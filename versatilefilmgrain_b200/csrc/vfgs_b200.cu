// vfgs_b200.cu -- C-ABI shim of libvfgs_b200.so: the host mirror of the reference's hardware
// state (vfgs_hw.c:49-63), its ten setters/entry points (vfgs_hw.c:288-388) and the additive
// frame-batch entry points of include/vfgs_b200.h. All sample processing happens in the CUDA
// kernels of vfgs_kernels.cuh; the host only keeps state, builds the table image, does the LFSR
// register bookkeeping by GF(2) jump-ahead and drives streams.
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <algorithm>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "../../include/vfgs_b200.h"
#include "../../include/vfgs_fw.h"
#include "../../include/vfgs_hw.h"
#include "../../include/yuv.h"
#include "vfgs_kernels.cuh"
#include "fw_host.h"

using namespace vfgs;

namespace {

// ------------------------------------------------------------------------------------ state
struct Slot { // one stage of the host pipeline
	uint8_t* d_in = nullptr;
	uint8_t* d_out = nullptr;
	uint32_t* d_streams = nullptr;
	size_t in_cap = 0, out_cap = 0, streams_cap = 0;
	cudaEvent_t h2d_done = nullptr, k_done = nullptr, d2h_done = nullptr;
};
constexpr int kPipeSlots = 4;
constexpr int kImageSets = 4;
constexpr size_t kImageBlobCap = 192u << 10, kImageFblobCap = 128u << 10; // upper bounds of build_tables' images
struct ImageSet {
	uint8_t* d_blob = nullptr;   // general image (+ negated slot copies)
	uint8_t* d_fblob = nullptr;  // fast-path image
	uint8_t* h_stage = nullptr;  // page-locked staging of both, the source of the asynchronous upload
	cudaEvent_t uploaded = nullptr, last_use = nullptr;
	bool in_use = false;
};
constexpr size_t kBlockTableBytes = sizeof(uint32_t) + 4 * sizeof(uint16_t); // per block: LFSR register + window offsets

struct Context {
	bool ready = false;
	int device = -1;
	int sm_count = 0;
	int max_smem_optin = 0;
	int fast_pad = 0;           // gap between the fast kernel's dynamic shared memory and the next 32 KB boundary (measured by a probe launch)
	uint32_t* d_pow2 = nullptr;
	// Table images (general + fast, vfgs_tables.h) live in a small ring of sets: a configuration change builds the next
	// set and uploads it asynchronously on the table stream, while frames already queued keep reading the set they were
	// launched with. A set is reused kImageSets changes later, after the last kernel that read it (last_use) is done.
	ImageSet img[kImageSets];
	int img_cur = -1;
	// firmware layer on the device (vfgs_b200_init_sei / _afgs1): constant tables, working memory, pattern store, staging
	FwTables* d_fw_tables = nullptr;
	FwScratch* d_fw_scratch = nullptr;
	int8_t* d_fw_pattern = nullptr;
	int8_t* h_fw_stage = nullptr;
	int fast_smem_attr = 0, gather_smem_attr = 0;
	uint32_t* d_streams = nullptr; // device entry point / line path
	size_t streams_cap = 0;
	cudaStream_t last_stream = nullptr;
	bool used_stream = false;
	cudaStream_t s_h2d = nullptr, s_k = nullptr, s_d2h = nullptr;
	// device entry point: the block tables of consecutive calls alternate between two buffers and are computed on a
	// side stream, so that the table kernel of call k + 1 runs under the grain kernel of call k
	cudaStream_t s_tab = nullptr;
	uint32_t* d_tab[2] = {nullptr, nullptr};
	size_t tab_cap[2] = {0, 0};
	cudaEvent_t tab_ready[2] = {nullptr, nullptr}, tab_free[2] = {nullptr, nullptr};
	bool tab_used[2] = {false, false};
	unsigned tab_next = 0;
	// descriptors of a batched call (vfgs_b200_add_grain_jobs_device): stream-kernel job table, per-job launch
	// parameters and task prefixes, staged in page-locked memory and copied on the table stream; they alternate with
	// d_tab (same tab_free events); desc_copied: the staging buffer may be rewritten
	uint8_t* h_desc[2] = {nullptr, nullptr};
	uint8_t* d_desc[2] = {nullptr, nullptr};
	size_t desc_cap[2] = {0, 0}, hdesc_cap[2] = {0, 0};
	cudaEvent_t desc_copied[2] = {nullptr, nullptr};
	bool desc_used[2] = {false, false};
	int multi_smem_attr[512] = {}; // per group key (group_key): the MULTI kernel's dynamic shared memory attribute
	int multi_occ_smem[512] = {}, multi_per_sm[512] = {}; // per group key: occupancy asked for that shared-memory size
	std::vector<std::shared_ptr<CUevent_st>> call_events; // end-of-call events of batched calls, reused once no session holds one
	Slot slot[kPipeSlots];
	uint8_t* d_line = nullptr; // compat line path staging
	size_t line_cap = 0;
	uint8_t* d_scratch = nullptr; // scratch output of in-place calls with sample-adaptive patterns
	size_t scratch_cap = 0;
	int smem_attr = 0;
	int last_launch[5] = {0, 0, 0, 0, 0};
	// optional per-launch timing of the grain kernel (vfgs_b200_kernel_timing)
	bool timing = false;
	std::vector<cudaEvent_t> ev_begin, ev_end;
	size_t ev_used = 0;
	double timed_ms = 0.0;
	uint64_t timed_launches = 0;
};

HwState g_hw;
bool g_hw_init = false;
Context g_ctx;
bool g_dirty = true; // table image must be rebuilt + uploaded
std::vector<uint8_t> g_blob;
TableInfo g_bi;
std::vector<uint8_t> g_fblob;
uint64_t g_launches = 0;
int g_kernel_mode = 0; // test hook: 0 auto, 1 general kernel everywhere, 2 gather kernel wherever it can run
char g_err[512] = "";
const JumpTable& jump_table()
{
	static const JumpTable t;
	return t;
}

HwState& hw()
{
	if (!g_hw_init) { g_hw.power_on(); g_hw_init = true; }
	return g_hw;
}

// frame pipeline hooks (yuv_pipeline.h, end of this file)
void pipe_before_state_change();
bool pipe_line(const void* Y, int y);

int set_err(int code, const char* fmt, ...)
{
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(g_err, sizeof(g_err), fmt, ap);
	va_end(ap);
	return code;
}

[[noreturn]] void fatal(const char* what)
{
	fprintf(stderr, "vfgs_b200: %s%s%s\n", what, g_err[0] ? ": " : "", g_err);
	abort();
}

#define REQUIRE(cond) \
	do { if (!(cond)) { snprintf(g_err, sizeof(g_err), "%s", #cond); fatal("precondition failed (the reference asserts here)"); } } while (0)

#define CUDA_TRY(expr) \
	do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return set_err(VFGS_B200_ERR_CUDA, "%s -> %s", #expr, cudaGetErrorString(e_)); } while (0)

// ------------------------------------------------------------------------------------ device ctx
int ensure_ctx(int device)
{
	static std::mutex mu; // the frame pipeline creates the context on its GPU-stage thread (yuv_pipeline.h)
	std::lock_guard<std::mutex> lock(mu);
	Context& c = g_ctx;
	if (c.ready && (device < 0 || device == c.device)) {
		CUDA_TRY(cudaSetDevice(c.device));
		return VFGS_B200_OK;
	}
	if (c.ready) return set_err(VFGS_B200_ERR_ARG, "library already bound to device %d", c.device);
	if (device < 0) CUDA_TRY(cudaGetDevice(&device));
	CUDA_TRY(cudaSetDevice(device));
	cudaDeviceProp prop;
	CUDA_TRY(cudaGetDeviceProperties(&prop, device));
	if (prop.major < 10)
		return set_err(VFGS_B200_ERR_CUDA, "device %d is sm_%d%d; this library carries sm_100a code only", device, prop.major, prop.minor);
	c.device = device;
	c.sm_count = prop.multiProcessorCount;
	c.max_smem_optin = (int)prop.sharedMemPerBlockOptin;
	CUDA_TRY(cudaMalloc(&c.d_pow2, sizeof(uint32_t) * kJumpBits * 32));
	{ // where the fast kernel's dynamic shared memory starts inside the shared window (behind the driver's reserved
	  // bytes and the kernel's static variables): asked of each variant by a one-thread probe launch, because the
	  // host lays the table images out for exactly that gap in front of the first LUT
		uint32_t* d_probe = (uint32_t*)c.d_pow2; // scratch: the jump table is uploaded right after
		FgsParams pp;
		memset(&pp, 0, sizeof(pp));
		pp.probe = d_probe;
		fgs_apply_fast_kernel<true, false><<<1, 32, 1024>>>(pp);
		pp.probe = d_probe + 1;
		fgs_apply_fast_kernel<true, true><<<1, 32, 1024>>>(pp);
		pp.probe = d_probe + 2;
		fgs_apply_fast_kernel<false, false><<<1, 32, 1024>>>(pp);
		pp.probe = d_probe + 3;
		fgs_apply_fast_kernel<true, false, false, true><<<1, 32, 1024>>>(pp);
		pp.probe = d_probe + 4;
		fgs_apply_fast_kernel<false, false, false, false, true><<<1, 32, 1024>>>(pp);
		pp.probe = d_probe + 5;
		fgs_apply_fast_kernel<true, true, false, false, true><<<1, 32, 1024>>>(pp);
		pp.probe = d_probe + 6;
		fgs_apply_fast_kernel<true, false, false, false, true><<<1, 32, 1024>>>(pp);
		pp.probe = d_probe + 7;
		fgs_apply_fast_kernel<true, false, false, true, true><<<1, 32, 1024>>>(pp);
		MultiParams mp; // the MULTI forms of the same variants (batched calls)
		memset(&mp, 0, sizeof(mp));
		mp.probe = d_probe + 8;
		fgs_apply_fast_multi_kernel<true, false><<<1, 32, 1024>>>(mp);
		mp.probe = d_probe + 9;
		fgs_apply_fast_multi_kernel<true, true><<<1, 32, 1024>>>(mp);
		mp.probe = d_probe + 10;
		fgs_apply_fast_multi_kernel<false, false><<<1, 32, 1024>>>(mp);
		mp.probe = d_probe + 11;
		fgs_apply_fast_multi_kernel<true, false, false, true><<<1, 32, 1024>>>(mp);
		mp.probe = d_probe + 12;
		fgs_apply_fast_multi_kernel<false, false, false, false, true><<<1, 32, 1024>>>(mp);
		mp.probe = d_probe + 13;
		fgs_apply_fast_multi_kernel<true, true, false, false, true><<<1, 32, 1024>>>(mp);
		mp.probe = d_probe + 14;
		fgs_apply_fast_multi_kernel<true, false, false, false, true><<<1, 32, 1024>>>(mp);
		mp.probe = d_probe + 15;
		fgs_apply_fast_multi_kernel<true, false, false, true, true><<<1, 32, 1024>>>(mp);
		uint32_t pads[16] = {};
		CUDA_TRY(cudaMemcpy(pads, d_probe, sizeof(pads), cudaMemcpyDeviceToHost));
		for (int i = 1; i < 16; i++)
			if (pads[i] != pads[0])
				return set_err(VFGS_B200_ERR_CUDA, "fast kernel variants place dynamic shared memory differently (%u, %u)", pads[0], pads[i]);
		c.fast_pad = (int)pads[0];
	}
	CUDA_TRY(cudaMemcpy(c.d_pow2, jump_table().pow2, sizeof(uint32_t) * kJumpBits * 32, cudaMemcpyHostToDevice));
	CUDA_TRY(cudaStreamCreateWithFlags(&c.s_h2d, cudaStreamNonBlocking));
	CUDA_TRY(cudaStreamCreateWithFlags(&c.s_k, cudaStreamNonBlocking));
	CUDA_TRY(cudaStreamCreateWithFlags(&c.s_d2h, cudaStreamNonBlocking));
	CUDA_TRY(cudaStreamCreateWithFlags(&c.s_tab, cudaStreamNonBlocking));
	for (int t = 0; t < 2; t++) {
		CUDA_TRY(cudaEventCreateWithFlags(&c.tab_ready[t], cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreateWithFlags(&c.tab_free[t], cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreateWithFlags(&c.desc_copied[t], cudaEventDisableTiming));
	}
	for (ImageSet& m : c.img) { // fixed-size allocations: nothing is (re)allocated, hence nothing synchronises, on a configuration change
		CUDA_TRY(cudaMalloc((void**)&m.d_blob, kImageBlobCap));
		CUDA_TRY(cudaMalloc((void**)&m.d_fblob, kImageFblobCap));
		CUDA_TRY(cudaHostAlloc((void**)&m.h_stage, kImageBlobCap + kImageFblobCap, cudaHostAllocDefault));
		CUDA_TRY(cudaEventCreateWithFlags(&m.uploaded, cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreateWithFlags(&m.last_use, cudaEventDisableTiming));
	}
	for (Slot& s : c.slot) {
		CUDA_TRY(cudaEventCreateWithFlags(&s.h2d_done, cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreateWithFlags(&s.k_done, cudaEventDisableTiming));
		CUDA_TRY(cudaEventCreateWithFlags(&s.d2h_done, cudaEventDisableTiming));
	}
	c.ready = true;
	g_dirty = true;
	return VFGS_B200_OK;
}

template <typename T>
int grow(T*& p, size_t& cap, size_t need)
{
	if (need <= cap) return VFGS_B200_OK;
	if (p) CUDA_TRY(cudaFree(p));
	p = nullptr; cap = 0;
	need = (need + 255) & ~(size_t)255;
	CUDA_TRY(cudaMalloc((void**)&p, need));
	cap = need;
	return VFGS_B200_OK;
}

// ------------------------------------------------------------------------------------ table image
void build_blob() { build_tables(hw(), g_bi, g_blob, g_fblob); }

int upload_blob()
{
	if (!g_dirty) return VFGS_B200_OK;
	Context& c = g_ctx;
	build_blob();
	if (g_bi.bytes > c.max_smem_optin - 1024)
		return set_err(VFGS_B200_ERR_STATE, "table image of %d bytes exceeds shared memory", g_bi.bytes);
	if ((size_t)g_bi.gbytes > kImageBlobCap || (size_t)g_bi.fbytes > kImageFblobCap)
		return set_err(VFGS_B200_ERR_STATE, "table images of %d + %d bytes exceed their buffers", g_bi.gbytes, g_bi.fbytes);
	// next set of the ring; frames in flight keep reading theirs. Only if the set is still being read by kernels
	// launched kImageSets configuration changes ago does the host wait, and then for those kernels alone.
	const int next = (c.img_cur + 1) % kImageSets;
	ImageSet& m = c.img[next];
	if (m.in_use) CUDA_TRY(cudaEventSynchronize(m.last_use));
	memcpy(m.h_stage, g_blob.data(), (size_t)g_bi.gbytes);
	memcpy(m.h_stage + kImageBlobCap, g_fblob.data(), (size_t)g_bi.fbytes);
	CUDA_TRY(cudaMemcpyAsync(m.d_blob, m.h_stage, (size_t)g_bi.gbytes, cudaMemcpyHostToDevice, c.s_tab));
	CUDA_TRY(cudaMemcpyAsync(m.d_fblob, m.h_stage + kImageBlobCap, (size_t)g_bi.fbytes, cudaMemcpyHostToDevice, c.s_tab));
	CUDA_TRY(cudaEventRecord(m.uploaded, c.s_tab));
	m.in_use = false;
	c.img_cur = next;
	if (g_bi.bytes > c.smem_attr) {
		CUDA_TRY(cudaFuncSetAttribute(fgs_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, g_bi.bytes));
		c.smem_attr = g_bi.bytes;
	}
	g_dirty = false;
	return VFGS_B200_OK;
}

// The state a grain launch works on: the global one (g_hw, g_bi, the current image set) or a session's copy.
struct StateRef {
	HwState* h;
	const TableInfo* bi;
	ImageSet* img;
};
StateRef global_state() { return {&hw(), &g_bi, g_ctx.img_cur >= 0 ? &g_ctx.img[g_ctx.img_cur] : nullptr}; }

// Grain kernels about to be launched on `stream` read the state's image set: they wait for its upload, and the set
// remembers the last stream position that reads it.
int images_before(const StateRef& s, cudaStream_t stream)
{
	CUDA_TRY(cudaStreamWaitEvent(stream, s.img->uploaded, 0));
	return VFGS_B200_OK;
}
int images_after(const StateRef& s, cudaStream_t stream)
{
	CUDA_TRY(cudaEventRecord(s.img->last_use, stream));
	s.img->in_use = true;
	return VFGS_B200_OK;
}

// ------------------------------------------------------------------------------------ launch
struct Geometry {
	int width, height, cw, ch, nb, R, spitch;
	int in_depth, out_depth;
	size_t in_sample, out_sample;
	size_t ysam, csam;
	size_t in_frame_bytes, out_frame_bytes;
};

int make_geometry(Geometry& g, const HwState& h, int width, int height, int out_depth)
{
	// what add_grain_block asserts (vfgs_hw.c:168-170)
	if (width <= 128) return set_err(VFGS_B200_ERR_STATE, "width must exceed 128 (vfgs_hw.c:168)");
	if (h.scale_shift + h.bs < 8 || h.scale_shift + h.bs > 13)
		return set_err(VFGS_B200_ERR_STATE, "scale_shift %d + bs %d outside 8..13 (vfgs_hw.c:170)", h.scale_shift, h.bs);
	if (height < 1) return set_err(VFGS_B200_ERR_ARG, "height %d", height);
	for (int c = 0; c < 3; c++)
		for (int i = 0; i < 256; i++)
			if ((h.plut[c][i] >> 4) >= kSlots)
				return set_err(VFGS_B200_ERR_STATE, "pattern LUT %d entry %d selects slot %d: the hardware has slots 0..8 (vfgs_hw.c:49,218)", c, i, h.plut[c][i] >> 4);
	g.in_depth = 8 + h.bs;
	g.out_depth = out_depth ? out_depth : g.in_depth;
	if (g.out_depth != g.in_depth && !(g.out_depth == 8 && g.in_depth == 10))
		return set_err(VFGS_B200_ERR_ARG, "out_depth %d with input depth %d", out_depth, g.in_depth);
	g.width = width; g.height = height;
	g.cw = width / h.csubx; g.ch = height / h.csuby; // yuv.c:72-77
	g.nb = (width + 15) / 16; g.R = (height + 15) / 16;
	g.spitch = g.nb + 2;
	g.in_sample = g.in_depth > 8 ? 2 : 1; g.out_sample = g.out_depth > 8 ? 2 : 1;
	g.ysam = (size_t)width * height; g.csam = (size_t)g.cw * g.ch;
	g.in_frame_bytes = (g.ysam + 2 * g.csam) * g.in_sample;
	g.out_frame_bytes = (g.ysam + 2 * g.csam) * g.out_sample;
	return VFGS_B200_OK;
}
int make_geometry(Geometry& g, int width, int height, int out_depth) { return make_geometry(g, hw(), width, height, out_depth); }

void fill_common(FgsParams& p, const Geometry& g, const StateRef& s)
{
	memset(&p, 0, sizeof(p));
	fill_state_params(p, *s.h, *s.bi);
	p.nb = g.nb; p.R = g.R;
	p.in_bytes = (int)g.in_sample; p.out_bytes = (int)g.out_sample;
	p.blob = s.img ? s.img->d_blob : nullptr;
	p.fblob = s.img ? s.img->d_fblob : nullptr;
	p.spitch = g.spitch;
}

typedef void (*GrainKernel)(const FgsParams);
enum KernelKind { kGeneral = 0, kFast = 1, kGather = 2, kFastEdge = 3 };

template <bool FOLD, bool SHIFT>
GrainKernel gather_kernel(const FgsParams& p)
{
	if (p.msb_in) // P010 luma of semi-planar frames
		return p.out_bytes == 1 ? fgs_apply_gather_kernel<true, true, FOLD, SHIFT, true> : fgs_apply_gather_kernel<true, false, FOLD, SHIFT, true>;
	return p.in_bytes == 1 ? fgs_apply_gather_kernel<false, false, FOLD, SHIFT>
	     : p.out_bytes == 1 ? fgs_apply_gather_kernel<true, true, FOLD, SHIFT> : fgs_apply_gather_kernel<true, false, FOLD, SHIFT>;
}
GrainKernel gather_kernel(const FgsParams& p, bool fold, bool shift)
{
	return fold ? (shift ? gather_kernel<true, true>(p) : gather_kernel<true, false>(p))
	            : (shift ? gather_kernel<false, true>(p) : gather_kernel<false, false>(p));
}

int launch_apply(const FgsParams& p, cudaStream_t stream, KernelKind kind = kGeneral, int gather_smem = 0, bool gather_fold = false,
                 bool gather_shift = false)
{
	Context& c = g_ctx;
	if (p.total_tasks <= 0) return VFGS_B200_OK;
	if (p.total_tasks >= (1ll << 31)) return set_err(VFGS_B200_ERR_ARG, "batch too large for one launch (%lld warp-tasks): split the call", p.total_tasks);
	GrainKernel kern = fgs_apply_kernel;
	int threads = kCtaThreads, smem = p.blob_bytes;
	if (kind == kFast || kind == kFastEdge) {
		const bool allwide = kind == kFast && p.in_bytes == 2 && p.out_bytes == 2 && p.fallwide;
		if (kind == kFast && p.ilv[1]) // semi-planar frames
			kern = allwide ? fgs_apply_fast_kernel<true, false, false, true, true>
			     : p.in_bytes == 1 ? fgs_apply_fast_kernel<false, false, false, false, true>
			     : p.out_bytes == 1 ? fgs_apply_fast_kernel<true, true, false, false, true> : fgs_apply_fast_kernel<true, false, false, false, true>;
		else if (allwide)
			kern = fgs_apply_fast_kernel<true, false, false, true>;
		else if (kind == kFast)
			kern = p.in_bytes == 1 ? fgs_apply_fast_kernel<false, false>
			     : p.out_bytes == 1 ? fgs_apply_fast_kernel<true, true> : fgs_apply_fast_kernel<true, false>;
		else
			kern = p.in_bytes == 1 ? fgs_apply_fast_kernel<false, false, true>
			     : p.out_bytes == 1 ? fgs_apply_fast_kernel<true, true, true> : fgs_apply_fast_kernel<true, false, true>;
		threads = fast_threads(p.in_bytes == 2, p.in_bytes == 2 && p.out_bytes == 1, kind == kFastEdge, allwide); smem = p.fsmem;
		if (smem > c.fast_smem_attr) {
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<false, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			CUDA_TRY(cudaFuncSetAttribute(fgs_apply_fast_kernel<true, false, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			c.fast_smem_attr = smem;
		}
	} else if (kind == kGather) {
		kern = gather_kernel(p, gather_fold, gather_shift);
		threads = kGatherThreads; smem = gather_smem;
		if (smem > c.gather_smem_attr) {
			FgsParams v = p; // every variant of the gather kernel
			for (int io = 0; io < 5; io++) {
				v.in_bytes = io == 0 ? 1 : 2; v.out_bytes = io == 2 || io == 4 ? 2 : 1;
				v.msb_in = io >= 3 ? 6 : 0;
				for (int fs = 0; fs < 4; fs++)
					CUDA_TRY(cudaFuncSetAttribute(gather_kernel(v, (fs & 1) != 0, (fs & 2) != 0), cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			}
			c.gather_smem_attr = smem;
		}
	}
	const int wpc = threads / 32;
	int per_sm = 0;
	CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, (size_t)smem));
	if (per_sm < 1) return set_err(VFGS_B200_ERR_CUDA, "grain kernel does not fit on an SM (smem %d)", smem);
	long long want = (p.total_tasks + wpc - 1) / wpc;
	long long cap = (long long)c.sm_count * per_sm; // persistent grid: a whole number of CTAs per SM
	int grid = (int)(want < cap ? want : cap);
	cudaEvent_t e0 = nullptr, e1 = nullptr;
	if (c.timing) {
		if (c.ev_used == c.ev_begin.size()) {
			cudaEvent_t a, b;
			CUDA_TRY(cudaEventCreate(&a));
			CUDA_TRY(cudaEventCreate(&b));
			c.ev_begin.push_back(a); c.ev_end.push_back(b);
		}
		e0 = c.ev_begin[c.ev_used]; e1 = c.ev_end[c.ev_used]; c.ev_used++;
		CUDA_TRY(cudaEventRecord(e0, stream));
	}
	kern<<<grid, threads, (size_t)smem, stream>>>(p);
	CUDA_TRY(cudaGetLastError());
	if (c.timing) CUDA_TRY(cudaEventRecord(e1, stream));
	g_launches++;
	c.last_launch[0] = grid; c.last_launch[1] = threads; c.last_launch[2] = smem; c.last_launch[3] = c.sm_count;
	c.last_launch[4] |= kind == kFast ? 1 : kind == kGather ? 4 : kind == kFastEdge ? 8 : 2;
	return VFGS_B200_OK;
}

int launch_streams(uint32_t epoch, uint32_t* d_streams, uint16_t* d_woffs, const WoffParams& wp, int nframes, const Geometry& g, uint64_t frame0, cudaStream_t stream)
{
	// 128-thread CTAs (4096 registers each) fit beside a resident 768-thread grain CTA
	const long long warps = (long long)nframes * g.R;
	const int grid = (int)((warps * 32 + kLfsrThreads - 1) / kLfsrThreads);
	lfsr_states_kernel<<<grid, kLfsrThreads, 0, stream>>>(epoch, g_ctx.d_pow2, d_streams, d_woffs, wp, nframes, g.R, g.nb, g.spitch, frame0);
	CUDA_TRY(cudaGetLastError());
	g_launches++;
	return VFGS_B200_OK;
}

// Register state after nframes whole frames (vfgs_hw.c:291-298,309-310 in closed form).
void advance_registers(HwState& h, const Geometry& g, uint64_t nframes) { advance_frames(h, g.R, g.nb, nframes, jump_table()); }

// One side of a frame call: three planes (planar), or a Y plane and one plane of interleaved U,V pairs (semi-planar:
// plane[1] holds both, plane[2] is unused).
struct FramePlanes {
	uint8_t* plane[3];
	int64_t stride[3];
	int64_t frame_stride;
	bool semi, msb; // msb: P010 samples (value in bits 15..6)
};
FramePlanes frame_planes(const vfgs_b200_planes& pl)
{
	FramePlanes f;
	f.plane[0] = (uint8_t*)pl.y; f.plane[1] = (uint8_t*)pl.u; f.plane[2] = (uint8_t*)pl.v;
	f.stride[0] = pl.stride_y; f.stride[1] = f.stride[2] = pl.stride_c;
	f.frame_stride = pl.frame_stride;
	f.semi = f.msb = false;
	return f;
}
FramePlanes frame_planes(const vfgs_b200_semiplanar& pl)
{
	FramePlanes f;
	f.plane[0] = (uint8_t*)pl.y; f.plane[1] = (uint8_t*)pl.uv; f.plane[2] = nullptr;
	f.stride[0] = pl.stride_y; f.stride[1] = pl.stride_uv; f.stride[2] = 0;
	f.frame_stride = pl.frame_stride;
	f.semi = true; f.msb = pl.format == VFGS_B200_P010;
	return f;
}
// Bytes of one frame's row of plane c and its line count (0 for the unused plane of a semi-planar side).
int64_t plane_row_bytes(const FramePlanes& f, int c, const Geometry& g, size_t sample)
{
	return (int64_t)(c ? (f.semi ? (c == 1 ? 2 * g.cw : 0) : g.cw) : g.width) * (int64_t)sample;
}
int64_t plane_lines(const FramePlanes& f, int c, const Geometry& g) { return (f.semi && c == 2) ? 0 : c ? g.ch : g.height; }

// Launch parameters and kernel assignment of a whole-frame call.
void plan_frames(const StateRef& s, const FramePlanes& in, const FramePlanes& out, int n, const Geometry& g, bool in_place,
                 uint32_t* d_streams, FgsParams& p, LaunchPlan& lp, uint16_t*& d_woffs)
{
	fill_common(p, g, s);
	p.nframes = n;
	p.y_begin = 0; p.y_end = g.height;
	p.row_begin = 0; p.rows = g.R;
	p.in_frame_bytes = in.frame_stride; p.out_frame_bytes = out.frame_stride;
	if (in.semi) {
		set_semiplanar_planes(p, in.plane[0], in.plane[1], in.stride[0], in.stride[1], out.plane[0], out.plane[1], out.stride[0],
		                      out.stride[1], g.width, g.height, g.cw, g.ch, in.msb, out.msb);
	} else {
		for (int c = 0; c < 3; c++) {
			p.comp[c].in = in.plane[c]; p.comp[c].out = out.plane[c];
			p.comp[c].in_row_bytes = in.stride[c];
			p.comp[c].out_row_bytes = out.stride[c];
			p.comp[c].width = c ? g.cw : g.width;
			p.comp[c].lines = c ? g.ch : g.height;
		}
	}
	// one allocation holds both per-block tables: uint32 registers, then 4 x uint16 window offsets
	d_woffs = (uint16_t*)(d_streams + (((size_t)n * g.R * g.spitch + 3) & ~(size_t)3)); // 16-byte aligned
	p.states = d_streams; p.woffs = d_woffs; p.stream_rows = g.R; p.stream_row0 = 0;
	finish_tasks(p);
	// every component goes to the cheapest kernel that can serve it (plan_launches)
	plan_launches(p, *s.bi, g_kernel_mode, in_place, g_ctx.max_smem_optin - 1024, g_ctx.fast_pad, lp);
}

// Streams + grain kernels for `n` frames whose epoch-relative index starts at frame0.
int run_frames_device(const StateRef& s, const FramePlanes& in, const FramePlanes& out, int n, const Geometry& g, bool in_place,
                      uint32_t epoch, uint64_t frame0, uint32_t* d_streams, cudaStream_t stream,
                      cudaStream_t table_stream = nullptr, cudaEvent_t table_ready = nullptr)
{
	FgsParams p;
	LaunchPlan lp;
	uint16_t* d_woffs = nullptr;
	plan_frames(s, in, out, n, g, in_place, d_streams, p, lp, d_woffs);
	g_ctx.last_launch[4] = 0;
	// the register table feeds the general kernel, the window-offset table the fast and gather kernels
	if (int rc = launch_streams(epoch, lp.any_general ? d_streams : nullptr, (lp.any_fast || lp.any_gather || lp.any_edge) ? d_woffs : nullptr,
	                            make_woff_params(p, lp.kind), n, g, frame0, table_stream ? table_stream : stream)) return rc;
	if (table_stream) { // the tables were computed beside the caller's stream: the grain kernels wait for them
		CUDA_TRY(cudaEventRecord(table_ready, table_stream));
		CUDA_TRY(cudaStreamWaitEvent(stream, table_ready, 0));
	}
	if (int rc = images_before(s, stream)) return rc;
	if (lp.any_fast)
		if (int rc = launch_apply(lp.fast, stream, kFast)) return rc;
	if (lp.any_edge)
		if (int rc = launch_apply(lp.edge, stream, kFastEdge)) return rc;
	if (lp.any_gather)
		if (int rc = launch_apply(lp.gather, stream, kGather, lp.gather_smem, lp.gather_fold, lp.gather_shift)) return rc;
	if (lp.any_general)
		if (int rc = launch_apply(lp.general, stream, kGeneral)) return rc;
	if (lp.any_fast && in.semi && lp.fast.fwide[1]) g_ctx.last_launch[4] |= 16; // the interleaved U/V lane ran
	return images_after(s, stream);
}

// How the output planes lie relative to the input planes: 0 disjoint, 1 in place (every overlapping plane pair is
// the same plane with the same strides and row bytes), -1 anything else (partial overlap: not supported).
// Planes of consecutive frames interleave in memory (Y0 U0 V0 Y1 ...), so plane pairs are compared frame by frame in
// closed form: with a common frame stride S, frame f1 of one plane meets frame f2 of the other iff their byte
// extents overlap for some k = f1 - f2 within the batch. A semi-planar side has two planes (Y, interleaved UV).
// One side of an overlap test: planes, frame count, geometry and bytes per sample.
struct Side {
	const FramePlanes& f;
	int n;
	const Geometry& g;
	size_t sample;
};
int64_t plane_extent(const Side& s, int c) // bytes one frame's plane spans
{
	const int64_t lines = plane_lines(s.f, c, s.g), row = plane_row_bytes(s.f, c, s.g, s.sample);
	if (lines < 1 || row < 1) return 0;
	return (lines - 1) * s.f.stride[c] + row;
}
// Bounding byte range [lo, hi) of a side's buffers (lo null: no bytes).
void side_span(const Side& s, const uint8_t*& lo, const uint8_t*& hi)
{
	lo = hi = nullptr;
	for (int c = 0; c < 3; c++) {
		const int64_t e = plane_extent(s, c);
		if (e <= 0) continue;
		const uint8_t* end = s.f.plane[c] + (int64_t)(s.n - 1) * s.f.frame_stride + e;
		if (!lo || s.f.plane[c] < lo) lo = s.f.plane[c];
		if (!hi || end > hi) hi = end;
	}
}
int overlap(const Side& a, const Side& b)
{
	const uint8_t *alo, *ahi, *blo, *bhi;
	side_span(a, alo, ahi);
	side_span(b, blo, bhi);
	if (!alo || !blo || ahi <= blo || bhi <= alo) return 0;
	if (a.n > 1 && b.n > 1 && a.f.frame_stride != b.f.frame_stride) return -1; // overlapping buffers walked with different strides
	const int64_t S = a.n > 1 ? a.f.frame_stride : b.f.frame_stride;
	int result = 0;
	for (int i = 0; i < 3; i++)
		for (int j = 0; j < 3; j++) {
			const int64_t ei = plane_extent(a, i), ej = plane_extent(b, j);
			if (ei <= 0 || ej <= 0) continue;
			const bool same = i == j && a.f.plane[i] == b.f.plane[j] && a.f.stride[i] == b.f.stride[j] &&
			                  plane_row_bytes(a.f, i, a.g, a.sample) == plane_row_bytes(b.f, j, b.g, b.sample) && a.f.msb == b.f.msb;
			bool hit;
			if ((a.n > 1 || b.n > 1) && S > 0) {
				// frame f1 of plane i against frame f2 of plane j: [f1 S, f1 S + ei) meets [D + f2 S, D + f2 S + ej)
				// iff D - ei < k S < D + ej for k = f1 - f2, -(b.n - 1) <= k <= a.n - 1
				const int64_t D = (int64_t)(b.f.plane[j] - a.f.plane[i]);
				auto floor_div = [](int64_t x, int64_t y) { int64_t q = x / y; return (x % y != 0 && ((x < 0) != (y < 0))) ? q - 1 : q; };
				int64_t k_lo = floor_div(D - ei, S) + 1, k_hi = -floor_div(-(D + ej), S) - 1;
				if (k_lo < -(int64_t)(b.n - 1)) k_lo = -(int64_t)(b.n - 1);
				if (k_hi > (int64_t)(a.n - 1)) k_hi = (int64_t)(a.n - 1);
				hit = k_lo <= k_hi;
			} else {
				hit = !(a.f.plane[i] + ei <= b.f.plane[j] || b.f.plane[j] + ej <= a.f.plane[i]);
			}
			if (!hit) continue;
			if (!same) return -1;
			result = 1;
		}
	return result;
}
int aliasing(const FramePlanes& in, const FramePlanes& out, int n, const Geometry& g)
{
	return overlap({in, n, g, g.in_sample}, {out, n, g, g.out_sample});
}

void packed_planes(vfgs_b200_planes& pl, const void* base, const Geometry& g, size_t sample, size_t frame_bytes)
{
	uint8_t* b = (uint8_t*)base;
	pl.y = b; pl.u = b + g.ysam * sample; pl.v = b + (g.ysam + g.csam) * sample;
	pl.stride_y = (int64_t)(g.width * sample); pl.stride_c = (int64_t)(g.cw * sample);
	pl.frame_stride = (int64_t)frame_bytes;
}

// Argument checks of a semi-planar call on state h, before any device work, and its geometry.
int semiplanar_geometry(Geometry& g, const HwState& h, const vfgs_b200_semiplanar& in, const vfgs_b200_semiplanar& out, int width, int height)
{
	if (!in.y || !in.uv || !out.y || !out.uv) return set_err(VFGS_B200_ERR_ARG, "null plane pointer");
	const int depth = 8 + h.bs;
	if (in.format != (depth == 10 ? VFGS_B200_P010 : VFGS_B200_NV12))
		return set_err(VFGS_B200_ERR_ARG, "input format %d does not match the configured depth %d (NV12 = 8, P010 = 10)", in.format, depth);
	if (out.format != in.format && !(out.format == VFGS_B200_NV12 && in.format == VFGS_B200_P010))
		return set_err(VFGS_B200_ERR_ARG, "output format %d from input format %d (same format, or NV12 from P010)", out.format, in.format);
	if (h.csubx != 2)
		return set_err(VFGS_B200_ERR_ARG, "semi-planar frames are 4:2:0 or 4:2:2 (4:4:4 frames are planar)");
	if (int rc = make_geometry(g, h, width, height, out.format == in.format ? 0 : 8)) return rc;
	for (int side = 0; side < 2; side++) {
		const vfgs_b200_semiplanar& f = side ? out : in;
		const int64_t sample = (int64_t)(side ? g.out_sample : g.in_sample);
		if (f.stride_y < (int64_t)g.width * sample || f.stride_uv < 2 * (int64_t)g.cw * sample)
			return set_err(VFGS_B200_ERR_ARG, "%s line stride shorter than a row", side ? "output" : "input");
		if (sample == 2 && (((uintptr_t)f.y | (uintptr_t)f.uv | (uint64_t)f.stride_y | (uint64_t)f.stride_uv | (uint64_t)f.frame_stride) & 1))
			return set_err(VFGS_B200_ERR_ARG, "%s P010 planes and strides must be 2-byte aligned", side ? "output" : "input");
	}
	return VFGS_B200_OK;
}

// Mirror of a hardware state in the layout of the reference's statics (see oracle/ref_harness.c refh_state):
// pattern[2][9][64][64], sLUT[3][256], pLUT[3][256], 4 LFSR registers, then scale_shift, bs, Y_min, Y_max, C_min, C_max,
// csubx, csuby as ints (vfgs_b200_get_state, vfgs_b200_session_get_state).
size_t state_dump(const HwState& h, void* dst, size_t cap)
{
	const size_t need = sizeof(h.pattern) + sizeof(h.slut) + sizeof(h.plut) + 4 * sizeof(uint32_t) + 8 * sizeof(int);
	if (!dst || cap < need) return need;
	uint8_t* p = (uint8_t*)dst;
	memcpy(p, h.pattern, sizeof(h.pattern)); p += sizeof(h.pattern);
	memcpy(p, h.slut, sizeof(h.slut)); p += sizeof(h.slut);
	memcpy(p, h.plut, sizeof(h.plut)); p += sizeof(h.plut);
	const uint32_t regs[4] = {h.rnd, h.rnd_up, h.line_rnd, h.line_rnd_up};
	memcpy(p, regs, sizeof(regs)); p += sizeof(regs);
	const int sc[8] = {h.scale_shift, h.bs, h.y_min, h.y_max, h.c_min, h.c_max, h.csubx, h.csuby};
	memcpy(p, sc, sizeof(sc));
	return need;
}

int prepare(int device)
{
	if (int rc = ensure_ctx(device)) return rc;
	return upload_blob();
}

// An in-place call whose plan puts a sample-adaptive component on the general kernel (in_place_needs_scratch).
bool needs_scratch(const StateRef& s, const FramePlanes& in, const FramePlanes& out, int nframes, const Geometry& g)
{
	FgsParams pp; LaunchPlan lpp; uint16_t* w = nullptr; // cheap host-side planning pass: which kernels would serve the components
	plan_frames(s, in, out, nframes, g, true, nullptr, pp, lpp, w);
	return in_place_needs_scratch(lpp, *s.bi);
}

int stream_switch(cudaStream_t st)
{
	Context& c = g_ctx;
	if (c.used_stream && c.last_stream != st) CUDA_TRY(cudaStreamSynchronize(c.last_stream)); // d_streams is shared
	c.last_stream = st; c.used_stream = true;
	return VFGS_B200_OK;
}

// Grain launches of one whole-frame call on state `s` (its registers advance), through a scratch output buffer where
// in place would not be safe. alias: what aliasing() found (0 or 1).
int run_job(const StateRef& s, const FramePlanes& in, const FramePlanes& out, int nframes, const Geometry& g, int alias, cudaStream_t st)
{
	const bool in_place = alias == 1;
	Context& c = g_ctx;
	if (in_place && needs_scratch(s, in, out, nframes, g)) {
		// In place with sample-adaptive pattern selection on a kernel that reads the neighbouring block's INPUT
		// sample (see in_place_needs_scratch), which another warp may already have overwritten. The frames go
		// through a scratch output buffer (packed, in the caller's layout) in sub-batches and are copied back (two
		// extra passes over the data; the reference's own in-place order, block after block along a line, has no
		// such hazard).
		const size_t fb = g.out_frame_bytes;
		int per = (int)((256u << 20) / fb);
		if (per < 1) per = 1;
		if (per > nframes) per = nframes;
		if (int rc = grow(c.d_scratch, c.scratch_cap, (size_t)per * fb)) return rc;
		if (int rc = grow(c.d_streams, c.streams_cap, (size_t)per * g.R * g.spitch * kBlockTableBytes + 16)) return rc;
		const uint32_t epoch = s.h->line_rnd;
		const int nplanes = in.semi ? 2 : 3;
		FramePlanes po = out;
		size_t soff[3] = {0, 0, 0};
		for (int k = 0; k < nplanes; k++) { // packed scratch frames: the planes back to back, rows tightly packed
			po.stride[k] = plane_row_bytes(out, k, g, g.out_sample);
			if (k + 1 < 3) soff[k + 1] = soff[k] + (size_t)po.stride[k] * (size_t)plane_lines(out, k, g);
		}
		po.frame_stride = (int64_t)fb;
		for (int f0 = 0; f0 < nframes; f0 += per) {
			const int n = nframes - f0 < per ? nframes - f0 : per;
			FramePlanes pi = in;
			for (int k = 0; k < nplanes; k++) {
				pi.plane[k] = in.plane[k] + (size_t)f0 * in.frame_stride;
				po.plane[k] = c.d_scratch + soff[k];
			}
			if (int rc = run_frames_device(s, pi, po, n, g, false, epoch, (uint64_t)f0, c.d_streams, st)) return rc;
			for (int f = 0; f < n; f++) // rows of the caller's planes may be padded: 2-D copies, plane by plane
				for (int k = 0; k < nplanes; k++) {
					const size_t row = (size_t)po.stride[k];
					CUDA_TRY(cudaMemcpy2DAsync(out.plane[k] + (size_t)(f0 + f) * out.frame_stride, (size_t)out.stride[k],
					                           c.d_scratch + (size_t)f * fb + soff[k], row, row, (size_t)plane_lines(out, k, g),
					                           cudaMemcpyDeviceToDevice, st));
				}
		}
		advance_registers(*s.h, g, (uint64_t)nframes);
		return VFGS_B200_OK;
	}
	const int t = (int)(c.tab_next++ & 1u);
	if (int rc = grow(c.d_tab[t], c.tab_cap[t], (size_t)nframes * g.R * g.spitch * kBlockTableBytes + 16)) return rc;
	if (c.tab_used[t]) CUDA_TRY(cudaStreamWaitEvent(c.s_tab, c.tab_free[t], 0)); // the grain kernels of two calls ago read this buffer
	if (int rc = run_frames_device(s, in, out, nframes, g, in_place, s.h->line_rnd, 0, c.d_tab[t], st, c.s_tab, c.tab_ready[t])) return rc;
	CUDA_TRY(cudaEventRecord(c.tab_free[t], st));
	c.tab_used[t] = true;
	advance_registers(*s.h, g, (uint64_t)nframes);
	return VFGS_B200_OK;
}

// Body of the device frame entry points, after their own argument checks: overlap check (before any device work),
// then the grain launches on the global state.
int run_call(const FramePlanes& in, const FramePlanes& out, int nframes, const Geometry& g, cudaStream_t st)
{
	const int alias = nframes ? aliasing(in, out, nframes, g) : 0; // argument check first: needs no device
	if (alias < 0)
		return set_err(VFGS_B200_ERR_ARG, g.in_depth != g.out_depth ? "in-place needs equal depths"
		               : "input and output planes overlap without being identical (same planes, strides and depth)");
	if (int rc = prepare(-1)) return rc;
	if (nframes == 0) return VFGS_B200_OK;
	if (int rc = stream_switch(st)) return rc;
	return run_job(global_state(), in, out, nframes, g, alias, st);
}

} // namespace

// A session: a snapshot of one complete hardware state with its own table images in device memory (built once, never
// rewritten, so no ring and no reuse wait). last_batch: the event after the last batched launch that read it; the
// image set's last_use covers the single-job route.
struct vfgs_b200_session {
	HwState hw;
	TableInfo bi;
	ImageSet img;
	bool uploaded = false; // the upload is known to be complete: launches need not wait for it
	std::shared_ptr<CUevent_st> last_batch;
};

namespace {

StateRef session_state(vfgs_b200_session* s) { return {&s->hw, &s->bi, &s->img}; }

// One job of a batched call after its argument checks.
struct JobPlan {
	vfgs_b200_session* s;
	FramePlanes in, out;
	Geometry g;
	int n, alias;
	bool batched;       // served by the MULTI launches (else by the single-job route)
	LaunchPlan lp;
	uint32_t epoch;     // the session's line_rnd at enqueue
	size_t tab_off;     // bytes into d_tab of its window-offset table
};

typedef void (*MultiKernel)(const MultiParams);

template <bool FOLD, bool SHIFT>
MultiKernel gather_multi_kernel(bool in16, bool out8, bool msb)
{
	if (msb) return out8 ? fgs_apply_gather_multi_kernel<true, true, FOLD, SHIFT, true> : fgs_apply_gather_multi_kernel<true, false, FOLD, SHIFT, true>;
	return !in16 ? fgs_apply_gather_multi_kernel<false, false, FOLD, SHIFT>
	     : out8 ? fgs_apply_gather_multi_kernel<true, true, FOLD, SHIFT> : fgs_apply_gather_multi_kernel<true, false, FOLD, SHIFT>;
}

// The MULTI instantiation of a group key (group_key; kinds numbered as LaunchPlan::kind: 0 fast, 1 gather, 3 EDGE) and
// its CTA size: the same choice launch_apply makes for one job.
MultiKernel multi_kernel(int key, int& threads)
{
	const int kind = key & 3;
	const bool in16 = key & 4, out8 = key & 8, allwide = key & 16, semi = key & 32;
	if (kind == 1) {
		threads = kGatherThreads;
		const bool fold = key & 64, shift = key & 128, msb = key & 256;
		return fold ? (shift ? gather_multi_kernel<true, true>(in16, out8, msb) : gather_multi_kernel<true, false>(in16, out8, msb))
		            : (shift ? gather_multi_kernel<false, true>(in16, out8, msb) : gather_multi_kernel<false, false>(in16, out8, msb));
	}
	threads = fast_threads(in16, in16 && out8, kind == 3, allwide);
	if (kind == 3)
		return !in16 ? fgs_apply_fast_multi_kernel<false, false, true> : out8 ? fgs_apply_fast_multi_kernel<true, true, true> : fgs_apply_fast_multi_kernel<true, false, true>;
	if (semi)
		return allwide ? fgs_apply_fast_multi_kernel<true, false, false, true, true>
		     : !in16 ? fgs_apply_fast_multi_kernel<false, false, false, false, true>
		     : out8 ? fgs_apply_fast_multi_kernel<true, true, false, false, true> : fgs_apply_fast_multi_kernel<true, false, false, false, true>;
	if (allwide) return fgs_apply_fast_multi_kernel<true, false, false, true>;
	return !in16 ? fgs_apply_fast_multi_kernel<false, false> : out8 ? fgs_apply_fast_multi_kernel<true, true> : fgs_apply_fast_multi_kernel<true, false>;
}

// Argument checks of one job against its session's state (what the single-job entry points refuse), and its geometry.
int check_job(const vfgs_b200_job& j, int k, JobPlan& jp)
{
	if (!j.session) return set_err(VFGS_B200_ERR_ARG, "job %d: null session", k);
	const bool planar = j.in || j.out, semi = j.sp_in || j.sp_out;
	if (planar == semi) return set_err(VFGS_B200_ERR_ARG, "job %d: set exactly one of the planar and the semi-planar pairs", k);
	if (planar ? !(j.in && j.out) : !(j.sp_in && j.sp_out)) return set_err(VFGS_B200_ERR_ARG, "job %d: null planes", k);
	if (j.nframes < 0) return set_err(VFGS_B200_ERR_ARG, "job %d: negative frame count", k);
	jp.s = j.session;
	jp.n = j.nframes;
	if (planar) {
		if (int rc = make_geometry(jp.g, j.session->hw, j.width, j.height, j.out_depth)) return rc;
		jp.in = frame_planes(*j.in); jp.out = frame_planes(*j.out);
	} else {
		if (j.out_depth) return set_err(VFGS_B200_ERR_ARG, "job %d: out_depth is 0 for semi-planar jobs (the output format selects it)", k);
		if (int rc = semiplanar_geometry(jp.g, j.session->hw, *j.sp_in, *j.sp_out, j.width, j.height)) return rc;
		jp.in = frame_planes(*j.sp_in); jp.out = frame_planes(*j.sp_out);
	}
	jp.alias = jp.n ? aliasing(jp.in, jp.out, jp.n, jp.g) : 0;
	if (jp.alias < 0)
		return set_err(VFGS_B200_ERR_ARG, jp.g.in_depth != jp.g.out_depth ? "job %d: in-place needs equal depths"
		               : "job %d: input and output planes overlap without being identical (same planes, strides and depth)", k);
	return VFGS_B200_OK;
}

// Refuses a call in which the buffers of two jobs overlap (in place within one job stays allowed): jobs sorted by the
// start of their bounding byte range, each tested against the following ones whose range starts before its own ends.
int check_disjoint(const std::vector<JobPlan>& jp)
{
	struct Span { const uint8_t *lo, *hi; int k; };
	std::vector<Span> sp;
	for (int k = 0; k < (int)jp.size(); k++) {
		const JobPlan& j = jp[k];
		if (!j.n) continue;
		const uint8_t *ilo, *ihi, *olo, *ohi;
		side_span({j.in, j.n, j.g, j.g.in_sample}, ilo, ihi);
		side_span({j.out, j.n, j.g, j.g.out_sample}, olo, ohi);
		if (!ilo && !olo) continue;
		sp.push_back({!ilo ? olo : !olo ? ilo : std::min(ilo, olo), std::max(ihi, ohi), k});
	}
	std::sort(sp.begin(), sp.end(), [](const Span& a, const Span& b) { return a.lo < b.lo; });
	for (size_t x = 0; x < sp.size(); x++)
		for (size_t y = x + 1; y < sp.size() && sp[y].lo < sp[x].hi; y++) {
			const JobPlan &a = jp[sp[x].k], &b = jp[sp[y].k];
			const Side as[2] = {{a.in, a.n, a.g, a.g.in_sample}, {a.out, a.n, a.g, a.g.out_sample}};
			const Side bs[2] = {{b.in, b.n, b.g, b.g.in_sample}, {b.out, b.n, b.g, b.g.out_sample}};
			for (int u = 0; u < 2; u++)
				for (int v = 0; v < 2; v++)
					if (overlap(as[u], bs[v]))
						return set_err(VFGS_B200_ERR_ARG, "the buffers of jobs %d and %d overlap", std::min(sp[x].k, sp[y].k), std::max(sp[x].k, sp[y].k));
		}
	return VFGS_B200_OK;
}

template <typename T>
int grow_host(T*& p, size_t& cap, size_t need)
{
	if (need <= cap) return VFGS_B200_OK;
	if (p) CUDA_TRY(cudaFreeHost(p));
	p = nullptr; cap = 0;
	need = (need + 4095) & ~(size_t)4095;
	CUDA_TRY(cudaHostAlloc((void**)&p, need, cudaHostAllocDefault));
	cap = need;
	return VFGS_B200_OK;
}

size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// The jobs of a call that the MULTI launches serve: one stream-kernel launch for all their block tables, then one grain
// launch per kernel instantiation (group_key).
int run_batched(std::vector<JobPlan>& jp, cudaStream_t st, int& bits)
{
	Context& c = g_ctx;
	size_t tab_bytes = 0;
	int njobs = 0;
	long long nwarps = 0;
	for (JobPlan& j : jp) {
		if (!j.batched) continue;
		j.tab_off = tab_bytes;
		tab_bytes += (align16((size_t)j.n * j.g.R * j.g.spitch * 4) + (size_t)j.n * j.g.R * j.g.spitch * 8 + 255) & ~(size_t)255;
		njobs++;
		nwarps += (long long)j.n * j.g.R;
	}
	if (!njobs) return VFGS_B200_OK;
	const int t = (int)(c.tab_next++ & 1u);
	if (int rc = grow(c.d_tab[t], c.tab_cap[t], tab_bytes)) return rc;
	uint8_t* tab = (uint8_t*)c.d_tab[t];
	std::vector<const LaunchPlan*> plans;
	for (JobPlan& j : jp) {
		if (!j.batched) continue;
		uint16_t* woffs = (uint16_t*)(tab + j.tab_off + align16((size_t)j.n * j.g.R * j.g.spitch * 4));
		for (FgsParams* q : {&j.lp.fast, &j.lp.edge, &j.lp.gather}) { q->states = nullptr; q->woffs = woffs; }
		plans.push_back(&j.lp);
		if (j.lp.any_fast && j.in.semi && j.lp.fast.fwide[1]) bits |= 16; // the interleaved U/V lane runs
	}
	std::vector<LaunchGroup> groups;
	group_launches(plans, groups);
	// descriptors: StreamJob[njobs], then per group FgsParams[m] and long long task0[m + 1]
	size_t bytes = align16(sizeof(StreamJob) * njobs);
	std::vector<size_t> goff(groups.size());
	for (size_t k = 0; k < groups.size(); k++) {
		goff[k] = bytes;
		bytes += align16(sizeof(FgsParams) * groups[k].p.size()) + align16(sizeof(long long) * (groups[k].p.size() + 1));
	}
	if (c.desc_used[t]) CUDA_TRY(cudaEventSynchronize(c.desc_copied[t])); // the staging buffer's previous copy has left it
	if (c.tab_used[t]) CUDA_TRY(cudaStreamWaitEvent(c.s_tab, c.tab_free[t], 0)); // the grain kernels of two calls ago read these buffers
	if (bytes > c.desc_cap[t]) { // the device copy may still be read: wait for the table stream before it is freed
		if (c.d_desc[t]) CUDA_TRY(cudaStreamSynchronize(c.s_tab));
		if (int rc = grow(c.d_desc[t], c.desc_cap[t], bytes)) return rc;
	}
	if (int rc = grow_host(c.h_desc[t], c.hdesc_cap[t], bytes)) return rc; // its last copy is done (desc_copied)
	uint8_t* h = c.h_desc[t];
	uint8_t* d = c.d_desc[t];
	StreamJob* sj = (StreamJob*)h;
	long long w0 = 0;
	int k = 0;
	for (const JobPlan& j : jp) {
		if (!j.batched) continue;
		StreamJob& s = sj[k++];
		s.warp0 = w0; s.epoch = j.epoch; s.R = j.g.R; s.nb = j.g.nb; s.spitch = j.g.spitch;
		s.states = nullptr; s.woffs = (uint16_t*)j.lp.fast.woffs;
		s.wp = make_woff_params(j.lp.fast, j.lp.kind);
		w0 += (long long)j.n * j.g.R;
	}
	for (size_t g = 0; g < groups.size(); g++) {
		FgsParams* fp = (FgsParams*)(h + goff[g]);
		long long* t0 = (long long*)(h + goff[g] + align16(sizeof(FgsParams) * groups[g].p.size()));
		t0[0] = 0;
		for (size_t m = 0; m < groups[g].p.size(); m++) {
			fp[m] = *groups[g].p[m];
			t0[m + 1] = t0[m] + fp[m].total_tasks;
		}
	}
	CUDA_TRY(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, c.s_tab));
	CUDA_TRY(cudaEventRecord(c.desc_copied[t], c.s_tab));
	c.desc_used[t] = true;
	{ // block tables of every job: one launch on the table stream
		const int grid = (int)((nwarps * 32 + kLfsrThreads - 1) / kLfsrThreads);
		lfsr_states_jobs_kernel<<<grid, kLfsrThreads, 0, c.s_tab>>>(c.d_pow2, (const StreamJob*)d, njobs, nwarps);
		CUDA_TRY(cudaGetLastError());
		g_launches++;
	}
	CUDA_TRY(cudaEventRecord(c.tab_ready[t], c.s_tab));
	CUDA_TRY(cudaStreamWaitEvent(st, c.tab_ready[t], 0));
	for (const JobPlan& j : jp) // images of sessions whose upload is not known to be complete
		if (j.batched && !j.s->uploaded) {
			if (cudaEventQuery(j.s->img.uploaded) == cudaSuccess) j.s->uploaded = true;
			else CUDA_TRY(cudaStreamWaitEvent(st, j.s->img.uploaded, 0));
		}
	for (size_t g = 0; g < groups.size(); g++) {
		const LaunchGroup& part = groups[g];
		MultiParams mp;
		memset(&mp, 0, sizeof(mp));
		mp.jobs = (const FgsParams*)(d + goff[g]);
		mp.task0 = (const long long*)(d + goff[g] + align16(sizeof(FgsParams) * part.p.size()));
		mp.njobs = (int)part.p.size();
		long long total = 0;
		for (const FgsParams* q : part.p) total += q->total_tasks;
		const int kind = part.key & 3, smem = part.smem;
		if (total <= 0) continue;
		int threads = 0;
		MultiKernel kern = multi_kernel(part.key, threads);
		if (smem > c.multi_smem_attr[part.key]) {
			CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
			c.multi_smem_attr[part.key] = smem;
		}
		int& per_sm = c.multi_per_sm[part.key]; // resident CTAs per SM, asked once per key and shared-memory size
		if (c.multi_occ_smem[part.key] != smem) {
			CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, (size_t)smem));
			c.multi_occ_smem[part.key] = smem;
		}
		if (per_sm < 1) return set_err(VFGS_B200_ERR_CUDA, "grain kernel does not fit on an SM (smem %d)", smem);
		const int wpc = threads / 32;
		const long long want = (total + wpc - 1) / wpc, cap = (long long)c.sm_count * per_sm;
		const int grid = (int)(want < cap ? want : cap);
		cudaEvent_t e0 = nullptr, e1 = nullptr;
		if (c.timing) {
			if (c.ev_used == c.ev_begin.size()) {
				cudaEvent_t a, b;
				CUDA_TRY(cudaEventCreate(&a));
				CUDA_TRY(cudaEventCreate(&b));
				c.ev_begin.push_back(a); c.ev_end.push_back(b);
			}
			e0 = c.ev_begin[c.ev_used]; e1 = c.ev_end[c.ev_used]; c.ev_used++;
			CUDA_TRY(cudaEventRecord(e0, st));
		}
		kern<<<grid, threads, (size_t)smem, st>>>(mp);
		CUDA_TRY(cudaGetLastError());
		if (c.timing) CUDA_TRY(cudaEventRecord(e1, st));
		g_launches++;
		c.last_launch[0] = grid; c.last_launch[1] = threads; c.last_launch[2] = smem; c.last_launch[3] = c.sm_count;
		bits |= kind == 0 ? 1 : kind == 1 ? 4 : 8;
	}
	CUDA_TRY(cudaEventRecord(c.tab_free[t], st));
	c.tab_used[t] = true;
	// the call's end, which its sessions keep: an event of the pool that no session holds any more, else a new one
	std::shared_ptr<CUevent_st> done;
	for (const std::shared_ptr<CUevent_st>& e : c.call_events)
		if (e.use_count() == 1) { done = e; break; }
	if (!done) {
		cudaEvent_t ev;
		CUDA_TRY(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
		done.reset(ev, [](cudaEvent_t e) { cudaEventDestroy(e); });
		c.call_events.push_back(done);
	}
	CUDA_TRY(cudaEventRecord(done.get(), st));
	for (JobPlan& j : jp)
		if (j.batched) j.s->last_batch = done;
	return VFGS_B200_OK;
}

int run_jobs(const vfgs_b200_job* jobs, int njobs, cudaStream_t st)
{
	if (njobs < 0) return set_err(VFGS_B200_ERR_ARG, "negative job count");
	if (njobs && !jobs) return set_err(VFGS_B200_ERR_ARG, "null job list");
	std::vector<JobPlan> jp((size_t)njobs);
	for (int k = 0; k < njobs; k++) // argument checks first: they need no device
		if (int rc = check_job(jobs[k], k, jp[k])) return rc;
	if (int rc = check_disjoint(jp)) return rc;
	for (JobPlan& j : jp) { // plans; a launch the kernels cannot take is refused before any device work
		if (!j.n) continue;
		uint16_t* w = nullptr;
		FgsParams p;
		plan_frames(session_state(j.s), j.in, j.out, j.n, j.g, j.alias == 1, nullptr, p, j.lp, w);
		// the general kernel and the in-place scratch detour take the single-job route
		const bool scratch = j.alias == 1 && in_place_needs_scratch(j.lp, j.s->bi);
		j.batched = !j.lp.any_general && !scratch;
		if (!scratch) // (the scratch detour cuts a job into sub-batches of 256 MB, far below the limit)
			for (const FgsParams* q : {&j.lp.fast, &j.lp.edge, &j.lp.gather, &j.lp.general})
				if (q->total_tasks >= (1ll << 31))
					return set_err(VFGS_B200_ERR_ARG, "batch too large for one launch (%lld warp-tasks): split the job", q->total_tasks);
	}
	if (!njobs) return VFGS_B200_OK;
	if (int rc = ensure_ctx(-1)) return rc;
	if (int rc = stream_switch(st)) return rc;
	int bits = 0;
	for (JobPlan& j : jp) { // registers advance in list order; single-job-route jobs launch here
		if (!j.n) continue;
		if (j.batched) {
			j.epoch = j.s->hw.line_rnd;
			advance_registers(j.s->hw, j.g, (uint64_t)j.n);
		} else {
			if (int rc = run_job(session_state(j.s), j.in, j.out, j.n, j.g, j.alias, st)) return rc;
			bits |= g_ctx.last_launch[4];
		}
	}
	const int rc = run_batched(jp, st, bits);
	g_ctx.last_launch[4] = bits;
	return rc;
}

int create_session(vfgs_b200_session** out)
{
	if (!out) return set_err(VFGS_B200_ERR_ARG, "null session pointer");
	*out = nullptr;
	const HwState& h = hw();
	// the geometry-independent conditions of make_geometry
	if (h.scale_shift + h.bs < 8 || h.scale_shift + h.bs > 13)
		return set_err(VFGS_B200_ERR_STATE, "scale_shift %d + bs %d outside 8..13 (vfgs_hw.c:170)", h.scale_shift, h.bs);
	for (int c = 0; c < 3; c++)
		for (int i = 0; i < 256; i++)
			if ((h.plut[c][i] >> 4) >= kSlots)
				return set_err(VFGS_B200_ERR_STATE, "pattern LUT %d entry %d selects slot %d: the hardware has slots 0..8 (vfgs_hw.c:49,218)", c, i, h.plut[c][i] >> 4);
	if (int rc = ensure_ctx(-1)) return rc;
	Context& c = g_ctx;
	std::unique_ptr<vfgs_b200_session> s(new vfgs_b200_session());
	s->hw = h;
	std::vector<uint8_t> blob, fblob;
	build_tables(s->hw, s->bi, blob, fblob);
	if (s->bi.bytes > c.max_smem_optin - 1024)
		return set_err(VFGS_B200_ERR_STATE, "table image of %d bytes exceeds shared memory", s->bi.bytes);
	ImageSet& m = s->img;
	auto fail = [&](int rc) {
		if (m.d_blob) cudaFree(m.d_blob);
		if (m.d_fblob) cudaFree(m.d_fblob);
		if (m.h_stage) cudaFreeHost(m.h_stage);
		if (m.uploaded) cudaEventDestroy(m.uploaded);
		if (m.last_use) cudaEventDestroy(m.last_use);
		return rc;
	};
	const size_t gb = (size_t)s->bi.gbytes, fb = (size_t)s->bi.fbytes;
#define SESSION_TRY(expr) do { cudaError_t e_ = (expr); if (e_ != cudaSuccess) return fail(set_err(VFGS_B200_ERR_CUDA, "%s -> %s", #expr, cudaGetErrorString(e_))); } while (0)
	SESSION_TRY(cudaMalloc((void**)&m.d_blob, gb));
	SESSION_TRY(cudaMalloc((void**)&m.d_fblob, fb));
	SESSION_TRY(cudaHostAlloc((void**)&m.h_stage, gb + fb, cudaHostAllocDefault));
	SESSION_TRY(cudaEventCreateWithFlags(&m.uploaded, cudaEventDisableTiming));
	SESSION_TRY(cudaEventCreateWithFlags(&m.last_use, cudaEventDisableTiming));
	memcpy(m.h_stage, blob.data(), gb);
	memcpy(m.h_stage + gb, fblob.data(), fb);
	SESSION_TRY(cudaMemcpyAsync(m.d_blob, m.h_stage, gb, cudaMemcpyHostToDevice, c.s_tab));
	SESSION_TRY(cudaMemcpyAsync(m.d_fblob, m.h_stage + gb, fb, cudaMemcpyHostToDevice, c.s_tab));
	SESSION_TRY(cudaEventRecord(m.uploaded, c.s_tab));
	if (s->bi.bytes > c.smem_attr) { // the general kernel of the single-job route
		SESSION_TRY(cudaFuncSetAttribute(fgs_apply_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, s->bi.bytes));
		c.smem_attr = s->bi.bytes;
	}
#undef SESSION_TRY
	*out = s.release();
	return VFGS_B200_OK;
}

} // namespace

// ====================================================================================== vfgs_hw.h
extern "C" {

void vfgs_set_luma_pattern(int index, int8_t* P) // vfgs_hw.c:314-318
{
	pipe_before_state_change();
	REQUIRE(index >= 0 && index < VFGS_MAX_PATTERNS);
	memcpy(hw().pattern[0][index], P, 64 * 64);
	g_dirty = true;
}

void vfgs_set_chroma_pattern(int index, int8_t* P) // vfgs_hw.c:320-325
{
	pipe_before_state_change();
	REQUIRE(index >= 0 && index < VFGS_MAX_PATTERNS);
	HwState& h = hw();
	const int rows = 64 / h.csuby, src_stride = 64 / h.csuby, ncopy = 64 / h.csubx;
	for (int r = 0; r < rows; r++) memcpy(h.pattern[1][index][r], P + (size_t)src_stride * r, (size_t)ncopy);
	g_dirty = true;
}

void vfgs_set_scale_lut(int c, uint8_t lut[]) // vfgs_hw.c:327-331
{
	pipe_before_state_change();
	REQUIRE(c >= 0 && c < 3);
	memcpy(hw().slut[c], lut, 256);
	g_dirty = true;
}

void vfgs_set_pattern_lut(int c, uint8_t lut[]) // vfgs_hw.c:333-337
{
	pipe_before_state_change();
	REQUIRE(c >= 0 && c < 3);
	// Any table is accepted, like the reference does (vfgs_hw.c:333-337). lut[i] >> 4 indexes pattern[..][9] in
	// vfgs_hw.c:218: an entry above slot 8 makes the reference read out of bounds if a sample ever hits it; here
	// such a table is refused when grain is requested (make_geometry: VFGS_B200_ERR_STATE), not in the setter.
	memcpy(hw().plut[c], lut, 256);
	g_dirty = true;
}

void vfgs_set_seed(uint32_t seed) // vfgs_hw.c:339-344
{
	pipe_before_state_change();
	HwState& h = hw();
	h.rnd = h.rnd_up = h.line_rnd = h.line_rnd_up = seed << 1;
}

void vfgs_set_scale_shift(int shift) // vfgs_hw.c:346-350
{
	pipe_before_state_change();
	REQUIRE(shift >= 2 && shift < 8);
	HwState& h = hw();
	h.scale_shift = shift + 6 - h.bs;
}

void vfgs_set_depth(int depth) // vfgs_hw.c:352-362
{
	pipe_before_state_change();
	REQUIRE(depth == 8 || depth == 10);
	HwState& h = hw();
	const int nbs = depth - 8;
	h.scale_shift = (h.scale_shift + h.bs - nbs) & 0xff;
	if (h.bs != nbs) g_dirty = true;
	h.bs = nbs;
}

void vfgs_set_legal_range(int legal) // vfgs_hw.c:364-380
{
	pipe_before_state_change();
	HwState& h = hw();
	h.y_min = h.c_min = legal ? 16 : 0;
	h.y_max = legal ? 235 : 255;
	h.c_max = legal ? 240 : 255;
}

void vfgs_set_chroma_subsampling(int subx, int suby) // vfgs_hw.c:382-388
{
	pipe_before_state_change();
	REQUIRE(subx == 1 || subx == 2);
	REQUIRE(suby == 1 || suby == 2);
	HwState& h = hw();
	if (h.csubx != subx || h.csuby != suby) g_dirty = true;
	h.csubx = subx; h.csuby = suby;
}

// vfgs_hw.c:288-312. Host line buffers, in place, synchronous. The register bookkeeping is the
// reference's; the samples go through the same kernels as the frame entry points.
void vfgs_add_grain_line(void* Y, void* U, void* V, int y, int width)
{
	if (pipe_line(Y, y)) return; // a slot of the frame pipeline (include/yuv.h): the whole frame is processed at flush time
	HwState& h = hw();
	Geometry g;
	if (make_geometry(g, width, 16 * ((y >> 4) + 1), 0)) fatal("vfgs_add_grain_line");
	if (prepare(-1)) fatal("vfgs_add_grain_line");
	Context& c = g_ctx;
	const JumpTable& jt = jump_table();

	if (y && (y & 15) == 0) { h.line_rnd_up = h.line_rnd; h.line_rnd = h.rnd; }

	// two rows of per-block registers (upper, current) stepped on the host: nb steps, trivial
	std::vector<uint32_t> rows((size_t)2 * g.spitch, 0);
	uint32_t su = h.line_rnd_up, sc = h.line_rnd;
	for (int b = 0; b < g.nb; b++) {
		rows[1 + b] = su; rows[(size_t)g.spitch + 1 + b] = sc;
		su = lfsr_step(su); sc = lfsr_step(sc);
	}
	const bool chroma = !((y & 1) && h.csuby > 1); // vfgs_hw.c:164-165
	const size_t lbytes = (size_t)width * g.in_sample, cbytes = (size_t)g.cw * g.in_sample;
	const size_t lpad = (lbytes + 255) & ~(size_t)255, cpad = (cbytes + 255) & ~(size_t)255;
	auto chk = [](cudaError_t e, const char* what) {
		if (e != cudaSuccess) { snprintf(g_err, sizeof(g_err), "%s -> %s", what, cudaGetErrorString(e)); fatal("vfgs_add_grain_line"); }
	};
	// the line is staged OUT OF PLACE (input region, then output region): with sample-adaptive pattern selection the
	// general kernel reads the neighbouring block's input sample, which another warp may already have overwritten
	const size_t region = lpad + 2 * cpad;
	if (grow(c.d_line, c.line_cap, 2 * region)) fatal("vfgs_add_grain_line");
	if (grow(c.d_streams, c.streams_cap, rows.size() * sizeof(uint32_t))) fatal("vfgs_add_grain_line");
	cudaStream_t st = c.s_k;
	if (c.used_stream && c.last_stream != st) chk(cudaStreamSynchronize(c.last_stream), "sync");
	c.last_stream = st; c.used_stream = true;
	chk(cudaMemcpyAsync(c.d_streams, rows.data(), rows.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st), "streams H2D");
	chk(cudaMemcpyAsync(c.d_line, Y, lbytes, cudaMemcpyHostToDevice, st), "Y H2D");
	if (chroma) {
		chk(cudaMemcpyAsync(c.d_line + lpad, U, cbytes, cudaMemcpyHostToDevice, st), "U H2D");
		chk(cudaMemcpyAsync(c.d_line + lpad + cpad, V, cbytes, cudaMemcpyHostToDevice, st), "V H2D");
	}
	FgsParams p;
	fill_common(p, g, global_state());
	p.nframes = 1;
	p.y_begin = y; p.y_end = y + 1;
	p.row_begin = y >> 4; p.rows = 1;
	uint8_t* base[3] = {c.d_line, c.d_line + lpad, c.d_line + lpad + cpad};
	for (int k = 0; k < 3; k++) {
		p.comp[k].in = base[k]; p.comp[k].out = base[k] + region;
		p.comp[k].in_row_bytes = p.comp[k].out_row_bytes = 0; // every line index maps to the staged line
		p.comp[k].width = k ? g.cw : width;
		p.comp[k].lines = (k && !chroma) ? 0 : 0x7fffffff;
	}
	p.states = c.d_streams; p.stream_rows = 2; p.stream_row0 = (y >> 4) - 1;
	finish_tasks(p);
	if (images_before(global_state(), st) || launch_apply(p, st) || images_after(global_state(), st)) fatal("vfgs_add_grain_line");
	chk(cudaMemcpyAsync(Y, c.d_line + region, lbytes, cudaMemcpyDeviceToHost, st), "Y D2H");
	if (chroma) {
		chk(cudaMemcpyAsync(U, c.d_line + region + lpad, cbytes, cudaMemcpyDeviceToHost, st), "U D2H");
		chk(cudaMemcpyAsync(V, c.d_line + region + lpad + cpad, cbytes, cudaMemcpyDeviceToHost, st), "V D2H");
	}
	chk(cudaStreamSynchronize(st), "line sync");

	h.rnd = jt.jump(h.line_rnd, (uint64_t)g.nb);
	h.rnd_up = jt.jump(h.line_rnd_up, (uint64_t)g.nb);
}

// ====================================================================================== vfgs_b200.h
int vfgs_b200_init(int device) { return ensure_ctx(device); }

int vfgs_b200_reset(void)
{
	g_hw.power_on();
	g_hw_init = true;
	g_dirty = true;
	return VFGS_B200_OK;
}

const char* vfgs_b200_last_error(void) { return g_err; }

size_t vfgs_b200_frame_bytes(int width, int height, int depth)
{
	const HwState& h = hw();
	const size_t s = depth > 8 ? 2 : 1;
	return ((size_t)width * height + 2 * (size_t)(width / h.csubx) * (height / h.csuby)) * s;
}

int vfgs_b200_add_grain_planes_device(const vfgs_b200_planes* in, const vfgs_b200_planes* out, int nframes,
                                      int width, int height, int out_depth, void* stream)
{
	if (!in || !out || nframes < 0) return set_err(VFGS_B200_ERR_ARG, "null planes or negative frame count");
	Geometry g;
	if (int rc = make_geometry(g, width, height, out_depth)) return rc;
	return run_call(frame_planes(*in), frame_planes(*out), nframes, g, (cudaStream_t)stream);
}

int vfgs_b200_add_grain_semiplanar_device(const vfgs_b200_semiplanar* in, const vfgs_b200_semiplanar* out, int nframes,
                                          int width, int height, void* stream)
{
	if (!in || !out || nframes < 0) return set_err(VFGS_B200_ERR_ARG, "null planes or negative frame count");
	Geometry g;
	if (int rc = semiplanar_geometry(g, hw(), *in, *out, width, height)) return rc;
	return run_call(frame_planes(*in), frame_planes(*out), nframes, g, (cudaStream_t)stream);
}

int vfgs_b200_add_grain_frames_device(const void* in, void* out, int nframes, int width, int height,
                                      int out_depth, void* stream)
{
	if (!in || !out) return set_err(VFGS_B200_ERR_ARG, "null buffer");
	Geometry g;
	if (int rc = make_geometry(g, width, height, out_depth)) return rc;
	vfgs_b200_planes pi, po;
	packed_planes(pi, in, g, g.in_sample, g.in_frame_bytes);
	packed_planes(po, out, g, g.out_sample, g.out_frame_bytes);
	return vfgs_b200_add_grain_planes_device(&pi, &po, nframes, width, height, out_depth, stream);
}

int vfgs_b200_add_grain_frames_host(const void* in, void* out, int nframes, int width, int height, int out_depth)
{
	if (!in || !out || nframes < 0) return set_err(VFGS_B200_ERR_ARG, "null buffer or negative frame count");
	Geometry g;
	if (int rc = make_geometry(g, width, height, out_depth)) return rc;
	if (int rc = prepare(-1)) return rc;
	if (nframes == 0) return VFGS_B200_OK;
	if (in == out && g.in_depth != g.out_depth) return set_err(VFGS_B200_ERR_ARG, "in-place needs equal depths");
	Context& c = g_ctx;
	if (c.used_stream) { CUDA_TRY(cudaStreamSynchronize(c.last_stream)); c.used_stream = false; }

	// chunk = as many frames as fit ~64 MB of input (measured ahead of 16 and 32 MB chunks, scripts/e2e_sweep.sh); the ring has kPipeSlots chunks in flight
	size_t chunk_bytes = 64u << 20;
	int nslots = 3;
	if (const char* e = getenv("VFGS_B200_CHUNK_MB")) { long v = atol(e); if (v > 0 && v <= 4096) chunk_bytes = (size_t)v << 20; }
	if (const char* e = getenv("VFGS_B200_SLOTS")) { int v = atoi(e); if (v >= 2 && v <= kPipeSlots) nslots = v; }
	int per = (int)(chunk_bytes / g.in_frame_bytes);
	if (per < 1) per = 1;
	if (per > nframes) per = nframes;
	const uint32_t epoch = hw().line_rnd;
	const uint8_t* hin = (const uint8_t*)in;
	uint8_t* hout = (uint8_t*)out;
	int idx = 0;
	for (int f0 = 0; f0 < nframes; f0 += per, idx++) {
		const int n = (nframes - f0 < per) ? nframes - f0 : per;
		Slot& s = c.slot[idx % nslots];
		if (int rc = grow(s.d_in, s.in_cap, (size_t)per * g.in_frame_bytes)) return rc;
		if (int rc = grow(s.d_out, s.out_cap, (size_t)per * g.out_frame_bytes)) return rc;
		if (int rc = grow(s.d_streams, s.streams_cap, (size_t)per * g.R * g.spitch * kBlockTableBytes + 16)) return rc;
		// the slot's previous chunk must have left the device before its buffers are overwritten
		if (idx >= nslots) {
			CUDA_TRY(cudaStreamWaitEvent(c.s_h2d, s.k_done, 0));   // d_in free once its kernel is done
			CUDA_TRY(cudaStreamWaitEvent(c.s_k, s.d2h_done, 0));   // d_out free once copied back
		}
		CUDA_TRY(cudaMemcpyAsync(s.d_in, hin + (size_t)f0 * g.in_frame_bytes, (size_t)n * g.in_frame_bytes, cudaMemcpyHostToDevice, c.s_h2d));
		CUDA_TRY(cudaEventRecord(s.h2d_done, c.s_h2d));
		CUDA_TRY(cudaStreamWaitEvent(c.s_k, s.h2d_done, 0));
		vfgs_b200_planes pi, po;
		packed_planes(pi, s.d_in, g, g.in_sample, g.in_frame_bytes);
		packed_planes(po, s.d_out, g, g.out_sample, g.out_frame_bytes);
		if (int rc = run_frames_device(global_state(), frame_planes(pi), frame_planes(po), n, g, false, epoch, (uint64_t)f0, s.d_streams, c.s_k)) return rc;
		CUDA_TRY(cudaEventRecord(s.k_done, c.s_k));
		CUDA_TRY(cudaStreamWaitEvent(c.s_d2h, s.k_done, 0));
		CUDA_TRY(cudaMemcpyAsync(hout + (size_t)f0 * g.out_frame_bytes, s.d_out, (size_t)n * g.out_frame_bytes, cudaMemcpyDeviceToHost, c.s_d2h));
		CUDA_TRY(cudaEventRecord(s.d2h_done, c.s_d2h));
	}
	CUDA_TRY(cudaStreamSynchronize(c.s_d2h));
	CUDA_TRY(cudaStreamSynchronize(c.s_k));
	CUDA_TRY(cudaStreamSynchronize(c.s_h2d));
	advance_registers(hw(), g, (uint64_t)nframes);
	return VFGS_B200_OK;
}

int vfgs_b200_skip_frames(int64_t nframes, int width, int height)
{
	if (nframes < 0) return set_err(VFGS_B200_ERR_ARG, "negative frame count");
	Geometry g;
	if (int rc = make_geometry(g, width, height, 0)) return rc;
	advance_registers(hw(), g, (uint64_t)nframes);
	return VFGS_B200_OK;
}

void vfgs_b200_get_lfsr(uint32_t regs[4])
{
	const HwState& h = hw();
	regs[0] = h.rnd; regs[1] = h.rnd_up; regs[2] = h.line_rnd; regs[3] = h.line_rnd_up;
}

void vfgs_b200_set_lfsr(const uint32_t regs[4])
{
	HwState& h = hw();
	h.rnd = regs[0]; h.rnd_up = regs[1]; h.line_rnd = regs[2]; h.line_rnd_up = regs[3];
}

// Mirror of the hardware state in the layout of the reference's statics (see oracle/ref_harness.c
// refh_state): pattern[2][9][64][64], sLUT[3][256], pLUT[3][256], 4 LFSR registers, then
// scale_shift, bs, Y_min, Y_max, C_min, C_max, csubx, csuby as ints.
size_t vfgs_b200_get_state(void* dst, size_t cap) { return state_dump(hw(), dst, cap); }

void* vfgs_b200_host_alloc(size_t bytes)
{
	if (ensure_ctx(-1)) return nullptr;
	void* p = nullptr;
	if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) {
		set_err(VFGS_B200_ERR_CUDA, "cudaHostAlloc(%zu) failed", bytes);
		return nullptr;
	}
	return p;
}

void vfgs_b200_host_free(void* p)
{
	if (p) cudaFreeHost(p);
}

uint64_t vfgs_b200_launch_count(void) { return g_launches; }

void vfgs_b200_force_general_kernel(int mode) { g_kernel_mode = mode; }

int vfgs_b200_kernel_timing(int enable)
{
	if (int rc = ensure_ctx(-1)) return rc;
	Context& c = g_ctx;
	c.timing = enable != 0;
	c.ev_used = 0; c.timed_ms = 0.0; c.timed_launches = 0;
	return VFGS_B200_OK;
}

int vfgs_b200_kernel_time(double* total_ms, uint64_t* launches)
{
	Context& c = g_ctx;
	if (!c.ready) return set_err(VFGS_B200_ERR_ARG, "no device bound");
	for (size_t i = 0; i < c.ev_used; i++) {
		CUDA_TRY(cudaEventSynchronize(c.ev_end[i]));
		float ms = 0.f;
		CUDA_TRY(cudaEventElapsedTime(&ms, c.ev_begin[i], c.ev_end[i]));
		c.timed_ms += ms; c.timed_launches++;
	}
	c.ev_used = 0;
	if (total_ms) *total_ms = c.timed_ms;
	if (launches) *launches = c.timed_launches;
	return VFGS_B200_OK;
}

void vfgs_b200_last_launch(int out[5])
{
	for (int i = 0; i < 5; i++) out[i] = g_ctx.last_launch[i];
}

int vfgs_b200_session_create(vfgs_b200_session** out) { return create_session(out); }

void vfgs_b200_session_destroy(vfgs_b200_session* s)
{
	if (!s) return;
	if (s->img.in_use) cudaEventSynchronize(s->img.last_use);
	if (s->last_batch) cudaEventSynchronize(s->last_batch.get());
	cudaFree(s->img.d_blob);
	cudaFree(s->img.d_fblob);
	cudaFreeHost(s->img.h_stage);
	cudaEventDestroy(s->img.uploaded);
	cudaEventDestroy(s->img.last_use);
	delete s;
}

void vfgs_b200_session_get_lfsr(const vfgs_b200_session* s, uint32_t regs[4])
{
	const HwState& h = s->hw;
	regs[0] = h.rnd; regs[1] = h.rnd_up; regs[2] = h.line_rnd; regs[3] = h.line_rnd_up;
}

void vfgs_b200_session_set_lfsr(vfgs_b200_session* s, const uint32_t regs[4])
{
	HwState& h = s->hw;
	h.rnd = regs[0]; h.rnd_up = regs[1]; h.line_rnd = regs[2]; h.line_rnd_up = regs[3];
}

int vfgs_b200_session_skip_frames(vfgs_b200_session* s, int64_t nframes, int width, int height)
{
	if (!s) return set_err(VFGS_B200_ERR_ARG, "null session");
	if (nframes < 0) return set_err(VFGS_B200_ERR_ARG, "negative frame count");
	Geometry g;
	if (int rc = make_geometry(g, s->hw, width, height, 0)) return rc;
	advance_registers(s->hw, g, (uint64_t)nframes);
	return VFGS_B200_OK;
}

size_t vfgs_b200_session_get_state(const vfgs_b200_session* s, void* dst, size_t cap) { return state_dump(s->hw, dst, cap); }

int vfgs_b200_add_grain_jobs_device(const vfgs_b200_job* jobs, int njobs, void* stream) { return run_jobs(jobs, njobs, (cudaStream_t)stream); }

} // extern "C"

// ====================================================================================== vfgs_fw.h
namespace {

int ensure_fw()
{
	Context& c = g_ctx;
	if (c.d_fw_tables) return VFGS_B200_OK;
	static FwTables tables;
	make_fw_tables(tables);
	CUDA_TRY(cudaMalloc((void**)&c.d_fw_tables, sizeof(FwTables)));
	CUDA_TRY(cudaMemcpy(c.d_fw_tables, &tables, sizeof(FwTables), cudaMemcpyHostToDevice));
	CUDA_TRY(cudaMalloc((void**)&c.d_fw_scratch, sizeof(FwScratch)));
	CUDA_TRY(cudaMemset(c.d_fw_scratch, 0, sizeof(FwScratch)));
	CUDA_TRY(cudaMalloc((void**)&c.d_fw_pattern, 2 * kSlots * 4096));
	CUDA_TRY(cudaMemset(c.d_fw_pattern, 0, 2 * kSlots * 4096));
	CUDA_TRY(cudaHostAlloc((void**)&c.h_fw_stage, 2 * kFwMaxPatterns * 4096, cudaHostAllocDefault));
	return VFGS_B200_OK;
}

// Pattern jobs on the table stream, results into the host mirror through the setters' copy rules, then LUTs and
// scalars through the setters themselves. The host waits for the job kernels only (tens of microseconds each; the
// auto-regressive filter is serial: ~0.2 ms): grain kernels queued on other streams keep running.
int fw_apply(FwPlan& plan)
{
	if (plan.error) return set_err(VFGS_B200_ERR_STATE, "%s", plan.error);
	if ((int)plan.jobs.size() > 2 * kFwMaxPatterns) return set_err(VFGS_B200_ERR_STATE, "too many patterns");
	pipe_before_state_change();
	if (int rc = ensure_ctx(-1)) return rc;
	if (int rc = ensure_fw()) return rc;
	Context& c = g_ctx;
	HwState& h = hw();
	for (size_t i = 0; i < plan.jobs.size(); i++) {
		const FwJob& j = plan.jobs[i];
		fw_pattern_kernel<<<1, kFwThreads, 0, c.s_tab>>>(j, c.d_fw_tables, c.d_fw_scratch, c.d_fw_pattern);
		CUDA_TRY(cudaGetLastError());
		g_launches++;
		CUDA_TRY(cudaMemcpyAsync(c.h_fw_stage + i * 4096, c.d_fw_pattern + ((size_t)j.bank * kSlots + j.slot) * 4096, 4096,
		                         cudaMemcpyDeviceToHost, c.s_tab));
	}
	CUDA_TRY(cudaStreamSynchronize(c.s_tab));
	for (size_t i = 0; i < plan.jobs.size(); i++) {
		const FwJob& j = plan.jobs[i];
		const int8_t* src = c.h_fw_stage + i * 4096;
		if (j.bank == 0) memcpy(h.pattern[0][j.slot], src, 4096);                 // vfgs_set_luma_pattern
		else                                                                     // vfgs_set_chroma_pattern: only the rows and columns it writes
			for (int r = 0; r < 64 / h.csuby; r++) memcpy(h.pattern[1][j.slot][r], src + 64 * r, (size_t)(64 / h.csubx));
	}
	g_dirty = true;
	if (plan.set_seed) vfgs_set_seed(plan.seed);
	for (int cc = 0; cc < 3; cc++) {
		vfgs_set_scale_lut(cc, plan.slut[cc]);
		vfgs_set_pattern_lut(cc, plan.plut[cc]);
	}
	if (plan.scale_shift < 2 || plan.scale_shift >= 8)
		return set_err(VFGS_B200_ERR_STATE, "scale shift %d outside 2..7 (the reference asserts, vfgs_hw.c:348)", plan.scale_shift);
	vfgs_set_scale_shift(plan.scale_shift);
	if (plan.set_legal) vfgs_set_legal_range(plan.legal);
	return VFGS_B200_OK;
}

} // namespace

extern "C" {

int vfgs_b200_init_sei(const fgs_sei* cfg) // vfgs_fw.c:517-644
{
	if (!cfg) return set_err(VFGS_B200_ERR_ARG, "null metadata");
	FwPlan plan;
	fw_plan_sei(*cfg, hw().csubx, hw().csuby, plan);
	return fw_apply(plan);
}

int vfgs_b200_init_afgs1(const fgs_afgs1* cfg) // vfgs_fw.c:663-708
{
	if (!cfg) return set_err(VFGS_B200_ERR_ARG, "null metadata");
	FwPlan plan;
	fw_plan_afgs1(*cfg, hw().csubx, hw().csuby, plan);
	return fw_apply(plan);
}

} // extern "C"

#include "yuv_pipeline.h"
