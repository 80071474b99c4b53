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
		uint32_t pads[8] = {0, 0, 0, 0, 0, 0, 0, 0};
		CUDA_TRY(cudaMemcpy(pads, d_probe, sizeof(pads), cudaMemcpyDeviceToHost));
		for (int i = 1; i < 8; i++)
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

// Grain kernels about to be launched on `stream` read the current image set: they wait for its upload, and the set
// remembers the last stream position that reads it.
int images_before(cudaStream_t stream)
{
	ImageSet& m = g_ctx.img[g_ctx.img_cur];
	CUDA_TRY(cudaStreamWaitEvent(stream, m.uploaded, 0));
	return VFGS_B200_OK;
}
int images_after(cudaStream_t stream)
{
	ImageSet& m = g_ctx.img[g_ctx.img_cur];
	CUDA_TRY(cudaEventRecord(m.last_use, stream));
	m.in_use = true;
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

int make_geometry(Geometry& g, int width, int height, int out_depth)
{
	const HwState& h = hw();
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

void fill_common(FgsParams& p, const Geometry& g)
{
	memset(&p, 0, sizeof(p));
	fill_state_params(p, hw(), g_bi);
	p.nb = g.nb; p.R = g.R;
	p.in_bytes = (int)g.in_sample; p.out_bytes = (int)g.out_sample;
	p.blob = g_ctx.img_cur >= 0 ? g_ctx.img[g_ctx.img_cur].d_blob : nullptr;
	p.fblob = g_ctx.img_cur >= 0 ? g_ctx.img[g_ctx.img_cur].d_fblob : nullptr;
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
void advance_registers(const Geometry& g, uint64_t nframes)
{
	if (!nframes) return;
	HwState& h = hw();
	const JumpTable& jt = jump_table();
	const uint32_t s0 = h.line_rnd;
	const uint64_t adv = nframes * (uint64_t)(g.R - 1) * (uint64_t)g.nb;
	if (g.R >= 2) {
		h.line_rnd_up = jt.jump(s0, adv - (uint64_t)g.nb);
		h.line_rnd = jt.jump(s0, adv);
	}
	h.rnd = jt.jump(h.line_rnd, (uint64_t)g.nb);
	h.rnd_up = jt.jump(h.line_rnd_up, (uint64_t)g.nb);
}

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
void plan_frames(const FramePlanes& in, const FramePlanes& out, int n, const Geometry& g, bool in_place,
                 uint32_t* d_streams, FgsParams& p, LaunchPlan& lp, uint16_t*& d_woffs)
{
	fill_common(p, g);
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
	plan_launches(p, g_bi, g_kernel_mode, in_place, g_ctx.max_smem_optin - 1024, g_ctx.fast_pad, lp);
}

// Streams + grain kernels for `n` frames whose epoch-relative index starts at frame0.
int run_frames_device(const FramePlanes& in, const FramePlanes& out, int n, const Geometry& g, bool in_place,
                      uint32_t epoch, uint64_t frame0, uint32_t* d_streams, cudaStream_t stream,
                      cudaStream_t table_stream = nullptr, cudaEvent_t table_ready = nullptr)
{
	FgsParams p;
	LaunchPlan lp;
	uint16_t* d_woffs = nullptr;
	plan_frames(in, out, n, g, in_place, d_streams, p, lp, d_woffs);
	g_ctx.last_launch[4] = 0;
	// the register table feeds the general kernel, the window-offset table the fast and gather kernels
	if (int rc = launch_streams(epoch, lp.any_general ? d_streams : nullptr, (lp.any_fast || lp.any_gather || lp.any_edge) ? d_woffs : nullptr,
	                            make_woff_params(p, lp.kind), n, g, frame0, table_stream ? table_stream : stream)) return rc;
	if (table_stream) { // the tables were computed beside the caller's stream: the grain kernels wait for them
		CUDA_TRY(cudaEventRecord(table_ready, table_stream));
		CUDA_TRY(cudaStreamWaitEvent(stream, table_ready, 0));
	}
	if (int rc = images_before(stream)) return rc;
	if (lp.any_fast)
		if (int rc = launch_apply(lp.fast, stream, kFast)) return rc;
	if (lp.any_edge)
		if (int rc = launch_apply(lp.edge, stream, kFastEdge)) return rc;
	if (lp.any_gather)
		if (int rc = launch_apply(lp.gather, stream, kGather, lp.gather_smem, lp.gather_fold, lp.gather_shift)) return rc;
	if (lp.any_general)
		if (int rc = launch_apply(lp.general, stream, kGeneral)) return rc;
	if (lp.any_fast && in.semi && lp.fast.fwide[1]) g_ctx.last_launch[4] |= 16; // the interleaved U/V lane ran
	return images_after(stream);
}

// How the output planes lie relative to the input planes: 0 disjoint, 1 in place (every overlapping plane pair is
// the same plane with the same strides and row bytes), -1 anything else (partial overlap: not supported).
// Planes of consecutive frames interleave in memory (Y0 U0 V0 Y1 ...), so plane pairs are compared frame by frame in
// closed form: with a common frame stride S, frame f1 of one plane meets frame f2 of the other iff their byte
// extents overlap for some k = f1 - f2 within the batch. A semi-planar side has two planes (Y, interleaved UV).
int aliasing(const FramePlanes& in, const FramePlanes& out, int n, const Geometry& g)
{
	auto extent = [&](const FramePlanes& pl, int c, size_t sample) { // bytes one frame's plane spans
		const int64_t lines = plane_lines(pl, c, g), row = plane_row_bytes(pl, c, g, sample);
		if (lines < 1 || row < 1) return (int64_t)0;
		return (lines - 1) * pl.stride[c] + row;
	};
	// bounding ranges of the two calls' buffers
	const uint8_t *ilo = nullptr, *ihi = nullptr, *olo = nullptr, *ohi = nullptr;
	for (int c = 0; c < 3; c++) {
		const int64_t ei = extent(in, c, g.in_sample), eo = extent(out, c, g.out_sample);
		if (ei > 0) {
			const uint8_t* e = in.plane[c] + (int64_t)(n - 1) * in.frame_stride + ei;
			if (!ilo || in.plane[c] < ilo) ilo = in.plane[c];
			if (!ihi || e > ihi) ihi = e;
		}
		if (eo > 0) {
			const uint8_t* e = out.plane[c] + (int64_t)(n - 1) * out.frame_stride + eo;
			if (!olo || out.plane[c] < olo) olo = out.plane[c];
			if (!ohi || e > ohi) ohi = e;
		}
	}
	if (!ilo || !olo || ihi <= olo || ohi <= ilo) return 0;
	if (n > 1 && in.frame_stride != out.frame_stride) return -1; // overlapping buffers walked with different strides
	const int64_t S = in.frame_stride;
	int result = 0;
	for (int i = 0; i < 3; i++)
		for (int j = 0; j < 3; j++) {
			const int64_t ei = extent(in, i, g.in_sample), ej = extent(out, j, g.out_sample);
			if (ei <= 0 || ej <= 0) continue;
			const bool same = i == j && in.plane[i] == out.plane[j] && in.stride[i] == out.stride[j] &&
			                  plane_row_bytes(in, i, g, g.in_sample) == plane_row_bytes(out, j, g, g.out_sample) && in.msb == out.msb;
			bool hit;
			if (n > 1 && S > 0) {
				// frame f1 of the input plane against frame f2 of the output plane: [f1 S, f1 S + ei) meets [D + f2 S, D + f2 S + ej)
				// iff D - ei < k S < D + ej for k = f1 - f2, |k| <= n - 1
				const int64_t D = (int64_t)(out.plane[j] - in.plane[i]);
				auto floor_div = [](int64_t a, int64_t b) { int64_t q = a / b; return (a % b != 0 && ((a < 0) != (b < 0))) ? q - 1 : q; };
				int64_t k_lo = floor_div(D - ei, S) + 1, k_hi = -floor_div(-(D + ej), S) - 1;
				if (k_lo < -(int64_t)(n - 1)) k_lo = -(int64_t)(n - 1);
				if (k_hi > (int64_t)(n - 1)) k_hi = (int64_t)(n - 1);
				hit = k_lo <= k_hi;
			} else {
				hit = !(in.plane[i] + ei <= out.plane[j] || out.plane[j] + ej <= in.plane[i]);
			}
			if (!hit) continue;
			if (!same) return -1;
			result = 1;
		}
	return result;
}

void packed_planes(vfgs_b200_planes& pl, const void* base, const Geometry& g, size_t sample, size_t frame_bytes)
{
	uint8_t* b = (uint8_t*)base;
	pl.y = b; pl.u = b + g.ysam * sample; pl.v = b + (g.ysam + g.csam) * sample;
	pl.stride_y = (int64_t)(g.width * sample); pl.stride_c = (int64_t)(g.cw * sample);
	pl.frame_stride = (int64_t)frame_bytes;
}

int prepare(int device)
{
	if (int rc = ensure_ctx(device)) return rc;
	return upload_blob();
}

// Body of the device frame entry points, after their own argument checks: overlap check (before any device work),
// then the grain launches, through a scratch output buffer where in place would not be safe.
int run_call(const FramePlanes& in, const FramePlanes& out, int nframes, const Geometry& g, cudaStream_t st)
{
	const int alias = nframes ? aliasing(in, out, nframes, g) : 0; // argument check first: needs no device
	if (alias < 0)
		return set_err(VFGS_B200_ERR_ARG, g.in_depth != g.out_depth ? "in-place needs equal depths"
		               : "input and output planes overlap without being identical (same planes, strides and depth)");
	if (int rc = prepare(-1)) return rc;
	if (nframes == 0) return VFGS_B200_OK;
	const bool in_place = alias == 1;
	Context& c = g_ctx;
	if (c.used_stream && c.last_stream != st) CUDA_TRY(cudaStreamSynchronize(c.last_stream)); // d_streams is shared
	c.last_stream = st; c.used_stream = true;
	bool scratch = false;
	if (in_place) { // cheap host-side planning pass: which kernels would serve the components
		FgsParams pp; LaunchPlan lpp; uint16_t* w = nullptr;
		plan_frames(in, out, nframes, g, true, nullptr, pp, lpp, w);
		scratch = in_place_needs_scratch(lpp, g_bi);
	}
	if (scratch) {
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
		const uint32_t epoch = hw().line_rnd;
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
			if (int rc = run_frames_device(pi, po, n, g, false, epoch, (uint64_t)f0, c.d_streams, st)) return rc;
			for (int f = 0; f < n; f++) // rows of the caller's planes may be padded: 2-D copies, plane by plane
				for (int k = 0; k < nplanes; k++) {
					const size_t row = (size_t)po.stride[k];
					CUDA_TRY(cudaMemcpy2DAsync(out.plane[k] + (size_t)(f0 + f) * out.frame_stride, (size_t)out.stride[k],
					                           c.d_scratch + (size_t)f * fb + soff[k], row, row, (size_t)plane_lines(out, k, g),
					                           cudaMemcpyDeviceToDevice, st));
				}
		}
		advance_registers(g, (uint64_t)nframes);
		return VFGS_B200_OK;
	}
	const int t = (int)(c.tab_next++ & 1u);
	if (int rc = grow(c.d_tab[t], c.tab_cap[t], (size_t)nframes * g.R * g.spitch * kBlockTableBytes + 16)) return rc;
	if (c.tab_used[t]) CUDA_TRY(cudaStreamWaitEvent(c.s_tab, c.tab_free[t], 0)); // the grain kernels of two calls ago read this buffer
	if (int rc = run_frames_device(in, out, nframes, g, in_place, hw().line_rnd, 0, c.d_tab[t], st, c.s_tab, c.tab_ready[t])) return rc;
	CUDA_TRY(cudaEventRecord(c.tab_free[t], st));
	c.tab_used[t] = true;
	advance_registers(g, (uint64_t)nframes);
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
	fill_common(p, g);
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
	if (images_before(st) || launch_apply(p, st) || images_after(st)) fatal("vfgs_add_grain_line");
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
	if (!in->y || !in->uv || !out->y || !out->uv) return set_err(VFGS_B200_ERR_ARG, "null plane pointer");
	const HwState& h = hw();
	const int depth = 8 + h.bs;
	if (in->format != (depth == 10 ? VFGS_B200_P010 : VFGS_B200_NV12))
		return set_err(VFGS_B200_ERR_ARG, "input format %d does not match the configured depth %d (NV12 = 8, P010 = 10)", in->format, depth);
	if (out->format != in->format && !(out->format == VFGS_B200_NV12 && in->format == VFGS_B200_P010))
		return set_err(VFGS_B200_ERR_ARG, "output format %d from input format %d (same format, or NV12 from P010)", out->format, in->format);
	if (h.csubx != 2)
		return set_err(VFGS_B200_ERR_ARG, "semi-planar frames are 4:2:0 or 4:2:2 (4:4:4 frames are planar)");
	Geometry g;
	if (int rc = make_geometry(g, width, height, out->format == in->format ? 0 : 8)) return rc;
	for (int side = 0; side < 2; side++) {
		const vfgs_b200_semiplanar& f = side ? *out : *in;
		const int64_t sample = (int64_t)(side ? g.out_sample : g.in_sample);
		if (f.stride_y < (int64_t)g.width * sample || f.stride_uv < 2 * (int64_t)g.cw * sample)
			return set_err(VFGS_B200_ERR_ARG, "%s line stride shorter than a row", side ? "output" : "input");
		if (sample == 2 && (((uintptr_t)f.y | (uintptr_t)f.uv | (uint64_t)f.stride_y | (uint64_t)f.stride_uv | (uint64_t)f.frame_stride) & 1))
			return set_err(VFGS_B200_ERR_ARG, "%s P010 planes and strides must be 2-byte aligned", side ? "output" : "input");
	}
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
		if (int rc = run_frames_device(frame_planes(pi), frame_planes(po), n, g, false, epoch, (uint64_t)f0, s.d_streams, c.s_k)) return rc;
		CUDA_TRY(cudaEventRecord(s.k_done, c.s_k));
		CUDA_TRY(cudaStreamWaitEvent(c.s_d2h, s.k_done, 0));
		CUDA_TRY(cudaMemcpyAsync(hout + (size_t)f0 * g.out_frame_bytes, s.d_out, (size_t)n * g.out_frame_bytes, cudaMemcpyDeviceToHost, c.s_d2h));
		CUDA_TRY(cudaEventRecord(s.d2h_done, c.s_d2h));
	}
	CUDA_TRY(cudaStreamSynchronize(c.s_d2h));
	CUDA_TRY(cudaStreamSynchronize(c.s_k));
	CUDA_TRY(cudaStreamSynchronize(c.s_h2d));
	advance_registers(g, (uint64_t)nframes);
	return VFGS_B200_OK;
}

int vfgs_b200_skip_frames(int64_t nframes, int width, int height)
{
	if (nframes < 0) return set_err(VFGS_B200_ERR_ARG, "negative frame count");
	Geometry g;
	if (int rc = make_geometry(g, width, height, 0)) return rc;
	advance_registers(g, (uint64_t)nframes);
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
size_t vfgs_b200_get_state(void* dst, size_t cap)
{
	const HwState& h = hw();
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
