// vfgs_kernels.cuh -- the two CUDA kernels of the hot path (sm_100a).
//
//   lfsr_states_kernel   replaces the serial LFSR chain of vfgs_hw.c:74-79,291-298,309-310: one warp
//                        per (frame, block-row) jumps the epoch state ahead by
//                        t = (f (R-1) + r) nb steps with 32x32 GF(2) matrix powers (one output bit
//                        per lane, gathered by a ballot) and emits the row's bit-stream, 32 bits per
//                        ballot, from which every block takes its 32-bit window.
//   fgs_apply_kernel     replaces add_grain_block + vfgs_add_grain_line + the frame walk of
//                        vfgs_main.c:664-682 + yuv_to_8bit: persistent CTAs copy the LUT/pattern image
//                        to shared memory with one bulk async copy (TMA engine, cp.async.bulk +
//                        mbarrier) and then loop over warp-tasks (fgs_task.h) with 128-bit global
//                        loads and stores.
#pragma once
#include <cuda_runtime.h>
#include "vfgs_tables.h"
#include "fw_device.h"

namespace vfgs {

constexpr int kCtaThreads = 256;
constexpr int kLfsrThreads = 128; // lfsr_states_kernel
constexpr int kWarpsPerCta = kCtaThreads / 32;

// ---- mbarrier / bulk-copy PTX -------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p)
{
	return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
	asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
	asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes)
{
	asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
	asm volatile(
	    "{\n"
	    ".reg .pred p;\n"
	    "WAIT_%=:\n"
	    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
	    "@p bra DONE_%=;\n"
	    "bra WAIT_%=;\n"
	    "DONE_%=:\n"
	    "}\n" :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}
// global -> shared bulk copy; bytes % 16 == 0, both addresses 16-byte aligned
__device__ __forceinline__ void bulk_copy_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
	asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
	             :: "r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// ---- LFSR registers per block -------------------------------------------------------------
// states[(f * R + r) * spitch + 1 + b] = LFSR register of block b of block-row r of frame frame0 + f
// (words 0 and nb + 1 of a row are padding; states may be null when only the general kernel's table is not needed); woffs, when not null, gets the same blocks' pattern-window
// offsets for the fast path (four uint16 per block: Y, U, V, unused). One warp per (frame, block-row): jump the epoch register
// ahead by t = ((frame0 + f) (R - 1) + r) nb steps with the matrix powers pow2 (JumpTable as
// uint32[64][32]; lane i owns output bit i, a ballot assembles the word), then walk the row 32 steps
// at a time: consecutive blocks are consecutive 32-bit windows of one bit-stream, so lane l takes
// window l of every {word k, word k+1} pair and the 32 registers go out as one coalesced store.
__device__ __forceinline__ void lfsr_row_tables(uint32_t epoch_state, const uint32_t* __restrict__ pow2, uint32_t* __restrict__ states,
                                                uint16_t* __restrict__ woffs, const WoffParams& wp, int warp, int R, int nb,
                                                int spitch, unsigned long long frame0, int lane)
{
	const int f = warp / R, r = warp - f * R;
	unsigned long long t = ((frame0 + (unsigned long long)f) * (unsigned long long)(R - 1) + (unsigned long long)r) *
	                       (unsigned long long)nb;
	uint32_t s = epoch_state;
	// matrix rows are fetched eight powers at a time, independently of the state, so the dependent
	// chain is only AND + POPC + ballot per set bit of t
	for (int k0 = 0; k0 < kJumpBits && (t >> k0) != 0; k0 += 8) {
		uint32_t rows[8];
#pragma unroll
		for (int j = 0; j < 8; j++) rows[j] = pow2[(k0 + j) * 32 + lane];
#pragma unroll
		for (int j = 0; j < 8; j++)
			if ((t >> (k0 + j)) & 1ull) s = __ballot_sync(0xffffffffu, __popc(rows[j] & s) & 1);
	}
	const uint32_t step32 = pow2[5 * 32 + lane];
	uint32_t* dst = states + (size_t)warp * spitch; // states == nullptr: only the window offsets are wanted
	if (states && lane == 0) { dst[0] = 0; dst[nb + 1] = 0; }
	for (int b0 = 0; b0 < nb; b0 += 32) {
		const uint32_t next = __ballot_sync(0xffffffffu, __popc(step32 & s) & 1);
		if (b0 + lane < nb) {
			const uint32_t st = __funnelshift_r(s, next, lane);
			if (states) dst[1 + b0 + lane] = st;
			if (woffs) { // pattern-window offsets of the block for the fast path, one 8-byte store
				uint2 v; // fast or gather format, per component
				v.x = window_offset<0>(st, wp.c[0]) | (window_offset<1>(st, wp.c[1]) << 16);
				v.y = window_offset<2>(st, wp.c[2]);
				*(uint2*)(woffs + ((size_t)warp * spitch + 1 + b0 + lane) * 4) = v;
			}
		}
		s = next;
	}
}

__global__ void __launch_bounds__(kLfsrThreads)
lfsr_states_kernel(uint32_t epoch_state, const uint32_t* __restrict__ pow2, uint32_t* __restrict__ states,
                   uint16_t* __restrict__ woffs, const WoffParams wp,
                   int nframes, int R, int nb, int spitch, unsigned long long frame0)
{
	const int warp = (int)((blockIdx.x * (unsigned)blockDim.x + threadIdx.x) >> 5);
	const int lane = threadIdx.x & 31;
	if (warp >= nframes * R) return; // warp-uniform
	lfsr_row_tables(epoch_state, pow2, states, woffs, wp, warp, R, nb, spitch, frame0, lane);
}

// Job-table form (vfgs_b200_add_grain_jobs_device): the block tables of every job of a call in one launch. One warp per
// (job, frame, block-row); the job is found by binary search over the prefix of nframes * R (StreamJob::warp0). Frame 0
// of a job is its session's register position at enqueue (StreamJob::epoch).
__global__ void __launch_bounds__(kLfsrThreads)
lfsr_states_jobs_kernel(const uint32_t* __restrict__ pow2, const StreamJob* __restrict__ jobs, int njobs, long long nwarps)
{
	const long long warp = (long long)((blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) >> 5);
	const int lane = threadIdx.x & 31;
	if (warp >= nwarps) return; // warp-uniform
	const StreamJob& J = jobs[stream_job_of(jobs, njobs, warp)];
	lfsr_row_tables(J.epoch, pow2, J.states, J.woffs, J.wp, (int)(warp - J.warp0), J.R, J.nb, J.spitch, 0ull, lane);
}

// ---- grain synthesis -----------------------------------------------------------------------
// the general task code wants ~128 registers: 2 CTAs per SM without spills measured ahead of 4 with (1366 x 768: 912 vs 681 GB/s)
#ifndef VFGS_GENERAL_CTAS
#define VFGS_GENERAL_CTAS 2
#endif
__global__ void __launch_bounds__(kCtaThreads, VFGS_GENERAL_CTAS)
fgs_apply_kernel(const __grid_constant__ FgsParams p)
{
	extern __shared__ __align__(128) uint8_t tab[];
	__shared__ __align__(8) uint64_t bar;

	if (threadIdx.x == 0) mbar_init(&bar, 1);
	__syncthreads();
	if (threadIdx.x == 0) {
		mbar_arrive_expect_tx(&bar, (uint32_t)p.blob_bytes);
		bulk_copy_g2s(tab, p.blob, (uint32_t)p.blob_bytes, &bar);
	}
	mbar_wait(&bar, 0);

	const int lane = threadIdx.x & 31;
	const long long stride = (long long)gridDim.x * kWarpsPerCta;
	for (long long task = (long long)blockIdx.x * kWarpsPerCta + (threadIdx.x >> 5); task < p.total_tasks; task += stride)
		process_task(p, tab, (uint32_t)task, lane);
}

// Fast path: single-pattern components (fgs_fast.h); EDGE: the variant for rows at any sample-aligned address and
// widths that are not a multiple of 8 samples (packed ragged pictures), everything else identical. One 1024-thread persistent CTA per
// SM (measured faster than 2 x 512: one table image per SM, more of the unified array left to L1, which
// the 16-bit-output variant uses as its landing buffer for the lines in flight).
// Shared memory: three per-lane replicated LUTs of scale << (16 - shift) (3 x 32 KB, each on a 32 KB
// boundary of the shared window, expanded here from the 1 KB compact LUT in global memory) and the
// components' +/- pattern copies, brought in by bulk async copies: in the gap between the start of dynamic
// shared memory and the first LUT as far as they fit (FgsParams::fimg_off < 0), else behind the third LUT.
// CTA size per variant, measured on B200 (scripts/ab_sweep.sh, same box, 4K/8K/1080p): the 8-bit-output kernel
// is bound by instruction issue and the shared-memory pipe and wants all 32 warps; the 16-bit-output kernel is
// HBM-bound with equal read and write streams and peaks at 24 warps x 4 lines in flight per lane (more
// outstanding lines per SM lower the DRAM efficiency again: 768 threads 95.6 %, 1024 threads 89 % of the
// measured copy bandwidth at 4K).
#ifndef VFGS_FAST_THREADS8
#define VFGS_FAST_THREADS8 768   // 16-bit in, 8-bit out
#endif
#ifndef VFGS_FAST_THREADS16
#define VFGS_FAST_THREADS16 768  // 16-bit in, 16-bit out
#endif
#ifndef VFGS_FAST_THREADS_IN8
#define VFGS_FAST_THREADS_IN8 896   // 8-bit in, 8-bit out (2 bytes per sample: issue-bound; 73 registers keep the 16-samples-per-lane path free of spills)
#endif
#ifndef VFGS_FAST_THREADS_EDGE
#define VFGS_FAST_THREADS_EDGE 768  // EDGE variants (ragged / unaligned rows): the piecewise accesses want the 85 registers of 24 warps
#endif
#ifndef VFGS_FAST_THREADS16W
#define VFGS_FAST_THREADS16W 512 // 16-bit in, 16-bit out, every component on the 16-samples-per-lane path (ALLWIDE): 128 registers hold four
                                 // 32-byte lines per lane; 4K 10-bit 0.93 (8 samples per lane) -> 0.965 (768 threads x 2 lines) -> 0.98
#endif
template <bool IN16, bool OUT8, bool EDGE = false, bool ALLWIDE = false> struct FastCta {
	static_assert(!ALLWIDE || (IN16 && !OUT8 && !EDGE), "ALLWIDE exists for 16-bit input and output only");
	static constexpr int threads = ALLWIDE ? VFGS_FAST_THREADS16W : EDGE ? VFGS_FAST_THREADS_EDGE : !IN16 ? VFGS_FAST_THREADS_IN8 : OUT8 ? VFGS_FAST_THREADS8 : VFGS_FAST_THREADS16;
};
inline int fast_threads(bool in16, bool out8, bool edge = false, bool allwide = false)
{
	return allwide ? VFGS_FAST_THREADS16W : edge ? VFGS_FAST_THREADS_EDGE : !in16 ? VFGS_FAST_THREADS_IN8 : out8 ? VFGS_FAST_THREADS8 : VFGS_FAST_THREADS16;
}

// SEMI: semi-planar frames (process_task_fast), same CTA sizes as the planar variants.
template <bool IN16, bool OUT8, bool EDGE = false, bool ALLWIDE = false, bool SEMI = false>
__global__ void __launch_bounds__(FastCta<IN16, OUT8, EDGE, ALLWIDE>::threads, 1)
fgs_apply_fast_kernel(const __grid_constant__ FgsParams p)
{
	constexpr int kFastThreads = FastCta<IN16, OUT8, EDGE, ALLWIDE>::threads, kFastWarps = kFastThreads / 32;
	extern __shared__ __align__(128) uint8_t smem[];
	__shared__ __align__(8) uint64_t bar;

	// the host laid the images out for the gap in front of the first LUT, which it measured with a probe launch
	const uint32_t pad = (0u - smem_u32(smem)) & (uint32_t)(kLutAlign - 1);
	if (p.probe) {
		if (threadIdx.x == 0) *p.probe = pad;
		return;
	}
#ifdef VFGS_DEBUG_ASSERTS
	if (pad != (uint32_t)p.fpad) __trap();
#endif
	uint8_t* lut_ptr = smem + pad;

	if (threadIdx.x == 0) mbar_init(&bar, 1);
	__syncthreads();
	if (threadIdx.x == 0) {
		mbar_arrive_expect_tx(&bar, (uint32_t)(p.fimg_bytes[0] + p.fimg_bytes[1] + p.fimg_bytes[2]));
		for (int c = 0; c < 3; c++)
			if (p.fimg_bytes[c]) bulk_copy_g2s(lut_ptr + p.fimg_off[c], p.fblob + p.fimg_src[c], (uint32_t)p.fimg_bytes[c], &bar);
	}
	expand_fast_luts((uint32_t*)lut_ptr, (const uint32_t*)p.fblob, (uint32_t)p.pow16, threadIdx.x, kFastThreads);
	mbar_wait(&bar, 0);
	__syncthreads();

	const int lane = threadIdx.x & 31;
	const smem_addr_t lut = smem_addr(lut_ptr);
	const long long stride = (long long)gridDim.x * kFastWarps;
	for (long long task = (long long)blockIdx.x * kFastWarps + (threadIdx.x >> 5); task < p.total_tasks; task += stride)
		process_task_fast<IN16, OUT8, EDGE, ALLWIDE, SEMI>(p, lut, (uint32_t)task, lane);
}

// Before a CTA overwrites tables the previous job's tasks read: every warp is done with them, and the generic-proxy
// reads are ordered before the bulk copy's async-proxy writes.
__device__ __forceinline__ void multi_switch_barrier()
{
	__syncthreads();
	if (threadIdx.x == 0) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// MULTI form (vfgs_b200_add_grain_jobs_device): the warp-tasks of several jobs of one instantiation, concatenated in job
// order, in one launch. CTA b takes the contiguous range multi_cta_range(b); inside each job's part of it its warps take
// tasks base + k * warps + w. Where the range enters the next job, the CTA waits for its warps, brings in that job's
// images (next mbarrier phase) and re-expands the LUTs with that job's scale shift. The job's FgsParams are read from
// global memory (uniform, L1-resident): no static shared memory is added, so the probe measures the same pad.
template <bool IN16, bool OUT8, bool EDGE = false, bool ALLWIDE = false, bool SEMI = false>
__global__ void __launch_bounds__(FastCta<IN16, OUT8, EDGE, ALLWIDE>::threads, 1)
fgs_apply_fast_multi_kernel(const __grid_constant__ MultiParams m)
{
	constexpr int kFastThreads = FastCta<IN16, OUT8, EDGE, ALLWIDE>::threads, kFastWarps = kFastThreads / 32;
	extern __shared__ __align__(128) uint8_t smem[];
	__shared__ __align__(8) uint64_t bar;

	const uint32_t pad = (0u - smem_u32(smem)) & (uint32_t)(kLutAlign - 1);
	if (m.probe) {
		if (threadIdx.x == 0) *m.probe = pad;
		return;
	}
	uint8_t* lut_ptr = smem + pad;
	if (threadIdx.x == 0) mbar_init(&bar, 1);
	__syncthreads();

	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const smem_addr_t lut = smem_addr(lut_ptr);
	MultiCursor cur;
	multi_begin(m.task0, m.njobs, (int)gridDim.x, (int)blockIdx.x, cur);
	uint32_t phase = 0;
	int j;
	long long lo, end;
	while (multi_next(m.task0, cur, j, lo, end)) {
		const long long t0 = m.task0[j];
		const FgsParams& p = m.jobs[j];
		if (phase) multi_switch_barrier();
		if (threadIdx.x == 0) {
			mbar_arrive_expect_tx(&bar, (uint32_t)(p.fimg_bytes[0] + p.fimg_bytes[1] + p.fimg_bytes[2]));
			for (int c = 0; c < 3; c++)
				if (p.fimg_bytes[c]) bulk_copy_g2s(lut_ptr + p.fimg_off[c], p.fblob + p.fimg_src[c], (uint32_t)p.fimg_bytes[c], &bar);
		}
		expand_fast_luts((uint32_t*)lut_ptr, (const uint32_t*)p.fblob, (uint32_t)p.pow16, threadIdx.x, kFastThreads);
		mbar_wait(&bar, phase & 1);
		phase++;
		__syncthreads();
		for (long long task = lo + warp; task < end; task += kFastWarps)
			process_task_fast<IN16, OUT8, EDGE, ALLWIDE, SEMI>(p, lut, (uint32_t)(task - t0), lane);
	}
}

// Gather path: components with sample-adaptive pattern selection (fgs_gather.h). Shared memory: one
// per-lane replicated LUT (32 KB, entry layouts: gather_lut_entry) per gather component, each on a
// 32 KB boundary, then the general table image (compact LUTs + pattern slots; FOLD: + the negated slots)
// brought in by one bulk copy.
#ifndef VFGS_GATHER_THREADS
#define VFGS_GATHER_THREADS 896
#define VFGS_GATHER_CTAS 1
#endif
constexpr int kGatherThreads = VFGS_GATHER_THREADS; // one CTA per SM at up to 72 registers (the gather path carries more per-lane state);
                                                    // measured ahead of 2 x 384 (one table image per SM) and of 640-832 and 960-1024 threads
constexpr int kGatherWarps = kGatherThreads / 32;

// MSB: P010 luma of semi-planar frames (16-bit input only).
template <bool IN16, bool OUT8, bool FOLD, bool SHIFT, bool MSB = false>
__global__ void __launch_bounds__(kGatherThreads, VFGS_GATHER_CTAS)
fgs_apply_gather_kernel(const __grid_constant__ FgsParams p)
{
	extern __shared__ __align__(128) uint8_t smem[];
	__shared__ __align__(8) uint64_t bar;

	uint8_t* lut_ptr = smem + ((0u - smem_u32(smem)) & (uint32_t)(kLutAlign - 1));
	uint8_t* img_ptr = lut_ptr + p.ngather * kLutBytes;

	if (threadIdx.x == 0) mbar_init(&bar, 1);
	__syncthreads();
	if (threadIdx.x == 0) {
		mbar_arrive_expect_tx(&bar, (uint32_t)p.blob_bytes);
		bulk_copy_g2s(img_ptr, p.blob, (uint32_t)p.blob_bytes, &bar);
	}
	mbar_wait(&bar, 0);
	for (int c = 0; c < 3; c++) {
		if (p.glut_index[c] < 0) continue;
		const uint16_t* compact = (const uint16_t*)(img_ptr + p.lut_off) + c * 256; // scale | slot << 8
		uint32_t* lut = (uint32_t*)(lut_ptr + p.glut_index[c] * kLutBytes);
		const uint32_t slot_bytes = (uint32_t)p.pat_size[c ? 1 : 0];
		for (int i = threadIdx.x; i < 256 * 32; i += kGatherThreads) {
			lut[i] = gather_lut_entry<IN16>(compact[i >> 5], slot_bytes);
		}
	}
	__syncthreads();

	const int lane = threadIdx.x & 31;
	const smem_addr_t luts = smem_addr(lut_ptr), img = smem_addr(img_ptr);
	const long long stride = (long long)gridDim.x * kGatherWarps;
	for (long long task = (long long)blockIdx.x * kGatherWarps + (threadIdx.x >> 5); task < p.total_tasks; task += stride)
		process_task_gather<IN16, OUT8, FOLD, SHIFT, MSB>(p, luts, img, (uint32_t)task, lane);
}

// MULTI form of the gather kernel: the schedule and the job switch of fgs_apply_fast_multi_kernel; a switch brings in the
// next job's general image and rebuilds its per-lane LUTs.
template <bool IN16, bool OUT8, bool FOLD, bool SHIFT, bool MSB = false>
__global__ void __launch_bounds__(kGatherThreads, VFGS_GATHER_CTAS)
fgs_apply_gather_multi_kernel(const __grid_constant__ MultiParams m)
{
	extern __shared__ __align__(128) uint8_t smem[];
	__shared__ __align__(8) uint64_t bar;

	uint8_t* lut_ptr = smem + ((0u - smem_u32(smem)) & (uint32_t)(kLutAlign - 1));
	if (threadIdx.x == 0) mbar_init(&bar, 1);
	__syncthreads();

	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const smem_addr_t luts = smem_addr(lut_ptr);
	MultiCursor cur;
	multi_begin(m.task0, m.njobs, (int)gridDim.x, (int)blockIdx.x, cur);
	uint32_t phase = 0;
	int j;
	long long lo, end;
	while (multi_next(m.task0, cur, j, lo, end)) {
		const long long t0 = m.task0[j];
		const FgsParams& p = m.jobs[j];
		uint8_t* img_ptr = lut_ptr + p.ngather * kLutBytes;
		if (phase) multi_switch_barrier();
		if (threadIdx.x == 0) {
			mbar_arrive_expect_tx(&bar, (uint32_t)p.blob_bytes);
			bulk_copy_g2s(img_ptr, p.blob, (uint32_t)p.blob_bytes, &bar);
		}
		mbar_wait(&bar, phase & 1);
		phase++;
		for (int c = 0; c < 3; c++) {
			if (p.glut_index[c] < 0) continue;
			const uint16_t* compact = (const uint16_t*)(img_ptr + p.lut_off) + c * 256;
			uint32_t* lut = (uint32_t*)(lut_ptr + p.glut_index[c] * kLutBytes);
			const uint32_t slot_bytes = (uint32_t)p.pat_size[c ? 1 : 0];
			for (int i = threadIdx.x; i < 256 * 32; i += kGatherThreads) lut[i] = gather_lut_entry<IN16>(compact[i >> 5], slot_bytes);
		}
		__syncthreads();
		const smem_addr_t img = smem_addr(img_ptr);
		for (long long task = lo + warp; task < end; task += kGatherWarps)
			process_task_gather<IN16, OUT8, FOLD, SHIFT, MSB>(p, luts, img, (uint32_t)(task - t0), lane);
	}
}

// ---- firmware layer: pattern jobs (fw_device.h) -------------------------------------------------
// One CTA per job, jobs of a configuration one after the other on the table stream (they share the firmware's pattern
// buffer, fw_device.h). The frequency-filtering job is two 64 x 64 x 64 integer matrix passes spread over the CTA; the
// auto-regressive filter takes the CTA for its noise term (lane-chunked LFSR walks from a jump-ahead each) and one warp
// for the causal filter itself, which runs as a wavefront over anti-diagonals (fw_ar_wave_step: 370 steps for the
// 82 x 73 luma field instead of a 5,986-sample serial walk).
constexpr int kFwThreads = 256;

// The job's pattern into scratch->P. gauss: the Gaussian table in shared memory (AR jobs); noise, field: shared buffers
// of 82 x 73 bytes.
__device__ __forceinline__ void fw_make_pattern(const FwJob& job, const FwTables* __restrict__ tables, const uint32_t* __restrict__ pow2,
                                                FwScratch* scratch, const int8_t* gauss, int8_t* noise, int8_t* field, int tid)
{
	if (job.kind == kFwAR) {
		const int sub = job.size == 32 ? 2 : 1, bytes = sub > 1 ? 44 * 38 : 82 * 73;
		fw_ar_noise(job, gauss, pow2, noise, tid, kFwThreads);
		__syncthreads();
		if (tid < 32) {
			const int steps = fw_ar_wave_steps(job);
			for (int t = 0; t < steps; t++) {
				fw_ar_wave_step(job, noise, field, scratch->Lbuf, t, tid);
				__syncwarp();
			}
		}
		__syncthreads();
		int8_t* keep = sub > 1 ? scratch->Cbuf : scratch->Lbuf; // the luma field stays for the chroma jobs (luma injection)
		for (int i = tid; i < bytes; i += kFwThreads) keep[i] = field[i];
		__syncthreads();
		fw_ar_phase1(job, *scratch, tid, kFwThreads);
	} else {
		if (tid == 0) fw_ff_phase0(job, *scratch);
		__syncthreads();
		fw_ff_phase1(job, *tables, *scratch, tid, kFwThreads);
		__syncthreads();
		fw_ff_phase2(job, *tables, *scratch, tid, kFwThreads);
		__syncthreads();
		fw_ff_phase3(job, *tables, *scratch, tid, kFwThreads);
	}
	__syncthreads();
}

__global__ void __launch_bounds__(kFwThreads)
fw_pattern_kernel(const FwJob job, const FwTables* __restrict__ tables, const uint32_t* __restrict__ pow2, FwScratch* scratch, int8_t* pattern)
{
	__shared__ int8_t field[73 * 82];
	__shared__ int8_t noise[73 * 82];
	__shared__ int8_t gauss[2048];
	const int tid = threadIdx.x;
	if (job.kind == kFwAR) {
		for (int i = tid; i < 2048; i += kFwThreads) gauss[i] = tables->gauss[i];
		__syncthreads();
	}
	fw_make_pattern(job, tables, pow2, scratch, gauss, noise, field, tid);
	fw_store_phase(job, *scratch, pattern, tid, kFwThreads);
}

// ---- firmware layer for sessions (vfgs_b200_session_init_metadata) ------------------------------------
// One entry of a metadata call: a session's pattern jobs in firmware order, its new LUTs and image layout (host-made),
// and where its firmware working memory, pattern store and table images live.
struct MetaEntry {
	FwJob jobs[2 * kFwMaxPatterns];
	int njobs;
	int csubx, csuby;
	uint8_t slut[3][256], plut[3][256];
	TableInfo bi;
	FwScratch* scratch;
	int8_t* pattern;       // int8 [2][9][64][64], the session's device pattern store
	uint8_t *blob, *fblob; // the session's general and fast images (kImageBlobCap / kImageFblobCap bytes)
	int8_t* out;           // njobs x 4096: each job's slot after its store, for the copy back to the host
};

// One CTA per entry: the entry's jobs one after the other against its session's working memory and pattern store, then
// both table images from the pattern store and the new LUTs (fill_tables, the code build_tables runs on the host).
__global__ void __launch_bounds__(kFwThreads)
fw_sessions_kernel(const MetaEntry* __restrict__ entries, const FwTables* __restrict__ tables, const uint32_t* __restrict__ pow2)
{
	__shared__ int8_t field[73 * 82];
	__shared__ int8_t noise[73 * 82];
	__shared__ int8_t gauss[2048];
	const MetaEntry& e = entries[blockIdx.x];
	const int tid = threadIdx.x;
	for (int i = tid; i < 2048; i += kFwThreads) gauss[i] = tables->gauss[i];
	__syncthreads();
	for (int k = 0; k < e.njobs; k++) {
		const FwJob& job = e.jobs[k];
		fw_make_pattern(job, tables, pow2, e.scratch, gauss, noise, field, tid);
		fw_store_phase(job, *e.scratch, e.pattern, tid, kFwThreads);
		__syncthreads();
		const int8_t* slot = e.pattern + ((size_t)job.bank * kSlots + job.slot) * 4096;
		for (int i = tid; i < 4096; i += kFwThreads) e.out[(size_t)k * 4096 + i] = slot[i];
	}
	__syncthreads();
	const TableSrc src = {e.pattern, &e.slut[0][0], &e.plut[0][0], e.csubx, e.csuby};
	fill_tables(src, e.bi, e.blob, e.fblob, tid, kFwThreads);
}

} // namespace vfgs
