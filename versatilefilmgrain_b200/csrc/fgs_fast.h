// fgs_fast.h -- the throughput path of the grain kernel: components whose pattern LUT selects one
// single pattern slot (every AFGS1 config, most FGC-SEI configs; SURVEY.md appendix A), rows
// aligned for 128-bit access, widths a multiple of 8 samples.
//
// Same decomposition as fgs_task.h (warp-task = 32 lane units x the lines of one stripe, neighbours'
// edge samples recomputed from their own LFSR window); a lane unit is 16 samples -- a whole 16-sample
// block, one 256-bit access per line -- where width and alignment allow it (wide_task_body, the form
// the usual picture sizes take), else 8 samples (fast_task_body). The per-sample work is cut to the bone:
//   * with one pattern slot the unscaled grain does not depend on the sample, so a lane's 8 grain
//     bytes per line are one contiguous octet of a pattern row: one 64-bit shared load (the image
//     keeps column-shifted copies so that every window starts on an 8-byte boundary, and skews the
//     row pitch so that the windows of a line spread over all banks);
//   * the block's random sign (vfgs_hw.c:218 "* s") is folded into WHICH COPY of the pattern is
//     read: the table image holds +pattern and -pattern (the host only takes this path when no
//     pattern byte is -128), so no per-sample sign multiply is left;
//   * the scale LUT (vfgs_hw.c:239) is replicated per lane in shared memory, one table of
//     [256][32] words = scale << (16 - shift) per component: a lane only ever touches its own bank,
//     so the 256-entry lookup with random intensities is conflict-free by construction, and the
//     rounded shift of vfgs_hw.c:263 is the upper half-word of one multiply-add;
//   * add + clip (vfgs_hw.c:265-267) run on two samples at a time with the packed 16-bit min/max
//     instructions (VIADDMNMX / VIMNMX .S16x2); 10-bit samples stay packed in their load words,
//     8-bit samples are widened two at a time into the same form.
// Host-compilable like fgs_task.h (tests/emu) -- the helpers below emulate the few PTX instructions.
#pragma once
#include <stddef.h>
#include <type_traits>
#include "fgs_task.h"

namespace vfgs {

// ---- byte permute and packed 16-bit helpers ------------------------------------------------
// PTX prmt.b32, default mode: selector nibble n (bits 2:0) picks byte n of {b,a}; nibble bit 3
// replicates that byte's sign bit instead.
VFGS_HD uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel)
{
#if defined(__CUDA_ARCH__)
	uint32_t d;
	asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
	return d;
#else
	const uint64_t src = ((uint64_t)b << 32) | a;
	uint32_t d = 0;
	for (int i = 0; i < 4; i++) {
		const uint32_t n = (sel >> (4 * i)) & 0xf;
		uint32_t byte = (uint32_t)(src >> (8 * (n & 7))) & 0xff;
		if (n & 8) byte = (byte & 0x80) ? 0xff : 0x00;
		d |= byte << (8 * i);
	}
	return d;
#endif
}
// sign-extended byte e (0..7) of the octet {w1,w0}. FMA_TOP: the top byte of each word comes out of a multiply-high
// (arithmetic shift by 24 on the FMA pipe). Round 1 measured that ahead for the issue-bound variants under its burst
// protocol; under the sustained protocol IMAD.HI is the expensive instruction and the PRMT wins, so it is off now.
#ifndef VFGS_OCTET_TOP_ON_FMA
#define VFGS_OCTET_TOP_ON_FMA 0 // round 1: 1. Under the sustained protocol the multiply-high costs more than the PRMT it saves (profiles/r02_wide16_ab.md, trips 4-5)
#endif
template <int E, bool FMA_TOP = false>
VFGS_HD int octet_byte(uint32_t w0, uint32_t w1)
{
	if (FMA_TOP && (E == 3 || E == 7)) {
		const int w = (int)(E == 3 ? w0 : w1);
#if defined(__CUDA_ARCH__)
		return __mulhi(w, 256);
#else
		return (int)(((long long)w * 256) >> 32);
#endif
	}
	constexpr uint32_t n = (uint32_t)E, s = 8u | (uint32_t)E;
	return (int)prmt(w0, w1, n | (s << 4) | (s << 8) | (s << 12));
}
VFGS_HD uint32_t add_max_s16x2(uint32_t a, uint32_t b, uint32_t c) // per half: max(a + b, c), signed
{
#if defined(__CUDA_ARCH__)
	return __viaddmax_s16x2(a, b, c);
#else
	uint32_t r = 0;
	for (int i = 0; i < 2; i++) {
		int16_t x = (int16_t)((int16_t)(a >> (16 * i)) + (int16_t)(b >> (16 * i)));
		const int16_t y = (int16_t)(c >> (16 * i));
		x = x > y ? x : y;
		r |= (uint32_t)(uint16_t)x << (16 * i);
	}
	return r;
#endif
}
VFGS_HD uint32_t min_s16x2(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
	return __vmins2(a, b);
#else
	uint32_t r = 0;
	for (int i = 0; i < 2; i++) {
		const int16_t x = (int16_t)(a >> (16 * i)), y = (int16_t)(b >> (16 * i));
		r |= (uint32_t)(uint16_t)(x < y ? x : y) << (16 * i);
	}
	return r;
#endif
}
VFGS_HD uint32_t min_u16x2(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
	return __vminu2(a, b);
#else
	uint32_t r = 0;
	for (int i = 0; i < 2; i++) {
		const uint16_t x = (uint16_t)(a >> (16 * i)), y = (uint16_t)(b >> (16 * i));
		r |= (uint32_t)(x < y ? x : y) << (16 * i);
	}
	return r;
#endif
}

VFGS_HD uint32_t mulhi_u32(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
	return __umulhi(a, b);
#else
	return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
// a >> N. Round 1 did this by a high multiply to move work from the ALU pipe to the FMA pipe; measured again in round 2
// under the sustained protocol the plain shift wins on every kernel (IMAD.HI is the expensive one of the two:
// profiles/r02_gather_ab.md, "LUT entry layout and shifts"), so the multiply is only a build-time knob now.
#ifndef VFGS_SHR_ON_FMA
#define VFGS_SHR_ON_FMA 0
#endif
template <int N>
VFGS_HD uint32_t shr_fma(uint32_t a)
{
	return VFGS_SHR_ON_FMA ? mulhi_u32(a, 1u << (32 - N)) : a >> N;
}

// ---- shared-memory image of the fast path --------------------------------------------------
//   lut   uint32 lut[3][256][32]: per component a per-lane replicated LUT of scale << (16 - scale_shift)
//         (built by the CTA from the compact LUT), each table on a 32 KB boundary of the shared window so
//         that "lane column | index bits" is a plain OR
//   img   per component its pattern slot as +pattern and -pattern, each in column-shifted copies
//         (fast_copies), rows packed to fpat_stride bytes; the image of component c starts fimg_off[c] bytes
//         from the first LUT (in front of it or behind the third one), fpat_off is relative to that
// Addresses are absolute: 32-bit shared-window addresses on the device, pointers in the host build.
constexpr int kLutBytes = 256 * 32 * 4;
constexpr int kLutAlign = 32768;

// lut[c][i][lane] = sLUT[c][i] << (16 - shift) from compact[i] = sLUT[Y][i] | sLUT[U][i] << 8 | sLUT[V][i] << 16;
// thread `tid` of `nthreads` does its share (the host build calls it with one thread).
VFGS_HD void expand_fast_luts(uint32_t* lut, const uint32_t* compact, uint32_t pow16, int tid, int nthreads)
{
	for (int i = tid; i < 3 * 256 * 32; i += nthreads) {
		const int c = i >> 13;
		lut[i] = ((compact[(i >> 5) & 255] >> (8 * c)) & 0xffu) * pow16;
	}
}

#if defined(__CUDA_ARCH__)
typedef uint32_t smem_addr_t;
__device__ __forceinline__ smem_addr_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t lds32(smem_addr_t a) { uint32_t v; asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ void lds64(smem_addr_t a, uint32_t& lo, uint32_t& hi) { asm("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(lo), "=r"(hi) : "r"(a)); }
__device__ __forceinline__ int lds_s8(smem_addr_t a) { int v; asm("ld.shared.s8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ int lds_u8(smem_addr_t a) { int v; asm("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
#else
typedef uintptr_t smem_addr_t;
inline smem_addr_t smem_addr(const void* p) { return (uintptr_t)p; }
inline uint32_t lds32(smem_addr_t a) { return *(const uint32_t*)a; }
inline void lds64(smem_addr_t a, uint32_t& lo, uint32_t& hi) { lo = ((const uint32_t*)a)[0]; hi = ((const uint32_t*)a)[1]; }
inline int lds_s8(smem_addr_t a) { return (int)*(const int8_t*)a; }
inline int lds_u8(smem_addr_t a) { return (int)*(const uint8_t*)a; }
#endif

// Measured on B200 (scripts/ab_sweep.sh, -DVFGS_FAST_L1_MODE=0|1|2): with 16-bit output the fast kernel is HBM-bound and runs
// ~2 % faster when the sample loads allocate in L1 (whole 128-byte lines are brought in ahead of the
// neighbouring lanes' requests); with 8-bit output it is issue-bound and the streaming operator is ahead.
#ifndef VFGS_FAST_L1_MODE
#define VFGS_FAST_L1_MODE 1 // 0: never, 1: with 16-bit output, 2: always (build-time knob for experiments)
#endif
template <bool L1_ALLOCATE>
VFGS_HD void ld_samples_16(const uint8_t* p, uint32_t r[4])
{
#if defined(__CUDA_ARCH__)
	if (L1_ALLOCATE) asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(p));
	else ld_global_16(p, r);
#else
	memcpy(r, p, 16);
#endif
}
template <bool L1_ALLOCATE>
VFGS_HD void ld_samples_16_if(const uint8_t* p, uint32_t r[4], bool pred)
{
#if defined(__CUDA_ARCH__)
	if (L1_ALLOCATE)
		asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %5, 0;\n\t@q ld.global.v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
		             : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]) : "l"(p), "r"((uint32_t)pred));
	else
		asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %5, 0;\n\t@q ld.global" VFGS_LD_OP ".v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
		             : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]) : "l"(p), "r"((uint32_t)pred));
#else
	if (pred) memcpy(r, p, 16);
#endif
}

// line prefetch into L1 (no destination register), only when pred is set
VFGS_HD void prefetch_l1(const uint8_t* p, bool pred)
{
#if defined(__CUDA_ARCH__)
	asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %1, 0;\n\t@q prefetch.global.L1 [%0];\n\t}" :: "l"(p), "r"((uint32_t)pred));
#else
	(void)p; (void)pred;
#endif
}

// global load that only happens when pred is set; the destination keeps its value otherwise
VFGS_HD void ld_global_16_if(const uint8_t* p, uint32_t r[4], bool pred)
{
#if defined(__CUDA_ARCH__)
	asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %5, 0;\n\t@q ld.global" VFGS_LD_OP ".v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
	             : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]) : "l"(p), "r"((uint32_t)pred));
#else
	if (pred) memcpy(r, p, 16);
#endif
}
VFGS_HD void ld_global_8_if(const uint8_t* p, uint32_t r[2], bool pred)
{
#if defined(__CUDA_ARCH__)
	asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q ld.global" VFGS_LD_OP ".v2.u32 {%0,%1}, [%2];\n\t}"
	             : "+r"(r[0]), "+r"(r[1]) : "l"(p), "r"((uint32_t)pred));
#else
	if (pred) memcpy(r, p, 8);
#endif
}

// 256-bit accesses (sm_100: LDG.256 / STG.256), 32-byte aligned: the wide 16-bit path, one per line and lane
VFGS_HD void ld_global_32(const uint8_t* p, uint32_t r[8])
{
#if defined(__CUDA_ARCH__)
	asm volatile("ld.global" VFGS_LD_OP ".v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
	             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "l"(p));
#else
	memcpy(r, p, 32);
#endif
}
VFGS_HD void ld_global_32_if(const uint8_t* p, uint32_t r[8], bool pred)
{
#if defined(__CUDA_ARCH__)
	asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %9, 0;\n\t@q ld.global" VFGS_LD_OP ".v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n\t}"
	             : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]) : "l"(p), "r"((uint32_t)pred));
#else
	if (pred) memcpy(r, p, 32);
#endif
}
VFGS_HD void st_global_32(uint8_t* p, const uint32_t r[8])
{
#if defined(__CUDA_ARCH__)
	asm volatile("st.global" VFGS_ST_OP ".v8.u32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
	             :: "l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]) : "memory");
#else
	memcpy(p, r, 32);
#endif
}

// 8 consecutive pattern bytes at address a, a % 8 == 0: the image holds every pattern in as many
// column-shifted copies as the window column has residues modulo 8 (fast_copies), and the block's window
// offset (window_offset) selects the copy in which the window starts on an 8-byte boundary.
#ifndef VFGS_FAST_LDS64
#define VFGS_FAST_LDS64 1 // build-time knob for experiments
#endif
VFGS_HD void octet(smem_addr_t a, uint32_t& w0, uint32_t& w1)
{
	if (VFGS_FAST_LDS64) lds64(a, w0, w1);
	else { w0 = lds32(a); w1 = lds32(a + 4); }
}

// ---- rows at any address, ragged widths (EDGE variant) ---------------------------------------
// The packed .yuv layout (src/yuv.c:162-214: stride = width) puts a row wherever the previous one ended: with a width
// that is not a multiple of 8 samples (1366 x 768, the 964-sample chroma rows of 1928 x 1080) row starts cycle through
// every alignment the sample size allows, and the last lane unit of a row is partial. A lane unit is still 8 samples
// that never straddle a block; only the way its bytes travel changes: the largest naturally aligned pieces the
// address allows (16 bytes at offset 0 of a 16-byte line; 4 + 8 + 4 at offsets 4 and 12; 8 + 8 at offset 8;
// 2 + 4 + 4 + 4 + 2 at the odd multiples of 2), each piece one coalesced warp-wide access. A partial unit goes
// sample by sample. N = bytes of a full unit (16: 16-bit samples, 8: 8-bit samples), nv = valid samples (1..8).
VFGS_HD void ld_piece16(const uint8_t* p, uint32_t* r)
{
#if defined(__CUDA_ARCH__)
	const uint4 v = *(const uint4*)p; r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
#else
	memcpy(r, p, 16);
#endif
}
VFGS_HD void ld_piece8(const uint8_t* p, uint32_t* r)
{
#if defined(__CUDA_ARCH__)
	const uint2 v = *(const uint2*)p; r[0] = v.x; r[1] = v.y;
#else
	memcpy(r, p, 8);
#endif
}
// (the callers guarantee natural alignment; the host build must not rely on it being exploitable)
VFGS_HD uint32_t ld_piece4(const uint8_t* p)
{
#if defined(__CUDA_ARCH__)
	return *(const uint32_t*)p;
#else
	uint32_t v; memcpy(&v, p, 4); return v;
#endif
}
VFGS_HD uint32_t ld_piece2(const uint8_t* p)
{
#if defined(__CUDA_ARCH__)
	return *(const uint16_t*)p;
#else
	uint16_t v; memcpy(&v, p, 2); return v;
#endif
}
VFGS_HD void st_piece16(uint8_t* p, const uint32_t* w)
{
#if defined(__CUDA_ARCH__)
	*(uint4*)p = make_uint4(w[0], w[1], w[2], w[3]);
#else
	memcpy(p, w, 16);
#endif
}
VFGS_HD void st_piece8(uint8_t* p, uint32_t w0, uint32_t w1)
{
#if defined(__CUDA_ARCH__)
	*(uint2*)p = make_uint2(w0, w1);
#else
	memcpy(p, &w0, 4); memcpy(p + 4, &w1, 4);
#endif
}
VFGS_HD void st_piece4(uint8_t* p, uint32_t w)
{
#if defined(__CUDA_ARCH__)
	*(uint32_t*)p = w;
#else
	memcpy(p, &w, 4);
#endif
}
VFGS_HD void st_piece2(uint8_t* p, uint32_t w)
{
	const uint16_t v = (uint16_t)w;
#if defined(__CUDA_ARCH__)
	*(uint16_t*)p = v;
#else
	memcpy(p, &v, 2);
#endif
}

// The loaded pieces stay as they came until the line is used (edge_fix): combining them at load time would make the
// lane wait for its loads right there instead of LB lines later. r[4] is only touched at the odd multiples of 2.
template <int N>
VFGS_HD void edge_load(const uint8_t* p, uint32_t r[5], int nv)
{
	constexpr int SB = N / 8; // bytes per sample
	if (nv < 8) { // partial last unit of a row, sample by sample; samples right of the picture read as 0 (one lane per row: it may wait)
		r[0] = r[1] = r[2] = r[3] = 0;
#pragma unroll
		for (int e = 0; e < 8; e++) {
			if (e < nv) {
				const uint32_t v = SB == 2 ? ld_piece2(p + 2 * e) : (uint32_t)p[e];
				if (SB == 2) r[e >> 1] |= v << (16 * (e & 1));
				else r[e >> 2] |= v << (8 * (e & 3));
			}
		}
		return;
	}
	const unsigned a = (unsigned)((uintptr_t)p & (N - 1));
	if (N == 16) {
		if (a == 0) ld_piece16(p, r);
		else if (a == 8) { ld_piece8(p, r); ld_piece8(p + 8, r + 2); }
		else if ((a & 3) == 0) { r[0] = ld_piece4(p); ld_piece8(p + 4, r + 1); r[3] = ld_piece4(p + 12); }
		else { r[0] = ld_piece2(p); r[1] = ld_piece4(p + 2); r[2] = ld_piece4(p + 6); r[3] = ld_piece4(p + 10); r[4] = ld_piece2(p + 14); } // odd multiple of 2
	} else {
		if (a == 0) ld_piece8(p, r);
		else if (a == 4) { r[0] = ld_piece4(p); r[1] = ld_piece4(p + 4); }
		else if ((a & 1) == 0) { r[0] = ld_piece2(p); r[1] = ld_piece4(p + 2); r[2] = ld_piece2(p + 6); }
		else { // odd addresses (8-bit samples, odd row pitch): bytes
			r[0] = r[1] = 0;
#pragma unroll
			for (int e = 0; e < 8; e++) r[e >> 2] |= (uint32_t)p[e] << (8 * (e & 3));
		}
	}
}
// pieces -> the unit's words, for a unit loaded from address offset a (p & (N - 1)) with nv valid samples
template <int N>
VFGS_HD void edge_fix(uint32_t r[5], unsigned a, int nv)
{
	if (nv < 8) return;
	if (N == 16) {
		if ((a & 3) == 2) {
			const uint32_t h0 = r[0], m0 = r[1], m1 = r[2], m2 = r[3], h1 = r[4];
			r[0] = h0 | (m0 << 16); r[1] = prmt(m0, m1, 0x5432); r[2] = prmt(m1, m2, 0x5432); r[3] = (m2 >> 16) | (h1 << 16);
		}
	} else if ((a & 3) == 2) {
		const uint32_t h0 = r[0], m = r[1], h1 = r[2];
		r[0] = h0 | (m << 16); r[1] = (m >> 16) | (h1 << 16);
	}
}
template <int N>
VFGS_HD void edge_store(uint8_t* p, const uint32_t w[4], int nv)
{
	constexpr int SB = N / 8;
	if (nv < 8) {
#pragma unroll
		for (int e = 0; e < 8; e++) {
			if (e < nv) {
				if (SB == 2) st_piece2(p + 2 * e, w[e >> 1] >> (16 * (e & 1)));
				else p[e] = (uint8_t)(w[e >> 2] >> (8 * (e & 3)));
			}
		}
		return;
	}
	const unsigned a = (unsigned)((uintptr_t)p & (N - 1));
	if (N == 16) {
		if (a == 0) st_piece16(p, w);
		else if (a == 8) { st_piece8(p, w[0], w[1]); st_piece8(p + 8, w[2], w[3]); }
		else if ((a & 3) == 0) { st_piece4(p, w[0]); st_piece8(p + 4, w[1], w[2]); st_piece4(p + 12, w[3]); }
		else {
			st_piece2(p, w[0]);
			st_piece4(p + 2, prmt(w[0], w[1], 0x5432)); st_piece4(p + 6, prmt(w[1], w[2], 0x5432)); st_piece4(p + 10, prmt(w[2], w[3], 0x5432));
			st_piece2(p + 14, w[3] >> 16);
		}
	} else {
		if (a == 0) st_piece8(p, w[0], w[1]);
		else if (a == 4) { st_piece4(p, w[0]); st_piece4(p + 4, w[1]); }
		else if ((a & 1) == 0) { st_piece2(p, w[0]); st_piece4(p + 2, prmt(w[0], w[1], 0x5432)); st_piece2(p + 6, w[1] >> 16); }
		else {
#pragma unroll
			for (int e = 0; e < 8; e++) p[e] = (uint8_t)(w[e >> 2] >> (8 * (e & 3)));
		}
	}
}

// Per-lane constants of a warp-task (pattern addresses have the block's sign folded in).
// Halo bytes feed the block-edge filter. With 16-sample blocks a lane holds one half of a block and has
// exactly one block edge (its left end if it is the first half, else its right end), so one halo address
// and one filter can serve (MergeHalo): lh. With 8-sample blocks the lane is a whole block and has both.
// Measured on B200 (scripts/ab_sweep.sh, same box): the merged form is +3 points of HBM roofline for the
// issue-bound 8-bit-output kernel and neutral for the HBM-bound 16-bit-output kernel at its CTA size.
#ifndef VFGS_FAST_MERGE_HALO
#define VFGS_FAST_MERGE_HALO 1 // 0 never, 1 always, 2 only with 8-bit output or input (build-time knob for experiments)
#endif
template <bool IN16, bool OUT8> struct MergeHalo { // mode 2: the issue-bound variants (8-bit output, 8-bit input)
	static constexpr bool value = VFGS_FAST_MERGE_HALO == 1 || (VFGS_FAST_MERGE_HALO == 2 && (OUT8 || !IN16));
};
struct FastLane {
	smem_addr_t own;         // the lane's octet, pattern row of line j = 0 of the current block
	smem_addr_t lh, rh;      // halo bytes: last column of block b-1 / first column of block b+1
	smem_addr_t lut;         // this lane's column of the component's LUT (index bits 7..14 are zero)
	int stride;              // pattern row pitch
	bool has_left, has_right;
	uint32_t lo2, hi2;       // clip range replicated in both 16-bit halves
};
// Same addresses for the block-row above, only alive while the overlap lines are processed.
struct FastUp {
	smem_addr_t own, lh, rh;
};

template <int E>
VFGS_HD int blend(int cur, uint32_t u0, uint32_t u1, int w_cur, int w_up) // vfgs_hw.c:225
{
	return (cur * w_cur + octet_byte<E>(u0, u1) * w_up + 16) >> 5;
}

// Scale, add, clip (vfgs_hw.c:239, 260-267) of 8 samples held in two words of four bytes: widened two at a time
// into the 16x2 form of the 16-bit path (no cap needed: v <= 255); LUT index = sample (vfgs_hw.c:211), times 128.
VFGS_HD void scale_add_clip_8bit(smem_addr_t lut, uint32_t lo2, uint32_t hi2, const int g[8], uint32_t raw0, uint32_t raw1,
                                 uint32_t& out0, uint32_t& out1)
{
	uint32_t r[4];
#pragma unroll
	for (int k = 0; k < 4; k++) {
		const uint32_t v2 = prmt(k < 2 ? raw0 : raw1, 0u, (k & 1) ? 0x4342 : 0x4140);
		const int s_lo = (int)lds32(lut | (smem_addr_t)((v2 << 7) & 0x7f80u));
		const int s_hi = (int)lds32(lut | (smem_addr_t)(shr_fma<9>(v2) & 0x7f80u));
		const int a_lo = s_lo * g[2 * k] + 0x8000;
		const int a_hi = s_hi * g[2 * k + 1] + 0x8000;
		const uint32_t d2 = prmt((uint32_t)a_lo, (uint32_t)a_hi, 0x7632);
		r[k] = min_s16x2(add_max_s16x2(v2, d2, lo2), hi2);
	}
	out0 = prmt(r[0], r[1], 0x6420);
	out1 = prmt(r[2], r[3], 0x6420);
}

// Scale, add, clip of 8 samples held in four words of two 10-bit samples (vfgs_hw.c:239, 260-267) and the optional
// 10 -> 8 bit conversion (yuv.c:231). The LUT holds scale * 2^(16 - shift), so the rounded quotient of vfgs_hw.c:263 is
// exactly the upper half-word of lut * grain + 0x8000. 8-bit output ((x + 2) >> 2): the + 2 rides on the rounding
// constant and on the clip range (the callers pass lo + 2, hi + 2): clip(v + d, lo, hi) + 2 == clip(v + d + 2, lo + 2, hi + 2).
// outw: 4 words (16-bit output) or 2 (8-bit).
#ifndef VFGS_OUT8_MUL64
#define VFGS_OUT8_MUL64 1 // 10 -> 8: the >> 2 as a multiply (FMA pipe), +1 point with the PRMT top byte (profiles/r02_wide16_ab.md, trips 4-5)
#endif
template <bool OUT8>
VFGS_HD void scale_add_clip_16bit(smem_addr_t lut, uint32_t lo2, uint32_t hi2, const int g[8], const uint32_t raw[4], uint32_t* outw)
{
	constexpr int kRound = OUT8 ? 0x28000 : 0x8000;
	uint32_t r[4];
#pragma unroll
	for (int k = 0; k < 4; k++) {
		// LUT index = (sample >> 2) & 0xff (vfgs_hw.c:211), times the 128-byte LUT row pitch
		const int s_lo = (int)lds32(lut | (smem_addr_t)((raw[k] << 5) & 0x7f80u));
		const int s_hi = (int)lds32(lut | (smem_addr_t)(shr_fma<11>(raw[k]) & 0x7f80u));
		const int a_lo = s_lo * g[2 * k] + kRound;
		const int a_hi = s_hi * g[2 * k + 1] + kRound;
		const uint32_t d2 = prmt((uint32_t)a_lo, (uint32_t)a_hi, 0x7632);
		// samples above 0x3fff clip to the ceiling whatever the grain: cap them so the signed 16-bit add cannot wrap
		const uint32_t v2 = min_u16x2(raw[k], 0x3fff3fffu);
		r[k] = min_s16x2(add_max_s16x2(v2, d2, lo2), hi2);  // vfgs_hw.c:265
	}
	if (OUT8) {
		if (VFGS_OUT8_MUL64) {
			// (x >> 2) & 0xff is byte 1 of x * 64 (FMA pipe instead of ALU); x <= hi + 2 <= (255 << 2) + 2 (the clip
			// ceiling, vfgs_hw.c:364-380), so x * 64 stays inside its half-word
#pragma unroll
			for (int k = 0; k < 4; k++) r[k] *= 64u;
			outw[0] = prmt(r[0], r[1], 0x7531);
			outw[1] = prmt(r[2], r[3], 0x7531);
		} else {
#pragma unroll
			for (int k = 0; k < 4; k++) r[k] >>= 2; // bits leaking across the half-words land in bytes 1 and 3, which are dropped
			outw[0] = prmt(r[0], r[1], 0x6420);
			outw[1] = prmt(r[2], r[3], 0x6420);
		}
	} else {
		outw[0] = r[0]; outw[1] = r[1]; outw[2] = r[2]; outw[3] = r[3];
	}
}

// One line of one lane. raw: the lane's 8 samples as loaded (IN16: 4 words of two 10-bit samples,
// else 2 words of four bytes). outw: result words ready to store (16-bit out: 4 words, 8-bit: 2).
// rc: byte offset of this line's row inside the current block's window; w_cur != 0 selects the
// vertical-overlap blend with row offset ru of the upper block's window.
template <bool IN16, bool OUT8, int NSH>
VFGS_HD void fast_line(const FastLane& L, int rc, int w_cur, int w_up, const FastUp& U, int ru,
                       const uint32_t raw[4], uint32_t outw[4])
{
	uint32_t c0, c1;
	octet(L.own + rc, c0, c1);
	int g[8];
	constexpr bool kFmaTop = VFGS_OCTET_TOP_ON_FMA && (OUT8 || !IN16);
	g[0] = octet_byte<0>(c0, c1); g[1] = octet_byte<1>(c0, c1); g[2] = octet_byte<2>(c0, c1); g[3] = octet_byte<3, kFmaTop>(c0, c1);
	g[4] = octet_byte<4>(c0, c1); g[5] = octet_byte<5>(c0, c1); g[6] = octet_byte<6>(c0, c1); g[7] = octet_byte<7, kFmaTop>(c0, c1);
	if (MergeHalo<IN16, OUT8>::value && NSH == 4) {
		// one edge per lane: halo h next to a, then b (left edge: h | g0 g1, right edge: g6 g7 | h mirrored)
		const bool edge = L.has_left || L.has_right;
		int h = edge ? lds_s8(L.lh + rc) : 0;
		if (w_cur) { // vertical overlap with the block-row above (vfgs_hw.c:173-188, 223-229)
			uint32_t u0, u1;
			octet(U.own + ru, u0, u1);
			g[0] = blend<0>(g[0], u0, u1, w_cur, w_up); g[1] = blend<1>(g[1], u0, u1, w_cur, w_up);
			g[2] = blend<2>(g[2], u0, u1, w_cur, w_up); g[3] = blend<3>(g[3], u0, u1, w_cur, w_up);
			g[4] = blend<4>(g[4], u0, u1, w_cur, w_up); g[5] = blend<5>(g[5], u0, u1, w_cur, w_up);
			g[6] = blend<6>(g[6], u0, u1, w_cur, w_up); g[7] = blend<7>(g[7], u0, u1, w_cur, w_up);
			if (edge) h = (h * w_cur + lds_s8(U.lh + ru) * w_up + 16) >> 5;
		}
		// block-edge filter (vfgs_hw.c:250-259), taps read unfiltered grain
		const int a = L.has_right ? g[7] : g[0], b = L.has_right ? g[6] : g[1];
		const int f = (h + 3 * a + b + 2) >> 2;
		g[0] = L.has_left ? f : g[0];
		g[7] = L.has_right ? f : g[7];
	} else {
		int hl = L.has_left ? lds_s8(L.lh + rc) : 0;
		int hr = L.has_right ? lds_s8(L.rh + rc) : 0;
		if (w_cur) {
			uint32_t u0, u1;
			octet(U.own + ru, u0, u1);
			g[0] = blend<0>(g[0], u0, u1, w_cur, w_up); g[1] = blend<1>(g[1], u0, u1, w_cur, w_up);
			g[2] = blend<2>(g[2], u0, u1, w_cur, w_up); g[3] = blend<3>(g[3], u0, u1, w_cur, w_up);
			g[4] = blend<4>(g[4], u0, u1, w_cur, w_up); g[5] = blend<5>(g[5], u0, u1, w_cur, w_up);
			g[6] = blend<6>(g[6], u0, u1, w_cur, w_up); g[7] = blend<7>(g[7], u0, u1, w_cur, w_up);
			if (L.has_left) hl = (hl * w_cur + lds_s8(U.lh + ru) * w_up + 16) >> 5;
			if (L.has_right) hr = (hr * w_cur + lds_s8(U.rh + ru) * w_up + 16) >> 5;
		}
		const int f0 = (hl + 3 * g[0] + g[1] + 2) >> 2;
		const int f7 = (g[6] + 3 * g[7] + hr + 2) >> 2;
		g[0] = L.has_left ? f0 : g[0];
		g[7] = L.has_right ? f7 : g[7];
	}

	if (IN16) {
		scale_add_clip_16bit<OUT8>(L.lut, L.lo2, L.hi2, g, raw, outw);
	} else {
		scale_add_clip_8bit(L.lut, L.lo2, L.hi2, g, raw[0], raw[1], outw[0], outw[1]);
	}
}

// Column-shifted copies of a pattern in the fast image: the window column ox is a multiple of 4 for
// 16-sample blocks (copies shifted by 0 and 4 bytes) and of 2 for 8-sample blocks (0, 2, 4, 6).
VFGS_HD int fast_copies(int block_samples) { return block_samples == 16 ? 2 : 4; }

// Per-component constants of the window-offset computation (host-made, make_woff_params).
struct WoffComp {
	int off0, doff;   // offset of the +pattern copies; -pattern copies minus +pattern copies (gather format: 0, 0x8000)
	int ystride;      // bytes per row step: stepy * row pitch
	int copy;         // bytes between column-shifted copies (0 in the gather format)
	int kmask, kshift; // copy index = qx & kmask, aligned column = (qx >> kshift) * xmul
	int xmul;
};

// Byte offset, inside the component's image, of a block's pattern window. The ten-bit fields of the register
// (vfgs_hw.c:99-138; decode_offsets) are moved to the top of a word, so that field * 13 >> 10 (column bin qx, 0..12)
// and field * 12 >> 10 (row bin qy, 0..11) are one multiply-high each; U's row field wraps around the word.
//   fast format    +pattern or -pattern copies according to the block's sign, among them the copy in which the
//                  window column (qx * 4 or qx * 2) sits on an 8-byte boundary, row qy * step, column rounded down to 8
//   gather format  qy * step * pitch + qx * step, bit 15 set when the block's sign is negative
// Precomputed per block by lfsr_states_kernel (FgsParams::woffs), so a lane only adds its column and the line's row pitch.
template <int C>
VFGS_HD uint32_t window_offset(uint32_t s, const WoffComp& w)
{
	constexpr uint32_t kTop = 0xffc00000u; // the bits below a field must not carry into the product
	const uint32_t xtop = C == 0 ? s << 22 : C == 1 ? (s << 12) & kTop : (s << 2) & kTop;
	const uint32_t ytop = C == 0 ? (s << 8) & kTop : C == 1 ? ((s << 30) | ((s >> 2) & 0x3fc00000u)) : (s << 18) & kTop;
	const uint32_t sign = C == 0 ? s >> 31 : C == 1 ? (s >> 2) & 1u : (s >> 15) & 1u;
	const uint32_t qx = mulhi_u32(xtop, 13u), qy = mulhi_u32(ytop, 12u);
	return (uint32_t)w.off0 + sign * (uint32_t)w.doff + qy * (uint32_t)w.ystride + (qx & (uint32_t)w.kmask) * (uint32_t)w.copy +
	       (qx >> w.kshift) * (uint32_t)w.xmul;
}

#ifndef VFGS_FAST_LB
#define VFGS_FAST_LB 4
#endif
constexpr int kFastLB = VFGS_FAST_LB; // lines in flight per lane (build-time knob for experiments)
#ifndef VFGS_FAST_PREFETCH16
#define VFGS_FAST_PREFETCH16 4 // lines ahead of the line loads prefetched into L1, 16-bit output: 1080p 0.867 -> 0.911, 4K 0.893 -> 0.918 of the HBM peak (profiles/r02_fast_prefetch_ab.md); 8 lines: no better
#endif
#ifndef VFGS_FAST_PREFETCH8
#define VFGS_FAST_PREFETCH8 0  // same, 8-bit output: the issue-bound variant loses with it (0.786 -> 0.743)
#endif
static_assert(kFastLB >= 2, "both vertical-overlap lines of a block-row must fall into the first group of lines");
#ifndef VFGS_FAST_LB16
#define VFGS_FAST_LB16 VFGS_FAST_LB // fast kernel, 16-bit (or 8-bit in, 8-bit out) stores
#endif
#ifndef VFGS_FAST_LB8
#define VFGS_FAST_LB8 VFGS_FAST_LB  // fast kernel, 16-bit in, 8-bit out
#endif
#ifndef VFGS_NARROW16_LB
#define VFGS_NARROW16_LB VFGS_FAST_LB16 // 16-bit in and out, 8 samples per lane (widths that are not a multiple of 16 samples)
#endif

// EDGE: rows at any sample-aligned address, partial last unit of a row (see edge_load / edge_store above)
template <bool IN16, bool OUT8, int NSH, bool EDGE = false>
VFGS_HD void fast_task_body(const FgsParams& p, smem_addr_t lut, const TaskGeom& t, int k0, int lane)
{
	const int c = t.c;
	const smem_addr_t img = lut + (smem_addr_t)(ptrdiff_t)p.fimg_off[c]; // the component's pattern image
	const Plane& pl = p.comp[c];
	const int ysh = (c && p.suby > 1) ? 1 : 0;
	constexpr int n = 1 << NSH;
	constexpr int LB = OUT8 ? VFGS_FAST_LB8 : IN16 ? VFGS_NARROW16_LB : VFGS_FAST_LB16; // lines in flight per lane

	// component lines of this stripe (whole stripes only: the host sends partial line ranges to
	// the general kernel)
	const int cl0 = (t.r * 16) >> ysh;
	int cl1 = cl0 + (16 >> ysh);
	if (cl1 > pl.lines) cl1 = pl.lines;
	const int nl = cl1 - cl0;
	if (nl <= 0) return;

	constexpr int IB = IN16 ? 2 : 1, OB = (IN16 && !OUT8) ? 2 : 1;
	constexpr int PF = OUT8 ? VFGS_FAST_PREFETCH8 : VFGS_FAST_PREFETCH16;            // lines prefetched ahead of the line loads
	constexpr bool kL1 = VFGS_FAST_L1_MODE == 2 || (VFGS_FAST_L1_MODE == 1 && !OUT8) || PF > 0; // sample loads allocate in L1
	const long long in_pitch = pl.in_row_bytes, out_pitch = pl.out_row_bytes;
	const uint8_t* src = pl.in + (long long)t.f * p.in_frame_bytes + (long long)cl0 * in_pitch + (long long)k0 * IB;
	uint8_t* dst = pl.out + (long long)t.f * p.out_frame_bytes + (long long)cl0 * out_pitch + (long long)k0 * OB;

	// The first LB lines are requested before anything else: the block decode below runs
	// while they are in flight. A stripe shorter than LB lines re-reads its last line.
	const int nv = EDGE ? (pl.width - k0 < kSamplesPerLane ? pl.width - k0 : kSamplesPerLane) : kSamplesPerLane; // valid samples of this unit
	uint32_t raw[LB][EDGE ? 5 : 4];
#pragma unroll
	for (int q = 0; q < LB; q++) {
		const int qq = q < nl ? q : nl - 1;
		if (EDGE) edge_load<IN16 ? 16 : 8>(src + qq * in_pitch, raw[q], nv);
		else if (IN16) ld_samples_16<kL1>(src + qq * in_pitch, raw[q]);
		else ld_global_8(src + qq * in_pitch, raw[q]);
	}

	if (IN16 && PF > 0) {
#pragma unroll
		for (int q = LB; q < LB + PF; q++) prefetch_l1(src + q * in_pitch, q < nl);
	}

	const int b = k0 >> NSH;
	const int i0 = k0 & (n - 1);
	FastLane L;
	L.has_left = (i0 == 0) && (b > 0);
	L.has_right = (i0 + kSamplesPerLane == n) && (b + 1 < p.nb);
	L.stride = p.fpat_stride[c];
	L.lut = lut + (smem_addr_t)(c * kLutBytes + lane * 4);
	constexpr int kOutBias = (IN16 && OUT8) ? 2 : 0; // see fast_line
	L.lo2 = (uint32_t)(p.lo[c] + kOutBias) * 0x00010001u; L.hi2 = (uint32_t)(p.hi[c] + kOutBias) * 0x00010001u;

	const int srow = t.r - p.stream_row0;
	const uint16_t* w_cur = p.woffs + (((long long)t.f * p.stream_rows + srow) * p.spitch + 1 + b) * 4 + c;
	L.own = img + (smem_addr_t)(w_cur[0] + i0);
	L.lh = L.rh = L.own;
	if (L.has_left) L.lh = img + (smem_addr_t)(w_cur[-4] + n - 1);
	if (L.has_right) (MergeHalo<IN16, OUT8>::value && NSH == 4 ? L.lh : L.rh) = img + (smem_addr_t)w_cur[4];

	// the first lines of a stripe overlap the block-row above (never in the first stripe, y <= 15)
	FastUp U;
	U.own = U.lh = U.rh = L.own;
	bool ovl = t.r > 0;
	if (ovl) {
		const uint16_t* w_up = w_cur - p.spitch * 4;
		U.own = img + (smem_addr_t)(w_up[0] + i0);
		if (L.has_left) U.lh = img + (smem_addr_t)(w_up[-4] + n - 1);
		if (L.has_right) (MergeHalo<IN16, OUT8>::value && NSH == 4 ? U.lh : U.rh) = img + (smem_addr_t)w_up[4];
	}

	int rc = 0;
	const uint8_t* nxt = src + LB * in_pitch; // line whose load refills the slot just consumed
	// WHOLE: the stripe is a whole number of LB-line groups (every stripe of a picture whose height is a
	// multiple of LB component lines): no per-line store predicate, one refill predicate per group.
	auto lines = [&](auto whole_tag) {
		constexpr bool WHOLE = decltype(whole_tag)::value;
#pragma unroll 1
		for (int base = 0; base < nl; base += LB) {
			const bool more = base + LB < nl;
#pragma unroll
			for (int q = 0; q < LB; q++) {
				const int line = base + q;
				uint32_t w[4];
				int w_cur = 0, w_up = 0, ru = 0;
				if (q == 0 && ovl) { w_cur = ysh ? 20 : 12; w_up = ysh ? 20 : 24; ru = (16 >> ysh) * L.stride; }
				if (q == 1 && ovl && !ysh) { w_cur = 24; w_up = 12; ru = 17 * L.stride; }
				if (EDGE) edge_fix<IN16 ? 16 : 8>(raw[q], (unsigned)((uintptr_t)(nxt - LB * in_pitch) & (IN16 ? 15 : 7)), nv);
				fast_line<IN16, OUT8, NSH>(L, rc, w_cur, w_up, U, ru, raw[q], w);
				// this slot's registers are free again: request the line LB further down
				const bool refill = WHOLE ? more : line + LB < nl;
				if (EDGE) { if (refill) edge_load<IN16 ? 16 : 8>(nxt, raw[q], nv); }
				else if (IN16) ld_samples_16_if<kL1>(nxt, raw[q], refill);
				else ld_global_8_if(nxt, raw[q], refill);
				if (IN16 && PF > 0) prefetch_l1(nxt + PF * in_pitch, line + LB + PF < nl);
				if (WHOLE || line < nl) {
					if (EDGE) edge_store<OB == 2 ? 16 : 8>(dst, w, nv);
					else if (OB == 2) st_global_16(dst, w);
					else st_global_8(dst, w);
				}
				rc += L.stride; nxt += in_pitch; dst += out_pitch;
			}
			ovl = false;
		}
	};
	if (nl % LB == 0) lines(std::true_type());
	else lines(std::false_type());
}

// ---- 16 samples per lane ---------------------------------------------------------------------
// A lane that owns a whole 16-sample block (or two 8-sample blocks) spreads the per-line work that does not depend on
// the sample count (addresses, loop control, halo loads, edge filters without left/right selection) and the per-task
// set-up over twice the samples. With 8-bit samples that is one 128-bit access per line; with 16-bit samples one
// 256-bit access (LDG.256 / STG.256, sm_100), 128-bit for the 8-bit output of the fused 10 -> 8 conversion. Taken when
// the component's width is a multiple of 16 and its rows are aligned to the access size (plan_launches, FgsParams::fwide).
// (Round 2, measured under the sustained protocol: profiles/r02_wide16_ab.md.)
// P010 samples (value in bits 15..6 of a uint16) to and from the LSB-aligned form of the arithmetic, two per word. The low
// six bits of the input are ignored; after the clip a value is at most 1020, so the shift back up cannot carry across the halves.
template <int N>
VFGS_HD void msb_to_lsb(const uint32_t* raw, uint32_t* out)
{
#pragma unroll
	for (int k = 0; k < N; k++) out[k] = (raw[k] >> 6) & 0x03ff03ffu;
}
template <int N>
VFGS_HD void lsb_to_msb(uint32_t* w)
{
#pragma unroll
	for (int k = 0; k < N; k++) w[k] <<= 6;
}

struct WideLane {
	smem_addr_t own0, own1;  // pattern rows of line j = 0: samples 0..7 and 8..15 (two blocks when the block size is 8)
	smem_addr_t lh, rh;      // halo bytes: last column of the block to the left / first column of the block to the right
	smem_addr_t lut;
	int stride;
	bool has_left, has_right;
	uint32_t lo2, hi2;
};
struct WideUp {
	smem_addr_t own0, own1, lh, rh;
};

VFGS_HD void octet_to_ints(uint32_t w0, uint32_t w1, int g[8])
{
	g[0] = octet_byte<0>(w0, w1); g[1] = octet_byte<1>(w0, w1); g[2] = octet_byte<2>(w0, w1); g[3] = octet_byte<3, VFGS_OCTET_TOP_ON_FMA != 0>(w0, w1);
	g[4] = octet_byte<4>(w0, w1); g[5] = octet_byte<5>(w0, w1); g[6] = octet_byte<6>(w0, w1); g[7] = octet_byte<7, VFGS_OCTET_TOP_ON_FMA != 0>(w0, w1);
}
VFGS_HD void blend_octet(int g[8], uint32_t u0, uint32_t u1, int w_cur, int w_up)
{
	g[0] = blend<0>(g[0], u0, u1, w_cur, w_up); g[1] = blend<1>(g[1], u0, u1, w_cur, w_up);
	g[2] = blend<2>(g[2], u0, u1, w_cur, w_up); g[3] = blend<3>(g[3], u0, u1, w_cur, w_up);
	g[4] = blend<4>(g[4], u0, u1, w_cur, w_up); g[5] = blend<5>(g[5], u0, u1, w_cur, w_up);
	g[6] = blend<6>(g[6], u0, u1, w_cur, w_up); g[7] = blend<7>(g[7], u0, u1, w_cur, w_up);
}
// One line of one wide lane: 16 samples in raw (8-bit: four words of four bytes, 16-bit: eight words of two samples),
// result in outw (four words of 8-bit samples or eight of 16-bit samples).
// MSB: 16-bit samples hold the value in bits 15..6 (P010 luma): shifted down here, the caller shifts the result back up.
template <bool IN16, bool OUT8, int NSH, bool MSB = false>
VFGS_HD void wide_line(const WideLane& L, int rc, int w_cur, int w_up, const WideUp& U, int ru,
                       const uint32_t* raw, uint32_t* outw)
{
	uint32_t a0, a1, b0, b1;
	octet(L.own0 + rc, a0, a1);
	octet(L.own1 + rc, b0, b1);
	int ga[8], gb[8];
	octet_to_ints(a0, a1, ga);
	octet_to_ints(b0, b1, gb);
	int hl = L.has_left ? lds_s8(L.lh + rc) : 0;
	int hr = L.has_right ? lds_s8(L.rh + rc) : 0;
	if (w_cur) { // vertical overlap with the block-row above (vfgs_hw.c:173-188, 223-229)
		uint32_t u0, u1;
		octet(U.own0 + ru, u0, u1);
		blend_octet(ga, u0, u1, w_cur, w_up);
		octet(U.own1 + ru, u0, u1);
		blend_octet(gb, u0, u1, w_cur, w_up);
		if (L.has_left) hl = (hl * w_cur + lds_s8(U.lh + ru) * w_up + 16) >> 5;
		if (L.has_right) hr = (hr * w_cur + lds_s8(U.rh + ru) * w_up + 16) >> 5;
	}
	// block-edge filters (vfgs_hw.c:250-259), taps read unfiltered grain
	const int f0 = (hl + 3 * ga[0] + ga[1] + 2) >> 2;
	const int f15 = (gb[6] + 3 * gb[7] + hr + 2) >> 2;
	if (NSH == 3) { // the lane holds two 8-sample blocks: the edge between them is lane-internal
		const int f7 = (ga[6] + 3 * ga[7] + gb[0] + 2) >> 2;
		const int f8 = (ga[7] + 3 * gb[0] + gb[1] + 2) >> 2;
		ga[7] = f7; gb[0] = f8;
	}
	ga[0] = L.has_left ? f0 : ga[0];
	gb[7] = L.has_right ? f15 : gb[7];
	if (IN16) {
		uint32_t cv[8];
		if (MSB) msb_to_lsb<8>(raw, cv);
		const uint32_t* r = MSB ? cv : raw;
		scale_add_clip_16bit<OUT8>(L.lut, L.lo2, L.hi2, ga, r, outw);
		scale_add_clip_16bit<OUT8>(L.lut, L.lo2, L.hi2, gb, r + 4, outw + (OUT8 ? 2 : 4));
	} else {
		scale_add_clip_8bit(L.lut, L.lo2, L.hi2, ga, raw[0], raw[1], outw[0], outw[1]);
		scale_add_clip_8bit(L.lut, L.lo2, L.hi2, gb, raw[2], raw[3], outw[2], outw[3]);
	}
}

// Lines in flight per lane of the wide 16-bit path (32 bytes each), measured with the CTA sizes of vfgs_kernels.cuh
// (profiles/r02_wide16_ab.md): odd counts lose 4-10 points (a stripe's 16 lines are then not a whole number of groups).
#ifndef VFGS_WIDE16_LB
#define VFGS_WIDE16_LB 2   // 16-bit output, kernel shared with 8-samples-per-lane components (768 threads)
#endif
#ifndef VFGS_WIDE16_LBW
#define VFGS_WIDE16_LBW 4  // 16-bit output, every component wide (ALLWIDE variant: 512 threads, 128 registers)
#endif
#ifndef VFGS_WIDE16_LB8
#define VFGS_WIDE16_LB8 2  // 8-bit output (768 threads)
#endif
template <bool IN16, bool OUT8, int NSH, bool ALLWIDE = false, bool MSB = false>
VFGS_HD void wide_task_body(const FgsParams& p, smem_addr_t lut, const TaskGeom& t, int k0, int lane)
{
	const int c = t.c;
	const smem_addr_t img = lut + (smem_addr_t)(ptrdiff_t)p.fimg_off[c];
	const Plane& pl = p.comp[c];
	const int ysh = (c && p.suby > 1) ? 1 : 0;
	constexpr int n = 1 << NSH;
	constexpr int LB = !IN16 ? VFGS_FAST_LB16 : OUT8 ? VFGS_WIDE16_LB8 : ALLWIDE ? VFGS_WIDE16_LBW : VFGS_WIDE16_LB;
	static_assert(LB >= 2, "both vertical-overlap lines of a block-row must fall into the first group of lines");
	constexpr int IB = IN16 ? 2 : 1, OB = (IN16 && !OUT8) ? 2 : 1;
	constexpr int RW = IN16 ? 8 : 4, OW = OB == 2 ? 8 : 4; // words per line: loaded, stored

	const int cl0 = (t.r * 16) >> ysh;
	int cl1 = cl0 + (16 >> ysh);
	if (cl1 > pl.lines) cl1 = pl.lines;
	const int nl = cl1 - cl0;
	if (nl <= 0) return;

	const long long in_pitch = pl.in_row_bytes, out_pitch = pl.out_row_bytes;
	const uint8_t* src = pl.in + (long long)t.f * p.in_frame_bytes + (long long)cl0 * in_pitch + (long long)k0 * IB;
	uint8_t* dst = pl.out + (long long)t.f * p.out_frame_bytes + (long long)cl0 * out_pitch + (long long)k0 * OB;

	uint32_t raw[LB][RW];
#pragma unroll
	for (int q = 0; q < LB; q++) {
		if (IN16) ld_global_32(src + (q < nl ? q : nl - 1) * in_pitch, raw[q]);
		else ld_global_16(src + (q < nl ? q : nl - 1) * in_pitch, raw[q]);
	}

	// first and last block of the lane (the same one with 16-sample blocks)
	const int b0 = k0 >> NSH, b1 = (k0 + 15) >> NSH;
	WideLane L;
	L.has_left = b0 > 0;
	L.has_right = b1 + 1 < p.nb;
	L.stride = p.fpat_stride[c];
	L.lut = lut + (smem_addr_t)(c * kLutBytes + lane * 4);
	constexpr int kOutBias = (IN16 && OUT8) ? 2 : 0; // see scale_add_clip_16bit
	L.lo2 = (uint32_t)(p.lo[c] + kOutBias) * 0x00010001u; L.hi2 = (uint32_t)(p.hi[c] + kOutBias) * 0x00010001u;

	const int srow = t.r - p.stream_row0;
	const uint16_t* w_cur = p.woffs + (((long long)t.f * p.stream_rows + srow) * p.spitch + 1 + b0) * 4 + c;
	auto windows = [&](const uint16_t* w, smem_addr_t& own0, smem_addr_t& own1, smem_addr_t& lh, smem_addr_t& rh) {
		own0 = img + (smem_addr_t)w[0];
		own1 = NSH == 4 ? own0 + 8 : img + (smem_addr_t)w[4];
		lh = rh = own0;
		if (L.has_left) lh = img + (smem_addr_t)(w[-4] + n - 1);
		if (L.has_right) rh = img + (smem_addr_t)w[NSH == 4 ? 4 : 8];
	};
	windows(w_cur, L.own0, L.own1, L.lh, L.rh);
	WideUp U;
	U.own0 = U.own1 = U.lh = U.rh = L.own0;
	bool ovl = t.r > 0;
	if (ovl) windows(w_cur - p.spitch * 4, U.own0, U.own1, U.lh, U.rh);

	int rc = 0;
	const uint8_t* nxt = src + LB * in_pitch;
#pragma unroll 1
	for (int base = 0; base < nl; base += LB) {
#pragma unroll
		for (int q = 0; q < LB; q++) {
			const int line = base + q;
			uint32_t w[OW];
			int wc = 0, wu = 0, ru = 0;
			if (q == 0 && ovl) { wc = ysh ? 20 : 12; wu = ysh ? 20 : 24; ru = (16 >> ysh) * L.stride; }
			if (q == 1 && ovl && !ysh) { wc = 24; wu = 12; ru = 17 * L.stride; }
			wide_line<IN16, OUT8, NSH, MSB>(L, rc, wc, wu, U, ru, raw[q], w);
			if (MSB && OB == 2) lsb_to_msb<OW>(w);
			if (IN16) ld_global_32_if(nxt, raw[q], line + LB < nl);
			else ld_global_16_if(nxt, raw[q], line + LB < nl);
			if (line < nl) {
				if (OB == 2) st_global_32(dst, w);
				else st_global_16(dst, w);
			}
			rc += L.stride; nxt += in_pitch; dst += out_pitch;
		}
		ovl = false;
	}
}

// ---- interleaved chroma (semi-planar frames) -------------------------------------------------------
// A UV line holds U0 V0 U1 V1 ...; with 4:2:0 / 4:2:2 a chroma block is 8 samples, so 16 consecutive samples of the line
// are one block of U and the same block of V. A lane unit is that pair: one 256-bit access per line for 16-bit samples
// (128-bit for 8-bit samples and for the 8-bit output of the fused 10 -> 8 conversion), two pattern octets (U's window
// from component 1's entry of the block, V's from component 2's), four halo bytes, and no lane-internal edge. Every packed
// 16-bit pair of the arithmetic is (U_k, V_k): U's LUT serves the low half, V's the high half, and the S16x2 add and clip
// run unchanged because U and V share the clip range.
template <bool OUT8>
VFGS_HD void scale_add_clip_uv_16bit(smem_addr_t lut_u, smem_addr_t lut_v, uint32_t lo2, uint32_t hi2, const int* gu, const int* gv,
                                     const uint32_t raw[4], uint32_t* outw)
{
	constexpr int kRound = OUT8 ? 0x28000 : 0x8000; // see scale_add_clip_16bit
	uint32_t r[4];
#pragma unroll
	for (int k = 0; k < 4; k++) {
		const int s_lo = (int)lds32(lut_u | (smem_addr_t)((raw[k] << 5) & 0x7f80u));
		const int s_hi = (int)lds32(lut_v | (smem_addr_t)(shr_fma<11>(raw[k]) & 0x7f80u));
		const int a_lo = s_lo * gu[k] + kRound;
		const int a_hi = s_hi * gv[k] + kRound;
		const uint32_t d2 = prmt((uint32_t)a_lo, (uint32_t)a_hi, 0x7632);
		const uint32_t v2 = min_u16x2(raw[k], 0x3fff3fffu);
		r[k] = min_s16x2(add_max_s16x2(v2, d2, lo2), hi2);
	}
	if (OUT8) {
#pragma unroll
		for (int k = 0; k < 4; k++) r[k] *= 64u;
		outw[0] = prmt(r[0], r[1], 0x7531);
		outw[1] = prmt(r[2], r[3], 0x7531);
	} else {
		outw[0] = r[0]; outw[1] = r[1]; outw[2] = r[2]; outw[3] = r[3];
	}
}
VFGS_HD void scale_add_clip_uv_8bit(smem_addr_t lut_u, smem_addr_t lut_v, uint32_t lo2, uint32_t hi2, const int* gu, const int* gv,
                                    uint32_t raw0, uint32_t raw1, uint32_t& out0, uint32_t& out1)
{
	uint32_t r[4];
#pragma unroll
	for (int k = 0; k < 4; k++) {
		const uint32_t v2 = prmt(k < 2 ? raw0 : raw1, 0u, (k & 1) ? 0x4342 : 0x4140);
		const int s_lo = (int)lds32(lut_u | (smem_addr_t)((v2 << 7) & 0x7f80u));
		const int s_hi = (int)lds32(lut_v | (smem_addr_t)(shr_fma<9>(v2) & 0x7f80u));
		const int a_lo = s_lo * gu[k] + 0x8000;
		const int a_hi = s_hi * gv[k] + 0x8000;
		const uint32_t d2 = prmt((uint32_t)a_lo, (uint32_t)a_hi, 0x7632);
		r[k] = min_s16x2(add_max_s16x2(v2, d2, lo2), hi2);
	}
	out0 = prmt(r[0], r[1], 0x6420);
	out1 = prmt(r[2], r[3], 0x6420);
}

struct UvLane {
	smem_addr_t own_u, own_v;              // pattern rows of line j = 0 of the block's U and V windows
	smem_addr_t lh_u, rh_u, lh_v, rh_v;    // halo bytes: last column of the block to the left / first of the block to the right
	smem_addr_t lut_u, lut_v;
	int stride;
	bool has_left, has_right;
	uint32_t lo2, hi2;
};
struct UvUp {
	smem_addr_t own_u, own_v, lh_u, rh_u, lh_v, rh_v;
};

// One grain octet of an 8-sample block: vertical overlap and both block-edge filters (vfgs_hw.c:223-229, 250-259).
VFGS_HD void block_octet(smem_addr_t own, smem_addr_t lh, smem_addr_t rh, smem_addr_t up_own, smem_addr_t up_lh, smem_addr_t up_rh,
                         bool has_left, bool has_right, int rc, int w_cur, int w_up, int ru, int g[8])
{
	uint32_t a0, a1;
	octet(own + rc, a0, a1);
	octet_to_ints(a0, a1, g);
	int hl = has_left ? lds_s8(lh + rc) : 0;
	int hr = has_right ? lds_s8(rh + rc) : 0;
	if (w_cur) {
		uint32_t u0, u1;
		octet(up_own + ru, u0, u1);
		blend_octet(g, u0, u1, w_cur, w_up);
		if (has_left) hl = (hl * w_cur + lds_s8(up_lh + ru) * w_up + 16) >> 5;
		if (has_right) hr = (hr * w_cur + lds_s8(up_rh + ru) * w_up + 16) >> 5;
	}
	const int f0 = (hl + 3 * g[0] + g[1] + 2) >> 2;
	const int f7 = (g[6] + 3 * g[7] + hr + 2) >> 2;
	g[0] = has_left ? f0 : g[0];
	g[7] = has_right ? f7 : g[7];
}

// One line of one interleaved-chroma lane. raw: 16 samples U0 V0 .. U7 V7 as loaded (16-bit: eight words, P010 when IN16;
// 8-bit: four words); outw: the same layout at the output depth.
template <bool IN16, bool OUT8>
VFGS_HD void uv_line(const UvLane& L, int rc, int w_cur, int w_up, const UvUp& U, int ru, const uint32_t* raw, uint32_t* outw)
{
	int gu[8], gv[8];
	block_octet(L.own_u, L.lh_u, L.rh_u, U.own_u, U.lh_u, U.rh_u, L.has_left, L.has_right, rc, w_cur, w_up, ru, gu);
	block_octet(L.own_v, L.lh_v, L.rh_v, U.own_v, U.lh_v, U.rh_v, L.has_left, L.has_right, rc, w_cur, w_up, ru, gv);
	if (IN16) {
		uint32_t cv[8];
		msb_to_lsb<8>(raw, cv);
		scale_add_clip_uv_16bit<OUT8>(L.lut_u, L.lut_v, L.lo2, L.hi2, gu, gv, cv, outw);
		scale_add_clip_uv_16bit<OUT8>(L.lut_u, L.lut_v, L.lo2, L.hi2, gu + 4, gv + 4, cv + 4, outw + (OUT8 ? 2 : 4));
	} else {
		scale_add_clip_uv_8bit(L.lut_u, L.lut_v, L.lo2, L.hi2, gu, gv, raw[0], raw[1], outw[0], outw[1]);
		scale_add_clip_uv_8bit(L.lut_u, L.lut_v, L.lo2, L.hi2, gu + 4, gv + 4, raw[2], raw[3], outw[2], outw[3]);
	}
}

// k0: first chroma sample (of U and of V) of the lane; the block is k0 / 8. Same line pipeline as wide_task_body.
template <bool IN16, bool OUT8, bool ALLWIDE = false>
VFGS_HD void uv_task_body(const FgsParams& p, smem_addr_t lut, const TaskGeom& t, int k0, int lane)
{
	const Plane& pl = p.comp[1];
	const int ysh = p.suby > 1 ? 1 : 0;
	constexpr int LB = !IN16 ? VFGS_FAST_LB16 : OUT8 ? VFGS_WIDE16_LB8 : ALLWIDE ? VFGS_WIDE16_LBW : VFGS_WIDE16_LB;
	static_assert(LB >= 2, "both vertical-overlap lines of a block-row must fall into the first group of lines");
	constexpr int IB = IN16 ? 2 : 1, OB = (IN16 && !OUT8) ? 2 : 1;
	constexpr int RW = IN16 ? 8 : 4, OW = OB == 2 ? 8 : 4;

	const int cl0 = (t.r * 16) >> ysh;
	int cl1 = cl0 + (16 >> ysh);
	if (cl1 > pl.lines) cl1 = pl.lines;
	const int nl = cl1 - cl0;
	if (nl <= 0) return;

	const long long in_pitch = pl.in_row_bytes, out_pitch = pl.out_row_bytes;
	const uint8_t* src = pl.in + (long long)t.f * p.in_frame_bytes + (long long)cl0 * in_pitch + (long long)k0 * 2 * IB;
	uint8_t* dst = pl.out + (long long)t.f * p.out_frame_bytes + (long long)cl0 * out_pitch + (long long)k0 * 2 * OB;

	uint32_t raw[LB][RW];
#pragma unroll
	for (int q = 0; q < LB; q++) {
		if (IN16) ld_global_32(src + (q < nl ? q : nl - 1) * in_pitch, raw[q]);
		else ld_global_16(src + (q < nl ? q : nl - 1) * in_pitch, raw[q]);
	}

	const int b = k0 >> 3;
	UvLane L;
	L.has_left = b > 0;
	L.has_right = b + 1 < p.nb;
	L.stride = p.fpat_stride[1]; // U's and V's images have the same geometry
	L.lut_u = lut + (smem_addr_t)(kLutBytes + lane * 4);
	L.lut_v = lut + (smem_addr_t)(2 * kLutBytes + lane * 4);
	constexpr int kOutBias = (IN16 && OUT8) ? 2 : 0;
	L.lo2 = (uint32_t)(p.lo[1] + kOutBias) * 0x00010001u; L.hi2 = (uint32_t)(p.hi[1] + kOutBias) * 0x00010001u;

	const smem_addr_t img_u = lut + (smem_addr_t)(ptrdiff_t)p.fimg_off[1], img_v = lut + (smem_addr_t)(ptrdiff_t)p.fimg_off[2];
	const int srow = t.r - p.stream_row0;
	const uint16_t* w_u = p.woffs + (((long long)t.f * p.stream_rows + srow) * p.spitch + 1 + b) * 4 + 1; // V: w_u + 1
	auto windows = [&](const uint16_t* w, UvUp& o) {
		o.own_u = img_u + (smem_addr_t)w[0];
		o.own_v = img_v + (smem_addr_t)w[1];
		o.lh_u = o.rh_u = o.own_u; o.lh_v = o.rh_v = o.own_v;
		if (L.has_left) { o.lh_u = img_u + (smem_addr_t)(w[-4] + 7); o.lh_v = img_v + (smem_addr_t)(w[-3] + 7); }
		if (L.has_right) { o.rh_u = img_u + (smem_addr_t)w[4]; o.rh_v = img_v + (smem_addr_t)w[5]; }
	};
	UvUp C;
	windows(w_u, C);
	L.own_u = C.own_u; L.own_v = C.own_v; L.lh_u = C.lh_u; L.rh_u = C.rh_u; L.lh_v = C.lh_v; L.rh_v = C.rh_v;
	UvUp U = C;
	bool ovl = t.r > 0;
	if (ovl) windows(w_u - p.spitch * 4, U);

	int rc = 0;
	const uint8_t* nxt = src + LB * in_pitch;
#pragma unroll 1
	for (int base = 0; base < nl; base += LB) {
#pragma unroll
		for (int q = 0; q < LB; q++) {
			const int line = base + q;
			uint32_t w[OW];
			int wc = 0, wu = 0, ru = 0;
			if (q == 0 && ovl) { wc = ysh ? 20 : 12; wu = ysh ? 20 : 24; ru = (16 >> ysh) * L.stride; }
			if (q == 1 && ovl && !ysh) { wc = 24; wu = 12; ru = 17 * L.stride; }
			uv_line<IN16, OUT8>(L, rc, wc, wu, U, ru, raw[q], w);
			if (OB == 2) lsb_to_msb<OW>(w);
			if (IN16) ld_global_32_if(nxt, raw[q], line + LB < nl);
			else ld_global_16_if(nxt, raw[q], line + LB < nl);
			if (line < nl) {
				if (OB == 2) st_global_32(dst, w);
				else st_global_16(dst, w);
			}
			rc += L.stride; nxt += in_pitch; dst += out_pitch;
		}
		ovl = false;
	}
}

// Dispatch on the component's block size (16 samples: luma and non-subsampled chroma; 8: chroma
// subsampled horizontally).
// Fast-kernel task numbering: per frame the components one after the other; inside a component the
// stripes' rows are one flat run of lane units (8 samples, or 16 on the wide path: FgsParams::fwide), 32
// consecutive units per warp-task, so only the very last task of a component can have idle lanes (a row need
// not be a multiple of 256 samples).
// ALLWIDE: every component of the launch takes the 16-samples-per-lane path (FgsParams::fallwide); the kernel variant then
// has its own CTA size and more lines in flight per lane.
// SEMI: semi-planar frames (NV12 / P010): component 1 is the interleaved UV plane (uv_task_body), component 2 has no
// tasks, luma is served here only on the wide path (16-bit luma MSB-aligned).
template <bool IN16, bool OUT8, bool EDGE = false, bool ALLWIDE = false, bool SEMI = false>
VFGS_HD void process_task_fast(const FgsParams& p, smem_addr_t lut, uint32_t task, int lane)
{
	TaskGeom t;
	t.f = (int)fastdiv(task, p.div_ftasks);
	uint32_t q = task - (uint32_t)t.f * (uint32_t)p.ftasks_per_frame;
	t.c = 0;
	if (q >= (uint32_t)p.ftasks[0]) { q -= (uint32_t)p.ftasks[0]; t.c = 1; }
	if (t.c == 1 && q >= (uint32_t)p.ftasks[1]) { q -= (uint32_t)p.ftasks[1]; t.c = 2; }
	const uint32_t unit = q * 32u + (uint32_t)lane;
	const uint32_t upr = (uint32_t)p.funits_per_row[t.c];
	if (unit >= upr * (uint32_t)p.rows) return;
	const uint32_t row = fastdiv(unit, p.div_funits[t.c]);
	t.r = p.row_begin + (int)row;
	t.seg = 0;
	static_assert(!(ALLWIDE && EDGE), "the EDGE variant has no wide path");
	static_assert(!(SEMI && EDGE), "the EDGE variant has no semi-planar form");
	if constexpr (SEMI) {
		const int u = (int)(unit - row * upr);
		if (t.c) uv_task_body<IN16, OUT8, ALLWIDE>(p, lut, t, u * 8, lane);
		else wide_task_body<IN16, OUT8, 4, ALLWIDE, IN16>(p, lut, t, u * 16, lane); // the host sends wide luma only
		return;
	}
	if (ALLWIDE || (!EDGE && p.fwide[t.c])) { // 16 samples per lane
		const int k0 = (int)(unit - row * upr) * 16;
		if (t.c && p.subx > 1) wide_task_body<IN16, OUT8, 3, ALLWIDE>(p, lut, t, k0, lane);
		else wide_task_body<IN16, OUT8, 4, ALLWIDE>(p, lut, t, k0, lane);
		return;
	}
	if (ALLWIDE) return;
	const int k0 = (int)(unit - row * upr) * kSamplesPerLane;
	if (t.c && p.subx > 1) fast_task_body<IN16, OUT8, 3, EDGE>(p, lut, t, k0, lane);
	else fast_task_body<IN16, OUT8, 4, EDGE>(p, lut, t, k0, lane);
}

} // namespace vfgs
