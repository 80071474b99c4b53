// fgs_gather.h -- grain kernel task code for components whose pattern LUT selects SEVERAL pattern
// slots (sample-adaptive pattern selection: the reference's built-in default SEI with 8 luma
// patterns, cfg/fgs_sei_ff_test5-7 chroma). Same memory pipeline as the single-pattern path
// (fgs_fast.h: lane = 8 samples, lines in flight with rotating refill, packed 16-bit clip), but the
// grain byte of every sample is a true gather:
//     entry = lut[intensity]            one conflict-free 32-bit shared load; the component has its own
//                                       per-lane replicated table, entry = scale + slot (layouts: gather_lut_entry)
//     grain = pattern[slot offset + window row + column]      one byte load, bank conflicts as they fall
// Second version (round 2). What changed against the first one, and why (profiles/r01_v13_fgs_apply_gather.md:
// 20 lane-instructions per sample, 45 shared-memory wavefronts per 256 samples, 53 % of them replays):
//   * The neighbour GRAIN an edge filter needs (vfgs_hw.c:250-259 reads the unfiltered grain of the two samples
//     on either side of a block edge) is no longer recomputed from the neighbour's input sample (a second LUT
//     lookup + gather per lane and line, plus global loads for the warp's end lanes): the adjacent lane has just
//     computed exactly that value, so it travels by ONE warp shuffle. Only a warp's two end lanes still recompute
//     their outer neighbour from its input sample (one predicated 2-byte global load per line, issued with the
//     line loads). The component's lane units are numbered flat (all stripes of a frame in one run, like the
//     fast kernel), 32 per warp, so that a warp's 512 bytes of a row start on a 512-byte boundary of the run.
//   * SHIFT variant (in-place calls, 16-sample blocks): a warp holds units 32q-1 .. 32q+30, so that the pairs
//     (second half of block b, first half of block b+1) never straddle two warps and NOTHING reads a neighbour's
//     input sample, which another warp may already have overwritten in place. Measured 11 % slower than the
//     aligned numbering (profiles/r02_gather_ab.md: the warp's row segment then starts 16 bytes before a 128-byte
//     line, every warp-wide access touches a fifth line and both end sectors are written half by half), so it is
//     only used where it saves the detour through a scratch buffer.
//   * The block's random sign (vfgs_hw.c:218 "* s") is folded into WHICH COPY of the slots is read (FOLD: the
//     table image carries the negated slots behind the plain ones; taken when no slot holds a -128 byte and the
//     copies fit into shared memory, else the sign is applied by one multiply per sample).
//   * The two (one) vertical-overlap lines of a stripe are peeled off the steady-state line loop.
// Restates vfgs_hw.c:140-284 per sample like fgs_task.h; host-compilable for tests/emu (the host build replays
// the shuffles from a table, see EmuWarp).
#pragma once
#include "fgs_fast.h"

namespace vfgs {

// Shared memory: [0, 32 KB * ngather) private LUTs of the gather components (each on a 32 KB
// boundary), then the general table image's pattern slots (gpat_off, relative to the image copy) and,
// with FOLD, their negated copies (gneg_off).
#ifndef VFGS_GATHER_LB
#define VFGS_GATHER_LB 2
#endif
constexpr int kGatherLB = VFGS_GATHER_LB; // lines in flight per lane
static_assert(kGatherLB >= 2, "both vertical-overlap lines of a block-row must fall into the first group of lines");

// ---- lane exchange -------------------------------------------------------------------------
// Device: a warp shuffle. Host build (tests/emu runs the lanes one after the other): every task is run twice,
// a recording pass that only notes what each lane sends at each exchange point, and a replaying pass that reads
// the neighbours' values from that table and is the only one that stores.
#if !defined(__CUDA_ARCH__)
struct EmuWarp {
	bool record = false;
	int lane = 0, point = 0;
	long long octet_lines = 0; // lane-lines that took the uniform-slot octet path (tests/emu: is it really taken?)
	int table[64][32];
};
inline EmuWarp& emu_warp() { static thread_local EmuWarp w; return w; }
#endif
VFGS_HD int lane_exchange(int v, int src_lane)
{
#if defined(__CUDA_ARCH__)
	return __shfl_sync(0xffffffffu, v, src_lane);
#else
	EmuWarp& w = emu_warp();
	const int pt = w.point++;
	if (w.record) { w.table[pt][w.lane] = v; return 0; }
	return w.table[pt][src_lane & 31];
#endif
}
VFGS_HD bool lane_stores()
{
#if defined(__CUDA_ARCH__)
	return true;
#else
	return !emu_warp().record;
#endif
}

// LUT index bits (intensity * 128) of sample e of a lane's raw words.
template <bool IN16, int E>
VFGS_HD uint32_t index_bits(const uint32_t raw[4])
{
	if (IN16) {
		const uint32_t w = raw[E >> 1];
		return (E & 1) ? (shr_fma<11>(w) & 0x7f80u) : ((w << 5) & 0x7f80u); // ((v >> 2) & 0xff) << 7
	} else {
		const uint32_t w = raw[E >> 2];
		constexpr int sh = (E & 3) * 8;
		return sh >= 7 ? (w >> (sh - 7)) & 0x7f80u : (w << (7 - sh)) & 0x7f80u;      // v << 7
	}
}

struct GatherLane {
	smem_addr_t own;        // window of the lane's block: slot bank (sign copy with FOLD) + oy * pitch + ox + i0
	smem_addr_t up;         // same for the block above (overlap lines only)
	smem_addr_t nb, nb_up;  // end lanes of a warp: the outer neighbour's edge column in ITS block's windows
	smem_addr_t lut;        // this lane's column of the component's private LUT
	int s_own, s_up;        // block signs (applied by multiplication when !FOLD)
	int s_nb, s_nb_up;
	bool word_aligned;      // own and up are multiples of 4: the lane's eight bytes of a slot row are two whole words
	int pow16;
	uint32_t slot_mul;      // TOP layout: bytes per slot
	uint32_t lo2, hi2;
};

// Layouts of a LUT entry (expanded from the table image's compact `scale | slot << 8` when a CTA starts).
//   TOP (10-bit input): scale | slot << 27. Both uses of the entry then take it WHOLE, without masking out the other
//     field: entry * pow16 = scale << (16 - ss) exactly, because the slot field leaves the 32-bit word (43 - ss >= 32:
//     ss = scale_shift <= 11 whenever the input is 10 bits deep, the library's entry check ss + bs <= 13 restating
//     vfgs_hw.c:170), and the slot's byte offset is (entry >> 27) * slot bytes (a shift and a multiply on the FMA pipe).
//     That is eight ALU-pipe instructions less per eight samples on a kernel whose ALU pipe is its busiest unit on
//     real pictures (profiles/r02_gather_natural.md).
//   else (8-bit input, ss up to 13): scale | slot byte offset << 8.
template <bool TOP>
VFGS_HD uint32_t gather_lut_entry(uint32_t compact, uint32_t slot_bytes)
{
	return TOP ? (compact & 0xffu) | ((compact >> 8) << 27) : (compact & 0xffu) | (((compact >> 8) * slot_bytes) << 8);
}
template <bool TOP>
VFGS_HD smem_addr_t entry_slot_offset(const GatherLane& L, uint32_t ent)
{
	return (smem_addr_t)(TOP ? (ent >> 27) * L.slot_mul : ent >> 8);
}
// scale << (16 - scale_shift)
template <bool TOP>
VFGS_HD int entry_scale16(const GatherLane& L, uint32_t ent)
{
	return (int)((TOP ? ent : ent & 0xffu) * (uint32_t)L.pow16);
}
template <bool TOP> struct EntrySlot { static constexpr uint32_t lsb = TOP ? 1u << 27 : 1u << 8; }; // lowest bit of the slot field

// Unfiltered grain (vertical overlap blended in, block sign applied) of sample E from its LUT entry: one byte gather
// (two on an overlap line), bank conflicts as the windows and slots fall.
template <bool TOP, bool FOLD, bool OVERLAP, int E>
VFGS_HD int gather_sample(const GatherLane& L, uint32_t ent, int rc, int ru, int wc, int wu)
{
	const smem_addr_t off = entry_slot_offset<TOP>(L, ent) + E;
	int g = lds_s8(L.own + rc + off);
	if (OVERLAP) g = (g * wc + lds_s8(L.up + ru + off) * wu + 16) >> 5; // vfgs_hw.c:223-229; wc / wu carry the signs when !FOLD
	else if (!FOLD) g *= L.s_own;
	return g;
}
template <bool FOLD, bool OVERLAP, int E>
VFGS_HD int octet_sample(const GatherLane& L, uint32_t c0, uint32_t c1, uint32_t u0, uint32_t u1, int wc, int wu)
{
	int g = octet_byte<E>(c0, c1);
	if (OVERLAP) g = (g * wc + octet_byte<E>(u0, u1) * wu + 16) >> 5;
	else if (!FOLD) g *= L.s_own;
	return g;
}

// One line of one lane, up to the exchange: g[] and sc[]. The eight LUT lookups come first. A lane whose eight samples all
// select the same pattern slot (the rule on real pictures: the slot changes with the intensity INTERVAL,
// vfgs_fw.c:598-622, and neighbouring samples mostly share one) and whose window is word aligned reads its eight
// grain bytes as two consecutive words of that slot's row. The branch is per lane: in a mixed warp the hardware runs
// both sides one after the other, each with its own lanes only, and a byte gather issued for a handful of lanes
// hardly conflicts, so the shared-memory wavefronts (the kernel's bound: profiles/r02_gather_uniform.md) shrink with every
// lane that qualifies. Uniformly random samples never qualify and pay five extra instructions per line for the test.
#ifndef VFGS_GATHER_OCTET_PATH
#define VFGS_GATHER_OCTET_PATH 1 // build-time knob for experiments
#endif
template <bool IN16, bool FOLD, bool OVERLAP>
VFGS_HD void gather_grain(const GatherLane& L, const uint32_t raw[4], int rc, int ru, int w_cur, int w_up, int g[8], int sc[8])
{
	const int wc = FOLD ? w_cur : w_cur * L.s_own, wu = FOLD ? w_up : w_up * L.s_up;
	uint32_t ent[8];
	ent[0] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 0>(raw)); ent[1] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 1>(raw));
	ent[2] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 2>(raw)); ent[3] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 3>(raw));
	ent[4] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 4>(raw)); ent[5] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 5>(raw));
	ent[6] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 6>(raw)); ent[7] = lds32(L.lut | (smem_addr_t)index_bits<IN16, 7>(raw));
#pragma unroll
	for (int e = 0; e < 8; e++) sc[e] = entry_scale16<IN16>(L, ent[e]);
	if (VFGS_GATHER_OCTET_PATH) {
		const uint32_t diff = ((ent[0] ^ ent[1]) | (ent[0] ^ ent[2]) | (ent[0] ^ ent[3])) | ((ent[0] ^ ent[4]) | (ent[0] ^ ent[5]) | (ent[0] ^ ent[6])) |
		                      (ent[0] ^ ent[7]);
		if (diff < EntrySlot<IN16>::lsb && L.word_aligned) {
#if !defined(__CUDA_ARCH__)
			emu_warp().octet_lines++;
#endif
			const smem_addr_t so = entry_slot_offset<IN16>(L, ent[0]);
			const smem_addr_t a = L.own + rc + so;
			const uint32_t c0 = lds32(a), c1 = lds32(a + 4);
			uint32_t u0 = 0, u1 = 0;
			if (OVERLAP) { const smem_addr_t b = L.up + ru + so; u0 = lds32(b); u1 = lds32(b + 4); }
			g[0] = octet_sample<FOLD, OVERLAP, 0>(L, c0, c1, u0, u1, wc, wu); g[1] = octet_sample<FOLD, OVERLAP, 1>(L, c0, c1, u0, u1, wc, wu);
			g[2] = octet_sample<FOLD, OVERLAP, 2>(L, c0, c1, u0, u1, wc, wu); g[3] = octet_sample<FOLD, OVERLAP, 3>(L, c0, c1, u0, u1, wc, wu);
			g[4] = octet_sample<FOLD, OVERLAP, 4>(L, c0, c1, u0, u1, wc, wu); g[5] = octet_sample<FOLD, OVERLAP, 5>(L, c0, c1, u0, u1, wc, wu);
			g[6] = octet_sample<FOLD, OVERLAP, 6>(L, c0, c1, u0, u1, wc, wu); g[7] = octet_sample<FOLD, OVERLAP, 7>(L, c0, c1, u0, u1, wc, wu);
			return;
		}
	}
	g[0] = gather_sample<IN16, FOLD, OVERLAP, 0>(L, ent[0], rc, ru, wc, wu); g[1] = gather_sample<IN16, FOLD, OVERLAP, 1>(L, ent[1], rc, ru, wc, wu);
	g[2] = gather_sample<IN16, FOLD, OVERLAP, 2>(L, ent[2], rc, ru, wc, wu); g[3] = gather_sample<IN16, FOLD, OVERLAP, 3>(L, ent[3], rc, ru, wc, wu);
	g[4] = gather_sample<IN16, FOLD, OVERLAP, 4>(L, ent[4], rc, ru, wc, wu); g[5] = gather_sample<IN16, FOLD, OVERLAP, 5>(L, ent[5], rc, ru, wc, wu);
	g[6] = gather_sample<IN16, FOLD, OVERLAP, 6>(L, ent[6], rc, ru, wc, wu); g[7] = gather_sample<IN16, FOLD, OVERLAP, 7>(L, ent[7], rc, ru, wc, wu);
}

// Unfiltered grain of the sample `v` next to a warp's end lane, from that sample's own intensity and its own block's
// window (the value the neighbouring warp's end lane computes for itself).
template <bool TOP, bool FOLD, bool OVERLAP>
VFGS_HD int gather_neighbour(const GatherLane& L, uint32_t v, int in_shift, int rc, int ru, int w_cur, int w_up)
{
	const smem_addr_t off = entry_slot_offset<TOP>(L, lds32(L.lut | (smem_addr_t)(((v >> in_shift) & 0xffu) << 7)));
	int g = lds_s8(L.nb + rc + off);
	if (OVERLAP) {
		const int wc = FOLD ? w_cur : w_cur * L.s_nb, wu = FOLD ? w_up : w_up * L.s_nb_up;
		g = (g * wc + lds_s8(L.nb_up + ru + off) * wu + 16) >> 5;
	} else if (!FOLD) g *= L.s_nb;
	return g;
}

// scale, add, clip (vfgs_hw.c:239, 260-267) and the optional 10 -> 8 bit conversion (yuv.c:231); sc[] = scale << (16 - scale_shift)
template <bool IN16, bool OUT8>
VFGS_HD void gather_finish(const GatherLane& L, const uint32_t raw[4], const int g[8], const int sc[8], uint32_t outw[4])
{
	if (IN16) {
		constexpr int kRound = OUT8 ? 0x28000 : 0x8000; // 8-bit output: the + 2 of yuv.c:231 rides on the rounding and the clip range (fast_line)
		uint32_t r[4];
#pragma unroll
		for (int k = 0; k < 4; k++) {
			const int a_lo = sc[2 * k] * g[2 * k] + kRound;
			const int a_hi = sc[2 * k + 1] * g[2 * k + 1] + kRound;
			const uint32_t d2 = prmt((uint32_t)a_lo, (uint32_t)a_hi, 0x7632);
			const uint32_t v2 = min_u16x2(raw[k], 0x3fff3fffu);
			r[k] = min_s16x2(add_max_s16x2(v2, d2, L.lo2), L.hi2);
		}
		if (OUT8) {
#pragma unroll
			for (int k = 0; k < 4; k++) r[k] >>= 2;
			outw[0] = prmt(r[0], r[1], 0x6420);
			outw[1] = prmt(r[2], r[3], 0x6420);
		} else {
			outw[0] = r[0]; outw[1] = r[1]; outw[2] = r[2]; outw[3] = r[3];
		}
	} else {
		uint32_t r[4];
#pragma unroll
		for (int k = 0; k < 4; k++) {
			const uint32_t v2 = prmt(k < 2 ? raw[0] : raw[1], 0u, (k & 1) ? 0x4342 : 0x4140);
			const int a_lo = sc[2 * k] * g[2 * k] + 0x8000;
			const int a_hi = sc[2 * k + 1] * g[2 * k + 1] + 0x8000;
			const uint32_t d2 = prmt((uint32_t)a_lo, (uint32_t)a_hi, 0x7632);
			r[k] = min_s16x2(add_max_s16x2(v2, d2, L.lo2), L.hi2);
		}
		outw[0] = prmt(r[0], r[1], 0x6420);
		outw[1] = prmt(r[2], r[3], 0x6420);
	}
}

// Window address (without slot offset) and sign of a block from its precomputed table entry
// (FgsParams::woffs, gather format: oy * pitch + ox, bit 15 = negative sign).
template <bool FOLD>
VFGS_HD smem_addr_t gather_window(smem_addr_t bank, int neg_off, uint32_t entry, int col, int& sign)
{
	const bool neg = (entry & 0x8000u) != 0;
	sign = neg ? -1 : 1;
	return bank + (smem_addr_t)((entry & 0x7fffu) + (uint32_t)col + (uint32_t)((FOLD && neg) ? neg_off : 0));
}

// one sample (IB bytes wide) when pred is set, else 0; volatile so that it is issued where it is written (a batch
// ahead of its use) instead of being sunk next to the use
template <int IB>
VFGS_HD uint32_t ld_sample_if(const uint8_t* p, bool pred)
{
#if defined(__CUDA_ARCH__)
	uint32_t v = 0;
	if (IB == 2)
		asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q ld.global.u16 %0, [%1];\n\t}" : "+r"(v) : "l"(p), "r"((uint32_t)pred));
	else
		asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q ld.global.u8 %0, [%1];\n\t}" : "+r"(v) : "l"(p), "r"((uint32_t)pred));
	return v;
#else
	if (!pred) return 0;
	return IB == 2 ? (uint32_t)*(const uint16_t*)p : (uint32_t)*p;
#endif
}
// The kernel keeps few lines in flight per lane (registers: LB = 2 at 28 warps = 28 KB per SM) and was bound by the
// latency of its line loads once the instruction count had come down (long_scoreboard 4.9 warps per issue cycle before,
// 1.4 after: profiles/r02_gather_natural.md). Lines further down the stripe are therefore prefetched into L1 (no registers),
// and the line loads are ordinary cached loads that find them there. Measured on B200 (profiles/r02_gather_ab.md, same
// box, two rounds): smooth pictures 0.747 -> 0.791 of the HBM peak, uniform random samples 0.724 -> 0.741.
#ifndef VFGS_GATHER_PREFETCH
#define VFGS_GATHER_PREFETCH 4 // lines ahead of the line loads that are prefetched into L1 (0: none, line loads bypass L1)
#endif
// (Prefetching the first lines of the warp's NEXT task as well was measured without gain and removed, profiles/r02_gather_ab.md.)
// line loads of the gather kernel: cached (they hit the prefetched lines) unless prefetching is off
template <bool IN16>
VFGS_HD void gather_ld_if(const uint8_t* p, uint32_t r[4], bool pred)
{
	if (VFGS_GATHER_PREFETCH > 0) {
#if defined(__CUDA_ARCH__)
		if (IN16)
			asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %5, 0;\n\t@q ld.global.v4.u32 {%0,%1,%2,%3}, [%4];\n\t}"
			             : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]) : "l"(p), "r"((uint32_t)pred));
		else
			asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %3, 0;\n\t@q ld.global.v2.u32 {%0,%1}, [%2];\n\t}"
			             : "+r"(r[0]), "+r"(r[1]) : "l"(p), "r"((uint32_t)pred));
#else
		if (pred) memcpy(r, p, IN16 ? 16 : 8);
#endif
	} else {
		if (IN16) ld_global_16_if(p, r, pred);
		else ld_global_8_if(p, r, pred);
	}
}
// One warp-task: 32 consecutive flat lane units of a component (lane = 8 samples: half a 16-sample block with one
// block edge, NSH = 4, or a whole 8-sample block with an edge at both ends, NSH = 3). Units run over all stripes of
// a frame; rows are padded to an even number of units so that the parity of a unit is the parity of its lane.
// SHIFT (NSH = 4 only): the warp holds units 32 q - 1 .. 32 q + 30 instead, see the head of this file.
// Every lane walks the full line count of a stripe (the exchange is a warp-wide shuffle); lanes outside the picture
// or past the end of a short last stripe neither load nor store.
// MSB: 16-bit samples hold the value in bits 15..6 (P010 luma of semi-planar frames), converted where a line is used.
template <bool IN16, bool OUT8, int NSH, bool FOLD, bool SHIFT, bool MSB = false>
VFGS_HD void gather_task_body(const FgsParams& p, smem_addr_t luts, smem_addr_t img, int f, int c, uint32_t q, int lane)
{
	constexpr bool PAIR = NSH == 4;
	static_assert(PAIR || !SHIFT, "the shifted numbering exists for 16-sample blocks only");
	constexpr int n = 1 << NSH;
	constexpr int LB = kGatherLB;
	const Plane& pl = p.comp[c];
	const int ysh = (c && p.suby > 1) ? 1 : 0;
	const int lines = 16 >> ysh;

	// which unit is this lane
	const long long u = (long long)q * 32 + lane - (SHIFT ? 1 : 0);
	const uint32_t upr = (uint32_t)p.gunits_per_row[c];                 // padded to even
	bool valid = u >= 0 && u < (long long)upr * (uint32_t)p.rows;
	const uint32_t uu = valid ? (uint32_t)u : 0u;
	const uint32_t row = fastdiv(uu, p.div_gunits[c]);
	const int j = (int)(uu - row * upr);
	const int k0 = j * kSamplesPerLane;
	valid = valid && k0 < pl.width;                                    // the padding unit of an odd row
	const int r = p.row_begin + (int)row;

	const int cl0 = (r * 16) >> ysh;
	int nl = pl.lines - cl0;
	nl = nl > lines ? lines : nl;
	if (!valid || nl < 0) nl = 0;

	constexpr int IB = IN16 ? 2 : 1, OB = (IN16 && !OUT8) ? 2 : 1;
	const long long in_pitch = pl.in_row_bytes, out_pitch = pl.out_row_bytes;
	const uint8_t* src = pl.in + (long long)f * p.in_frame_bytes + (long long)cl0 * in_pitch + (long long)k0 * IB;
	uint8_t* dst = pl.out + (long long)f * p.out_frame_bytes + (long long)cl0 * out_pitch + (long long)k0 * OB;
	const bool stores = lane_stores();

	const int b = valid ? (k0 >> NSH) : 0; // idle lanes must not index past the table row
	const int i0 = k0 & (n - 1);
	const bool has_left = valid && (i0 == 0) && (b > 0);
	const bool has_right = valid && (i0 + kSamplesPerLane == n) && (b + 1 < p.nb);
	const bool odd = i0 != 0; // PAIR: second half of a block, its one edge is on the right
	// a warp's end lanes fetch their outer neighbour's sample from memory (never with SHIFT: every pair is inside a warp);
	// the host build runs lane by lane with the same rule
	const bool mem_left = !SHIFT && lane == 0 && has_left;
	const bool mem_right = !SHIFT && lane == 31 && has_right && k0 + kSamplesPerLane < pl.width; // samples right of the picture read as 0
	const bool mem_halo = mem_left || mem_right;
	const long long halo_off = mem_right ? (long long)kSamplesPerLane * IB : -(long long)IB;

	uint32_t raw[LB][4] = {}, vh[LB];
#pragma unroll
	for (int qq = 0; qq < LB; qq++) {
		gather_ld_if<IN16>(src + qq * in_pitch, raw[qq], qq < nl);
		vh[qq] = SHIFT ? 0u : ld_sample_if<IB>(src + qq * in_pitch + halo_off, mem_halo && qq < nl);
	}
	if (VFGS_GATHER_PREFETCH > 0) {
#pragma unroll
		for (int qq = LB; qq < LB + VFGS_GATHER_PREFETCH; qq++) prefetch_l1(src + qq * in_pitch, qq < nl);
	}

	const int bank = c ? 1 : 0;
	const int stride = p.pat_stride[bank];
	GatherLane L;
	L.lut = luts + (smem_addr_t)(p.glut_index[c] * kLutBytes + lane * 4);
	L.pow16 = p.pow16;
	L.slot_mul = p.gslot_mul[c ? 1 : 0];
	constexpr int kOutBias = (IN16 && OUT8) ? 2 : 0;
	L.lo2 = (uint32_t)(p.lo[c] + kOutBias) * 0x00010001u; L.hi2 = (uint32_t)(p.hi[c] + kOutBias) * 0x00010001u;

	const int srow = r - p.stream_row0;
	const uint16_t* w_cur = p.woffs + (((long long)f * p.stream_rows + (valid ? srow : 0)) * p.spitch + 1 + b) * 4 + c;
	const smem_addr_t bank_addr = img + (smem_addr_t)p.gpat_off[bank];
	const int neg_off = p.gneg_off[bank];
	L.own = gather_window<FOLD>(bank_addr, neg_off, w_cur[0], i0, L.s_own);
	L.up = L.nb = L.nb_up = L.own; L.s_up = L.s_nb = L.s_nb_up = 1;
	const bool ovl = valid && r > 0; // the first lines of a stripe overlap the block-row above (never in the first stripe, y <= 15)
	if (ovl) L.up = gather_window<FOLD>(bank_addr, neg_off, (w_cur - p.spitch * 4)[0], i0, L.s_up);
	L.word_aligned = ((L.own | L.up) & 3) == 0; // pattern rows and slots are multiples of 4 bytes apart (vfgs_tables.h)
	if (!SHIFT && mem_halo) { // the neighbouring block's window: its last column (left neighbour) or its first (right neighbour)
		const int nbo = mem_right ? 4 : -4, col = mem_right ? 0 : n - 1;
		L.nb = gather_window<FOLD>(bank_addr, neg_off, w_cur[nbo], col, L.s_nb);
		if (ovl) L.nb_up = gather_window<FOLD>(bank_addr, neg_off, (w_cur - p.spitch * 4)[nbo], col, L.s_nb_up);
	}

	// exchange partner of a 16-sample-block lane: the other side of its one block edge
	const int partner = odd ? lane + 1 : lane - 1;

	int rc = 0;
	const uint8_t* nxt = src + LB * in_pitch;
	// one group of LB lines; FIRST: the group that holds the vertical-overlap lines
	auto group = [&](int base, auto first_tag) {
		constexpr bool FIRST = decltype(first_tag)::value;
#pragma unroll
		for (int qq = 0; qq < LB; qq++) {
			const int line = base + qq;
			int g[8], sc[8], gh = 0;
			bool done = false;
			if constexpr (MSB) { // in place: the slot is refilled after this line
				msb_to_lsb<4>(raw[qq], raw[qq]);
				vh[qq] >>= 6;
			}
			if (FIRST && qq < 2 && !(qq == 1 && ysh)) { // vfgs_hw.c:173-188: lines 0 and 1 (line 0 only for vertically subsampled chroma)
				if (ovl) { // per lane: a warp may hold the end of the first stripe and the start of the second
					const int w_c = qq == 0 ? (ysh ? 20 : 12) : 24, w_u = qq == 0 ? (ysh ? 20 : 24) : 12;
					const int ru = ((16 + qq) >> ysh) * stride;
					gather_grain<IN16, FOLD, true>(L, raw[qq], rc, ru, w_c, w_u, g, sc);
					if (!SHIFT) gh = gather_neighbour<IN16, FOLD, true>(L, vh[qq], p.bs, rc, ru, w_c, w_u);
					done = true;
				}
			}
			if (!done) {
				gather_grain<IN16, FOLD, false>(L, raw[qq], rc, 0, 0, 0, g, sc);
				if (!SHIFT) gh = gather_neighbour<IN16, FOLD, false>(L, vh[qq], p.bs, rc, 0, 0, 0);
			}

			// block-edge filter (vfgs_hw.c:250-259): both sides read the unfiltered grain of the other side
			if (PAIR) {
				int got = lane_exchange(odd ? g[7] : g[0], partner);
				if (!SHIFT) got = mem_halo ? gh : got;
				const int a = odd ? g[7] : g[0], bb = odd ? g[6] : g[1];
				const int fl = (got + 3 * a + bb + 2) >> 2;
				g[0] = has_left ? fl : g[0];
				g[7] = has_right ? fl : g[7];
			} else {
				int gl = lane_exchange(g[7], lane - 1), gr = lane_exchange(g[0], lane + 1);
				gl = mem_left ? gh : gl; gr = mem_right ? gh : gr;
				const int f0 = (gl + 3 * g[0] + g[1] + 2) >> 2;
				const int f7 = (g[6] + 3 * g[7] + gr + 2) >> 2;
				g[0] = has_left ? f0 : g[0];
				g[7] = has_right ? f7 : g[7];
			}
			uint32_t w[4];
			gather_finish<IN16, OUT8>(L, raw[qq], g, sc, w);
			if constexpr (MSB && OB == 2) lsb_to_msb<4>(w);
			const bool more = line + LB < nl;
			gather_ld_if<IN16>(nxt, raw[qq], more);
			if (!SHIFT) vh[qq] = ld_sample_if<IB>(nxt + halo_off, mem_halo && more);
			if (VFGS_GATHER_PREFETCH > 0) prefetch_l1(nxt + VFGS_GATHER_PREFETCH * in_pitch, line + LB + VFGS_GATHER_PREFETCH < nl);
			if (line < nl && stores) {
				if (OB == 2) st_global_16(dst, w);
				else st_global_8(dst, w);
			}
			rc += stride; nxt += in_pitch; dst += out_pitch;
		}
	};
	group(0, std::true_type());
#pragma unroll 1
	for (int base = LB; base < lines; base += LB) group(base, std::false_type());
}

// Gather-kernel task numbering: per frame the gather components one after the other, each cut into warp-tasks of
// 32 consecutive flat units.
template <bool IN16, bool OUT8, bool FOLD, bool SHIFT, bool MSB = false>
VFGS_HD void process_task_gather(const FgsParams& p, smem_addr_t luts, smem_addr_t img, uint32_t task, int lane)
{
	const int f = (int)fastdiv(task, p.div_gtasks);
	uint32_t q = task - (uint32_t)f * (uint32_t)p.gtasks_per_frame;
	int c = 0;
	if (q >= (uint32_t)p.gtasks[0]) { q -= (uint32_t)p.gtasks[0]; c = 1; }
	if (c == 1 && q >= (uint32_t)p.gtasks[1]) { q -= (uint32_t)p.gtasks[1]; c = 2; }
#if !defined(__CUDA_ARCH__)
	emu_warp().lane = lane; emu_warp().point = 0;
#endif
	if constexpr (MSB) { // luma only
		if (SHIFT) gather_task_body<IN16, OUT8, 4, FOLD, true, true>(p, luts, img, f, c, q, lane);
		else gather_task_body<IN16, OUT8, 4, FOLD, false, true>(p, luts, img, f, c, q, lane);
		return;
	}
	if (SHIFT) gather_task_body<IN16, OUT8, 4, FOLD, true>(p, luts, img, f, c, q, lane); // the host never sends 8-sample blocks here
	else if (c && p.subx > 1) gather_task_body<IN16, OUT8, 3, FOLD, false>(p, luts, img, f, c, q, lane);
	else gather_task_body<IN16, OUT8, 4, FOLD, false>(p, luts, img, f, c, q, lane);
}

} // namespace vfgs
