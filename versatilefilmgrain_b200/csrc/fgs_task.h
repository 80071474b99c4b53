// fgs_task.h -- one warp-task of the grain kernel, written per lane with no cross-lane exchange.
//
// A warp-task is (frame f, block-row r, component c, segment s): 256 consecutive samples of every
// line of that component inside the 16-luma-line stripe r. Lane l owns the 8 samples starting at
// k0 = 256 s + 8 l on each line, so a lane never straddles a block (blocks are 16 or 8 samples)
// and every block edge falls on a lane boundary. The one neighbour sample an edge filter needs
// from the adjacent block is RECOMPUTED by the lane itself from that block's LFSR window
// (same bit-stream, one bit earlier/later), so lanes, warps and CTAs are fully independent.
//
// Restates, per sample, the reference's add_grain_block (vfgs_hw.c:140-284):
//   intensity / LUTs 209-215,239 | pattern fetch 218 | vertical overlap 173-188,223-229 |
//   horizontal edge filter 250-259 | scale, add, clip 260-268 | 10->8 output yuv.c:216-258
// The same source is compiled for the device (kernels) and, by tests/emu only, for the host.
#pragma once
#include "vfgs_core.h"
#include <string.h>

namespace vfgs {

// ---- global memory access -------------------------------------------------------------------
// Samples are streamed: read once, written once. Cache operators of the 128-bit loads / stores
// (overridable at build time for experiments: -DVFGS_LD_OP='".cs"').
#ifndef VFGS_LD_OP
#define VFGS_LD_OP ".L1::no_allocate"
#endif
#ifndef VFGS_ST_OP
#define VFGS_ST_OP ".L1::no_allocate"
#endif
VFGS_HD void ld_global_16(const uint8_t* p, uint32_t r[4])
{
#if defined(__CUDA_ARCH__)
	asm volatile("ld.global" VFGS_LD_OP ".v4.u32 {%0,%1,%2,%3}, [%4];"
	             : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "l"(p));
#else
	memcpy(r, p, 16);
#endif
}
VFGS_HD void ld_global_8(const uint8_t* p, uint32_t r[2])
{
#if defined(__CUDA_ARCH__)
	asm volatile("ld.global" VFGS_LD_OP ".v2.u32 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "l"(p));
#else
	memcpy(r, p, 8);
#endif
}
VFGS_HD void st_global_16(uint8_t* p, const uint32_t r[4])
{
#if defined(__CUDA_ARCH__)
	asm volatile("st.global" VFGS_ST_OP ".v4.u32 [%0], {%1,%2,%3,%4};"
	             :: "l"(p), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
#else
	memcpy(p, r, 16);
#endif
}
VFGS_HD void st_global_8(uint8_t* p, const uint32_t r[2])
{
#if defined(__CUDA_ARCH__)
	asm volatile("st.global" VFGS_ST_OP ".v2.u32 [%0], {%1,%2};" :: "l"(p), "r"(r[0]), "r"(r[1]) : "memory");
#else
	memcpy(p, r, 8);
#endif
}
VFGS_HD int ld_sample(const uint8_t* row, int k, int bytes)
{
	return bytes == 2 ? (int)((const uint16_t*)row)[k] : (int)row[k];
}

// ---- table access (shared memory on the device) -------------------------------------------
// 8 consecutive pattern bytes starting at any byte address: three aligned words + funnel shifts.
VFGS_HD void fetch8(const uint8_t* p, uint32_t out[2])
{
	const uintptr_t a = (uintptr_t)p;
	const uint32_t* w = (const uint32_t*)(a & ~(uintptr_t)3);
	const int sh = (int)(a & 3) * 8;
	const uint32_t w0 = w[0], w1 = w[1];
	if (sh == 0) {
		out[0] = w0; out[1] = w1;
	} else {
		const uint32_t w2 = w[2];
		out[0] = (w0 >> sh) | (w1 << (32 - sh));
		out[1] = (w1 >> sh) | (w2 << (32 - sh));
	}
}
VFGS_HD int sbyte(const uint32_t w[2], int e) // signed byte e (0..7) of a fetched octet
{
	return (int)(int8_t)(w[e >> 2] >> ((e & 3) * 8));
}

VFGS_HD int rshift_round(int a, int s) { return (a + (1 << (s - 1))) >> s; } // vfgs_hw.c:43

// What a lane needs to know about one block for one line.
struct BlockLine {
	const uint8_t* cur; // pattern bank base + row of the current block's window + ox
	const uint8_t* up;  // same for the block above (overlap rows)
	int s_cur, s_up;    // signs
};

// Unfiltered grain of one sample: column `col` of the block window, pattern slot offset `slot_off`.
VFGS_HD int grain_sample(const BlockLine& bl, int slot_off, int col, int w_cur, int w_up)
{
	int p = (int)(int8_t)bl.cur[slot_off + col] * bl.s_cur;
	if (w_cur) p = rshift_round(p * w_cur + (int)(int8_t)bl.up[slot_off + col] * bl.s_up * w_up, 5);
	return p;
}

struct TaskGeom {
	int f, r, c, seg;
};

VFGS_HD TaskGeom decode_task(const FgsParams& p, uint32_t task)
{
	TaskGeom g;
	const uint32_t fr = fastdiv(task, p.div_tps);
	int q = (int)(task - fr * (uint32_t)p.tasks_per_stripe);
	g.f = (int)fastdiv(fr, p.div_rows);
	g.r = p.row_begin + (int)(fr - (uint32_t)g.f * (uint32_t)p.rows);
	if (q < p.nseg[0]) { g.c = 0; g.seg = q; }
	else if (q < p.nseg[0] + p.nseg[1]) { g.c = 1; g.seg = q - p.nseg[0]; }
	else { g.c = 2; g.seg = q - p.nseg[0] - p.nseg[1]; }
	return g;
}

// One line of one lane: 8 samples in v[] (zero beyond the picture), neighbours' intensities in
// vl/vr when the pattern slot depends on the sample.
struct LaneCtx {
	const uint16_t* lut;   // scale | slot<<8, this component
	const uint8_t* bank;   // pattern slots of this component's bank
	int slot_size, stride;
	int uniform_slot;      // >=0: every sample uses this slot
	int bs, ss, lo, hi;
	int n;                 // samples per block
	int i0;                // first column of the lane inside its block
	bool has_left, has_right;
	BlockOfs cur, up, lcur, lup, rcur, rup;
};

VFGS_HD void lane_line(const LaneCtx& L, int y, int ysh, const int v[8], int vl, int vr, int out[8])
{
	const int j = y & 15;
	int w_cur = 0, w_up = 0; // vfgs_hw.c:173-188
	if (y > 15) {
		if (j == 0) { w_cur = ysh ? 20 : 12; w_up = ysh ? 20 : 24; }
		else if (j == 1) { w_cur = 24; w_up = 12; }
	}
	const int rc = j >> ysh, ru = (16 + j) >> ysh;

	BlockLine me;
	me.cur = L.bank + (L.cur.oy + rc) * L.stride + L.cur.ox + L.i0;
	me.up = L.bank + (L.up.oy + ru) * L.stride + L.up.ox + L.i0;
	me.s_cur = L.cur.sign; me.s_up = L.up.sign;

	int g[8], sc[8];
	if (L.uniform_slot >= 0) {
		// single pattern slot: the lane's 8 grain bytes are contiguous in the pattern row
		const int so = L.uniform_slot * L.slot_size;
		uint32_t pc[2], pu[2];
		fetch8(me.cur + so, pc);
		if (w_cur) fetch8(me.up + so, pu);
#pragma unroll
		for (int e = 0; e < 8; e++) {
			int p = sbyte(pc, e) * me.s_cur;
			if (w_cur) p = rshift_round(p * w_cur + sbyte(pu, e) * me.s_up * w_up, 5);
			g[e] = p;
			sc[e] = L.lut[(v[e] >> L.bs) & 0xff] & 0xff;
		}
	} else {
		// sample-adaptive pattern selection: byte gathers
#pragma unroll
		for (int e = 0; e < 8; e++) {
			const int ent = L.lut[(v[e] >> L.bs) & 0xff];
			sc[e] = ent & 0xff;
			g[e] = grain_sample(me, (ent >> 8) * L.slot_size, e, w_cur, w_up);
		}
	}

	// block-edge filter (vfgs_hw.c:250-259); both taps read unfiltered neighbours
	int g0 = g[0], g7 = g[7];
	if (L.has_left) {
		BlockLine nb;
		nb.cur = L.bank + (L.lcur.oy + rc) * L.stride + L.lcur.ox;
		nb.up = L.bank + (L.lup.oy + ru) * L.stride + L.lup.ox;
		nb.s_cur = L.lcur.sign; nb.s_up = L.lup.sign;
		const int slot = L.uniform_slot >= 0 ? L.uniform_slot : (L.lut[(vl >> L.bs) & 0xff] >> 8);
		const int gl = grain_sample(nb, slot * L.slot_size, L.n - 1, w_cur, w_up);
		g0 = (gl + 3 * g[0] + g[1] + 2) >> 2;
	}
	if (L.has_right) {
		BlockLine nb;
		nb.cur = L.bank + (L.rcur.oy + rc) * L.stride + L.rcur.ox;
		nb.up = L.bank + (L.rup.oy + ru) * L.stride + L.rup.ox;
		nb.s_cur = L.rcur.sign; nb.s_up = L.rup.sign;
		const int slot = L.uniform_slot >= 0 ? L.uniform_slot : (L.lut[(vr >> L.bs) & 0xff] >> 8);
		const int gr = grain_sample(nb, slot * L.slot_size, 0, w_cur, w_up);
		g7 = (g[6] + 3 * g[7] + gr + 2) >> 2;
	}
	g[0] = g0; g[7] = g7;

	// scale, add, clip (vfgs_hw.c:260-268)
	const int rnd = 1 << (L.ss - 1);
#pragma unroll
	for (int e = 0; e < 8; e++) {
		int o = v[e] + ((sc[e] * g[e] + rnd) >> L.ss);
		o = o > L.hi ? L.hi : o;
		o = o < L.lo ? L.lo : o;
		out[e] = o;
	}
}

// Whole warp-task for one lane.
VFGS_HD void process_task(const FgsParams& p, const uint8_t* tab, uint32_t task, int lane)
{
	const TaskGeom t = decode_task(p, task);
	const Plane& pl = p.comp[t.c];
	const int c = t.c;
	const int suby = c ? p.suby : 1;
	const int ysh = suby > 1 ? 1 : 0;                 // chroma line = luma line >> ysh
	const int nsh = (c && p.subx > 1) ? 3 : 4;        // samples per block = 1 << nsh
	const int n = 1 << nsh;
	const int k0 = t.seg * kSegSamples + lane * kSamplesPerLane;
	if (k0 >= pl.width) return;

	// picture lines of this stripe that carry this component
	int y0 = t.r * 16, y1 = y0 + 16;
	if (y0 < p.y_begin) y0 = p.y_begin;
	if (y1 > p.y_end) y1 = p.y_end;
	if (suby > 1) y0 = (y0 + 1) & ~1;
	if (y0 >= y1) return;

	LaneCtx L;
	L.lut = (const uint16_t*)(tab + p.lut_off) + c * 256;
	const int bankid = c ? 1 : 0;
	L.bank = tab + p.pat_off[bankid];
	L.slot_size = p.pat_size[bankid];
	L.stride = p.pat_stride[bankid];
	L.uniform_slot = p.uniform_pi[c];
	L.bs = p.bs; L.ss = p.ss; L.lo = p.lo[c]; L.hi = p.hi[c];
	L.n = n;
	const int b = k0 >> nsh;
	L.i0 = k0 & (n - 1);
	L.has_left = (L.i0 == 0) && (b > 0);
	L.has_right = (L.i0 + kSamplesPerLane == n) && (b + 1 < p.nb);

	// LFSR registers of this block and its neighbours, current and upper block-row
	const int srow = t.r - p.stream_row0;
	const uint32_t* row_cur = p.states + ((long long)t.f * p.stream_rows + srow) * p.spitch + 1;
	const uint32_t* row_up = srow > 0 ? row_cur - p.spitch : row_cur; // only read when y > 15
	L.cur = decode_offsets(c, row_cur[b], p.subx, p.suby);
	L.up = decode_offsets(c, row_up[b], p.subx, p.suby);
	if (L.has_left) {
		L.lcur = decode_offsets(c, row_cur[b - 1], p.subx, p.suby);
		L.lup = decode_offsets(c, row_up[b - 1], p.subx, p.suby);
	} else { L.lcur = L.cur; L.lup = L.up; }
	if (L.has_right) {
		L.rcur = decode_offsets(c, row_cur[b + 1], p.subx, p.suby);
		L.rup = decode_offsets(c, row_up[b + 1], p.subx, p.suby);
	} else { L.rcur = L.cur; L.rup = L.up; }

	const uint8_t* fin = pl.in + (long long)t.f * p.in_frame_bytes;
	uint8_t* fout = pl.out + (long long)t.f * p.out_frame_bytes;
	const int ilv = p.ilv[c], msb_in = p.msb_in, msb_out = p.msb_out; // semi-planar: sample index k is at k << ilv
	const bool full = pl.vec && !ilv && (k0 + kSamplesPerLane <= pl.width);
	const bool need_nb = L.uniform_slot < 0;
	const bool to8 = p.in_bytes == 2 && p.out_bytes == 1;

	constexpr int LB = 4; // lines whose loads are issued back to back
	for (int yb = y0; yb < y1; yb += LB * suby) {
		uint32_t raw[LB][4];
		int vl[LB], vr[LB];
#pragma unroll
		for (int q = 0; q < LB; q++) {
			const int y = yb + q * suby;
			const int cl = y >> ysh;
			if (y < y1 && cl < pl.lines) {
				const uint8_t* row = fin + (long long)cl * pl.in_row_bytes;
				if (full) {
					if (p.in_bytes == 2) ld_global_16(row + k0 * 2, raw[q]);
					else ld_global_8(row + k0, raw[q]);
				} else {
					// picture tail or unaligned rows: sample by sample, zero right of the picture
					int s[8];
#pragma unroll
					for (int e = 0; e < 8; e++) s[e] = (k0 + e < pl.width) ? ld_sample(row, (k0 + e) << ilv, p.in_bytes) : 0;
					if (p.in_bytes == 2) {
#pragma unroll
						for (int e = 0; e < 4; e++) raw[q][e] = (uint32_t)s[2 * e] | ((uint32_t)s[2 * e + 1] << 16);
					} else {
#pragma unroll
						for (int e = 0; e < 2; e++)
							raw[q][e] = (uint32_t)s[4 * e] | ((uint32_t)s[4 * e + 1] << 8) | ((uint32_t)s[4 * e + 2] << 16) | ((uint32_t)s[4 * e + 3] << 24);
					}
				}
				vl[q] = (need_nb && L.has_left) ? ld_sample(row, (k0 - 1) << ilv, p.in_bytes) >> msb_in : 0;
				vr[q] = (need_nb && L.has_right && k0 + 8 < pl.width) ? ld_sample(row, (k0 + 8) << ilv, p.in_bytes) >> msb_in : 0;
			}
		}
#pragma unroll
		for (int q = 0; q < LB; q++) {
			const int y = yb + q * suby;
			const int cl = y >> ysh;
			if (y < y1 && cl < pl.lines) {
				int v[8], o[8];
				if (p.in_bytes == 2) {
#pragma unroll
					for (int e = 0; e < 4; e++) { v[2 * e] = (raw[q][e] & 0xffff) >> msb_in; v[2 * e + 1] = raw[q][e] >> (16 + msb_in); }
				} else {
#pragma unroll
					for (int e = 0; e < 8; e++) v[e] = (raw[q][e >> 2] >> ((e & 3) * 8)) & 0xff;
				}
				lane_line(L, y, ysh, v, vl[q], vr[q], o);
				if (to8) {
#pragma unroll
					for (int e = 0; e < 8; e++) o[e] = (o[e] + 2) >> 2; // yuv.c:231
				}
				uint8_t* orow = fout + (long long)cl * pl.out_row_bytes;
				if (full) {
					if (p.out_bytes == 2) {
						uint32_t w[4];
#pragma unroll
						for (int e = 0; e < 4; e++) w[e] = ((uint32_t)o[2 * e] << msb_out) | ((uint32_t)o[2 * e + 1] << (16 + msb_out));
						st_global_16(orow + k0 * 2, w);
					} else {
						uint32_t w[2];
#pragma unroll
						for (int e = 0; e < 2; e++)
							w[e] = (uint32_t)o[4 * e] | ((uint32_t)o[4 * e + 1] << 8) | ((uint32_t)o[4 * e + 2] << 16) | ((uint32_t)o[4 * e + 3] << 24);
						st_global_8(orow + k0, w);
					}
				} else {
#pragma unroll
					for (int e = 0; e < 8; e++)
						if (k0 + e < pl.width) {
							if (p.out_bytes == 2) ((uint16_t*)orow)[(k0 + e) << ilv] = (uint16_t)(o[e] << msb_out);
							else orow[(k0 + e) << ilv] = (uint8_t)o[e];
						}
				}
			}
		}
	}
}

} // namespace vfgs
