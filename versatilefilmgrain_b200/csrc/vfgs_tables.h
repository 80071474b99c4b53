// vfgs_tables.h -- host-side mirror of the hardware state and the construction of the table images
// and launch parameters the kernels consume. Plain C++ (no CUDA runtime), shared by the C-ABI shim
// (vfgs_b200.cu) and, for the GPU-less logic tests only, by tests/emu/emu.cpp.
#pragma once
#include <stdint.h>
#include <string.h>
#include <vector>

#include "fgs_gather.h"

#ifndef VFGS_PAT_ROW_SKEW
#define VFGS_PAT_ROW_SKEW 8 // bytes (general image: gather and general kernels; build-time knob for experiments)
#endif
#ifndef VFGS_FAST_WIDE8
#define VFGS_FAST_WIDE8 1 // 8-bit input: 16 samples per lane where possible (build-time knob for experiments)
#endif
#ifndef VFGS_FAST_WIDE16
#define VFGS_FAST_WIDE16 1 // 16-bit input: the same with 256-bit accesses (build-time knob for experiments)
#endif
#ifndef VFGS_FAST_ROW_SKEW
#define VFGS_FAST_ROW_SKEW 8 // bytes, multiple of 8 (build-time knob for experiments)
#endif

namespace vfgs {

constexpr int kSlots = 9; // 8 settable + the always-zero slot 8 (vfgs_hw.c:49)

struct HwState {
	int8_t pattern[2][kSlots][64][64];
	uint8_t slut[3][256];
	uint8_t plut[3][256];
	uint32_t rnd, rnd_up, line_rnd, line_rnd_up;
	int scale_shift, bs;
	int y_min, y_max, c_min, c_max;
	int csubx, csuby;
	void power_on()
	{
		memset(pattern, 0, sizeof(pattern));
		memset(slut, 0, sizeof(slut));
		memset(plut, 0, sizeof(plut));
		rnd = rnd_up = line_rnd = line_rnd_up = 0xdeadbeefu; // vfgs_hw.c:52-55
		scale_shift = 5 + 6;                                 // vfgs_hw.c:56
		bs = 0;
		y_min = c_min = 0; y_max = c_max = 255;
		csubx = csuby = 2;
	}
};

struct TableInfo {
	// general image (fgs_task.h)
	int lut_off, pat_off[2], pat_size[2], pat_stride[2], uniform_pi[3], bytes;
	// sign-folded gather launches: the slots in use once more, negated, behind the general image (a bank takes part
	// when none of its slots in use holds a -128 byte); gbytes = size of the image including them
	int nslot[2], neg_off[2], gbytes;
	bool neg_ok[2];
	// fast image (fgs_fast.h): usable for a component when its pattern LUT selects one slot and that
	// slot has no -128 byte (so that -pattern fits int8)
	bool fast_ok[3];
	int fimg_src[3], fimg_bytes[3]; // component images inside the fast image (bytes 0 when !fast_ok)
	bool fshare_cbcr;               // Cr reads Cb's image (same pattern slot)
	int fpat_off[3][2], fpat_stride[3], fpat_copy[3], fbytes; // fpat_off: relative to the component image; fpat_copy: bytes from one column-shifted copy to the next
};

// General image layout (all offsets multiples of 16): LUT uint16[3][256] = scale | slot << 8, then the
// luma slots in use (64 rows), then the chroma slots in use packed to (64/csuby) rows x (64/csubx) bytes;
// rows cols + VFGS_PAT_ROW_SKEW bytes apart.
inline void build_tables(const HwState& h, TableInfo& g_bi, std::vector<uint8_t>& g_blob, std::vector<uint8_t>& g_fblob)
{
	int nslot[2] = {1, 1};
	for (int c = 0; c < 3; c++) {
		int first = h.plut[c][0] >> 4, uni = first;
		for (int i = 0; i < 256; i++) {
			int s = h.plut[c][i] >> 4;
			if (s != first) uni = -1;
			if (s + 1 > nslot[c ? 1 : 0]) nslot[c ? 1 : 0] = s + 1;
		}
		g_bi.uniform_pi[c] = uni;
	}
	const int crows = 64 / h.csuby, ccols = 64 / h.csubx;
	// pattern rows are stored cols + VFGS_PAT_ROW_SKEW bytes apart: the window rows are multiples of 4 (or 2), so
	// with the natural power-of-two pitch the byte gathers of a line would fall into half of the banks
	const int lpitch = 64 + VFGS_PAT_ROW_SKEW, cpitch = ccols + VFGS_PAT_ROW_SKEW;
	g_bi.lut_off = 0;
	g_bi.pat_off[0] = 3 * 256 * 2;
	g_bi.pat_size[0] = 64 * lpitch; g_bi.pat_stride[0] = lpitch;
	g_bi.pat_off[1] = g_bi.pat_off[0] + nslot[0] * g_bi.pat_size[0];
	g_bi.pat_size[1] = crows * cpitch; g_bi.pat_stride[1] = cpitch;
	g_bi.bytes = (g_bi.pat_off[1] + nslot[1] * g_bi.pat_size[1] + 16 + 15) & ~15; // +16: fetch8 may touch one word past an octet
	g_bi.gbytes = g_bi.bytes;
	for (int b = 0; b < 2; b++) { // negated copies of the banks' slots (gather kernel, sign folding)
		g_bi.nslot[b] = nslot[b];
		g_bi.neg_ok[b] = true;
		for (int s = 0; s < nslot[b] && g_bi.neg_ok[b]; s++)
			for (int r = 0; r < 64 && g_bi.neg_ok[b]; r++)
				for (int x = 0; x < 64; x++)
					if (h.pattern[b][s][r][x] == -128) { g_bi.neg_ok[b] = false; break; }
		g_bi.neg_off[b] = g_bi.gbytes - g_bi.pat_off[b]; // relative to the bank's plain slots
		g_bi.gbytes += nslot[b] * g_bi.pat_size[b];
	}
	g_bi.gbytes = (g_bi.gbytes + 15) & ~15;
	g_blob.assign((size_t)g_bi.gbytes, 0);
	uint16_t* lut = (uint16_t*)g_blob.data();
	for (int c = 0; c < 3; c++)
		for (int i = 0; i < 256; i++) lut[c * 256 + i] = (uint16_t)(h.slut[c][i] | ((h.plut[c][i] >> 4) << 8));
	for (int s = 0; s < nslot[0]; s++)
		for (int r = 0; r < 64; r++)
			memcpy(&g_blob[g_bi.pat_off[0] + s * g_bi.pat_size[0] + r * lpitch], h.pattern[0][s][r], 64);
	for (int s = 0; s < nslot[1]; s++)
		for (int r = 0; r < crows; r++)
			memcpy(&g_blob[g_bi.pat_off[1] + s * g_bi.pat_size[1] + r * cpitch], h.pattern[1][s][r], (size_t)ccols);
	for (int b = 0; b < 2; b++) {
		if (!g_bi.neg_ok[b]) continue;
		const int rows = b ? crows : 64, cols = b ? ccols : 64, pitch = g_bi.pat_stride[b];
		for (int s = 0; s < nslot[b]; s++)
			for (int r = 0; r < rows; r++)
				for (int x = 0; x < cols; x++)
					g_blob[g_bi.pat_off[b] + g_bi.neg_off[b] + s * g_bi.pat_size[b] + r * pitch + x] = (uint8_t)(int8_t)-h.pattern[b][s][r][x];
	}

	// fast-path image: compact scale LUT, then per component the single slot as +pattern and -pattern, each in
	// fast_copies() column-shifted copies (copy k holds the pattern moved left by k * 8 / copies bytes), so that
	// every window column has a copy in which it sits on an 8-byte boundary (fgs_fast.h, window_offset)
	int off = 256 * 4;
	g_bi.fshare_cbcr = false;
	for (int c = 0; c < 3; c++) {
		const int rows = c ? crows : 64, cols = c ? ccols : 64;
		const int ncopy = fast_copies((c && h.csubx > 1) ? 8 : 16);
		const int slot = g_bi.uniform_pi[c];
		bool ok = slot >= 0;
		for (int r = 0; ok && r < rows; r++)
			for (int x = 0; x < cols; x++)
				if (h.pattern[c ? 1 : 0][slot][r][x] == -128) { ok = false; break; }
		g_bi.fast_ok[c] = ok;
		// row pitch = cols + VFGS_FAST_ROW_SKEW: the window rows oy are multiples of 4 (or 2), so with a power-of-two
		// pitch every window of a line would start in the same few banks; the skew spreads them over all banks
		const int pitch = cols + VFGS_FAST_ROW_SKEW;
		g_bi.fpat_stride[c] = pitch;
		g_bi.fpat_copy[c] = rows * pitch;
		g_bi.fpat_off[c][0] = 0;
		g_bi.fpat_off[c][1] = ncopy * rows * pitch;
		g_bi.fimg_src[c] = off;
		g_bi.fimg_bytes[c] = ok ? 2 * ncopy * rows * pitch : 0;
		if (c == 2 && ok && g_bi.fast_ok[1] && g_bi.uniform_pi[1] == slot) { // Cb and Cr read the same slot: one image
			g_bi.fimg_src[2] = g_bi.fimg_src[1];
			g_bi.fshare_cbcr = true;
		} else {
			off += g_bi.fimg_bytes[c];
		}
	}
	g_bi.fbytes = (off + 15) & ~15;
	g_fblob.assign((size_t)g_bi.fbytes, 0);
	uint32_t* clut = (uint32_t*)g_fblob.data();
	for (int i = 0; i < 256; i++) clut[i] = (uint32_t)h.slut[0][i] | ((uint32_t)h.slut[1][i] << 8) | ((uint32_t)h.slut[2][i] << 16);
	for (int c = 0; c < 3; c++) {
		if (!g_bi.fast_ok[c] || (c == 2 && g_bi.fshare_cbcr)) continue;
		const int rows = c ? crows : 64, cols = c ? ccols : 64;
		const int ncopy = fast_copies((c && h.csubx > 1) ? 8 : 16), shift = 8 / ncopy;
		for (int k = 0; k < ncopy; k++) {
			const int pitch = g_bi.fpat_stride[c];
			int8_t* plus = (int8_t*)&g_fblob[g_bi.fimg_src[c] + g_bi.fpat_off[c][0] + k * g_bi.fpat_copy[c]];
			int8_t* minus = (int8_t*)&g_fblob[g_bi.fimg_src[c] + g_bi.fpat_off[c][1] + k * g_bi.fpat_copy[c]];
			for (int r = 0; r < rows; r++)
				for (int x = 0; x + k * shift < cols; x++) {
					const int8_t v = h.pattern[c ? 1 : 0][g_bi.uniform_pi[c]][r][x + k * shift];
					plus[r * pitch + x] = v; minus[r * pitch + x] = (int8_t)-v;
				}
		}
	}
}


// State- and table-dependent part of the launch parameters (pointers to the device copies of the
// images are filled in by the caller).
inline void fill_state_params(FgsParams& p, const HwState& h, const TableInfo& bi)
{
	p.subx = h.csubx; p.suby = h.csuby;
	p.bs = h.bs; p.ss = h.scale_shift;
	p.pow16 = 1 << (16 - h.scale_shift);
	for (int c = 0; c < 3; c++) {
		p.lo[c] = (c ? h.c_min : h.y_min) << h.bs;
		p.hi[c] = (c ? h.c_max : h.y_max) << h.bs;
		p.uniform_pi[c] = bi.uniform_pi[c];
		p.fpat_off[c][0] = bi.fpat_off[c][0]; p.fpat_off[c][1] = bi.fpat_off[c][1];
		p.fpat_stride[c] = bi.fpat_stride[c];
		p.fpat_copy[c] = bi.fpat_copy[c];
		p.fimg_src[c] = bi.fimg_src[c]; p.fimg_bytes[c] = bi.fimg_bytes[c];
	}
	p.blob_bytes = bi.bytes;
	p.lut_off = bi.lut_off;
	for (int b = 0; b < 2; b++) { p.pat_off[b] = bi.pat_off[b]; p.pat_size[b] = bi.pat_size[b]; p.pat_stride[b] = bi.pat_stride[b]; }
}

inline bool aligned_for(const void* base, long long row, long long frame, size_t unit)
{
	return ((uintptr_t)base % unit) == 0 && (row % (long long)unit) == 0 && (frame % (long long)unit) == 0;
}

// Planes of a semi-planar call (NV12 / P010): comp[0] is the luma plane, comp[1] / comp[2] are views of the interleaved
// UV plane that start at U0 / V0 and step over the other component's samples (FgsParams::ilv). msb_*: 16-bit samples
// in bits 15..6. Set before finish_tasks.
inline void set_semiplanar_planes(FgsParams& p, const uint8_t* y_in, const uint8_t* uv_in, long long sy_in, long long suv_in,
                                  uint8_t* y_out, uint8_t* uv_out, long long sy_out, long long suv_out, int width, int height,
                                  int cw, int ch, bool msb_in, bool msb_out)
{
	for (int c = 0; c < 3; c++) {
		p.comp[c].in = c ? uv_in + (c - 1) * p.in_bytes : y_in;
		p.comp[c].out = c ? uv_out + (c - 1) * p.out_bytes : y_out;
		p.comp[c].in_row_bytes = c ? suv_in : sy_in;
		p.comp[c].out_row_bytes = c ? suv_out : sy_out;
		p.comp[c].width = c ? cw : width;
		p.comp[c].lines = c ? ch : height;
		p.ilv[c] = c ? 1 : 0;
	}
	p.msb_in = msb_in ? 6 : 0;
	p.msb_out = msb_out ? 6 : 0;
}

// Segments per line, vector-access eligibility and the task count, once planes and sizes are set.
inline void finish_tasks(FgsParams& p)
{
	for (int c = 0; c < 3; c++) {
		p.nseg[c] = (p.comp[c].width + kSegSamples - 1) / kSegSamples;
		p.comp[c].vec = aligned_for(p.comp[c].in, p.comp[c].in_row_bytes, p.in_frame_bytes, 8 * (size_t)p.in_bytes) &&
		                aligned_for(p.comp[c].out, p.comp[c].out_row_bytes, p.out_frame_bytes, 8 * (size_t)p.out_bytes);
	}
	p.tasks_per_stripe = p.nseg[0] + p.nseg[1] + p.nseg[2];
	p.total_tasks = (long long)p.nframes * p.rows * p.tasks_per_stripe;
	p.div_tps = make_fastdiv((uint32_t)(p.tasks_per_stripe > 0 ? p.tasks_per_stripe : 1));
	p.div_rows = make_fastdiv((uint32_t)(p.rows > 0 ? p.rows : 1));
}

#ifndef VFGS_FAST_EXTRA_SMEM
#define VFGS_FAST_EXTRA_SMEM 0 // unused bytes added to the launch (build-time knob: moves the L1/shared carveout)
#endif
// Shared-memory placement of the fast kernel's component images. pad = bytes between the start of the
// kernel's dynamic shared memory and the next 32 KB boundary of the shared window, where the first LUT
// goes: images are packed downwards from that boundary while they fit, the others upwards from the end of
// the third LUT. served[c]: the fast kernel processes component c in this launch. Cr shares Cb's image
// when both read the same pattern slot (fimg_bytes[2] = 0: nothing to copy).
inline void place_fast_images(FgsParams& p, const TableInfo& bi, int pad, const bool served[3])
{
	int front = 0, back = 0;
	for (int c = 0; c < 3; c++) {
		p.fimg_bytes[c] = served[c] ? bi.fimg_bytes[c] : 0;
		const int n = p.fimg_bytes[c];
		p.fimg_off[c] = 0;
		if (!n) continue;
		if (c == 2 && bi.fshare_cbcr && p.fimg_bytes[1]) { // shares Cb's image (and Cb's is resident): nothing to copy
			p.fimg_off[2] = p.fimg_off[1]; p.fimg_bytes[2] = 0;
			continue;
		}
		if (front + n <= pad) { front += n; p.fimg_off[c] = -front; }
		else { p.fimg_off[c] = 3 * kLutBytes + back; back += n; }
	}
	p.fpad = pad;
	p.fsmem = pad + 3 * kLutBytes + back + VFGS_FAST_EXTRA_SMEM;
}

// Which grain kernel serves which component of a whole-frame launch:
//   fast    one pattern slot (no -128 byte), vector-aligned rows, width % 8 == 0        (fgs_fast.h)
//   gather  several pattern slots (or a -128 byte), same alignment conditions, out of place (fgs_gather.h)
//   general everything else: ragged widths, unaligned rows                               (fgs_task.h)
// mode: 0 = as above, 1 = general kernel for everything, 2 = gather kernel wherever it can run
// (1 and 2 exist for the tests). smem_limit: opt-in shared memory per block of the device.
struct LaunchPlan {
	FgsParams fast, gather, general, edge;
	bool any_fast, any_gather, any_general, any_edge;
	int kind[3];     // per component: 0 fast, 1 gather, 2 general kernel, 3 fast kernel's EDGE variant (ragged / unaligned rows)
	int gather_smem; // dynamic shared memory of the gather launch
	bool gather_fold; // the gather launch reads sign-folded slot copies (fgs_gather.h, FOLD)
	bool gather_shift; // in-place call: the gather launch uses the shifted unit numbering (fgs_gather.h, SHIFT)
};

inline void plan_launches(const FgsParams& p, const TableInfo& bi, int mode, bool in_place, int smem_limit, int fast_pad, LaunchPlan& lp)
{
	lp.fast = lp.gather = lp.general = lp.edge = p;
	lp.any_fast = lp.any_gather = lp.any_general = lp.any_edge = false;
	int* kind = lp.kind;
	int ngather = 0;
	// semi-planar frames (FgsParams::ilv): U and V alternate on one plane, so they take ONE kind of kernel (two launches
	// must not write alternate samples of the same words): the fast kernel's interleaved lane when both are single-slot
	// and the plane allows one access per line and lane, else the general kernel. 16-bit (P010) luma takes the wide fast
	// path or the gather kernel, both with the MSB conversion, else the general kernel; 8-bit (NV12) luma is a planar plane,
	// except that the SEMI fast kernel serves it on the wide path only: where planar rows would take 8 samples per lane,
	// it takes the (planar) EDGE variant.
	const bool semi = p.ilv[1] != 0;
	for (int c = 0; c < 3; c++) {
		const bool aligned = p.comp[c].vec && (p.comp[c].width % kSamplesPerLane) == 0;
		kind[c] = 2;
		if (semi && c) {
			if (mode == 0 && bi.fast_ok[1] && bi.fast_ok[2] && p.comp[0].width % 16 == 0 &&
			    aligned_for(p.comp[1].in, p.comp[1].in_row_bytes, p.in_frame_bytes, (size_t)(16 * p.in_bytes)) &&
			    aligned_for(p.comp[1].out, p.comp[1].out_row_bytes, p.out_frame_bytes, (size_t)(16 * p.out_bytes)))
				kind[c] = 0;
			continue;
		}
		if (semi && p.msb_in) {
			const bool wide = VFGS_FAST_WIDE16 != 0 && p.comp[0].width % 16 == 0 &&
			                  aligned_for(p.comp[0].in, p.comp[0].in_row_bytes, p.in_frame_bytes, (size_t)(16 * p.in_bytes)) &&
			                  aligned_for(p.comp[0].out, p.comp[0].out_row_bytes, p.out_frame_bytes, (size_t)(16 * p.out_bytes));
			if (mode == 0 && bi.fast_ok[0] && wide) kind[c] = 0;
			else if (mode != 1 && aligned && (!bi.fast_ok[0] || mode == 2)) kind[c] = 1;
			if (kind[c] == 1) ngather++;
			continue;
		}
		if (aligned && mode != 1) {
			// in place: the gather kernel's shifted numbering (SHIFT) reads nothing but a lane's own samples, but exists for
			// 16-sample blocks only; the aligned numbering recomputes the warps' outer neighbours from INPUT samples
			// another warp may already have overwritten
			const bool block8 = c && p.subx > 1;
			if (bi.fast_ok[c] && mode != 2) kind[c] = 0;
			else if (!in_place || !block8) kind[c] = 1;
		}
#ifndef VFGS_NO_EDGE_KERNEL
		// ragged width or rows that do not start on a vector boundary: the fast kernel's EDGE variant, provided every row
		// starts on a sample boundary (always, for a sane buffer)
		if (!aligned && mode == 0 && bi.fast_ok[c] &&
		    aligned_for(p.comp[c].in, p.comp[c].in_row_bytes, p.in_frame_bytes, (size_t)p.in_bytes) &&
		    aligned_for(p.comp[c].out, p.comp[c].out_row_bytes, p.out_frame_bytes, (size_t)p.out_bytes))
			kind[c] = 3;
#endif
		if (semi && kind[c] == 0 &&
		    !(VFGS_FAST_WIDE8 != 0 && p.comp[0].width % 16 == 0 && aligned_for(p.comp[0].in, p.comp[0].in_row_bytes, p.in_frame_bytes, 16) &&
		      aligned_for(p.comp[0].out, p.comp[0].out_row_bytes, p.out_frame_bytes, 16)))
			kind[c] = 3;
		if (kind[c] == 1) ngather++;
	}
	for (int which = 0; which < 2; which++) { // the fast kernel's tables must fit as well (plain launch, EDGE launch)
		const int k = which ? 3 : 0;
		FgsParams& f = which ? lp.edge : lp.fast;
		bool served[3];
		for (int c = 0; c < 3; c++) served[c] = kind[c] == k;
		place_fast_images(f, bi, fast_pad, served);
		if (f.fsmem + 64 > smem_limit) {
			for (int c = 0; c < 3; c++) if (kind[c] == k) { kind[c] = 2; served[c] = false; }
			place_fast_images(f, bi, fast_pad, served);
		}
	}
	// sign folding needs the negated copies of every bank a gather component reads, and room for them
	lp.gather_fold = ngather > 0;
	for (int c = 0; c < 3; c++) if (kind[c] == 1 && !bi.neg_ok[c ? 1 : 0]) lp.gather_fold = false;
	if (lp.gather_fold && kLutAlign + ngather * kLutBytes + bi.gbytes > smem_limit) lp.gather_fold = false;
#ifdef VFGS_GATHER_NO_FOLD
	lp.gather_fold = false; // build-time knob for experiments
#endif
	lp.gather_smem = kLutAlign + ngather * kLutBytes + (lp.gather_fold ? bi.gbytes : bi.bytes);
	if (ngather && lp.gather_smem > smem_limit) { // tables do not fit: those components take the general kernel
		for (int c = 0; c < 3; c++) if (kind[c] == 1) kind[c] = 2;
		ngather = 0; lp.gather_fold = false;
	}
	int gi = 0;
	for (int c = 0; c < 3; c++) {
		lp.gather.glut_index[c] = kind[c] == 1 ? gi++ : -1;
		if (kind[c] != 0) lp.fast.nseg[c] = 0;
		if (kind[c] != 1) lp.gather.nseg[c] = 0;
		if (kind[c] != 2) lp.general.nseg[c] = 0;
		if (kind[c] != 3) lp.edge.nseg[c] = 0;
		(kind[c] == 0 ? lp.any_fast : kind[c] == 1 ? lp.any_gather : kind[c] == 3 ? lp.any_edge : lp.any_general) = true;
	}
	// the fast kernel numbers its tasks over flat runs of lane units (process_task_fast); the EDGE launch has a partial
	// last unit per row where the width is not a multiple of 8
	for (int which = 0; which < 2; which++) {
		const int k = which ? 3 : 0;
		FgsParams& f = which ? lp.edge : lp.fast;
		f.ftasks_per_frame = 0;
		for (int c = 0; c < 3; c++) {
			// 16 samples per lane where the rows allow one access per line and lane (128-bit for 8-bit samples, 256-bit for 16-bit ones)
			const bool wide_on = f.in_bytes == 1 ? VFGS_FAST_WIDE8 != 0 : VFGS_FAST_WIDE16 != 0;
			f.fwide[c] = wide_on && kind[c] == 0 && k == 0 && f.comp[c].width % 16 == 0 &&
			             aligned_for(f.comp[c].in, f.comp[c].in_row_bytes, f.in_frame_bytes, (size_t)(16 * f.in_bytes)) &&
			             aligned_for(f.comp[c].out, f.comp[c].out_row_bytes, f.out_frame_bytes, (size_t)(16 * f.out_bytes));
			f.funits_per_row[c] = kind[c] == k ? (f.comp[c].width + (f.fwide[c] ? 16 : kSamplesPerLane) - 1) / (f.fwide[c] ? 16 : kSamplesPerLane) : 0;
			if (semi && c) { // the interleaved lane: one unit per chroma block of U and V (8 samples each), on component 1 only
				f.fwide[c] = c == 1 && kind[1] == k;
				f.funits_per_row[c] = f.fwide[c] ? f.comp[1].width / 8 : 0;
			}
			f.ftasks[c] = (f.funits_per_row[c] * f.rows + 31) / 32;
			f.ftasks_per_frame += f.ftasks[c];
			f.div_funits[c] = make_fastdiv((uint32_t)(f.funits_per_row[c] > 0 ? f.funits_per_row[c] : 1));
		}
		f.div_ftasks = make_fastdiv((uint32_t)(f.ftasks_per_frame > 0 ? f.ftasks_per_frame : 1));
		int served = 0, wide = 0;
		for (int c = 0; c < (semi ? 2 : 3); c++) if (kind[c] == k) { served++; wide += f.fwide[c] ? 1 : 0; }
		f.fallwide = served > 0 && wide == served;
	}
	lp.gather_shift = in_place && ngather > 0;
	lp.gather.ngather = ngather;
	lp.gather.gpat_off[0] = bi.pat_off[0]; lp.gather.gpat_off[1] = bi.pat_off[1];
	lp.gather.gneg_off[0] = bi.neg_off[0]; lp.gather.gneg_off[1] = bi.neg_off[1];
	lp.gather.gslot_mul[0] = (uint32_t)bi.pat_size[0]; lp.gather.gslot_mul[1] = (uint32_t)bi.pat_size[1];
	lp.gather.blob_bytes = lp.gather_fold ? bi.gbytes : bi.bytes;
	{ // the gather kernel numbers its tasks over flat runs of lane units as well (gather_task_body)
		FgsParams& g = lp.gather;
		g.gtasks_per_frame = 0;
		for (int c = 0; c < 3; c++) {
			const bool block8 = c && g.subx > 1;
			const int upr = kind[c] == 1 ? ((g.comp[c].width + kSamplesPerLane - 1) / kSamplesPerLane + 1) & ~1 : 0;
			const long long units = (long long)upr * g.rows;
			g.gunits_per_row[c] = upr;
			(void)block8;
			g.gtasks[c] = kind[c] != 1 ? 0 : (int)((units + (lp.gather_shift ? 1 : 0) + 31) / 32);
			g.gtasks_per_frame += g.gtasks[c];
			g.div_gunits[c] = make_fastdiv((uint32_t)(upr > 0 ? upr : 1));
		}
		g.div_gtasks = make_fastdiv((uint32_t)(g.gtasks_per_frame > 0 ? g.gtasks_per_frame : 1));
	}
	for (FgsParams* q : {&lp.fast, &lp.gather, &lp.general, &lp.edge}) {
		q->tasks_per_stripe = q->nseg[0] + q->nseg[1] + q->nseg[2];
		q->total_tasks = (long long)q->nframes * q->rows * q->tasks_per_stripe;
		q->div_tps = make_fastdiv((uint32_t)(q->tasks_per_stripe > 0 ? q->tasks_per_stripe : 1));
	}
	lp.fast.total_tasks = (long long)lp.fast.nframes * lp.fast.ftasks_per_frame;
	lp.edge.total_tasks = (long long)lp.edge.nframes * lp.edge.ftasks_per_frame;
	lp.gather.total_tasks = (long long)lp.gather.nframes * lp.gather.gtasks_per_frame;
}

// In place, a kernel must not read what another warp may already have overwritten. The fast kernel and the gather
// kernel's 16-sample-block lanes read nothing but their own samples; the general kernel (and the gather kernel's
// 8-sample-block halo lanes, which plan_launches therefore never uses in place) read a neighbouring block's INPUT
// sample when the pattern slot depends on the sample: those calls go through a scratch output buffer.
inline bool in_place_needs_scratch(const LaunchPlan& lp, const TableInfo& bi)
{
	for (int c = 0; c < 3; c++)
		if (lp.kind[c] == 2 && bi.uniform_pi[c] < 0) return true;
	return false;
}

// What lfsr_states_kernel needs to turn a block register into a pattern-window offset (FgsParams::woffs).
// Per component the entry has the format of the kernel that serves it:
//   fast    offset inside the fast image of the +pattern / -pattern copies (block sign folded in), there of the
//           copy shifted by ox % 8, + oy * stride + ox rounded down to 8
//   gather  oy * stride + ox inside a pattern slot, bit 15 set when the block sign is negative
struct WoffParams {
	WoffComp c[3];
};
inline WoffParams make_woff_params(const FgsParams& p, const int kind[3])
{
	WoffParams w;
	for (int c = 0; c < 3; c++) {
		const int stepx = (c && p.subx > 1) ? 2 : 4, stepy = (c && p.suby > 1) ? 2 : 4; // vfgs_hw.c:103-137
		WoffComp& k = w.c[c];
		if (kind[c] == 1) { // gather format
			k.off0 = 0; k.doff = 0x8000; k.ystride = stepy * p.pat_stride[c ? 1 : 0];
			k.copy = 0; k.kmask = 0; k.kshift = 0; k.xmul = stepx;
		} else {            // fast format: 2 copies (columns multiples of 4) or 4 (multiples of 2)
			k.off0 = p.fpat_off[c][0]; k.doff = p.fpat_off[c][1] - p.fpat_off[c][0]; k.ystride = stepy * p.fpat_stride[c];
			k.copy = p.fpat_copy[c]; k.kmask = stepx == 4 ? 1 : 3; k.kshift = stepx == 4 ? 1 : 2; k.xmul = 8;
		}
	}
	return w;
}

// ---- batched calls (vfgs_b200_add_grain_jobs_device) ------------------------------------------------
// One job of the job-table form of the LFSR stream kernel: its warps are [warp0, warp0 + nframes * R) of the launch.
struct StreamJob {
	long long warp0;
	uint32_t epoch; // the session's line_rnd at enqueue: frame 0 of the job
	int R, nb, spitch;
	uint32_t* states; // register table (null: not needed), window-offset table
	uint16_t* woffs;
	WoffParams wp;
};

// Launch block of the MULTI grain kernels: the per-job launch parameters of one kernel instantiation and the prefix of
// their task counts (task0[j] = first task of job j in the concatenation, task0[njobs] = total), in device memory.
struct MultiParams {
	const FgsParams* jobs;
	const long long* task0;
	int njobs;
	uint32_t* probe; // not null: the fast kernel only reports its shared-memory pad here (as FgsParams::probe)
};

// Static schedule of a MULTI launch: CTA b of `grid` takes the concatenated tasks [lo, hi), contiguous and in job order.
VFGS_HD void multi_cta_range(long long total, int grid, int b, long long& lo, long long& hi)
{
	lo = total * b / grid;
	hi = total * (b + 1) / grid;
}
// The job holding concatenated task t: the first j with task0[j + 1] > t (jobs without tasks are passed over).
VFGS_HD int multi_first_job(const long long* task0, int njobs, long long t)
{
	int lo = 0, hi = njobs - 1;
	while (lo < hi) {
		const int mid = (lo + hi) >> 1;
		if (task0[mid + 1] > t) hi = mid; else lo = mid + 1;
	}
	return lo;
}
// A CTA's walk over its range, one job at a time (the loop of the MULTI kernels and of the host replay in tests/emu):
// multi_next gives the next job j the range enters and the part [lo, end) of the range inside it; the CTA loads job j's
// tables, then its warps take tasks lo + k * warps + w below end (job-local index: task - task0[j]).
struct MultiCursor {
	long long lo, hi;
	int j;
};
VFGS_HD void multi_begin(const long long* task0, int njobs, int grid, int b, MultiCursor& c)
{
	multi_cta_range(task0[njobs], grid, b, c.lo, c.hi);
	c.j = multi_first_job(task0, njobs, c.lo);
}
VFGS_HD bool multi_next(const long long* task0, MultiCursor& c, int& j, long long& lo, long long& end)
{
	while (c.lo < c.hi) {
		const int k = c.j++;
		const long long e = task0[k + 1] < c.hi ? task0[k + 1] : c.hi;
		if (e <= c.lo) continue; // a job without tasks
		j = k; lo = c.lo; end = e;
		c.lo = e;
		return true;
	}
	return false;
}
// The job of warp `warp` of the job-table stream kernel: the last job whose first warp is <= warp (jobs without frames
// share warp0 with the next one).
VFGS_HD int stream_job_of(const StreamJob* jobs, int njobs, long long warp)
{
	int lo = 0, hi = njobs - 1;
	while (lo < hi) {
		const int mid = (lo + hi + 1) >> 1;
		if (jobs[mid].warp0 <= warp) lo = mid; else hi = mid - 1;
	}
	return lo;
}

// Which kernel instantiation serves a planned launch: the launches of the jobs of one call are grouped by this key.
// kind: 0 fast, 1 gather, 3 the fast kernel's EDGE variant (the general kernel is never batched).
//   fast  IN16 | OUT8 | ALLWIDE | SEMI   (the template flags of fgs_apply_fast_kernel)
//   gather IN16 | OUT8 | FOLD | SHIFT | MSB
inline int group_key(const FgsParams& p, int kind, bool fold, bool shift)
{
	const bool in16 = p.in_bytes == 2, out8 = p.out_bytes == 1;
	int k = kind | (in16 ? 4 : 0) | (out8 ? 8 : 0);
	if (kind == 0) k |= (in16 && !out8 && p.fallwide ? 16 : 0) | (p.ilv[1] ? 32 : 0);
	if (kind == 1) k |= (fold ? 64 : 0) | (shift ? 128 : 0) | (p.msb_in ? 256 : 0);
	return k;
}

// Registers after nframes whole frames of R block-rows of nb blocks (vfgs_hw.c:291-298,309-310 in closed form).
inline void advance_frames(HwState& h, int R, int nb, uint64_t nframes, const JumpTable& jt)
{
	if (!nframes) return;
	const uint32_t s0 = h.line_rnd;
	const uint64_t adv = nframes * (uint64_t)(R - 1) * (uint64_t)nb;
	if (R >= 2) {
		h.line_rnd_up = jt.jump(s0, adv - (uint64_t)nb);
		h.line_rnd = jt.jump(s0, adv);
	}
	h.rnd = jt.jump(h.line_rnd, (uint64_t)nb);
	h.rnd_up = jt.jump(h.line_rnd_up, (uint64_t)nb);
}

// The launches of a batched call: the planned launches of its jobs, grouped by group_key in order of first appearance,
// each group's jobs in list order, with the largest dynamic shared memory of its jobs' launches.
struct LaunchGroup {
	int key;
	std::vector<const FgsParams*> p;
	int smem;
};
inline void group_launches(const std::vector<const LaunchPlan*>& plans, std::vector<LaunchGroup>& groups)
{
	groups.clear();
	auto add = [&](const FgsParams& q, int kind, bool fold, bool shift, int smem) {
		const int key = group_key(q, kind, fold, shift);
		for (LaunchGroup& g : groups)
			if (g.key == key) {
				g.p.push_back(&q);
				if (smem > g.smem) g.smem = smem;
				return;
			}
		groups.push_back({key, {&q}, smem});
	};
	for (const LaunchPlan* lp : plans) {
		if (lp->any_fast) add(lp->fast, 0, false, false, lp->fast.fsmem);
		if (lp->any_edge) add(lp->edge, 3, false, false, lp->edge.fsmem);
		if (lp->any_gather) add(lp->gather, 1, lp->gather_fold, lp->gather_shift, lp->gather_smem);
	}
}

} // namespace vfgs
