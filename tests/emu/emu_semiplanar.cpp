// emu_semiplanar.cpp -- TEST TOOL, never part of the product library.
// Host build of the semi-planar (NV12 / P010) form of the kernels' task code: the fast kernel's SEMI variants (interleaved
// U/V lane, MSB-aligned wide luma), the gather kernel's MSB variants and the general task code with its sample step, run
// lane by lane like emu.cpp does for planar frames, with the shim's planner (vfgs_tables.h). What it cannot cover -- the
// launch, the bulk copies, the LFSR stream kernel -- the -m gpu tests cover (tests/test_gpu_semiplanar.py).
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "../../versatilefilmgrain_b200/csrc/vfgs_tables.h"

using namespace vfgs;

namespace {
void f_check(bool ok) { if (!ok) abort(); }
struct StateDump { // == refh_state / oracle_dump
	int8_t pattern[2][9][64][64];
	uint8_t slut[3][256];
	uint8_t plut[3][256];
	uint32_t rnd, rnd_up, line_rnd, line_rnd_up;
	int scale_shift, bs, y_min, y_max, c_min, c_max, csubx, csuby;
};

template <bool IN16, bool OUT8, bool EDGE, bool ALLWIDE = false, bool SEMI = false>
void run_fast(const FgsParams& p, const uint8_t* lut)
{
	for (long long task = 0; task < p.total_tasks; task++)
		for (int lane = 0; lane < 32; lane++) process_task_fast<IN16, OUT8, EDGE, ALLWIDE, SEMI>(p, smem_addr(lut), (uint32_t)task, lane);
}

// the gather task code exchanges grain values between lanes: every task runs twice, recording, then replaying (emu.cpp)
template <bool IN16, bool OUT8, bool FOLD, bool SHIFT, bool MSB = false>
void run_gather(const FgsParams& p, const uint8_t* luts, const uint8_t* img)
{
	for (long long task = 0; task < p.total_tasks; task++)
		for (int pass = 0; pass < 2; pass++) {
			emu_warp().record = pass == 0;
			for (int lane = 0; lane < 32; lane++)
				process_task_gather<IN16, OUT8, FOLD, SHIFT, MSB>(p, smem_addr(luts), smem_addr(img), (uint32_t)task, lane);
		}
}
template <bool FOLD, bool SHIFT>
void run_gather_any(const FgsParams& g, size_t isz, size_t osz, const uint8_t* gl, const uint8_t* gi)
{
	if (isz == 1) run_gather<false, false, FOLD, SHIFT>(g, gl, gi);
	else if (osz == 1) run_gather<true, true, FOLD, SHIFT>(g, gl, gi);
	else run_gather<true, false, FOLD, SHIFT>(g, gl, gi);
}
} // namespace

extern "C" int emus_state_size(void) { return (int)sizeof(StateDump); }

// Semi-planar frames (NV12 / P010), whole frames, like vfgs_b200_add_grain_semiplanar_device: luma plane y (stride sy), then
// one plane of interleaved U,V pairs (stride suv), frames fs bytes apart, for input and output. p010_in / p010_out: 16-bit
// samples in bits 15..6 (the input format must match the state's depth; the caller checks formats). In place (same
// pointers) with a plan that reads neighbours' input samples goes through a packed scratch buffer, like the library.
// Returns the mask of emu_add_grain_frames (emu.cpp) plus 128 = the fast task code's interleaved U/V lane ran.
extern "C" int emu_add_grain_semiplanar(const void* state, const void* y_in, const void* uv_in, long long sy_in, long long suv_in,
                                        long long fs_in, void* y_out, void* uv_out, long long sy_out, long long suv_out, long long fs_out,
                                        int nframes, int width, int height, int p010_out, int first_frame_index, int mode)
{
	const StateDump& d = *(const StateDump*)state;
	static const JumpTable jt;
	HwState h;
	memcpy(h.pattern, d.pattern, sizeof(h.pattern));
	memcpy(h.slut, d.slut, sizeof(h.slut));
	memcpy(h.plut, d.plut, sizeof(h.plut));
	h.rnd = d.rnd; h.rnd_up = d.rnd_up; h.line_rnd = d.line_rnd; h.line_rnd_up = d.line_rnd_up;
	h.scale_shift = d.scale_shift; h.bs = d.bs;
	h.y_min = d.y_min; h.y_max = d.y_max; h.c_min = d.c_min; h.c_max = d.c_max;
	h.csubx = d.csubx; h.csuby = d.csuby;
	f_check(h.csubx == 2);
	const bool p010_in = h.bs == 2;
	const size_t isz = p010_in ? 2 : 1, osz = p010_out ? 2 : 1;
	const int cw = width / h.csubx, ch = height / h.csuby;
	const int nb = (width + 15) / 16, R = (height + 15) / 16, spitch = nb + 2;

	TableInfo bi;
	std::vector<uint8_t> blob, fblob;
	build_tables(h, bi, blob, fblob);
	std::vector<uint32_t> tab_store((blob.size() + 64) / 4);
	uint8_t* tab = (uint8_t*)tab_store.data();
	memcpy(tab, blob.data(), (size_t)bi.bytes);
	constexpr int kEmuPad = kLutAlign - 1152;
	std::vector<uint8_t> smem_store((size_t)2 * kLutAlign + 3 * kLutBytes + fblob.size() + 64);
	uint8_t* lut_ptr = (uint8_t*)(((uintptr_t)smem_store.data() + 2 * kLutAlign - 1) & ~(uintptr_t)(kLutAlign - 1));
	std::vector<uint32_t> states((size_t)nframes * R * spitch, 0);
	for (int f = 0; f < nframes; f++)
		for (int r = 0; r < R; r++) {
			uint64_t t = ((uint64_t)(first_frame_index + f) * (uint64_t)(R - 1) + (uint64_t)r) * (uint64_t)nb;
			uint32_t s = jt.jump(h.line_rnd, t);
			for (int b = 0; b < nb; b++) { states[((size_t)f * R + r) * spitch + 1 + b] = s; s = lfsr_step(s); }
		}
	std::vector<uint16_t> woffs(states.size() * 4, 0);

	auto plan = [&](uint8_t* yo, uint8_t* uvo, long long syo, long long suvo, long long fso, bool in_place, FgsParams& p, LaunchPlan& lp) {
		memset(&p, 0, sizeof(p));
		fill_state_params(p, h, bi);
		p.woffs = woffs.data();
		p.nframes = nframes; p.nb = nb; p.R = R; p.row_begin = 0; p.rows = R;
		p.y_begin = 0; p.y_end = height;
		p.in_bytes = (int)isz; p.out_bytes = (int)osz;
		p.in_frame_bytes = fs_in; p.out_frame_bytes = fso;
		set_semiplanar_planes(p, (const uint8_t*)y_in, (const uint8_t*)uv_in, sy_in, suv_in, yo, uvo, syo, suvo, width, height, cw, ch,
		                      p010_in, p010_out != 0);
		p.states = states.data(); p.spitch = spitch; p.stream_rows = R; p.stream_row0 = 0;
		finish_tasks(p);
		plan_launches(p, bi, mode, in_place, 227 * 1024, kEmuPad, lp);
	};
	const bool in_place = y_in == y_out;
	FgsParams p;
	LaunchPlan lp;
	plan((uint8_t*)y_out, (uint8_t*)uv_out, sy_out, suv_out, fs_out, in_place, p, lp);
	std::vector<uint8_t> scratch;
	const size_t yrow = (size_t)width * osz, uvrow = (size_t)2 * cw * osz, sfb = yrow * height + uvrow * ch;
	const bool use_scratch = in_place && in_place_needs_scratch(lp, bi);
	if (use_scratch) { // packed scratch output frames, copied back below
		scratch.assign(sfb * nframes, 0);
		plan(scratch.data(), scratch.data() + yrow * height, (long long)yrow, (long long)uvrow, (long long)sfb, false, p, lp);
	}
	{
		const WoffParams wp = make_woff_params(p, lp.kind);
		for (size_t i = 0; i < states.size(); i++) {
			woffs[i * 4 + 0] = (uint16_t)window_offset<0>(states[i], wp.c[0]);
			woffs[i * 4 + 1] = (uint16_t)window_offset<1>(states[i], wp.c[1]);
			woffs[i * 4 + 2] = (uint16_t)window_offset<2>(states[i], wp.c[2]);
		}
	}
	if (lp.any_fast) { // the SEMI variants of the fast kernel
		const FgsParams& f = lp.fast;
		f_check(f.fpad == kEmuPad && f.fsmem <= kEmuPad + 3 * kLutBytes + (int)fblob.size());
		for (int c = 0; c < 3; c++)
			if (f.fimg_bytes[c]) memcpy(lut_ptr + f.fimg_off[c], fblob.data() + f.fimg_src[c], (size_t)f.fimg_bytes[c]);
		expand_fast_luts((uint32_t*)lut_ptr, (const uint32_t*)fblob.data(), (uint32_t)(1 << (16 - h.scale_shift)), 0, 1);
		if (isz == 1) run_fast<false, false, false, false, true>(f, lut_ptr);
		else if (osz == 1) run_fast<true, true, false, false, true>(f, lut_ptr);
		else if (f.fallwide) run_fast<true, false, false, true, true>(f, lut_ptr);
		else run_fast<true, false, false, false, true>(f, lut_ptr);
	}
	if (lp.any_edge) { // 8-bit luma that is not wide: the planar EDGE variant
		const FgsParams& f = lp.edge;
		for (int c = 0; c < 3; c++)
			if (f.fimg_bytes[c]) memcpy(lut_ptr + f.fimg_off[c], fblob.data() + f.fimg_src[c], (size_t)f.fimg_bytes[c]);
		expand_fast_luts((uint32_t*)lut_ptr, (const uint32_t*)fblob.data(), (uint32_t)(1 << (16 - h.scale_shift)), 0, 1);
		f_check(isz == 1);
		run_fast<false, false, true>(f, lut_ptr);
	}
	if (lp.any_gather) {
		const FgsParams& g = lp.gather;
		std::vector<uint8_t> gstore((size_t)kLutAlign + (size_t)g.ngather * kLutBytes + blob.size() + 64);
		uint8_t* gl = (uint8_t*)(((uintptr_t)gstore.data() + kLutAlign - 1) & ~(uintptr_t)(kLutAlign - 1));
		uint8_t* gi = gl + (size_t)g.ngather * kLutBytes;
		memcpy(gi, blob.data(), blob.size());
		for (int c = 0; c < 3; c++) {
			if (g.glut_index[c] < 0) continue;
			const uint16_t* compact = (const uint16_t*)(gi + g.lut_off) + c * 256;
			uint32_t* lut = (uint32_t*)(gl + (size_t)g.glut_index[c] * kLutBytes);
			const uint32_t slot_bytes = (uint32_t)g.pat_size[c ? 1 : 0];
			for (int i = 0; i < 256 * 32; i++)
				lut[i] = isz == 2 ? gather_lut_entry<true>(compact[i >> 5], slot_bytes) : gather_lut_entry<false>(compact[i >> 5], slot_bytes);
		}
		if (isz == 1) { // NV12 luma: the planar gather kernel
			if (lp.gather_fold) { if (lp.gather_shift) run_gather_any<true, true>(g, isz, osz, gl, gi); else run_gather_any<true, false>(g, isz, osz, gl, gi); }
			else { if (lp.gather_shift) run_gather_any<false, true>(g, isz, osz, gl, gi); else run_gather_any<false, false>(g, isz, osz, gl, gi); }
		} else if (osz == 1) { // P010 luma: the MSB variants
			if (lp.gather_fold) { if (lp.gather_shift) run_gather<true, true, true, true, true>(g, gl, gi); else run_gather<true, true, true, false, true>(g, gl, gi); }
			else { if (lp.gather_shift) run_gather<true, true, false, true, true>(g, gl, gi); else run_gather<true, true, false, false, true>(g, gl, gi); }
		} else {
			if (lp.gather_fold) { if (lp.gather_shift) run_gather<true, false, true, true, true>(g, gl, gi); else run_gather<true, false, true, false, true>(g, gl, gi); }
			else { if (lp.gather_shift) run_gather<true, false, false, true, true>(g, gl, gi); else run_gather<true, false, false, false, true>(g, gl, gi); }
		}
	}
	if (lp.any_general)
		for (long long task = 0; task < lp.general.total_tasks; task++)
			for (int lane = 0; lane < 32; lane++) process_task(lp.general, tab, (uint32_t)task, lane);
	if (use_scratch)
		for (int f = 0; f < nframes; f++) {
			const uint8_t* s = scratch.data() + (size_t)f * sfb;
			for (int r = 0; r < height; r++) memcpy((uint8_t*)y_out + f * fs_out + r * sy_out, s + r * yrow, yrow);
			for (int r = 0; r < ch; r++) memcpy((uint8_t*)uv_out + f * fs_out + r * suv_out, s + yrow * height + r * uvrow, uvrow);
		}
	return (lp.any_fast ? 1 : 0) | (lp.any_general ? 2 : 0) | (lp.any_gather ? 4 : 0) | (lp.any_gather && lp.gather_fold ? 8 : 0) |
	       (lp.any_gather && lp.gather_shift ? 16 : 0) | (lp.any_edge ? 32 : 0) | (lp.any_fast && (lp.fast.fwide[0] || lp.fast.fwide[1]) ? 64 : 0) |
	       (lp.any_fast && lp.fast.fwide[1] ? 128 : 0);
}
