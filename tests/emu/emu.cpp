// emu.cpp -- TEST TOOL, never part of the product library.
// Compiles the per-lane task code of the CUDA kernels (versatilefilmgrain_b200/csrc/fgs_task.h and
// fgs_fast.h) and the shim's table/parameter construction (vfgs_tables.h) with the HOST compiler and
// runs every (task, lane) pair serially, so the kernels' logic can be checked against the oracle in
// the GPU-less container before a GPU trip. What it cannot cover is covered by the -m gpu tests: the
// launch itself, the bulk copy, the LFSR stream kernel.
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

template <bool IN16, bool OUT8, bool EDGE, bool ALLWIDE = false>
void run_fast(const FgsParams& p, const uint8_t* lut)
{
	for (long long task = 0; task < p.total_tasks; task++)
		for (int lane = 0; lane < 32; lane++) process_task_fast<IN16, OUT8, EDGE, ALLWIDE>(p, smem_addr(lut), (uint32_t)task, lane);
}

// the gather task code exchanges grain values between lanes (warp shuffle on the device): every task runs twice,
// first recording what each lane sends, then replaying with the neighbours' values (fgs_gather.h, EmuWarp)
template <bool IN16, bool OUT8, bool FOLD, bool SHIFT>
void run_gather(const FgsParams& p, const uint8_t* luts, const uint8_t* img)
{
	for (long long task = 0; task < p.total_tasks; task++)
		for (int pass = 0; pass < 2; pass++) {
			emu_warp().record = pass == 0;
			for (int lane = 0; lane < 32; lane++)
				process_task_gather<IN16, OUT8, FOLD, SHIFT>(p, smem_addr(luts), smem_addr(img), (uint32_t)task, lane);
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

extern "C" int emu_state_size(void) { return (int)sizeof(StateDump); }
// lane-lines of the gather task code that took the uniform-slot octet path since the last call (fgs_gather.h)
extern "C" long long emu_octet_lines(void) { const long long v = emu_warp().octet_lines; emu_warp().octet_lines = 0; return v; }

// Packed planar frames, whole frames, like vfgs_b200_add_grain_frames_device.
// mode: 0 automatic kernel choice, 1 general task code everywhere, 2 gather task code wherever it can
// run (plan_launches). Returns a bit mask: 1 = fast, 2 = general, 4 = gather task code ran, 8 = with sign-folded slot copies, 16 = with the shifted unit numbering (in place),
// 32 = the fast task code's EDGE variant ran (ragged / unaligned rows).
extern "C" int emu_add_grain_frames(const void* state, const void* in, void* out, int nframes, int width,
                                    int height, int out_depth, int first_frame_index, int mode)
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

	const int in_depth = 8 + h.bs;
	if (!out_depth) out_depth = in_depth;
	const int cw = width / h.csubx, ch = height / h.csuby;
	const int nb = (width + 15) / 16, R = (height + 15) / 16, spitch = nb + 2;
	const size_t isz = in_depth > 8 ? 2 : 1, osz = out_depth > 8 ? 2 : 1;
	const size_t ysam = (size_t)width * height, csam = (size_t)cw * ch;

	TableInfo bi;
	std::vector<uint8_t> blob, fblob;
	build_tables(h, bi, blob, fblob);

	// "shared memory" of the two kernels (the fast kernel's LUT on a 32 KB boundary, like on the device)
	std::vector<uint32_t> tab_store((blob.size() + 64) / 4);
	uint8_t* tab = (uint8_t*)tab_store.data();
	memcpy(tab, blob.data(), (size_t)bi.bytes); // the general kernel copies the image without the negated slot copies
	// the fast kernel's shared window: LUTs on a 32 KB boundary, dynamic shared memory starting kEmuPad bytes
	// in front of it (1 KB reserved by the driver + 128 B of static variables on the device)
	constexpr int kEmuPad = kLutAlign - 1152;
	std::vector<uint8_t> smem_store((size_t)2 * kLutAlign + 3 * kLutBytes + fblob.size() + 64);
	uint8_t* lut_ptr = (uint8_t*)(((uintptr_t)smem_store.data() + 2 * kLutAlign - 1) & ~(uintptr_t)(kLutAlign - 1));

	// per-block LFSR registers (what lfsr_states_kernel produces)
	std::vector<uint32_t> states((size_t)nframes * R * spitch, 0);
	for (int f = 0; f < nframes; f++)
		for (int r = 0; r < R; r++) {
			uint64_t t = ((uint64_t)(first_frame_index + f) * (uint64_t)(R - 1) + (uint64_t)r) * (uint64_t)nb;
			uint32_t s = jt.jump(h.line_rnd, t);
			for (int b = 0; b < nb; b++) { states[((size_t)f * R + r) * spitch + 1 + b] = s; s = lfsr_step(s); }
		}

	FgsParams p;
	memset(&p, 0, sizeof(p));
	fill_state_params(p, h, bi);
	std::vector<uint16_t> woffs(states.size() * 4, 0);
	p.woffs = woffs.data();
	p.nframes = nframes; p.nb = nb; p.R = R; p.row_begin = 0; p.rows = R;
	p.y_begin = 0; p.y_end = height;
	p.in_bytes = (int)isz; p.out_bytes = (int)osz;
	p.in_frame_bytes = (long long)((ysam + 2 * csam) * isz);
	p.out_frame_bytes = (long long)((ysam + 2 * csam) * osz);
	const size_t off[3] = {0, ysam, ysam + csam};
	for (int c = 0; c < 3; c++) {
		p.comp[c].in = (const uint8_t*)in + off[c] * isz;
		p.comp[c].out = (uint8_t*)out + off[c] * osz;
		p.comp[c].in_row_bytes = (long long)((c ? cw : width) * isz);
		p.comp[c].out_row_bytes = (long long)((c ? cw : width) * osz);
		p.comp[c].width = c ? cw : width;
		p.comp[c].lines = c ? ch : height;
	}
	p.states = states.data(); p.spitch = spitch; p.stream_rows = R; p.stream_row0 = 0;
	finish_tasks(p);

	LaunchPlan lp;
	plan_launches(p, bi, mode, in == out, 227 * 1024, kEmuPad, lp);
	{ // window offsets of every block (the second table lfsr_states_kernel writes), in the serving kernel's format
		const WoffParams wp = make_woff_params(p, lp.kind);
		for (size_t i = 0; i < states.size(); i++)
		{
			woffs[i * 4 + 0] = (uint16_t)window_offset<0>(states[i], wp.c[0]);
			woffs[i * 4 + 1] = (uint16_t)window_offset<1>(states[i], wp.c[1]);
			woffs[i * 4 + 2] = (uint16_t)window_offset<2>(states[i], wp.c[2]);
		}
	}
	if (lp.any_fast) { // what fgs_apply_fast_kernel builds in shared memory
		const FgsParams& f = lp.fast;
		f_check(f.fpad == kEmuPad && f.fsmem <= kEmuPad + 3 * kLutBytes + (int)fblob.size());
		for (int c = 0; c < 3; c++)
			if (f.fimg_bytes[c]) memcpy(lut_ptr + f.fimg_off[c], fblob.data() + f.fimg_src[c], (size_t)f.fimg_bytes[c]);
		expand_fast_luts((uint32_t*)lut_ptr, (const uint32_t*)fblob.data(), (uint32_t)(1 << (16 - h.scale_shift)), 0, 1);
		if (isz == 1) run_fast<false, false, false>(f, lut_ptr);
		else if (osz == 1) run_fast<true, true, false>(f, lut_ptr);
		else if (f.fallwide) run_fast<true, false, false, true>(f, lut_ptr); // the ALLWIDE kernel variant, like launch_apply
		else run_fast<true, false, false>(f, lut_ptr);
	}
	if (lp.any_edge) { // the EDGE launch of the fast kernel: same shared-memory image, its own components
		const FgsParams& f = lp.edge;
		f_check(f.fpad == kEmuPad && f.fsmem <= kEmuPad + 3 * kLutBytes + (int)fblob.size());
		for (int c = 0; c < 3; c++)
			if (f.fimg_bytes[c]) memcpy(lut_ptr + f.fimg_off[c], fblob.data() + f.fimg_src[c], (size_t)f.fimg_bytes[c]);
		expand_fast_luts((uint32_t*)lut_ptr, (const uint32_t*)fblob.data(), (uint32_t)(1 << (16 - h.scale_shift)), 0, 1);
		if (isz == 1) run_fast<false, false, true>(f, lut_ptr);
		else if (osz == 1) run_fast<true, true, true>(f, lut_ptr);
		else run_fast<true, false, true>(f, lut_ptr);
	}
	if (lp.any_gather) {
		// what fgs_apply_gather_kernel builds in shared memory: one private LUT per gather component, then the image
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
		if (lp.gather_fold) { if (lp.gather_shift) run_gather_any<true, true>(g, isz, osz, gl, gi); else run_gather_any<true, false>(g, isz, osz, gl, gi); }
		else { if (lp.gather_shift) run_gather_any<false, true>(g, isz, osz, gl, gi); else run_gather_any<false, false>(g, isz, osz, gl, gi); }
	}
	if (lp.any_general)
		for (long long task = 0; task < lp.general.total_tasks; task++)
			for (int lane = 0; lane < 32; lane++) process_task(lp.general, tab, (uint32_t)task, lane);
	return (lp.any_fast ? 1 : 0) | (lp.any_general ? 2 : 0) | (lp.any_gather ? 4 : 0) | (lp.any_gather && lp.gather_fold ? 8 : 0) | (lp.any_gather && lp.gather_shift ? 16 : 0) | (lp.any_edge ? 32 : 0) |
	       (lp.any_fast && (lp.fast.fwide[0] || lp.fast.fwide[1] || lp.fast.fwide[2]) ? 64 : 0);
}

// Launch planning of a whole-frame call, without running anything (host logic only): which kernel serves each
// component, the fast kernel's shared-memory layout and lane-unit width. out (ints): kind[3], fsmem, fpad,
// fimg_off[3], fimg_bytes[3], fwide[3], funits_per_row[3], gather_smem, fallwide, warp-tasks per frame of the fast,
// EDGE, gather and general launches, gather_fold, gather_shift, EDGE funits_per_row[3], gather gunits_per_row[3]
// (31 ints).
extern "C" void emu_plan(const void* state, int width, int height, int out_depth, int in_place, int mode, int* out)
{
	const StateDump& d = *(const StateDump*)state;
	HwState h;
	memcpy(h.pattern, d.pattern, sizeof(h.pattern));
	memcpy(h.slut, d.slut, sizeof(h.slut));
	memcpy(h.plut, d.plut, sizeof(h.plut));
	h.rnd = d.rnd; h.rnd_up = d.rnd_up; h.line_rnd = d.line_rnd; h.line_rnd_up = d.line_rnd_up;
	h.scale_shift = d.scale_shift; h.bs = d.bs;
	h.y_min = d.y_min; h.y_max = d.y_max; h.c_min = d.c_min; h.c_max = d.c_max;
	h.csubx = d.csubx; h.csuby = d.csuby;
	const int in_depth = 8 + h.bs;
	if (!out_depth) out_depth = in_depth;
	const int cw = width / h.csubx, ch = height / h.csuby;
	const size_t isz = in_depth > 8 ? 2 : 1, osz = out_depth > 8 ? 2 : 1;
	const size_t ysam = (size_t)width * height, csam = (size_t)cw * ch;
	TableInfo bi;
	std::vector<uint8_t> blob, fblob;
	build_tables(h, bi, blob, fblob);
	FgsParams p;
	memset(&p, 0, sizeof(p));
	fill_state_params(p, h, bi);
	p.nframes = 1; p.nb = (width + 15) / 16; p.R = (height + 15) / 16; p.row_begin = 0; p.rows = p.R;
	p.y_begin = 0; p.y_end = height;
	p.in_bytes = (int)isz; p.out_bytes = (int)osz;
	p.in_frame_bytes = (long long)((ysam + 2 * csam) * isz);
	p.out_frame_bytes = (long long)((ysam + 2 * csam) * osz);
	static uint8_t* const base_in = (uint8_t*)0x10000000, * const base_out = (uint8_t*)0x40000000; // aligned dummies, never dereferenced
	const size_t off[3] = {0, ysam, ysam + csam};
	for (int c = 0; c < 3; c++) {
		p.comp[c].in = base_in + off[c] * isz;
		p.comp[c].out = (in_place ? base_in : base_out) + off[c] * osz;
		p.comp[c].in_row_bytes = (long long)((c ? cw : width) * isz);
		p.comp[c].out_row_bytes = (long long)((c ? cw : width) * osz);
		p.comp[c].width = c ? cw : width;
		p.comp[c].lines = c ? ch : height;
	}
	p.spitch = p.nb + 2; p.stream_rows = p.R;
	finish_tasks(p);
	LaunchPlan lp;
	plan_launches(p, bi, mode, in_place != 0, 227 * 1024, kLutAlign - 1152, lp);
	int k = 0;
	for (int c = 0; c < 3; c++) out[k++] = lp.kind[c];
	out[k++] = lp.fast.fsmem; out[k++] = lp.fast.fpad;
	for (int c = 0; c < 3; c++) out[k++] = lp.fast.fimg_off[c];
	for (int c = 0; c < 3; c++) out[k++] = lp.fast.fimg_bytes[c];
	for (int c = 0; c < 3; c++) out[k++] = lp.fast.fwide[c];
	for (int c = 0; c < 3; c++) out[k++] = lp.fast.funits_per_row[c];
	out[k++] = lp.gather_smem;
	out[k++] = lp.fast.fallwide;
	// warp-tasks of one frame per launch: fast, EDGE, gather, general
	out[k++] = lp.fast.ftasks_per_frame; out[k++] = lp.edge.ftasks_per_frame; out[k++] = lp.gather.gtasks_per_frame;
	out[k++] = lp.general.rows * lp.general.tasks_per_stripe;
	out[k++] = lp.gather_fold; out[k++] = lp.gather_shift;
	for (int c = 0; c < 3; c++) out[k++] = lp.edge.funits_per_row[c];
	for (int c = 0; c < 3; c++) out[k++] = lp.gather.gunits_per_row[c];
}

// ---- firmware layer (fw_host.h + fw_device.h run with one host thread) ---------------------------
#include "../../versatilefilmgrain_b200/csrc/fw_host.h"

// What vfgs_b200_init_sei / vfgs_b200_init_afgs1 do, on a freshly powered-on hardware state with the given depth and
// chroma subsampling (vfgs_main.c:750-757); the setters' arithmetic is restated from vfgs_hw.c:339-380 (test tool).
// cfg: raw fgs_sei / fgs_afgs1 bytes. state_out: StateDump. Returns 0, or 1 where the reference asserts.
extern "C" int emu_fw_init(const void* cfg, int is_afgs1, int depth, int csubx, int csuby, void* state_out)
{
	static HwState h; // 73 KB
	h.power_on();
	const int nbs = depth - 8;
	h.scale_shift = (h.scale_shift + h.bs - nbs) & 0xff; h.bs = nbs; // vfgs_set_depth
	h.csubx = csubx; h.csuby = csuby;
	FwPlan plan;
	if (is_afgs1) fw_plan_afgs1(*(const fgs_afgs1*)cfg, csubx, csuby, plan);
	else fw_plan_sei(*(const fgs_sei*)cfg, csubx, csuby, plan);
	if (plan.error) return 1;
	static FwTables tables;
	static bool have_tables = false;
	if (!have_tables) { make_fw_tables(tables); have_tables = true; }
	static FwScratch scratch;
	memset(&scratch, 0, sizeof(scratch));
	for (const FwJob& j : plan.jobs) fw_run_job_serial(j, tables, scratch, &h.pattern[0][0][0][0]);
	memcpy(h.slut, plan.slut, sizeof(h.slut));
	memcpy(h.plut, plan.plut, sizeof(h.plut));
	if (plan.set_seed) h.rnd = h.rnd_up = h.line_rnd = h.line_rnd_up = plan.seed << 1;
	if (plan.scale_shift < 2 || plan.scale_shift >= 8) return 1; // vfgs_hw.c:348
	h.scale_shift = plan.scale_shift + 6 - h.bs;
	if (plan.set_legal) { h.y_min = h.c_min = plan.legal ? 16 : 0; h.y_max = plan.legal ? 235 : 255; h.c_max = plan.legal ? 240 : 255; }
	StateDump& d = *(StateDump*)state_out;
	memcpy(d.pattern, h.pattern, sizeof(d.pattern));
	memcpy(d.slut, h.slut, sizeof(d.slut));
	memcpy(d.plut, h.plut, sizeof(d.plut));
	d.rnd = h.rnd; d.rnd_up = h.rnd_up; d.line_rnd = h.line_rnd; d.line_rnd_up = h.line_rnd_up;
	d.scale_shift = h.scale_shift; d.bs = h.bs; d.y_min = h.y_min; d.y_max = h.y_max; d.c_min = h.c_min; d.c_max = h.c_max;
	d.csubx = h.csubx; d.csuby = h.csuby;
	return 0;
}

extern "C" void emu_fw_tables(int8_t* gauss, int8_t* dct)
{
	FwTables t;
	make_fw_tables(t);
	memcpy(gauss, t.gauss, sizeof(t.gauss));
	memcpy(dct, t.dct, sizeof(t.dct));
}
