// emu_jobs.cpp -- TEST TOOL, never part of the product library.
// Host build of a batched call (vfgs_b200_add_grain_jobs_device) with the shim's own planning and grouping code
// (vfgs_tables.h: plan_launches, group_key / group_launches, advance_frames) and the kernels' own schedule and job
// lookup (multi_begin / multi_next, stream_job_of):
//   * every job is planned against its session's state; jobs the single-job route serves (general kernel, in-place
//     scratch detour) are reported and left to the single-job emulators (emu.cpp, emu_semiplanar.cpp);
//   * the window-offset tables of the batched jobs come from one walk over the warps of the job-table stream kernel;
//   * each group is replayed CTA by CTA: one "shared memory" buffer per CTA, kept across its job switches, into which
//     every switch copies that job's images and re-expands its LUTs; the task code then runs lane by lane.
// What it cannot cover -- the launches, the bulk copies, the device build of the code -- the -m gpu tests cover
// (tests/test_gpu_sessions.py).
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
// the fast kernel's shared window on the device: dynamic shared memory starts this far in front of a 32 KB boundary
constexpr int kEmuPad = kLutAlign - 1152;

struct Session {
	HwState h;
	TableInfo bi;
	std::vector<uint8_t> blob, fblob;
};

template <bool IN16, bool OUT8, bool EDGE, bool ALLWIDE, bool SEMI>
void fast_task(const FgsParams& p, const uint8_t* lut, uint32_t task)
{
	for (int lane = 0; lane < 32; lane++) process_task_fast<IN16, OUT8, EDGE, ALLWIDE, SEMI>(p, smem_addr(lut), task, lane);
}
// the instantiation fgs_apply_fast_multi_kernel takes for a group key (vfgs_b200.cu, multi_kernel)
void fast_task_of(int key, const FgsParams& p, const uint8_t* lut, uint32_t task)
{
	const bool in16 = key & 4, out8 = key & 8, allwide = key & 16, semi = key & 32, edge = (key & 3) == 3;
	if (edge) {
		if (!in16) fast_task<false, false, true, false, false>(p, lut, task);
		else if (out8) fast_task<true, true, true, false, false>(p, lut, task);
		else fast_task<true, false, true, false, false>(p, lut, task);
	} else if (semi) {
		if (allwide) fast_task<true, false, false, true, true>(p, lut, task);
		else if (!in16) fast_task<false, false, false, false, true>(p, lut, task);
		else if (out8) fast_task<true, true, false, false, true>(p, lut, task);
		else fast_task<true, false, false, false, true>(p, lut, task);
	} else if (allwide) {
		fast_task<true, false, false, true, false>(p, lut, task);
	} else if (!in16) {
		fast_task<false, false, false, false, false>(p, lut, task);
	} else if (out8) {
		fast_task<true, true, false, false, false>(p, lut, task);
	} else {
		fast_task<true, false, false, false, false>(p, lut, task);
	}
}

// the gather task code exchanges grain values between lanes: every task runs twice, recording, then replaying (emu.cpp)
template <bool IN16, bool OUT8, bool FOLD, bool SHIFT, bool MSB>
void gather_task(const FgsParams& p, const uint8_t* luts, const uint8_t* img, uint32_t task)
{
	for (int pass = 0; pass < 2; pass++) {
		emu_warp().record = pass == 0;
		for (int lane = 0; lane < 32; lane++) process_task_gather<IN16, OUT8, FOLD, SHIFT, MSB>(p, smem_addr(luts), smem_addr(img), task, lane);
	}
}
template <bool FOLD, bool SHIFT>
void gather_io(bool in16, bool out8, bool msb, const FgsParams& p, const uint8_t* luts, const uint8_t* img, uint32_t task)
{
	if (msb) {
		if (out8) gather_task<true, true, FOLD, SHIFT, true>(p, luts, img, task);
		else gather_task<true, false, FOLD, SHIFT, true>(p, luts, img, task);
	} else if (!in16) {
		gather_task<false, false, FOLD, SHIFT, false>(p, luts, img, task);
	} else if (out8) {
		gather_task<true, true, FOLD, SHIFT, false>(p, luts, img, task);
	} else {
		gather_task<true, false, FOLD, SHIFT, false>(p, luts, img, task);
	}
}
void gather_task_of(int key, const FgsParams& p, const uint8_t* luts, const uint8_t* img, uint32_t task)
{
	const bool in16 = key & 4, out8 = key & 8, fold = key & 64, shift = key & 128, msb = key & 256;
	if (fold) { if (shift) gather_io<true, true>(in16, out8, msb, p, luts, img, task); else gather_io<true, false>(in16, out8, msb, p, luts, img, task); }
	else { if (shift) gather_io<false, true>(in16, out8, msb, p, luts, img, task); else gather_io<false, false>(in16, out8, msb, p, luts, img, task); }
}
} // namespace

extern "C" int emuj_state_size(void) { return (int)sizeof(StateDump); }

// One job of a batched call. Planar jobs: packed frames at in_y / out_y (the other fields unused), out_depth as in
// vfgs_b200_add_grain_planes_device. Semi-planar jobs: Y and UV planes with their strides and the frame stride;
// out_depth 8 = NV12 output from P010 input, else the input format.
struct EmuJob {
	int session, semi, nframes, width, height, out_depth;
	const uint8_t* in_y;
	const uint8_t* in_uv;
	long long sy_in, suv_in, fs_in;
	uint8_t* out_y;
	uint8_t* out_uv;
	long long sy_out, suv_out, fs_out;
};

// states: nsess state dumps (registers included), the sessions' states at the call. mode: kernel selection as
// vfgs_b200_force_general_kernel. grid / warps: persistent grid and warps per CTA of every replayed launch.
// Outputs: regs (nsess x 4) the sessions' registers afterwards; batched[k] 1 when job k went to the MULTI launches;
// keys (up to 16) the group keys of the grain launches in launch order. Returns the number of grain launches, or -1
// when a job's plan was not what the shim would accept.
extern "C" int emuj_run_jobs(const void* states, int nsess, const EmuJob* jobs, int njobs, int mode, int grid, int warps,
                             uint32_t* regs, int* batched, int* keys)
{
	static const JumpTable jt;
	std::vector<Session> S((size_t)nsess);
	for (int k = 0; k < nsess; k++) {
		const StateDump& d = ((const StateDump*)states)[k];
		HwState& h = S[k].h;
		memcpy(h.pattern, d.pattern, sizeof(h.pattern));
		memcpy(h.slut, d.slut, sizeof(h.slut));
		memcpy(h.plut, d.plut, sizeof(h.plut));
		h.rnd = d.rnd; h.rnd_up = d.rnd_up; h.line_rnd = d.line_rnd; h.line_rnd_up = d.line_rnd_up;
		h.scale_shift = d.scale_shift; h.bs = d.bs;
		h.y_min = d.y_min; h.y_max = d.y_max; h.c_min = d.c_min; h.c_max = d.c_max;
		h.csubx = d.csubx; h.csuby = d.csuby;
		build_tables(h, S[k].bi, S[k].blob, S[k].fblob); // vfgs_b200_session_create
	}
	std::vector<LaunchPlan> lps((size_t)njobs);
	std::vector<std::vector<uint16_t>> woffs((size_t)njobs);
	std::vector<StreamJob> sj;
	std::vector<const LaunchPlan*> plans;
	long long nwarps = 0;
	for (int k = 0; k < njobs; k++) { // planning and registers in list order (run_jobs)
		const EmuJob& J = jobs[k];
		batched[k] = 0;
		if (!J.nframes) continue;
		Session& s = S[J.session];
		const HwState& h = s.h;
		const int in_depth = 8 + h.bs, out_depth = J.out_depth ? J.out_depth : in_depth;
		const int cw = J.width / h.csubx, ch = J.height / h.csuby;
		const int nb = (J.width + 15) / 16, R = (J.height + 15) / 16, spitch = nb + 2;
		const int isz = in_depth > 8 ? 2 : 1, osz = out_depth > 8 ? 2 : 1;
		FgsParams p;
		memset(&p, 0, sizeof(p));
		fill_state_params(p, h, s.bi);
		p.blob = s.blob.data(); p.fblob = s.fblob.data();
		p.nframes = J.nframes; p.nb = nb; p.R = R; p.row_begin = 0; p.rows = R;
		p.y_begin = 0; p.y_end = J.height;
		p.in_bytes = isz; p.out_bytes = osz;
		bool in_place;
		if (J.semi) {
			p.in_frame_bytes = J.fs_in; p.out_frame_bytes = J.fs_out;
			set_semiplanar_planes(p, J.in_y, J.in_uv, J.sy_in, J.suv_in, J.out_y, J.out_uv, J.sy_out, J.suv_out, J.width, J.height, cw,
			                      ch, in_depth == 10, out_depth == 10);
			in_place = J.in_y == J.out_y;
		} else {
			const size_t ysam = (size_t)J.width * J.height, csam = (size_t)cw * ch;
			p.in_frame_bytes = (long long)((ysam + 2 * csam) * isz);
			p.out_frame_bytes = (long long)((ysam + 2 * csam) * osz);
			const size_t off[3] = {0, ysam, ysam + csam};
			for (int c = 0; c < 3; c++) {
				p.comp[c].in = J.in_y + off[c] * isz;
				p.comp[c].out = J.out_y + off[c] * osz;
				p.comp[c].in_row_bytes = (long long)(c ? cw : J.width) * isz;
				p.comp[c].out_row_bytes = (long long)(c ? cw : J.width) * osz;
				p.comp[c].width = c ? cw : J.width;
				p.comp[c].lines = c ? ch : J.height;
			}
			in_place = J.in_y == J.out_y;
		}
		p.spitch = spitch; p.stream_rows = R; p.stream_row0 = 0;
		finish_tasks(p);
		LaunchPlan& lp = lps[k];
		plan_launches(p, s.bi, mode, in_place, 227 * 1024, kEmuPad, lp);
		const bool scratch = in_place && in_place_needs_scratch(lp, s.bi);
		if (!lp.any_general && !scratch) {
			batched[k] = 1;
			woffs[k].assign((size_t)J.nframes * R * spitch * 4, 0);
			for (FgsParams* q : {&lp.fast, &lp.edge, &lp.gather}) { q->states = nullptr; q->woffs = woffs[k].data(); }
			StreamJob t;
			t.warp0 = nwarps; t.epoch = h.line_rnd; t.R = R; t.nb = nb; t.spitch = spitch;
			t.states = nullptr; t.woffs = woffs[k].data(); t.wp = make_woff_params(lp.fast, lp.kind);
			sj.push_back(t);
			plans.push_back(&lp);
			nwarps += (long long)J.nframes * R;
		}
		advance_frames(s.h, R, nb, (uint64_t)J.nframes, jt);
	}
	for (int k = 0; k < nsess; k++) {
		regs[4 * k] = S[k].h.rnd; regs[4 * k + 1] = S[k].h.rnd_up; regs[4 * k + 2] = S[k].h.line_rnd; regs[4 * k + 3] = S[k].h.line_rnd_up;
	}
	// the job-table stream kernel: one warp per (job, frame, block-row), its job found by stream_job_of
	for (long long w = 0; w < nwarps; w++) {
		const StreamJob& t = sj[(size_t)stream_job_of(sj.data(), (int)sj.size(), w)];
		const long long local = w - t.warp0;
		const long long f = local / t.R, r = local - f * t.R;
		uint32_t st = jt.jump(t.epoch, ((uint64_t)f * (uint64_t)(t.R - 1) + (uint64_t)r) * (uint64_t)t.nb);
		for (int b = 0; b < t.nb; b++) {
			uint16_t* o = t.woffs + ((size_t)local * t.spitch + 1 + b) * 4;
			o[0] = (uint16_t)window_offset<0>(st, t.wp.c[0]);
			o[1] = (uint16_t)window_offset<1>(st, t.wp.c[1]);
			o[2] = (uint16_t)window_offset<2>(st, t.wp.c[2]);
			st = lfsr_step(st);
		}
	}
	std::vector<LaunchGroup> groups;
	group_launches(plans, groups);
	size_t max_blob = 0;
	for (const Session& s : S) max_blob = s.blob.size() > max_blob ? s.blob.size() : max_blob;
	int launches = 0;
	for (const LaunchGroup& g : groups) {
		const int kind = g.key & 3;
		std::vector<FgsParams> fp; // the device copy of the group's launch parameters
		std::vector<long long> task0(1, 0);
		for (const FgsParams* q : g.p) { fp.push_back(*q); task0.push_back(task0.back() + q->total_tasks); }
		if (task0.back() <= 0) continue;
		if (launches < 16) keys[launches] = g.key;
		launches++;
		for (int b = 0; b < grid; b++) {
			// this CTA's shared memory, filled with garbage once: a switch that forgot to reload something shows
			std::vector<uint8_t> store((size_t)3 * kLutAlign + 3 * kLutBytes + 256 * 1024 + max_blob, 0xa5);
			uint8_t* lut_ptr = (uint8_t*)(((uintptr_t)store.data() + 2 * kLutAlign - 1) & ~(uintptr_t)(kLutAlign - 1));
			MultiCursor cur;
			multi_begin(task0.data(), (int)fp.size(), grid, b, cur);
			int j;
			long long lo, end;
			while (multi_next(task0.data(), cur, j, lo, end)) {
				const FgsParams& p = fp[(size_t)j];
				if (kind == 1) { // fgs_apply_gather_multi_kernel: the job's image behind its gather LUTs, the LUTs rebuilt
					uint8_t* img = lut_ptr + (size_t)p.ngather * kLutBytes;
					memcpy(img, p.blob, (size_t)p.blob_bytes);
					for (int c = 0; c < 3; c++) {
						if (p.glut_index[c] < 0) continue;
						const uint16_t* compact = (const uint16_t*)(img + p.lut_off) + c * 256;
						uint32_t* lut = (uint32_t*)(lut_ptr + (size_t)p.glut_index[c] * kLutBytes);
						const uint32_t slot_bytes = (uint32_t)p.pat_size[c ? 1 : 0];
						for (int i = 0; i < 256 * 32; i++)
							lut[i] = (g.key & 4) ? gather_lut_entry<true>(compact[i >> 5], slot_bytes) : gather_lut_entry<false>(compact[i >> 5], slot_bytes);
					}
					for (int w = 0; w < warps; w++)
						for (long long task = lo + w; task < end; task += warps) gather_task_of(g.key, p, lut_ptr, img, (uint32_t)(task - task0[j]));
				} else { // fgs_apply_fast_multi_kernel: the job's component images, the LUTs with its scale shift
					if (p.fpad != kEmuPad) return -1;
					for (int c = 0; c < 3; c++)
						if (p.fimg_bytes[c]) memcpy(lut_ptr + p.fimg_off[c], p.fblob + p.fimg_src[c], (size_t)p.fimg_bytes[c]);
					expand_fast_luts((uint32_t*)lut_ptr, (const uint32_t*)p.fblob, (uint32_t)p.pow16, 0, 1);
					for (int w = 0; w < warps; w++)
						for (long long task = lo + w; task < end; task += warps) fast_task_of(g.key, p, lut_ptr, (uint32_t)(task - task0[j]));
				}
			}
		}
	}
	return launches;
}

// Schedule coverage alone, for the kernels' walk (multi_begin / multi_next) over given task counts: hits (size sum of
// ntasks) how often each (job, task) ran, switches[b] how many jobs CTA b loaded. Returns 0, -1 when CTA ranges are not
// contiguous and in order, -2 when a task index falls outside its job.
extern "C" int emuj_replay(const long long* ntasks, int njobs, int grid, int warps, int* hits, int* switches)
{
	std::vector<long long> task0((size_t)njobs + 1, 0);
	for (int j = 0; j < njobs; j++) task0[j + 1] = task0[j] + ntasks[j];
	long long prev_hi = 0;
	for (int b = 0; b < grid; b++) {
		MultiCursor cur;
		multi_begin(task0.data(), njobs, grid, b, cur);
		if (cur.lo != prev_hi || cur.hi < cur.lo) return -1;
		prev_hi = cur.hi;
		switches[b] = 0;
		int j;
		long long lo, end;
		while (multi_next(task0.data(), cur, j, lo, end)) {
			switches[b]++;
			for (int w = 0; w < warps; w++)
				for (long long task = lo + w; task < end; task += warps) {
					const long long local = task - task0[j];
					if (local < 0 || local >= ntasks[j]) return -2;
					hits[task0[j] + local]++;
				}
		}
	}
	return prev_hi == task0[njobs] ? 0 : -1;
}
