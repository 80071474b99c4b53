// emu_meta.cpp -- TEST TOOL, never part of the product library.
// Host build of the device half of vfgs_b200_session_init_metadata with the library's own code:
//   * the auto-regressive filter's data-parallel form (fw_device.h: fw_ar_noise with nthreads = 32, then
//     fw_ar_wave_step run lane by lane in step order, as one warp runs it) against the serial fw_ar_phase0;
//   * the shared image fill (vfgs_tables.h: layout_tables + fill_tables with any thread count) against a restatement of
//     the serial image builder as it was before the fill was split out of it (reference_build_tables below);
//   * the layout from the -128 flags a session keeps against the layout from scanning the patterns;
//   * the host half of an update (fw_host.h: fw_apply_host) on a fresh state.
// What it cannot cover -- the launch, the CTA barriers, the copies -- the -m gpu tests cover
// (tests/test_gpu_session_metadata.py).
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "../../versatilefilmgrain_b200/csrc/fw_host.h"

using namespace vfgs;

namespace {
struct StateDump { // == refh_state / oracle_dump
	int8_t pattern[2][9][64][64];
	uint8_t slut[3][256];
	uint8_t plut[3][256];
	uint32_t rnd, rnd_up, line_rnd, line_rnd_up;
	int scale_shift, bs, y_min, y_max, c_min, c_max, csubx, csuby;
};

void to_hw(const StateDump& d, HwState& h)
{
	memcpy(h.pattern, d.pattern, sizeof(h.pattern));
	memcpy(h.slut, d.slut, sizeof(h.slut));
	memcpy(h.plut, d.plut, sizeof(h.plut));
	h.rnd = d.rnd; h.rnd_up = d.rnd_up; h.line_rnd = d.line_rnd; h.line_rnd_up = d.line_rnd_up;
	h.scale_shift = d.scale_shift; h.bs = d.bs; h.y_min = d.y_min; h.y_max = d.y_max; h.c_min = d.c_min; h.c_max = d.c_max;
	h.csubx = d.csubx; h.csuby = d.csuby;
}
void to_dump(const HwState& h, StateDump& d)
{
	memcpy(d.pattern, h.pattern, sizeof(d.pattern));
	memcpy(d.slut, h.slut, sizeof(d.slut));
	memcpy(d.plut, h.plut, sizeof(d.plut));
	d.rnd = h.rnd; d.rnd_up = h.rnd_up; d.line_rnd = h.line_rnd; d.line_rnd_up = h.line_rnd_up;
	d.scale_shift = h.scale_shift; d.bs = h.bs; d.y_min = h.y_min; d.y_max = h.y_max; d.c_min = h.c_min; d.c_max = h.c_max;
	d.csubx = h.csubx; d.csuby = h.csuby;
}

const FwTables& tables()
{
	static FwTables t;
	static bool made = false;
	if (!made) { make_fw_tables(t); made = true; }
	return t;
}
const uint32_t* pow2()
{
	static const JumpTable jt;
	return &jt.pow2[0].row[0]; // uint32[64][32], the layout of the device copy
}

// The data-parallel AR phase as the device runs it: noise by 32 threads, then the wavefront, lane by lane per step.
void ar_wave(const FwJob& j, int8_t* buf, const int8_t* buf0)
{
	static int8_t noise[82 * 73];
	for (int tid = 0; tid < 32; tid++) fw_ar_noise(j, tables().gauss, pow2(), noise, tid, 32);
	for (int t = 0; t < fw_ar_wave_steps(j); t++)
		for (int lane = 0; lane < 32; lane++) fw_ar_wave_step(j, noise, buf, buf0, t, lane);
}

// One AR job both ways on the same luma field; true when the fields agree byte for byte.
bool ar_same(const FwJob& j, const int8_t* luma)
{
	const int bytes = j.size == 32 ? 44 * 38 : 82 * 73;
	std::vector<int8_t> a((size_t)bytes, 0x55), b((size_t)bytes, -0x33);
	fw_ar_phase0(j, tables().gauss, a.data(), luma);
	ar_wave(j, b.data(), luma);
	return memcmp(a.data(), b.data(), (size_t)bytes) == 0;
}

uint64_t rng_next(uint64_t& s)
{
	s ^= s << 13; s ^= s >> 7; s ^= s << 17;
	return s;
}
int rng_int(uint64_t& s, int lo, int hi) { return lo + (int)(rng_next(s) % (uint64_t)(hi - lo + 1)); }

// The serial image builder before the fill was split out of it (restated verbatim, test tool).
void reference_build_tables(const HwState& h, TableInfo& g_bi, std::vector<uint8_t>& g_blob, std::vector<uint8_t>& g_fblob)
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
	const int lpitch = 64 + VFGS_PAT_ROW_SKEW, cpitch = ccols + VFGS_PAT_ROW_SKEW;
	g_bi.lut_off = 0;
	g_bi.pat_off[0] = 3 * 256 * 2;
	g_bi.pat_size[0] = 64 * lpitch; g_bi.pat_stride[0] = lpitch;
	g_bi.pat_off[1] = g_bi.pat_off[0] + nslot[0] * g_bi.pat_size[0];
	g_bi.pat_size[1] = crows * cpitch; g_bi.pat_stride[1] = cpitch;
	g_bi.bytes = (g_bi.pat_off[1] + nslot[1] * g_bi.pat_size[1] + 16 + 15) & ~15;
	g_bi.gbytes = g_bi.bytes;
	for (int b = 0; b < 2; b++) {
		g_bi.nslot[b] = nslot[b];
		g_bi.neg_ok[b] = true;
		for (int s = 0; s < nslot[b] && g_bi.neg_ok[b]; s++)
			for (int r = 0; r < 64 && g_bi.neg_ok[b]; r++)
				for (int x = 0; x < 64; x++)
					if (h.pattern[b][s][r][x] == -128) { g_bi.neg_ok[b] = false; break; }
		g_bi.neg_off[b] = g_bi.gbytes - g_bi.pat_off[b];
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
		const int pitch = cols + VFGS_FAST_ROW_SKEW;
		g_bi.fpat_stride[c] = pitch;
		g_bi.fpat_copy[c] = rows * pitch;
		g_bi.fpat_off[c][0] = 0;
		g_bi.fpat_off[c][1] = ncopy * rows * pitch;
		g_bi.fimg_src[c] = off;
		g_bi.fimg_bytes[c] = ok ? 2 * ncopy * rows * pitch : 0;
		if (c == 2 && ok && g_bi.fast_ok[1] && g_bi.uniform_pi[1] == slot) {
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

bool same_info(const TableInfo& a, const TableInfo& b) { return memcmp(&a, &b, sizeof(TableInfo)) == 0; }

bool plan_of(const void* cfg, int is_afgs1, int csubx, int csuby, FwPlan& plan)
{
	if (is_afgs1) fw_plan_afgs1(*(const fgs_afgs1*)cfg, csubx, csuby, plan);
	else fw_plan_sei(*(const fgs_sei*)cfg, csubx, csuby, plan);
	return plan.error == nullptr;
}
} // namespace

extern "C" int emum_state_size(void) { return (int)sizeof(StateDump); }

// Every AR job of a configuration's plan, in firmware order on one working memory: the wavefront against the serial
// filter on the same inputs (the luma field the previous jobs left). Returns the number of jobs that differ, -1 where
// the plan fails; *njobs: AR jobs compared.
extern "C" int emum_ar_plan(const void* cfg, int is_afgs1, int csubx, int csuby, int* njobs)
{
	FwPlan plan;
	if (!plan_of(cfg, is_afgs1, csubx, csuby, plan)) return -1;
	static FwScratch s;
	memset(&s, 0, sizeof(s));
	static int8_t pattern[2][9][64][64];
	int bad = 0, n = 0;
	for (const FwJob& j : plan.jobs) {
		if (j.kind == kFwAR) {
			n++;
			std::vector<int8_t> luma(s.Lbuf, s.Lbuf + sizeof(s.Lbuf)); // the serial run of a luma job overwrites Lbuf
			if (!ar_same(j, luma.data())) bad++;
		}
		fw_run_job_serial(j, tables(), s, &pattern[0][0][0][0]);
	}
	*njobs = n;
	return bad;
}

// n random AR jobs: lags 1..3 (with and without the luma coefficient) and the SEI 6-tap layout, random shifts, scales
// and seeds, luma and chroma sizes, luma injection on a random luma field. Returns the number of jobs that differ.
extern "C" int emum_ar_random(unsigned long long seed, int n)
{
	uint64_t s = seed * 0x9E3779B97F4A7C15ull + 1;
	int bad = 0;
	std::vector<int8_t> luma(73 * 82 + 1024, 0);
	for (int k = 0; k < n; k++) {
		for (size_t i = 0; i < 73 * 82; i++) luma[i] = (int8_t)rng_int(s, -127, 127);
		const int layout = rng_int(s, 0, 6); // 0: SEI 6 taps; 1..6: lag 1..3, without / with the luma coefficient
		const int size = rng_int(s, 0, 1) ? 64 : 32;
		const int scale = rng_int(s, 1, 9);
		FwJob j = fw_ar_job(size == 32 ? 1 : 0, 0, 2, 2, size, rng_int(s, 0, 3) != 0, rng_int(s, 1, 4), scale, (uint32_t)rng_next(s));
		int16_t ar[25];
		const int amp = rng_int(s, 0, 2) == 0 ? 512 : 128;
		for (int i = 0; i < 25; i++) ar[i] = (int16_t)rng_int(s, -amp, amp);
		static const int ncoef[7] = {6, 4, 5, 12, 13, 24, 25};
		if (!fw_ar_taps(j, ar, ncoef[layout], scale)) abort();
		if (!ar_same(j, luma.data())) bad++;
	}
	return bad;
}

// Synthetic jobs with a luma coefficient and the luma field present, for both sizes. Returns the number that differ.
extern "C" int emum_ar_luma_injection(unsigned long long seed, int n)
{
	uint64_t s = seed * 0xD1B54A32D192ED03ull + 7;
	int bad = 0;
	std::vector<int8_t> luma(73 * 82 + 1024, 0);
	for (int k = 0; k < n; k++) {
		for (size_t i = 0; i < 73 * 82; i++) luma[i] = (int8_t)rng_int(s, -127, 127);
		const int size = k & 1 ? 64 : 32, lag = rng_int(s, 1, 3), scale = rng_int(s, 4, 9);
		FwJob j = fw_ar_job(size == 32 ? 1 : 0, 0, 2, 2, size, true, rng_int(s, 1, 3), scale, (uint32_t)rng_next(s));
		int16_t ar[25];
		for (int i = 0; i < 25; i++) ar[i] = (int16_t)rng_int(s, -200, 200);
		const int nc = 2 * lag * (lag + 1) + 1;
		ar[nc - 1] = (int16_t)(rng_int(s, 1, 127) * (rng_int(s, 0, 1) ? 1 : -1));
		if (!fw_ar_taps(j, ar, nc, scale) || !j.cx) abort();
		if (!ar_same(j, luma.data())) bad++;
	}
	return bad;
}

// The shared fill with nthreads threads (run one after the other) against the serial builder, for one state.
// Returns 0 when layout and both images agree byte for byte, 1 for the layout, 2 for the general image, 3 for the fast one.
extern "C" int emum_fill(const void* state, int nthreads)
{
	static HwState h;
	to_hw(*(const StateDump*)state, h);
	TableInfo want, got;
	memset(&want, 0, sizeof(want)); memset(&got, 0, sizeof(got));
	std::vector<uint8_t> wb, wf;
	reference_build_tables(h, want, wb, wf);
	Minus128 m;
	scan_minus128(h, m);
	layout_tables(h.plut, h.csubx, h.csuby, m, got);
	if (!same_info(want, got)) return 1;
	std::vector<uint8_t> gb((size_t)got.gbytes, 0xa5), gf((size_t)got.fbytes, 0x5a); // every byte must be written
	const TableSrc src = {&h.pattern[0][0][0][0], &h.slut[0][0], &h.plut[0][0], h.csubx, h.csuby};
	for (int tid = nthreads - 1; tid >= 0; tid--) fill_tables(src, got, gb.data(), gf.data(), tid, nthreads);
	if (gb != wb) return 2;
	if (gf != wf) return 3;
	return 0;
}

// What a session created on state `before` keeps and what a metadata update makes of it: the -128 flags of the
// snapshot, cleared for the slots the plan writes, give the layout; the state after the update (`after`, in which the
// pattern jobs have run) scanned gives it as well. Returns 0 when the two layouts agree, 1 when not, -1 on a plan error.
extern "C" int emum_flag_layout(const void* before, const void* cfg, int is_afgs1, const void* after)
{
	static HwState hb, ha;
	to_hw(*(const StateDump*)before, hb);
	to_hw(*(const StateDump*)after, ha);
	FwPlan plan;
	if (!plan_of(cfg, is_afgs1, hb.csubx, hb.csuby, plan)) return -1;
	Minus128 m;
	scan_minus128(hb, m);
	for (const FwJob& j : plan.jobs) m.used[j.bank][j.slot] = false;
	TableInfo a, b;
	memset(&a, 0, sizeof(a)); memset(&b, 0, sizeof(b));
	layout_tables(plan.plut, hb.csubx, hb.csuby, m, a);
	Minus128 ms;
	scan_minus128(ha, ms);
	layout_tables(ha.plut, ha.csubx, ha.csuby, ms, b);
	return same_info(a, b) ? 0 : 1;
}

// The host half of an update (fw_apply_host) on a freshly powered-on state of the given depth and subsampling.
// Returns 0, 1 where the plan fails or the reference asserts.
extern "C" int emum_host_half(const void* cfg, int is_afgs1, int depth, int csubx, int csuby, void* state_out)
{
	static HwState h;
	h.power_on();
	const int nbs = depth - 8;
	h.scale_shift = (h.scale_shift + h.bs - nbs) & 0xff; h.bs = nbs; // vfgs_set_depth
	h.csubx = csubx; h.csuby = csuby;
	FwPlan plan;
	if (!plan_of(cfg, is_afgs1, csubx, csuby, plan)) return 1;
	if (!fw_apply_host(h, plan)) return 1;
	to_dump(h, *(StateDump*)state_out);
	return 0;
}

// Serial firmware jobs of a plan on a given state and working memory (the state a session reaches on the host), for
// building `after` states: state in/out, scratch in/out (sizeof(FwScratch) bytes).
extern "C" int emum_scratch_size(void) { return (int)sizeof(FwScratch); }
extern "C" int emum_run_plan(const void* cfg, int is_afgs1, void* state, void* scratch)
{
	static HwState h;
	to_hw(*(const StateDump*)state, h);
	FwPlan plan;
	if (!plan_of(cfg, is_afgs1, h.csubx, h.csuby, plan)) return 1;
	for (const FwJob& j : plan.jobs) fw_run_job_serial(j, tables(), *(FwScratch*)scratch, &h.pattern[0][0][0][0]);
	if (!fw_apply_host(h, plan)) return 1;
	to_dump(h, *(StateDump*)state);
	return 0;
}
