// fw_device.h -- grain pattern synthesis of the firmware layer as data-parallel "jobs" (one CTA each).
//
// Restates, from the reference's src/vfgs_fw.c:
//   vfgs_make_sei_ff_pattern64 / 32   :362-408   Gaussian samples placed by an LFSR in the low-frequency corner of a
//                                                64 x 64 (32 x 32) block, then
//   idct2_64 / idct2_32               :297-360   two integer matrix passes with the H.266 64-point DCT-II and a clip
//   vfgs_make_ar_pattern              :410-502   causal auto-regressive filter over an 82 x 73 (44 x 38) field in raster
//                                                order (+ optional luma injection), cropped to 64 x 64 (32 x 32)
// and the copy semantics of vfgs_set_luma_pattern / vfgs_set_chroma_pattern (src/vfgs_hw.c:314-325), including the
// firmware's habit of reusing ONE pattern buffer P for every pattern (a 32 x 32 pattern leaves the rest of P as it was,
// and the chroma setter of a non-4:2:0 format reads that rest).
// The constant tables come from h274_tables.h. The phase functions are written for `nthreads` cooperating threads
// with a barrier between phases: a CTA on the device (fw_pattern_kernel), one thread in the host build (tests/emu).
#pragma once
#include <stdint.h>
#include <string.h>
#include "h274_tables.h"
#include "vfgs_core.h"

namespace vfgs {

struct FwTables {
	int8_t gauss[2048];
	int8_t dct[64][64];
};

// Gaussian table from its packed form; DCT matrix from its 65 cosine magnitudes: entry (k, n) is c[0] for k = 0, else
// the angle index j = (2n + 1) k mod 256 folded into [0, 64] with the sign of cos(pi j / 128).
inline void make_fw_tables(FwTables& t)
{
	auto hex = [](char ch) { return ch <= '9' ? ch - '0' : ch - 'a' + 10; };
	for (int i = 0; i < 2048; i++) t.gauss[i] = (int8_t)(uint8_t)(hex(kGaussianHex[2 * i]) * 16 + hex(kGaussianHex[2 * i + 1]));
	for (int k = 0; k < 64; k++)
		for (int n = 0; n < 64; n++) {
			int v = kDct64Cos[0];
			if (k) {
				int j = ((2 * n + 1) * k) % 256;
				if (j > 128) j = 256 - j;
				v = j <= 64 ? kDct64Cos[j] : -(int)kDct64Cos[128 - j];
			}
			t.dct[k][n] = (int8_t)v;
		}
}

enum FwKind { kFwFF64 = 0, kFwFF32 = 1, kFwAR = 2 };

constexpr int kFwMaxPatterns = 8; // VFGS_MAX_PATTERNS, vfgs_hw.h:49

struct FwJob {
	int kind;
	int bank, slot;       // destination pattern[bank][slot] (bank 0: vfgs_set_luma_pattern, 1: vfgs_set_chroma_pattern)
	int csubx, csuby;     // chroma setter repacking (vfgs_hw.c:320-325)
	int fh, fv;           // FF: horizontal / vertical cut-off (comp_model_value[1], [2])
	int size;             // AR: 64 | 32
	int16_t coef[4][7];   // AR: taps, [3][3] is the current sample (vfgs_fw.c:421-463)
	int cx;               // AR: luma injection coefficient (0: none)
	int use_luma;         // AR: the luma field of the previous job is available (buf0 != NULL)
	int shift, scale;     // AR: Gaussian scale-down, coefficient scale-down
	uint32_t seed;        // start of the LFSR
};

// Working memory of the jobs, persistent from job to job like the firmware's locals (vfgs_fw.c:519-521, 666-669).
struct FwScratch {
	int8_t P[64 * 64];
	int8_t Lbuf[73 * 82 + 1024]; // + slack: the reference's luma injection indexes the luma field with a pitch of 88 and runs
	int8_t Cbuf[38 * 44];        //   up to 428 bytes past its 82 x 73 bytes (vfgs_fw.c:478-481); here that slack reads as zeros
	uint32_t nseq[1024];
	int16_t X[64 * 64];
};

VFGS_HD int fw_round(int a, int s) { return (a + (1 << (s - 1))) >> s; } // vfgs_fw.c:43

// ---- frequency-filtering pattern ------------------------------------------------------------
// phase 0 (one thread): the LFSR state of every group of 4 (2) coefficients, vfgs_fw.c:371-383 / 395-405
VFGS_HD void fw_ff_phase0(const FwJob& j, FwScratch& s)
{
	const int S = j.kind == kFwFF64 ? 64 : 32, step = j.kind == kFwFF64 ? 4 : 2;
	uint32_t n = j.seed; // Seed_LUT[0] (64 x 64) or Seed_LUT[1] (32 x 32)
	int idx = 0;
	for (int l = 0; l < S; l++)
		for (int k = 0; k < S; k += step) { s.nseq[idx++] = n; n = lfsr_step(n); } // the firmware's prng is the hardware's LFSR step (vfgs_fw.c:284-294)
}
// phase 1: coefficient block B (kept in P), zero outside the [0, fh) x [0, fv) corner, DC removed
VFGS_HD void fw_ff_phase1(const FwJob& j, const FwTables& t, FwScratch& s, int tid, int nthreads)
{
	const int S = j.kind == kFwFF64 ? 64 : 32, step = j.kind == kFwFF64 ? 4 : 2;
	const int fh = step * (j.fh + 1), fv = step * (j.fv + 1);
	for (int i = tid; i < S * S; i += nthreads) {
		const int l = i / S, k = i % S, kk = k - k % step;
		int8_t v = 0;
		if (kk < fh && l < fv) v = t.gauss[(s.nseq[l * (S / step) + kk / step] + (uint32_t)(k - kk)) & 2047];
		if (i == 0) v = 0;
		s.P[i] = v;
	}
}
// phase 2: vertical pass X = (D' B) (vfgs_fw.c:303-313 / 335-345)
VFGS_HD void fw_ff_phase2(const FwJob& j, const FwTables& t, FwScratch& s, int tid, int nthreads)
{
	const bool big = j.kind == kFwFF64;
	const int S = big ? 64 : 32;
	for (int idx = tid; idx < S * S; idx += nthreads) {
		const int jj = idx / S, i = idx % S;
		int acc = big ? 256 : 128;
		for (int k = 0; k < S; k++) acc += (int)t.dct[big ? k : 2 * k][jj] * s.P[k * S + i];
		s.X[idx] = (int16_t)(acc >> (big ? 9 : 8));
	}
}
// phase 3: horizontal pass + clip (vfgs_fw.c:315-327 / 347-359), result back into P
VFGS_HD void fw_ff_phase3(const FwJob& j, const FwTables& t, FwScratch& s, int tid, int nthreads)
{
	const bool big = j.kind == kFwFF64;
	const int S = big ? 64 : 32;
	for (int idx = tid; idx < S * S; idx += nthreads) {
		const int jj = idx / S, i = idx % S;
		int acc = 256;
		for (int k = 0; k < S; k++) acc += (int)s.X[jj * S + k] * t.dct[big ? k : 2 * k][i];
		acc >>= 9;
		acc = acc > 127 ? 127 : acc < -127 ? -127 : acc;
		s.P[idx] = (int8_t)acc;
	}
}

// ---- auto-regressive pattern ------------------------------------------------------------------
// phase 0 (one thread): the causal filter in raster order, vfgs_fw.c:465-495 (the host reference of the wavefront below)
// buf: the field being generated (82 x 73 or 44 x 38 bytes; shared memory on the device), buf0: the luma field,
// gauss: the Gaussian table
VFGS_HD void fw_ar_phase0(const FwJob& j, const int8_t* gauss, int8_t* buf, const int8_t* buf0)
{
	const int sub = j.size == 32 ? 2 : 1;
	const int width = sub > 1 ? 44 : 82, height = sub > 1 ? 38 : 73;
	uint32_t rnd = j.seed;
	for (int y = 0; y < height; y++)
		for (int x = 0; x < width; x++) {
			int g = 0;
			if (y >= 3 && x >= 3 && x < width - 3) {
				for (int jj = -3; jj <= 0; jj++)
					for (int i = -3; i <= 3 && (i < 0 || jj < 0); i++)
						g += (int)j.coef[3 + jj][3 + i] * buf[width * (y + jj) + x + i];
				if (j.cx && j.use_luma) { // luma injection; the luma field is indexed with a pitch of width * sub like the reference does
					const int i = (x - 3) * sub + 3, jj = (y - 3) * sub + 3;
					int Z = buf0[width * sub * jj + i];
					if (sub > 1) Z += buf0[width * sub * jj + i + 1];
					if (sub > 1) Z += buf0[width * sub * (jj + 1) + i] + buf0[width * sub * (jj + 1) + i + 1];
					g += j.cx * fw_round(Z, 2 * sub - 2);
				}
				g = fw_round(g, j.scale);
			}
			g += fw_round((int)gauss[rnd & 2047], j.shift);
			rnd = lfsr_step(rnd);
			buf[width * y + x] = (int8_t)(g > 127 ? 127 : g < -127 ? -127 : g);
		}
}
// The same filter as data-parallel phases (the device form, fw_pattern_kernel and fw_sessions_kernel).
// Noise: the Gaussian term of sample (x, y) is read at the LFSR after y * width + x steps from the seed. Thread tid of
// nthreads takes one contiguous run of samples: one jump-ahead to its start (pow2: JumpTable as uint32[64][32]), then a
// walk. noise: width * height bytes.
VFGS_HD int fw_parity(uint32_t x)
{
#if defined(__CUDA_ARCH__)
	return __popc(x) & 1;
#else
	return __builtin_popcount(x) & 1;
#endif
}
VFGS_HD uint32_t fw_lfsr_jump(const uint32_t* pow2, uint32_t x, uint32_t n)
{
	for (int k = 0; n; k++, n >>= 1)
		if (n & 1u) {
			uint32_t y = 0;
			for (int i = 0; i < 32; i++) y |= (uint32_t)fw_parity(pow2[k * 32 + i] & x) << i;
			x = y;
		}
	return x;
}
VFGS_HD void fw_ar_noise(const FwJob& j, const int8_t* gauss, const uint32_t* pow2, int8_t* noise, int tid, int nthreads)
{
	const int sub = j.size == 32 ? 2 : 1;
	const int n = sub > 1 ? 44 * 38 : 82 * 73;
	const int chunk = (n + nthreads - 1) / nthreads, i0 = tid * chunk, i1 = i0 + chunk < n ? i0 + chunk : n;
	if (i0 >= i1) return;
	uint32_t rnd = fw_lfsr_jump(pow2, j.seed, (uint32_t)i0);
	for (int i = i0; i < i1; i++) {
		noise[i] = (int8_t)fw_round((int)gauss[rnd & 2047], j.shift);
		rnd = lfsr_step(rnd);
	}
}
// Wavefront: sample (x, y) reads (x-3..x-1, y) and (x-3..x+3, y-3..y-1), all of smaller t = x + 4y, so the samples of
// one t are independent: step t computes them, one per lane (at most ceil(82 / 4) = 21 of them), and a warp barrier
// separates the steps. The tap sum is integer, so the order does not change it: the result is fw_ar_phase0's, byte for
// byte. buf0 (the luma field) must not overlap buf.
VFGS_HD int fw_ar_wave_steps(const FwJob& j) { return j.size == 32 ? 44 + 4 * 37 : 82 + 4 * 72; }
VFGS_HD void fw_ar_wave_step(const FwJob& j, const int8_t* noise, int8_t* buf, const int8_t* buf0, int t, int lane)
{
	const int sub = j.size == 32 ? 2 : 1;
	const int width = sub > 1 ? 44 : 82, height = sub > 1 ? 38 : 73;
	const int y = (t >= width ? (t - width + 4) >> 2 : 0) + lane; // smallest y with x = t - 4y < width, + lane
	const int x = t - 4 * y;
	if (x < 0 || y >= height) return;
	int g = 0;
	if (y >= 3 && x >= 3 && x < width - 3) {
		for (int jj = -3; jj <= 0; jj++)
			for (int i = -3; i <= 3 && (i < 0 || jj < 0); i++)
				g += (int)j.coef[3 + jj][3 + i] * buf[width * (y + jj) + x + i];
		if (j.cx && j.use_luma) { // luma injection, indexed as in fw_ar_phase0
			const int i = (x - 3) * sub + 3, jj = (y - 3) * sub + 3;
			int Z = buf0[width * sub * jj + i];
			if (sub > 1) Z += buf0[width * sub * jj + i + 1];
			if (sub > 1) Z += buf0[width * sub * (jj + 1) + i] + buf0[width * sub * (jj + 1) + i + 1];
			g += j.cx * fw_round(Z, 2 * sub - 2);
		}
		g = fw_round(g, j.scale);
	}
	g += noise[width * y + x];
	buf[width * y + x] = (int8_t)(g > 127 ? 127 : g < -127 ? -127 : g);
}

// phase 1: cropped area to P (vfgs_fw.c:497-501)
VFGS_HD void fw_ar_phase1(const FwJob& j, FwScratch& s, int tid, int nthreads)
{
	const int sub = j.size == 32 ? 2 : 1, width = sub > 1 ? 44 : 82;
	const int8_t* buf = j.size == 32 ? s.Cbuf : s.Lbuf;
	for (int idx = tid; idx < j.size * j.size; idx += nthreads) {
		const int y = idx / j.size, x = idx % j.size;
		s.P[idx] = (y < 64 / sub && x < 64 / sub) ? buf[width * (3 + 6 / sub + y) + (3 + 6 / sub + x)] : (int8_t)0;
	}
}

// ---- setter: P -> pattern[bank][slot] (vfgs_hw.c:314-325) ----------------------------------------
VFGS_HD void fw_store_phase(const FwJob& j, const FwScratch& s, int8_t* pattern /* [2][9][64][64] */, int tid, int nthreads)
{
	int8_t* dst = pattern + ((size_t)j.bank * 9 + j.slot) * 4096;
	if (j.bank == 0) {
		for (int i = tid; i < 4096; i += nthreads) dst[i] = s.P[i];
	} else {
		const int rows = 64 / j.csuby, src_stride = 64 / j.csuby, ncopy = 64 / j.csubx;
		for (int i = tid; i < rows * ncopy; i += nthreads) {
			const int r = i / ncopy, x = i % ncopy;
			dst[r * 64 + x] = s.P[src_stride * r + x];
		}
	}
}

// Whole job with one thread (host build).
inline void fw_run_job_serial(const FwJob& j, const FwTables& t, FwScratch& s, int8_t* pattern)
{
	if (j.kind == kFwAR) { fw_ar_phase0(j, t.gauss, j.size == 32 ? s.Cbuf : s.Lbuf, s.Lbuf); fw_ar_phase1(j, s, 0, 1); }
	else { fw_ff_phase0(j, s); fw_ff_phase1(j, t, s, 0, 1); fw_ff_phase2(j, t, s, 0, 1); fw_ff_phase3(j, t, s, 0, 1); }
	fw_store_phase(j, s, pattern, 0, 1);
}

} // namespace vfgs
