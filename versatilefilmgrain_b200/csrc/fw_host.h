// fw_host.h -- the cheap, serial half of the firmware layer: from film grain metadata to (a) the list of pattern jobs
// the device runs (fw_device.h) and (b) the LUTs and scalars, which go through the ordinary vfgs_hw.h setters.
// Restates src/vfgs_fw.c:504-708 (vfgs_init_sei, vfgs_make_lut_piecewise_linear, vfgs_init_afgs1) and the tap layout
// part of vfgs_make_ar_pattern (:421-463). Plain C++, shared by the shim and, for the GPU-less tests, by tests/emu.
#pragma once
#include <stdint.h>
#include <string.h>
#include <vector>

#include "../../include/vfgs_fw.h"
#include "fw_device.h"
#include "vfgs_tables.h"

namespace vfgs {

struct FwPlan {
	std::vector<FwJob> jobs;    // in the firmware's order (they share one pattern buffer, fw_device.h)
	uint8_t slut[3][256], plut[3][256];
	int scale_shift = 0;        // argument of vfgs_set_scale_shift
	bool set_seed = false; uint32_t seed = 0;
	bool set_legal = false; int legal = 0;
	const char* error = nullptr; // the reference asserts here
};

// Tap layout of the auto-regressive filter (vfgs_fw.c:421-463). Returns false where the reference asserts.
inline bool fw_ar_taps(FwJob& j, const int16_t ar[], int nb_coef, int scale)
{
	memset(j.coef, 0, sizeof(j.coef));
	j.cx = 0;
	int L = 0;
	switch (nb_coef) {
	case 6: // SEI auto-regressive mode
		j.coef[3][2] = ar[1];                                            // left
		j.coef[2][3] = (int16_t)((ar[1] * ar[4]) >> scale);              // top
		j.coef[2][2] = (int16_t)((ar[3] * ar[4]) >> scale);              // top-left
		j.coef[2][4] = (int16_t)((ar[3] * ar[4]) >> scale);              // top-right
		j.coef[3][1] = ar[5];                                            // left-left
		j.coef[1][3] = (int16_t)(((int32_t)ar[5] * ar[4] * ar[4]) >> (2 * scale)); // top-top
		return true;
	case 5: j.cx = ar[4]; /* fall through */
	case 4: L = 1; break;
	case 13: j.cx = ar[12]; /* fall through */
	case 12: L = 2; break;
	case 25: j.cx = ar[24]; /* fall through */
	case 24: L = 3; break;
	default: return false;
	}
	int k = 0;
	for (int y = -L; y <= 0; y++)
		for (int x = -L; x <= L && (x < 0 || y < 0); x++, k++) j.coef[3 + y][3 + x] = ar[k];
	return true;
}

inline FwJob fw_ar_job(int bank, int slot, int csubx, int csuby, int size, bool use_luma, int shift, int scale, uint32_t seed)
{
	FwJob j;
	memset(&j, 0, sizeof(j));
	j.kind = kFwAR; j.bank = bank; j.slot = slot; j.csubx = csubx; j.csuby = csuby;
	j.size = size; j.use_luma = use_luma ? 1 : 0; j.shift = shift; j.scale = scale; j.seed = seed;
	return j;
}

// vfgs_init_sei, vfgs_fw.c:517-644
inline void fw_plan_sei(const fgs_sei& cfg, int csubx, int csuby, FwPlan& plan)
{
	const int16_t* flat = &cfg.comp_model_value[0][0][0];
	// two models are "the same pattern" when their values 1..5 agree (the scale, value 0, lives in the scale LUT);
	// an unused list entry is the index -1, whose "values 1..5" are the first five values of the whole array
	auto same_pattern = [&](int32_t a, int32_t b) {
		for (int i = 1; i < SEI_MAX_MODEL_VALUES; i++)
			if (flat[a + i] != flat[b + i]) return false;
		return true;
	};
	uint8_t slut[256], plut[256];
	uint8_t intensities[kFwMaxPatterns];
	int32_t patterns[kFwMaxPatterns];
	int np = 0;
	for (int c = 0; c < 3; c++) {
		memset(slut, 0, sizeof(slut)); // once per component of the OUTER loop: Cr starts from Cb's entries (c == 2 fills both)
		if (c < 2) {
			np = 0;
			memset(intensities, 0, sizeof(intensities));
			for (int i = 0; i < kFwMaxPatterns; i++) patterns[i] = -1;
		}
		// 1. distinct patterns of the component, sorted by the lower bound of their first interval
		if (cfg.comp_model_present_flag[c])
			for (int k = 0; k < cfg.num_intensity_intervals[c]; k++) {
				const uint8_t a = cfg.intensity_interval_lower_bound[c][k];
				const int32_t id = SEI_MAX_MODEL_VALUES * (k + 256 * c);
				int i = 0;
				for (; i < kFwMaxPatterns; i++)
					if (same_pattern(patterns[i], id)) break;
				if (i == kFwMaxPatterns && np < kFwMaxPatterns) {
					for (i = np; i > 0; i--) {
						if (intensities[i - 1] > a) { intensities[i] = intensities[i - 1]; patterns[i] = patterns[i - 1]; }
						else break;
					}
					intensities[i] = a; patterns[i] = id;
					np++;
				}
			}
		if (c == 1) continue;
		// 2. pattern jobs, in list order
		for (int i = 0; i < np; i++) {
			const int16_t* coef = flat + patterns[i];
			FwJob j;
			if (cfg.model_id) {
				j = fw_ar_job(c ? 1 : 0, i, csubx, csuby, c ? 32 : 64, c != 0, 1, cfg.log2_scale_factor, kSeedLut[c ? 1 : 0]);
				fw_ar_taps(j, coef, 6, cfg.log2_scale_factor);
			} else {
				memset(&j, 0, sizeof(j));
				j.kind = c ? kFwFF32 : kFwFF64; j.bank = c ? 1 : 0; j.slot = i; j.csubx = csubx; j.csuby = csuby;
				j.fh = coef[1]; j.fv = coef[2]; j.seed = kSeedLut[c ? 1 : 0];
			}
			plan.jobs.push_back(j);
		}
		// 3. LUTs of the component(s)
		for (int cc = c < 1 ? c : 1; cc <= c; cc++) {
			if (cfg.comp_model_present_flag[cc]) {
				memset(plut, 255, sizeof(plut));
				for (int k = 0; k < cfg.num_intensity_intervals[cc]; k++) {
					const uint8_t a = cfg.intensity_interval_lower_bound[cc][k], b = cfg.intensity_interval_upper_bound[cc][k];
					const int32_t id = SEI_MAX_MODEL_VALUES * (k + 256 * cc);
					int i = 0;
					for (; i < kFwMaxPatterns; i++)
						if (same_pattern(patterns[i], id)) break;
					for (int l = a; l <= b; l++) {
						slut[l] = (uint8_t)cfg.comp_model_value[cc][k][0];
						if (i < kFwMaxPatterns) plut[l] = (uint8_t)(i << 4);
					}
				}
				uint8_t last = 0; // holes repeat the previous entry
				for (int k = 0; k < 256; k++) {
					if (plut[k] == 255) plut[k] = last;
					else last = plut[k];
				}
			} else {
				memset(plut, 0, sizeof(plut));
			}
			memcpy(plan.slut[cc], slut, 256);
			memcpy(plan.plut[cc], plut, 256);
		}
	}
	plan.scale_shift = cfg.log2_scale_factor - (cfg.model_id ? 1 : 0); // the AR patterns were generated one shift down
}

// vfgs_make_lut_piecewise_linear, vfgs_fw.c:649-660 (C division: truncation toward zero)
inline bool fw_piecewise_linear(uint8_t lut[256], const uint8_t in[], const uint8_t out[], int n)
{
	memset(lut, 0, 256);
	for (int k = 1; k < n; k++) {
		const int din = in[k] - in[k - 1], dout = (int)out[k] - out[k - 1];
		if (din <= 0) return false; // the reference asserts
		for (int i = 0; i <= din; i++) lut[in[k - 1] + i] = (uint8_t)(out[k - 1] + (dout * i + din / 2) / din);
	}
	return true;
}

// vfgs_init_afgs1, vfgs_fw.c:663-708
inline void fw_plan_afgs1(const fgs_afgs1& cfg, int csubx, int csuby, FwPlan& plan)
{
	plan.set_seed = true;
	plan.seed = (uint32_t)cfg.grain_seed | ((uint32_t)cfg.grain_seed << 16);
	uint8_t lut[256];
	bool ok = fw_piecewise_linear(lut, cfg.point_y_values, cfg.point_y_scaling, cfg.num_y_points);
	memcpy(plan.slut[0], lut, 256);
	if (!cfg.chroma_scaling_from_luma) ok = fw_piecewise_linear(lut, cfg.point_cb_values, cfg.point_cb_scaling, cfg.num_cb_points) && ok;
	memcpy(plan.slut[1], lut, 256);
	if (!cfg.chroma_scaling_from_luma) ok = fw_piecewise_linear(lut, cfg.point_cr_values, cfg.point_cr_scaling, cfg.num_cr_points) && ok;
	memcpy(plan.slut[2], lut, 256);
	if (!ok) { plan.error = "scaling points must be strictly increasing (vfgs_fw.c:656)"; return; }

	// grain_scale_shift + 1: the AOM Gaussian table has sigma 512, this one 63 (three shifts less than the spec's + 4)
	const int n = 2 * cfg.ar_coeff_lag * (cfg.ar_coeff_lag + 1);
	const int16_t* ar[3] = {cfg.ar_coeffs_y, cfg.ar_coeffs_cb, cfg.ar_coeffs_cr};
	for (int c = 0; c < 3; c++) {
		FwJob j = fw_ar_job(c ? 1 : 0, c == 2 ? 1 : 0, csubx, csuby, c ? 32 : 64, c != 0, cfg.grain_scale_shift + 1, cfg.ar_coeff_shift, kSeedLut[c]);
		if (!fw_ar_taps(j, ar[c], n, cfg.ar_coeff_shift)) { plan.error = "ar_coeff_lag must be 1..3 (vfgs_fw.c:454)"; return; }
		plan.jobs.push_back(j);
	}
	memset(plan.plut[0], 0, 256);
	memset(plan.plut[1], 0, 256);
	memset(plan.plut[2], 1, 256); // >> 4 in the hardware: Cr reads chroma slot 0 as well (vfgs_hw.c:212)
	plan.scale_shift = cfg.grain_scaling - 6;
	plan.set_legal = true; plan.legal = cfg.clip_to_restricted_range;
}

// The host half of a firmware update (vfgs_fw.c:592-643, :697-707 through the setters): seed, LUTs, scale shift and clip
// range into h, in the firmware's order. Returns false where the reference asserts on the scale shift (vfgs_hw.c:348);
// the seed and the LUTs are then already set, as in the reference.
inline bool fw_apply_host(HwState& h, const FwPlan& plan)
{
	if (plan.set_seed) hw_set_seed(h, plan.seed);
	for (int cc = 0; cc < 3; cc++) {
		hw_set_scale_lut(h, cc, plan.slut[cc]);
		hw_set_pattern_lut(h, cc, plan.plut[cc]);
	}
	if (plan.scale_shift < 2 || plan.scale_shift >= 8) return false;
	hw_set_scale_shift(h, plan.scale_shift);
	if (plan.set_legal) hw_set_legal_range(h, plan.legal);
	return true;
}

} // namespace vfgs
