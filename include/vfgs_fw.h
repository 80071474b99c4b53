/*
 * vfgs_fw.h -- the reference's firmware-layer interface (src/vfgs_fw.h:40-96) with the pattern synthesis on the GPU.
 *
 * The reference's firmware (src/vfgs_fw.c) turns film grain metadata -- an FGC SEI message in frequency-filtering
 * or auto-regressive mode, or AOM AFGS1 metadata -- into "hardware" state through the setters of vfgs_hw.h: up to
 * 8 + 8 grain patterns, six 256-entry LUTs and a few scalars. Everything is cheap except the patterns (a 64 x 64
 * integer inverse DCT, src/vfgs_fw.c:297-408, or a causal auto-regressive filter in raster order, :410-502), which
 * matter when the metadata changes per picture.
 *
 * vfgs_b200_init_sei / vfgs_b200_init_afgs1 do what vfgs_init_sei / vfgs_init_afgs1 do (same structs, same
 * resulting hardware state, bit for bit), but synthesise the patterns with CUDA kernels on the library's table
 * stream. Frames already queued keep the tables they were launched with; the call waits only for its own small
 * kernels, never for the grain kernels (no device-wide synchronisation).
 *
 * They are additive: the reference's own vfgs_fw.c keeps working unchanged on top of the vfgs_hw.h setters
 * (tests/test_fw_dropin.py). To switch a caller over, replace its two calls (src/vfgs_main.c:754-757, 777-780):
 *     vfgs_init_afgs1(&afgs1)  ->  vfgs_b200_init_afgs1(&afgs1)
 *     vfgs_init_sei(&sei)      ->  vfgs_b200_init_sei(&sei)
 * The struct layouts below are those of src/vfgs_fw.h:53-91 (the interface, not an implementation).
 */
#ifndef VFGS_B200_FW_H
#define VFGS_B200_FW_H

#include <stdint.h>

#include "vfgs_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

#define SEI_MAX_MODEL_VALUES 6

/* FGC SEI message (ITU-T H.274 8.5 film grain characteristics), src/vfgs_fw.h:53-62 */
typedef struct fgs_sei_s {
	uint8_t  model_id;                    /* 0 frequency filtering, 1 auto-regressive */
	uint8_t  log2_scale_factor;
	uint8_t  comp_model_present_flag[3];
	uint16_t num_intensity_intervals[3];
	uint8_t  num_model_values[3];
	uint8_t  intensity_interval_lower_bound[3][256];
	uint8_t  intensity_interval_upper_bound[3][256];
	int16_t  comp_model_value[3][256][SEI_MAX_MODEL_VALUES];
} fgs_sei;

/* AOM AFGS1 metadata (ITU-T T.35), src/vfgs_fw.h:64-91 */
typedef struct fgs_afgs1_s {
	uint16_t grain_seed;
	uint8_t  num_y_points;
	uint8_t  point_y_values[14];
	uint8_t  point_y_scaling[14];
	uint8_t  chroma_scaling_from_luma;
	uint8_t  num_cb_points;
	uint8_t  point_cb_values[10];
	uint8_t  point_cb_scaling[10];
	uint8_t  num_cr_points;
	uint8_t  point_cr_values[10];
	uint8_t  point_cr_scaling[10];
	uint8_t  grain_scaling;
	uint8_t  ar_coeff_lag;
	int16_t  ar_coeffs_y[24];
	int16_t  ar_coeffs_cb[25];
	int16_t  ar_coeffs_cr[25];
	uint8_t  ar_coeff_shift;
	uint8_t  grain_scale_shift;
	uint8_t  cb_mult;
	uint8_t  cb_luma_mult;
	uint16_t cb_offset;
	uint8_t  cr_mult;
	uint8_t  cr_luma_mult;
	uint16_t cr_offset;
	uint8_t  overlap_flag;
	uint8_t  clip_to_restricted_range;
} fgs_afgs1;

/* src/vfgs_fw.c:517-644 and :663-708 with the pattern synthesis on the device. Return VFGS_B200_OK or an error code
 * of vfgs_b200.h (text in vfgs_b200_last_error()); depth and chroma subsampling must have been set before, as for
 * the reference (src/vfgs_main.c:750-757). */
int vfgs_b200_init_sei(const fgs_sei* cfg);
int vfgs_b200_init_afgs1(const fgs_afgs1* cfg);

/* ---- Metadata of grain sessions (vfgs_b200.h): many sessions re-programmed in one asynchronous device call ----------
 *
 * Film grain metadata can change with every picture. One entry gives one session new metadata; one call takes a whole
 * list, e.g. every stream of a round, and costs one kernel launch, one copy of the entries to the device and one copy
 * of the new patterns back. The global state, its table images and the global firmware's working memory are not
 * touched. */
typedef struct vfgs_b200_session_metadata {
	vfgs_b200_session* session;
	const fgs_sei*     sei;    /* exactly one of the two is set */
	const fgs_afgs1*   afgs1;
} vfgs_b200_session_metadata;

/* n entries, asynchronous on `stream` (a cudaStream_t, NULL = default stream).
 *   State: each entry leaves its session in exactly the state vfgs_b200_init_sei / _afgs1 would leave the global state
 *   in, were the session's state the global one: patterns, LUTs, scale shift, clip range and registers (AFGS1 reseeds
 *   and sets the clip range; SEI leaves the registers alone: vfgs_b200_session_set_seed). Each session has its own copy
 *   of the firmware's working memory, taken from the global one when the session was created, so a session behaves like
 *   its own copy of the reference's process from that point on (with 4:2:2 / 4:4:4, the chroma patterns of an SEI
 *   message read what earlier patterns left in that memory).
 *   Ordering: jobs enqueued after the call, on any stream, use the new metadata; jobs enqueued before keep the old
 *   tables, even while they still run (the call's device work waits on the device for them). The call never waits on
 *   the host for device work, except to reuse its own page-locked staging two calls later, or when that staging grows.
 *   vfgs_b200_session_get_state waits for the new patterns to arrive on the host.
 *   Refused with VFGS_B200_ERR_ARG / _ERR_STATE before any device work or any change to any session: n < 0, a null
 *   list or session, both or neither metadata pointers set, the same session twice, non-increasing AFGS1 scaling points,
 *   ar_coeff_lag outside 1..3, more patterns than the hardware holds, a scale shift outside 2..7 (scale_shift + bs
 *   outside 8..13), table images that do not fit shared memory. A refused call leaves every session as it was. (This is
 *   stricter than vfgs_b200_init_sei / _afgs1, which, like the reference, have already set the LUTs when they refuse a
 *   scale shift.) */
int vfgs_b200_session_init_metadata(const vfgs_b200_session_metadata* list, int n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VFGS_B200_FW_H */
