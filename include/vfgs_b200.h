/*
 * vfgs_b200.h -- additive C-ABI of libvfgs_b200.so (plain pointers and sizes, no C++/torch types).
 *
 * The reference drives its hardware layer one picture line at a time (src/vfgs_main.c:664-682
 * calling vfgs_add_grain_line, src/vfgs_hw.c:288). A GPU wants whole frames, so the frame loop of
 * src/vfgs_main.c:771-790 (read -> vfgs_add_grain -> optional yuv_to_8bit -> write) gets these
 * batch entry points. They share one hardware state (the mirror of src/vfgs_hw.c:49-63) with the
 * drop-in setters of vfgs_hw.h and leave the LFSR registers exactly where the reference's line walk
 * would, so frame calls and line calls can be interleaved bit-exactly.
 *
 * Frame layout ("packed planar", the .yuv file layout of src/yuv.c:162-214): per frame the Y plane
 * (width x height), then U, then V (each (width/subx) x (height/suby)), rows tightly packed, frames
 * back to back. Samples are uint8 when the configured depth is 8 and little-endian uint16 when it
 * is 10. out_depth = 0 keeps the input depth; out_depth = 8 with 10-bit input fuses the
 * (v + 2) >> 2 conversion of src/yuv.c:216-258 into the store.
 *
 * All functions return VFGS_B200_OK or an error code; vfgs_b200_last_error() gives the text.
 * Nothing here falls back to the CPU.
 */
#ifndef VFGS_B200_H
#define VFGS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VFGS_B200_OK         0
#define VFGS_B200_ERR_ARG    1 /* bad argument (size, depth, null pointer, aliasing) */
#define VFGS_B200_ERR_STATE  2 /* hw state the reference would assert on (src/vfgs_hw.c:167-170) */
#define VFGS_B200_ERR_CUDA   3 /* CUDA runtime error, text in vfgs_b200_last_error() */

/* Planes with explicit strides, for callers whose frames are not packed (src/yuv.c:54-87 pads
 * strides to 64 samples). All strides are in BYTES. */
typedef struct vfgs_b200_planes {
	void*   y;
	void*   u;
	void*   v;
	int64_t stride_y;      /* between luma lines */
	int64_t stride_c;      /* between chroma lines */
	int64_t frame_stride;  /* between consecutive frames, same for the three planes */
} vfgs_b200_planes;

/* Semi-planar frames, the layout of hardware video decoders and encoders: per frame a Y plane, then one plane in which
 * U and V alternate on every chroma line. All strides are in BYTES. */
#define VFGS_B200_NV12 1  /* 8-bit samples: Y plane, then one plane of interleaved U,V pairs (NV12 / NV16) */
#define VFGS_B200_P010 2  /* 10-bit samples in bits 15..6 of little-endian uint16 (P010 / P210) */

typedef struct vfgs_b200_semiplanar {
	void*   y;
	void*   uv;            /* U0 V0 U1 V1 ... on every chroma line */
	int64_t stride_y;      /* bytes between luma lines */
	int64_t stride_uv;     /* bytes between chroma lines */
	int64_t frame_stride;  /* bytes between consecutive frames, same for both planes */
	int     format;        /* VFGS_B200_NV12 | VFGS_B200_P010 */
} vfgs_b200_semiplanar;

/* Bind the library to a CUDA device (default: the current device at first use). */
int vfgs_b200_init(int device);
/* Hardware state back to the power-on values of src/vfgs_hw.c:49-63. */
int vfgs_b200_reset(void);
const char* vfgs_b200_last_error(void);

/* Bytes of one packed planar frame at the given depth with the configured chroma subsampling. */
size_t vfgs_b200_frame_bytes(int width, int height, int depth);

/* nframes packed planar frames already in DEVICE memory; asynchronous on `stream` (a cudaStream_t,
 * NULL = default stream). in == out (every plane identical, same strides) is allowed when the depths
 * match: the kernels then read nothing but what they overwrite themselves; only components with
 * sample-adaptive pattern selection AND 8-sample blocks or ragged / unaligned rows take a detour through a
 * scratch buffer (two extra passes over the data). Input and output that overlap in any other way are
 * refused with VFGS_B200_ERR_ARG. */
int vfgs_b200_add_grain_frames_device(const void* in, void* out, int nframes, int width, int height,
                                      int out_depth, void* stream);

/* Same with explicit planes/strides (device memory). Any sample-aligned pointers and strides are accepted and give the
 * same output; the speed depends on them: planes, line strides and the frame stride that are multiples of 32 bytes
 * (16 for 8-bit samples), with widths that are multiples of 16 samples, take the 16-samples-per-lane kernels
 * (packed frames of the usual picture sizes in cudaMalloc'd memory qualify); multiples of 16 bytes / 8 samples the
 * 8-samples-per-lane form; anything else the EDGE variant (DESIGN.md section 4). */
int vfgs_b200_add_grain_planes_device(const vfgs_b200_planes* in, const vfgs_b200_planes* out,
                                      int nframes, int width, int height, int out_depth, void* stream);

/* nframes semi-planar frames in DEVICE memory; asynchronous on `stream`. The chroma geometry is that of the planar
 * calls: a UV line holds cw = width / subx pairs, the plane has ch = height / suby lines.
 *   Output: the input deinterleaved, P010 samples taken as word >> 6, run through the planar path, and the result
 *   reinterleaved with P010 samples written as value << 6, bit for bit; the LFSR registers advance exactly as for a
 *   planar call of the same size, so semi-planar, planar and line calls and vfgs_b200_skip_frames interleave
 *   bit-exactly. The low 6 bits of P010 input are ignored and written as zero.
 *   Formats: in->format must match the configured depth (NV12 <-> 8, P010 <-> 10); out->format is in->format, or
 *   NV12 from P010 (the fused (v + 2) >> 2 conversion of out_depth = 8). Only 4:2:0 and 4:2:2 are accepted (4:4:4
 *   frames are planar: vfgs_b200_add_grain_planes_device).
 *   in == out (same pointers, strides and format) is allowed; any other overlap, null pointers, line strides shorter
 *   than a row and P010 planes or strides that are not 2-byte aligned are refused with VFGS_B200_ERR_ARG before any
 *   device work.
 *   Speed: with single-pattern chroma, widths that are multiples of 16 and planes, line strides and frame stride that
 *   are multiples of 32 bytes (P010; 16 for NV12), U and V run on the fast kernel's interleaved lane; P010 luma takes
 *   the 16-samples-per-lane fast path under the same conditions, or the gather kernel for sample-adaptive patterns.
 *   Everything else takes the general kernel, which is correct everywhere and not fast (DESIGN.md section 13). */
int vfgs_b200_add_grain_semiplanar_device(const vfgs_b200_semiplanar* in, const vfgs_b200_semiplanar* out,
                                          int nframes, int width, int height, void* stream);

/* nframes packed planar frames in HOST memory; returns when `out` is complete. Frames are cut into
 * chunks that flow through a ring of device buffers on three streams (H2D / kernels / D2H) so the
 * copies of neighbouring chunks overlap the kernels. Give it pinned buffers (vfgs_b200_host_alloc)
 * for the copies to be asynchronous; pageable buffers work, but the CUDA runtime then stages them
 * and the overlap is lost. in == out is allowed when the depths match. */
int vfgs_b200_add_grain_frames_host(const void* in, void* out, int nframes, int width, int height,
                                    int out_depth);

/* Advance the LFSR registers as if `nframes` frames of this size had been processed (GF(2)
 * jump-ahead, no GPU work): this is how a rank that owns frames [k, k+m) of a sequence gets the
 * state of frame k without touching frames 0..k-1. */
int vfgs_b200_skip_frames(int64_t nframes, int width, int height);

/* Raw LFSR registers in the order rnd, rnd_up, line_rnd, line_rnd_up (src/vfgs_hw.c:52-55). */
void vfgs_b200_get_lfsr(uint32_t regs[4]);
void vfgs_b200_set_lfsr(const uint32_t regs[4]);

/* Copy of the mirrored hardware state, laid out like the reference's statics (src/vfgs_hw.c:49-63):
 * int8 pattern[2][9][64][64], uint8 sLUT[3][256], uint8 pLUT[3][256], uint32 rnd, rnd_up, line_rnd,
 * line_rnd_up, then int scale_shift, bs, Y_min, Y_max, C_min, C_max, csubx, csuby. Returns the size
 * needed; nothing is written when cap is smaller. Needs no GPU. */
size_t vfgs_b200_get_state(void* dst, size_t cap);

/* Page-locked host memory for the host entry point. */
void* vfgs_b200_host_alloc(size_t bytes);
void  vfgs_b200_host_free(void* p);

/* Number of CUDA kernels this library has launched since load (for launch accounting). */
uint64_t vfgs_b200_launch_count(void);

/* Measurement aid: with timing enabled every grain-kernel launch is bracketed by CUDA events on its
 * own stream; vfgs_b200_kernel_time() waits for them and returns the accumulated device time and
 * launch count since timing was (re-)enabled. */
int vfgs_b200_kernel_timing(int enable);
int vfgs_b200_kernel_time(double* total_ms, uint64_t* launches);

/* Test aid: kernel selection. 0 = automatic (fast kernel for single-pattern components -- its EDGE variant
 * for ragged / unaligned rows --, gather kernel for sample-adaptive ones, general kernel for sample-adaptive
 * components on ragged / unaligned rows), 1 = general kernel for everything, 2 = gather kernel wherever it
 * can run. All of them are CUDA paths. */
void vfgs_b200_force_general_kernel(int mode);

/* Frame pipeline behind include/yuv.h: out[0] = frames processed, out[1] = batches flushed. */
void vfgs_b200_pipeline_stats(unsigned long long out[2]);

/* Geometry of the last grain kernel launch: out[0]=grid, out[1]=block, out[2]=dynamic smem bytes,
 * out[3]=SM count of the bound device, out[4]=which grain kernels the last frame call launched
 * (bit 0 fast, bit 1 general, bit 2 gather, bit 3 the fast kernel's EDGE variant, bit 4 the fast kernel's interleaved
 * U/V lane of semi-planar frames). */
void vfgs_b200_last_launch(int out[5]);

/* ---- Grain sessions: many video streams, each with its own grain state, served by one batched call ----------------
 *
 * A session owns a copy of one complete hardware state (patterns, LUTs, scalars, the four LFSR registers) and that
 * state's table images in device memory, built once. Calls on sessions neither read nor change the global state of the
 * setters, vfgs_b200_init_sei / _afgs1 and the frame entry points above; setters do not affect existing sessions, and
 * vfgs_b200_reset leaves them alive. A session belongs to the device the library is bound to. Like the rest of the
 * library, sessions and job calls are used from one thread at a time. */
typedef struct vfgs_b200_session vfgs_b200_session;

/* Snapshot of the current hardware state (whatever the setters / vfgs_b200_init_sei / _afgs1 programmed, LFSR registers
 * included), with its table images uploaded asynchronously to session-owned device memory. VFGS_B200_ERR_STATE when
 * the state could never add grain (a pattern LUT entry above slot 8, scale_shift + bs outside 8..13). */
int  vfgs_b200_session_create(vfgs_b200_session** out);
/* Waits for the kernels that read this session (its last use only), then frees it. NULL is a no-op. */
void vfgs_b200_session_destroy(vfgs_b200_session* s);
/* The session's LFSR registers, order as vfgs_b200_get_lfsr. */
void vfgs_b200_session_get_lfsr(const vfgs_b200_session* s, uint32_t regs[4]);
void vfgs_b200_session_set_lfsr(vfgs_b200_session* s, const uint32_t regs[4]);
/* vfgs_b200_skip_frames on the session's registers. */
int  vfgs_b200_session_skip_frames(vfgs_b200_session* s, int64_t nframes, int width, int height);
/* vfgs_set_seed on the session's registers: seed << 1 into all four (src/vfgs_hw.c:339-344). SEI metadata never seeds
 * (the reference's CLI seeds separately, src/vfgs_main.c:759-760). */
int  vfgs_b200_session_set_seed(vfgs_b200_session* s, uint32_t seed);
/* The session's state in the layout of vfgs_b200_get_state. */
size_t vfgs_b200_session_get_state(const vfgs_b200_session* s, void* dst, size_t cap);

/* One job: nframes frames of one session, in device memory. */
typedef struct vfgs_b200_job {
	vfgs_b200_session* session;
	const vfgs_b200_planes* in;         /* planar frames ... */
	const vfgs_b200_planes* out;
	const vfgs_b200_semiplanar* sp_in;  /* ... or semi-planar ones: exactly one of the two pairs is set */
	const vfgs_b200_semiplanar* sp_out;
	int nframes, width, height;
	int out_depth;                      /* planar jobs, as in vfgs_b200_add_grain_planes_device; 0 for semi-planar */
} vfgs_b200_job;

/* njobs jobs in DEVICE memory, asynchronous on `stream`. Output and the registers of every session afterwards are
 * exactly what one vfgs_b200_add_grain_planes_device / _semiplanar_device call per job, in list order, would give, each
 * made on its session's state and registers. A session may appear in several jobs; each then starts where the previous
 * one left its registers (which advance on the host at enqueue).
 *   Launches: one LFSR stream-kernel launch for all jobs, then one grain launch per kernel instantiation the jobs need
 *   (the fast kernel's variants, its EDGE variant, the gather kernel's variants). A job whose plan needs the general
 *   kernel, or in place the scratch detour, runs on its own through the single-job route.
 *   Refused with VFGS_B200_ERR_ARG / _ERR_STATE before any device work: everything the single-job entry points refuse,
 *   a null session, both or neither plane pairs set, njobs < 0, and buffers of two jobs that overlap (in place within
 *   one job is allowed as in the single-job calls). */
int vfgs_b200_add_grain_jobs_device(const vfgs_b200_job* jobs, int njobs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VFGS_B200_H */
