// vfgs_core.h -- arithmetic shared by the host shim and the CUDA kernels: the LFSR and its GF(2)
// jump-ahead, the per-block offset decode, and the launch parameter block.
//
// Reference behaviour restated here (file:line under the reference's src/):
//   LFSR step                     vfgs_hw.c:74-79
//   offset bit-fields             vfgs_hw.c:99-138
//   per-line register bookkeeping vfgs_hw.c:288-312 (closed form: SURVEY.md section 8a, row A2)
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define VFGS_HD __host__ __device__ __forceinline__
#else
#define VFGS_HD inline
#endif

namespace vfgs {

// ------------------------------------------------------------------------------------ LFSR
// 31-bit Fibonacci LFSR living in bits 31..1 of the register, bit 0 is a one-step delay tail.
// Viewed as a bit-stream z[], the register after t steps is the window z[t..t+31] (bit i = z[t+i]),
// so consecutive blocks of a row are consecutive 32-bit windows of one stream.
VFGS_HD uint32_t lfsr_step(uint32_t x)
{
	return (x >> 1) | ((((x >> 1) ^ (x >> 29)) & 1u) << 31);
}

// 32-bit window starting at bit `bit` of a stream stored LSB-first in 32-bit words.
VFGS_HD uint32_t stream_window(const uint32_t* words, int bit)
{
	const int w = bit >> 5, sh = bit & 31;
	const uint32_t lo = words[w], hi = words[w + 1];
#if defined(__CUDA_ARCH__)
	return __funnelshift_r(lo, hi, sh);
#else
	return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
}

// Transition matrices over GF(2) in row form: bit i of (M x) = parity(row[i] & x).
struct Gf2Matrix {
	uint32_t row[32];
};

inline uint32_t gf2_apply(const Gf2Matrix& m, uint32_t x)
{
	uint32_t y = 0;
	for (int i = 0; i < 32; i++) y |= (uint32_t)(__builtin_popcount(m.row[i] & x) & 1) << i;
	return y;
}

inline Gf2Matrix gf2_mul(const Gf2Matrix& a, const Gf2Matrix& b) // apply b, then a
{
	Gf2Matrix o;
	for (int i = 0; i < 32; i++) {
		uint32_t acc = 0;
		for (uint32_t sel = a.row[i]; sel; sel &= sel - 1) acc ^= b.row[__builtin_ctz(sel)];
		o.row[i] = acc;
	}
	return o;
}

constexpr int kJumpBits = 64;

// pow2[k] = (one LFSR step)^(2^k), k = 0..63. Shared by the host bookkeeping and (as a flat
// uint32[64][32] table in device memory) by the stream kernel.
struct JumpTable {
	Gf2Matrix pow2[kJumpBits];
	JumpTable()
	{
		for (int i = 0; i < 31; i++) pow2[0].row[i] = 1u << (i + 1);
		pow2[0].row[31] = (1u << 1) | (1u << 29);
		for (int k = 1; k < kJumpBits; k++) pow2[k] = gf2_mul(pow2[k - 1], pow2[k - 1]);
	}
	uint32_t jump(uint32_t x, uint64_t n) const
	{
		for (int k = 0; n; k++, n >>= 1)
			if (n & 1u) x = gf2_apply(pow2[k], x);
		return x;
	}
};

// ------------------------------------------------------------------------------------ offsets
struct BlockOfs {
	int sign; // +1 / -1
	int ox;   // column of the block's window inside the pattern
	int oy;   // row (before the line-in-block term)
};

// 10-bit field -> one of 13 (x) or 12 (y) bins, times the component's step.
VFGS_HD BlockOfs decode_offsets(int c, uint32_t s, int subx, int suby)
{
	uint32_t sb, fx, fy;
	int stepx = 4, stepy = 4;
	if (c == 0) {
		sb = s >> 31;
		fx = s & 0x3ffu;
		fy = (s >> 14) & 0x3ffu;
	} else if (c == 1) {
		sb = (s >> 2) & 1u;
		fx = (s >> 10) & 0x3ffu;
		fy = (s >> 24) | ((s & 3u) << 8); // field wraps around the word
		stepx = subx > 1 ? 2 : 4; stepy = suby > 1 ? 2 : 4;
	} else {
		sb = (s >> 15) & 1u;
		fx = (s >> 20) & 0x3ffu;
		fy = (s >> 4) & 0x3ffu;
		stepx = subx > 1 ? 2 : 4; stepy = suby > 1 ? 2 : 4;
	}
	BlockOfs o;
	o.sign = sb ? -1 : 1;
	o.ox = (int)((fx * 13u) >> 10) * stepx;
	o.oy = (int)((fy * 12u) >> 10) * stepy;
	return o;
}

// ------------------------------------------------------------------------------------ division by launch constants
// q = n / d for n < 2^31 with a precomputed 33-bit reciprocal (Granlund-Montgomery round-up method):
// two instructions instead of the ~25 of a 32-bit hardware-less division, once per warp-task.
struct FastDiv {
	uint32_t m;
	int s;
};
inline FastDiv make_fastdiv(uint32_t d)
{
	FastDiv f;
	f.s = 0;
	while ((1ull << f.s) < d) f.s++;
	f.m = (uint32_t)((((1ull << f.s) - d) << 32) / d + 1);
	return f;
}
VFGS_HD uint32_t fastdiv(uint32_t n, FastDiv f)
{
#if defined(__CUDA_ARCH__)
	return (__umulhi(f.m, n) + n) >> f.s;
#else
	return (uint32_t)((((uint64_t)f.m * n) >> 32) + n) >> f.s;
#endif
}

// ------------------------------------------------------------------------------------ launch block
struct Plane {
	const uint8_t* in;
	uint8_t* out;
	long long in_row_bytes, out_row_bytes;
	int width; // in-picture samples per line
	int lines; // in-picture lines
	int vec;   // 1: every row start of in and out is aligned for 8-sample vector access
	int pad;
};

constexpr int kSamplesPerLane = 8;
constexpr int kSegSamples = 32 * kSamplesPerLane; // one warp-task covers 256 samples of a line

struct FgsParams {
	Plane comp[3];
	long long in_frame_bytes, out_frame_bytes;
	long long total_tasks;  // < 2^31 (the host splits larger batches)
	int nframes, nb, R;
	int row_begin, rows;    // block-rows [row_begin, row_begin + rows) of every frame carry tasks
	int y_begin, y_end;     // luma line range to process inside each frame
	int subx, suby;         // chroma subsampling
	int in_bytes, out_bytes; // bytes per sample (1 | 2)
	int bs, ss;             // depth - 8, effective scale shift
	int pow16;              // 1 << (16 - ss), kept opaque so the kernels multiply (FMA pipe) instead of shifting (ALU pipe)
	int lo[3], hi[3];       // clip range per component, already << bs
	int uniform_pi[3];      // pattern slot when the pattern LUT selects a single slot, else -1
	int nseg[3], tasks_per_stripe;
	FastDiv div_tps, div_rows; // reciprocals of tasks_per_stripe and rows
	// fast kernel task numbering: a component's stripes are one flat run of 8-sample lane units
	// (units_per_row * rows of them per frame), cut into warp-tasks of 32 units regardless of row ends
	int funits_per_row[3], ftasks[3], ftasks_per_frame;
	int fwide[3];           // the component's lane units are 16 samples (fgs_fast.h, wide_task_body)
	int fallwide;           // every component this launch serves is wide (selects the ALLWIDE kernel variant)
	FastDiv div_funits[3], div_ftasks;
	// table image ("blob") copied to shared memory by every CTA
	const uint8_t* blob;
	int blob_bytes;
	int lut_off;            // uint16[3][256]: scale | slot << 8
	int pat_off[2];         // luma / chroma pattern slots
	int pat_size[2];        // bytes per slot
	int pat_stride[2];      // bytes per pattern row
	// table image of the fast path (fgs_fast.h), in global memory: uint32 lut[256] = sLUT[Y] | sLUT[U]<<8 | sLUT[V]<<16,
	// then per component its single pattern slot as +pattern and -pattern, each in column-shifted copies.
	// In shared memory the three expanded LUTs sit on 32 KB boundaries of the shared window; the component
	// images go into the gap in front of the first LUT as far as they fit, the rest behind the last LUT.
	const uint8_t* fblob;
	int fimg_src[3];        // byte offset of the component's image inside fblob
	int fimg_bytes[3];      // its size (0: the component is not served by the fast kernel)
	int fimg_off[3];        // where it goes in shared memory, relative to the first LUT (negative: in front of it)
	int fpad;               // bytes between the start of dynamic shared memory and the first LUT (measured by a probe launch)
	uint32_t* probe;        // not null: the fast kernel only reports that gap here and returns (vfgs_b200.cu, ensure_ctx)
	int fsmem;              // dynamic shared memory of the launch
	int fpat_off[3][2];     // +pattern / -pattern copies, relative to the component's image
	int fpat_stride[3];
	int fpat_copy[3];       // bytes between the column-shifted copies of a pattern
	// gather path (fgs_gather.h): private LUT slot of each component (-1: none), the pattern banks' offsets inside
	// the general image and (sign-folded launches) the distance from a bank's slots to their negated copies
	int glut_index[3], ngather;
	int gpat_off[2], gneg_off[2];
	uint32_t gslot_mul[2];  // bytes per slot of each bank (fgs_gather.h, TOP layout)
	// gather kernel task numbering: a component's stripes are one flat run of 8-sample lane units, rows padded to an
	// even number of units; a warp-task holds 32 (16-sample blocks) or 30 (8-sample blocks) consecutive units
	int gunits_per_row[3], gtasks[3], gtasks_per_frame;
	FastDiv div_gunits[3], div_gtasks;
	// LFSR register per block: row (f * stream_rows + r - stream_row0) holds spitch words, word b + 1 is
	// the register of block b of that block-row (words 0 and nb + 1 are padding for the b-1 / b+1 reads)
	const uint32_t* states;
	int spitch, stream_rows, stream_row0;
	// same indexing, four uint16 per block: byte offset (inside the fast image, block sign folded in) of the
	// block's pattern window for Y, U, V (fast path only; written by lfsr_states_kernel)
	const uint16_t* woffs;
	// semi-planar frames (NV12 / P010, vfgs_b200_add_grain_semiplanar_device): U and V alternate on one plane.
	// General kernel: comp[1] / comp[2] are views of that plane starting at U0 / V0 whose samples are every second
	// one (ilv). Fast kernel (SEMI variants): comp[1] is the whole interleaved plane, comp[2] carries no tasks.
	// msb_in / msb_out: 16-bit samples hold the value in bits 15..6 (P010): shift on load / store.
	int ilv[3];
	int msb_in, msb_out;
};

} // namespace vfgs
