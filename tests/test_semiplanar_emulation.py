"""Semi-planar frames (NV12 / P010) through the host build of the kernels' task code (tests/emu/emu_semiplanar.cpp,
emu_add_grain_semiplanar), against the oracle's planar output converted; and the argument checks of
vfgs_b200_add_grain_semiplanar_device, which need no GPU."""

import numpy as np
import pytest

from tests.semiplanar import INTERLEAVED, Surface, load_emu, planar_to_semi, run_emu_semi, semi_to_planar
from tests.util import Oracle, load_golden, program_case, synth_frames

G = load_golden()
CASES = [c for c in G.runnable() if G.cases[c]["fmt"] in ("420", "422")]
WIDE = 64


@pytest.fixture(scope="module")
def emu():
    return load_emu()


def csub(fmt):
    return 2 if fmt == "420" else 1


def run_case(emu, case, w, h, n, p010_out=None, mode=0, offset=0, pad_y=0, pad_uv=0, seed=1, in_place=False, frames=None,
             legal=None):
    """One semi-planar call of golden case `case` on synthetic frames; returns (got planar, want planar, mask, out Y, out UV)."""
    meta = G.cases[case]
    depth, fmt = meta["depth"], meta["fmt"]
    p010 = depth == 10
    p010_out = p010 if p010_out is None else p010_out
    o = Oracle(); program_case(o, G, case)
    if legal is not None:
        o.vfgs_set_legal_range(legal)
    if frames is None:
        frames = synth_frames(n, w, h, fmt, depth, seed=seed)
    rng = np.random.default_rng(seed)
    Y, UV = planar_to_semi(frames, n, w, h, fmt, p010, rng=rng)  # P010: random low bits, which must be ignored
    ch = h // csub(fmt)
    isz, osz = (2 if p010 else 1), (2 if p010_out else 1)
    src = Surface(n, w, h, ch, isz, w * isz + pad_y, w * isz + pad_uv, offset)
    src.fill(Y, UV)
    dst = src if in_place else Surface(n, w, h, ch, osz, w * osz + pad_y, w * osz + pad_uv, offset)
    mask = run_emu_semi(emu, o, src, dst, n, w, h, p010_out, mode=mode)
    want = o.add_grain_frames(frames, n, w, h, 8 if (p010 and not p010_out) else 0)
    oy, ouv = dst.planes()
    return semi_to_planar(oy, ouv, p010_out), want, mask, oy, ouv


def formats(case):
    return (True, False) if G.cases[case]["depth"] == 10 else (False,)


@pytest.mark.parametrize("case", CASES)
def test_semiplanar_equals_oracle(emu, case):
    """NV12 (8-bit), P010 and P010 -> NV12 (10-bit), modes 0/1/2, a few geometries: the output converted to planar is the
    oracle's planar output; P010 input carries random low bits, P010 output has them zero."""
    for (w, h, n) in ((512, 56, 2), (264, 40, 2), (144, 34, 1)):
        for p010_out in formats(case):
            for mode in (0, 1, 2):
                got, want, mask, oy, ouv = run_case(emu, case, w, h, n, p010_out=p010_out, mode=mode, seed=w + mode)
                assert np.array_equal(got, want), (case, w, h, p010_out, mode, int(np.count_nonzero(got != want)))
                assert mode != 1 or mask == 2
                if p010_out and G.cases[case]["depth"] == 10:
                    assert not (oy & 63).any() and not (ouv & 63).any()


def test_interleaved_path_is_taken_where_expected(emu):
    """The fast kernel's interleaved U/V lane runs when both chroma components are single-slot, the width is a multiple of
    16 and the UV plane allows one 32-byte (P010) / 16-byte (NV12) access per line and lane; otherwise U and V take the
    general code together. P010 luma: wide fast path or general; NV12 luma keeps its planar kernels (EDGE if not wide)."""
    afgs, nv = "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei_ff_test1.cfg|d8|420|g100"

    def check(case, w, h, expect, **kw):
        got, want, mask, _, _ = run_case(emu, case, w, h, 1, **kw)
        assert np.array_equal(got, want), (case, w, h, kw)
        assert mask == expect, (case, w, h, kw, mask)

    F = 1 | WIDE | INTERLEAVED
    check(afgs, 512, 64, F)                                  # P010, aligned: everything on the fast kernel
    check(afgs, 512, 64, F, p010_out=False)                  # P010 -> NV12
    check(afgs, 512, 64, F, pad_y=64, pad_uv=32)             # padded pitches, multiples of 32 bytes
    check(afgs, 512, 64, 2, offset=16)                       # P010 planes 16 bytes off a 32-byte boundary: general code
    check(afgs, 512, 64, 1 | WIDE | 2, pad_uv=16)            # UV pitch not a multiple of 32: U and V general, luma wide
    check(afgs, 520, 40, 2)                                  # width a multiple of 8, not of 16
    check(nv, 512, 64, F)                                    # NV12, aligned
    check(nv, 512, 64, 2 | 32, offset=8)                     # NV12 8 bytes off: UV general, luma the planar EDGE variant
    check(nv, 520, 40, 2 | 32)                               # NV12 width % 16 == 8
    check(afgs, 1366, 768, 2)                                # ragged picture sizes: interleaved chroma and P010 luma general
    check(afgs, 1928, 1080, 2)
    check(nv, 1366, 768, 2 | 32)                             # NV12 luma keeps its planar kernel
    check(nv, 1928, 1080, 2 | 32)
    check("fgs_sei.cfg|d10|420|g100", 512, 64, F | 4 | 8)           # default SEI: P010 luma on the gather kernel
    check("fgs_sei_ff_test5.cfg|d10|420|g100", 512, 64, 1 | WIDE | 2)     # sample-adaptive chroma: U and V general


def test_p010_low_bits_are_ignored(emu):
    """Two inputs that differ only in the low 6 bits of every P010 word give the same output, with zero low bits."""
    case = "fgs_afgs1_test1.cfg|d10|420|g100"
    for w in (512, 264):
        a = run_case(emu, case, w, 40, 1, seed=3)
        b = run_case(emu, case, w, 40, 1, seed=4, frames=synth_frames(1, w, 40, "420", 10, seed=3))
        assert np.array_equal(a[3], b[3]) and np.array_equal(a[4], b[4]) and np.array_equal(a[0], a[1])
        assert not (a[3] & 63).any() and not (a[4] & 63).any()


def test_10_to_8_at_the_ceiling(emu):
    """P010 -> NV12 of samples at the 10-bit ceiling with the full range legal: (x + 2) >> 2 tops out at 255."""
    case = "fgs_afgs1_test1.cfg|d10|420|g100"
    rng = np.random.default_rng(9)
    for (w, h) in ((512, 40), (272, 34)):
        frames = rng.integers(1016, 1024, size=w * h * 3 // 2, dtype=np.uint16)
        got, want, mask, _, _ = run_case(emu, case, w, h, 1, p010_out=False, frames=frames, legal=0)
        assert np.array_equal(got, want) and want.max() == 255, (w, h, mask)


@pytest.mark.parametrize("case,expect_general", [("fgs_afgs1_test1.cfg|d10|420|g100", False), ("fgs_sei_ff_test1.cfg|d8|420|g100", False),
                                                 ("fgs_sei_ff_test5.cfg|d10|420|g100", True), ("fgs_sei.cfg|d10|420|g100", False)])
def test_in_place(emu, case, expect_general):
    """in == out: single-slot configs stay on the fast kernel; sample-adaptive chroma (ff_test5) runs the general code
    through the two-plane scratch buffer; sample-adaptive P010 luma takes the gather kernel's shifted numbering."""
    for (w, h, n) in ((512, 56, 2), (264, 40, 1)):
        got, want, mask, _, _ = run_case(emu, case, w, h, n, in_place=True, pad_uv=32, seed=w)
        assert np.array_equal(got, want), (case, w, h, mask)
        assert bool(mask & 2) == (expect_general or w == 264), mask  # width 264: not a multiple of 16


# ---- argument checks of the library (no GPU needed) ------------------------------------------------------------------
@pytest.fixture(scope="module")
def hw():
    from versatilefilmgrain_b200 import VfgsHw
    h = VfgsHw()
    yield h
    h.reset()


def rc_of(hw, pin, pout, n, w, h):
    from versatilefilmgrain_b200.api import VfgsError
    try:
        hw.add_grain_semiplanar_device(pin, pout, n, w, h)
    except VfgsError as e:
        return int(str(e).split("error ")[1].split(":")[0])
    return 0


def test_arguments_are_refused_before_any_device_work(hw):
    import torch
    from versatilefilmgrain_b200.api import NV12, P010, SemiPlanes
    w, h, n = 256, 144, 3
    ok = (0,) if torch.cuda.is_available() else (3,)  # legal calls get past the checks: VFGS_B200_ERR_CUDA without a device
    base = 0x10000000

    def surf(b, fmt, sample=2):
        pitch = w * sample
        return SemiPlanes(b, b + h * pitch, pitch, pitch, (h + h // 2) * pitch, fmt)

    hw.reset()
    hw.vfgs_set_depth(10)
    fb = (h + h // 2) * w * 2
    if not torch.cuda.is_available():
        assert rc_of(hw, surf(base, P010), surf(base, P010), n, w, h) in ok                  # in place
        assert rc_of(hw, surf(base, P010), surf(base + n * fb, P010), n, w, h) in ok         # disjoint
        assert rc_of(hw, surf(base, P010), surf(base + n * fb, NV12, 1), n, w, h) in ok      # P010 -> NV12
    assert rc_of(hw, surf(base, NV12, 1), surf(base + n * fb, NV12, 1), n, w, h) == 1       # format / depth mismatch
    assert rc_of(hw, surf(base, P010), surf(base + fb, P010), n, w, h) == 1                 # output one frame behind
    assert rc_of(hw, surf(base, P010), surf(base + 64, P010), n, w, h) == 1                 # shifted by a few bytes
    assert rc_of(hw, surf(base, P010), surf(base, NV12, 1), n, w, h) == 1                   # in place across formats
    shared_uv = surf(base + n * fb, P010); shared_uv.uv = surf(base, P010).uv                # only the UV planes alias
    if not torch.cuda.is_available():
        assert rc_of(hw, surf(base, P010), shared_uv, n, w, h) in ok                         # (identical: in place for that plane)
    y_over_uv = surf(base + n * fb, P010); y_over_uv.y = surf(base, P010).uv                # output luma over the input chroma
    assert rc_of(hw, surf(base, P010), y_over_uv, n, w, h) == 1
    odd = surf(base, P010); odd.uv += 1
    assert rc_of(hw, odd, surf(base + n * fb, P010), n, w, h) == 1                          # odd P010 address
    odd = surf(base, P010); odd.stride_uv += 1; odd.frame_stride += 2 * h
    assert rc_of(hw, odd, surf(base + n * fb, P010), n, w, h) == 1                          # odd P010 stride
    short = surf(base, P010); short.stride_y = w * 2 - 2
    assert rc_of(hw, short, surf(base + n * fb, P010), n, w, h) == 1                        # stride shorter than a row
    null = surf(base, P010); null.uv = None
    assert rc_of(hw, null, surf(base + n * fb, P010), n, w, h) == 1                         # null plane
    hw.vfgs_set_chroma_subsampling(1, 1)
    assert rc_of(hw, surf(base, P010), surf(base + 4 * n * fb, P010), n, w, h) == 1         # 4:4:4
    hw.reset()
    hw.vfgs_set_depth(8)
    assert rc_of(hw, surf(base, NV12, 1), surf(base + n * fb, P010), n, w, h) == 1          # NV12 -> P010
    assert rc_of(hw, surf(base, P010), surf(base + n * fb, P010), n, w, h) == 1             # P010 at depth 8
    hw.reset()
