"""The C-ABI library builds for sm_100a, loads without a GPU and exports every symbol that
include/*.h declares; the host-side state machine behaves like the reference's setters."""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

from tests.util import Oracle, load_golden, program_case, states_equal
from versatilefilmgrain_b200 import api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = load_golden()


def declared_functions():
    names = []
    for hdr in ("vfgs_hw.h", "vfgs_b200.h", "vfgs_fw.h"):
        text = open(os.path.join(ROOT, "include", hdr)).read()
        text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
        names += re.findall(r"\b(vfgs_[a-z0-9_]+)\s*\(", text)
    return sorted(set(names))


def test_headers_declare_what_the_module_binds():
    assert set(declared_functions()) == set(api.HW_SYMBOLS + api.B200_SYMBOLS)


def test_library_exports_every_declared_symbol(hw_lib):
    for name in declared_functions():
        assert hasattr(hw_lib.L, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", api.LIB_PATH], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (vfgs_\w+)", out))
    assert set(declared_functions()) <= exported


def test_library_exports_the_yuv_layer(hw_lib):
    """include/yuv.h: the reference's seven yuv.h entry points (src/yuv.h:60-66), batched implementation."""
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "yuv.h")).read(), flags=re.S)
    names = sorted(set(re.findall(r"\b(yuv_[a-z0-9_]+)\s*\(", text)))
    assert names == ["yuv_alloc", "yuv_free", "yuv_pad", "yuv_read", "yuv_skip", "yuv_to_8bit", "yuv_write"]
    for n in names:
        assert hasattr(hw_lib.L, n), n


def test_library_carries_sm100a_code_only():
    out = subprocess.run(["cuobjdump", "-lelf", api.LIB_PATH], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, out


def test_headers_compile_as_c(tmp_path):
    src = tmp_path / "t.c"
    src.write_text('#include "vfgs_hw.h"\n#include "vfgs_b200.h"\nint main(void){ vfgs_b200_planes p; (void)p; return VFGS_MAX_PATTERNS == 8 ? 0 : 1; }\n')
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-c", str(src), "-o", str(tmp_path / "t.o")], check=True)


@pytest.mark.parametrize("case", [c for c in G.runnable()][::6])
def test_setters_mirror_reference_state(hw_lib, case):
    """Programming the shim through vfgs_hw.h reproduces the state the reference firmware left in
    vfgs_hw.c's statics (golden fixture)."""
    hw_lib.reset()
    st = program_case(hw_lib, G, case)
    assert states_equal(hw_lib.state(), st) == []


def test_scale_shift_depth_ordering(hw_lib):
    for seq in ([("depth", 10), ("shift", 5), ("depth", 8)], [("shift", 3), ("depth", 10), ("depth", 10)],
                [("depth", 10), ("depth", 8), ("shift", 7), ("depth", 10)]):
        hw_lib.reset()
        o = Oracle()
        for what, v in seq:
            for hw in (hw_lib, o):
                (hw.vfgs_set_depth if what == "depth" else hw.vfgs_set_scale_shift)(v)
        assert np.array_equal(hw_lib.state()["scalars"], o.state()["scalars"]), seq


def test_chroma_pattern_repacking_uses_current_subsampling(hw_lib):
    rng = np.random.default_rng(3)
    for sx, sy in ((2, 2), (2, 1), (1, 1)):
        hw_lib.reset()
        o = Oracle()
        P = rng.integers(-127, 128, size=64 * 64, dtype=np.int8)
        for hw in (hw_lib, o):
            hw.vfgs_set_chroma_subsampling(sx, sy)
            hw.vfgs_set_chroma_pattern(3, P)
            hw.vfgs_set_luma_pattern(7, P)
        assert states_equal(hw_lib.state(), o.state()) == []


def test_seed_and_skip_frames_bookkeeping(hw_lib):
    """vfgs_set_seed stores seed<<1; skip_frames lands where processing the frames would
    (closed form of vfgs_hw.c:291-298; oracle runs the real thing)."""
    from tests.util import synth_frames
    case = "fgs_sei_ff_test1.cfg|d10|420|g100"
    for (w, h, n) in ((256, 152, 3), (208, 136, 1), (256, 16 * 9, 5), (144, 16, 2) if False else (256, 144, 2)):
        hw_lib.reset()
        program_case(hw_lib, G, case)
        hw_lib.vfgs_set_seed(4242)
        assert hw_lib.get_lfsr() == [8484] * 4
        o = Oracle(); program_case(o, G, case); o.vfgs_set_seed(4242)
        o.add_grain_frames(synth_frames(n, w, h, "420", 10, seed=1), n, w, h, 0)
        hw_lib.skip_frames(n, w, h)
        assert hw_lib.get_lfsr() == o.get_lfsr(), (w, h, n)


def test_lfsr_jump_known_answers(hw_lib):
    """Host jump-ahead of the shim against the reference's serial prng (fixture KATs): a 1-block-row
    frame geometry makes skip_frames(n) == n * nb single steps on line_rnd... use nb = 9, R = 2."""
    o = Oracle()
    for start in (0xdeadbeef, 0x615f615e, 24690):
        for n in (1, 2, 7, 1000, 123457):
            hw_lib.reset()
            hw_lib.set_lfsr([start] * 4)
            hw_lib.skip_frames(n, 144, 32)  # nb = 9, R = 2 -> advance n * 9 steps
            regs = hw_lib.get_lfsr()
            assert regs[2] == o.lfsr_jump(start, 9 * n)
            assert regs[3] == o.lfsr_jump(start, 9 * n - 9)
            assert regs[0] == o.lfsr_jump(start, 9 * n + 9)


def test_frame_api_rejects_bad_arguments_without_touching_a_gpu(hw_lib):
    hw_lib.reset()
    L = hw_lib.L
    buf = np.zeros(16, dtype=np.uint16)
    p = buf.ctypes.data_as(C.c_void_p)
    assert L.vfgs_b200_add_grain_frames_device(p, p, 1, 64, 64, 0, None) == 2   # width <= 128 (hw.c:168)
    hw_lib.vfgs_set_depth(8)
    assert L.vfgs_b200_add_grain_frames_device(p, p, 1, 256, 64, 10, None) == 1  # out depth > in depth
    assert b"out_depth" in L.vfgs_b200_last_error()
    assert L.vfgs_b200_add_grain_frames_host(None, p, 1, 256, 64, 0) == 1


def test_random_setter_sequences_match_the_reference(hw_lib):
    """Random interleavings of every vfgs_hw.h setter (the state machine is order-dependent: scale_shift follows the
    depth in force, chroma patterns are repacked with the subsampling in force) leave the shim's mirror, the oracle
    and, where it is mounted, the live reference in the same state."""
    from oracle import pyoracle
    from tests.util import states_equal
    ref = None
    if pyoracle.have_reference():
        ref = pyoracle.Reference()
    rng = np.random.default_rng(77)
    for trial in range(40):
        hw_lib.reset()
        o = Oracle()
        targets = [hw_lib, o]
        if ref is not None:
            ref.reset()
            targets.append(ref)
        for _ in range(int(rng.integers(5, 40))):
            op = int(rng.integers(0, 9))
            if op == 0:
                args = ("vfgs_set_depth", (int(rng.choice([8, 10])),))
            elif op == 1:
                sx, sy = [(2, 2), (2, 1), (1, 1), (1, 2)][int(rng.integers(0, 4))]
                args = ("vfgs_set_chroma_subsampling", (sx, sy))
            elif op == 2:
                args = ("vfgs_set_scale_shift", (int(rng.integers(2, 8)),))
            elif op == 3:
                args = ("vfgs_set_legal_range", (int(rng.integers(0, 2)),))
            elif op == 4:
                args = ("vfgs_set_seed", (int(rng.integers(0, 1 << 32)),))
            elif op == 5:
                args = ("vfgs_set_luma_pattern", (int(rng.integers(0, 8)), rng.integers(-128, 128, size=(64, 64), dtype=np.int8)))
            elif op == 6:
                args = ("vfgs_set_chroma_pattern", (int(rng.integers(0, 8)), rng.integers(-128, 128, size=(64, 64), dtype=np.int8)))
            elif op == 7:
                args = ("vfgs_set_scale_lut", (int(rng.integers(0, 3)), rng.integers(0, 256, size=256, dtype=np.uint8)))
            else:
                args = ("vfgs_set_pattern_lut", (int(rng.integers(0, 3)), (rng.integers(0, 8, size=256).astype(np.uint8) << 4)))
            for t in targets:
                getattr(t, args[0])(*args[1])
        want = o.state()
        assert states_equal(hw_lib.state(), want) == [], trial
        if ref is not None:
            assert states_equal(ref.state(), want) == [], trial


def test_pattern_lut_with_out_of_range_slots_is_accepted_then_refused_at_use(hw_lib):
    """The reference setter copies any table (vfgs_hw.c:333-337); an entry above slot 8 only matters when a sample
    hits it (out-of-bounds read of pattern[2][9], vfgs_hw.c:218). The shim mirrors the table like the reference
    (compared with the live reference where it is built) and refuses to synthesise grain with it
    (VFGS_B200_ERR_STATE, no GPU needed), instead of aborting in the setter."""
    from oracle import pyoracle
    from versatilefilmgrain_b200.api import VfgsError
    hw_lib.reset()
    lut = np.arange(256, dtype=np.uint8)  # slots 0..15
    hw_lib.vfgs_set_pattern_lut(1, lut)
    assert np.array_equal(hw_lib.state()["plut"][1], lut)
    if pyoracle.have_reference():
        reference = pyoracle.Reference()
        reference.reset()
        reference.vfgs_set_pattern_lut(1, lut)
        assert states_equal(hw_lib.state(), reference.state()) == []
    with pytest.raises(VfgsError, match="slot"):
        hw_lib.add_grain_frames_device_ptr(0x1000, 0x2000, 1, 256, 144)
    hw_lib.reset()


def test_overlapping_buffers_are_classified_before_any_device_work(hw_lib):
    """in == out (all planes identical) is in place; any other overlap of input and output planes -- output one frame
    behind the input, only the chroma planes aliased, Cb written over Cr -- is refused with VFGS_B200_ERR_ARG.
    The check needs no GPU: without one, legal calls get past it and fail with the CUDA error instead."""
    import torch
    from versatilefilmgrain_b200.api import Planes, VfgsError
    hw_lib.reset()
    w, h, n = 256, 144, 3
    ys, cs = w * h * 2, (w // 2) * (h // 2) * 2  # power-on state: 8-bit ... set 10-bit 4:2:0 explicitly
    hw_lib.vfgs_set_depth(10)
    fb = ys + 2 * cs
    base = 0x10000000

    def planes(b):
        return Planes(b, b + ys, b + ys + cs, 2 * w, w, fb)

    def rc_of(pin, pout):
        try:
            hw_lib.add_grain_planes_device(pin, pout, n, w, h)
        except VfgsError as e:
            return int(str(e).split("error ")[1].split(":")[0])
        return 0

    ok = (0,) if torch.cuda.is_available() else (3,)  # VFGS_B200_ERR_CUDA without a device
    if not torch.cuda.is_available():
        assert rc_of(planes(base), planes(base)) in ok                    # in place
        assert rc_of(planes(base), planes(base + n * fb)) in ok            # disjoint, back to back
    assert rc_of(planes(base), planes(base + fb)) == 1                     # output one frame behind the input
    assert rc_of(planes(base), planes(base + 64)) == 1                     # shifted by a few bytes
    mixed = planes(base + 2 * n * fb); mixed.u = base + ys                 # only Cb aliases (exactly): in place for that plane
    if not torch.cuda.is_available():
        assert rc_of(planes(base), mixed) in ok
    swapped = planes(base + 2 * n * fb); swapped.u = base + ys + cs        # Cb written over the input's Cr
    assert rc_of(planes(base), swapped) == 1
    hw_lib.reset()
