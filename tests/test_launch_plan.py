"""Host-side launch planning (versatilefilmgrain_b200/csrc/vfgs_tables.h: plan_launches, place_fast_images), through
the host build of the shared headers (tests/emu): which kernel serves which component, the fast kernel's
shared-memory layout, the 16-samples-per-lane path of 8-bit input. No GPU, nothing is executed."""
import ctypes as C

import numpy as np
import pytest

from oracle.pyoracle import RefState
from tests.util import Oracle, build_emu, load_golden, program_case, program_random_state

G = load_golden()
FAST, GATHER, GENERAL = 0, 1, 2


@pytest.fixture(scope="module")
def emu():
    L = C.CDLL(build_emu())
    L.emu_plan.argtypes = [C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    return L


def plan(emu, o, w, h, od=0, in_place=0, mode=0):
    st = RefState(); o.L.oracle_get_state(o.h, C.byref(st))
    out = np.zeros(32, dtype=np.int32)
    emu.emu_plan(C.byref(st), w, h, od, in_place, mode, out.ctypes.data_as(C.c_void_p))
    return {"kind": list(out[0:3]), "fsmem": int(out[3]), "fpad": int(out[4]), "fimg_off": list(out[5:8]),
            "fimg_bytes": list(out[8:11]), "fwide": list(out[11:14]), "units": list(out[14:17]), "gather_smem": int(out[17]),
            "allwide": int(out[18])}


def test_headline_config_layout(emu):
    """AFGS1 4:2:0 10-bit: everything on the fast kernel; luma image and the shared Cb/Cr image sit in the gap in front
    of the LUTs, so the launch needs gap + 96 KB (<= 132 KB carve-out with the driver's reserved KB)."""
    o = Oracle(); program_case(o, G, "fgs_afgs1_test1.cfg|d10|420|g100")
    p = plan(emu, o, 3840, 2160)
    assert p["kind"] == [FAST, FAST, FAST]
    assert p["fpad"] == 32768 - 1152 and p["fsmem"] == p["fpad"] + 3 * 32768
    assert p["fimg_bytes"][0] == 2 * 2 * 64 * 72 and p["fimg_bytes"][1] == 2 * 4 * 32 * 40
    assert p["fimg_bytes"][2] == 0 and p["fimg_off"][2] == p["fimg_off"][1]  # Cr shares Cb's image
    assert all(off < 0 for off in p["fimg_off"])                           # in front of the first LUT
    assert p["units"] == [240, 120, 120] and p["fwide"] == [1, 1, 1]         # 16 samples per lane, one 256-bit access per line


def test_kernel_choice(emu):
    o = Oracle(); program_case(o, G, "fgs_sei.cfg|d10|420|g100")           # 8 luma patterns
    assert plan(emu, o, 512, 64)["kind"] == [GATHER, FAST, FAST]
    assert plan(emu, o, 512, 64, in_place=1)["kind"] == [GATHER, FAST, FAST]   # 16-sample-block gather lanes read only their own samples
    o5 = Oracle(); program_case(o5, G, "fgs_sei_ff_test5.cfg|d10|420|g100")  # sample-adaptive 4:2:0 chroma: 8-sample blocks
    assert plan(emu, o5, 512, 64)["kind"] == [FAST, GATHER, GATHER]
    assert plan(emu, o5, 512, 64, in_place=1)["kind"] == [FAST, GENERAL, GENERAL]  # halo lanes would read overwritten input: the shim takes the scratch route
    assert plan(emu, o, 512, 64, mode=1)["kind"] == [GENERAL] * 3
    assert plan(emu, o, 204, 64)["kind"] == [GENERAL, 3, 3]                # 204 % 8 != 0: sample-adaptive luma on the general kernel, chroma on the fast kernel's EDGE variant
    o = Oracle(); program_case(o, G, "fgs_afgs1_test1.cfg|d10|420|g100")
    assert plan(emu, o, 200, 64)["kind"] == [FAST, 3, 3]                   # chroma width 100: EDGE variant
    assert plan(emu, o, 512, 64, mode=2)["kind"] == [GATHER] * 3


def test_444_images_spill_behind_the_luts(emu):
    o = Oracle(); program_case(o, G, "fgs_sei_ff_test4.cfg|d10|444|g150")
    p = plan(emu, o, 512, 64)
    assert p["kind"] == [FAST] * 3
    assert p["fimg_off"][0] < 0 and p["fimg_off"][1] >= 3 * 32768           # 2 x 18 KB do not fit in the 31 KB gap
    assert p["fsmem"] <= 227 * 1024


def test_wide_path_of_8bit_input(emu):
    o = Oracle(); program_random_state(o, 2, 8, "444", 1, 1, 1, 7, False)
    assert plan(emu, o, 512, 64)["fwide"] == [1, 1, 1] and plan(emu, o, 512, 64)["units"] == [32, 32, 32]
    assert plan(emu, o, 520, 64)["fwide"] == [0, 0, 0]                      # 520 % 16 == 8: 8 samples per lane
    o = Oracle(); program_case(o, G, "fgs_sei_ff_test1.cfg|d8|420|g100")
    p = plan(emu, o, 1920, 1080)
    assert p["fwide"] == [1, 1, 1] and p["units"] == [120, 60, 60]
    p = plan(emu, o, 1936, 1080)                                            # chroma width 968 = 16 * 60.5
    assert p["fwide"] == [1, 0, 0] and p["units"] == [121, 121, 121]


def test_wide_path_of_16bit_input(emu):
    """10-bit samples: 16 per lane where width % 16 == 0 and rows, planes and frames are 32-byte aligned (256-bit loads;
    the output of the fused 10 -> 8 conversion needs 16)."""
    o = Oracle(); program_case(o, G, "fgs_afgs1_test1.cfg|d10|420|g100")
    p = plan(emu, o, 1920, 1080)
    assert p["fwide"] == [1, 1, 1] and p["units"] == [120, 60, 60] and p["allwide"] == 1   # the 512-thread ALLWIDE kernel variant
    p = plan(emu, o, 1936, 1080)                                            # chroma width 968 = 16 * 60.5: 8 samples per lane
    assert p["fwide"] == [1, 0, 0] and p["units"] == [121, 121, 121] and p["allwide"] == 0  # mixed launch: the 768-thread kernel
    p = plan(emu, o, 1928, 1080)                                            # luma 1928 = 16 * 120.5; chroma 964 is ragged (EDGE)
    assert p["fwide"] == [0, 0, 0] and p["kind"] == [FAST, 3, 3] and p["allwide"] == 0
    o = Oracle(); program_case(o, G, "fgs_sei.cfg|d10|420|g100")            # luma on the gather kernel: the fast launch serves chroma only
    p = plan(emu, o, 1920, 1080)
    assert p["kind"] == [GATHER, FAST, FAST] and p["fwide"] == [0, 1, 1] and p["allwide"] == 1
