"""Metadata calls on sessions (vfgs_b200_session_init_metadata) through the host build of their device code
(tests/emu/emu_meta.cpp): the auto-regressive filter's wavefront form against the serial filter, the shared table-image
fill against the serial image builder, the layout from a session's -128 flags against the scanned one, and the host
half of an update against the restated firmware (tests/emu/emu.cpp, emu_fw_init). Needs no GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import RefState
from tests.fixtures import SUBSAMPLING
from tests.util import RANDOM_STATES, Oracle, build_emu, load_golden, program_case, program_random_state

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
G = load_golden()
CASES = G.runnable()
AR_CASES = [c for c in CASES if G.cases[c]["afgs1"] or np.frombuffer(G.struct(c), dtype=np.uint8)[0] == 1]  # model_id 1: SEI AR


def build_emu_meta() -> str:
    """Host build of emu_meta.cpp (test tool only), rebuilt when it or a shared header is newer."""
    so, src = os.path.join(HERE, "libemu_meta.so"), os.path.join(HERE, "emu_meta.cpp")
    csrc = os.path.join(HERE, "..", "..", "versatilefilmgrain_b200", "csrc")
    deps = [src] + [os.path.join(csrc, n) for n in os.listdir(csrc) if n.endswith(".h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-Wno-unknown-pragmas", "-o", so, src],
                       check=True)
    return so


@pytest.fixture(scope="module")
def emu():
    L = C.CDLL(build_emu_meta())
    assert L.emum_state_size() == C.sizeof(RefState)
    L.emum_ar_plan.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
    L.emum_ar_random.argtypes = [C.c_ulonglong, C.c_int]
    L.emum_ar_luma_injection.argtypes = [C.c_ulonglong, C.c_int]
    L.emum_fill.argtypes = [C.c_void_p, C.c_int]
    L.emum_flag_layout.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    L.emum_host_half.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    L.emum_run_plan.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return L


def raw(case):
    return np.frombuffer(G.struct(case), dtype=np.uint8).copy()


def ref_state(st: dict) -> RefState:
    r = RefState()
    C.memmove(r.pattern, np.ascontiguousarray(st["pattern"], dtype=np.int8).ctypes.data, 2 * 9 * 64 * 64)
    C.memmove(r.slut, np.ascontiguousarray(st["slut"], dtype=np.uint8).ctypes.data, 768)
    C.memmove(r.plut, np.ascontiguousarray(st["plut"], dtype=np.uint8).ctypes.data, 768)
    r.rnd, r.rnd_up, r.line_rnd, r.line_rnd_up = [int(v) for v in st["lfsr"]]
    (r.scale_shift, r.bs, r.y_min, r.y_max, r.c_min, r.c_max, r.csubx, r.csuby) = [int(v) for v in st["scalars"]]
    return r


def power_on(depth, fmt) -> RefState:
    o = Oracle()
    o.vfgs_set_depth(depth)
    o.vfgs_set_chroma_subsampling(*SUBSAMPLING[fmt])
    return ref_state(o.state())


# ---- the wavefront ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["420", "422", "444"])
def test_wavefront_equals_serial_filter_on_golden_jobs(emu, fmt):
    """Every AR job of the golden AFGS1 and SEI auto-regressive cases, in 4:2:0, 4:2:2 and 4:4:4, run in firmware order
    on one working memory (the chroma jobs read the luma field the luma job left)."""
    sx, sy = SUBSAMPLING[fmt]
    seen, total = set(), 0
    for case in AR_CASES:
        key = G.struct(case)
        if key in seen:
            continue
        seen.add(key)
        n = C.c_int(0)
        bad = emu.emum_ar_plan(raw(case).ctypes.data, 1 if G.cases[case]["afgs1"] else 0, sx, sy, C.byref(n))
        assert bad == 0, case
        total += n.value
    assert total >= 3 and len(seen) >= 2


@pytest.mark.parametrize("seed", range(8))
def test_wavefront_equals_serial_filter_on_random_taps(emu, seed):
    """Random taps for lags 1-3 (with and without a luma coefficient) and the SEI 6-tap layout, random shifts, scales
    and seeds, luma and chroma field sizes, with and without the luma field."""
    assert emu.emum_ar_random(seed, 60) == 0


@pytest.mark.parametrize("seed", range(4))
def test_wavefront_equals_serial_filter_with_luma_injection(emu, seed):
    """Synthetic jobs with cx != 0 and the luma field present (the firmware never enables the injection)."""
    assert emu.emum_ar_luma_injection(seed, 40) == 0


# ---- the image fill --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nthreads", [1, 32, 256])
def test_fill_reproduces_builder_on_golden_states(emu, nthreads):
    assert len(CASES) >= 70
    for case in CASES:
        st = ref_state(G.state(case))
        assert emu.emum_fill(C.byref(st), nthreads) == 0, case


@pytest.mark.parametrize("nthreads", [1, 32, 256])
@pytest.mark.parametrize("args", RANDOM_STATES)
def test_fill_reproduces_builder_on_random_states(emu, nthreads, args):
    """Random states, several slots per bank, some with -128 bytes (no sign folding, no fast image for those slots)."""
    o = Oracle()
    program_random_state(o, *args)
    st = ref_state(o.state())
    assert emu.emum_fill(C.byref(st), nthreads) == 0


def test_fill_on_minus128_in_unread_chroma_bytes(emu):
    """A -128 byte in the part of a chroma slot the images never read (4:2:0): sign folding is off for the bank, as the
    scan of the whole slot has it."""
    o = Oracle()
    program_random_state(o, 3, 8, "420", 1, 2)
    st = o.state()
    st["pattern"][1, 1, 40, 50] = -128
    r = ref_state(st)
    for n in (1, 32, 256):
        assert emu.emum_fill(C.byref(r), n) == 0


# ---- the -128 flags of a session ----------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_flag_layout_equals_scanned_layout(emu, case):
    """A session on the power-on state given a case's metadata: the layout planned from the flags equals the layout of
    the state the firmware leaves (scanned), and that state is the golden one."""
    meta = G.cases[case]
    before = power_on(meta["depth"], meta["fmt"])
    after = power_on(meta["depth"], meta["fmt"])
    scratch = (C.c_uint8 * emu.emum_scratch_size())()
    af = 1 if meta["afgs1"] else 0
    assert emu.emum_run_plan(raw(case).ctypes.data, af, C.byref(after), scratch) == 0
    assert emu.emum_flag_layout(C.byref(before), raw(case).ctypes.data, af, C.byref(after)) == 0
    want = G.state(case)
    got = after.as_dict()
    for bank in range(2):
        n = meta["nslot"][bank]
        assert np.array_equal(got["pattern"][bank, :n], want["pattern"][bank, :n]), (case, bank)


@pytest.mark.parametrize("args", RANDOM_STATES[:6])
def test_flag_layout_after_a_random_snapshot(emu, args):
    """A session created from a random state (-128 bytes in some of them) and given golden metadata of its depth and
    format: the slots the firmware writes lose their -128 flags, the others keep them."""
    depth, fmt = args[1], args[2]
    cases = [c for c in CASES if G.cases[c]["depth"] == depth and G.cases[c]["fmt"] == fmt]
    o = Oracle()
    program_random_state(o, *args)
    for case in cases[:4]:
        before = ref_state(o.state())
        after = ref_state(o.state())
        scratch = (C.c_uint8 * emu.emum_scratch_size())()
        af = 1 if G.cases[case]["afgs1"] else 0
        assert emu.emum_run_plan(raw(case).ctypes.data, af, C.byref(after), scratch) == 0
        assert emu.emum_flag_layout(C.byref(before), raw(case).ctypes.data, af, C.byref(after)) == 0, case


# ---- the host half ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_host_half_equals_restated_firmware(emu, case):
    """LUTs, scalars and registers of an update, applied on the host at enqueue, equal the whole restated firmware's."""
    meta = G.cases[case]
    sx, sy = SUBSAMPLING[meta["fmt"]]
    af = 1 if meta["afgs1"] else 0
    got, want = RefState(), RefState()
    assert emu.emum_host_half(raw(case).ctypes.data, af, meta["depth"], sx, sy, C.byref(got)) == 0
    full = C.CDLL(build_emu())
    full.emu_fw_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    assert full.emu_fw_init(raw(case).ctypes.data, af, meta["depth"], sx, sy, C.byref(want)) == 0
    g, w = got.as_dict(), want.as_dict()
    for k in ("slut", "plut", "lfsr", "scalars"):
        assert np.array_equal(g[k], w[k]), (case, k)
