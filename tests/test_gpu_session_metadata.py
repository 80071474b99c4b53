"""Metadata calls on grain sessions (vfgs_b200_session_init_metadata, fw_sessions_kernel) on the GPU: every golden
configuration programmed into a session that was created from another state, against the golden state, the global
firmware route and the oracle's frames; 64- and 300-entry calls; updates queued between jobs on two CUDA streams; the
firmware's working memory per session; refusals; lifetime and seeding. Run with -m gpu on a B200."""
import ctypes as C

import numpy as np
import pytest

from tests.fixtures import SUBSAMPLING
from tests.util import Oracle, first_mismatch, load_golden, program_case, program_random_state, states_equal, synth_frames

pytestmark = pytest.mark.gpu

G = load_golden()
CASES = G.runnable()


@pytest.fixture(scope="module")
def hw():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from versatilefilmgrain_b200 import VfgsHw
    return VfgsHw(device=0)


def kind(case):
    return "afgs1" if G.cases[case]["afgs1"] else "sei"


def other_state(case, seed=11):
    """A random state of the case's depth and format (the session's state before its metadata arrives). Its clip range
    is the full one, as in the golden states: SEI metadata leaves the clip range alone."""
    m = G.cases[case]
    return (seed, m["depth"], m["fmt"], 3, 2, 0, 4, False)


def new_session(hw, state):
    hw.reset()
    program_random_state(hw, *state)
    return hw.create_session()


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a.view(np.int16) if a.dtype == np.uint16 else a)).cuda()


def from_dev(t):
    a = t.cpu().numpy()
    return a.view(np.uint16) if a.dtype == np.int16 else a


def out_buffer(n, depth, od):
    import torch
    return torch.zeros(n, dtype=torch.uint8 if (od == 8 or depth == 8) else torch.int16, device="cuda")


def golden_regs(case):
    return [int(v) for v in G.state(case)["lfsr"]]


def golden_diff(got, case, lfsr=True):
    """states_equal against the golden state, over the slots the case's LUTs select. The chroma bank only where the
    metadata writes chroma patterns: an SEI message without chroma models leaves the session's chroma slots as they
    were (the golden states start from power-on, the sessions here from another state)."""
    want = dict(G.state(case))
    if not lfsr:
        want["lfsr"] = got["lfsr"]
    raw = G.struct(case)
    nslot = list(G.cases[case]["nslot"])
    if not G.cases[case]["afgs1"] and not (raw[3] or raw[4]):  # comp_model_present_flag[1], [2]
        nslot[1] = 0
    return states_equal(got, want, nslot)


def oracle_update(o, case):
    """The oracle's side of a metadata update: the golden state of the case, except what SEI metadata leaves alone
    (the registers and the clip range)."""
    regs, legal = o.get_lfsr(), int(o.state()["scalars"][2]) == 16
    program_case(o, G, case)
    if not G.cases[case]["afgs1"]:
        o.set_lfsr(regs)
        o.vfgs_set_legal_range(1 if legal else 0)


def finish_seed(session, case):
    """What test_gpu_firmware.py does after the firmware: the CLI seeds SEI streams (vfgs_main.c:759-760)."""
    if not G.cases[case]["afgs1"]:
        session.set_seed(G.seed)


# ---- every golden case ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", CASES)
def test_session_programmed_from_metadata(hw, case):
    """A session created from another state of the same depth and format takes the case's metadata: its state equals the
    golden state and the state the global firmware route leaves from the same start, and frames through a jobs call
    (10-bit input also to 8-bit output) equal the oracle's."""
    from versatilefilmgrain_b200 import Job
    import torch
    meta = G.cases[case]
    state = other_state(case)
    s = new_session(hw, state)
    before = hw.launch_count()
    hw.init_sessions([(s, kind(case), G.struct(case))])
    assert hw.launch_count() == before + 1
    if not meta["afgs1"]:  # SEI leaves the registers alone
        o = Oracle(); program_random_state(o, *state)
        assert s.get_lfsr() == o.get_lfsr()
    finish_seed(s, case)
    got = s.get_state()
    assert golden_diff(got, case) == [], case
    # the global route from the same start (same state, same firmware working memory)
    hw.reset(); program_random_state(hw, *state)
    (hw.init_afgs1 if meta["afgs1"] else hw.init_sei)(G.struct(case))
    if not meta["afgs1"]:
        hw.vfgs_set_seed(G.seed)
    assert states_equal(got, hw.state()) == [], case
    w, h, n = 512, 152, 2
    frames = synth_frames(n, w, h, meta["fmt"], meta["depth"], seed=41)
    src = to_dev(frames.reshape(-1))
    for od in ((0, 8) if meta["depth"] == 10 else (0,)):
        s.set_lfsr(golden_regs(case))
        o = Oracle(); program_case(o, G, case)
        want = o.add_grain_frames(frames, n, w, h, od)
        dst = out_buffer(want.size, meta["depth"], od)
        hw.add_grain_jobs_device([Job.packed(s, src, dst, n, w, h, od)])
        torch.cuda.synchronize()
        res = from_dev(dst)
        assert np.array_equal(res, want), (case, od, first_mismatch(res, want, w, h, meta["fmt"], n))
        assert s.get_lfsr() == o.get_lfsr(), (case, od)
    s.close()


# ---- batch sizes --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nsess", [64, 300])
def test_batched_update_then_jobs(hw, nsess):
    """nsess sessions of every depth and format take mixed SEI / AFGS1 metadata in ONE call (one launch), then one jobs
    call serves one frame of each; every output and register set equals the oracle's."""
    from versatilefilmgrain_b200 import Job
    import torch
    rng = np.random.default_rng(nsess)
    cases = [CASES[int(i)] for i in rng.integers(0, len(CASES), size=nsess)]
    sessions = [new_session(hw, other_state(c, seed=100 + k)) for k, c in enumerate(cases)]
    before = hw.launch_count()
    hw.init_sessions([(s, kind(c), G.struct(c)) for s, c in zip(sessions, cases)])
    assert hw.launch_count() == before + 1
    w, h = 256, 48
    jobs, wants, oracles = [], [], []
    for k, (s, c) in enumerate(zip(sessions, cases)):
        m = G.cases[c]
        finish_seed(s, c)
        frames = synth_frames(1, w, h, m["fmt"], m["depth"], seed=k)
        o = Oracle(); program_case(o, G, c)
        o.set_lfsr(s.get_lfsr())
        wants.append(o.add_grain_frames(frames, 1, w, h, 0)); oracles.append(o)
        dst = out_buffer(wants[-1].size, m["depth"], 0)
        jobs.append(Job.packed(s, to_dev(frames.reshape(-1)), dst, 1, w, h))
    hw.add_grain_jobs_device(jobs)
    torch.cuda.synchronize()
    for k, (j, want, o, s) in enumerate(zip(jobs, wants, oracles, sessions)):
        res = from_dev(j.tensors[1])
        assert np.array_equal(res, want), (k, cases[k], first_mismatch(res, want, w, h, G.cases[cases[k]]["fmt"], 1))
        assert s.get_lfsr() == o.get_lfsr(), k
    for k, (s, c) in enumerate(zip(sessions, cases)):
        assert golden_diff(s.get_state(), c, lfsr=False) == [], (k, c)
        s.close()


# ---- in flight ------------------------------------------------------------------------------------------------------------
def test_updates_between_jobs_in_flight(hw):
    """Six rounds of (jobs, update) on two CUDA streams with no synchronisation in between: each round's frames come
    out under the metadata that was current when they were queued, although the next update is already queued behind
    them (the update's kernel waits on the device for the jobs that read the old images)."""
    from versatilefilmgrain_b200 import Job
    import torch
    order = ["fgs_sei.cfg|d10|420|g100", "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei_ff_test5.cfg|d10|420|g100",
             "fgs_afgs1_test3.cfg|d10|420|g100", "fgs_sei_ar_test1.cfg|d10|420|g100", "fgs_afgs1_test7.cfg|d10|420|g100"]
    order = [c for c in order if c in G.cases]
    assert len(order) >= 4
    w, h, n = 1920, 1080, 3
    frames = [synth_frames(n, w, h, "420", 10, seed=70 + k) for k in range(2)]
    srcs = [to_dev(f.reshape(-1)) for f in frames]
    start = (5, 10, "420", 2, 2, 0, 5, False)
    sessions = [new_session(hw, start) for _ in range(2)]
    oracles = []
    for _ in range(2):
        o = Oracle(); program_random_state(o, *start); oracles.append(o)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = [[out_buffer(frames[0].size, 10, 0) for _ in range(2)] for _ in range(6)]
    torch.cuda.synchronize()  # inputs and outputs exist before the side streams touch them
    updates = []
    for r in range(6):  # enqueue only: nothing waits for the device in this loop
        hw.add_grain_jobs_device([Job.packed(sessions[k], srcs[k], outs[r][k], n, w, h) for k in range(2)], stream=streams[r % 2])
        cases = [order[(r + k) % len(order)] for k in range(2)]
        hw.init_sessions([(sessions[k], kind(cases[k]), G.struct(cases[k])) for k in range(2)], stream=streams[(r + 1) % 2])
        updates.append(cases)
    torch.cuda.synchronize()
    for r in range(6):
        for k in range(2):
            want = oracles[k].add_grain_frames(frames[k], n, w, h, 0)
            res = from_dev(outs[r][k])
            assert np.array_equal(res, want), (r, k, first_mismatch(res, want, w, h, "420", n))
            oracle_update(oracles[k], updates[r][k])
    for k in range(2):
        assert sessions[k].get_lfsr() == oracles[k].get_lfsr()
        sessions[k].close()


# ---- the firmware's working memory -------------------------------------------------------------------------------------
@pytest.mark.parametrize("fmt", ["422", "444"])
def test_working_memory_is_per_session(hw, fmt):
    """An SEI message without a luma model after one with a luma model: in 4:2:2 / 4:4:4 its chroma patterns read what
    the luma pattern left in the firmware's pattern buffer. A global init_sei in between must not change that."""
    a = "builtin_default|d10|420|g100"  # luma and chroma models; its metadata is applied here in 4:2:2 / 4:4:4
    b_raw = bytearray(G.struct(a))
    b_raw[2] = 0  # comp_model_present_flag[0]: no luma model
    assert b_raw[3] and b_raw[4]
    unrelated = G.struct(next(c for c in CASES if G.cases[c]["fmt"] == fmt and not G.cases[c]["afgs1"]))
    hw.reset(); hw.vfgs_set_depth(10); hw.vfgs_set_chroma_subsampling(*SUBSAMPLING[fmt])
    s = hw.create_session()
    hw.init_sei(G.struct(a)); hw.init_sei(bytes(b_raw))
    want = hw.state()
    s.init_sei(G.struct(a))
    hw.init_sei(unrelated)
    s.init_sei(bytes(b_raw))
    assert states_equal(s.get_state(), want) == []
    s.close()


# ---- refusals -------------------------------------------------------------------------------------------------------------
class Afgs1(C.Structure):
    """fgs_afgs1 (include/vfgs_fw.h)."""
    _fields_ = [("grain_seed", C.c_uint16), ("num_y_points", C.c_uint8), ("point_y_values", C.c_uint8 * 14),
                ("point_y_scaling", C.c_uint8 * 14), ("chroma_scaling_from_luma", C.c_uint8), ("num_cb_points", C.c_uint8),
                ("point_cb_values", C.c_uint8 * 10), ("point_cb_scaling", C.c_uint8 * 10), ("num_cr_points", C.c_uint8),
                ("point_cr_values", C.c_uint8 * 10), ("point_cr_scaling", C.c_uint8 * 10), ("grain_scaling", C.c_uint8),
                ("ar_coeff_lag", C.c_uint8), ("ar_coeffs_y", C.c_int16 * 24), ("ar_coeffs_cb", C.c_int16 * 25),
                ("ar_coeffs_cr", C.c_int16 * 25), ("ar_coeff_shift", C.c_uint8), ("grain_scale_shift", C.c_uint8),
                ("cb_mult", C.c_uint8), ("cb_luma_mult", C.c_uint8), ("cb_offset", C.c_uint16), ("cr_mult", C.c_uint8),
                ("cr_luma_mult", C.c_uint8), ("cr_offset", C.c_uint16), ("overlap_flag", C.c_uint8),
                ("clip_to_restricted_range", C.c_uint8)]


def afgs1_variant(case, **fields):
    raw = G.struct(case)
    assert C.sizeof(Afgs1) == len(raw)
    a = Afgs1.from_buffer_copy(raw)
    for k, v in fields.items():
        if k == "y_points_equal":
            a.point_y_values[1] = a.point_y_values[0]
        else:
            setattr(a, k, v)
    return bytes(a)


def test_refusals_change_nothing(hw):
    """Every refusal is decided on the host before any device work: all sessions' states and registers, the global
    state and the launch count stay as they were, even where valid entries come first. (Too many patterns and images
    larger than shared memory cannot come out of the firmware's planner, which makes at most 8 + 8 patterns.)"""
    from versatilefilmgrain_b200 import VfgsError
    from versatilefilmgrain_b200.api import _CMetadata
    af = next(c for c in CASES if G.cases[c]["afgs1"] and G.cases[c]["depth"] == 10)
    se = next(c for c in CASES if not G.cases[c]["afgs1"] and G.cases[c]["depth"] == 10 and G.cases[c]["fmt"] == "420")
    a = new_session(hw, other_state(af, 3))
    b = new_session(hw, other_state(af, 4))
    hw.init_sessions([(a, "afgs1", G.struct(af))])  # one session that has had metadata already
    hw.reset(); program_random_state(hw, 9, 10, "420")
    sei_raw = bytearray(G.struct(se))
    sei_raw[1] = 1  # log2_scale_factor 1 in frequency-filtering mode: scale shift 1
    bad = [
        [(a, "afgs1", afgs1_variant(af, y_points_equal=True, num_y_points=max(2, Afgs1.from_buffer_copy(G.struct(af)).num_y_points)))],
        [(b, "afgs1", G.struct(af)), (a, "afgs1", afgs1_variant(af, ar_coeff_lag=0))],
        [(b, "afgs1", G.struct(af)), (a, "afgs1", afgs1_variant(af, ar_coeff_lag=4))],
        [(a, "afgs1", afgs1_variant(af, grain_scaling=7))],
        [(b, "sei", G.struct(se)), (a, "sei", bytes(sei_raw))],
        [(a, "afgs1", G.struct(af)), (a, "sei", G.struct(se))],
        [(b, "afgs1", G.struct(af)), (None, "afgs1", G.struct(af))],
    ]

    def snapshot():
        return [a.get_state(), b.get_state(), hw.state(), hw.launch_count()]

    def same(x, y):
        assert states_equal(x[0], y[0]) == [] and states_equal(x[1], y[1]) == [] and states_equal(x[2], y[2]) == []
        assert x[3] == y[3]

    ref = snapshot()
    for entries in bad:
        with pytest.raises(VfgsError):
            hw.init_sessions(entries)
        same(snapshot(), ref)
    # malformed lists through the C entry point
    L = hw.L
    arr = (_CMetadata * 2)()
    raw = (C.c_uint8 * len(G.struct(af))).from_buffer_copy(G.struct(af))
    arr[0].session = a.handle; arr[0].afgs1 = C.cast(raw, C.c_void_p); arr[0].sei = C.cast(raw, C.c_void_p)  # both set
    arr[1].session = b.handle  # neither set
    assert L.vfgs_b200_session_init_metadata(arr, 1, None) == 1
    arr[0].sei = None
    assert L.vfgs_b200_session_init_metadata(arr, 2, None) == 1
    assert L.vfgs_b200_session_init_metadata(arr, -1, None) == 1
    assert L.vfgs_b200_session_init_metadata(None, 1, None) == 1
    assert L.vfgs_b200_session_init_metadata(None, 0, None) == 0
    same(snapshot(), ref)
    a.close(); b.close()


# ---- lifetime and seeding -------------------------------------------------------------------------------------------------
def test_destroy_right_after_update_and_set_seed(hw):
    """A session destroyed right after its update (nothing synchronised) takes its kernel with it cleanly; the other
    session of the same call is programmed correctly. session_set_seed is vfgs_set_seed on the session's registers."""
    import torch
    af = next(c for c in CASES if G.cases[c]["afgs1"] and G.cases[c]["fmt"] == "420")
    a = new_session(hw, other_state(af, 5))
    b = new_session(hw, other_state(af, 6))
    hw.init_sessions([(a, "afgs1", G.struct(af)), (b, "afgs1", G.struct(af))])
    a.close()
    torch.cuda.synchronize()
    assert golden_diff(b.get_state(), af) == []
    for seed in (0, 1, 0x12345678, 0xFFFFFFFF):
        b.set_seed(seed)
        hw.vfgs_set_seed(seed)
        assert b.get_lfsr() == hw.get_lfsr()
    b.close()
