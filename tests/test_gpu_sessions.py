"""Grain sessions and vfgs_b200_add_grain_jobs_device on the GPU: random job lists over the golden cases against one
oracle per session and against the same jobs run one by one through the global entry points, repeated sessions,
interleaving with global calls, launch accounting, in place, refusals, lifetime, two CUDA streams and one bench-sized
call. Run with -m gpu on a B200."""
import numpy as np
import pytest

from tests.semiplanar import planar_to_semi, semi_to_planar
from tests.util import Oracle, load_golden, program_case, program_random_state, synth_frames

pytestmark = pytest.mark.gpu

G = load_golden()
CASES = G.runnable()
GEOMS = [(512, 56, 2), (264, 40, 1), (1366, 768, 1), (1928, 1080, 1), (640, 34, 2), (200, 24, 3)]


@pytest.fixture(scope="module")
def hw():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from versatilefilmgrain_b200 import VfgsHw
    h = VfgsHw(device=0)
    yield h
    h.force_general_kernel(0)


def program(target, state):
    """state: a golden case name or the argument tuple of program_random_state."""
    if isinstance(state, str):
        program_case(target, G, state)
    else:
        program_random_state(target, *state)


def meta(state):
    if isinstance(state, str):
        m = G.cases[state]
        return m["depth"], m["fmt"]
    return state[1], state[2]


def new_session(hw, state, regs=None):
    hw.reset(); program(hw, state)
    if regs is not None:
        hw.set_lfsr(regs)
    return hw.create_session()


def oracle(state, regs):
    o = Oracle(); program(o, state)
    o.set_lfsr(regs)
    return o


def to_dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a.view(np.int16) if a.dtype == np.uint16 else a)).cuda()


def from_dev(t):
    a = t.cpu().numpy()
    return a.view(np.uint16) if a.dtype == np.int16 else a


def surface(Y, UV):
    n, h, w = Y.shape
    s = np.zeros((n, h + UV.shape[1], w), dtype=Y.dtype)
    s[:, :h, :], s[:, h:, :UV.shape[2]] = Y, UV
    return to_dev(s)


class Spec:
    """One job: session index, frames, geometry, planar / semi-planar, output depth, in place."""

    def __init__(self, sess, state, w, h, n, semi, out8, in_place, seed):
        depth, fmt = meta(state)
        self.sess, self.state, self.w, self.h, self.n, self.semi = sess, state, w, h, n, semi
        self.out8 = out8 and depth == 10 and not in_place
        self.in_place, self.fmt, self.depth = in_place, fmt, depth
        self.frames = synth_frames(n, w, h, fmt, depth, seed=seed)

    def buffers(self):
        import torch
        dt = torch.uint8 if self.out8 or self.depth == 8 else torch.int16
        if self.semi:
            Y, UV = planar_to_semi(self.frames, self.n, self.w, self.h, self.fmt, self.depth == 10)
            self.src = surface(Y, UV)
            self.dst = self.src if self.in_place else torch.zeros(self.src.shape, dtype=dt, device="cuda")
        else:
            self.src = to_dev(self.frames.reshape(-1))
            self.dst = self.src if self.in_place else torch.zeros(self.src.numel(), dtype=dt, device="cuda")

    def out_format(self):
        from versatilefilmgrain_b200.api import NV12, P010
        return NV12 if self.out8 or self.depth == 8 else P010

    def job(self, session):
        from versatilefilmgrain_b200 import Job
        self.buffers()
        if self.semi:
            return Job.surfaces(session, self.src, self.dst, self.n, self.w, self.h, out_format=self.out_format())
        return Job.packed(session, self.src, self.dst, self.n, self.w, self.h, out_depth=8 if self.out8 else 0)

    def result(self):
        a = from_dev(self.dst)
        if not self.semi:
            return a
        return semi_to_planar(a[:, :self.h, :self.w], a[:, self.h:, :], not (self.out8 or self.depth == 8))

    def want(self, o):
        return o.add_grain_frames(self.frames, self.n, self.w, self.h, 8 if self.out8 else 0)

    def run_global(self, hw):
        """The same job through the global single-job entry points (state programmed and registers set by the caller)."""
        import torch
        self.buffers()
        if self.semi:
            hw.add_grain_surfaces(self.src, self.dst, self.n, self.w, self.h, out_format=self.out_format())
        else:
            hw.add_grain_frames_device(self.src, self.dst, self.n, self.w, self.h, 8 if self.out8 else 0)
        torch.cuda.synchronize()
        return self.result()


def random_specs(rng, nsess, njobs, cases, geoms=GEOMS):
    states = [cases[int(rng.integers(len(cases)))] for _ in range(nsess)]
    specs = []
    for k in range(njobs):
        s = int(rng.integers(nsess))
        depth, fmt = meta(states[s])
        w, h, n = geoms[int(rng.integers(len(geoms)))]
        semi = fmt != "444" and bool(rng.integers(2))
        specs.append(Spec(s, states[s], w, h, n, semi, bool(rng.integers(2)), bool(rng.integers(4) == 0), seed=1000 + k))
    return states, specs


def run_and_check(hw, states, specs, stream=None):
    """One batched call of specs over fresh sessions; every output and every session's registers equal one oracle per
    session fed the jobs in list order."""
    import torch
    sessions = [new_session(hw, s) for s in states]
    epochs = [x.get_lfsr() for x in sessions]
    jobs = [sp.job(sessions[sp.sess]) for sp in specs]
    hw.add_grain_jobs_device(jobs, stream=stream)
    torch.cuda.synchronize()
    oracles = [oracle(s, e) for s, e in zip(states, epochs)]
    for k, sp in enumerate(specs):
        want = sp.want(oracles[sp.sess])
        got = sp.result()
        assert np.array_equal(got, want), (k, sp.state, sp.w, sp.h, sp.n, sp.semi, sp.out8, sp.in_place, int(np.count_nonzero(got != want)))
    for x, o in zip(sessions, oracles):
        assert x.get_lfsr() == o.get_lfsr()
    return sessions, epochs


@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("seed", [1, 2, 3])
def test_case_matrix(hw, mode, seed):
    """Seeded random job lists over the golden cases x geometries (1366 x 768 and 1928 x 1080 among them) x planar /
    semi-planar x 10 -> 8: output and registers equal the oracle's, and equal the same jobs run one by one through the
    global entry points with the state programmed and the registers set."""
    rng = np.random.default_rng(seed * 10 + mode)
    states, specs = random_specs(rng, 6, 14, CASES)
    hw.force_general_kernel(mode)
    try:
        sessions, epochs = run_and_check(hw, states, specs)
        batched = [sp.result() for sp in specs]
        regs = [list(e) for e in epochs]
        for k, sp in enumerate(specs):
            hw.reset(); program(hw, sp.state); hw.set_lfsr(regs[sp.sess])
            got = sp.run_global(hw)
            regs[sp.sess] = hw.get_lfsr()
            assert np.array_equal(got, batched[k]), k
        for x, r in zip(sessions, regs):
            assert x.get_lfsr() == r
            x.close()
    finally:
        hw.force_general_kernel(0)


def test_random_states(hw):
    """Random states of the fuzzed list (several pattern slots, 4:2:2 / 4:4:4, legal range, -128 bytes), mixed in one call."""
    from tests.util import RANDOM_STATES
    rng = np.random.default_rng(11)
    states, specs = random_specs(rng, len(RANDOM_STATES), 20, RANDOM_STATES, geoms=[(512, 56, 2), (264, 40, 1), (640, 34, 2)])
    for x in run_and_check(hw, states, specs)[0]:
        x.close()


def test_every_golden_case(hw):
    """Every golden case gets one session in a single call: one job each, semi-planar for every second 4:2:0 / 4:2:2
    case, 10 -> 8 for every third 10-bit one; outputs and registers equal the oracle's."""
    specs = []
    for k, case in enumerate(CASES):
        depth, fmt = meta(case)
        specs.append(Spec(k, case, (264, 512, 200)[k % 3], 40, 1, fmt != "444" and k % 2 == 1, depth == 10 and k % 3 == 0,
                          False, seed=k))
    for x in run_and_check(hw, CASES, specs)[0]:
        x.close()


def test_session_repeated_and_interleaved(hw):
    """One session in several jobs of one call, calls on sessions interleaved with global calls and skip_frames: neither
    side disturbs the other, and a session's state is a snapshot that later setters do not change."""
    import torch
    a, b = "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei.cfg|d8|420|g100"
    w, h = 512, 64
    sa = new_session(hw, a)
    ea = sa.get_lfsr()
    st_before = sa.get_state()
    hw.reset(); program(hw, b)  # the global state is now b
    eg = hw.get_lfsr()
    oa, og = oracle(a, ea), oracle(b, eg)
    for rnd in range(3):
        specs = [Spec(0, a, w, h, 1 + k % 2, k % 2 == 1, False, False, seed=rnd * 10 + k) for k in range(4)]
        hw.add_grain_jobs_device([sp.job(sa) for sp in specs])
        wants = [sp.want(oa) for sp in specs]
        g = synth_frames(2, w, h, "420", 8, seed=50 + rnd)
        src = to_dev(g.reshape(-1)); dst = torch.zeros_like(src)
        hw.add_grain_frames_device(src, dst, 2, w, h)
        want_g = og.add_grain_frames(g, 2, w, h, 0)
        sa.skip_frames(3, w, h); oa.skip_frames(3, w, h)
        hw.skip_frames(5, w, h); og.skip_frames(5, w, h)
        hw.vfgs_set_seed(rnd + 7); og.vfgs_set_seed(rnd + 7)  # a setter between calls: the session keeps its state
        torch.cuda.synchronize()
        for sp, want in zip(specs, wants):
            assert np.array_equal(sp.result(), want), rnd
        assert np.array_equal(from_dev(dst), want_g), rnd
        assert sa.get_lfsr() == oa.get_lfsr()
        assert hw.get_lfsr() == og.get_lfsr()
    hw.reset()  # reset leaves the session alive
    st_after = sa.get_state()
    for k in ("pattern", "slut", "plut", "scalars"):
        assert np.array_equal(st_before[k], st_after[k]), k
    sp = Spec(0, a, w, h, 1, False, False, False, seed=99)
    hw.add_grain_jobs_device([sp.job(sa)])
    torch.cuda.synchronize()
    assert np.array_equal(sp.result(), sp.want(oa))
    sa.close()


def test_launch_accounting(hw):
    """N jobs of one instantiation cost one stream-kernel launch plus one grain launch (N = 1, 64, 300); a mixed list
    costs one launch per instantiation plus the single-job-route jobs' own launches."""
    import torch
    a = "fgs_afgs1_test1.cfg|d10|420|g100"
    w, h = 512, 32
    s = new_session(hw, a)
    for n in (1, 64, 300):
        specs = [Spec(0, a, w, h, 1, False, False, False, seed=k) for k in range(n)]
        jobs = [sp.job(s) for sp in specs]
        c0 = hw.launch_count()
        hw.add_grain_jobs_device(jobs)
        assert hw.launch_count() - c0 == 2, n
        assert hw.last_launch()["kernels"] == ["fgs_apply_fast_kernel"]
    torch.cuda.synchronize()
    s.close()

    b, ragged = "fgs_sei_ff_test1.cfg|d8|420|g100", "fgs_sei_ff_test5.cfg|d10|420|g100"
    sa, sb, sc = new_session(hw, a), new_session(hw, b), new_session(hw, ragged)

    def launches(jobs):
        c0 = hw.launch_count()
        hw.add_grain_jobs_device(jobs)
        torch.cuda.synchronize()
        return hw.launch_count() - c0
    mk = lambda sess, st, seed, gw=w: Spec(0, st, gw, h, 1, False, False, False, seed=seed).job(sess)
    da = launches([mk(sa, a, k) for k in range(5)])
    db = launches([mk(sb, b, k) for k in range(5)])
    dc = launches([mk(sc, ragged, 0, 200)])  # sample-adaptive chroma on a ragged width: the general kernel
    assert da == 2 and db >= 2 and dc >= 2
    mixed = [mk(sa, a, k) for k in range(5)] + [mk(sb, b, k) for k in range(5)] + [mk(sc, ragged, 9, 200)]
    assert launches(mixed) == 1 + (da - 1) + (db - 1) + dc
    for x in (sa, sb, sc):
        x.close()


def test_in_place(hw):
    """In-place jobs: single-pattern and sample-adaptive configurations, among them 4:2:0 with sample-adaptive chroma
    (8-sample blocks), which takes the single-job route's scratch detour, next to batched in-place jobs."""
    states = ["fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei.cfg|d10|420|g100", (8, 8, "420", 5, 3, 0, 5, True),
              (6, 10, "420", 2, 1, 0, 2, False), (4, 10, "422", 1, 4, 1, 3, False)]
    specs = []
    for k in range(10):
        s = k % len(states)
        depth, fmt = meta(states[s])
        specs.append(Spec(s, states[s], (512, 264, 640)[k % 3], 40, 1 + k % 2, fmt != "444" and k % 3 == 1, False, True, seed=k))
    for x in run_and_check(hw, states, specs)[0]:
        x.close()


def test_refusals(hw):
    """Overlapping jobs, a null session, both or neither pair, negative njobs, a state the kernels cannot run: refused
    before any device work, nothing written (guard bands and outputs keep their sentinel)."""
    import ctypes as C
    import torch
    from versatilefilmgrain_b200 import Job, VfgsError
    from versatilefilmgrain_b200.api import Planes, _CJob
    a = "fgs_afgs1_test1.cfg|d10|420|g100"
    w, h = 512, 32
    s = new_session(hw, a)
    fb = s.frame_bytes(w, h, 10) // 2
    guard = 4096
    raw = torch.full((4 * fb + 2 * guard,), 0x5a5a, dtype=torch.int16, device="cuda")
    src = to_dev(synth_frames(2, w, h, "420", 10, seed=3).reshape(-1))
    src2 = to_dev(synth_frames(1, w, h, "420", 10, seed=4).reshape(-1))  # disjoint from src
    o1, o2 = raw[guard:guard + 2 * fb], raw[guard + fb:guard + 3 * fb]  # o2 overlaps o1's second frame
    lfsr = s.get_lfsr()

    def refused(jobs, n=None):
        with pytest.raises(VfgsError, match="error 1"):
            if n is None:
                hw.add_grain_jobs_device(jobs)
            else:
                hw._chk(hw.L.vfgs_b200_add_grain_jobs_device((_CJob * 1)(), n, None))
        torch.cuda.synchronize()
        assert bool((raw == 0x5a5a).all())
        assert s.get_lfsr() == lfsr

    refused([Job.packed(s, src, o1, 2, w, h), Job.packed(s, src2, o2, 1, w, h)])  # outputs overlap, inputs disjoint
    first, third = raw[guard:guard + fb], raw[guard + 2 * fb:guard + 3 * fb]
    refused([Job.packed(s, src2, first, 1, w, h), Job.packed(s, first, third, 1, w, h)])  # one job reads the other's output
    refused([Job.packed(s, first, third, 1, w, h), Job.packed(s, src2, first, 1, w, h)])  # the same, in the other order
    refused([Job.packed(s, src, o1, 1, w, h), Job.packed(s, src, raw[guard + 3 * fb:guard + 4 * fb], 1, w, h)])  # shared input
    j = Job.packed(s, src, o1, 1, w, h)
    j.session = None
    refused([j])
    j = Job.packed(s, src, o1, 1, w, h)
    j.dst = None
    refused([j])  # half a pair
    j = Job.packed(s, src, o1, 1, w, h)
    j.src = j.dst = None
    refused([j])  # neither pair
    refused([], n=-1)
    both = (_CJob * 1)()
    pl = Job.packed(s, src, o1, 1, w, h)
    from versatilefilmgrain_b200.api import SemiPlanes
    sp = SemiPlanes(src.data_ptr(), src.data_ptr() + w * h * 2, w * 2, w * 2, 0, 2)
    both[0].session, both[0].in_, both[0].out = s.handle, C.pointer(pl.src), C.pointer(pl.dst)
    both[0].sp_in, both[0].sp_out = C.pointer(sp), C.pointer(sp)
    both[0].nframes, both[0].width, both[0].height = 1, w, h
    with pytest.raises(VfgsError, match="error 1"):
        hw._chk(hw.L.vfgs_b200_add_grain_jobs_device(both, 1, None))
    torch.cuda.synchronize()
    assert bool((raw == 0x5a5a).all())
    hw.reset(); program(hw, a)
    bad = np.full(256, 9 << 4, dtype=np.uint8)
    hw.vfgs_set_pattern_lut(1, bad)
    with pytest.raises(VfgsError, match="error 2"):
        hw.create_session()
    hw.reset(); program(hw, a)
    s.close()


def test_destroy_after_enqueue_and_two_streams(hw):
    """session_destroy right after the enqueue still yields the right output; calls on two CUDA streams are correct."""
    import torch
    a, b = "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei.cfg|d10|420|g100"
    w, h = 1920, 1080
    sa, sb = new_session(hw, a), new_session(hw, b)
    ea, eb = sa.get_lfsr(), sb.get_lfsr()
    spa = [Spec(0, a, w, h, 2, False, False, False, seed=k) for k in range(3)]
    spb = [Spec(0, b, w, h, 1, True, False, False, seed=10 + k) for k in range(3)]
    st1, st2 = torch.cuda.Stream(), torch.cuda.Stream()
    ja, jb = [sp.job(sa) for sp in spa], [sp.job(sb) for sp in spb]
    torch.cuda.synchronize()
    hw.add_grain_jobs_device(ja, stream=st1)
    hw.add_grain_jobs_device(jb, stream=st2)
    sa.close(); sb.close()
    torch.cuda.synchronize()
    oa, ob = oracle(a, ea), oracle(b, eb)
    for sp in spa:
        assert np.array_equal(sp.result(), sp.want(oa))
    for sp in spb:
        assert np.array_equal(sp.result(), sp.want(ob))


def test_bench_sized_call(hw):
    """One call of 256 one-frame 1080p jobs and 16 4K jobs over a pool larger than L2, sessions past 2^32 LFSR steps
    (session_skip_frames), every frame checked against the oracle."""
    import torch
    from versatilefilmgrain_b200 import Job
    from versatilefilmgrain_b200.api import P010
    states = ["fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei.cfg|d10|420|g100", "fgs_afgs1_test5.cfg|d10|420|g100",
              "fgs_sei_ff_test1.cfg|d10|420|g100"]
    sessions, epochs = [], []
    for k, st in enumerate(states * 4):  # 16 sessions
        x = new_session(hw, st)
        e = x.get_lfsr()
        x.skip_frames(600_000 + k, 1920, 1080)  # 600k 1080p frames = 4.8e9 LFSR steps
        sessions.append(x); epochs.append(e)
    g = torch.Generator(device="cuda"); g.manual_seed(5)
    jobs, meta_ = [], []
    for k in range(256):
        fb = 1920 * 1080 * 3 // 2
        src = torch.randint(0, 1024, (fb,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
        dst = torch.empty_like(src)
        jobs.append(Job.packed(sessions[k % 16], src, dst, 1, 1920, 1080)); meta_.append((k % 16, src, dst, 1920, 1080, False))
    for k in range(16):
        w, h = 3840, 2160
        src = (torch.randint(0, 1024, (1, h * 3 // 2, w), dtype=torch.int32, device="cuda", generator=g) << 6).to(torch.int16)
        dst = torch.empty_like(src)
        jobs.append(Job.surfaces(sessions[k], src, dst, 1, w, h, out_format=P010)); meta_.append((k, src, dst, w, h, True))
    total = sum(m[1].numel() * 4 for m in meta_)
    assert total > 126 << 20
    hw.add_grain_jobs_device(jobs)
    torch.cuda.synchronize()
    oracles = []
    for k, (st, e) in enumerate(zip(states * 4, epochs)):
        o = oracle(st, e); o.skip_frames(600_000 + k, 1920, 1080)
        oracles.append(o)
    for (s, src, dst, w, h, semi) in meta_:
        o = oracles[s]
        if semi:
            a, b = from_dev(src)[0], from_dev(dst)[0]
            frames = semi_to_planar(a[None, :h], a[None, h:], True)
            want = o.add_grain_frames(frames, 1, w, h, 0)
            assert np.array_equal(semi_to_planar(b[None, :h], b[None, h:], True), want)
        else:
            want = o.add_grain_frames(from_dev(src), 1, w, h, 0)
            assert np.array_equal(from_dev(dst), want)
    for x, o in zip(sessions, oracles):
        assert x.get_lfsr() == o.get_lfsr()
        x.close()
