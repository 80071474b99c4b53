"""Batched calls (vfgs_b200_add_grain_jobs_device) through the host build of the task code (tests/emu/emu_jobs.cpp): job
lists planned and grouped with the shim's own code, block tables from the job-table stream kernel's walk, every group
replayed CTA by CTA with the kernels' schedule and a table reload at every job switch. Outputs and session registers
against one Oracle per session; the jobs the single-job route serves go through the single-job emulators. Needs no GPU."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle.pyoracle import RefState
from tests.semiplanar import Surface, load_emu as load_emu_semi, planar_to_semi, run_emu_semi, semi_to_planar
from tests.util import Oracle, aligned_empty, build_emu, load_golden, program_case, program_random_state, synth_frames

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
G = load_golden()


class EmuJob(C.Structure):
    _fields_ = [("session", C.c_int), ("semi", C.c_int), ("nframes", C.c_int), ("width", C.c_int), ("height", C.c_int),
                ("out_depth", C.c_int), ("in_y", C.c_void_p), ("in_uv", C.c_void_p), ("sy_in", C.c_longlong),
                ("suv_in", C.c_longlong), ("fs_in", C.c_longlong), ("out_y", C.c_void_p), ("out_uv", C.c_void_p),
                ("sy_out", C.c_longlong), ("suv_out", C.c_longlong), ("fs_out", C.c_longlong)]


@pytest.fixture(scope="module")
def emu():
    so, src = os.path.join(HERE, "libemu_jobs.so"), os.path.join(HERE, "emu_jobs.cpp")
    csrc = os.path.join(HERE, "..", "..", "versatilefilmgrain_b200", "csrc")
    deps = [src] + [os.path.join(csrc, n) for n in os.listdir(csrc) if n.endswith(".h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-Wno-unknown-pragmas", "-o", so, src],
                       check=True)
    L = C.CDLL(so)
    assert L.emuj_state_size() == C.sizeof(RefState)
    L.emuj_replay.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    L.emuj_run_jobs.argtypes = [C.c_void_p, C.c_int, C.POINTER(EmuJob), C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                C.c_void_p, C.c_void_p]
    return L


@pytest.fixture(scope="module")
def single():
    """The single-job emulators (planar, semi-planar), which the single-job route's jobs go through."""
    L = C.CDLL(build_emu())
    L.emu_add_grain_frames.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 6
    return L, load_emu_semi()


# ---- schedule ----------------------------------------------------------------------------------------------------
def replay(emu, ntasks, grid, warps):
    nt = np.ascontiguousarray(ntasks, dtype=np.int64)
    hits = np.zeros(max(int(nt.sum()), 1), dtype=np.int32)
    sw = np.zeros(grid, dtype=np.int32)
    rc = emu.emuj_replay(nt.ctypes.data, len(nt), grid, warps, hits.ctypes.data, sw.ctypes.data)
    return rc, hits[:int(nt.sum())], sw


@pytest.mark.parametrize("seed", range(40))
def test_every_task_once_in_order(emu, seed):
    """Random job lists (1-300 jobs, mixed sizes, empty jobs) and grids, walked with the kernels' own multi_begin /
    multi_next: exact coverage, contiguous ranges in order, and one table load per job a CTA range touches."""
    rng = np.random.default_rng(seed)
    njobs = int(rng.integers(1, 301))
    kind = rng.integers(0, 4, size=njobs)
    sizes = np.where(kind == 0, 0, np.where(kind == 1, rng.integers(1, 40, size=njobs),
                                            np.where(kind == 2, rng.integers(40, 3000, size=njobs), rng.integers(3000, 60000, size=njobs))))
    grid = int(rng.integers(1, 300))
    warps = int(rng.choice([16, 24, 28, 32]))
    rc, hits, sw = replay(emu, sizes, grid, warps)
    assert rc == 0
    assert (hits == 1).all()
    assert int(sw.sum()) <= int((sizes > 0).sum()) + grid - 1
    total = int(sizes.sum())
    bounds = np.concatenate([[0], np.cumsum(sizes)])
    for b in range(grid):
        lo, hi = total * b // grid, total * (b + 1) // grid
        assert sw[b] == int(((bounds[:-1] < hi) & (bounds[1:] > lo) & (sizes > 0)).sum())


def test_single_job_and_repeated_jobs(emu):
    """One job: every CTA loads once, balanced contiguous ranges; only empty jobs: nothing runs; one size repeated."""
    rc, hits, sw = replay(emu, [100_003], 148, 24)
    assert rc == 0 and (hits == 1).all() and (sw == 1).all()
    rc, hits, sw = replay(emu, [0, 0, 0], 8, 32)
    assert rc == 0 and hits.size == 0 and (sw == 0).all()
    rc, hits, sw = replay(emu, [64] * 300, 148, 32)
    assert rc == 0 and (hits == 1).all() and int(sw.sum()) <= 300 + 147


# ---- outputs -----------------------------------------------------------------------------------------------------
def program(target, state):
    if isinstance(state, str):
        program_case(target, G, state)
    else:
        program_random_state(target, *state)


def meta(state):
    if isinstance(state, str):
        return G.cases[state]["depth"], G.cases[state]["fmt"]
    return state[1], state[2]


def dump(o):
    st = RefState()
    o.L.oracle_get_state(o.h, C.byref(st))
    return st


class Spec:
    def __init__(self, sess, state, w, h, n, semi, out8, in_place, seed):
        self.depth, self.fmt = meta(state)
        self.sess, self.w, self.h, self.n = sess, w, h, n
        self.semi, self.in_place = semi and self.fmt != "444", in_place
        self.out8 = out8 and self.depth == 10 and not in_place
        self.frames = synth_frames(n, w, h, self.fmt, self.depth, seed=seed)
        isz, osz = (2 if self.depth == 10 else 1), (1 if self.out8 or self.depth == 8 else 2)
        if self.semi:
            ch = h // (2 if self.fmt == "420" else 1)
            Y, UV = planar_to_semi(self.frames, n, w, h, self.fmt, self.depth == 10)
            self.src = Surface(n, w, h, ch, isz)
            self.src.fill(Y, UV)
            self.dst = self.src if in_place else Surface(n, w, h, ch, osz)
        else:
            self.src = aligned_empty(self.frames.size, self.frames.dtype)
            self.src[:] = self.frames.reshape(-1)
            self.dst = self.src if in_place else aligned_empty(self.frames.size, np.uint8 if osz == 1 else np.uint16)

    def cjob(self):
        j = EmuJob()
        j.session, j.semi, j.nframes, j.width, j.height = self.sess, int(self.semi), self.n, self.w, self.h
        j.out_depth = 8 if self.out8 else 0
        if self.semi:
            j.in_y, j.in_uv, j.sy_in, j.suv_in, j.fs_in = self.src.args()
            j.out_y, j.out_uv, j.sy_out, j.suv_out, j.fs_out = self.dst.args()
        else:
            j.in_y, j.out_y = self.src.ctypes.data, self.dst.ctypes.data
        return j

    def run_single(self, single, st, o, mode):
        """The single-job route's emulation, with the session's state before this job."""
        L, semi = single
        if self.semi:
            run_emu_semi(semi, o, self.src, self.dst, self.n, self.w, self.h, not (self.out8 or self.depth == 8), mode=mode)
        else:  # in place, the route goes through a scratch output buffer (emu.cpp has no such detour of its own)
            out = aligned_empty(self.dst.size, self.dst.dtype) if self.in_place else self.dst
            L.emu_add_grain_frames(C.byref(st), self.src.ctypes.data, out.ctypes.data, self.n, self.w, self.h,
                                   8 if self.out8 else 0, 0, mode)
            self.dst[:] = out

    def result(self):
        if self.semi:
            y, uv = self.dst.planes()
            return semi_to_planar(y, uv, not (self.out8 or self.depth == 8))
        return self.dst


def run_call(emu, single, states, specs, mode=0, grid=5, warps=24):
    """One emulated batched call; checks every output and every session's registers against one Oracle per session."""
    oracles = []
    for s in states:
        o = Oracle(); program(o, s)
        oracles.append(o)
    dumps = (RefState * len(states))(*[dump(o) for o in oracles])
    arr = (EmuJob * len(specs))(*[sp.cjob() for sp in specs])
    regs = np.zeros(4 * len(states), dtype=np.uint32)
    batched = np.zeros(len(specs), dtype=np.int32)
    keys = np.zeros(16, dtype=np.int32)
    wants = []
    singles = []
    for sp in specs:  # the oracle in list order; the single-job route's jobs start from the state their session has then
        o = oracles[sp.sess]
        singles.append((dump(o), o.get_lfsr()))
        wants.append(o.add_grain_frames(sp.frames, sp.n, sp.w, sp.h, 8 if sp.out8 else 0))
    launches = emu.emuj_run_jobs(dumps, len(states), arr, len(specs), mode, grid, warps, regs.ctypes.data,
                                 batched.ctypes.data, keys.ctypes.data)
    assert launches >= 0
    for sp, b, (st, lfsr) in zip(specs, batched, singles):
        if not b:
            o = Oracle(); program(o, states[sp.sess]); o.set_lfsr(lfsr)
            sp.run_single(single, st, o, mode)
    for k, (sp, want) in enumerate(zip(specs, wants)):
        got = sp.result()
        assert np.array_equal(got, want), (k, states[sp.sess], sp.w, sp.h, sp.n, sp.semi, sp.out8, sp.in_place, bool(batched[k]),
                                           int(np.count_nonzero(got != want)))
    for k, o in enumerate(oracles):
        assert [int(v) for v in regs[4 * k:4 * k + 4]] == o.get_lfsr(), k
    return batched, [int(v) for v in keys[:min(launches, 16)]]


STATES = ["fgs_afgs1_test1.cfg|d10|420|g100", "fgs_afgs1_test1.cfg|d8|420|g100", "fgs_sei.cfg|d10|420|g100",
          "fgs_sei.cfg|d8|420|g100", "fgs_sei_ff_test1.cfg|d10|422|g100", "fgs_sei_ff_test1.cfg|d10|444|g100",
          "fgs_sei_ar_test1.cfg|d10|422|g150", "fgs_sei_ff_test5.cfg|d10|420|g100",
          (8, 8, "420", 5, 3, 0, 5, True), (6605739, 10, "422", 4, 2, 0, 7, False), (3, 8, "444", 3, 2, 0, 4, False)]
GEOMS = [(264, 40, 1), (512, 34, 2), (204, 36, 1), (640, 18, 1), (328, 20, 2)]


@pytest.mark.parametrize("mode", [0, 2])
@pytest.mark.parametrize("seed", range(6))
def test_mixed_lists_equal_oracle(emu, single, seed, mode):
    """Mixed lists: 8-bit, 10-bit and 10 -> 8; 4:2:0, 4:2:2 and 4:4:4; semi-planar; ragged widths (EDGE); sample-adaptive
    (gather) states; in place; one session in several jobs. Every output and every session's registers equal the oracle's."""
    rng = np.random.default_rng(100 + seed)
    states = [STATES[int(i)] for i in rng.choice(len(STATES), size=5, replace=False)]
    specs = []
    for k in range(int(rng.integers(6, 11))):
        s = int(rng.integers(len(states)))
        w, h, n = GEOMS[int(rng.integers(len(GEOMS)))]
        specs.append(Spec(s, states[s], w, h, n, bool(rng.integers(2)), bool(rng.integers(2)), bool(rng.integers(4) == 0),
                          seed=seed * 100 + k))
    batched, _ = run_call(emu, single, states, specs, mode=mode, grid=int(rng.integers(1, 8)), warps=int(rng.choice([16, 24, 28])))
    assert mode != 0 or batched.any()


def test_every_kind_of_group_in_one_call(emu, single):
    """One call whose batched jobs need the fast kernel (planar 10-bit, 8-bit, 10 -> 8, semi-planar P010 and NV12), its
    EDGE variant (ragged width) and the gather kernel (default SEI, sample-adaptive random states), several jobs per group,
    next to jobs of the single-job route (general kernel on a ragged sample-adaptive state, in-place scratch detour)."""
    states = ["fgs_afgs1_test1.cfg|d10|420|g100", "fgs_afgs1_test1.cfg|d8|420|g100", "fgs_sei.cfg|d10|420|g100",
              (8, 8, "420", 5, 3, 0, 5, True), "fgs_sei_ff_test1.cfg|d10|444|g100"]
    specs = [Spec(0, states[0], 264, 40, 1, False, False, False, 1), Spec(0, states[0], 512, 34, 2, False, True, False, 2),
             Spec(0, states[0], 512, 34, 1, True, False, False, 3), Spec(1, states[1], 264, 40, 1, False, False, False, 4),
             Spec(1, states[1], 512, 40, 1, True, False, False, 5), Spec(1, states[1], 204, 36, 1, False, False, False, 6),
             Spec(2, states[2], 512, 40, 1, False, False, False, 7), Spec(2, states[2], 264, 40, 2, False, True, False, 8),
             Spec(3, states[3], 512, 40, 1, False, False, False, 9), Spec(3, states[3], 204, 36, 1, False, False, False, 10),
             Spec(3, states[3], 512, 32, 1, False, False, True, 11), Spec(4, states[4], 328, 20, 2, False, False, False, 12),
             Spec(0, states[0], 264, 40, 1, False, False, True, 13), Spec(2, states[2], 512, 40, 1, False, False, True, 14)]
    batched, keys = run_call(emu, single, states, specs, grid=3, warps=24)
    kinds = {k & 3 for k in keys}
    assert kinds == {0, 1, 3}, keys
    assert len(keys) >= 5
    assert not batched.all()  # the ragged sample-adaptive job takes the general kernel on its own
