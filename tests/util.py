"""Shared helpers for the test-suite (fixtures decoding, state programming, digests)."""
from __future__ import annotations

import hashlib
import json
import os

import numpy as np

from oracle.pyoracle import Oracle, program_hw_from_state, synth_frames  # noqa: F401

from tests.fixtures import GOLDEN, Golden, load_golden, parse_output_key, program_case, sha  # noqa: E402,F401


def states_equal(a: dict, b: dict, nslot=None) -> list:
    """Names of the fields that differ. nslot = [luma, chroma] restricts the pattern comparison to
    the slots the pattern LUTs can select (the fixtures keep only those)."""
    bad = []
    for k in ("slut", "plut", "scalars", "lfsr"):
        if not np.array_equal(np.asarray(a[k]), np.asarray(b[k])):
            bad.append(k)
    pa, pb = np.asarray(a["pattern"]), np.asarray(b["pattern"])
    if nslot is None:
        if not np.array_equal(pa, pb):
            bad.append("pattern")
    else:
        for bank in range(2):
            if not np.array_equal(pa[bank, :nslot[bank]], pb[bank, :nslot[bank]]):
                bad.append(f"pattern[{bank}]")
    return bad


def first_mismatch(a: np.ndarray, b: np.ndarray, width, height, fmt, nframes):
    """Human-readable location of the first differing sample of two packed planar buffers."""
    from oracle.pyoracle import frame_samples
    idx = np.nonzero(a != b)[0]
    if idx.size == 0:
        return "identical"
    i = int(idx[0])
    ys, cs, cw, _ = frame_samples(width, height, fmt)
    per = ys + 2 * cs
    f, r = divmod(i, per)
    if r < ys:
        c, y, x = 0, r // width, r % width
    else:
        r -= ys
        c = 1 + r // cs
        r %= cs
        y, x = r // cw, r % cw
    return f"{idx.size} samples differ; first at frame {f} comp {c} line {y} col {x}: got {int(a[i])} want {int(b[i])}"


def build_emu() -> str:
    """Host build of the kernel's per-lane task code (tests/emu/emu.cpp), test tool only."""
    import subprocess
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
    so, src = os.path.join(here, "libemu.so"), os.path.join(here, "emu.cpp")
    csrc = os.path.join(os.path.dirname(here), "..", "versatilefilmgrain_b200", "csrc")
    deps = [src] + [os.path.join(csrc, n) for n in os.listdir(csrc) if n.endswith(".h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        # -Bsymbolic: the inline functions of the shared headers must bind to this library's own copies, not to
        # those libvfgs_b200.so exports when a test has loaded it first
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-Wl,-Bsymbolic", "-Wno-unknown-pragmas", "-o", so, src], check=True)
    return so


def program_random_state(target, seed: int, depth: int, fmt: str, nluma: int = 1, nchroma: int = 1, legal: int = 0,
                         shift: int = 5, with_minus128: bool = False) -> None:
    """Programs `target` (Oracle, Reference or VfgsHw: same setter names as src/vfgs_hw.h) with a random but
    legal hardware state through the setters, in the order the reference's firmware uses (vfgs_main.c:750-760,
    vfgs_fw.c:578-643): nluma / nchroma pattern slots selected by random pattern LUTs, random scale LUTs."""
    rng = np.random.default_rng(seed)
    sx, sy = {"420": (2, 2), "422": (2, 1), "444": (1, 1)}[fmt]
    target.vfgs_set_depth(depth)
    target.vfgs_set_chroma_subsampling(sx, sy)
    lo = -128 if with_minus128 else -127
    for i in range(nluma):
        target.vfgs_set_luma_pattern(i, rng.integers(lo, 128, size=(64, 64), dtype=np.int8))
    for i in range(nchroma):
        # a full 64 x 64 buffer: the reference reads 64/csubx bytes every 64/csuby bytes (vfgs_hw.c:320-325), which
        # for 4:2:2 reaches past a packed 64 x 32 array
        target.vfgs_set_chroma_pattern(i, rng.integers(lo, 128, size=(64, 64), dtype=np.int8))
    for c in range(3):
        n = nluma if c == 0 else nchroma
        slots = rng.integers(0, n, size=8)
        plut = (np.repeat(slots, 32).astype(np.uint8) << 4) | rng.integers(0, 16, size=256, dtype=np.uint8)  # low nibble is ignored (>> 4)
        target.vfgs_set_scale_lut(c, rng.integers(0, 256, size=256, dtype=np.uint8))
        target.vfgs_set_pattern_lut(c, np.ascontiguousarray(plut.astype(np.uint8)))
    target.vfgs_set_scale_shift(shift)
    target.vfgs_set_legal_range(legal)
    target.vfgs_set_seed(int(rng.integers(1, 1 << 31)))


# (seed, depth, fmt, luma slots, chroma slots, legal range, scale shift, -128 bytes in the patterns)
RANDOM_STATES = [
    (1, 8, "422", 1, 1, 0, 2, False), (2, 8, "444", 1, 1, 1, 7, False), (3, 8, "444", 3, 2, 0, 4, False),
    (4, 10, "422", 1, 4, 1, 3, False), (5, 10, "444", 8, 8, 0, 6, False), (6, 10, "420", 2, 1, 0, 2, False),
    (7, 10, "420", 1, 1, 1, 7, True), (8, 8, "420", 5, 3, 0, 5, True), (9, 10, "444", 1, 1, 0, 5, False),
    # found by fuzzing the emulated kernels: Cb sample-adaptive (gather kernel), Cr one slot (fast kernel, own image)
    (6605739, 10, "422", 4, 2, 0, 7, False), (765400224, 10, "444", 6, 2, 1, 5, False),
]


# bench.py's default run (--steps 20 --warmup 5) on the largest box the project reports on (--gpus 8)
BENCH_STEPS, BENCH_WARMUP, BENCH_GPUS = 20, 5, 8


def bench_call(workload: str, gpus: int = BENCH_GPUS):
    """(frames per call, calls per step, first frame of the last call) of a default weak-scaling bench.py run of
    `workload`, computed the way bench.py computes them: the last call is the last pass of the last step on the
    highest rank, which starts furthest into the sequence."""
    import bench
    _, w, h, fmt, depth, od = bench.WORKLOADS[workload]
    _, in_bytes, out_bytes = bench.frame_geometry(w, h, fmt, depth, od)
    frames = int(max(8, min(4096, bench.POOL_INPUT_BYTES // in_bytes)))
    passes = max(1, int(round(4.0e11 / (frames * (in_bytes + out_bytes)))))
    s, p, rank = BENCH_WARMUP + BENCH_STEPS - 1, passes - 1, gpus - 1
    return frames, passes, ((s * passes + p) * gpus + rank) * frames


def bench_last_call_first_frame(workload: str) -> int:
    return bench_call(workload)[2]


def aligned_empty(n, dtype, offset=0):
    """n zeroed elements whose first byte sits `offset` bytes after a 64-byte boundary (numpy itself only promises 16):
    the 16-samples-per-lane paths of the fast kernel need 16 / 32-byte aligned rows."""
    item = np.dtype(dtype).itemsize
    raw = np.zeros(n * item + 128, dtype=np.uint8)
    start = (-raw.ctypes.data) % 64 + offset
    return raw[start:start + n * item].view(dtype)
