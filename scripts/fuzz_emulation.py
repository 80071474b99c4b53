#!/usr/bin/env python
"""Fuzzes the kernels' task code (host build, tests/emu) against the oracle: random hardware states programmed
through the setters (depth, format, 1-8 pattern slots per bank, legal range, scale shift, -128 pattern bytes),
random picture sizes, in-range and garbage samples, frame offsets into a running sequence, in-place operation, every
kernel-selection mode. Test tool, no GPU.

    python scripts/fuzz_emulation.py [seed] [seconds] [--semiplanar]

--semiplanar: semi-planar frames (vfgs_b200_add_grain_semiplanar_device, tests/emu/emu_semiplanar.cpp) instead, 4:2:0 / 4:2:2,
NV12 / P010 / P010 -> NV12, random widths, base alignments, padded pitches and in place.

(Found in round 1: a Cr component with its own fast-kernel image next to a sample-adaptive Cb got an empty image.)"""
import ctypes as C
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

from oracle.pyoracle import RefState, _ptr  # noqa: E402
from tests.util import Oracle, aligned_empty, build_emu, first_mismatch, program_random_state, synth_frames  # noqa: E402

WIDTHS = [136, 144, 152, 160, 200, 203, 256, 264, 270, 272, 366, 512, 520, 523, 528, 1040]


def one_case(emu, rng):
    depth = int(rng.choice([8, 10])); fmt = str(rng.choice(["420", "422", "444"]))
    one = rng.integers(0, 4) == 0  # a quarter of the cases with one pattern per bank (fast kernel everywhere)
    spec = (int(rng.integers(1, 1 << 30)), depth, fmt, 1 if one else int(rng.integers(1, 9)), 1 if one else int(rng.integers(1, 9)),
            int(rng.integers(0, 2)), int(rng.integers(2, 8)), bool(rng.integers(0, 4) == 0))
    w = int(rng.choice(WIDTHS)); h = max(2, int(rng.integers(1, 70))); n = int(rng.integers(1, 4))
    for od in ((0, 8) if depth == 10 else (0,)):
        kind = "natural" if rng.integers(0, 3) == 0 else "uniform"  # smooth frames exercise the gather code's octet path
        frames = synth_frames(n, w, h, fmt, depth, seed=spec[0] % 1000, kind=kind)
        if depth == 10 and rng.integers(0, 3) == 0:
            frames = rng.integers(0, 65536, size=frames.size, dtype=np.uint16)  # codes far outside 10 bits
        o = Oracle(); program_random_state(o, *spec)
        st = RefState(); o.L.oracle_get_state(o.h, C.byref(st))
        first = int(rng.integers(0, 5000)) if rng.integers(0, 3) == 0 else 0  # frames of a sequence already under way
        # buffer alignment decides between 16 samples per lane (32-byte aligned rows), 8 samples per lane and the EDGE variant
        offset = int(rng.choice([0, 0, 0, 32, 16, 8, 4, 2])) & ~(frames.itemsize - 1)
        src = aligned_empty(frames.size, frames.dtype, offset); src[:] = frames.reshape(-1)
        frames = src
        outs = []
        for mode in (0, 1, 2):
            out = aligned_empty(frames.size, np.uint8 if (od == 8 or depth == 8) else np.uint16, int(rng.choice([offset, 0])))
            emu.emu_add_grain_frames(C.byref(st), _ptr(frames), _ptr(out), n, w, h, od, first, mode)
            outs.append((f"mode={mode} offset={offset}", out))
        if od == 0:  # same depth in and out: in place as well
            buf = aligned_empty(frames.size, frames.dtype, offset); buf[:] = frames
            mask = emu.emu_add_grain_frames(C.byref(st), _ptr(buf), _ptr(buf), n, w, h, od, first, 0)
            # sample-adaptive components on the general task code read neighbouring input samples: the shim sends those
            # calls through a scratch buffer (vfgs_b200.cu, in_place_needs_scratch), the emulation has none
            if (spec[3] == 1 and spec[4] == 1) or not (mask & 2):
                outs.append((f"in place (mask {mask})", buf))
        o.skip_frames(first, w, h)
        want = o.add_grain_frames(frames, n, w, h, od)
        for what, got in outs:
            if not np.array_equal(got, want):
                return f"MISMATCH spec={spec} w={w} h={h} n={n} od={od} first={first} {what}: {first_mismatch(got, want, w, h, fmt, n)}"
    return None


def one_semiplanar_case(emu, rng):
    from tests.semiplanar import Surface, planar_to_semi, run_emu_semi, semi_to_planar
    depth = int(rng.choice([8, 10])); fmt = str(rng.choice(["420", "422"]))
    one = rng.integers(0, 2) == 0  # half of the cases with one pattern per bank (the interleaved fast lane)
    spec = (int(rng.integers(1, 1 << 30)), depth, fmt, 1 if one else int(rng.integers(1, 9)), 1 if one else int(rng.integers(1, 9)),
            int(rng.integers(0, 2)), int(rng.integers(2, 8)), bool(rng.integers(0, 4) == 0))
    w = int(rng.choice(WIDTHS)) & ~1; h = max(2, int(rng.integers(1, 70))) & ~1; n = int(rng.integers(1, 4))
    ch = h // (2 if fmt == "420" else 1)
    p010 = depth == 10
    frames = synth_frames(n, w, h, fmt, depth, seed=spec[0] % 1000)
    first = int(rng.integers(0, 5000)) if rng.integers(0, 3) == 0 else 0
    for p010_out in ((True, False) if p010 else (False,)):
        for in_place in ((False, True) if p010_out == p010 else (False,)):
            mode = int(rng.choice([0, 0, 1, 2]))
            o = Oracle(); program_random_state(o, *spec)
            isz, osz = (2 if p010 else 1), (2 if p010_out else 1)
            offset = int(rng.choice([0, 0, 32, 16, 8, 4, 2])) & ~(isz - 1)
            pads = [int(rng.choice([0, 0, 16, 32, 64, 2])) & ~(max(isz, osz) - 1) for _ in range(2)]
            src = Surface(n, w, h, ch, isz, w * isz + pads[0], w * isz + pads[1], offset)
            Y, UV = planar_to_semi(frames, n, w, h, fmt, p010, rng=rng)
            src.fill(Y, UV)
            dst = src if in_place else Surface(n, w, h, ch, osz, w * osz + pads[0], w * osz + pads[1], int(rng.choice([offset, 0])) & ~(osz - 1))
            mask = run_emu_semi(emu, o, src, dst, n, w, h, p010_out, first=first, mode=mode)
            o.skip_frames(first, w, h)
            want = o.add_grain_frames(frames, n, w, h, 0 if p010_out == p010 else 8)
            got = semi_to_planar(*dst.planes(), p010_out)
            if not np.array_equal(got, want):
                return (f"MISMATCH semiplanar spec={spec} w={w} h={h} n={n} p010_out={p010_out} in_place={in_place} mode={mode} "
                        f"offset={offset} pads={pads} mask={mask}: {first_mismatch(got, want, w, h, fmt, n)}")
    return None


def run(seed: int, seconds: float, max_cases: int = 0, semiplanar: bool = False):
    if semiplanar:
        from tests.semiplanar import load_emu
        emu = load_emu()
    else:
        emu = C.CDLL(build_emu())
        emu.emu_add_grain_frames.argtypes = [C.c_void_p] * 3 + [C.c_int] * 6
    rng = np.random.default_rng(seed)
    t0, n = time.time(), 0
    while time.time() - t0 < seconds and (max_cases == 0 or n < max_cases):
        bad = one_semiplanar_case(emu, rng) if semiplanar else one_case(emu, rng)
        if bad:
            return n, bad
        n += 1
    return n, None


if __name__ == "__main__":
    semi = "--semiplanar" in sys.argv
    argv = [a for a in sys.argv[1:] if a != "--semiplanar"]
    n, bad = run(int(argv[0]) if argv else 0, float(argv[1]) if len(argv) > 1 else 60, semiplanar=semi)
    print(bad or f"fuzz ok: {n} cases")
    sys.exit(1 if bad else 0)
