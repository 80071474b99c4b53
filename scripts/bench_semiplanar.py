"""Semi-planar (NV12 / P010) frames against planar frames of the same workload, in one process on one GPU.

    python scripts/bench_semiplanar.py --out profiles/r03_semiplanar_bench.json

Same protocol as bench.py: resident pools well over L2 (~6.4 GB of input per layout), one warm-up call, timed regions of
over a second, grain-kernel time from vfgs_b200_kernel_timing, algorithmic bytes = samples x (bytes in + bytes out)
(identical for both layouts at the same depth), a sustained plain copy in the same process, GPU name and power limit read
in the same run. Frame rates come from the host clock around synchronised calls. Each workload runs semi-planar and planar alternately, twice. For 4K P010 -> P010 it also times the
workaround a user has without this entry point: deinterleave and shift down into planar scratch buffers, the planar call,
shift up and reinterleave (frames per second of the whole sequence).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

POOL_INPUT_BYTES = 6.4e9
MIN_SECONDS = 1.0

# name: (golden case, width, height, fmt, depth, semi-planar output P010?, in place)
WORKLOADS = {
    "4k420_afgs1_p010_to_p010": ("fgs_afgs1_test1.cfg|d10|420|g100", 3840, 2160, "420", 10, True, False),
    "4k420_afgs1_p010_in_place": ("fgs_afgs1_test1.cfg|d10|420|g100", 3840, 2160, "420", 10, True, True),
    "4k420_afgs1_p010_to_nv12": ("fgs_afgs1_test1.cfg|d10|420|g100", 3840, 2160, "420", 10, False, False),
    "4k420_afgs1_nv12_to_nv12": ("fgs_afgs1_test1.cfg|d8|420|g100", 3840, 2160, "420", 8, False, False),
    "4k420_sei_default_p010": ("fgs_sei.cfg|d10|420|g100", 3840, 2160, "420", 10, True, False),
    "4k422_ff_test4_gain150_p210": ("fgs_sei_ff_test4.cfg|d10|422|g150", 3840, 2160, "422", 10, True, False),
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn, sync, start=None):
    """After one warm-up call (then start()), calls fn() until MIN_SECONDS of wall time have passed, synchronising after
    each call; returns (calls, seconds)."""
    fn(); sync()  # warm-up
    if start:
        start()
    calls, t0 = 0, time.perf_counter()
    while True:
        fn(); calls += 1
        sync()
        dt = time.perf_counter() - t0
        if dt >= MIN_SECONDS:
            return calls, dt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_semiplanar_bench.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()

    import torch
    from tests.util import load_golden, program_case
    from versatilefilmgrain_b200 import VfgsHw
    from versatilefilmgrain_b200.api import NV12, P010, SemiPlanes

    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    G = load_golden()
    hw = VfgsHw(device=0)
    sync = torch.cuda.synchronize
    stream = torch.cuda.current_stream().cuda_stream
    result = {"gpu": gpu_info(), "protocol": __doc__.split("\n\n")[2].replace("\n", " ").strip(), "workloads": {}}

    # sustained plain copy of a pool of the same size
    a = torch.empty(int(POOL_INPUT_BYTES), dtype=torch.uint8, device="cuda"); b = torch.empty_like(a)
    calls, dt = timed(lambda: b.copy_(a), sync)
    result["copy_GBps"] = 2 * a.numel() * calls / dt / 1e9
    del a, b

    for name in args.workloads.split(","):
        case, w, h, fmt, depth, p010_out, in_place = WORKLOADS[name]
        sy = 2 if fmt == "420" else 1
        cw, ch = w // 2, h // sy
        isz = 2 if depth == 10 else 1
        osz = 2 if p010_out else 1
        samples = w * h + 2 * cw * ch
        fin, fout = samples * isz, samples * osz
        F = int(max(8, min(4096, POOL_INPUT_BYTES // fin)))
        idt = torch.int16 if isz == 2 else torch.uint8
        odt = torch.int16 if osz == 2 else torch.uint8
        g = torch.Generator(device="cuda"); g.manual_seed(1)
        hi = 1 << (16 if isz == 2 else 8)
        # semi-planar surfaces (n, h + ch, w) and planar packed frames
        s_in = torch.randint(0, hi, (F, h + ch, w), dtype=torch.int32, device="cuda", generator=g).to(idt)
        s_out = s_in if in_place else torch.empty((F, h + ch, w), dtype=odt, device="cuda")
        p_in = torch.randint(0, 1 << depth, (F * samples,), dtype=torch.int32, device="cuda", generator=g).to(idt)
        p_out = p_in if in_place else torch.empty((F * samples,), dtype=odt, device="cuda")
        hw.reset(); program_case(hw, G, case)
        pin = SemiPlanes(s_in.data_ptr(), s_in.data_ptr() + h * w * isz, w * isz, w * isz, (h + ch) * w * isz, P010 if isz == 2 else NV12)
        pout = SemiPlanes(s_out.data_ptr(), s_out.data_ptr() + h * w * osz, w * osz, w * osz, (h + ch) * w * osz, P010 if osz == 2 else NV12)
        od = 8 if (depth == 10 and not p010_out) else 0

        def semi():
            hw.add_grain_semiplanar_device(pin, pout, F, w, h, stream)

        def planar():
            hw.add_grain_frames_device_ptr(p_in.data_ptr(), p_out.data_ptr(), F, w, h, od, stream)

        arms = {"semiplanar": semi, "planar": planar}
        if name == "4k420_afgs1_p010_to_p010":
            ys, cs = w * h, cw * ch
            scratch_in = torch.empty((F, samples), dtype=torch.int16, device="cuda")
            scratch_out = torch.empty_like(scratch_in)

            def workaround():
                y, uv = s_in[:, :h, :], s_in[:, h:, :].reshape(F, ch, cw, 2)
                scratch_in[:, :ys].view(F, h, w).copy_(torch.bitwise_right_shift(y.to(torch.int32) & 0xffff, 6))
                scratch_in[:, ys:ys + cs].view(F, ch, cw).copy_(torch.bitwise_right_shift(uv[..., 0].to(torch.int32) & 0xffff, 6))
                scratch_in[:, ys + cs:].view(F, ch, cw).copy_(torch.bitwise_right_shift(uv[..., 1].to(torch.int32) & 0xffff, 6))
                hw.add_grain_frames_device_ptr(scratch_in.data_ptr(), scratch_out.data_ptr(), F, w, h, 0, stream)
                s_out[:, :h, :].copy_(scratch_out[:, :ys].view(F, h, w).to(torch.int32).bitwise_left_shift(6).to(torch.int16))
                o = s_out[:, h:, :].reshape(F, ch, cw, 2)
                o[..., 0].copy_(scratch_out[:, ys:ys + cs].view(F, ch, cw).to(torch.int32).bitwise_left_shift(6).to(torch.int16))
                o[..., 1].copy_(scratch_out[:, ys + cs:].view(F, ch, cw).to(torch.int32).bitwise_left_shift(6).to(torch.int16))

            arms["workaround"] = workaround
        rows = {k: [] for k in arms}
        for _ in range(2):
            for arm, fn in arms.items():
                calls, dt = timed(fn, sync, start=lambda: hw.kernel_timing(True))
                kms, launches = hw.kernel_time()
                hw.kernel_timing(False)
                frames = calls * F
                rows[arm].append({"fps": frames / dt, "kernel_ms": kms, "grain_launches": launches,
                                  "kernel_GBps": (samples * (isz + osz) * frames) / (kms / 1e3) / 1e9 if kms else None})
        summary = {arm: {"fps": max(r["fps"] for r in rs), "kernel_GBps": max((r["kernel_GBps"] or 0) for r in rs), "runs": rs}
                   for arm, rs in rows.items()}
        summary["frames_per_call"] = F
        summary["algorithmic_bytes_per_frame"] = samples * (isz + osz)
        summary["semi_over_planar_fps"] = summary["semiplanar"]["fps"] / summary["planar"]["fps"]
        if "workaround" in summary:
            summary["semi_over_workaround_fps"] = summary["semiplanar"]["fps"] / summary["workaround"]["fps"]
        for arm in arms:
            summary[arm]["kernel_share_of_copy"] = summary[arm]["kernel_GBps"] / result["copy_GBps"]
        result["workloads"][name] = summary
        print(name, json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "runs"})
                                for k, v in summary.items()}), flush=True)
        del s_in, s_out, p_in, p_out
        arms.clear()
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"gpu": result["gpu"], "copy_GBps": result["copy_GBps"]}))


if __name__ == "__main__":
    main()
