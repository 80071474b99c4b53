"""Many video streams, each with its own grain state, in one process on one GPU.

    python scripts/bench_sessions.py --out profiles/r04_sessions_bench.json

Each workload is a list of streams; one call processes the next frames of every stream. Arms: (a) one batched call
(vfgs_b200_add_grain_jobs_device over one session per stream); (b) the same jobs as one jobs call per job; (c) the
workaround without sessions: per stream, the global state re-programmed through the setters and the stream's registers
set before and read after its single-job call; (d) the upper bound: the same total frames as one planar call of a
single configuration. Every stream owns its input and output buffers, the pool is well over L2 (126 MB). Frame rates come
from the host clock around synchronised calls (one warm-up call, timed regions of over a second, arms alternated, twice);
grain-kernel time from vfgs_b200_kernel_timing; algorithmic bytes = samples x (bytes in + bytes out); a plain copy is
timed in the same process; the GPU name and power limit are read in the same run.
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

MIN_SECONDS = 1.0
AFGS, SEI = "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei.cfg|d10|420|g100"
AFGS8, FF1 = "fgs_afgs1_test1.cfg|d8|420|g100", "fgs_sei_ff_test1.cfg|d10|420|g100"
# name: list of (count, golden case, width, height, frames per call, semi-planar P010)
WORKLOADS = {
    "64x1080p_10bit_single_pattern": [(64, AFGS, 1920, 1080, 1, False)],
    "16x4k_p010_2_frames": [(16, AFGS, 3840, 2160, 2, True)],
    "mix_32x1080p_8x4k": [(12, AFGS, 1920, 1080, 1, False), (10, SEI, 1920, 1080, 1, False), (10, AFGS8, 1920, 1080, 1, False),
                          (4, FF1, 3840, 2160, 1, True), (4, SEI, 3840, 2160, 1, False)],
}


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn, sync, start=None):
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_sessions_bench.json"))
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()

    import torch
    from tests.util import load_golden, program_case, program_hw_from_state
    from versatilefilmgrain_b200 import Job, VfgsHw

    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    G = load_golden()
    hw = VfgsHw(device=0)
    sync = torch.cuda.synchronize
    result = {"gpu": gpu_info(), "protocol": __doc__.split("\n\n")[2].replace("\n", " ").strip(), "workloads": {}}

    a = torch.empty(4 << 30, dtype=torch.uint8, device="cuda"); b = torch.empty_like(a)
    calls, dt = timed(lambda: b.copy_(a), sync)
    result["copy_GBps"] = 2 * a.numel() * calls / dt / 1e9
    del a, b

    g = torch.Generator(device="cuda"); g.manual_seed(1)
    for name in args.workloads.split(","):
        streams = []  # (case, session, job, state dict)
        total_frames, total_bytes = 0, 0
        for count, case, w, h, n, semi in WORKLOADS[name]:
            depth = G.cases[case]["depth"]
            hw.reset(); program_case(hw, G, case)
            state = hw.state()
            samples = w * h * 3 // 2
            dt_ = torch.int16 if depth == 10 else torch.uint8
            for k in range(count):
                s = hw.create_session()
                if semi:
                    src = (torch.randint(0, 1 << depth, (n, h * 3 // 2, w), dtype=torch.int32, device="cuda", generator=g) << 6).to(dt_)
                    job = Job.surfaces(s, src, torch.empty_like(src), n, w, h)
                else:
                    src = torch.randint(0, 1 << depth, (n * samples,), dtype=torch.int32, device="cuda", generator=g).to(dt_)
                    job = Job.packed(s, src, torch.empty_like(src), n, w, h)
                streams.append((case, s, job, state))
                total_frames += n
                total_bytes += n * samples * 2 * (2 if depth == 10 else 1)

        def batched():
            hw.add_grain_jobs_device([j for _, _, j, _ in streams])

        def per_job():
            for _, _, j, _ in streams:
                hw.add_grain_jobs_device([j])

        regs = [s.get_lfsr() for _, s, _, _ in streams]

        def workaround():
            for k, (case, s, j, st) in enumerate(streams):
                program_hw_from_state(hw, st)
                hw.set_lfsr(regs[k])
                if j.src.__class__.__name__ == "SemiPlanes":
                    hw.add_grain_semiplanar_device(j.src, j.dst, j.nframes, j.width, j.height, torch.cuda.current_stream().cuda_stream)
                else:
                    hw.add_grain_planes_device(j.src, j.dst, j.nframes, j.width, j.height, 0, torch.cuda.current_stream().cuda_stream)
                regs[k] = hw.get_lfsr()

        # upper bound: the same number of frames as one planar call of one configuration (1080p / 4K by the workload's bulk)
        w0, h0 = (3840, 2160) if "4k" in name and "mix" not in name else (1920, 1080)
        fb = w0 * h0 * 3 // 2
        nb = max(1, total_bytes // (fb * 4))
        ub_in = torch.randint(0, 1024, (nb * fb,), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
        ub_out = torch.empty_like(ub_in)

        def upper():
            hw.add_grain_frames_device(ub_in, ub_out, nb, w0, h0)

        def upper_config():  # (d) is one AFGS1 10-bit 4:2:0 configuration, whatever the other arms left programmed
            hw.reset(); program_case(hw, G, AFGS)

        arms = {"a_batched": (batched, total_frames), "b_one_call_per_job": (per_job, total_frames),
                "c_global_reprogram": (workaround, total_frames), "d_single_config_call": (upper, nb)}
        rows = {k: [] for k in arms}
        for _ in range(2):
            for arm, (fn, frames_per_call) in arms.items():
                if arm == "d_single_config_call":
                    upper_config()
                c0 = hw.launch_count()
                fn(); sync()
                launches = hw.launch_count() - c0
                calls, dt = timed(fn, sync, start=lambda: hw.kernel_timing(True))
                kms, _ = hw.kernel_time()
                hw.kernel_timing(False)
                byts = total_bytes if arm != "d_single_config_call" else nb * fb * 4
                rows[arm].append({"fps": calls * frames_per_call / dt, "launches_per_call": launches,
                                  "kernel_GBps": byts * calls / (kms / 1e3) / 1e9 if kms else None})
        summary = {arm: {"fps": max(r["fps"] for r in rs), "launches_per_call": rs[-1]["launches_per_call"],
                         "kernel_GBps": max((r["kernel_GBps"] or 0) for r in rs), "runs": rs} for arm, rs in rows.items()}
        for arm in summary:
            summary[arm]["kernel_share_of_copy"] = summary[arm]["kernel_GBps"] / result["copy_GBps"]
        summary["streams"] = len(streams)
        summary["frames_per_call"] = total_frames
        summary["a_over_b"] = summary["a_batched"]["fps"] / summary["b_one_call_per_job"]["fps"]
        summary["a_over_c"] = summary["a_batched"]["fps"] / summary["c_global_reprogram"]["fps"]
        summary["a_over_d"] = summary["a_batched"]["fps"] / summary["d_single_config_call"]["fps"]
        result["workloads"][name] = summary
        print(name, json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "runs"})
                                for k, v in summary.items()}), flush=True)
        sync()
        for _, s, _, _ in streams:
            s.close()
        del streams, ub_in, ub_out
        torch.cuda.empty_cache()

    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"gpu": result["gpu"], "copy_GBps": result["copy_GBps"]}))


if __name__ == "__main__":
    main()
