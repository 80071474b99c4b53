"""Per-picture metadata on grain sessions: one batched vfgs_b200_session_init_metadata call per round against the
route without it (global init, session_create, destroy of the previous session), and the device time of one
auto-regressive pattern, serial (the parent build's fw_pattern_kernel, loaded from --serial-lib) against the wavefront.

    python scripts/bench_session_metadata.py --out profiles/r05_session_metadata_bench.json [--serial-lib PATH]

Workloads:
  afgs1_64x1080p  64 streams, 1920 x 1080 10-bit 4:2:0, AFGS1; each round every stream gets new metadata (new seed,
                  perturbed scaling points and AR coefficients of the golden AFGS1 configurations) and one frame
  sei_8x4k        8 streams, 3840 x 2160 10-bit 4:2:0, the default FGC SEI (8 frequency-filtering luma patterns)
Arms, alternated round by round in one process:
  (a) batched     one init_sessions call + one jobs call per round
  (b) recipe      per stream: global init_afgs1 / init_sei, session_create, destroy of its previous session; then the
                  jobs call
  (c) update      the batched call alone (updates/s over host time, and its device time from CUDA events)
  (d) jobs        the jobs call with unchanged metadata (the ceiling)
Every arm ends in a device synchronise; its time is host time over whole rounds."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tests.fixtures import load_golden, synth_frames  # noqa: E402

G = load_golden()


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


def perturbed_afgs1(raw: bytes, rng) -> bytes:
    a = Afgs1.from_buffer_copy(raw)
    a.grain_seed = int(rng.integers(0, 1 << 16))
    for k in range(a.num_y_points):  # scaling values move, points stay strictly increasing
        a.point_y_scaling[k] = int(np.clip(a.point_y_scaling[k] + rng.integers(-8, 9), 0, 255))
    n = 2 * a.ar_coeff_lag * (a.ar_coeff_lag + 1)
    for arr, m in ((a.ar_coeffs_y, n), (a.ar_coeffs_cb, n + 1), (a.ar_coeffs_cr, n + 1)):
        for k in range(m):
            arr[k] = int(np.clip(arr[k] + rng.integers(-3, 4), -128, 127))
    return bytes(a)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # noqa: BLE001
        return f"unknown ({e})"


def run_workload(hw, name, nstreams, w, h, cases, kind, rounds, rng):
    import torch
    from versatilefilmgrain_b200 import Job
    depth, fmt = 10, "420"

    def program_global(raw):
        hw.vfgs_set_depth(depth)
        hw.vfgs_set_chroma_subsampling(2, 2)
        (hw.init_afgs1 if kind == "afgs1" else hw.init_sei)(raw)
        if kind == "sei":
            hw.vfgs_set_seed(int(rng.integers(1, 1 << 31)))

    base = [G.struct(cases[k % len(cases)]) for k in range(nstreams)]
    # metadata of every round, made before any timing
    meta = [[perturbed_afgs1(b, rng) if kind == "afgs1" else b for b in base] for _ in range(rounds + 1)]
    hw.reset()
    sessions = []
    for k in range(nstreams):
        program_global(base[k])
        sessions.append(hw.create_session())
    frames = synth_frames(1, w, h, fmt, depth, seed=3)
    srcs = [torch.from_numpy(frames.view(np.int16)).cuda() for _ in range(nstreams)]  # the buffers of two jobs never overlap
    dsts = [torch.empty_like(srcs[0]) for _ in range(nstreams)]
    torch.cuda.synchronize()

    def jobs_call(sess):
        hw.add_grain_jobs_device([Job.packed(s, a, d, 1, w, h) for s, a, d in zip(sess, srcs, dsts)])

    def update(r):
        hw.init_sessions([(s, kind, m) for s, m in zip(sessions, meta[r])])
        if kind == "sei":
            for s in sessions:
                s.set_seed(int(rng.integers(1, 1 << 31)))

    recipe_sessions = list(sessions)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    times = {"a_batched": [], "b_recipe": [], "c_update": [], "c_update_device_ms": [], "d_jobs": []}
    for warm in (True, False):
        for r in range(2 if warm else rounds):
            # (a) one batched update + one jobs call
            t0 = time.perf_counter(); update(r); jobs_call(sessions); torch.cuda.synchronize()
            ta = time.perf_counter() - t0
            # (b) global init, session_create, destroy of the previous session, per stream; then the jobs call
            t0 = time.perf_counter()
            for k in range(nstreams):
                program_global(meta[r][k])
                new = hw.create_session()
                recipe_sessions[k].close() if recipe_sessions[k] is not sessions[k] else None
                recipe_sessions[k] = new
            jobs_call(recipe_sessions); torch.cuda.synchronize()
            tb = time.perf_counter() - t0
            # (c) the batched update alone, with its device time
            t0 = time.perf_counter(); ev0.record(); update(r + 1); ev1.record(); torch.cuda.synchronize()
            tc = time.perf_counter() - t0
            # (d) the jobs call with unchanged metadata
            t0 = time.perf_counter(); jobs_call(sessions); torch.cuda.synchronize()
            td = time.perf_counter() - t0
            if not warm:
                times["a_batched"].append(ta); times["b_recipe"].append(tb); times["c_update"].append(tc)
                times["c_update_device_ms"].append(ev0.elapsed_time(ev1)); times["d_jobs"].append(td)
    for s in recipe_sessions:
        if s not in sessions:
            s.close()
    for s in sessions:
        s.close()
    med = {k: float(np.median(v)) for k, v in times.items()}
    out = {
        "workload": name, "streams": nstreams, "width": w, "height": h, "depth": depth, "format": fmt, "metadata": kind,
        "rounds": rounds,
        "median_round_s": {k: v for k, v in med.items() if k != "c_update_device_ms"},
        "update_device_ms_median": med["c_update_device_ms"],
        "a_batched_frames_per_s": nstreams / med["a_batched"],
        "b_recipe_frames_per_s": nstreams / med["b_recipe"],
        "c_updates_per_s_host": nstreams / med["c_update"],
        "c_updates_per_s_device": nstreams / (med["c_update_device_ms"] / 1e3),
        "d_jobs_frames_per_s": nstreams / med["d_jobs"],
    }
    out["ratio_a_over_b"] = out["a_batched_frames_per_s"] / out["b_recipe_frames_per_s"]
    out["ratio_a_over_d"] = out["a_batched_frames_per_s"] / out["d_jobs_frames_per_s"]
    return out


def ar_pattern_times(serial_lib: str | None, iters: int):
    """Device time of fw_pattern_kernel per AR pattern (luma 64 x 64: first job of an AFGS1 configuration; chroma
    32 x 32: the other two), from torch.profiler, for this build and, if given, the serial build."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from versatilefilmgrain_b200 import VfgsHw
    case = next(c for c in G.runnable() if G.cases[c]["afgs1"] and G.cases[c]["depth"] == 10 and G.cases[c]["fmt"] == "420")
    raw = G.struct(case)
    libs = [("wavefront", None)] + ([("serial", serial_lib)] if serial_lib else [])
    res = {}
    for label, path in libs:
        if path:
            L = C.CDLL(path)
            L.vfgs_b200_init.argtypes = [C.c_int]
            L.vfgs_set_depth.argtypes = [C.c_int]
            L.vfgs_set_chroma_subsampling.argtypes = [C.c_int, C.c_int]
            L.vfgs_b200_init_afgs1.argtypes = [C.c_void_p]
            assert L.vfgs_b200_init(0) == 0
            buf = (C.c_uint8 * len(raw)).from_buffer_copy(raw)

            def init():
                L.vfgs_set_depth(10); L.vfgs_set_chroma_subsampling(2, 2)
                assert L.vfgs_b200_init_afgs1(buf) == 0
        else:
            hw = VfgsHw(device=0)

            def init():
                hw.vfgs_set_depth(10); hw.vfgs_set_chroma_subsampling(2, 2); hw.init_afgs1(raw)
        for _ in range(3):
            init()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(iters):
                init()
            torch.cuda.synchronize()
        durs = [e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
                for e in prof.events() if "fw_pattern_kernel" in e.name]
        durs = [d for d in durs if d > 0]
        if len(durs) < 3 * iters:
            res[label] = {"error": f"{len(durs)} kernel records for {3 * iters} launches"}
            continue
        durs = np.array(durs[-3 * iters:], dtype=float).reshape(iters, 3)
        res[label] = {"luma_64_us_median": float(np.median(durs[:, 0])), "chroma_32_us_median": float(np.median(durs[:, 1:])),
                      "launches": int(durs.size)}
    if "serial" in res and "error" not in res["serial"] and "error" not in res["wavefront"]:
        res["serial_over_wavefront_luma"] = res["serial"]["luma_64_us_median"] / res["wavefront"]["luma_64_us_median"]
        res["serial_over_wavefront_chroma"] = res["serial"]["chroma_32_us_median"] / res["wavefront"]["chroma_32_us_median"]
    elif "serial" not in res:
        res["serial"] = "not measured"
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="")
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--serial-lib", default="", help="a parent build of libvfgs_b200.so (serial AR filter)")
    ap.add_argument("--ar-iters", type=int, default=50)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this benchmark measures the GPU"
    from versatilefilmgrain_b200 import VfgsHw
    hw = VfgsHw(device=0)
    rng = np.random.default_rng(1)
    afgs1 = [c for c in G.runnable() if G.cases[c]["afgs1"] and G.cases[c]["depth"] == 10 and G.cases[c]["fmt"] == "420"]
    result = {"card": card(), "torch_device": torch.cuda.get_device_name(0), "workloads": []}
    result["workloads"].append(run_workload(hw, "afgs1_64x1080p", 64, 1920, 1080, afgs1, "afgs1", args.rounds, rng))
    result["workloads"].append(run_workload(hw, "sei_8x4k", 8, 3840, 2160, ["builtin_default|d10|420|g100"], "sei", args.rounds, rng))
    result["ar_pattern_device_time"] = ar_pattern_times(args.serial_lib or None, args.ar_iters)
    result["card_after"] = card()
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
