#!/usr/bin/env python
"""bench.py -- throughput of the VFGS hardware-layer hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

One "step" is one batch of synthetic frames of the workload's size through the hot path (default: the
BASELINE.json headline, 3840x2160 10-bit 4:2:0): PASSES calls of the C-ABI device entry point, each over
a resident pool of distinct frames several GB large (inputs larger than L2, so every call streams from and
to HBM), with the frame index -- hence the LFSR state -- running on from call to call. PASSES is sized so
that a step moves ~400 GB (about 65 ms on one B200): the default 20 steps time more than a second.

  --total-frames T   strong scaling (BASELINE.json configs[4]: --workload 8k420_ff_test1 --total-frames 2400):
             a step is the WHOLE job of T frames; rank r owns the contiguous shard shard_range(T, r, N), jumps
             to its first frame (vfgs_b200_skip_frames) and cycles its resident pool while the frame index
             runs over the shard. "scaling": "strong".

  value      frames/s, device-resident (inputs already in HBM), CUDA events on the launching stream,
             max over ranks; whole job over all N GPUs
  e2e        same metric through the host entry point of the C-ABI (pinned host buffers; H2D, kernels
             and D2H inside the timed region)
  roofline   grain kernel alone: algorithmic bytes (samples x (bytes in + bytes out)) / its average
             launch duration (CUDA events around each launch), against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the reference's own CPU implementation (oracle/_ref, unmodified sources compiled with
             gcc -O3 -mavx2) on this host's cores, on a bounded sample of the same workload
  --impl reference  times that CPU implementation instead of the CUDA path (rank 0 only)

Multi-GPU: one process per GPU (torchrun). Frames are sharded: every rank owns a contiguous run of
each call's global batch (weak scaling, default) or of the whole job (--total-frames) and derives its LFSR
start state by jump-ahead; there is no collective on the data path (NCCL is used only for the barrier and
the max-over-ranks of the timings). Before anything is timed every rank reproduces reference digests at
NON-ZERO frame offsets (tests/golden "shards": groups g = rank, rank + N, ... of the reference's
continuous run), so a wrong shard start cannot go unnoticed.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "4k_10bit_420_frames_per_sec_device_resident"
UNIT = "frames/s"

# name -> (golden case, width, height, fmt, depth, out_depth)
WORKLOADS = {
    "4k420_afgs1_10to10": ("fgs_afgs1_test1.cfg|d10|420|g100", 3840, 2160, "420", 10, 0),
    "4k420_afgs1_10to8": ("fgs_afgs1_test1.cfg|d10|420|g100", 3840, 2160, "420", 10, 8),
    "4k420_afgs1_8to8": ("fgs_afgs1_test1.cfg|d8|420|g100", 3840, 2160, "420", 8, 0),
    "1366x768_ragged": ("fgs_afgs1_test1.cfg|d10|420|g100", 1366, 768, "420", 10, 0),  # rows not 16-byte aligned: general kernel
    "4k420_sei_default": ("fgs_sei.cfg|d10|420|g100", 3840, 2160, "420", 10, 0),
    "4k420_ff_test5": ("fgs_sei_ff_test5.cfg|d10|420|g100", 3840, 2160, "420", 10, 0),
    "1080p420_ff_test1": ("fgs_sei_ff_test1.cfg|d10|420|g100", 1920, 1080, "420", 10, 0),
    "1080p420_ar_test1": ("fgs_sei_ar_test1.cfg|d10|420|g100", 1920, 1080, "420", 10, 0),
    "4k422_ff_test4_gain150": ("fgs_sei_ff_test4.cfg|d10|422|g150", 3840, 2160, "422", 10, 0),
    "4k444_ff_test4_gain150": ("fgs_sei_ff_test4.cfg|d10|444|g150", 3840, 2160, "444", 10, 0),
    "8k420_ff_test1": ("fgs_sei_ff_test1.cfg|d10|420|g100", 7680, 4320, "420", 10, 0),
}
DEFAULT_WORKLOAD = "4k420_afgs1_10to10"
POOL_INPUT_BYTES = 6.4e9  # per GPU; x2 with the output pool, far above the 126 MB L2


def frame_geometry(w, h, fmt, depth, out_depth):
    sx, sy = {"420": (2, 2), "422": (2, 1), "444": (1, 1)}[fmt]
    samples = w * h + 2 * (w // sx) * (h // sy)
    isz = 2 if depth > 8 else 1
    osz = 2 if (out_depth or depth) > 8 else 1
    return samples, samples * isz, samples * osz


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """Polls SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4}

    def __init__(self, index: int, period_s: float = 0.004):
        super().__init__(daemon=True)
        self.index, self.period, self.stop_flag = index, period_s, threading.Event()
        self.sm, self.reasons, self.max_mhz, self.err = [], 0, None, None
        self.nvml = self.handle = None
        try:  # NVML is initialised here, before the timed region, so that the thread samples from its first instant
            import pynvml
            pynvml.nvmlInit()
            self.nvml, self.handle = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception as e:  # NVML missing: report it, do not invent numbers
            self.err = repr(e)

    def run(self):
        if self.handle is None:
            return
        pynvml, h = self.nvml, self.handle
        try:
            while not self.stop_flag.is_set():
                self.sm.append(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                try:
                    self.reasons |= int(pynvml.nvmlDeviceGetCurrentClocksEventReasons(h))
                except Exception:
                    self.reasons |= int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                time.sleep(self.period)
        except Exception as e:  # NVML missing: report it, do not invent numbers
            self.err = repr(e)

    def result(self):
        self.stop_flag.set()
        self.join(timeout=2)
        names = [n for n, bit in {**self.BAD, **self.NOTE}.items() if self.reasons & bit]
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
               "reasons": names, "samples": len(self.sm)}
        if self.err:
            out["error"] = self.err
        return out


# ------------------------------------------------------------------------------------- CPU arm
_W = {}


def _cpu_worker_init(case, w, h, fmt, depth, out_depth, frames_per_worker, use_ref):
    from oracle import pyoracle
    from tests.fixtures import load_golden
    G = load_golden()
    hw = pyoracle.Reference() if use_ref else pyoracle.Oracle()
    st = G.state(case)
    pyoracle.program_hw_from_state(hw, st)
    rng = np.random.default_rng(os.getpid())
    samples, _, _ = frame_geometry(w, h, fmt, depth, out_depth)
    maxv = (1 << depth) - 1
    data = rng.integers(0, maxv + 1, size=frames_per_worker * samples, dtype=np.uint16 if depth > 8 else np.uint8)
    _W.update(hw=hw, st=st, data=data, work=data.copy(), n=frames_per_worker, w=w, h=h, fmt=fmt, depth=depth,
              od=out_depth, use_ref=use_ref, out8=np.empty(data.size, dtype=np.uint8))


def _cpu_worker_step(_):
    from oracle import pyoracle
    from oracle.pyoracle import _ptr
    W = _W
    np.copyto(W["work"], W["data"])
    _, _, cw, ch = pyoracle.frame_samples(W["w"], W["h"], W["fmt"])
    t0 = time.perf_counter()
    if W["use_ref"]:
        # the reference's own line walk (vfgs_main.c:664-682 -> vfgs_hw.c:288) and yuv_to_8bit
        W["hw"].L.refh_add_grain_frames_packed(_ptr(W["work"]), W["n"], W["w"], W["h"], cw, ch, W["depth"])
        if W["od"] == 8 and W["depth"] == 10:
            W["hw"].L.refh_to_8bit_packed(_ptr(W["out8"]), _ptr(W["work"]), W["n"], W["w"], W["h"], cw, ch)
    else:
        W["hw"].add_grain_frames(W["work"], W["n"], W["w"], W["h"], W["od"])
    return time.perf_counter() - t0


class CpuArm:
    """The reference CPU implementation on all host cores: one forked process per core (the reference
    keeps its state in file-scope statics and is single-threaded), each on its own frames."""

    def __init__(self, workload, frames_per_worker):
        import multiprocessing as mp
        from oracle import pyoracle
        pyoracle.build()
        self.use_ref = pyoracle.have_reference()
        try:
            self.cores = len(os.sched_getaffinity(0))
        except Exception:
            self.cores = os.cpu_count() or 1
        case, w, h, fmt, depth, od = WORKLOADS[workload]
        self.fpw = frames_per_worker
        self.pool = mp.get_context("fork").Pool(self.cores, _cpu_worker_init, (case, w, h, fmt, depth, od, frames_per_worker, self.use_ref))

    def step(self):
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker_step, range(self.cores), chunksize=1)
        return time.perf_counter() - t0

    def step_one_core(self):
        """The same work on a single worker while the others idle: the reference as it ships (one thread)."""
        t0 = time.perf_counter()
        self.pool.map(_cpu_worker_step, range(1), chunksize=1)
        return time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()

    @property
    def kind(self):
        return "reference" if self.use_ref else "port"

    def describe(self):
        what = "oracle/_ref (unmodified reference, gcc -O3 -mavx2, asserts on)" if self.use_ref else "oracle port (oracle/vfgs_oracle.c)"
        return f"{what}; {self.cores} forked workers x {self.fpw} frames per step, in-memory frames, file I/O excluded"


def cpu_frames_per_worker(w, h):
    return max(1, int(round(6 * (3840 * 2160) / (w * h))))  # ~0.5 s of work per worker per step


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    case, w, h, fmt, depth, od = WORKLOADS[args.workload]
    fpw = cpu_frames_per_worker(w, h)
    arm = CpuArm(args.workload, fpw)
    for _ in range(args.warmup):
        arm.step()
    t = [arm.step() for _ in range(args.steps)]
    arm.close()
    total = sum(t)
    frames = arm.cores * fpw * args.steps
    value = frames / total
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic", "impl": "reference",
        "config": workload_config(args.workload), "frames_per_step": arm.cores * fpw,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.describe()},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_config(name):
    """Identical in both arms (the driver compares the dicts); per-arm quantities are top-level keys of the line."""
    case, w, h, fmt, depth, od = WORKLOADS[name]
    return {"workload": f"{w}x{h} {depth}-bit {fmt[0]}:{fmt[1]}:{fmt[2]} -> {od or depth}-bit, grain config {case.split('|')[0]}"
                        f"{' gain ' + case.split('|g')[1] if not case.endswith('g100') else ''}, uniform random samples",
            "name": name,
            "l2": "inputs larger than L2: every call streams a resident pool of distinct frames (GBs, >> 126 MB L2) once"}


# ------------------------------------------------------------------------------------- CUDA arm
def bind_to_gpu_numa_node(index: int):
    """Pin this process to the CPUs NVML reports as local to GPU `index` (same NUMA node / PCIe root), so
    that the page-locked staging buffers it allocates afterwards are local too: with several ranks on one
    host the H2D/D2H copies otherwise cross the socket interconnect. Returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        allowed = os.sched_getaffinity(0)
        cpus = (cpus & allowed) or allowed
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} cpus local to gpu {index}"
    except Exception as e:  # affinity is an optimisation, never a requirement
        return f"not bound ({type(e).__name__})"


def parity_gate(hw, G, case, fmt, depth, od, rank, world):
    """Before anything is timed: the workload's grain configuration on golden inputs must reproduce the digests
    the unmodified reference produced (tests/golden/golden.npz). Every rank does the plain golden cases and, from
    the reference's continuous multi-group run ("shards"), the groups g = rank, rank + world, ...: each of those
    starts at a non-zero frame offset reached by jump-ahead, which is exactly what a shard start is.
    Returns (checks done, error text or None)."""
    import torch
    from tests.fixtures import parse_output_key, program_case, sha, synth_frames
    from versatilefilmgrain_b200.sharding import position_shard
    meta = G.cases[case]
    epoch = [int(v) for v in G.state(case)["lfsr"]]

    def run(frames, n, w, h, first):
        hw.reset()
        program_case(hw, G, case)
        position_shard(hw, epoch, first, w, h)
        d_s = torch.from_numpy(frames.view(np.int16) if depth > 8 else frames).cuda()
        d_o = torch.zeros(frames.size, dtype=torch.int16 if (od or depth) > 8 else torch.uint8, device="cuda")
        hw.add_grain_frames_device(d_s, d_o, n, w, h, od)
        torch.cuda.synchronize()
        got = d_o.cpu().numpy()
        return got.view(np.uint16) if (od or depth) > 8 else got

    done = 0
    for key, want in meta["outputs"].items():
        gw, gh, gn, gseed, god = parse_output_key(key)
        if god != od:
            continue
        got = run(synth_frames(gn, gw, gh, fmt, depth, seed=gseed), gn, gw, gh, 0)
        if sha(got) != want["sha256"] or hw.get_lfsr() != want["lfsr_after"]:
            return done, f"golden {key}: CUDA output differs from the reference digest"
        done += 1
    for key, groups in meta["shards"].items():
        gw, gh, gn, gseed, god = parse_output_key(key)
        if god != od:
            continue
        frames = synth_frames(gn, gw, gh, fmt, depth, seed=gseed)
        for g in range(rank % len(groups), len(groups), world):
            got = run(frames, gn, gw, gh, g * gn)
            if sha(got) != groups[g]["sha256"] or hw.get_lfsr() != groups[g]["lfsr_after"]:
                return done, f"shard start at frame {g * gn} of {key}: CUDA output differs from the reference digest"
            done += 1
    return done, None


DUMP_SAMPLES = 1 << 22  # output samples written by --dump-outputs over all ranks: 16 MB of values + 32 MB of indices


def dump_outputs(out_dir, dst, hw, rank=0, world=1):
    """What the last timed step left in the output pool, for comparing two builds on the same inputs: a fixed,
    seeded sample of the output samples (all of them if the pool is smaller) as float32, their flat indices into the
    pool as float64, and the four LFSR registers the next call would start from. With several ranks each writes its
    share of the sample, so the files stay within the same total size."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if world == 1 else f"_rank{rank}"
    n, k = dst.numel(), DUMP_SAMPLES // world
    if n <= k:
        idx = np.arange(n, dtype=np.int64)
    else:
        idx = np.unique(np.random.default_rng(2024 + rank).integers(0, n, size=k, dtype=np.int64))
    vals = dst.index_select(0, torch.from_numpy(idx).to(dst.device)).cpu().numpy()
    if vals.dtype == np.int16:
        vals = vals.view(np.uint16)  # 10-bit codes travel as int16 tensors
    np.save(os.path.join(out_dir, f"output_sample{suffix}.npy"), vals.astype(np.float32))
    np.save(os.path.join(out_dir, f"output_sample_index{suffix}.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, f"lfsr_after{suffix}.npy"), np.array(hw.get_lfsr(), dtype=np.float64))


def run_b200_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus > 1 and world == 1:
        # not under torchrun: re-launch ourselves the way the driver does
        import subprocess
        port = 29500 + (os.getpid() % 2000)
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    case, w, h, fmt, depth, od = WORKLOADS[args.workload]
    cpu_baseline = None
    if rank == 0 and not args.no_cpu_baseline:
        # timed first, before this process creates a CUDA context (the workers are forked); with several ranks the
        # others wait in init_process_group meanwhile
        fpw = cpu_frames_per_worker(w, h)
        arm = CpuArm(args.workload, fpw)
        arm.step()
        tt = [arm.step() for _ in range(3)]
        t1 = arm.step_one_core()
        arm.close()
        cpu_baseline = {"value": arm.cores * fpw * len(tt) / sum(tt), "unit": UNIT, "cores": arm.cores, "kind": arm.kind,
                        "sample": arm.describe() + f"; {len(tt)} timed steps after 1 warm-up",
                        "one_core": {"value": fpw / t1, "unit": UNIT, "what": "one worker alone (the reference is single-threaded), 1 step"}}

    placement = bind_to_gpu_numa_node(local) if world > 1 else "single rank, not bound"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from tests.fixtures import load_golden, program_case  # nothing from oracle/ here
    from versatilefilmgrain_b200 import VfgsHw
    from versatilefilmgrain_b200.sharding import position_shard, shard_range

    samples, in_bytes, out_bytes = frame_geometry(w, h, fmt, depth, od)
    G = load_golden()
    hw = VfgsHw(device=local)

    checks, err = (0, None) if args.skip_parity_gate else parity_gate(hw, G, case, fmt, depth, od, rank, world)
    bad = torch.tensor([1 if err else 0], dtype=torch.int32, device="cuda")
    if world > 1:
        dist.all_reduce(bad, op=dist.ReduceOp.MAX)
    if err:
        print(json.dumps({"error": "parity gate failed: " + err, "workload": args.workload, "rank": rank}), flush=True)
    if int(bad.item()):
        return 2
    hw.reset()
    st = program_case(hw, G, case)
    epoch = [int(v) for v in st["lfsr"]]

    # resident pool of distinct frames (uniform random codes: worst case for the LUT/pattern gathers)
    F = args.frames_per_step or int(max(8, min(4096, POOL_INPUT_BYTES // in_bytes)))
    strong = args.total_frames > 0
    if strong:
        my_first, my_count = shard_range(args.total_frames, rank, world)
        F = max(1, min(F, (args.total_frames + world - 1) // world))
        passes = None
    else:
        # calls per step: ~400 GB of algorithmic traffic per step and GPU, so that 20 steps time > 1 s
        passes = args.passes or max(1, int(round(4.0e11 / (F * (in_bytes + out_bytes)))))
    gen = torch.Generator(device="cuda"); gen.manual_seed(1234 + rank)
    sdt = torch.int16 if depth > 8 else torch.uint8
    if args.data == "uniform":
        src = torch.randint(0, 1 << depth, (F * samples,), dtype=sdt, device="cuda", generator=gen)
    else:
        # "natural": smooth horizontal gradient inside the legal range + small noise, so neighbouring samples
        # mostly share LUT entries and pattern slots (best case for the gathers); generated frame by frame
        src = torch.empty(F * samples, dtype=sdt, device="cuda")
        lo, hi = 16 << (depth - 8), 235 << (depth - 8)
        for f in range(F):
            idx = torch.arange(samples, device="cuda", dtype=torch.float32)
            base = lo + (hi - lo) * (0.5 + 0.45 * torch.sin(idx * (6.2831853 / w) + f * 0.37))
            noise = torch.randint(-3, 4, (samples,), device="cuda", generator=gen)
            src[f * samples:(f + 1) * samples] = (base.to(torch.int32) + noise).clamp_(0, (1 << depth) - 1).to(sdt)
        del idx, base, noise
    ddt = torch.int16 if (od or depth) > 8 else torch.uint8
    if args.in_place and ddt == sdt:
        dst = src  # diagnostic: the reference CLI's own mode (vfgs_main.c:664-682 adds grain in place)
    else:
        # --dst-offset (diagnostic): shifts the output pool relative to the input pool by a multiple of 256 bytes
        pad = args.dst_offset // (2 if ddt == torch.int16 else 1)
        dst = torch.empty(F * samples + pad, dtype=ddt, device="cuda")[pad:]
    stream = torch.cuda.current_stream()

    def step(s):
        if strong:
            # the whole job: this rank's contiguous shard, the pool cycled while the frame index runs over the shard
            done = 0
            while done < my_count:
                n = min(F, my_count - done)
                position_shard(hw, epoch, my_first + done, w, h)
                hw.add_grain_frames_device(src, dst, n, w, h, od, stream)
                done += n
        else:
            # call p of step s: rank r owns frames [r*F, (r+1)*F) of that call's global batch of world*F frames
            for p in range(passes):
                position_shard(hw, epoch, ((s * passes + p) * world + rank) * F, w, h)
                hw.add_grain_frames_device(src, dst, F, w, h, od, stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for s in range(args.warmup):
        step(s)
    barrier()
    sampler = ClockSampler(local); sampler.start()
    hw.kernel_timing(True)
    launches0 = hw.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for s in range(args.steps):
        step(args.warmup + s)
    e1.record(stream)
    barrier()
    clocks = sampler.result()
    if args.dump_outputs:
        # before the copy below overwrites the output pool
        dump_outputs(args.dump_outputs, dst, hw, rank, world)
    ms = e0.elapsed_time(e1)
    k_ms, k_n = hw.kernel_time()
    hw.kernel_timing(False)
    gpu_launches = hw.launch_count() - launches0
    t = torch.tensor([ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    frames_per_step = args.total_frames if strong else world * F * passes  # whole job, all ranks
    my_frames_per_step = my_count if strong else F * passes
    value = frames_per_step * args.steps / (ms_max * 1e-3)

    # What a plain device-to-device copy sustains on this GPU over the same kind of region (about a second, same pools,
    # clocks sampled): MEASURED_PEAKS.json's hbm_gbs is a best-of-10 burst figure, and over a second the power cap pulls
    # the SM clock down (reported next to the roofline; `frac` stays achieved / MEASURED_PEAKS as the contract says).
    sustained = None
    if not args.no_sustained_copy and src.data_ptr() != dst.data_ptr():
        a8, b8 = src.view(torch.uint8), dst.view(torch.uint8)
        nbytes = min(a8.numel(), b8.numel())
        a8, b8 = a8[:nbytes], b8[:nbytes]
        for _ in range(3):
            b8.copy_(a8)
        reps = max(4, int(1.0 * 6.0e12 / (2 * nbytes)))
        barrier()
        cs = ClockSampler(local); cs.start()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(reps):
            b8.copy_(a8)
        c1.record(stream)
        torch.cuda.synchronize()
        ck = cs.result()
        cms = c0.elapsed_time(c1)
        sustained = {"gbs": 2 * nbytes * reps / (cms * 1e-3) / 1e9, "seconds": cms * 1e-3, "what": "torch copy_ (cudaMemcpy D2D) of the input pool onto the output pool, read + write bytes",
                     "sm_mhz": ck["sm_mhz"], "reasons": ck["reasons"]}

    # ---- end to end through the host entry point: pinned host buffers, H2D + kernels + D2H timed -------------------
    Fe = min(F, args.e2e_frames or int(max(8, min(128, 2.4e9 // in_bytes))))
    if world > 1 and not args.e2e_frames:
        Fe = max(8, Fe * 2 // 3)  # several ranks pin their buffers on one host: keep the total below what one rank used to take times N
    e2e_steps = max(3, min(args.steps, 20))
    # The GPUs of one box do not sit behind equally fast host links (profiles/r02_pcie_matrix.json: with all eight busy,
    # four of them get 8.5 GB/s each way, four 11.5), so with several ranks the step's world * Fe frames are dealt out in
    # proportion to the copy rate every rank measures here, with all ranks copying at once: this step's H2D and D2H
    # copies alone, concurrently on two streams from pinned buffers, no kernels. Summed over the ranks it is also the
    # box's PCIe ceiling for the step (`pcie_copies_alone`).
    cap = Fe if world == 1 else int(Fe * 1.35) + 1  # frames a rank may be dealt
    h_in = torch.empty(cap * samples, dtype=src.dtype).pin_memory()
    h_in[: Fe * samples].copy_(src[: Fe * samples])
    if cap > Fe:
        h_in[Fe * samples:].copy_(src[: (cap - Fe) * samples])
    h_out = torch.empty(cap * samples, dtype=dst.dtype).pin_memory()
    del src, dst
    torch.cuda.empty_cache()
    d_in, d_out = torch.empty(Fe * samples, dtype=h_in.dtype, device="cuda"), torch.empty(Fe * samples, dtype=h_out.dtype, device="cuda")
    s_up, s_down = torch.cuda.Stream(), torch.cuda.Stream()

    def copies():
        with torch.cuda.stream(s_up):
            d_in.copy_(h_in[: Fe * samples], non_blocking=True)
        with torch.cuda.stream(s_down):
            h_out[: Fe * samples].copy_(d_out, non_blocking=True)

    copies()
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        copies()
    torch.cuda.synchronize()
    my_copy_s = time.perf_counter() - t0
    t = torch.tensor([my_copy_s], dtype=torch.float64, device="cuda")
    rates = torch.zeros(world, dtype=torch.float64, device="cuda")
    rates[rank] = Fe * e2e_steps / my_copy_s
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(rates, op=dist.ReduceOp.SUM)
    copy_only_value = world * Fe * e2e_steps / float(t.item())
    del d_in, d_out
    from versatilefilmgrain_b200.sharding import weighted_shard_ranges
    shards = weighted_shard_ranges(world * Fe, [min(float(r), 1.35 * float(rates.min().item())) for r in rates.tolist()]) if world > 1 else [(0, Fe)]
    my_e2e_first, my_e2e = shards[rank]
    my_e2e = min(my_e2e, cap)

    def e2e_step(s):
        position_shard(hw, epoch, s * world * Fe + my_e2e_first, w, h)
        hw.add_grain_frames_host(h_in, h_out, my_e2e, w, h, od)

    for s in range(2):
        e2e_step(s)
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        e2e_step(2 + s)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    t = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = sum(c for _, c in shards) * e2e_steps / float(t.item())

    peak, peak_src = measured_peak_gbs()
    # the grain kernels of one C-ABI call (one launch for single-pattern configs, two when components split between
    # the fast and the gather kernel) move the call's algorithmic bytes: bytes of all calls / their summed device time
    my_algo_bytes = my_frames_per_step * args.steps * (in_bytes + out_bytes)
    achieved = my_algo_bytes / (k_ms * 1e-3) / 1e9 if k_n else None
    calls_per_step = (k_n / max(args.steps, 1)) / max(1, len(hw.last_launch()["kernels"]))
    frames_per_call = my_frames_per_step / max(calls_per_step, 1e-9)
    traffic = traffic_src = None
    try:  # DRAM bytes per frame of the grain kernel from the committed ncu capture of this workload
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f).get(args.workload) or {}
        if tj.get("dram_bytes_per_frame") and args.data == "uniform":
            traffic = tj["dram_bytes_per_frame"] * frames_per_call
            traffic_src = (f"{tj['source']}: dram__bytes_read.sum + dram__bytes_write.sum per frame of that capture, "
                           f"scaled to the {frames_per_call:.0f} frames of one call here")
    except Exception:
        pass
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic" if args.data == "uniform" else "synthetic (smooth gradient + noise)",
        "config": workload_config(args.workload),
        "frames_per_step": frames_per_step, "frames_per_call_per_gpu": frames_per_call,
        "pool_gb_per_gpu": F * (in_bytes + out_bytes) / 1e9,
        "timed_region_s": ms_max * 1e-3,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": sum(c for _, c in shards) * in_bytes, "d2h_bytes_per_step": sum(c for _, c in shards) * out_bytes,
                "frames_per_step": sum(c for _, c in shards), "frames_per_rank": [c for _, c in shards],
                "shards": "one step = world x %d frames, dealt to the ranks in proportion to the copy rate each measured with all ranks copying" % Fe if world > 1 else "single rank",
                "steps": e2e_steps, "host_buffers": "pinned", "cpu_placement": placement, "scaling": "weak",
                "gbs_each_way": [e2e_value * in_bytes / 1e9, e2e_value * out_bytes / 1e9],
                "pcie_copies_alone": {"value": copy_only_value, "unit": UNIT,
                                      "what": "the same H2D and D2H copies without kernels, concurrently, all ranks: the box's PCIe ceiling for this step"}},
        "gpu_launches": int(gpu_launches),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": (achieved / peak) if achieved else None, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "kernel": "+".join(hw.last_launch()["kernels"]), "launches_per_step": k_n / max(args.steps, 1),
                     "bytes_per_launch": frames_per_call * (in_bytes + out_bytes),
                     "avg_launch_ms": (k_ms / max(calls_per_step * args.steps, 1e-9)) if k_n else None,
                     "kernel_share_of_step": (k_ms / ms) if ms else None,
                     "frac_of_nominal_8TBs": (achieved / 8000.0) if achieved else None,
                     "sustained_copy": sustained,
                     "frac_of_sustained_copy": (achieved / sustained["gbs"]) if (achieved and sustained) else None},
        "bytes_per_frame": in_bytes + out_bytes,
        "device_resident_gbs": value * (in_bytes + out_bytes) / 1e9,
        "parity": ("SKIPPED (--skip-parity-gate: profiling / experiment run, not a bench value)" if args.skip_parity_gate else
                   f"{checks} golden digests of the unmodified reference reproduced on every rank before timing, "
                   f"incl. shard starts at non-zero frame offsets (tests/golden)"),
    }
    if strong:
        line["total_frames"] = args.total_frames
        line["shard"] = {"first": my_first, "count": my_count, "of_rank": rank}

    if cpu_baseline is not None:
        line["cpu_baseline"] = cpu_baseline
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    ap.add_argument("--frames-per-step", type=int, default=0, help="frames of the resident pool = frames per C-ABI call (default: 6.4 GB of input)")
    ap.add_argument("--passes", type=int, default=0, help="C-ABI calls per step (default: ~400 GB of traffic per step)")
    ap.add_argument("--total-frames", type=int, default=0, help="strong scaling: a step is this whole job, sharded over the ranks")
    ap.add_argument("--e2e-frames", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sustained-copy", action="store_true", help="skip the one-second device-to-device copy measured for comparison")
    ap.add_argument("--skip-parity-gate", action="store_true", help="diagnostic (ncu captures, experiments with deliberately wrong build knobs): the line says so")
    ap.add_argument("--dst-offset", type=int, default=0, help="diagnostic: extra bytes (multiple of 256) in front of the output pool")
    ap.add_argument("--in-place", action="store_true", help="diagnostic: output written over the input (same depth only)")
    ap.add_argument("--data", default="uniform", choices=["uniform", "natural"],
                    help="sample distribution of the synthetic frames (uniform random codes = worst case for the LUT/pattern gathers)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write a seeded sample of the last step's output frames and the LFSR "
                         "registers as DIR/*.npy (CUDA path only)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    sys.exit(run_reference_arm(args) if args.impl == "reference" else run_b200_arm(args))


if __name__ == "__main__":
    main()
