"""The device entry point at the scale bench.py times it, against the oracle, bit for bit.

bench.py's calls are one C-ABI call over a resident pool of several GB (input offsets past 2^32 bytes), every warp
of the persistent grain kernels runs hundreds of warp-tasks across row, component and frame boundaries, and the LFSR
starts more than 2^32 steps from the epoch. The parity tests use small batches, where no warp runs more than a few
tasks. Here every frame of such calls is checked: chunks of the output are copied to the host and compared with the
oracle on a thread pool (one Oracle per worker; ctypes releases the GIL), and the LFSR registers afterwards with the
oracle's. Each case skips, naming the shortfall, where the device has less free memory than it needs. Run with
-m gpu on a B200."""
import concurrent.futures as cf
import ctypes as C
import os
import threading

import numpy as np
import pytest

import bench
from oracle.pyoracle import RefState
from tests.util import (Oracle, bench_call, build_emu, first_mismatch, load_golden, program_case, program_hw_from_state,
                        program_random_state)
from versatilefilmgrain_b200.sharding import position_shard, steps_per_frame

pytestmark = pytest.mark.gpu

G = load_golden()
GUARD_BYTES = 1 << 20            # sentinel bands on each side of every output pool
CHUNK_BYTES = 48 << 20           # input bytes per oracle chunk
KERNEL_NAMES = {0: "fgs_apply_fast_kernel", 3: "fgs_apply_fast_kernel<EDGE>", 1: "fgs_apply_gather_kernel", 2: "fgs_apply_kernel"}
LAUNCH_ORDER = (0, 3, 1, 2)      # the order in which one call launches its grain kernels (run_frames_device)
TPF_INDEX = {0: 19, 3: 20, 1: 21, 2: 22}  # emu_plan: warp-tasks per frame of each launch


@pytest.fixture(scope="module")
def hw():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from versatilefilmgrain_b200 import VfgsHw
    h = VfgsHw(device=0)
    Oracle().lfsr_jump(1, 1)  # builds the oracle's jump table before worker threads share it
    yield h
    h.force_general_kernel(0)


@pytest.fixture(scope="module")
def emu():
    L = C.CDLL(build_emu())
    L.emu_plan.argtypes = [C.c_void_p] + [C.c_int] * 5 + [C.c_void_p]
    return L


WORKERS = max(1, min(16, os.cpu_count() or 1))


@pytest.fixture(scope="module")
def pool():
    with cf.ThreadPoolExecutor(max_workers=WORKERS) as ex:
        yield ex


# ------------------------------------------------------------------------------------------------ helpers
def need_device_memory(nbytes):
    import torch
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 1e9:.1f} GB of free device memory, {free / 1e9:.1f} GB free "
                    f"({(nbytes - free) / 1e9:.1f} GB short)")


def plan(emu, setup, w, h, od=0, in_place=False, mode=0):
    """The host planner's view of a packed call (tests/emu): per component the kernel kind and lane units per stripe
    row of the kernel that serves it (0 for the general kernel, which numbers its tasks by segments), and warp-tasks
    per frame of every launch."""
    o = Oracle(); setup(o)
    st = RefState(); o.L.oracle_get_state(o.h, C.byref(st))
    out = np.zeros(32, dtype=np.int32)
    emu.emu_plan(C.byref(st), w, h, od, 1 if in_place else 0, mode, out.ctypes.data_as(C.c_void_p))
    kinds = [int(k) for k in out[0:3]]
    units = [int(out[{0: 14, 3: 25, 1: 28}[k] + c]) if k != 2 else 0 for c, k in enumerate(kinds)]
    return {"kind": kinds, "units": units, "tasks_per_frame": {k: int(out[TPF_INDEX[k]]) for k in set(kinds)},
            "gather_fold": int(out[23]), "gather_shift": int(out[24])}


def assert_regime(hw, p, nframes, min_last, min_other):
    """The kernels the call launched are the ones the planner predicts, and the warps of the persistent grids ran many
    warp-tasks each: at least `min_last` in the call's last launch, whose grid and block are recorded, and at least
    `min_other` in any earlier launch of the call, counted against the most warps the device can hold at once."""
    import torch
    ll = hw.last_launch()
    assert sorted(ll["kernels"]) == sorted(KERNEL_NAMES[k] for k in set(p["kind"])), (ll, p)
    last = [k for k in LAUNCH_ORDER if k in p["kind"]][-1]
    warps = ll["grid"] * ll["block"] // 32
    assert nframes * p["tasks_per_frame"][last] >= min_last * warps, (KERNEL_NAMES[last], nframes, p, ll)
    max_warps = ll["sms"] * torch.cuda.get_device_properties(0).max_threads_per_multi_processor // 32
    for k in p["tasks_per_frame"]:
        if k != last:
            assert nframes * p["tasks_per_frame"][k] >= min_other * max_warps, (KERNEL_NAMES[k], nframes, p)


_tls = threading.local()


def _check_chunk(key, setup, epoch, frame0, inp, got, n, w, h, fmt, od):
    """Oracle on `n` frames that start `frame0` frames after the epoch; (mismatch text or None, registers after)."""
    if getattr(_tls, "key", None) != key:  # one Oracle per worker thread, programmed once per configuration
        _tls.o = Oracle(); setup(_tls.o); _tls.key = key
    o = _tls.o
    o.set_lfsr(epoch)
    o.skip_frames(frame0, w, h)
    exp = o.add_grain_frames(inp, n, w, h, od)
    bad = None if np.array_equal(got, exp) else f"frames {frame0}+: " + first_mismatch(got, exp, w, h, fmt, n)
    return bad, o.get_lfsr()


def check_against_oracle(ex, setup, epoch, first, nframes, w, h, fmt, od, fetch):
    """Every frame of a call whose frame 0 is `first` frames after the epoch. fetch(k0, k1) -> (input, output) of
    frames [k0, k1) as host arrays. Returns the oracle's registers after the last frame."""
    samples = w * h + 2 * (w // {"420": 2, "422": 2, "444": 1}[fmt]) * (h // {"420": 2, "422": 1, "444": 1}[fmt])
    per = max(1, CHUNK_BYTES // (2 * samples))
    key = object()
    todo, bad, regs = [], [], None
    for k0 in range(0, nframes, per):
        k1 = min(nframes, k0 + per)
        inp, got = fetch(k0, k1)
        todo.append((k1, ex.submit(_check_chunk, key, setup, epoch, first + k0, inp, got, k1 - k0, w, h, fmt, od)))
        while len(todo) > 2 * WORKERS:  # bounded host memory
            regs = _collect(todo.pop(0), nframes, bad) or regs
    while todo:
        regs = _collect(todo.pop(0), nframes, bad) or regs
    assert not bad, bad[:4]
    return regs


def _collect(item, nframes, bad):
    k1, fut = item
    msg, regs = fut.result()
    if msg:
        bad.append(msg)
    return regs if k1 == nframes else None


def to_host(t):
    a = t.cpu().numpy()
    return a.view(np.uint16) if a.dtype == np.int16 else a


def sentinel_pool(n, dtype):
    """(whole allocation, the n-element pool inside it, guard elements per side): everything holds the sentinel."""
    import torch
    item = 2 if dtype == torch.int16 else 1
    guard = GUARD_BYTES // item
    raw = torch.empty(n + 2 * guard, dtype=dtype, device="cuda")
    raw.fill_(0x5A5A if item == 2 else 0xA5)
    return raw, raw[guard:guard + n], guard


def assert_guards_untouched(raw, guard):
    s = 0x5A5A if raw.dtype.itemsize == 2 else 0xA5
    assert bool((raw[:guard] == s).all()) and bool((raw[-guard:] == s).all()), "a write landed outside the output pool"


def bench_input(F, samples, w, depth, data, seed):
    """The resident input pool the way bench.py makes it (seeded torch.Generator on the device)."""
    import torch
    gen = torch.Generator(device="cuda"); gen.manual_seed(seed)
    sdt = torch.int16 if depth > 8 else torch.uint8
    if data == "uniform":
        return torch.randint(0, 1 << depth, (F * samples,), dtype=sdt, device="cuda", generator=gen)
    src = torch.empty(F * samples, dtype=sdt, device="cuda")
    lo, hi = 16 << (depth - 8), 235 << (depth - 8)
    idx = torch.arange(samples, device="cuda", dtype=torch.float32)
    for f in range(F):
        base = lo + (hi - lo) * (0.5 + 0.45 * torch.sin(idx * (6.2831853 / w) + f * 0.37))
        noise = torch.randint(-3, 4, (samples,), device="cuda", generator=gen)
        src[f * samples:(f + 1) * samples] = (base.to(torch.int32) + noise).clamp_(0, (1 << depth) - 1).to(sdt)
    return src


def golden_setup(case):
    return lambda target: program_case(target, G, case)


# ------------------------------------------------------------------------------------------------ 1b
def test_back_to_back_calls_like_a_bench_step(hw, pool):
    """Calls queued on one stream with no host synchronisation, the way a bench step queues them: successive frame
    positions of one input pool, two output pools taken in turn, so that the block tables of consecutive calls (two
    buffers used alternately, computed on a side stream) are reused while earlier grain kernels are still queued.
    Midway the configuration changes through the setters (a new set of table images while frames of the old one are
    in flight), and the geometry changes 4K -> 1080p -> 4K (the 1080p call needs larger block tables: the buffers grow
    while calls are queued). The output of a call whose pool a later call overwrites is copied aside on the stream."""
    import torch
    case_a, case_b = "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei.cfg|d10|420|g100"
    F4 = 15
    geo = {"4k": (3840, 2160, F4), "1080p": (1920, 1080, 4 * F4)}  # a 4K frame holds four 1080p frames
    samples4 = bench.frame_geometry(3840, 2160, "420", 10, 0)[0]
    n = F4 * samples4
    need_device_memory(10 * n * 2 + (1 << 30))
    # (configuration, geometry) of each call; frame positions run on per geometry
    calls = [("a", "4k"), ("a", "4k"), ("a", "4k"), ("b", "4k"), ("b", "1080p"), ("b", "1080p"), ("b", "4k"), ("b", "4k")]

    hw.reset()
    epoch = [int(v) for v in program_case(hw, G, case_a)["lfsr"]]
    src = bench_input(1, n, 3840, 10, "uniform", 99)
    outs = [sentinel_pool(n, torch.int16) for _ in range(2)]
    stream = torch.cuda.current_stream()
    pos, record = {"4k": 0, "1080p": 0}, []
    cfg = "a"
    for i, (c, gname) in enumerate(calls):
        if c != cfg:
            program_hw_from_state(hw, G.state(case_b))  # setters only: the registers stay where they are
            cfg = c
        w, h, F = geo[gname]
        position_shard(hw, epoch, 1000 + pos[gname], w, h)
        dst = outs[i % 2][1]
        hw.add_grain_frames_device(src, dst, F, w, h, 0, stream)
        overwritten = i + 2 < len(calls)
        snap = dst.clone() if overwritten else dst             # stream-ordered copy: no host synchronisation
        record.append((c, w, h, F, 1000 + pos[gname], snap))
        pos[gname] += F
    torch.cuda.synchronize()
    regs = hw.get_lfsr()
    for raw, _, guard in outs:
        assert_guards_untouched(raw, guard)
    for c, w, h, F, first, out in record:
        setup = golden_setup(case_a if c == "a" else case_b)
        samples = w * h * 3 // 2
        want = check_against_oracle(pool, setup, epoch, first, F, w, h, "420", 0,
                                    lambda k0, k1: (to_host(src[k0 * samples:k1 * samples]), to_host(out[k0 * samples:k1 * samples])))
    assert regs == want
    del src, outs, record
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ 1a
FULL_POOL = [(name, "uniform") for name in bench.WORKLOADS] + [("4k420_sei_default", "natural")]


@pytest.mark.parametrize("workload,data", FULL_POOL, ids=[n if d == "uniform" else f"{n}-natural" for n, d in FULL_POOL])
def test_bench_workload_full_pool(hw, emu, pool, workload, data):
    """One call exactly as bench.py makes it: the whole resident pool (frames per call as the bench sizes them), at the
    frame position of the last call of a default 8-GPU run (rank 7), input drawn the bench's way on the device."""
    import torch
    case, w, h, fmt, depth, od = bench.WORKLOADS[workload]
    samples, in_bytes, out_bytes = bench.frame_geometry(w, h, fmt, depth, od)
    F, _, first = bench_call(workload)
    assert F == int(max(8, min(4096, bench.POOL_INPUT_BYTES // in_bytes)))
    assert F * in_bytes > 1 << 32                               # input offsets past 2^32 bytes
    assert first * steps_per_frame(w, h) > 1 << 32              # more than 2^32 LFSR steps from the epoch
    need_device_memory(F * (in_bytes + out_bytes) + 2 * GUARD_BYTES + (1 << 30))

    setup = golden_setup(case)
    hw.reset()
    epoch = [int(v) for v in program_case(hw, G, case)["lfsr"]]
    src = bench_input(F, samples, w, depth, data, 1234 + 7)
    raw, dst, guard = sentinel_pool(F * samples, torch.int16 if (od or depth) > 8 else torch.uint8)
    position_shard(hw, epoch, first, w, h)
    hw.add_grain_frames_device(src, dst, F, w, h, od)
    torch.cuda.synchronize()
    regs = hw.get_lfsr()

    p = plan(emu, setup, w, h, od)
    assert_regime(hw, p, F, 64, 16)
    assert_guards_untouched(raw, guard)
    want = check_against_oracle(pool, setup, epoch, first, F, w, h, fmt, od,
                                lambda k0, k1: (to_host(src[k0 * samples:k1 * samples]), to_host(dst[k0 * samples:k1 * samples])))
    assert regs == want
    del src, dst, raw
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ 1c
def rand_setup(*params):
    return lambda target: program_random_state(target, *params)


AFGS10, AFGS8 = "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_afgs1_test1.cfg|d8|420|g100"
# name -> (setup, fmt, depth, width, height, out depth, in place, kernel mode, kernel kinds the planner must pick)
MANY_TASKS = {
    "fast_allwide_10to10": (golden_setup(AFGS10), "420", 10, 1280, 720, 0, False, 0, [0, 0, 0]),
    "fast_mixed_768": (golden_setup(AFGS10), "420", 10, 720, 480, 0, False, 0, [0, 0, 0]),
    "fast_10to8": (golden_setup(AFGS10), "420", 10, 1280, 720, 8, False, 0, [0, 0, 0]),
    "fast_8to8_wide": (golden_setup(AFGS8), "420", 8, 1280, 720, 0, False, 0, [0, 0, 0]),
    "fast_8to8_narrow": (rand_setup(2, 8, "444", 1, 1, 1, 7, False), "444", 8, 1096, 616, 0, False, 0, [0, 0, 0]),
    "edge": (golden_setup(AFGS10), "420", 10, 1366, 768, 0, False, 0, [3, 3, 3]),
    "gather_fold": (golden_setup("fgs_sei.cfg|d10|420|g100"), "420", 10, 1280, 720, 0, False, 0, [1, 0, 0]),
    "gather_no_fold": (rand_setup(7, 10, "420", 1, 1, 1, 7, True), "420", 10, 1280, 720, 0, False, 0, [1, 1, 1]),
    "gather_shift_in_place": (golden_setup("fgs_sei.cfg|d10|420|g100"), "420", 10, 1280, 720, 0, True, 0, [1, 0, 0]),
    "general": (golden_setup(AFGS10), "420", 10, 1280, 720, 0, False, 1, [2, 2, 2]),
    "fmt422": (golden_setup("fgs_sei_ff_test4.cfg|d10|422|g150"), "422", 10, 1280, 720, 0, False, 0, None),
    "fmt444": (golden_setup("fgs_sei_ff_test4.cfg|d10|444|g150"), "444", 10, 1280, 720, 0, False, 0, None),
}
MIN_TASKS_PER_WARP = 32


def frames_for_many_tasks(p, sms, threads_per_sm):
    """An odd frame count that gives even the most warps the device can hold at once at least MIN_TASKS_PER_WARP
    warp-tasks of the call's last launch, and a quarter of that in any earlier one."""
    warps = sms * threads_per_sm // 32
    last = [k for k in LAUNCH_ORDER if k in p["kind"]][-1]
    F = max(-(-(MIN_TASKS_PER_WARP if k == last else MIN_TASKS_PER_WARP // 4) * warps // t) for k, t in p["tasks_per_frame"].items())
    return F | 1


@pytest.mark.parametrize("variant", list(MANY_TASKS))
def test_many_tasks_per_warp(hw, emu, pool, variant):
    """Small pictures, many frames per call: every warp of the persistent grid runs at least 32 warp-tasks, one case
    per kernel instance. Unit runs per component that are not multiples of 32 and an odd frame count make tasks
    straddle stripe rows, component ends and frame ends."""
    import torch
    from tests.util import synth_frames
    setup, fmt, depth, w, h, od, in_place, mode, kinds = MANY_TASKS[variant]
    p = plan(emu, setup, w, h, od, in_place, mode)
    if kinds is not None:
        assert p["kind"] == kinds, p
    assert p["gather_fold"] == (variant in ("gather_fold", "gather_shift_in_place"))
    assert p["gather_shift"] == (variant == "gather_shift_in_place")
    R = (h + 15) // 16
    if mode != 1:
        assert any(u * R % 32 for u in p["units"]), p  # some component's run of lane units ends inside a warp-task
    props = torch.cuda.get_device_properties(0)
    F = frames_for_many_tasks(p, props.multi_processor_count, props.max_threads_per_multi_processor)
    samples, in_bytes, out_bytes = bench.frame_geometry(w, h, fmt, depth, od)
    need_device_memory(F * (2 * in_bytes + out_bytes) + 2 * GUARD_BYTES + (1 << 30))

    # synth_frames input, made chunk by chunk (a chunk's frames from their own seed) on the worker threads
    per = max(1, CHUNK_BYTES // in_bytes)
    starts = list(range(0, F, per))
    sdt = torch.int16 if depth > 8 else torch.uint8
    src = torch.empty(F * samples, dtype=sdt, device="cuda")
    gen = lambda k0: synth_frames(min(per, F - k0), w, h, fmt, depth, seed=1000 + k0)
    for k0, a in zip(starts, pool.map(gen, starts)):
        src[k0 * samples:k0 * samples + a.size].copy_(torch.from_numpy(a.view(np.int16) if depth > 8 else a))

    hw.reset(); setup(hw)
    epoch = hw.get_lfsr()
    ddt = torch.int16 if (od or depth) > 8 else torch.uint8
    raw, dst, guard = sentinel_pool(F * samples, ddt)
    if in_place:
        dst.copy_(src)
    hw.force_general_kernel(mode)
    try:
        hw.add_grain_frames_device(dst if in_place else src, dst, F, w, h, od)
        torch.cuda.synchronize()
    finally:
        hw.force_general_kernel(0)
    regs = hw.get_lfsr()
    assert_regime(hw, p, F, MIN_TASKS_PER_WARP, MIN_TASKS_PER_WARP // 4)
    assert_guards_untouched(raw, guard)
    want = check_against_oracle(pool, setup, epoch, 0, F, w, h, fmt, od,
                                lambda k0, k1: (to_host(src[k0 * samples:k1 * samples]), to_host(dst[k0 * samples:k1 * samples])))
    assert regs == want
    del src, dst, raw
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ 1d
@pytest.mark.parametrize("layout", ["packed", "padded_planes"])
def test_in_place_scratch_route_spans_sub_batches(hw, emu, pool, layout):
    """In place with sample-adaptive 8-sample-block chroma (fgs_sei_ff_test5): the library runs the frames through a
    256 MB scratch output buffer in sub-batches (10 frames at 4K) and copies them back plane by plane. 25 frames make
    three sub-batches, the last one partial: the later ones start at a non-zero frame of the call. Once on packed
    frames, once on planes with padded rows and frames: the pictures match the oracle, and the row padding, the frame
    padding and the guard bands around the buffer are untouched."""
    import torch
    from versatilefilmgrain_b200.api import Planes
    case, w, h, F = "fgs_sei_ff_test5.cfg|d10|420|g100", 3840, 2160, 25
    setup = golden_setup(case)
    assert plan(emu, setup, w, h, 0, True)["kind"] == [0, 2, 2]   # the general kernel in place: the scratch route
    sub = plan(emu, setup, w, h)                                  # each sub-batch runs out of place into the scratch buffer
    assert sub["kind"] == [0, 1, 1]
    cw, ch = w // 2, h // 2
    samples = w * h + 2 * cw * ch
    assert samples * 2 * 10 <= 256 << 20 < samples * 2 * 11       # ten frames per sub-batch
    if layout == "packed":
        sy, sc, fs = w, cw, samples
    else:
        sy, sc = w + 64, cw + 96                                  # elements per row (row padding)
        fs = sy * h + 2 * sc * ch + 128                           # elements per frame (frame padding)
    need_device_memory(3 * F * fs * 2 + 2 * GUARD_BYTES + (1 << 30))

    hw.reset()
    epoch = [int(v) for v in program_case(hw, G, case)["lfsr"]]
    raw, buf, guard = sentinel_pool(F * fs, torch.int16)
    gen = torch.Generator(device="cuda"); gen.manual_seed(5)
    buf.copy_(torch.randint(0, 1 << 10, (F * fs,), dtype=torch.int16, device="cuda", generator=gen))
    before = buf.clone()
    frames = buf.view(F, fs)

    def plane_views(t):
        fr = t.view(F, fs)
        y = fr[:, :sy * h].view(F, h, sy)
        u = fr[:, sy * h:sy * h + sc * ch].view(F, ch, sc)
        v = fr[:, sy * h + sc * ch:sy * h + 2 * sc * ch].view(F, ch, sc)
        return y, u, v

    def packed(t, k0, k1):  # frames [k0, k1) of planes `t` as packed host frames
        y, u, v = plane_views(t)
        return np.concatenate([to_host(x[k0:k1, :, :width].reshape(k1 - k0, -1)) for x, width in ((y, w), (u, cw), (v, cw))],
                              axis=1).reshape(-1)

    base, item = buf.data_ptr(), 2
    pl = Planes(base, base + sy * h * item, base + (sy * h + sc * ch) * item, sy * item, sc * item, fs * item)
    launches = hw.launch_count()
    if layout == "packed":
        hw.add_grain_frames_device(buf, buf, F, w, h, 0)
    else:
        hw.add_grain_planes_device(pl, pl, F, w, h, 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    regs = hw.get_lfsr()
    # three sub-batches, each a block-table launch and the out-of-place plan's grain kernels (a single in-place pass
    # would be one table launch and two grain launches)
    assert sorted(hw.last_launch()["kernels"]) == sorted({KERNEL_NAMES[k] for k in sub["kind"]})
    assert hw.launch_count() - launches == 3 * (1 + len(set(sub["kind"])))
    assert_guards_untouched(raw, guard)
    # nothing but the pictures changed
    mask = torch.ones(F * fs, dtype=torch.bool, device="cuda")
    my, mu, mv = plane_views(mask)
    my[:, :, :w] = False; mu[:, :, :cw] = False; mv[:, :, :cw] = False
    assert bool((buf[mask] == before[mask]).all()), "in-place call wrote outside the pictures"
    want = check_against_oracle(pool, setup, epoch, 0, F, w, h, "420", 0,
                                lambda k0, k1: (packed(before, k0, k1), packed(buf, k0, k1)))
    assert regs == want
    del raw, buf, before, frames, mask
    torch.cuda.empty_cache()
