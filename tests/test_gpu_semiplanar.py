"""vfgs_b200_add_grain_semiplanar_device on the GPU: NV12 / P010 frames against the oracle's planar output converted, the
reference's digests, register continuity with planar calls, decoder-style surfaces, kernel selection and one
bench-sized 4K P010 call. Run with -m gpu on a B200."""
import numpy as np
import pytest

from tests.semiplanar import planar_to_semi, semi_to_planar
from tests.util import Oracle, bench_call, load_golden, parse_output_key, program_case, sha, synth_frames

pytestmark = pytest.mark.gpu

G = load_golden()
CASES = [c for c in G.runnable() if G.cases[c]["fmt"] in ("420", "422")]


@pytest.fixture(scope="module")
def hw():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from versatilefilmgrain_b200 import VfgsHw
    return VfgsHw(device=0)


def surface(Y, UV, pitch_pad=0):
    """Decoder-style surface (n, h + ch, pitch) on the device holding Y then UV rows; pitch_pad extra samples per row."""
    import torch
    n, h, w = Y.shape
    ch = UV.shape[1]
    s = np.zeros((n, h + ch, w + pitch_pad), dtype=Y.dtype)
    s[:, :h, :w], s[:, h:, :UV.shape[2]] = Y, UV
    return torch.from_numpy(s.view(np.int16) if s.dtype == np.uint16 else s).cuda()


def unpack(t, h, w, cw2):
    a = t.cpu().numpy()
    a = a.view(np.uint16) if a.dtype == np.int16 else a
    return a[:, :h, :w].copy(), a[:, h:, :cw2].copy()


def run_surfaces(hw, frames, n, w, h, fmt, depth, p010_out, pitch_pad=0, in_place=False, seed=0):
    import torch
    from versatilefilmgrain_b200.api import NV12, P010
    p010 = depth == 10
    Y, UV = planar_to_semi(frames, n, w, h, fmt, p010, rng=np.random.default_rng(seed))
    src = surface(Y, UV, pitch_pad)
    if in_place:
        dst = src
    else:
        dst = torch.zeros(src.shape, dtype=torch.int16 if p010_out else torch.uint8, device="cuda")
    hw.add_grain_surfaces(src, dst, n, w, h, out_format=P010 if p010_out else NV12)
    torch.cuda.synchronize()
    oy, ouv = unpack(dst, h, w, UV.shape[2])
    if p010_out:
        assert not (oy & 63).any() and not (ouv & 63).any()
    return semi_to_planar(oy, ouv, p010_out)


@pytest.mark.parametrize("case", CASES)
def test_semiplanar_case_matrix(hw, case):
    """Every 4:2:0 / 4:2:2 golden case, NV12 / P010 / P010 -> NV12, kernel modes 0/1/2, plain and padded pitches:
    the output converted to planar equals the oracle's, the registers afterwards equal the oracle's."""
    meta = G.cases[case]
    for (w, h, n, pad) in ((512, 56, 2, 0), (264, 40, 2, 0), (640, 34, 1, 64)):
        for p010_out in ((True, False) if meta["depth"] == 10 else (False,)):
            frames = synth_frames(n, w, h, meta["fmt"], meta["depth"], seed=w)
            o = Oracle(); program_case(o, G, case)
            want = o.add_grain_frames(frames, n, w, h, 0 if p010_out or meta["depth"] == 8 else 8)
            for mode in (0, 1, 2):
                hw.reset(); program_case(hw, G, case)
                hw.force_general_kernel(mode)
                try:
                    got = run_surfaces(hw, frames, n, w, h, meta["fmt"], meta["depth"], p010_out, pitch_pad=pad, seed=mode)
                finally:
                    hw.force_general_kernel(0)
                assert np.array_equal(got, want), (case, w, h, p010_out, mode, int(np.count_nonzero(got != want)))
                assert hw.get_lfsr() == o.get_lfsr()


@pytest.mark.parametrize("case", CASES)
def test_reference_digests_and_shards(hw, case):
    """The semi-planar output converted to planar reproduces the digests the unmodified reference recorded, for the
    continuous run and for shards started at non-zero frame offsets through vfgs_b200_skip_frames."""
    meta = G.cases[case]
    epoch = [int(v) for v in G.state(case)["lfsr"]]
    for key, want in meta["outputs"].items():
        w, h, n, iseed, od = parse_output_key(key)
        frames = synth_frames(n, w, h, meta["fmt"], meta["depth"], seed=iseed)
        hw.reset(); program_case(hw, G, case)
        got = run_surfaces(hw, frames, n, w, h, meta["fmt"], meta["depth"], meta["depth"] == 10 and od != 8)
        assert sha(got) == want["sha256"], (case, key)
        assert hw.get_lfsr() == want["lfsr_after"], (case, key)
    for key, groups in meta.get("shards", {}).items():
        w, h, n, iseed, od = parse_output_key(key)
        frames = synth_frames(n, w, h, meta["fmt"], meta["depth"], seed=iseed)
        for g in (1, 5):
            if g >= len(groups):
                continue
            hw.reset(); program_case(hw, G, case)
            hw.set_lfsr(epoch); hw.skip_frames(g * n, w, h)
            got = run_surfaces(hw, frames, n, w, h, meta["fmt"], meta["depth"], meta["depth"] == 10 and od != 8)
            assert sha(got) == groups[g]["sha256"], (case, key, g)
            assert hw.get_lfsr() == groups[g]["lfsr_after"], (case, key, g)


def test_semiplanar_planar_semiplanar_back_to_back(hw):
    """Three calls queued without a synchronisation in between: semi-planar, planar, semi-planar; each equals the
    oracle's continuous run, and so do the registers."""
    import torch
    from versatilefilmgrain_b200.api import P010
    case, w, h, n = "fgs_afgs1_test1.cfg|d10|420|g100", 1920, 136, 3
    frames = [synth_frames(n, w, h, "420", 10, seed=s) for s in (1, 2, 3)]
    o = Oracle(); program_case(o, G, case)
    want = [o.add_grain_frames(f, n, w, h, 0) for f in frames]
    hw.reset(); program_case(hw, G, case)
    srcs, dsts = [], []
    for k, f in enumerate(frames):
        if k == 1:
            src = torch.from_numpy(f.view(np.int16)).cuda(); dst = torch.zeros_like(src)
            hw.add_grain_frames_device(src, dst, n, w, h)
        else:
            Y, UV = planar_to_semi(f, n, w, h, "420", True)
            src = surface(Y, UV); dst = torch.zeros_like(src)
            hw.add_grain_surfaces(src, dst, n, w, h, out_format=P010)
        srcs.append(src); dsts.append(dst)
    torch.cuda.synchronize()
    for k in range(3):
        if k == 1:
            got = dsts[k].cpu().numpy().view(np.uint16)
        else:
            got = semi_to_planar(*unpack(dsts[k], h, w, w), True)
        assert np.array_equal(got, want[k]), k
    assert hw.get_lfsr() == o.get_lfsr()


@pytest.mark.parametrize("case", ["fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei_ff_test1.cfg|d8|420|g100",
                                  "fgs_sei_ff_test5.cfg|d10|420|g100", "fgs_sei.cfg|d10|420|g100"])
def test_separate_allocations_and_in_place(hw, case):
    """Y and UV in separate allocations with pitched rows (out of place and in place), and pitched surfaces in place."""
    import torch
    from versatilefilmgrain_b200.api import NV12, P010, SemiPlanes
    meta = G.cases[case]
    p010 = meta["depth"] == 10
    w, h, n = 1920, 72, 2
    frames = synth_frames(n, w, h, "420", meta["depth"], seed=5)
    o = Oracle(); program_case(o, G, case)
    want = o.add_grain_frames(frames, n, w, h, 0)
    Y, UV = planar_to_semi(frames, n, w, h, "420", p010)
    dt = torch.int16 if p010 else torch.uint8
    sz = 2 if p010 else 1
    pitch = w + 128

    for in_place in (False, True):
        ty = torch.zeros((n, h, pitch), dtype=dt, device="cuda")
        tuv = torch.zeros((n, h // 2, pitch), dtype=dt, device="cuda")
        ty[:, :, :w] = torch.from_numpy(Y.view(np.int16) if p010 else Y).cuda()
        tuv[:, :, :w] = torch.from_numpy(UV.view(np.int16) if p010 else UV).cuda()
        # separate allocations: one frame per call so that a common frame stride is not needed
        hw.reset(); program_case(hw, G, case)
        outs = []
        for f in range(n):
            pin = SemiPlanes(ty[f].data_ptr(), tuv[f].data_ptr(), pitch * sz, pitch * sz, 0, P010 if p010 else NV12)
            if in_place:
                pout = pin
                outs.append((ty[f], tuv[f]))
            else:
                oy, ouv = torch.zeros_like(ty[f]), torch.zeros_like(tuv[f])
                pout = SemiPlanes(oy.data_ptr(), ouv.data_ptr(), pitch * sz, pitch * sz, 0, P010 if p010 else NV12)
                outs.append((oy, ouv))
            hw.add_grain_semiplanar_device(pin, pout, 1, w, h, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        gy = np.stack([a.cpu().numpy()[:, :w] for a, _ in outs]); guv = np.stack([b.cpu().numpy()[:, :w] for _, b in outs])
        if p010:
            gy, guv = gy.view(np.uint16), guv.view(np.uint16)
        assert np.array_equal(semi_to_planar(gy, guv, p010), want), (case, in_place)
        assert hw.get_lfsr() == o.get_lfsr()
    hw.reset(); program_case(hw, G, case)
    got = run_surfaces(hw, frames, n, w, h, "420", meta["depth"], p010, pitch_pad=64, in_place=True)
    assert np.array_equal(got, want), (case, "pitched surface in place")


def test_kernel_selection(hw):
    """last_launch: AFGS1 at 4K runs the fast kernel with the interleaved lane, default-SEI P010 luma the gather kernel,
    ff_test5 chroma (sample-adaptive) the general kernel."""
    import torch
    from versatilefilmgrain_b200.api import P010
    w, h = 3840, 2160
    src = torch.zeros((1, h + h // 2, w), dtype=torch.int16, device="cuda")
    dst = torch.zeros_like(src)
    for case, want in (("fgs_afgs1_test1.cfg|d10|420|g100", {"fgs_apply_fast_kernel", "fgs_apply_fast_kernel<interleaved UV>"}),
                       ("fgs_sei.cfg|d10|420|g100", {"fgs_apply_gather_kernel", "fgs_apply_fast_kernel", "fgs_apply_fast_kernel<interleaved UV>"}),
                       ("fgs_sei_ff_test5.cfg|d10|420|g100", {"fgs_apply_fast_kernel", "fgs_apply_kernel"})):
        hw.reset(); program_case(hw, G, case)
        hw.add_grain_surfaces(src, dst, 1, w, h, out_format=P010)
        torch.cuda.synchronize()
        assert set(hw.last_launch()["kernels"]) == want, (case, hw.last_launch())


def test_bench_sized_4k_p010_call(hw):
    """One 4K P010 -> P010 call whose input passes 2^32 bytes, at the frame position of the last call of a default
    bench.py run, every frame checked against the oracle, guard bands around the output untouched."""
    import torch
    from versatilefilmgrain_b200.api import P010, SemiPlanes
    case, w, h = "fgs_afgs1_test1.cfg|d10|420|g100", 3840, 2160
    ch, fs = h // 2, (h + h // 2) * w * 2
    n = (1 << 32) // fs + 4
    free, _ = torch.cuda.mem_get_info()
    if free < 2 * n * fs + (1 << 30):
        pytest.skip(f"needs {2 * n * fs / 1e9:.1f} GB of free device memory")
    _, _, first = bench_call("4k420_afgs1_10to10")
    g = torch.Generator(device="cuda"); g.manual_seed(7)
    src = torch.randint(0, 1 << 16, (n, h + ch, w), dtype=torch.int32, device="cuda", generator=g).to(torch.int16)
    guard = 1 << 20
    sentinel = 0x5a5a
    raw = torch.full((n * (h + ch) * w + 2 * guard,), sentinel, dtype=torch.int16, device="cuda")
    dst = raw[guard:guard + n * (h + ch) * w].view(n, h + ch, w)
    hw.reset(); program_case(hw, G, case)
    epoch = hw.get_lfsr()
    hw.skip_frames(first, w, h)
    pin = SemiPlanes(src.data_ptr(), src.data_ptr() + h * w * 2, w * 2, w * 2, fs, P010)
    pout = SemiPlanes(dst.data_ptr(), dst.data_ptr() + h * w * 2, w * 2, w * 2, fs, P010)
    hw.add_grain_semiplanar_device(pin, pout, n, w, h, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    assert n * fs > 1 << 32
    assert bool((raw[:guard] == sentinel).all()) and bool((raw[-guard:] == sentinel).all())
    o = Oracle(); program_case(o, G, case)
    o.set_lfsr(epoch); o.skip_frames(first, w, h)
    for f0 in range(0, n, 4):
        k = min(4, n - f0)
        iy, iuv = unpack(src[f0:f0 + k], h, w, w)
        frames = semi_to_planar(iy, iuv, True)
        want = o.add_grain_frames(frames, k, w, h, 0)
        got = semi_to_planar(*unpack(dst[f0:f0 + k], h, w, w), True)
        assert np.array_equal(got, want), f0
    assert hw.get_lfsr() == o.get_lfsr()
