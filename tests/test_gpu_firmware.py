"""The firmware layer with the pattern synthesis on the GPU (include/vfgs_fw.h: vfgs_b200_init_sei / _afgs1; kernels
fw_pattern_kernel, versatilefilmgrain_b200/csrc/fw_device.h) against the hardware state the UNMODIFIED reference
firmware (vfgs_fw.c:517-708) programmed for every golden case, and the table-image ring that lets a configuration
change happen while frames are still in flight."""
import numpy as np
import pytest

from tests.fixtures import SUBSAMPLING
from tests.util import Oracle, first_mismatch, load_golden, program_case, states_equal, synth_frames

pytestmark = pytest.mark.gpu

G = load_golden()
CASES = G.runnable()


@pytest.fixture(scope="module")
def hw():
    import torch
    assert torch.cuda.is_available(), "these tests need a CUDA device"
    from versatilefilmgrain_b200 import VfgsHw
    return VfgsHw(device=0)


def init_from_golden(hw, case):
    """What vfgs_main.c:750-760 does, with the device firmware in place of vfgs_init_*."""
    meta = G.cases[case]
    hw.reset()
    hw.vfgs_set_depth(meta["depth"])
    hw.vfgs_set_chroma_subsampling(*SUBSAMPLING[meta["fmt"]])
    (hw.init_afgs1 if meta["afgs1"] else hw.init_sei)(G.struct(case))
    if not meta["afgs1"]:
        hw.vfgs_set_seed(G.seed)


@pytest.mark.parametrize("case", CASES)
def test_device_firmware_programs_the_reference_state(hw, case):
    before = hw.launch_count()
    init_from_golden(hw, case)
    assert hw.launch_count() > before  # the patterns came out of CUDA kernels
    assert states_equal(hw.state(), G.state(case), G.cases[case]["nslot"]) == [], case


@pytest.mark.parametrize("case", CASES)
def test_device_firmware_then_frames(hw, case):
    """Frames through the tables the device firmware built, for every golden configuration; 10-bit input also to
    8-bit output (the CLI's --outdepth 8)."""
    import torch
    meta = G.cases[case]
    w, h, n = 512, 152, 3
    frames = synth_frames(n, w, h, meta["fmt"], meta["depth"], seed=31)
    src = torch.from_numpy(frames.view(np.int16) if frames.dtype == np.uint16 else frames).cuda()
    for od in ((0, 8) if meta["depth"] == 10 else (0,)):
        init_from_golden(hw, case)
        o = Oracle(); program_case(o, G, case)
        want = o.add_grain_frames(frames, n, w, h, od)
        dst = torch.empty(frames.size, dtype=torch.uint8 if (od == 8 or meta["depth"] == 8) else torch.int16, device="cuda")
        hw.add_grain_frames_device(src, dst, n, w, h, od)
        torch.cuda.synchronize()
        got = dst.cpu().numpy()
        got = got.view(np.uint16) if got.dtype == np.int16 else got
        assert np.array_equal(got, want), (od, first_mismatch(got, want, w, h, meta["fmt"], n))
        assert hw.get_lfsr() == o.get_lfsr(), od


def test_configuration_switch_with_frames_in_flight(hw):
    """Per-picture metadata updates (vfgs_main.c:773-781): a long batch is queued, the configuration is replaced at once
    (new patterns, LUTs, scale shift, clip range, seed), a second batch is queued -- nothing waits for the first batch.
    Each batch must come out under the configuration it was queued with: the kernels of the first keep reading their
    own table images (ring of image sets, vfgs_b200.cu upload_blob)."""
    import torch
    a, b, c3 = "fgs_sei.cfg|d10|420|g100", "fgs_afgs1_test1.cfg|d10|420|g100", "fgs_sei_ff_test5.cfg|d10|420|g100"
    w, h, n = 1920, 1080, 12
    frames = synth_frames(n, w, h, "420", 10, seed=5)
    src = torch.from_numpy(frames.view(np.int16)).cuda()
    outs = [torch.empty_like(src) for _ in range(6)]
    stream = torch.cuda.Stream()
    order = [a, b, c3, a, b, c3]  # six changes: the ring of four sets wraps around
    with torch.cuda.stream(stream):
        for case, dst in zip(order, outs):
            init_from_golden(hw, case)
            hw.add_grain_frames_device(src, dst, n, w, h, 0, stream)
    torch.cuda.synchronize()
    want = {}
    for case in (a, b, c3):
        o = Oracle(); program_case(o, G, case)
        want[case] = o.add_grain_frames(frames, n, w, h, 0)
    for case, dst in zip(order, outs):
        got = dst.cpu().numpy().view(np.uint16)
        assert np.array_equal(got, want[case]), (case, first_mismatch(got, want[case], w, h, "420", n))
