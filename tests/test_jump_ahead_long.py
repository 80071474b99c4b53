"""The LFSR jump-ahead at long step counts, against plain serial stepping (no GPU).

The library never steps the LFSR serially across frames: it moves whole frames by GF(2) matrix powers
(vfgs_core.h JumpTable, vfgs_b200_skip_frames), and so does the oracle (oracle_lfsr_jump). The reference's
serial known answers in tests/golden stop at 1,000,003 steps, so matrix powers 2^20 and above would otherwise
be checked only against the oracle, which builds them the same way. Here a tiny C program steps the register
one step at a time past 2^32 steps, reports it at a sorted list of checkpoints in one pass and measures the
period on the way; the period carries the check on to the 2^33 .. 2^36 step counts a multi-GPU bench run
reaches (bench.py moves every call to its first frame with skip_frames)."""
import os
import subprocess

import pytest

from tests.util import Oracle, bench_last_call_first_frame, load_golden

SERIAL_C = r"""
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
/* argv: start register, then checkpoints in increasing order. Prints "<n> <register after n steps>" per
   checkpoint, then "period <p>": the least p > 0 with x(p + 1) == x(1). One step is vfgs_hw.c:74-79: a 31-bit
   Fibonacci LFSR in bits 31..1, new top bit = bit 1 ^ bit 29, bit 0 trails (so x(0) itself may be off the cycle). */
int main(int argc, char** argv)
{
	uint32_t x = (uint32_t)strtoul(argv[1], 0, 0), x1 = 0;
	uint64_t period = 0, n = 0;
	for (int k = 2; k < argc; k++) {
		const uint64_t next = strtoull(argv[k], 0, 0);
		for (; n < next; n++) {
			x = (x >> 1) | ((((x >> 1) ^ (x >> 29)) & 1u) << 31);
			if (n == 0) x1 = x;
			else if (!period && x == x1) period = n;
		}
		printf("%llu %u\n", (unsigned long long)n, x);
	}
	printf("period %llu\n", (unsigned long long)period);
	return 0;
}
"""

G = load_golden()
W4K, H4K = 3840, 2160
NB4K = (W4K + 15) // 16
STEPS_PER_4K_FRAME = ((H4K + 15) // 16 - 1) * NB4K  # 32160: the library moves in whole frames of this many steps
P = (1 << 31) - 1

# where the registers start: the golden epochs (the reference's power-on 0xdeadbeef, odd, and the registers the
# cfg files seed) and a freshly seeded register (vfgs_set_seed: seed << 1) whose bit 0 is off the cycle
SEEDED = 0x0C0FFEE5 << 1 & 0xFFFFFFFF
STARTS = sorted({0xdeadbeef, SEEDED} | {int(G.state(c)["lfsr"][2]) for c in G.runnable()})

BENCH_FRAME = bench_last_call_first_frame("4k420_afgs1_10to10")
# exact step counts checked against the jump-ahead
EXACT = [(1 << 31) - 2, (1 << 31) - 1, 1 << 31, (1 << 32) - 1, 1 << 32, BENCH_FRAME * STEPS_PER_4K_FRAME] + \
        [(1 << e) + d for e in range(33, 37) for d in (-1, 0, 1)]
# whole 4K frames on both sides of each exact count (and the bench's own frame), for the library's bookkeeping
FRAMES = sorted({f for n in EXACT for f in (n // STEPS_PER_4K_FRAME, n // STEPS_PER_4K_FRAME + 1)} | {BENCH_FRAME})
# steps the serial pass covers: everything up to just past 2^32 directly, longer counts through the period
SERIAL_END = (1 << 32) + 2 * STEPS_PER_4K_FRAME


def frame_counts(f):
    """Step counts of the four registers after f whole 4K frames (advance_registers): rnd, rnd_up, line_rnd, line_rnd_up."""
    adv = f * STEPS_PER_4K_FRAME
    return [adv + NB4K, adv, adv, adv - NB4K]


def reduce(n, period):
    """A step count >= 1 folded onto the cycle: x(n) == x(((n - 1) mod p) + 1); counts inside the serial pass stay."""
    return n if n <= SERIAL_END else (n - 1) % period + 1


@pytest.fixture(scope="module")
def serial(tmp_path_factory):
    """{start register: ({step count: register}, period)}, one serial pass per start register, run side by side."""
    d = tmp_path_factory.mktemp("lfsr_serial")
    src, exe = os.path.join(d, "serial.c"), os.path.join(d, "serial")
    with open(src, "w") as f:
        f.write(SERIAL_C)
    subprocess.run(["gcc", "-O2", "-o", exe, src], check=True)
    counts = {n for n in EXACT if n <= SERIAL_END} | {n for f in FRAMES for n in frame_counts(f) if n <= SERIAL_END}
    # the folded counts are known only once the period is; it is (2^31 - 1), asserted below, so they can be listed now
    counts |= {reduce(n, P) for n in EXACT} | {reduce(n, P) for f in FRAMES for n in frame_counts(f)}
    counts |= {0, 1, P, P + 1, SERIAL_END}
    args = [str(n) for n in sorted(counts)]
    procs = {s: subprocess.Popen([exe, str(s)] + args, stdout=subprocess.PIPE, text=True) for s in STARTS}
    out = {}
    for s, p in procs.items():
        text, _ = p.communicate(timeout=600)
        assert p.returncode == 0
        regs, period = {}, None
        for line in text.split("\n"):
            if line.startswith("period"):
                period = int(line.split()[1])
            elif line:
                n, x = line.split()
                regs[int(n)] = int(x)
        out[s] = (regs, period)
    return out


def test_period_is_that_of_the_cycle(serial):
    """Every start register comes back after 2^31 - 1 steps (x^31 + x^3 + 1 is primitive); a register whose bit 0 does
    not follow from its other bits (the odd default, a seed with bit 27 set) is off the cycle: it never comes back
    itself, its successor does."""
    for s, (regs, period) in serial.items():
        assert period == P, hex(s)
        assert regs[P + 1] == regs[1], hex(s)
        on_cycle = (s >> 31) == ((s ^ (s >> 28)) & 1)
        assert (regs[P] == s) == on_cycle, hex(s)
    assert serial[0xdeadbeef][0][P] != 0xdeadbeef and serial[SEEDED][0][P] != SEEDED


def test_oracle_jump_matches_serial_steps(serial):
    o = Oracle()
    for s, (regs, period) in serial.items():
        for n in EXACT:
            assert o.lfsr_jump(s, n) == regs[reduce(n, period)], (hex(s), n)


def test_library_skip_frames_matches_serial_steps(serial, hw_lib):
    """vfgs_b200_skip_frames from each start register, to the whole 4K frames next to every checkpoint and to the
    bench's last frame position: all four registers against the serial pass. No device is involved."""
    for s, (regs, period) in serial.items():
        for f in FRAMES:
            hw_lib.reset()
            hw_lib.set_lfsr([s] * 4)
            hw_lib.skip_frames(f, W4K, H4K)
            want = [regs[reduce(n, period)] for n in frame_counts(f)]
            assert hw_lib.get_lfsr() == want, (hex(s), f)


def test_checkpoints_reach_the_bench_regime():
    """The counts above are the ones that matter: past 2^32 steps, and the bench's last position is among them."""
    assert BENCH_FRAME * STEPS_PER_4K_FRAME > 1 << 35
    assert max(FRAMES) * STEPS_PER_4K_FRAME > 1 << 36
    assert SERIAL_END > 1 << 32
