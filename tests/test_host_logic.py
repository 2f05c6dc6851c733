"""CPU checks of host-side logic and of closed forms the kernels rely on (no GPU, no native code)."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_fire_clock_closed_form_equals_the_reference_predicate():
    """same_lane.cuh:fire_clock uses c* = floor(until - 0.5) + 1 for 1 <= until < 2^22 without evaluating the
    reference's predicate (receiver.rs:352-353: r = until - c as f32; fire if r <= 0 || |r| < 0.5).  Check in f32
    arithmetic that c* fires and c* - 1 does not, on random and adversarial values."""
    rng = np.random.default_rng(1)
    vals = [rng.uniform(1.0, 64.0, 400000), rng.uniform(1.0, 4.0e6, 200000),
            np.arange(1, 4000, dtype=np.float64)[:, None] + np.array([0.0, 0.5, -0.5, 0.49999997, 0.50000006, 1e-7, -1e-7])[None, :]]
    until = np.concatenate([np.asarray(v).reshape(-1) for v in vals]).astype(np.float32)
    # neighbours in f32 of every half-integer: the worst cases for the 0.5 threshold
    half = (np.arange(1, 5000, dtype=np.float32) + np.float32(0.5))
    until = np.concatenate([until, half, np.nextafter(half, np.float32(0)), np.nextafter(half, np.float32(1e9))])
    until = until[(until >= 1.0) & (until < 4.0e6)]

    def fires(u, c):
        r = (u - c.astype(np.float32)).astype(np.float32)
        return (r <= 0) | (np.abs(r) < np.float32(0.5))

    cstar = np.floor((until - np.float32(0.5)).astype(np.float32)).astype(np.int64) + 1
    assert np.all(cstar >= 1)
    assert np.all(fires(until, cstar))
    prev = cstar - 1
    assert not np.any(fires(until, prev)[prev >= 1])


def test_bench_stripes_ranks_over_the_device_range():
    import bench
    assert [bench.device_for_rank(r, 8, 8) for r in range(8)] == list(range(8))
    assert [bench.device_for_rank(r, 4, 8) for r in range(4)] == [0, 4, 1, 5]
    assert [bench.device_for_rank(r, 2, 8) for r in range(2)] == [0, 4]
    assert [bench.device_for_rank(r, 2, 4) for r in range(2)] == [0, 2]
    assert bench.device_for_rank(0, 1, 8) == 0
    assert [bench.device_for_rank(r, 4, 4) for r in range(4)] == [0, 1, 2, 3]      # nothing to choose
    assert sorted(bench.device_for_rank(r, 3, 7) for r in range(3)) == [0, 1, 3]   # odd device counts stay distinct
    for world, ndev in [(2, 8), (4, 8), (3, 8), (5, 8), (2, 3), (6, 7)]:
        got = [bench.device_for_rank(r, world, ndev) for r in range(world)]
        assert len(set(got)) == world and all(0 <= d < ndev for d in got)


def test_speculative_agc_blocks_coalesce_bitwise_on_the_corpus_noise():
    """The long-stream path (same_long.cu) runs the unlocked AGC in blocks that warm up 1024 samples early from a guessed
    gain and uses a block only if its start gain equals the sequential trajectory bit for bit.  Modelled here on the
    oracle's own DCBlocker/Agc: on the corpus noise (sigma 3663, samedec limits) every hand-over matches and the
    trajectories coalesce within a few hundred samples, from the gain the stream starts with as well as from the far
    clamp; on exact silence the gain runs into its upper clamp and matches too.  This does not hold at every level:
    noise of sigma ~300-1000 fails nearly every hand-over (the band is pinned in tests/test_levels_cpu.py)."""
    from oracle import agc_block_model, synth_cpu
    from oracle.pyoracle import default_config
    from sameold_b200 import synth
    cfg = default_config(22050, samedec=True)
    plan = synth.plan_stream(900, 22050, 120.0)
    plan.burst_starts, plan.burst_payloads = [], []            # noise only: the AGC stays unlocked
    x = synth_cpu([plan], 120 * 22050, 22050, 1)[0]
    for guess in (None, 0.005, 3.0e-4):
        nb, bad, worst = agc_block_model(cfg, x, 2048, 1024, guess)
        assert nb > 1000 and bad == 0, (guess, nb, bad)
        assert 0 < worst < 700, worst
    nb, bad, _ = agc_block_model(cfg, np.zeros(30 * 22050, np.int16), 2048, 1024, None)
    assert bad == 0 and nb > 300
    # a warm-up that is too short is caught by the bitwise check (that is what the verification is for)
    nb, bad, _ = agc_block_model(cfg, x, 2048, 64, 0.005)
    assert bad > nb // 2
