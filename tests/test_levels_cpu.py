"""CPU checks of the properties the kernels rely on away from the corpus's operating point (no GPU):

* the band of noise levels where the long-stream path's speculative AGC hand-overs fail to verify (same_long.cu),
  on the oracle's model of that speculation;
* the exactness of the integer DC blocker (same_fast.cuh) at its bound: the reference's f32 recursion and the exact
  integer one agree bit for bit on the worst-case s16 inputs, and |D| stays below 2^24;
* the test-signal renderer of tests/test_levels_gpu.py: deterministic, and at the levels it claims."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from test_levels_gpu import HEADER, event_bursts, render, worst_dc_pattern  # noqa: E402

RATE = 22050


# ---------------------------------------------------------------------------------------------------------------------
# The AGC coalescence band
# ---------------------------------------------------------------------------------------------------------------------
def _model(cfg, x, guess):
    from oracle import agc_block_model
    return agc_block_model(cfg, x, 2048, 1024, guess)


def _guesses(cfg):
    """where the device's warm-up starts: the gain at the pass start (the stream's initial gain for the first pass),
    and the far limit"""
    from oracle import Oracle
    return (Oracle.derived(cfg)["agc_gain0"], cfg.agc_gain_max)


@pytest.mark.parametrize("sigma", [300, 500, 700])
def test_speculative_agc_hand_overs_fail_on_quiet_noise(sigma):
    """samedec limits [1/32767, 1/200]: between about -40 and -33 dBFS of noise the warm-started and the sequential
    gain trajectories do not meet bit for bit within the 1024-sample warm-up, so nearly every block fails its check"""
    from oracle.pyoracle import default_config
    cfg = default_config(RATE, samedec=True)
    x = render(60 * RATE, sigma=sigma, seed=sigma)
    for guess in _guesses(cfg):
        nb, bad, _ = _model(cfg, x, guess)
        assert nb == 645 and bad >= 0.9 * nb, (sigma, guess, nb, bad)


@pytest.mark.parametrize("sigma", [1, 30, 100, 220, 2000, 3663])
def test_speculative_agc_hand_overs_verify_outside_the_band(sigma):
    """below the band the gain is pinned at gmax; above it the trajectories coalesce within the warm-up"""
    from oracle.pyoracle import default_config
    cfg = default_config(RATE, samedec=True)
    x = render(60 * RATE, sigma=sigma, seed=sigma)
    for guess in _guesses(cfg):
        nb, bad, worst = _model(cfg, x, guess)
        assert nb == 645 and bad == 0, (sigma, guess, nb, bad)
        assert worst <= 1024


def test_speculative_agc_hand_overs_verify_on_the_recordings():
    from oracle import load_golden_recording
    from oracle.pyoracle import default_config
    cfg = default_config(RATE, samedec=True)
    for name in ("long_message", "npt", "two_and_two"):
        for guess in _guesses(cfg):
            nb, bad, _ = _model(cfg, load_golden_recording(name), guess)
            assert nb > 50 and bad == 0, (name, guess, nb, bad)


def test_speculative_agc_hand_overs_fail_with_library_default_limits():
    """gain limits [0, 1e6]: nothing pins the gain, and sigma 300 noise fails as well"""
    from oracle.pyoracle import default_config
    cfg = default_config(RATE, samedec=False)
    x = render(60 * RATE, sigma=300, seed=300)
    for guess in (None, 1.0 / 300):
        nb, bad, _ = _model(cfg, x, guess)
        assert bad >= 0.9 * nb, (guess, nb, bad)


# ---------------------------------------------------------------------------------------------------------------------
# The integer DC blocker at its bound
# ---------------------------------------------------------------------------------------------------------------------
def dc_exact(x, L=16):
    """dcblock.rs:45-49,104-108 in exact integers (Python ints): D = 256 * x[n-15] - S2, output = D / 256, with
    S1 = sum of the last L inputs (ff moving sum) and S2 = sum of the last L values of S1 (16 x fb moving sum)"""
    raw, s1h = [0] * L, [0] * L
    s1 = s2 = 0
    out = []
    for v in (int(t) for t in x):
        s1 += v - raw[0]
        raw = raw[1:] + [v]
        s2 += s1 - s1h[0]
        s1h = s1h[1:] + [s1]
        out.append((256 * raw[0] - s2, s1, s2))
    return out


def dc_float32(x, L=16):
    """the reference's recursion literally, in its operation order, in f32: per moving average
    aged = window.push(input); moving_sum += input - aged; avg = moving_sum * (1/L); delayed = window.front();
    then out = sig - 1.0 * ma1"""
    f = np.float32
    inv = f(1.0) / f(L)
    ffw, fbw = [f(0)] * L, [f(0)] * L
    ffs = fbs = f(0)
    out = []
    for v in (f(t) for t in x):
        aged = ffw[0]
        ffw = ffw[1:] + [v]
        ffs = f(ffs + f(v - aged))
        ma0 = f(ffs * inv)
        sig = ffw[0]
        aged1 = fbw[0]
        fbw = fbw[1:] + [ma0]
        fbs = f(fbs + f(ma0 - aged1))
        ma1 = f(fbs * inv)
        out.append((f(sig - f(f(1.0) * ma1)), ffs, fbs))
    return out


def dc_inputs():
    w, wn = worst_dc_pattern(1), worst_dc_pattern(-1)
    alt = np.tile(np.array([32767, -32768], np.int16), 200)
    steps = np.concatenate([np.full(50, -32768), np.full(50, 32767), np.full(37, -32768), np.full(3, 32767),
                            np.full(45, -32768)]).astype(np.int16)
    return {"worst +": np.concatenate([w, w, np.zeros(40, np.int16)]), "worst -": np.concatenate([wn, wn]),
            "alternating": alt, "steps": steps,
            "mixed": np.concatenate([alt[:33], w, steps, wn, alt[:7], w])}


@pytest.mark.parametrize("name", list(dc_inputs()))
def test_integer_dc_blocker_is_exact_at_its_bound(name):
    x = dc_inputs()[name]
    ex, fl = dc_exact(x), dc_float32(x)
    for n, ((D, s1, s2), (y, ffs, fbs)) in enumerate(zip(ex, fl)):
        assert abs(D) < 1 << 24 and abs(s2) < 1 << 24
        assert np.float32(D) == D                                          # the integer is exact in f32
        assert (np.float32(D) * np.float32(0.00390625)).view(np.uint32) == y.view(np.uint32), (name, n, D, y)
        assert np.float32(s1).view(np.uint32) == ffs.view(np.uint32)
        assert (np.float32(s2) * np.float32(0.0625)).view(np.uint32) == fbs.view(np.uint32)


def test_integer_dc_blocker_bound_is_reached():
    """max |D| over s16 input is 240 * 65535: x[n-15] has weight 256 - 16 = 240 and the other 30 samples of the
    window weights summing to 240, so one rail there and the other everywhere else"""
    for name in ("worst +", "worst -"):
        m = max(abs(D) for D, _, _ in dc_exact(dc_inputs()[name]))
        assert m == 240 * 65535 == 15728400
    rng = np.random.default_rng(4)
    x = rng.choice(np.array([-32768, 32767], np.int16), 20000)
    assert max(abs(D) for D, _, _ in dc_exact(x)) <= 15728400


# ---------------------------------------------------------------------------------------------------------------------
# The test-signal renderer
# ---------------------------------------------------------------------------------------------------------------------
def test_renderer_is_deterministic_and_at_its_levels():
    bursts = event_bursts(0.5 * RATE, 2000.0, n_eom=0)
    a = render(12 * RATE, bursts, 300.0, seed=4, dc=-700.0, dc_step=(9 * RATE, 1500.0))
    assert np.array_equal(a, render(12 * RATE, bursts, 300.0, seed=4, dc=-700.0, dc_step=(9 * RATE, 1500.0)))
    assert not np.array_equal(a, render(12 * RATE, bursts, 300.0, seed=5, dc=-700.0, dc_step=(9 * RATE, 1500.0)))
    end = int(np.ceil(bursts[-1][0] + len(HEADER) * 8 * RATE / 520.83))
    quiet = a[end + 100:9 * RATE].astype(np.float64)                    # noise + dc only
    assert abs(quiet.mean() + 700.0) < 10 and abs(quiet.std() - 300.0) < 5
    after = a[9 * RATE:].astype(np.float64)
    assert abs(after.mean() - 800.0) < 10
    b0 = int(bursts[0][0]) + 100
    tone = render(12 * RATE, bursts)[b0:b0 + RATE // 2].astype(np.float64)
    assert abs(np.sqrt(np.mean(tone ** 2)) - 2000.0 / np.sqrt(2)) < 15  # burst RMS = amplitude / sqrt 2
    # clipping: a full-scale burst driven x2 is clipped to the rails a large part of the time
    od = render(3 * RATE, [(0.0, HEADER, 65534.0, 520.83)])[: RATE]
    frac = np.mean((od == 32767) | (od == -32768))
    assert 0.5 < frac < 0.8, frac
    assert np.mean(np.abs(render(3 * RATE, [(0.0, HEADER, 32767.0, 520.83)])[: RATE]) >= 32767) < 0.05
    # off-rate bursts last 1 / (1 + deviation) as long
    fast = render(4 * RATE, [(0.0, HEADER, 1000.0, 520.83 * 1.02)])
    assert abs(np.flatnonzero(fast)[-1] + 1 - np.ceil(len(HEADER) * 8 * RATE / (520.83 * 1.02))) <= 1
    # splices land where asked and the worst-case pattern is what the DC bound needs
    s = render(1000, splice=[(100, worst_dc_pattern(1))])
    assert s[115] == 32767 and np.all(s[100:115] == -32768) and np.all(s[116:131] == -32768) and not s[131:].any()
