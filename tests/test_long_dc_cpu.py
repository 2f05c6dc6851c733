"""The long-stream path's DC front at general geometry (sameold_b200/csrc/same_long.cu, "A, general") restated in
numpy, checked bit for bit against the literal f32 recursion of dcblock.rs:45-49,104-108 (as same_rx_generic_kernel and
same_rx_wide_kernel run it) for s16 input:

  ffsum[n] = D + (x[n-L+1] + ... + x[n])          integer, time-parallel
  ma0[n]   = ffsum[n] * inv_len                   time-parallel
  fbsum[n] = fbsum[n-1] + (ma0[n] - ma0[n-L])     the one sequential scan
  d[n]     = x[n-L+1] - gate * (fbsum[n] * inv_len)

and the DC state a commit writes at any position p, from the windows the chunk started with where p < L.  Signed
zeros are compared too (bits, not values)."""
import numpy as np
import pytest

F = np.float32
LENGTHS = [8, 32, 35, 70, 84, 140, 368, 512]


def literal(x, L, state=None):
    """the reference recursion over s16 samples x from `state` = (ff window, fb window, ffsum, fbsum) (None: reset):
    (d [len(x)] f32, state after the last sample)"""
    if state is None:
        ff, fb, ffsum, fbsum = [F(0)] * L, [F(0)] * L, F(0), F(0)
    else:
        ff, fb, ffsum, fbsum = list(state[0]), list(state[1]), state[2], state[3]
    inv, gate = F(1) / F(L), F(1) if L > 1 else F(0)
    d = np.empty(len(x), F)
    hf = hb = 0   # ring heads: oldest entries
    for n, xi in enumerate(x):
        v = F(int(xi))
        aged = ff[hf]
        ff[hf] = v
        hf = (hf + 1) % L
        ffsum = F(ffsum + F(v - aged))
        ma0 = F(ffsum * inv)
        sig = ff[hf]                              # oldest after the push: x[n - L + 1]
        aged2 = fb[hb]
        fb[hb] = ma0
        hb = (hb + 1) % L
        fbsum = F(fbsum + F(ma0 - aged2))
        d[n] = F(sig - F(gate * F(fbsum * inv)))
    rot = lambda w, h: np.array(w[h:] + w[:h], F)
    return d, (rot(ff, hf), rot(fb, hb), ffsum, fbsum)


def decomposed(x, L, state=None):
    """the same by the three phases: (d, ma0, fbsum, commit) with commit(p) the state after sample p - 1"""
    if state is None:
        state = (np.zeros(L, F), np.zeros(L, F), F(0), F(0))
    ff0, fb0, ffsum0, fbsum0 = state
    inv, gate = F(1) / F(L), F(1) if L > 1 else F(0)
    n = len(x)
    xe = np.concatenate([ff0.astype(np.int64), np.asarray(x, np.int64)])          # x[m] at xe[m + L]
    D = int(np.rint(ffsum0)) - int(ff0.astype(np.int64).sum())
    c = np.concatenate([[0], np.cumsum(xe)])
    ffsum = D + (c[L + 1:] - c[1:n + 1])                                          # sum xe[n+1 .. n+L] = x[n-L+1 .. n]
    assert np.all(np.abs(ffsum) <= 1 << 24)
    ma0 = ffsum.astype(F) * inv                                                   # exact conversion, one rounding
    ma0e = np.concatenate([fb0, ma0])                                             # ma0[m] at ma0e[m + L]
    delta = ma0 - ma0e[:n]
    fbsum = np.empty(n, F)
    f = F(fbsum0)
    for i in range(n):
        f = F(f + delta[i])
        fbsum[i] = f
    sig = xe[1:n + 1].astype(F)                                                   # x[n - L + 1]
    d = sig - gate * (fbsum * inv)

    def commit(p):
        assert 1 <= p <= n
        w = xe[p:p + L]                                                           # x[p-L .. p-1]
        return w.astype(F), ma0e[p:p + L].copy(), F(D + int(w.sum())), fbsum[p - 1]

    return d, ma0, fbsum, commit


def signals(n, seed):
    rng = np.random.default_rng(seed)
    alt = np.tile(np.array([32767, -32768], np.int16), n // 2 + 1)[:n]
    steps = np.where((np.arange(n) // 97) % 2 == 0, 32767, -32768).astype(np.int16)
    dc = np.clip(np.rint(20000 * np.sign(np.sin(np.arange(n) / 300.0) + 1e-9) + rng.normal(0, 3000, n)), -32768, 32767)
    noise = np.clip(np.rint(rng.normal(0, 3663, n)), -32768, 32767)
    zeros_then = np.concatenate([np.zeros(n // 3), rng.integers(-32768, 32768, n - n // 3)])
    return {"full-scale alternation": alt, "rail-to-rail steps": steps, "dc +-20000": dc.astype(np.int16),
            "noise": noise.astype(np.int16), "zeros then uniform": zeros_then.astype(np.int16)}


def bits(a):
    return np.asarray(a, F).view(np.uint32)


def same_state(a, b):
    return all(np.array_equal(bits(u), bits(v)) for u, v in zip(a, b))


@pytest.mark.parametrize("L", LENGTHS)
@pytest.mark.parametrize("start", ["reset", "mid-stream"])
def test_three_phase_dc_equals_the_literal_recursion(L, start):
    n = 3 * L + 700
    for name, sig in signals(2 * n, L).items():
        state = None
        if start == "mid-stream":
            _, state = literal(sig[:n], L)
        x = sig[n:] if start == "mid-stream" else sig[:n]
        want_d, want_state = literal(x, L, state)
        d, ma0, fbsum, commit = decomposed(x, L, state)
        assert np.array_equal(bits(d), bits(want_d)), f"L={L}, {name}, {start}: d differs"
        assert same_state(commit(len(x)), want_state), f"L={L}, {name}, {start}: state at the end"
        for p in sorted({1, L // 2 + 1, L - 1, L, L + 1, 2 * L + 3, len(x) - 1} - {0}):
            _, want_p = literal(x[:p], L, state)
            assert same_state(commit(p), want_p), f"L={L}, {name}, {start}: state at {p}"


def test_fbsum_leaves_the_exact_range():
    """the cases the scan is for: at L = 32 |fbsum| exceeds 2^19 (off the 1/32 grid), and at L = 35 inv_len is not
    dyadic, so an integer restatement of the feedback sum would differ from the reference"""
    for L in (32, 35):
        x = np.full(4 * L, 32767, np.int16)
        _, ma0, fbsum, _ = decomposed(x, L)
        if L == 32:
            assert np.max(np.abs(fbsum)) > 2 ** 19
        else:
            exact = np.cumsum(ma0.astype(np.float64) - np.concatenate([np.zeros(L), ma0[:-L].astype(np.float64)]))
            assert not np.array_equal(fbsum.astype(np.float64), exact)
