"""CPU tests of the lookahead true-peak limiter (no GPU): a float64 numpy / scipy reference of the kkx.h "limiter"
rule (steps 1-8) built on test_loudness.py's loudness and true-peak references, checked against known answers.  The
GPU tests in test_limiter_gpu.py compare the kernels and the model's output with the same reference."""
import math

import numpy as np
from scipy.ndimage import minimum_filter1d
from scipy.signal import resample_poly

from tests.test_loudness import loudness_ref, tone, true_peak_ref

HA, HB, RMAX, SLOPE = 120, 10, 12.0, 0.0025     # lookahead, FIR guard (samples), largest reduction, release (dB / sample)
W = int(round(RMAX / SLOPE))                    # release window: 4800 samples


def static_gain_ref(x, target, ceiling):
    """Step 1: (L, tp, g) -- the loudness gain when target != 0 and L is defined, capped at Rmax above the ceiling."""
    L = loudness_ref(x) if len(x) else float("nan")
    tp = true_peak_ref(x)
    g = 1.0
    if target != 0 and not math.isnan(L):
        g = 10.0 ** ((target - L) / 20.0)
    cap = 10.0 ** ((ceiling + RMAX) / 20.0)
    if tp * g > cap:
        g = cap / tp
    return L, tp, g


def envelope_ref(x, g, ceiling):
    """Steps 2-5 in float64: (q, e, G) over the item's samples."""
    x = np.asarray(x, np.float64)
    n = len(x)
    p = np.abs(resample_poly(x, 4, 1)).reshape(n, 4).max(axis=1)
    q = np.zeros(n)
    nz = p > 0
    q[nz] = np.minimum(0.0, ceiling - 20.0 * np.log10(g * p[nz]))
    # h[m] = min of q over [m - Hb, m + Ha + Hb] for m in [-o, n) (o = Ha + Hb: the lookahead reaches before the
    # item's start), q = 0 outside [0, n)
    o = HA + HB
    size = HA + 2 * HB + 1
    h = minimum_filter1d(np.concatenate([np.zeros(o), q]), size, mode="constant", cval=0.0, origin=-(size // 2 - HB))
    m = np.arange(-o, n, dtype=np.float64)
    # e[i] = min(0, min over m in [i - W, i] of h[m] + (i - m) s); older terms are >= 0 since h >= -Rmax
    e = np.minimum(0.0, m * SLOPE + np.minimum.accumulate(h - m * SLOPE))[o:]
    E = np.concatenate([np.ones(HA), 10.0 ** (e / 20.0)])                    # e = 0 before the first sample
    c = np.concatenate([[0.0], np.cumsum(E)])
    G = (c[HA + 1:] - c[: n]) / (HA + 1)
    return q, e, G


def limiter_ref(x, target, ceiling):
    """Steps 1-7 for one item of float32 samples: g, G, v (float32), t and the report (max reduction dB, dBTP)."""
    x = np.asarray(x, np.float32)
    L, tp, g = static_gain_ref(x.astype(np.float64), target, ceiling)
    q, e, G = envelope_ref(x, g, ceiling)
    v = x * (g * G).astype(np.float32)
    tpv = true_peak_ref(v)
    c = 10.0 ** (ceiling / 20.0)
    t = min(1.0, c / tpv) if tpv > 0 else 1.0
    red = -20.0 * math.log10(t * G.min()) if len(G) else 0.0
    out_db = 20.0 * math.log10(t * tpv) if tpv > 0 else -math.inf
    return dict(L=L, tp=tp, g=g, q=q, e=e, G=G, v=v, t=t, red=red, out_db=out_db)


def output_ref(x, target, ceiling):
    """Step 8 at 24 kHz: the returned float32 samples fp32(v t)."""
    r = limiter_ref(x, target, ceiling)
    return (r["v"] * np.float32(r["t"])).astype(np.float32), r


def speech_with_transients(n, seed):
    """Speech-like noise (test_loudness_gpu.py's generator, its noise clipped at 3 sigma so that the body has a speech-
    like crest factor) plus a 2 ms burst every 2 s: a peak-to-loudness ratio near 20 dB, in the range of unprocessed
    speech."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 24000.0
    env = np.maximum(np.sin(2 * np.pi * 3.1 * t + seed), 0.0) ** 2 + 0.02
    x = 0.1 * env * np.clip(rng.standard_normal(n), -3.0, 3.0)
    k = np.arange(48)
    for s in range(6000, n - 100, 48000):
        x[s:s + 48] += 0.6 * np.sin(2 * np.pi * 2000 * k / 24000) * np.hanning(48)
    return x.astype(np.float32)


def test_tone_under_the_ceiling_is_untouched():
    x = tone(48000, 24000, dbfs_rms=-23.0).astype(np.float32)
    r = limiter_ref(x, -23.0, -1.0)
    assert abs(r["L"] - (-23.0)) < 1.0
    assert np.all(r["G"] == 1.0) and r["t"] == 1.0 and r["red"] == 0.0
    assert np.all(r["v"] == (x * np.float32(r["g"])))


def test_isolated_click_on_a_tone():
    n, c0 = 48000, 24000
    x = tone(n, 24000, dbfs_rms=-40.0)
    x[c0] += 0.9
    x = x.astype(np.float32)
    ceiling = -6.0
    r = limiter_ref(x, 0.0, ceiling)
    q, e, G = r["q"], r["e"], r["G"]
    assert r["g"] == 1.0
    qmin = q.min()
    assert abs(int(np.argmin(q)) - c0) <= 1 and qmin < -5.0
    # the reduction starts no earlier than Ha + 2 Hb samples before the click
    first = int(np.flatnonzero(G < 1.0)[0])
    assert first >= c0 - HA - 2 * HB, (first, c0)
    assert np.all(G[: c0 - HA - 2 * HB] == 1.0)
    # full depth over the click's FIR support (its true-peak filter reaches Hb samples either side)
    depth = 10.0 ** (qmin / 20.0)
    span = slice(c0 - HB, c0 + HB + 1)
    assert np.allclose(G[span], depth, rtol=0, atol=1e-12)
    np.testing.assert_allclose(e[span], qmin, rtol=0, atol=1e-9)
    # after the hold, e recovers at exactly s dB per sample until it is back at 0
    m = int(np.argmin(q)) + HB
    k = int(-qmin / SLOPE) - 1
    np.testing.assert_allclose(np.diff(e[m: m + k]), SLOPE, rtol=0, atol=1e-9)
    assert np.all(e[m + k + 2:] > -1e-9)
    # the ceiling holds and the report says what happened
    y, r = output_ref(x, 0.0, ceiling)
    assert true_peak_ref(y) <= 10.0 ** (ceiling / 20.0) * (1 + 1e-6)
    assert r["red"] > 5.0 and abs(r["out_db"] - 20 * math.log10(true_peak_ref(y))) < 1e-4


def test_speech_with_transients_reaches_the_streaming_target():
    # measured with this reference: L = -23.97 LUFS, true peak -3.20 dBTP (PLR 20.8 dB); the static rule lands at
    # -21.77 LUFS (7.8 LU short of -14), the limiter at -14.71 LUFS with its true peak at -1.00 dBTP (max reduction
    # 7.77 dB)
    x = speech_with_transients(24000 * 12, 3)
    target, ceiling = -14.0, -1.0
    L, tp = loudness_ref(x.astype(np.float64)), true_peak_ref(x)
    plr = 20 * math.log10(tp) - L
    assert 18.0 <= plr <= 22.0, plr
    cap = 10.0 ** (ceiling / 20.0)
    g_static = min(10.0 ** ((target - L) / 20.0), cap / tp)
    L_static = loudness_ref((x * g_static).astype(np.float64))
    assert L_static < target - 4.0, L_static
    y, r = output_ref(x, target, ceiling)
    L_out = loudness_ref(y.astype(np.float64))
    assert abs(L_out - target) <= 1.0, L_out
    assert 20 * math.log10(true_peak_ref(y)) <= ceiling + 1e-4
    assert r["red"] > 0.0


def test_without_normalisation_only_the_ceiling_is_enforced():
    x = (1.5 * np.sin(2 * np.pi * 440 * np.arange(24000) / 24000)).astype(np.float32)
    y, r = output_ref(x, 0.0, -1.0)
    assert r["g"] == 1.0 and r["red"] > 4.0
    assert true_peak_ref(y) <= 10.0 ** (-1.0 / 20.0) * (1 + 1e-6)
    z = np.zeros(5000, np.float32)
    y, r = output_ref(z, 0.0, -1.0)
    assert np.all(y == 0.0) and r["red"] == 0.0 and r["t"] == 1.0


def test_static_cap_is_rmax_above_the_ceiling():
    x = np.zeros(24000, np.float32)
    x[12000] = 1.0
    L, tp, g = static_gain_ref(x.astype(np.float64), 0.0, -20.0)
    assert abs(20 * math.log10(tp * g) - (-20.0 + RMAX)) < 1e-9
    q, e, G = envelope_ref(x, g, -20.0)
    assert abs(q.min() + RMAX) < 1e-9
