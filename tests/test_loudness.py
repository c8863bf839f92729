"""CPU tests of loudness normalisation (no GPU): a float64 numpy / scipy reference of the kkx.h "loudness_target" rules
(K-weighting, 400 ms gating, 4x true peak, the gain rule), checked against the BS.1770-4 coefficient table and known
answers, and the filters the library designs (kkx_test_loudness_design) against that reference.  The GPU tests in
test_loudness_gpu.py compare the kernels and the model's output with the same reference."""
import ctypes as C
import math

import numpy as np
import pytest
from scipy.signal import firwin, freqz, lfilter, resample_poly

# ITU-R BS.1770-4, Table 1 and 2 (fs = 48 kHz): pre-filter (shelf) and RLB high-pass
BS1770_48K = ((1.53512485958697, -2.69169618940638, 1.19839281085285, -1.69065929318241, 0.73248077421585),
              (1.0, -2.0, 1.0, -1.99004745483398, 0.99007225036621))


def kweight_design(fs):
    """The two K-weighting biquads ((b, a), (b, a)) in float64: libebur128's analog parameters, bilinear transform."""
    f0, G, Q = 1681.974450955533, 3.999843853973347, 0.7071752369554196
    K = math.tan(math.pi * f0 / fs)
    Vh = 10.0 ** (G / 20.0)
    Vb = Vh ** 0.4996667741545416
    a0 = 1.0 + K / Q + K * K
    shelf = (np.array([(Vh + Vb * K / Q + K * K) / a0, 2.0 * (K * K - Vh) / a0, (Vh - Vb * K / Q + K * K) / a0]),
             np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0]))
    f0, Q = 38.13547087602444, 0.5003270373238773
    K = math.tan(math.pi * f0 / fs)
    a0 = 1.0 + K / Q + K * K
    hp = (np.array([1.0, -2.0, 1.0]), np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0]))
    return shelf, hp


def kweight(x, fs=24000):
    (b1, a1), (b2, a2) = kweight_design(fs)
    return lfilter(b2, a2, lfilter(b1, a1, np.asarray(x, np.float64)))


def block_energies(x, fs=24000):
    """z_j of every whole 400 ms block on a 100 ms hop from sample 0."""
    y = kweight(x, fs)
    blk, hop = int(0.4 * fs), int(0.1 * fs)
    n = (len(y) - blk) // hop + 1 if len(y) >= blk else 0
    c = np.concatenate([[0.0], np.cumsum(y * y)])
    return np.array([(c[j * hop + blk] - c[j * hop]) / blk for j in range(n)])


def loudness_ref(x, fs=24000):
    """Integrated loudness L (LUFS) with BS.1770-4 gating; NaN when no block passes."""
    z = block_energies(x, fs)
    with np.errstate(divide="ignore"):
        l = -0.691 + 10.0 * np.log10(z)
    a = l > -70.0
    if not a.any():
        return float("nan")
    rel = -0.691 + 10.0 * math.log10(z[a].mean()) - 10.0
    g = a & (l > rel)
    return -0.691 + 10.0 * math.log10(z[g].mean())


def true_peak_ref(x):
    """max |resample_poly(x, 4, 1)| (scipy's default Kaiser filter, zeros outside the item)."""
    x = np.asarray(x, np.float64)
    return float(np.abs(resample_poly(x, 4, 1)).max()) if len(x) else 0.0


def gain_ref(L, tp, target, ceiling):
    if math.isnan(L):
        return 1.0
    g = 10.0 ** ((target - L) / 20.0)
    cap = 10.0 ** (ceiling / 20.0)
    if tp * g > cap:
        g = cap / tp
    return g


def tone(n, fs, f=997.0, dbfs_rms=-23.0, phase=0.0):
    a = math.sqrt(2.0) * 10.0 ** (dbfs_rms / 20.0)
    return a * np.sin(2 * np.pi * f * np.arange(n) / fs + phase)


@pytest.fixture(scope="module")
def lib():
    from kokorox_b200 import build
    build.build()
    from kokorox_b200.onn import load_library
    return load_library()


def lib_design(lib, fs):
    kw = np.zeros(10, np.float64)
    n = lib.kkx_test_loudness_design(fs, kw.ctypes.data_as(C.POINTER(C.c_double)), None, 0)
    taps = np.zeros(n, np.float32)
    assert lib.kkx_test_loudness_design(fs, None, taps.ctypes.data_as(C.POINTER(C.c_float)), n) == n
    return kw, taps


def test_kweighting_at_48k_is_the_bs1770_table(lib):
    kw, _ = lib_design(lib, 48000.0)
    want = np.array(BS1770_48K[0] + BS1770_48K[1])
    assert np.abs(kw - want).max() <= 1e-12
    # the numpy design agrees with the table too
    (b1, a1), (b2, a2) = kweight_design(48000)
    assert np.abs(np.concatenate([b1, a1[1:], b2, a2[1:]]) - want).max() <= 1e-12


def test_kweighting_at_24k_matches_the_numpy_design(lib):
    kw, _ = lib_design(lib, 24000.0)
    (b1, a1), (b2, a2) = kweight_design(24000)
    assert np.abs(kw - np.concatenate([b1, a1[1:], b2, a2[1:]])).max() <= 1e-12


def test_true_peak_taps_are_scipy_resample_poly_4_1(lib):
    _, taps = lib_design(lib, 24000.0)
    want = (4 * firwin(81, 0.25, window=("kaiser", 5.0))).astype(np.float32)
    assert len(taps) == 81
    ulp = np.spacing(np.abs(want)).astype(np.float64)
    assert np.all(np.abs(taps.astype(np.float64) - want.astype(np.float64)) <= ulp)
    assert np.array_equal(taps, taps[::-1])


def test_997hz_sine_at_minus_23_dbfs():
    assert abs(loudness_ref(tone(20 * 48000, 48000), 48000) - (-23.0)) <= 0.01
    # at 24 kHz the bilinear transform warps the shelf: -22.97
    assert abs(loudness_ref(tone(20 * 24000, 24000), 24000) - (-22.97)) <= 0.01


def test_silence_after_a_tone_does_not_count():
    t = tone(10 * 24000, 24000)
    short = np.concatenate([t, np.zeros(24000)])
    long = np.concatenate([t, np.zeros(10 * 24000)])
    # blocks of silence alone fail the absolute gate; only the 3 blocks that straddle the edge differ from the tone
    assert loudness_ref(short) == loudness_ref(long)
    assert abs(loudness_ref(long) - loudness_ref(t)) <= 0.1


def test_relative_gate_drops_a_quiet_part():
    fs, f = 24000, 997.0
    na = 20 * fs                      # 20 s at -20 dBFS, then 20 s at -40 dBFS (phase-continuous)
    x = np.concatenate([tone(na, fs, f, -20.0), tone(na, fs, f, -40.0, 2 * np.pi * f * na / fs)])
    (b1, a1), (b2, a2) = kweight_design(fs)
    h2 = abs(freqz(b1, a1, [f], fs=fs)[1][0] * freqz(b2, a2, [f], fs=fs)[1][0]) ** 2
    za = 10.0 ** (-20.0 / 10.0) * h2          # steady K-weighted mean square of the loud part
    zb = za / 100.0
    blk, hop = int(0.4 * fs), int(0.1 * fs)
    n_loud = (na - blk) // hop + 1            # blocks inside the loud part
    straddle = [za * (k / 4) + zb * (1 - k / 4) for k in (3, 2, 1)]
    # every quiet-only block is 20 LU below the loud ones, beyond the 10 LU relative gate; the straddling ones are not
    want = -0.691 + 10 * math.log10((n_loud * za + sum(straddle)) / (n_loud + 3))
    got = loudness_ref(x)
    assert abs(got - want) <= 0.01
    assert got > -20.0 - 0.691 + 10 * math.log10(h2) - 0.1     # nowhere near the -30 LUFS an ungated mean would give


@pytest.mark.parametrize("n", (1, 9599))
def test_short_items_are_undefined(n):
    assert math.isnan(loudness_ref(tone(n, 24000)))
    assert gain_ref(loudness_ref(tone(n, 24000)), 0.1, -16.0, -1.0) == 1.0


def test_silence_is_undefined():
    assert math.isnan(loudness_ref(np.zeros(5 * 24000)))
    assert true_peak_ref(np.zeros(100)) == 0.0


def test_true_peak_exceeds_sample_peak_near_fs_over_4():
    # a 6 kHz tone (fs / 4) sampled 45 degrees off its crests: every sample is at 0.707 of the peak
    fs = 24000
    x = 0.5 * np.sin(2 * np.pi * 6000 * np.arange(fs) / fs + np.pi / 4)
    assert np.abs(x).max() < 0.36
    assert true_peak_ref(x) > 0.49


def test_gain_rule():
    # not peak-limited: -20 LUFS with peak 0.1 to -23 LUFS
    assert gain_ref(-20.0, 0.1, -23.0, -1.0) == pytest.approx(10 ** (-3 / 20), rel=1e-15)
    # peak-limited: -30 LUFS with peak 0.5 to -16 LUFS would peak at 2.5; the ceiling -1 dBTP wins
    g = gain_ref(-30.0, 0.5, -16.0, -1.0)
    assert g == pytest.approx(10 ** (-1 / 20) / 0.5, rel=1e-15)
    assert 0.5 * g <= 10 ** (-1 / 20) * (1 + 1e-15)
    # a 0 dBTP ceiling and an exact fit
    assert gain_ref(-20.0, 10 ** (-3 / 20), -17.0, 0.0) == pytest.approx(10 ** (3 / 20), rel=1e-12)
    assert gain_ref(float("nan"), 0.9, -16.0, -1.0) == 1.0
    # vector form as the GPU tests use it
    L = np.array([-20.0, -30.0, float("nan")])
    tp = np.array([0.1, 0.5, 0.3])
    g = np.array([gain_ref(a, b, -23.0, -1.0) for a, b in zip(L, tp)])
    assert g[0] == pytest.approx(10 ** (-3 / 20)) and g[1] == pytest.approx(10 ** (-1 / 20) / 0.5) and g[2] == 1.0
