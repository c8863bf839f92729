"""GPU tests (-m gpu): the signal-path kernels in isolation -- harmonic source (K9), STFT (K10), iSTFT head (K11),
duration head and length regulator (K4/K5), pool_up, conv_post (tensor-core configuration), curve_conv and
add_rows_stats -- against float64 references, or against the oracle's own fp32 arithmetic where that arithmetic is
the contract.  Items are packed with NaN gap rows and every output buffer carries sentinels, so that stray reads and
writes show.  Hooks: include/kkx_test.h."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from tests.test_signal_ops import (STFT_BOUND_C, emulate_phase_upsampling, istft_reference, level,  # noqa: E402
                                   stft_reference)

pytestmark = pytest.mark.gpu

GAP = 32
SENT = np.float32(-777.0)        # sentinel of output buffers: a kernel that writes outside its items changes it
NAN = np.float32("nan")


@pytest.fixture(scope="module")
def lib():
    from kokorox_b200.onn import load_library
    lib = load_library()
    lib.kkx_test_last_error.restype = C.c_char_p
    lib.kkx_test_durations.restype = C.c_int64
    return lib


def ptr(a, t=C.c_float):
    return None if a is None else a.ctypes.data_as(C.POINTER(t))


def i32(a):
    return np.ascontiguousarray(a, dtype=np.int32)


def i64(a):
    return np.ascontiguousarray(a, dtype=np.int64)


def ok(lib, rc):
    assert rc == 0, lib.kkx_test_last_error()


def bf16_bits(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16)


def bf16_round(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


# ============================================================================ K9 harmonic source
def run_sine(lib, f0s, noise=None, seed=0, lin_w=None, lin_b=0.0, want_phase=True):
    """f0s: list of per-item coarse curves (L_b = 2T_b) -> (phase list [9][L_b], har list [300 L_b])."""
    lens = [len(f) for f in f0s]
    off, rows = level(lens)
    f0 = np.full(rows, NAN, np.float32)
    for o, f in zip(off, f0s):
        f0[o:o + len(f)] = f
    lw = np.asarray(lin_w, np.float32)
    lb = np.asarray([lin_b], np.float32)
    nph, ns = 9 * sum(lens), 300 * sum(lens)
    phase = np.full(nph, SENT, np.float32) if want_phase else None
    har = np.full(ns, SENT, np.float32)
    nz = None if noise is None else np.ascontiguousarray(noise, np.float32).reshape(-1)
    ok(lib, lib.kkx_test_sine_source(0, ptr(f0), rows, len(lens), ptr(i32(off), C.c_int), ptr(i32(lens), C.c_int), ptr(nz),
                                     C.c_int64(0 if nz is None else nz.size), C.c_uint64(seed), ptr(lw), ptr(lb),
                                     ptr(phase), ptr(har)))
    phs, hs, p, s = [], [], 0, 0
    for L in lens:
        if want_phase:
            phs.append(phase[p:p + 9 * L].reshape(9, L))
        hs.append(har[s:s + 300 * L])
        p += 9 * L
        s += 300 * L
    return phs, hs


def oracle_source(f0, noise, lin_w, lin_b):
    """KokoroOracle.harmonic_source on a weight dict holding only m_source.l_linear, and the coarse phase its lines
    compute on the way (cumsum(rad) * 2 pi * 300, fp32), mirrored line for line."""
    from oracle.kokoro_ref import HOP_F0, N_HARM, SAMPLE_RATE, KokoroOracle
    o = KokoroOracle({"decoder.generator.m_source.l_linear.weight": np.asarray(lin_w, np.float32).reshape(1, 9),
                      "decoder.generator.m_source.l_linear.bias": np.asarray([lin_b], np.float32)})
    f = torch.from_numpy(np.asarray(f0, np.float32))
    with torch.no_grad():
        f0_up = f.repeat_interleave(HOP_F0).view(1, -1, 1)
        fn = f0_up * torch.arange(1, N_HARM + 1, dtype=torch.float32).view(1, 1, -1)
        rad = (fn / SAMPLE_RATE) % 1
        del fn, f0_up
        rad = F.interpolate(rad.transpose(1, 2), scale_factor=1 / HOP_F0, mode="linear").transpose(1, 2)
        coarse = ((torch.cumsum(rad, dim=1) * 2 * np.pi).transpose(1, 2) * HOP_F0)[0].numpy().copy()   # [9, L]
        del rad
        har = None
        if noise is not None:
            har = o.harmonic_source(f, torch.from_numpy(np.asarray(noise, np.float32).reshape(-1, 9))).numpy().copy()
    return coarse, har


def f0_profile(kind, L, seed):
    rng = np.random.default_rng(seed)
    if kind == "zero":
        return np.zeros(L, np.float32)
    if kind == "ten":            # exactly at the voicing edge: f > 10 is false
        return np.full(L, 10.0, np.float32)
    if kind == "negative":       # the python-style % 1 of negative numbers
        return (-rng.uniform(0, 400, L)).astype(np.float32)
    t = np.arange(L) / 200.0     # speech-like contour 50..500 Hz with unvoiced stretches and exact zeros
    f = 275 + 225 * np.sin(2 * np.pi * (0.3 * t + rng.uniform())) * np.cos(2 * np.pi * 0.07 * t)
    f = f + rng.normal(0, 5, L)
    f[(np.arange(L) // 37) % 5 == 0] = 0.0
    return np.clip(f, 50, 500).astype(np.float32) * (f > 0)


# T = 1, 128, 129: L = 2T around the 256-wide scan chunk; 1000: the parity length; 14 500: 8.7 M samples (past 2^23);
# 28 500: 17.1 M samples (past 2^24: (float)n is no longer exact)
@pytest.mark.parametrize("T,kind", [(1, "contour"), (128, "contour"), (129, "negative"), (64, "zero"), (64, "ten"),
                                    (1000, "contour"), (14500, "contour"), (28500, "contour")])
def test_sine_source_matches_oracle(lib, T, kind):
    L = 2 * T
    f0 = f0_profile(kind, L, seed=T)
    rng = np.random.default_rng(T + 1)
    noise = rng.standard_normal((300 * L, 9)).astype(np.float32)
    lin_w = rng.uniform(-0.6, 0.6, 9).astype(np.float32)
    lin_b = np.float32(0.05)
    (ph,), (har,) = run_sine(lib, [f0], noise, lin_w=lin_w, lin_b=lin_b)
    coarse, ref = oracle_source(f0, noise, lin_w, lin_b)
    # coarse phase: the kernel's fp64 scan adds in another order than torch's sequential double cumsum, so a flip of
    # the fp32 rounding is possible in principle; the count of such flips is zero at every length tested
    flips = int((ph.view(np.uint32) != coarse.view(np.uint32)).sum())
    assert flips == 0, f"{flips} coarse phases differ from the oracle's fp32 cumsum(rad) * 2 pi * 300"
    # har_source: the interpolated phase is the oracle's bit for bit (tests/test_signal_ops.py), sin_reduced is within
    # 2e-7 of sin, scaled by 0.1 -> 2e-8; Linear(9 -> 1) in another order than torch's: <= 9 * 2^-24 * sum |w_h v_h|
    # ~ 3e-8; tanhf vs torch.tanh: 2 ulp of |out| <= 1 -> 2.4e-7.  Sum: 3e-7; the bound is 1e-6.
    err = np.abs(har.astype(np.float64) - ref).max()
    print(f"T={T} {kind}: har_source max err {err:.2e}, phase max {np.abs(coarse).max():.3e} rad")
    assert err <= 1e-6


def test_sine_source_ragged_batch(lib):
    """A ragged batch is the items run alone, bit for bit (noise injected: one buffer all items read from offset 0)."""
    Ts = [129, 1, 700, 64]
    f0s = [f0_profile("contour", 2 * T, seed=10 + T) for T in Ts]
    noise = np.random.default_rng(3).standard_normal((300 * 2 * max(Ts), 9)).astype(np.float32)
    lin_w = np.random.default_rng(4).uniform(-0.6, 0.6, 9).astype(np.float32)
    phs, hs = run_sine(lib, f0s, noise, lin_w=lin_w, lin_b=0.01)
    for f0, ph, h in zip(f0s, phs, hs):
        (p1,), (h1,) = run_sine(lib, [f0], noise, lin_w=lin_w, lin_b=0.01)
        assert np.array_equal(ph, p1) and np.array_equal(h, h1)
        coarse, ref = oracle_source(f0, noise[:300 * len(f0)], lin_w, np.float32(0.01))
        assert np.array_equal(ph.view(np.uint32), coarse.view(np.uint32))
        assert np.abs(h.astype(np.float64) - ref).max() <= 1e-6


def test_sin_reduced_bound_at_large_phases(lib):
    """uv = 1, noise 0, one-hot lin_w: out = tanhf(fp32(0.1 sin_reduced(phi))), so atanh(out) / 0.1 recovers
    sin_reduced(phi) of the interpolated fp32 phase phi (emulated bit for bit, tests/test_signal_ops.py).  f0 = 2666 Hz
    makes harmonic 9 advance 0.99975 turns per sample, so phases reach 1.3e7 rad.
    Bound: the claim (2e-7) + the recovery: tanhf 2 ulp and the 0.1 product half an ulp at |out| < 0.125 (ulp 7.45e-9)
    -> 2.5 * 7.45e-9 / 0.1 = 1.9e-7 -> 3.9e-7."""
    T = 3000
    L = 2 * T
    f0 = np.full(L, 2666.0, np.float32)
    f0[::7] = 1234.5
    noise = np.zeros((300 * L, 9), np.float32)
    worst = 0.0
    ph_all = None
    for h in (0, 4, 8):
        lw = np.zeros(9, np.float32)
        lw[h] = 1.0
        (ph,), (out,) = run_sine(lib, [f0], noise, lin_w=lw, lin_b=0.0)
        phi = emulate_phase_upsampling(ph[h], 300)
        s_got = np.arctanh(out.astype(np.float64)) / 0.1
        e = np.abs(s_got - np.sin(phi.astype(np.float64))).max()
        worst = max(worst, e)
        ph_all = phi
    print(f"sin_reduced: max recovered error {worst:.2e} at phases up to {np.abs(ph_all).max():.2e} rad")
    assert np.abs(ph_all).max() > 1e7
    assert worst <= 3.9e-7


def production_noise(lib, seed, S_items, slot=0):
    """The on-device N(0, 1) noise of every harmonic for items of S_items[b] samples (f0 = 0: uv = 0, amplitude
    fp32(0.1 / 3)); returns per harmonic the noise of item `slot`.  One-hot lin_w, so out = tanhf(namp * z)."""
    namp = np.float64(np.float32(np.float32(0.1) / np.float32(3.0)))
    f0s = [np.zeros(S // 300, np.float32) for S in S_items]
    z = []
    for h in range(9):
        lw = np.zeros(9, np.float32)
        lw[h] = 1.0
        _, hs = run_sine(lib, f0s, None, seed=seed, lin_w=lw, lin_b=0.0, want_phase=False)
        z.append(np.arctanh(hs[slot].astype(np.float64)) / namp)
    return np.stack(z)           # [9, S]


@pytest.fixture(scope="module")
def noise_streams(lib):
    S = 300 * 2 * 17000          # 10.2 M samples per harmonic, 92 M in all
    return production_noise(lib, 12345, [S])


def test_production_noise_is_standard_normal(noise_streams):
    from scipy import stats
    z = noise_streams
    n = z.shape[1]
    se = 1 / math.sqrt(n)
    for h in range(9):
        m, v = z[h].mean(), z[h].var()
        assert abs(m) < 5 * se and abs(v - 1) < 5 * math.sqrt(2) * se, (h, m, v)
        p = stats.kstest(z[h][:2_000_000], "norm").pvalue
        assert p > 1e-6, (h, p)
    # Box-Muller of 24-bit uniforms u = (k + 0.5) 2^-24: |z| <= sqrt(-2 ln 2^-25) = 5.887
    assert np.abs(z).max() <= math.sqrt(-2 * math.log(2.0 ** -25)) + 1e-5
    tail = int((np.abs(z) > 4.5).sum())
    p45 = 2 * stats.norm.sf(4.5)
    exp = p45 * z.size
    assert abs(tail - exp) < 5 * math.sqrt(exp), (tail, exp)


def test_production_noise_is_uncorrelated(lib, noise_streams):
    z = noise_streams
    n = z.shape[1]
    bound = 5 / math.sqrt(n)     # 5 standard errors of a correlation of independent unit variables
    c = np.corrcoef(z)
    off_diag = np.abs(c - np.eye(9)).max()
    lag1 = max(abs(np.corrcoef(z[h, :-1], z[h, 1:])[0, 1]) for h in range(9))
    print(f"noise: max cross-harmonic |r| {off_diag:.2e}, max lag-1 |r| {lag1:.2e}, bound {bound:.2e} (n = {n})")
    assert off_diag < bound and lag1 < bound
    # another seed: an independent stream
    z2 = production_noise(lib, 777, [300 * 2 * 4000])
    n2 = z2.shape[1]
    for h in (0, 5, 8):
        assert abs(np.corrcoef(z[h, :n2], z2[h])[0, 1]) < 5 / math.sqrt(n2)


def test_production_noise_is_keyed_by_sample_not_batch_slot(lib):
    """Same seed: an item alone and at batch position 2 behind other items gets the same noise, bit for bit."""
    S = 300 * 2 * 50
    lw = np.asarray([0.3, -0.2, 0.1, 0.25, -0.15, 0.05, 0.2, -0.3, 0.12], np.float32)
    f0 = np.zeros(S // 300, np.float32)
    _, (alone,) = run_sine(lib, [f0], None, seed=99, lin_w=lw, want_phase=False)
    _, hs = run_sine(lib, [np.zeros(2 * 7, np.float32), np.zeros(2 * 300, np.float32), f0], None, seed=99, lin_w=lw,
                     want_phase=False)
    assert np.array_equal(hs[2], alone)
    assert np.array_equal(hs[1][:S], alone)              # the same sample indices of a longer item
    _, (other,) = run_sine(lib, [f0], None, seed=100, lin_w=lw, want_phase=False)
    assert not np.array_equal(other, alone)


# ============================================================================ K10 STFT
def stft_signal(kind, S, seed):
    rng = np.random.default_rng(seed)
    if kind == "zero":
        return np.zeros(S, np.float32)
    if kind == "const":
        return np.full(S, 0.37, np.float32)
    t = np.arange(S) / 24000.0
    x = sum(a * np.sin(2 * np.pi * f * t + p) for a, f, p in zip(rng.uniform(0.1, 0.6, 5), rng.uniform(80, 9000, 5),
                                                               rng.uniform(0, 6.3, 5)))
    x = x + 0.05 * rng.standard_normal(S)
    return np.tanh(x).astype(np.float32)


@pytest.mark.parametrize("replicate", [0, 1])
def test_stft_matches_float64(lib, replicate):
    # T = 1 (F = 121), 16 (F = 1921: 15 CTAs of 128 frames + 1 frame), 32 (F = 3841 = 30 CTAs + 1)
    items = [(1, "speech"), (16, "speech"), (2, "zero"), (3, "const"), (32, "speech")]
    Fs = [120 * T + 1 for T, _ in items]
    xs = [stft_signal(k, 600 * T, seed=i) for i, (T, k) in enumerate(items)]
    s_off, n_x = [], 0
    for x in xs:
        s_off.append(n_x)
        n_x += len(x) + 8
    xcat = np.full(n_x, NAN, np.float32)
    for o, x in zip(s_off, xs):
        xcat[o:o + len(x)] = x
    h_off, rows = level(Fs)
    har = np.full((rows, 24), SENT, np.float32)
    ok(lib, lib.kkx_test_stft(0, ptr(xcat), C.c_int64(n_x), len(Fs), ptr(i64(s_off), C.c_int64), ptr(i32(h_off), C.c_int),
                              ptr(i32(Fs), C.c_int), rows, replicate, ptr(har)))
    inside = np.zeros(rows, bool)
    for o, Fb in zip(h_off, Fs):
        inside[o:o + Fb] = True
    assert np.all(har[~inside] == SENT) and np.all(har[inside, 22:] == SENT)
    u = 2.0 ** -24
    for (T, kind), x, o, Fb in zip(items, xs, h_off, Fs):
        mag, ph = har[o:o + Fb, :11].T, har[o:o + Fb, 11:22].T          # [11, F]
        X, l1 = stft_reference(x, replicate)                             # complex128 [11, F], float64 [F]
        if kind == "zero":
            assert np.all(mag == 0) and np.all(ph == 0)
            continue
        bound = np.broadcast_to(STFT_BOUND_C * u * l1[None, :] + 1e-30, X.shape)
        # magnitude and complex value (the phase of a near-zero bin is not compared on its own)
        e_mag = np.abs(mag - np.abs(X)) / bound
        # (atan2f and hypotf: a few ulp each, 1e-6 of |X| in all; a bin the cut rule sets to +pi drops an imaginary part
        # of up to 4e-6 l1 by design)
        cut_drop = np.where(ph == np.float32(math.pi), 4e-6 * l1[None, :], 0.0)
        e_cplx = np.abs(mag * np.exp(1j * ph.astype(np.float64)) - X) / (bound + cut_drop + 1e-6 * np.abs(X))
        print(f"T={T} {kind} replicate={replicate}: mag err {e_mag.max():.3f}, complex err {e_cplx.max():.3f} of the bound")
        assert e_mag.max() <= 1 and e_cplx.max() <= 1
        # branch-cut rule: inside the fp32 rounding floor -> exactly fp32(pi); clearly outside -> the plain atan2
        re, im = X.real, X.imag
        cut = (re < -bound) & (np.abs(im) <= 2e-6 * l1[None, :])
        assert np.all(ph[cut] == np.float32(math.pi))
        plain = np.abs(im) >= 8e-6 * l1[None, :]
        d = np.abs(ph[plain].astype(np.float64) - np.angle(X[plain]))      # raw difference: -pi for +pi would be 2 pi
        assert np.all(d <= 2 * bound[plain] / np.abs(X[plain]) + 1e-6)
        if kind == "const":
            assert cut.sum() > 0     # the constant item lands bins inside the band


# ============================================================================ K11 iSTFT head
# conv_post logits: log-magnitudes in [-20, 8] and phase logits up to |x| = 100 (the suite's model runs use random
# weights, so the checkpoint's range is not known here: this is the range tested).
def istft_case(lib, Ts, fast, phase_max, mag_lo=-20.0, mag_hi=8.0, seed=0, pcm=False):
    Fs = [120 * T + 1 for T in Ts]
    h_off, rows = level(Fs)
    rng = np.random.default_rng(seed)
    cp = np.full((rows, 24), NAN, np.float32)       # gap rows and columns 22, 23: NaN, never read
    for o, Fb in zip(h_off, Fs):
        cp[o:o + Fb, :11] = rng.uniform(mag_lo, mag_hi, (Fb, 11))
        cp[o:o + Fb, 11:22] = rng.uniform(-phase_max, phase_max, (Fb, 11))
    s_off, n = [], 0
    for T in Ts:
        s_off.append(n)
        n += 600 * T + 12            # 12 sentinel samples behind every item
    audio = np.full(n, SENT, np.float32)
    pc = np.full(n, -12345, np.int16) if pcm else None
    ok(lib, lib.kkx_test_istft(0, ptr(cp), rows, len(Ts), ptr(i32(h_off), C.c_int), ptr(i32(Fs), C.c_int), fast,
                               C.c_int64(n), ptr(i64(s_off), C.c_int64), ptr(audio), ptr(pc, C.c_int16)))
    outs, refs = [], []
    for T, o, so, Fb in zip(Ts, h_off, s_off, Fs):
        S = 600 * T
        assert np.all(audio[so + S:so + S + 12] == SENT), "write behind the item"
        if pcm:
            assert np.all(pc[so + S:so + S + 12] == -12345)
        outs.append(audio[so:so + S])
        refs.append(istft_reference(cp[o:o + Fb, :22]))
    return outs, refs, (pc, s_off) if pcm else None


@pytest.mark.parametrize("fast", [0, 1])
def test_istft_matches_float64(lib, fast):
    # T = 31: 3720 groups = 30 whole 124-group CTAs; T = 30: a 4-group last CTA; T = 1, 2: one CTA; 100, 1000: many
    Ts = [1, 2, 30, 31, 100, 1000]
    bound = 1e-4 if fast else 1e-5
    for pmax in (1.0, 10.0, 100.0):
        outs, refs, _ = istft_case(lib, Ts, fast, pmax, seed=int(pmax))
        worst = 0.0
        for T, y, r in zip(Ts, outs, refs):
            assert y.shape == r.shape and np.isfinite(y).all()
            worst = max(worst, np.abs(y - r).max() / np.abs(r).max())
        print(f"istft fast={fast} |phase logit| <= {pmax:g}: max error {worst:.2e} of the item's peak")
        # measured on a B200 (1000 W): fp32 2.1e-7 / 2.5e-7 / 2.8e-7 of the peak at |x| <= 1 / 10 / 100; FAST 4.0e-7 /
        # 7.0e-7 / 6.2e-6 -- __sinf's error grows with |x| (its argument is scaled by 1 / 2 pi in fp32 before the SFU),
        # about 6e-8 |x|.  Bounds: 1e-5 (fp32) and 1e-4 (FAST, 16x the measured worst case at |x| <= 100)
        assert worst <= bound


def test_istft_pcm16_twin(lib):
    Ts = [1, 30, 31, 77]
    outs, refs, (pc, s_off) = istft_case(lib, Ts, 1, 100.0, mag_lo=-20.0, mag_hi=0.0, seed=5, pcm=True)
    for T, y, r, so in zip(Ts, outs, refs, s_off):
        p = pc[so:so + 600 * T]
        # bit-equal to trunc(clamp(kernel float) * 32767) of the kernel's own float
        want = np.trunc(np.clip(y, np.float32(-1), np.float32(1)) * np.float32(32767)).astype(np.int16)
        assert np.array_equal(p, want)
        # within one LSB of the float64 reference
        ref = np.trunc(np.clip(r, -1, 1) * 32767)
        assert np.abs(p.astype(np.float64) - ref).max() <= 1


# ============================================================================ K4 / K5 durations and length regulator
def run_durations(lib, logits_items, speeds, C_, ldo, ocol, seed=0):
    Ns = [len(l) for l in logits_items]
    B = len(Ns)
    t_off, rows_tok = level(Ns)
    lg = np.full((rows_tok, 50), NAN, np.float32)
    rng = np.random.default_rng(seed)
    feat = np.full((rows_tok, C_), NAN, np.float32)
    for o, l in zip(t_off, logits_items):
        lg[o:o + len(l)] = l
        feat[o:o + len(l)] = rng.standard_normal((len(l), C_))
    sp = np.asarray(speeds, np.float32)
    durf = np.full(rows_tok, SENT, np.float32)
    pd = np.full(rows_tok, -5, np.int32)
    cum = np.zeros((B, 512), np.int32)
    tot = np.zeros(B, np.int32)
    fro = np.zeros(B, np.int32)
    args = (ptr(lg), ptr(sp), ptr(feat), C_, ldo, ocol, B, ptr(i32(t_off), C.c_int), ptr(i32(Ns), C.c_int), rows_tok,
            ptr(durf), ptr(pd, C.c_int32), ptr(cum, C.c_int32), ptr(tot, C.c_int32), ptr(fro, C.c_int32))
    rows_fr = lib.kkx_test_durations(0, *args, None, None, C.c_int64(0))
    assert rows_fr > 0, lib.kkx_test_last_error()
    idx = np.full(rows_fr, -7, np.int32)
    out = np.full((rows_fr, ldo), SENT, np.float32)
    assert lib.kkx_test_durations(0, *args, ptr(idx, C.c_int32), ptr(out), C.c_int64(rows_fr)) == rows_fr
    return dict(t_off=t_off, Ns=Ns, lg=lg, feat=feat, durf=durf, pd=pd, cum=cum, tot=tot, fro=fro, idx=idx, out=out)


def check_durations(r, speeds, ldo, ocol):
    C_ = r["feat"].shape[1]
    rows_fr = r["out"].shape[0]
    covered = np.zeros(rows_fr, bool)
    for b, (o, N) in enumerate(zip(r["t_off"], r["Ns"])):
        lg = r["lg"][o:o + N].astype(np.float64)
        with np.errstate(over="ignore", invalid="ignore"):
            sig = 1.0 / (1.0 + np.exp(-lg))
        s64 = sig.sum(axis=1)
        d = r["durf"][o:o + N]
        ref = s64 / np.float64(np.float32(speeds[b]))
        # |d - s64 / speed| <= sum_k 2^-22 sigma_k / speed (expf 2 ulp + two roundings per sigmoid) + one ulp of d (the
        # fp32 rounding of the fp64 sum and the correctly rounded division, half an ulp each); a sigmoid below fp32's
        # normal range (logit < -87: expf overflows) is 0, which adds at most 50 * FLT_MIN / speed
        fin = np.isfinite(ref)
        tol = (2.0 ** -22 * s64[fin] + 50 * np.finfo(np.float32).tiny) / speeds[b] + np.spacing(np.abs(d[fin]))
        assert np.all(np.abs(d[fin].astype(np.float64) - ref[fin]) <= tol)
        assert np.all(np.isnan(d[~fin]))
        # pred_dur = rint-half-even(dur_float) clamped to [1, 1000] (NaN -> 1), exactly
        with np.errstate(invalid="ignore"):
            want = np.where(np.isnan(d), 1, np.clip(np.rint(d), 1, 1000)).astype(np.int32)
        pd = r["pd"][o:o + N]
        assert np.array_equal(pd, want)
        cum = np.concatenate([[0], np.cumsum(pd.astype(np.int64))])
        assert np.array_equal(r["cum"][b, :N], cum[:-1]) and r["tot"][b] == cum[-1]
        T, fo = int(cum[-1]), r["fro"][b]
        idx = np.repeat(np.arange(N), pd)
        assert np.array_equal(r["idx"][fo:fo + T], idx)
        got = r["out"][fo:fo + T]
        assert np.array_equal(got[:, ocol:ocol + C_].view(np.uint32), r["feat"][o + idx].view(np.uint32))
        assert np.all(got[:, :ocol] == SENT) and np.all(got[:, ocol + C_:] == SENT)
        covered[fo:fo + T] = True
    assert np.all(r["out"][~covered] == SENT), "gather_rows wrote a gap row"


def test_durations_ties_and_specials(lib):
    # logits of +-100 make sigma exactly 1 or 0: 25 ones / 2.0 = 12.5 -> 12 (half to even; roundf would give 13),
    # 23 / 2 = 11.5 -> 12, 21 / 2 = 10.5 -> 10, 27 / 2 = 13.5 -> 14
    rows = []
    for ones in (25, 23, 21, 27, 1, 0, 50):
        rows.append(np.where(np.arange(50) < ones, 100.0, -100.0))
    special = np.zeros((5, 50))
    special[0, 3] = np.nan                 # NaN -> duration 1
    special[1, :] = np.inf                 # sigma(+inf) = 1: 50 / 2 = 25
    special[2, :] = -np.inf                # sigma(-inf) = 0 -> clamped to 1
    special[3, :10] = np.inf
    special[3, 10:] = -np.inf
    special[4, :] = 0.0                    # 50 * 0.5 = 25 / 2 = 12.5 -> 12
    lg = np.concatenate([np.asarray(rows), special]).astype(np.float32)
    r = run_durations(lib, [lg], [2.0], 512, 520, 0)
    check_durations(r, [2.0], 520, 0)
    assert list(r["pd"][r["t_off"][0]:r["t_off"][0] + 7]) == [12, 12, 10, 14, 1, 1, 25]
    assert list(r["pd"][r["t_off"][0] + 7:r["t_off"][0] + 12]) == [1, 25, 1, 5, 12]


def test_durations_speeds_and_cap(lib):
    rng = np.random.default_rng(1)
    lg = [rng.uniform(-6, 6, (n, 50)).astype(np.float32) for n in (40, 33, 17)]
    lg[2][:5] = 100.0                     # 50 / 0.01 = 5000 -> the 1000 cap (0.01 is below the model's 0.1 minimum)
    speeds = [0.1, 1.7, 0.01]
    r = run_durations(lib, lg, speeds, 512, 520, 0, seed=2)
    check_durations(r, speeds, 520, 0)
    assert np.all(r["pd"][r["t_off"][2]:r["t_off"][2] + 5] == 1000)


@pytest.mark.parametrize("Ns", [[1], [31, 32, 33], [511, 512], [512, 1, 200]])
def test_length_regulator_exact(lib, Ns):
    # durations up to 1000 per token: logits around the sigmoid's middle at speed 0.03 -> sums 0..50 / 0.03
    rng = np.random.default_rng(sum(Ns))
    lg = [rng.normal(0, 3, (n, 50)).astype(np.float32) for n in Ns]
    speeds = [0.03 + 0.01 * b for b in range(len(Ns))]
    r = run_durations(lib, lg, speeds, 24, 40, 9, seed=len(Ns))
    check_durations(r, speeds, 40, 9)
    if sum(Ns) > 30:
        assert r["pd"][r["pd"] > 0].max() >= 900


# ============================================================================ pool_up (fp32) and pool_up_bf16
@pytest.mark.parametrize("C_,Cpad", [(512, 512), (256, 256), (1090, 1152)])
def test_pool_up_kernels(lib, C_, Cpad):
    Ts = [1, 130, 7, 257]
    B = len(Ts)
    rng = np.random.default_rng(C_)
    in_off, rows_in = level(Ts)
    out_off, rows_out = level([2 * T for T in Ts])
    x = np.full((rows_in, C_), NAN, np.float32)
    for o, T in zip(in_off, Ts):
        x[o:o + T] = rng.standard_normal((T, C_))
    sc = (1 + 0.3 * rng.standard_normal((B, C_))).astype(np.float32)
    sh = (0.3 * rng.standard_normal((B, C_))).astype(np.float32)
    w = (0.5 * rng.standard_normal((C_, 3))).astype(np.float32)
    bias = (0.1 * rng.standard_normal(C_)).astype(np.float32)
    base = [ptr(x), rows_in, C_, B, ptr(i32(in_off), C.c_int), ptr(i32(Ts), C.c_int), ptr(sc), ptr(sh), C.c_float(0.2),
            ptr(w), ptr(bias), ptr(i32(out_off), C.c_int), rows_out]
    y = np.full((rows_out, C_), SENT, np.float32)
    ok(lib, lib.kkx_test_pool_up(0, *base, 0, y.ctypes.data_as(C.c_void_p)))
    yb = np.full((rows_out, Cpad), 0xFFFF, np.uint16)     # NaN bits: gap rows and pad columns must come back zero
    ok(lib, lib.kkx_test_pool_up(0, *base, Cpad, yb.ctypes.data_as(C.c_void_p)))
    inside = np.zeros(rows_out, bool)
    u = 2.0 ** -24
    for b, (oi, oo, T) in enumerate(zip(in_off, out_off, Ts)):
        inside[oo:oo + 2 * T] = True
        xa = x[oi:oi + T].astype(np.float64)
        a = xa * sc[b] + sh[b]
        a = np.where(a > 0, a, a * np.float64(np.float32(0.2)))
        ref = F.conv_transpose1d(torch.from_numpy(np.ascontiguousarray(a.T))[None],
                                 torch.from_numpy(w.astype(np.float64)[:, None, :]), torch.from_numpy(bias.astype(np.float64)),
                                 stride=2, padding=1, output_padding=1, groups=C_)[0].T.numpy()
        # magnitude of the terms: each fp32 operation (x * sc + sh, the slope product, w * a, the two additions) adds
        # at most one rounding of the running magnitude -> <= 8 u * m
        am = np.abs(xa * sc[b]) + np.abs(sh[b])
        m = np.zeros((2 * T, C_))
        m[0::2] = np.abs(w[:, 1]) * am + np.abs(bias)
        m[1::2] = np.abs(w[:, 2]) * am + np.abs(bias)
        m[1:-1:2] += np.abs(w[:, 0]) * am[1:]
        got = y[oo:oo + 2 * T]
        assert np.all(np.abs(got - ref) <= 8 * u * m + 1e-30)
        # bf16 operand: the same expression rounded to bf16.  The two kernels are compiled separately and nvcc may contract
        # w2 * a0 + w0 * a1 + bias into FMAs differently in each, so their fp32 values v, v' can differ -- each is within
        # 8 u m of the exact value, so |v - v'| <= 16 u m (more than an ulp of v only where the terms cancel).  Rounding
        # v' to bf16 adds at most one bf16 ulp: |bf16(v') - bf16(v)| <= ulp_bf16 + 16 u m; measured on a B200, the two
        # differ in about 1e-5 of the elements
        want = bf16_bits(got)
        have = yb[oo:oo + 2 * T, :C_]
        wf = (want.astype(np.uint32) << 16).view(np.float32)
        hf = (have.astype(np.uint32) << 16).view(np.float32)
        ulp = np.abs(np.spacing(wf)) * 65536.0
        assert np.all(np.abs(hf - wf) <= ulp + 16 * u * m)
        mism = float((have != want).mean())
        print(f"pool_up_bf16 C={C_}: {mism:.2e} of the elements differ from bf16(pool_up)")
        assert mism < 1e-2
    assert np.all(y[~inside] == SENT), "pool_up wrote outside the items"
    assert np.all(yb[~inside] == 0) and np.all(yb[:, C_:] == 0), "gap rows / pad columns of the bf16 operand not zero"


# ============================================================================ conv_post (tensor-core configuration)
@pytest.mark.parametrize("lens", [[1], [127], [128], [129], [128 * 150 + 5], [300, 1, 129, 256],
                                  [3 + (i * 7) % 29 for i in range(512)]], ids=lambda v: f"B{len(v)}-L{max(v)}")
def test_post_conv_matches_float64_reference(lib, lens):
    B = len(lens)
    rng = np.random.default_rng(len(lens) + max(lens))
    off, rows = level(lens)
    x = np.full((rows, 128), NAN, np.float32)
    for o, L in zip(off, lens):
        x[o:o + L] = rng.standard_normal((L, 128))
    w = (rng.standard_normal((22, 128, 7)) / np.sqrt(128 * 7)).astype(np.float32)
    b = (0.1 * rng.standard_normal(22)).astype(np.float32)
    out = np.full((rows, 24), SENT, np.float32)
    ok(lib, lib.kkx_test_post_conv(0, ptr(x), rows, B, ptr(i32(off), C.c_int), ptr(i32(lens), C.c_int),
                                   ptr(np.ascontiguousarray(w.transpose(0, 2, 1))), ptr(b), C.c_float(0.01), ptr(out)))
    inside = np.zeros(rows, bool)
    wb = torch.from_numpy(bf16_round(w).astype(np.float64))
    for o, L in zip(off, lens):
        inside[o:o + L] = True
        xi = torch.from_numpy(x[o:o + L])
        a = bf16_round(F.leaky_relu(xi, 0.01).numpy()).astype(np.float64)
        ref = F.conv1d(torch.from_numpy(a.T)[None], wb, torch.from_numpy(b.astype(np.float64)), padding=3)[0].T.numpy()
        got = out[o:o + L, :22]
        # fp32 accumulation of 896 exact bf16 products (test_tc_conv_matches_torch_on_bf16_operands' bound)
        np.testing.assert_allclose(got, ref, atol=3e-4, rtol=1e-4)
        if L >= 128:
            ref32 = F.conv1d(F.leaky_relu(xi, 0.01).T[None], torch.from_numpy(w), torch.from_numpy(b), padding=3)[0].T.numpy()
            assert np.sqrt(((got - ref32) ** 2).sum() / (ref32 ** 2).sum()) < 6e-3
    assert np.all(out[inside, 22:] == SENT), "conv_post wrote columns 22, 23"
    assert np.all(out[~inside] == SENT), "conv_post wrote outside the items"


# ============================================================================ curve_conv and add_rows_stats
def test_curve_conv_matches_float64(lib):
    Ts = [1, 255, 256, 257, 3000]
    B = len(Ts)
    rng = np.random.default_rng(8)
    x_off, rows_x = level([2 * T for T in Ts])
    out_off, rows_out = level(Ts)
    x = np.full(rows_x, NAN, np.float32)
    for o, T in zip(x_off, Ts):
        x[o:o + 2 * T] = rng.uniform(0, 400, 2 * T)
    w3 = rng.standard_normal(3).astype(np.float32)
    bias = np.asarray([0.3], np.float32)
    u = 2.0 ** -24
    for ocol in (512, 513):
        out = np.full((rows_out, 520), SENT, np.float32)
        ok(lib, lib.kkx_test_curve_conv(0, ptr(x), rows_x, B, ptr(i32(x_off), C.c_int), ptr(i32([2 * T for T in Ts]), C.c_int),
                                        ptr(w3), ptr(bias), ptr(out), rows_out, 520, ocol, ptr(i32(out_off), C.c_int),
                                        ptr(i32(Ts), C.c_int)))
        mask = np.ones_like(out, bool)
        for o, oo, T in zip(x_off, out_off, Ts):
            xi = torch.from_numpy(x[o:o + 2 * T].astype(np.float64)).view(1, 1, -1)
            ref = F.conv1d(xi, torch.from_numpy(w3.astype(np.float64)).view(1, 1, 3),
                           torch.from_numpy(bias.astype(np.float64)), stride=2, padding=1)[0, 0].numpy()
            m = F.conv1d(xi.abs(), torch.from_numpy(np.abs(w3).astype(np.float64)).view(1, 1, 3), stride=2,
                         padding=1)[0, 0].numpy() + abs(bias[0])
            assert np.all(np.abs(out[oo:oo + T, ocol] - ref) <= 4 * u * m)     # three FMA roundings + the bias add
            mask[oo:oo + T, ocol] = False
        assert np.all(out[mask] == SENT)


@pytest.mark.parametrize("C_,lens", [(128, [1, 128, 129, 700]), (256, [255, 256, 1000])])
@pytest.mark.parametrize("to_bf16", [False, True])
def test_add_rows_stats(lib, C_, lens, to_bf16):
    B = len(lens)
    rng = np.random.default_rng(C_ + len(lens))
    off, rows = level(lens)
    a = np.full((rows, C_), SENT, np.float32)
    bb = np.full((rows, C_), NAN, np.float32)
    for o, L in zip(off, lens):
        a[o:o + L] = rng.standard_normal((L, C_)) * 3
        bb[o:o + L] = rng.standard_normal((L, C_))
    a0 = a.copy()
    ob = np.full((rows, C_), 0x7FC1, np.uint16) if to_bf16 else None
    nch = (max(lens) + 127) // 128
    part = np.zeros((B, nch, 2, C_), np.float32)
    ok(lib, lib.kkx_test_add_rows_stats(0, ptr(a), ptr(bb), rows, C_, B, ptr(i32(off), C.c_int), ptr(i32(lens), C.c_int),
                                        ptr(ob, C.c_uint16), ptr(part)))
    u = 2.0 ** -24
    for i, (o, L) in enumerate(zip(off, lens)):
        s = a0[o:o + L] + bb[o:o + L]                    # numpy fp32 a + b
        if to_bf16:
            assert np.array_equal(a, a0), "`out` must stay untouched with bf16 output"
            assert np.array_equal(ob[o:o + L], bf16_bits(s))
        else:
            assert np.array_equal(a[o:o + L].view(np.uint32), s.view(np.uint32))
        s64 = s.astype(np.float64)
        n = (L + 127) // 128
        S = part[i, :n, 0].astype(np.float64).sum(axis=0)
        Q = part[i, :n, 1].astype(np.float64).sum(axis=0)
        # fp32 sums over <= 128 rows per chunk (a chain of <= 128 additions): <= 130 u * sum |v| (squares: sum v^2)
        assert np.all(np.abs(S - s64.sum(axis=0)) <= 130 * u * np.abs(s64).sum(axis=0))
        assert np.all(np.abs(Q - (s64 ** 2).sum(axis=0)) <= 130 * u * (s64 ** 2).sum(axis=0))
    if not to_bf16:
        inside = np.zeros(rows, bool)
        for o, L in zip(off, lens):
            inside[o:o + L] = True
        assert np.array_equal(a[~inside], a0[~inside])
    else:
        inside = np.zeros(rows, bool)
        for o, L in zip(off, lens):
            inside[o:o + L] = True
        assert np.all(ob[~inside] == 0x7FC1)
