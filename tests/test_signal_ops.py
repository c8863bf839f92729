"""CPU tests: the references tests/test_signal_ops_gpu.py holds the signal-path kernels to.

- the numpy emulation of sine_source_kernel's x300 phase interpolation (index, lambda and fma in fp32) is the oracle's
  fp32 F.interpolate bit for bit, past 2^24 samples, so that a GPU mismatch there is the kernel's fault;
- the x1/300 down-sampling of the oracle's rad curve reproduces each 300-sample plateau (what sine_phase relies on);
- the float64 STFT / iSTFT references equal torch.stft / torch.istft, and the STFT branch-cut classification the GPU
  test uses agrees with KokoroOracle.stft."""
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

GAP_ROWS = 32
# STFT rounding bound in units of 2^-24 * sum_j |x_j w_j|: the fp32 window (1 rounding) and product (1), the twiddle
# tables (1), 20 accumulating FMAs (20) -> 23 per real / imaginary part, sqrt(2) * 23 for the modulus plus hypotf -> 34
STFT_BOUND_C = 34.0


def level(lens, first=GAP_ROWS):
    """Row offsets of ragged items as Model::make_level packs them (32 gap rows, 8-row alignment) and the row count."""
    off, o = [], first
    for n in lens:
        off.append(o)
        o = (o + n + GAP_ROWS + 7) & ~7
    return off, o


def emulate_phase_upsampling(p, scale=300):
    """fp32 per-sample phase of sine_source_kernel: src = fma(fp32(1/300), fp32(n) + 0.5, -0.5) clamped at 0,
    i0 = (int)src, i1 = min(i0 + 1, L - 1), lambda = src - i0, value = fma(p[i0], 1 - lambda, p[i1] * lambda).
    An fma is exact in float64 here (the product of two fp32 values has 48 bits, and the addend's bits fall inside
    the 53) and then rounded once to fp32."""
    p = np.asarray(p, np.float32)
    L = p.shape[-1]
    n = np.arange(L * scale, dtype=np.int64)
    t = n.astype(np.float32) + np.float32(0.5)
    src = (np.float64(np.float32(1.0 / scale)) * t.astype(np.float64) - 0.5).astype(np.float32)
    del t
    src = np.maximum(src, np.float32(0))
    i0 = src.astype(np.int64)
    i1 = np.minimum(i0 + 1, L - 1)
    lam = np.clip(src - i0.astype(np.float32), np.float32(0), np.float32(1))
    del src
    w0 = np.float32(1) - lam
    prod = p[i1] * lam
    return (p[i0].astype(np.float64) * w0.astype(np.float64) + prod.astype(np.float64)).astype(np.float32)


def hann64():
    return 0.5 - 0.5 * np.cos(2 * np.pi * np.arange(20) / 20)


def stft_reference(x, replicate):
    """float64 STFT (n_fft 20, hop 5, periodic Hann, center) of fp32 x -> X [11, F] complex128 and the per-frame
    l1 = sum_j |x_j w_j| [F]."""
    xd = np.asarray(x, np.float64)
    pad = np.pad(xd, 10, mode="edge" if replicate else "reflect")
    frames = np.lib.stride_tricks.sliding_window_view(pad, 20)[::5] * hann64()
    return np.fft.rfft(frames, axis=1).T.copy(), np.abs(frames).sum(axis=1)


def istft_reference(cp):
    """float64 head + iSTFT of conv_post rows cp [F, 22]: X = exp(cp[:, :11]) e^{i sin(cp[:, 11:])}, inverse real DFT
    (the imaginary parts of bins 0 and 10 dropped), periodic Hann synthesis window, overlap-add, division by the summed
    squared window, n_fft / 2 trimmed at both ends -> 5 (F - 1) samples."""
    cp = np.asarray(cp, np.float64)
    X = np.exp(cp[:, :11]) * np.exp(1j * np.sin(cp[:, 11:22]))
    w = hann64()
    fr = np.fft.irfft(X, n=20, axis=1) * w
    Fn = cp.shape[0]
    n = 20 + 5 * (Fn - 1)
    y, env = np.zeros(n), np.zeros(n)
    for j in range(20):
        y[j:j + 5 * Fn:5] += fr[:, j]
        env[j:j + 5 * Fn:5] += w[j] ** 2
    return (y / np.where(env > 1e-11, env, 1.0))[10:n - 10]


@pytest.mark.parametrize("T", [25, 14500, 28500])
def test_phase_interpolation_emulation_is_the_oracle_bit_for_bit(T):
    # coarse phases as the oracle makes them (fp32 ((cumsum(rad) * 2) * pi) * 300) for a 50..500 Hz fundamental's
    # ninth harmonic: up to ~1e7 rad; T = 28 500 is 17.1 M samples, past 2^24
    L = 2 * T
    rng = np.random.default_rng(T)
    rad = torch.from_numpy(((rng.uniform(50, 500, L).astype(np.float32) * np.float32(9)) / np.float32(24000)) % 1)
    coarse = ((torch.cumsum(rad.view(1, -1, 1), dim=1) * 2 * np.pi).transpose(1, 2) * 300)
    ref = F.interpolate(coarse, scale_factor=300, mode="linear")[0, 0].numpy()
    got = emulate_phase_upsampling(coarse[0, 0].numpy(), 300)
    assert got.shape == ref.shape
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))


def test_rad_downsampling_reproduces_each_plateau():
    L = 3000
    f0 = np.random.default_rng(1).uniform(-100, 600, L).astype(np.float32)
    f0_up = torch.from_numpy(f0).repeat_interleave(300).view(1, -1, 1)
    fn = f0_up * torch.arange(1, 10, dtype=torch.float32).view(1, 1, -1)
    rad_full = (fn / 24000) % 1
    rad = F.interpolate(rad_full.transpose(1, 2), scale_factor=1 / 300, mode="linear").transpose(1, 2)
    assert torch.equal(rad[0], rad_full[0, ::300])


@pytest.mark.parametrize("replicate", [0, 1])
def test_stft_reference_is_torch_stft(replicate):
    x = np.tanh(np.random.default_rng(2).standard_normal(600 * 3)).astype(np.float32)
    X, _ = stft_reference(x, replicate)
    ref = torch.stft(torch.from_numpy(x.astype(np.float64)), 20, 5, 20, window=torch.hann_window(20, dtype=torch.float64),
                     center=True, pad_mode="replicate" if replicate else "reflect", return_complex=True).numpy()
    np.testing.assert_allclose(X, ref, rtol=0, atol=1e-12)


@pytest.mark.parametrize("replicate", [0, 1])
def test_stft_cut_rule_reference_agrees_with_the_oracle(replicate):
    """The GPU test's classification -- re < 0 with |im| <= 2e-6 l1 must be fp32(pi), |im| >= 8e-6 l1 must be the
    plain angle -- holds for the oracle's own fp32 STFT, which cuts at 4e-6 l1 (KokoroOracle.stft)."""
    from oracle.kokoro_ref import KokoroOracle
    o = KokoroOracle({}, stft_pad_mode="replicate" if replicate else "reflect")
    rng = np.random.default_rng(3)
    xs = [np.full(600 * 2, 0.37, np.float32), np.tanh(rng.standard_normal(600 * 4)).astype(np.float32),
          np.repeat(rng.standard_normal(600 * 4 // 20), 20).astype(np.float32)]
    u = 2.0 ** -24
    ncut = 0
    for x in xs:
        mag, ph = (t.numpy() for t in o.stft(torch.from_numpy(x)))
        X, l1 = stft_reference(x, replicate)
        bound = np.broadcast_to(STFT_BOUND_C * u * l1[None, :], X.shape)
        cut = (X.real < -bound) & (np.abs(X.imag) <= 2e-6 * l1[None, :])
        assert np.all(ph[cut] == np.float32(math.pi))
        plain = np.abs(X.imag) >= 8e-6 * l1[None, :]
        assert np.all(np.abs(ph[plain].astype(np.float64) - np.angle(X[plain])) <= 2 * bound[plain] / np.abs(X[plain]) + 1e-6)
        ncut += int(cut.sum())
    assert ncut > 100


def test_istft_reference_is_torch_istft():
    rng = np.random.default_rng(4)
    for T in (1, 2, 7):
        Fn = 120 * T + 1
        cp = np.concatenate([rng.uniform(-20, 8, (Fn, 11)), rng.uniform(-100, 100, (Fn, 11))], axis=1)
        got = istft_reference(cp)
        X = torch.from_numpy(np.exp(cp[:, :11]) * np.exp(1j * np.sin(cp[:, 11:]))).T
        ref = torch.istft(X[None], 20, 5, 20, window=torch.hann_window(20, dtype=torch.float64))[0].numpy()
        assert got.shape == ref.shape == (600 * T,)
        np.testing.assert_allclose(got, ref, rtol=0, atol=1e-12 * np.abs(ref).max())


def test_level_layout_matches_the_model():
    off, rows = level([1, 300, 17])
    assert off == [32, 72, 408] and rows == 464
