"""CPU tests of the output-format path (no GPU): the resampling filter the library designs (kkx_test_resample_taps)
against scipy, and the numpy G.711 reference the GPU tests use against Python's audioop."""
import ctypes as C
import math
import warnings

import numpy as np
import pytest

RATES = (8000, 11025, 12000, 16000, 22050, 24000, 32000, 44100, 48000)

# ---- G.711 reference (Sun g711.c, the encoder behind audioop.lin2ulaw / lin2alaw(..., 2)) -----------------------
_SEG_U = np.array([0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF, 0x1FFF])
_SEG_A = np.array([0x1F, 0x3F, 0x7F, 0xFF, 0x1FF, 0x3FF, 0x7FF, 0xFFF])


def ulaw_ref(pcm16):
    """mu-law codes of 16-bit samples: the 14-bit value p >> 2, bias 33, clip 8159."""
    v = np.asarray(pcm16, np.int32) >> 2
    mask = np.where(v < 0, 0x7F, 0xFF)
    v = np.minimum(np.abs(v), 8159) + 33
    seg = np.searchsorted(_SEG_U, v, side="left")
    s7 = np.minimum(seg, 7)
    code = np.where(seg >= 8, 0x7F, (s7 << 4) | ((v >> (s7 + 1)) & 0xF))
    return (code ^ mask).astype(np.uint8)


def alaw_ref(pcm16):
    """A-law codes of 16-bit samples: the 13-bit value p >> 3."""
    v = np.asarray(pcm16, np.int32) >> 3
    mask = np.where(v >= 0, 0xD5, 0x55)
    v = np.where(v >= 0, v, -v - 1)
    seg = np.searchsorted(_SEG_A, v, side="left")
    s7 = np.minimum(seg, 7)
    q = np.where(s7 < 2, v >> 1, v >> s7) & 0xF
    code = np.where(seg >= 8, 0x7F, (s7 << 4) | q)
    return (code ^ mask).astype(np.uint8)


def pcm16_ref(y):
    """trunc(clamp(y, -1, 1) * 32767) in f32, the library's f32 -> i16 conversion."""
    return np.trunc(np.clip(np.asarray(y, np.float32), -1.0, 1.0) * np.float32(32767.0)).astype(np.int16)


def ratio(rate):
    g = math.gcd(rate, 24000)
    return rate // g, 24000 // g


@pytest.fixture(scope="module")
def lib():
    from kokorox_b200 import build
    build.build()
    from kokorox_b200.onn import load_library
    return load_library()


@pytest.mark.parametrize("rate", RATES)
def test_resample_taps_match_scipy_firwin(lib, rate):
    from scipy.signal import firwin
    U, D = ratio(rate)
    if U == D:     # 24 kHz: resample_poly copies its input (firwin has no filter with cutoff 1): the identity
        H, want = 0, np.ones(1, np.float32)
    else:
        H = 10 * max(U, D)
        want = (U * firwin(2 * H + 1, 1.0 / max(U, D), window=("kaiser", 5.0))).astype(np.float32)
    n = lib.kkx_test_resample_taps(rate, None, 0)
    assert n == 2 * H + 1
    got = np.zeros(n, np.float32)
    assert lib.kkx_test_resample_taps(rate, got.ctypes.data_as(C.POINTER(C.c_float)), n) == n
    # within one fp32 ulp per tap (both are designed in double and rounded once)
    ulp = np.spacing(np.abs(want)).astype(np.float64)
    assert np.all(np.abs(got.astype(np.float64) - want.astype(np.float64)) <= ulp), rate
    assert np.array_equal(got, got[::-1])     # linear phase: the design is symmetric


@pytest.mark.parametrize("rate", (7999, 48001, 44099, 0, -8000, 96000))
def test_resample_taps_reject_unsupported_rates(lib, rate):
    assert lib.kkx_test_resample_taps(rate, None, 0) < 0


def test_g711_reference_matches_audioop():
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", DeprecationWarning)
        audioop = pytest.importorskip("audioop")
    p = np.arange(-32768, 32768, dtype=np.int16)
    assert np.array_equal(ulaw_ref(p), np.frombuffer(audioop.lin2ulaw(p.tobytes(), 2), np.uint8))
    assert np.array_equal(alaw_ref(p), np.frombuffer(audioop.lin2alaw(p.tobytes(), 2), np.uint8))
