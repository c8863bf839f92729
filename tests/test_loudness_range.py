"""CPU tests of the EBU R128 loudness report (no GPU): a float64 numpy reference of the kkx.h "loudness_report" rules
1-5 (maximum momentary and short-term loudness, the EBU Tech 3342 loudness range), built on test_loudness.py's
K-weighting and block energies, checked against known answers.  The GPU tests in test_loudness_range_gpu.py compare
the kernels and the model's report with the same reference."""
import math

import numpy as np
import pytest

from tests.test_loudness import block_energies, kweight, tone

FS = 24000
SEG = FS // 10                  # the 100 ms hop, 2400 samples
BLOCK, WINDOW = 4 * SEG, 30 * SEG


def short_term_energies(x, fs=FS):
    """s_j of every whole 3 s window on a 100 ms hop from sample 0 (cumulative sums of the K-weighted square)."""
    y = kweight(x, fs)
    win, hop = 3 * fs, fs // 10
    n = (len(y) - win) // hop + 1 if len(y) >= win else 0
    c = np.concatenate([[0.0], np.cumsum(y * y)])
    return np.array([(c[j * hop + win] - c[j * hop]) / win for j in range(n)])


def lufs(z):
    with np.errstate(divide="ignore"):
        return -0.691 + 10.0 * np.log10(z)


def ranks(m):
    """Rule 4: the nearest ranks of the 10 % and 95 % points of m sorted values, halves rounded up, in integers."""
    return (10 * (m - 1) + 50) // 100, (95 * (m - 1) + 50) // 100


def range_ref(x):
    """Rules 1-5 for one item: (LRA in LU, max momentary and max short-term loudness in LUFS); NaN = undefined."""
    x = np.asarray(x, np.float64)
    z = block_energies(x) if len(x) else np.zeros(0)
    M = float(lufs(z.max())) if len(z) else float("nan")
    s = short_term_energies(x) if len(x) else np.zeros(0)
    if not len(s):
        return float("nan"), M, float("nan")
    S = float(lufs(s.max()))
    ls = lufs(s)
    a = ls > -70.0
    if not a.any():
        return float("nan"), M, S
    rel = -0.691 + 10.0 * math.log10(s[a].mean()) - 20.0
    g = np.sort(s[a & (ls > rel)])
    if not len(g):
        return float("nan"), M, S
    lo, hi = ranks(len(g))
    return 10.0 * math.log10(g[hi] / g[lo]), M, S


def levels(dbfs, seconds=20.0, f=1000.0, fs=FS):
    """EBU Tech 3342's test signals: a phase-continuous 1 kHz tone, `seconds` at each level in turn."""
    n = int(round(seconds * fs))
    parts = [tone(n, fs, f, d, 2 * np.pi * f * n * k / fs) for k, d in enumerate(dbfs)]
    return np.concatenate(parts)


# (levels in dBFS, expected LRA): the first four cases of EBU Tech 3342; the tone is steady over every 3 s window
# (3000 whole periods), so a window that lies inside one level has exactly that level's energy and the 10 % and 95 %
# points fall inside the quietest and the loudest gated level: the LRA is exactly their difference.
TECH3342 = (((-20.0, -30.0), 10.0), ((-20.0, -15.0), 5.0), ((-40.0, -20.0), 20.0),
            ((-50.0, -35.0, -20.0, -35.0, -50.0), 15.0))


@pytest.mark.parametrize("pattern,want", TECH3342)
def test_tech3342_loudness_range(pattern, want):
    lra, M, S = range_ref(levels(pattern))
    assert abs(lra - want) <= 1.0                  # Tech 3342's tolerance
    assert abs(lra - want) <= 1e-6                 # and the analytic value
    assert M >= S - 1e-9                            # a 400 ms block inside the loudest part is at least any 3 s window


def test_quiet_parts_fall_under_the_relative_gate():
    x = levels((-50.0, -35.0, -20.0, -35.0, -50.0))
    s = short_term_energies(x)
    rel = -0.691 + 10.0 * math.log10(s[lufs(s) > -70.0].mean()) - 20.0
    quiet = lufs(s[:171])                           # windows inside the first -50 dBFS part
    assert quiet.max() < rel < lufs(s[200 + 30:200 + 171]).min()   # ... under the gate; the -35 part over it


def test_steady_tone():
    lra, M, S = range_ref(tone(20 * FS, FS))
    # the 24 kHz value test_loudness.py pins for the integrated loudness of this tone
    assert abs(M - (-22.97)) <= 0.01 and abs(S - (-22.97)) <= 0.01
    assert 0.0 <= lra <= 0.01


def test_isolated_burst():
    # 1 s of the tone between 5 s of silence on each side, starting on a 2400-sample boundary
    x = np.concatenate([np.zeros(5 * FS), tone(FS, FS), np.zeros(5 * FS)])
    assert (5 * FS) % SEG == 0
    lra, M, S = range_ref(x)
    assert abs(M - (-22.97)) <= 0.01
    assert abs(S - (-22.97 + 10.0 * math.log10(1.0 / 3.0))) <= 0.02


@pytest.mark.parametrize("m,lo,hi", ((1, 0, 0), (2, 0, 1), (10, 1, 9), (21, 2, 19)))
def test_rank_rule(m, lo, hi):
    assert ranks(m) == (lo, hi)
    # the nearest rank of p (m - 1) with halves rounded up
    assert ranks(m) == (math.floor(0.10 * (m - 1) + 0.5), math.floor(0.95 * (m - 1) + 0.5))


def test_one_window_has_no_range():
    lra, M, S = range_ref(tone(WINDOW, FS))
    assert len(short_term_energies(tone(WINDOW, FS))) == 1
    assert lra == 0.0 and abs(S - (-22.97)) <= 0.01


@pytest.mark.parametrize("n", (1, BLOCK - 1))
def test_no_whole_block_is_undefined(n):
    lra, M, S = range_ref(tone(n, FS))
    assert math.isnan(M) and math.isnan(S) and math.isnan(lra)


def test_no_whole_window_is_undefined():
    lra, M, S = range_ref(tone(WINDOW - 1, FS))
    assert not math.isnan(M) and math.isnan(S) and math.isnan(lra)
    lra, M, S = range_ref(tone(WINDOW, FS))
    assert not math.isnan(S) and not math.isnan(lra)


def test_silence():
    lra, M, S = range_ref(np.zeros(5 * FS))
    assert M == -np.inf and S == -np.inf and math.isnan(lra)
