"""GPU tests (-m gpu) of the EBU R128 loudness report ("loudness_report", kernels_loudness.cu loud_short / loud_range):
the kernels against the float64 reference of test_loudness_range.py (kkx_test_loudness_range, synthetic signals from
1 sample to 2^25 samples), measure-only output bit-identical to the option off in every encoding and at several rates,
the model's report equal to the op-level report on the same samples (programs, frame groups, "max_tokens" passes), no
side effects with normalisation and the limiter on, the launch count, and argument errors."""
import ctypes as C
import math

import numpy as np
import pytest

from tests.conftest import synth_case
from tests.test_loudness_range import TECH3342, levels, range_ref

pytestmark = pytest.mark.gpu

# no block, one block, no window, one window, several, long
OP_LENS = (1, 9599, 9600, 71999, 72000, 180001, 1000003)
HUGE = (1 << 25) + 2400 * 3 + 7            # ~14 000 short-term windows: every radix pass loops over the CTA many times
ENCODINGS = ("f32", "pcm16", "ulaw", "alaw", "flac")


@pytest.fixture(scope="module")
def lib():
    from kokorox_b200.onn import load_library
    lib = load_library()
    lib.kkx_test_last_error.restype = C.c_char_p
    return lib


@pytest.fixture(scope="module")
def model(weights_path):
    from kokorox_b200.onn import B200Koko, init_ort
    init_ort()
    m = B200Koko.new(weights_path)      # the default (tensor-core) configuration
    yield m
    m.close()


@pytest.fixture
def opts(model):
    """Sets session options for one test and restores the defaults afterwards."""
    def set_opts(**kw):
        for k, v in kw.items():
            model.set_option(k, v)
    yield set_opts
    for k, v in (("loudness_report", 0), ("limiter", 0), ("loudness_target", 0), ("true_peak_max", -100),
                 ("out_rate", 24000), ("max_frames", 49152), ("max_tokens", 40960)):
        model.set_option(k, v)


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _pack(items):
    lens = np.asarray([len(x) for x in items], np.int64)
    x = np.ascontiguousarray(np.concatenate(items).astype(np.float32))
    return x, lens, lens.ctypes.data_as(C.POINTER(C.c_int64))


def op_range(lib, items):
    """kkx_test_loudness_range on packed items: [3][B] float32 (LRA, max momentary, max short-term)."""
    x, lens, lp = _pack(items)
    out = np.zeros((3, len(items)), np.float32)
    rc = lib.kkx_test_loudness_range(0, _fp(x), len(items), lp, _fp(out[0]), _fp(out[1]), _fp(out[2]))
    assert rc == 0, lib.kkx_test_last_error()
    return out


def op_loudness(lib, items):
    """kkx_test_loudness on packed items: [2][B] float32 (L, dBTP)."""
    x, lens, lp = _pack(items)
    out = np.zeros((3, len(items)), np.float32)
    rc = lib.kkx_test_loudness(0, _fp(x), len(items), lp, -2300, -100, _fp(out[0]), _fp(out[1]), _fp(out[2]))
    assert rc == 0, lib.kkx_test_last_error()
    return out[:2]


def speechlike(n, seed, level=0.1, swing_db=0.0):
    """Noise with a syllable-rate envelope and pauses; swing_db > 0 adds a slow level change (a 40 s sine in dB), so
    that the short-term values are spread out and the range is wide."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 24000.0
    env = np.maximum(np.sin(2 * np.pi * 3.1 * t + seed), 0.0) ** 2 + 0.02
    if swing_db:
        env = env * 10.0 ** (swing_db / 20.0 * np.sin(2 * np.pi * t / 40.0))
    return (level * env * rng.standard_normal(n)).astype(np.float32)


def check_values(got, x, what):
    want = range_ref(x.astype(np.float64))
    for k, name in enumerate(("LRA", "M", "S")):
        g, w = float(got[k]), want[k]
        if math.isnan(w) or math.isinf(w):
            assert (math.isnan(g) and math.isnan(w)) or g == w, (what, name, g, w)
        else:
            assert abs(g - w) <= 0.01, (what, name, g, w)
    return want


def check_alone(lib, items, out):
    for b, x in enumerate(items):
        one = op_range(lib, [x])
        assert np.array_equal(one[:, 0], out[:, b], equal_nan=True), b


def test_kernels_match_reference(lib):
    items = [speechlike(n, i) for i, n in enumerate(OP_LENS)]
    items.append(np.zeros(96000, np.float32))                                  # silence
    items += [levels(p).astype(np.float32) for p, _ in TECH3342]
    out = op_range(lib, items)
    for b, x in enumerate(items):
        check_values(out[:, b], x, (b, len(x)))
    assert math.isnan(out[1, 1]) and not math.isnan(out[1, 2])                # 9599: no block; 9600: one
    assert math.isnan(out[2, 3]) and math.isnan(out[0, 3]) and out[0, 4] == 0.0   # 71999: no window; 72000: one
    assert out[1, 7] == -np.inf and out[2, 7] == -np.inf and math.isnan(out[0, 7])
    for k, (_, want) in enumerate(TECH3342):
        assert abs(out[0, 8 + k] - want) <= 0.01, (k, out[0, 8 + k])
    check_alone(lib, items, out)


def test_kernels_on_a_long_item(lib):
    items = [speechlike(HUGE, 7, swing_db=10.0), speechlike(180001, 8, swing_db=10.0)]
    out = op_range(lib, items)
    for b, x in enumerate(items):
        check_values(out[:, b], x, b)
    assert out[0, 0] > 10.0                     # a wide range: the 10 % and 95 % points are far apart
    check_alone(lib, items, out)


def _batch(n_items=3, seed=0, lens=(140, 37, 260, 61, 190, 90)):
    cases = [synth_case(int(lens[i % len(lens)]), 9200 + seed + i, 9300 + seed + i) for i in range(n_items)]
    speeds = [(1.0, 1.25, 0.85, 1.1, 0.95, 1.2)[i % 6] for i in range(n_items)]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


def per_item(model, enc, toks, styles, speeds):
    if enc == "f32":
        return [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    if enc == "pcm16":
        return [a.copy() for a in model.infer_batch_pcm16(toks, styles, speeds)]
    if enc in ("ulaw", "alaw"):
        return [a.copy() for a in model.infer_batch_g711(toks, styles, speeds, law=enc)]
    return model.infer_batch_flac(toks, styles, speeds)


def programs(model, enc, toks, styles, speeds, poffs):
    out = model.infer_programs(toks, styles, speeds, poffs, encoding=enc)
    return out if enc == "flac" else [a.copy() for a in out]


def same(a, b):
    return a == b if isinstance(a, bytes) else np.array_equal(a, b)


@pytest.mark.parametrize("rate", (24000, 8000, 22050))
def test_measure_only_is_invisible(lib, model, opts, rate):
    toks, styles, speeds = _batch(4, seed=10)
    poffs = [0, 1, 4]
    plain24 = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    progs24 = [plain24[0], np.concatenate(plain24[1:4])]
    want_items, want_progs = op_loudness(lib, plain24), op_loudness(lib, progs24)
    # a ceiling under the loudest item's true peak: rule 5 would scale it, measuring must not
    ceiling = int(np.clip(math.floor(want_items[1].max()) - 3, -20, 0))
    assert want_items[1].max() > ceiling
    opts(out_rate=rate, true_peak_max=100 * ceiling)
    off_items = {e: per_item(model, e, toks, styles, speeds) for e in ENCODINGS}
    off_progs = {e: programs(model, e, toks, styles, speeds, poffs) for e in ENCODINGS}
    opts(loudness_report=1)
    for e in ENCODINGS:
        got = per_item(model, e, toks, styles, speeds)
        assert all(same(a, b) for a, b in zip(got, off_items[e])), (rate, e, "items")
        L, tp, g = model.last_loudness()
        assert np.all(g == 1.0), (rate, e, g)
        assert np.array_equal(L, want_items[0], equal_nan=True) and np.array_equal(tp, want_items[1]), (rate, e)
        got = programs(model, e, toks, styles, speeds, poffs)
        assert all(same(a, b) for a, b in zip(got, off_progs[e])), (rate, e, "programs")
        L, tp, g = model.last_loudness()
        assert np.all(g == 1.0), (rate, e, g)
        assert np.array_equal(L, want_progs[0], equal_nan=True) and np.array_equal(tp, want_progs[1]), (rate, e)


def test_model_report_is_the_op_level_report(lib, model, opts):
    toks, styles, speeds = _batch(6, seed=20)
    plain24, dur = model.infer_batch(toks, styles, speeds, return_durations=True)
    plain24 = [a.copy() for a in plain24]
    poffs = [0, 2, 3, 6]
    want = op_range(lib, [np.concatenate(plain24[a:b]) for a, b in zip(poffs[:-1], poffs[1:])])
    want_all = op_range(lib, [np.concatenate(plain24)])
    assert np.isfinite(want_all).all()          # long enough for whole 3 s windows
    opts(loudness_report=1)

    def check(where):
        model.infer_programs(toks, styles, speeds, poffs)
        assert np.array_equal(np.asarray(model.last_loudness_range(), np.float32), want, equal_nan=True), where
        model.infer_programs(toks, styles, speeds, [0, 6])
        assert np.array_equal(np.asarray(model.last_loudness_range(), np.float32), want_all), where

    check("one group")
    opts(max_frames=max(int(d.sum()) for d in dur))     # a program spans several frame groups
    check("frame groups")
    assert model.get_stat("frame_groups") > 1
    # per item, over the passes of a "max_tokens" split
    opts(max_frames=49152, max_tokens=512)
    model.infer_batch(toks, styles, speeds)
    assert np.array_equal(np.asarray(model.last_loudness_range(), np.float32), op_range(lib, plain24), equal_nan=True)


@pytest.mark.parametrize("limiter", (0, 1))
def test_no_side_effects_with_normalisation(model, opts, limiter):
    toks, styles, speeds = _batch(3, seed=30)
    opts(loudness_target=-1600, limiter=limiter)

    def run():
        outs = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
        rep = [np.asarray(model.last_loudness(), np.float32)]
        if limiter:
            rep.append(np.asarray(model.last_limiter(), np.float32))
        prog = model.infer_programs(toks, styles, speeds, [0, 3])[0].copy()
        rep.append(np.asarray(model.last_loudness(), np.float32))
        return outs, rep, prog

    outs0, rep0, prog0 = run()
    opts(loudness_report=1)
    outs1, rep1, prog1 = run()
    assert all(np.array_equal(a, b) for a, b in zip(outs0, outs1)) and np.array_equal(prog0, prog1)
    assert all(np.array_equal(a, b, equal_nan=True) for a, b in zip(rep0, rep1))
    assert len(model.last_loudness_range()[0]) == 1


def test_default_off_and_launch_count(model, opts, weights_path):
    from kokorox_b200.onn import B200Koko, KkxError
    toks, styles, speeds = _batch(3, seed=40)
    fresh = B200Koko.new(weights_path)
    try:
        want = [a.copy() for a in fresh.infer_batch(toks, styles, speeds)]
        want_launches = fresh.get_stat("launches")
        assert fresh.get_stat("loudness_report") == 0
        with pytest.raises(KkxError) as e:      # report off: nothing to report
            fresh.last_loudness_range()
        assert e.value.code == -5
    finally:
        fresh.close()
    got = model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") == want_launches
    assert all(np.array_equal(a, b) for a, b in zip(got, want))
    for mf in (49152, 300):
        opts(max_frames=mf, loudness_report=0)
        model.infer_batch(toks, styles, speeds)
        plain, groups = model.get_stat("launches"), model.get_stat("frame_groups")
        # measure-only at 24 kHz: the loudness kernels, loud_short, loud_range and the resampling pass-through
        opts(loudness_report=1)
        model.infer_batch(toks, styles, speeds)
        assert model.get_stat("launches") - plain == (3 + 2 + 1) * groups, mf
        assert model.get_stat("frame_groups") == groups
        # with a target (and with the limiter as well): the two report kernels
        for lim in (0, 1):
            opts(loudness_report=0, loudness_target=-1600, limiter=lim)
            model.infer_batch(toks, styles, speeds)
            base = model.get_stat("launches")
            opts(loudness_report=1)
            model.infer_batch(toks, styles, speeds)
            assert model.get_stat("launches") - base == 2 * groups, (mf, lim)
        opts(loudness_target=0, limiter=0)
    assert groups > 1


def test_rejected_values_and_report_errors(model, opts):
    from kokorox_b200.onn import KkxError
    opts(loudness_report=1)
    for v in (2, -1):
        with pytest.raises(KkxError):
            model.set_option("loudness_report", v)
        assert model.get_stat("loudness_report") == 1
    toks, styles, speeds = _batch(2, seed=50)
    model.infer_batch(toks, styles, speeds)
    assert model.get_stat("loudness_items") == 2
    lra = np.zeros(3, np.float32)
    assert model._lib.kkx_last_loudness_range(model._ctx, 3, _fp(lra), None, None) == -1
    assert model._lib.kkx_last_loudness_range(model._ctx, 2, None, None, None) == 0
    model.set_option("loudness_report", 0)
    model.infer_batch(toks, styles, speeds)
    assert model._lib.kkx_last_loudness_range(model._ctx, 2, None, None, None) == -5
    assert model.get_stat("loudness_items") == 0
    with pytest.raises(KkxError) as e:
        model.last_loudness()
    assert e.value.code == -5
