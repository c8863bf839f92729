"""GPU tests (-m gpu) of loudness normalisation ("loudness_target" / "true_peak_max", kernels_loudness.cu): the kernels
against the float64 reference of test_loudness.py, the model's normalised output against its own unnormalised output
and the reported gain at several "out_rate" values (PCM16, G.711 and FLAC included), bit-identity of an item across
batches, frame groups, passes, coalesced and asynchronous batches, the default-off guarantee, and argument errors."""
import ctypes as C
import math
import threading

import numpy as np
import pytest

from tests.conftest import synth_case
from tests.test_flac import flac_decode_ref
from tests.test_loudness import gain_ref, loudness_ref, true_peak_ref
from tests.test_resample import alaw_ref, pcm16_ref, ulaw_ref

pytestmark = pytest.mark.gpu

OP_LENS = (1, 9599, 9600, 9601, 24000, 180001, 1000003)


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
    for k, v in (("loudness_target", 0), ("true_peak_max", -100), ("out_rate", 24000), ("max_frames", 49152),
                 ("max_tokens", 40960), ("coalesce", 0), ("coalesce_wait_us", 0)):
        model.set_option(k, v)


def op_loudness(lib, items, target=-2300, ceiling=-100):
    lens = np.asarray([len(x) for x in items], np.int64)
    x = np.ascontiguousarray(np.concatenate(items).astype(np.float32))
    B = len(items)
    L, tp, g = (np.zeros(B, np.float32) for _ in range(3))
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    rc = lib.kkx_test_loudness(0, fp(x), B, lens.ctypes.data_as(C.POINTER(C.c_int64)), target, ceiling, fp(L), fp(tp),
                               fp(g))
    assert rc == 0, lib.kkx_test_last_error()
    return L, tp, g


def speechlike(n, seed, level=0.1):
    """Noise with a syllable-rate envelope and pauses: the gates have something to do."""
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 24000.0
    env = np.maximum(np.sin(2 * np.pi * 3.1 * t + seed), 0.0) ** 2 + 0.02
    return (level * env * rng.standard_normal(n)).astype(np.float32)


def op_items():
    items = [speechlike(n, i) for i, n in enumerate(OP_LENS)]
    items.append(np.zeros(48000, np.float32))                                  # silence: undefined
    n = 72000                                                                  # fs / 4, 3 s: true peak > sample peak
    items.append((0.5 * np.sin(2 * np.pi * 6000 * np.arange(n) / 24000 + np.pi / 4)).astype(np.float32))
    return items


def test_kernels_match_reference(lib):
    items = op_items()
    L, tp, g = op_loudness(lib, items, -2300, -100)
    for b, x in enumerate(items):
        Lr = loudness_ref(x.astype(np.float64))
        tpr = true_peak_ref(x.astype(np.float64))
        if math.isnan(Lr):
            assert math.isnan(L[b]) and g[b] == 1.0, b
        else:
            assert abs(L[b] - Lr) <= 0.01, (b, L[b], Lr)
            gr = gain_ref(Lr, tpr, -23.0, -1.0)
            assert abs(20 * math.log10(g[b] / gr)) <= 0.02, (b, g[b], gr)
        if tpr == 0.0:
            assert tp[b] == -np.inf
        else:
            assert abs(tp[b] - 20 * math.log10(tpr)) <= 0.01, (b, tp[b], tpr)
    assert len(items[0]) < 9600 and math.isnan(L[0]) and math.isnan(L[1]) and not math.isnan(L[2])
    sine = items[-1]
    assert tp[-1] > 20 * math.log10(np.abs(sine).max()) + 2.0     # the 4x peak sees the crests between the samples
    # peak-limited: -5 LUFS would put the sine's true peak near -5.3 dBTP; a -10 dBTP ceiling holds it there
    Ls, tps, gs = op_loudness(lib, [sine], -500, -1000)
    assert -5.0 - Ls[0] + tps[0] > -10.0
    assert abs(20 * math.log10(gs[0]) + tps[0] - (-10.0)) <= 1e-4
    # each item alone gives the same bits as in the batch
    for b, x in enumerate(items):
        one = op_loudness(lib, [x], -2300, -100)
        for k in range(3):
            assert np.array_equal(one[k], np.asarray([(L, tp, g)[k][b]]), equal_nan=True), (b, k)


def _batch(n_items=3, seed=0, lens=(140, 37, 260)):
    cases = [synth_case(int(lens[i % len(lens)]), 9500 + seed + i, 9600 + seed + i) for i in range(n_items)]
    speeds = [1.0, 1.25, 0.85, 1.1, 0.95, 1.2][:n_items]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


@pytest.mark.parametrize("r", (24000, 8000, 22050, 48000))
def test_normalised_output_is_the_plain_output_times_the_gain(model, opts, r):
    toks, styles, speeds = _batch()
    opts(out_rate=24000)
    w24 = [a.astype(np.float64) for a in model.infer_batch(toks, styles, speeds)]
    opts(out_rate=r)
    off = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    opts(loudness_target=-2300)
    on = model.infer_batch(toks, styles, speeds)
    L, tp, g = model.last_loudness()
    assert len(L) == 3
    for b in range(3):
        assert np.array_equal(on[b], np.float32(off[b] * g[b])), (r, b)
        # measured on the 24 kHz waveform, whatever the output rate
        Lr = loudness_ref(w24[b])
        assert abs(L[b] - Lr) <= 0.01, (r, b, L[b], Lr)
        assert abs(tp[b] - 20 * math.log10(true_peak_ref(w24[b]))) <= 0.01
    # 16-bit PCM, G.711 and FLAC are derived from the normalised value
    p = model.infer_batch_pcm16(toks, styles, speeds)
    assert np.array_equal(model.last_loudness()[2], g)
    u = model.infer_batch_g711(toks, styles, speeds, law="ulaw")
    a = model.infer_batch_g711(toks, styles, speeds, law="alaw")
    files = model.infer_batch_flac(toks, styles, speeds)
    for b in range(3):
        assert np.array_equal(p[b], pcm16_ref(on[b]))
        assert np.array_equal(u[b], ulaw_ref(p[b])) and np.array_equal(a[b], alaw_ref(p[b]))
        assert np.array_equal(flac_decode_ref(files[b])[0], p[b])


def test_low_target_is_reached(model, opts):
    toks, styles, speeds = _batch(seed=10)
    opts(loudness_target=-4000)
    out = model.infer_batch(toks, styles, speeds)
    L = model.last_loudness()[0]
    for b in range(3):
        assert not math.isnan(L[b])
        assert abs(loudness_ref(out[b].astype(np.float64)) - (-40.0)) <= 0.02, b


def test_true_peak_ceiling_holds(model, opts):
    toks, styles, speeds = _batch(seed=20)
    opts(loudness_target=-500, true_peak_max=-100)
    out = model.infer_batch(toks, styles, speeds)
    for b in range(3):
        assert 20 * math.log10(true_peak_ref(out[b].astype(np.float64))) <= -1.0 + 0.01, b
    for r in (24000, 8000, 22050, 48000):
        opts(out_rate=r)
        for p in model.infer_batch_pcm16(toks, styles, speeds):
            assert np.abs(p.astype(np.int32)).max() < 32767, r


def _run_threads(fn, n):
    res, errs = [None] * n, [None] * n

    def work(i):
        try:
            res[i] = fn(i)
        except Exception as e:  # noqa: BLE001 -- collected and asserted by the caller
            errs[i] = e
    ts = [threading.Thread(target=work, args=(i,)) for i in range(n)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return res, errs


@pytest.mark.parametrize("r", (24000, 22050))
def test_item_bits_do_not_depend_on_the_batch(model, opts, r):
    toks, styles, speeds = _batch(5, seed=50, lens=(200, 61, 333, 148, 90))
    opts(out_rate=r, loudness_target=-1600)
    alone, rep = [], []
    for t, s, sp in zip(toks, styles, speeds):
        alone.append(model.infer_one(t, s, sp).copy())
        rep.append([v[0] for v in model.last_loudness()])
    rep = np.asarray(rep, np.float32).T          # [3][5]

    def same(outs, what):
        for b in range(5):
            assert np.array_equal(outs[b], alone[b]), f"{what}: item {b} differs from its own call"

    def same_report(what):
        got = np.asarray(model.last_loudness(), np.float32)
        assert np.array_equal(got, rep, equal_nan=True), what

    same(model.infer_batch(toks, styles, speeds), "batch")
    same_report("batch")
    opts(max_frames=300)                          # several frame groups
    same(model.infer_batch(toks, styles, speeds), "frame groups")
    assert model.get_stat("frame_groups") > 1
    same_report("frame groups")
    opts(max_frames=49152, max_tokens=512)      # several passes of one call
    same(model.infer_batch(toks, styles, speeds), "passes")
    same_report("passes")
    opts(max_tokens=40960, coalesce=5, coalesce_wait_us=500000)
    res, errs = _run_threads(lambda i: model.infer_one(toks[i], styles[i], speeds[i]), 5)
    opts(coalesce=0, coalesce_wait_us=0)
    assert all(e is None for e in errs), errs
    same(res, "coalesced")
    t = model.submit(toks[2], styles[2], speeds[2])
    assert np.array_equal(model.wait(t), alone[2]), "submit"


def test_short_item_is_left_alone(model, opts):
    tok, style = synth_case(3, 9700, 9701)
    plain = model.infer_one(tok, style, 10.0).copy()
    assert model.get_stat("last_frames") < 16
    opts(loudness_target=-1600)
    got = model.infer_one(tok, style, 10.0)
    assert np.array_equal(got, plain)
    L, _, g = model.last_loudness()
    assert math.isnan(L[0]) and g[0] == 1.0


def test_default_off_and_launch_count(model, opts, weights_path):
    from kokorox_b200.onn import B200Koko, KkxError
    toks, styles, speeds = _batch(seed=90)
    fresh = B200Koko.new(weights_path)
    try:
        want = [a.copy() for a in fresh.infer_batch(toks, styles, speeds)]
        want_launches = fresh.get_stat("launches")
        assert fresh.get_stat("loudness_target") == 0 and fresh.get_stat("true_peak_max") == -100
        with pytest.raises(KkxError) as e:      # normalisation off: nothing to report
            fresh.last_loudness()
        assert e.value.code == -5
    finally:
        fresh.close()
    opts(loudness_target=-2300)
    model.infer_batch(toks, styles, speeds)
    on_launches = model.get_stat("launches")
    groups = model.get_stat("frame_groups")
    opts(loudness_target=0)
    got = model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") == want_launches
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    # at 24 kHz: 3 loudness kernels + the resampling pass-through per frame group; at other rates 3
    assert on_launches - want_launches == 4 * groups
    opts(out_rate=16000)
    model.infer_batch(toks, styles, speeds)
    l16 = model.get_stat("launches")
    opts(loudness_target=-2300)
    model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") - l16 == 3 * model.get_stat("frame_groups")


def test_rejected_values_and_report_errors(model, opts):
    from kokorox_b200.onn import KkxError
    opts(loudness_target=-1600, true_peak_max=-200)
    for v in (1, -499, -7001, 100, -100000):
        with pytest.raises(KkxError):
            model.set_option("loudness_target", v)
        assert model.get_stat("loudness_target") == -1600
    for v in (1, -2001, 100):
        with pytest.raises(KkxError):
            model.set_option("true_peak_max", v)
        assert model.get_stat("true_peak_max") == -200
    for v in (-7000, -500):
        model.set_option("loudness_target", v)
        assert model.get_stat("loudness_target") == v
    toks, styles, speeds = _batch(2, seed=30)
    model.infer_batch(toks, styles, speeds)
    n = C.c_int32(2)
    L = np.zeros(3, np.float32)
    assert model._lib.kkx_last_loudness(model._ctx, 3, L.ctypes.data_as(C.POINTER(C.c_float)), None, None) == -1
    assert model._lib.kkx_last_loudness(model._ctx, n, None, None, None) == 0
    model.set_option("loudness_target", 0)
    model.infer_batch(toks, styles, speeds)
    assert model._lib.kkx_last_loudness(model._ctx, 2, None, None, None) == -5
