"""GPU tests (-m gpu) of the lookahead true-peak limiter ("limiter", kernels_loudness.cu): the kernels against the
float64 reference of test_limiter.py (kkx_test_limiter, synthetic signals of many lengths), the model's limited output
against the reference applied to the same session's plain 24 kHz output at several "out_rate" values and encodings,
the no-op cases, bit-identity of an item across batches, frame groups, passes, coalesced and asynchronous batches and
programs, the default-off guarantee with the launch count, and argument errors."""
import ctypes as C
import math
import threading

import numpy as np
import pytest
from scipy.signal import resample_poly

from tests.conftest import synth_case
from tests.test_flac import flac_decode_ref
from tests.test_limiter import limiter_ref, speech_with_transients
from tests.test_loudness import true_peak_ref
from tests.test_resample import alaw_ref, pcm16_ref, ratio, ulaw_ref

pytestmark = pytest.mark.gpu

# 1, below the lookahead, around the 8192-sample tile, across several tiles, and long
OP_LENS = (1, 100, 8191, 8192, 8193, 24000, 180001, 1000003)
LONG = 65536 * 600 + 2400 * 7 + 1        # a program beyond one call's 65 536-frame cap (test_programs_gpu.py)


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
    for k, v in (("limiter", 0), ("loudness_target", 0), ("true_peak_max", -100), ("out_rate", 24000),
                 ("max_frames", 49152), ("max_tokens", 40960), ("coalesce", 0), ("coalesce_wait_us", 0)):
        model.set_option(k, v)


def op_limiter(lib, items, target, ceiling):
    """kkx_test_limiter on packed items: per item (g, G, v, t, max reduction dB, output dBTP)."""
    lens = np.asarray([len(x) for x in items], np.int64)
    x = np.ascontiguousarray(np.concatenate(items).astype(np.float32))
    B, N = len(items), len(x)
    g, t, red, tp = (np.zeros(B, np.float32) for _ in range(4))
    G, v = np.zeros(N, np.float32), np.zeros(N, np.float32)
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    rc = lib.kkx_test_limiter(0, fp(x), B, lens.ctypes.data_as(C.POINTER(C.c_int64)), target, ceiling, fp(g), fp(G),
                              fp(v), fp(t), fp(red), fp(tp))
    assert rc == 0, lib.kkx_test_last_error()
    off = np.concatenate([[0], np.cumsum(lens)])
    return [(g[b], G[off[b]:off[b + 1]], v[off[b]:off[b + 1]], t[b], red[b], tp[b]) for b in range(B)]


def db(a):
    return 20.0 * np.log10(np.asarray(a, np.float64))


def op_items():
    items = []
    for i, n in enumerate(OP_LENS):
        # at 3x the speech-like items' true peak is ~ +6 dBTP: limited also without normalisation
        x = 3 * speech_with_transients(n, i) if n >= 24000 else np.zeros(n, np.float32)
        if n < 24000:                       # short items: a burst near the end, reaching beyond the item
            x[max(0, n - 60):] = 1.4 * np.cos(np.arange(min(n, 60)) * 0.7)
        items.append(x)
    items.append(np.zeros(30000, np.float32))                                      # silence
    items.append((0.05 * np.sin(2 * np.pi * 440 * np.arange(30000) / 24000)).astype(np.float32))   # under the ceiling
    return items


def check_item(got, x, target, ceiling, what):
    g, G, v, t, red, tp = got
    r = limiter_ref(x, target / 100.0, ceiling / 100.0)
    assert abs(db(g) - db(r["g"])) <= 0.01, (what, g, r["g"])
    assert np.abs(db(G) - db(r["G"])).max() <= 0.01, what
    assert abs(db(t) - db(r["t"])) <= 0.01, (what, t, r["t"])
    assert abs(red - r["red"]) <= 0.01, (what, red, r["red"])
    if math.isinf(r["out_db"]):
        assert math.isinf(tp) and tp < 0, what
    else:
        assert abs(tp - r["out_db"]) <= 0.01, (what, tp, r["out_db"])
        assert 20 * math.log10(true_peak_ref(v * np.float32(t))) <= ceiling / 100.0 + 0.001, what
    # v is the rule's product of the device's own g and G
    assert np.array_equal(v, (x * (np.float32(g) * G.astype(np.float32)).astype(np.float32)).astype(np.float32)), what
    return r


@pytest.mark.parametrize("target", (-1400, 0))
def test_kernels_match_reference(lib, target):
    items = op_items()
    ceiling = -100
    out = op_limiter(lib, items, target, ceiling)
    for b, x in enumerate(items):
        r = check_item(out[b], x, target, ceiling, (target, len(x), b))
        if not x.any() or r["red"] == 0.0:    # silence and the quiet tone: untouched, bit for bit
            assert np.all(out[b][1] == 1.0) and out[b][3] == 1.0 and out[b][4] == 0.0, b
            assert np.array_equal(out[b][2], x * np.float32(out[b][0])), b
    assert out[-3][4] > 3.0 and out[-4][4] > 3.0      # the speech-like items were limited
    # purity: each item alone gives the same bits as in the batch
    for b, x in enumerate(items):
        one = op_limiter(lib, [x], target, ceiling)[0]
        for k in range(6):
            assert np.array_equal(np.asarray(one[k]), np.asarray(out[b][k])), (b, k)


def test_kernels_at_program_length(lib):
    items = [speech_with_transients(24000, 1), speech_with_transients(LONG, 2), speech_with_transients(9601, 3)]
    out = op_limiter(lib, items, -1400, -100)
    for b, x in enumerate(items):
        check_item(out[b], x, -1400, -100, b)


def _batch(n_items=3, seed=0, lens=(140, 37, 260)):
    cases = [synth_case(int(lens[i % len(lens)]), 9800 + seed + i, 9900 + seed + i) for i in range(n_items)]
    speeds = [1.0, 1.25, 0.85, 1.1, 0.95, 1.2][:n_items]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


def _expected(plain24, target, ceiling, rate):
    """The reference pipeline (steps 1-8) on the session's plain 24 kHz output of one item."""
    r = limiter_ref(plain24, target, ceiling)
    y = r["v"].astype(np.float64)
    if rate != 24000:
        U, D = ratio(rate)
        y = resample_poly(y, U, D)
    return y * r["t"], r


@pytest.mark.parametrize("rate", (24000, 8000, 22050, 48000))
def test_limited_output_matches_reference(model, opts, rate):
    toks, styles, speeds = _batch()
    plain = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    opts(out_rate=rate, loudness_target=-500, limiter=1)      # a high target: the random-weight audio is limited
    on = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    red, tp = model.last_limiter()
    g = model.last_loudness()[2]
    assert len(red) == 3
    for b in range(3):
        want, r = _expected(plain[b], -5.0, -1.0, rate)
        assert len(on[b]) == len(want)
        assert r["red"] > 0.0 and red[b] > 0.0, b
        assert abs(db(g[b]) - db(r["g"])) <= 0.01
        assert abs(red[b] - r["red"]) <= 0.01 and abs(tp[b] - r["out_db"]) <= 0.01, (b, red[b], r["red"])
        assert np.abs(on[b] - want).max() <= 3e-3 * np.abs(want).max(), (rate, b)
        if rate == 24000:
            assert 20 * math.log10(true_peak_ref(on[b])) <= -1.0 + 0.001, b
    # 16-bit PCM, G.711 and FLAC are derived from the limited value
    p = model.infer_batch_pcm16(toks, styles, speeds)
    u = model.infer_batch_g711(toks, styles, speeds, law="ulaw")
    a = model.infer_batch_g711(toks, styles, speeds, law="alaw")
    files = model.infer_batch_flac(toks, styles, speeds)
    for b in range(3):
        assert np.array_equal(p[b], pcm16_ref(on[b]))
        assert np.abs(p[b].astype(np.int32)).max() < 32767
        assert np.array_equal(u[b], ulaw_ref(p[b])) and np.array_equal(a[b], alaw_ref(p[b]))
        assert np.array_equal(flac_decode_ref(files[b])[0], p[b])


def test_limiter_without_loudness(model, opts):
    from kokorox_b200.onn import KkxError
    toks, styles, speeds = _batch(seed=10)
    plain = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    # a ceiling 6 dB under the quietest item's true peak (within the option's range): limited without any target
    C = int(np.clip(round(min(20 * math.log10(true_peak_ref(a)) for a in plain) - 6.0), -20, 0))
    opts(limiter=1, true_peak_max=100 * C)
    on = model.infer_batch(toks, styles, speeds)
    red, tp = model.last_limiter()
    with pytest.raises(KkxError) as e:                        # loudness is off: nothing to report there
        model.last_loudness()
    assert e.value.code == -5
    for b in range(3):
        want, r = _expected(plain[b], 0.0, float(C), 24000)
        assert r["g"] <= 1.0 and red[b] > 0.0
        assert np.abs(on[b] - want).max() <= 3e-3 * np.abs(want).max(), b
        assert 20 * math.log10(true_peak_ref(on[b])) <= C + 0.001, b
        assert abs(red[b] - r["red"]) <= 0.01, b


def test_untouched_items_are_bit_identical(model, opts):
    toks, styles, speeds = _batch(seed=20)
    # quiet target: g tp stays under the ceiling, so G = 1 and t = 1; same g as with the limiter off
    opts(loudness_target=-4000)
    off = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    g_off = model.last_loudness()[2].copy()
    opts(limiter=1)
    on = model.infer_batch(toks, styles, speeds)
    red, _ = model.last_limiter()
    assert np.array_equal(model.last_loudness()[2], g_off)
    for b in range(3):
        assert red[b] == 0.0 and np.array_equal(on[b], off[b]), b
    # a short item (L undefined) under the ceiling, loudness off: exactly the plain output
    tok, style = synth_case(3, 9700, 9701)
    opts(loudness_target=0, limiter=0)
    plain = model.infer_one(tok, style, 10.0).copy()
    assert model.get_stat("last_frames") < 16
    tp_db = 20 * math.log10(true_peak_ref(plain))
    assert tp_db < -0.5, tp_db
    opts(limiter=1, true_peak_max=0)
    got = model.infer_one(tok, style, 10.0)
    assert np.array_equal(got, plain)
    red, tp = model.last_limiter()
    assert red[0] == 0.0 and abs(tp[0] - tp_db) <= 0.01


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


@pytest.mark.parametrize("rate", (24000, 22050))
def test_item_bits_do_not_depend_on_the_batch(model, opts, rate):
    toks, styles, speeds = _batch(5, seed=50, lens=(200, 61, 333, 148, 90))
    opts(out_rate=rate, loudness_target=-500, limiter=1)      # a high target: every item is limited
    alone, rep = [], []
    for t, s, sp in zip(toks, styles, speeds):
        alone.append(model.infer_one(t, s, sp).copy())
        rep.append([v[0] for v in model.last_limiter()])
    rep = np.asarray(rep, np.float32).T          # [2][5]
    assert (rep[0] > 0).all()

    def same(outs, what):
        for b in range(5):
            assert np.array_equal(outs[b], alone[b]), f"{what}: item {b} differs from its own call"

    def same_report(what):
        assert np.array_equal(np.asarray(model.last_limiter(), np.float32), rep), what

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
    # one-item programs are the per-item calls, report included
    progs = [a.copy() for a in model.infer_programs(toks, styles, speeds, [0, 1, 2, 3, 4, 5])]
    same(progs, "one-item programs")
    same_report("one-item programs")
    # a program of items 1..3 is one utterance: its bits do not depend on the programs around it or on frame groups
    whole = model.infer_programs(toks[1:4], styles[1:4], speeds[1:4], [0, 3])[0].copy()
    whole_rep = np.asarray(model.last_limiter(), np.float32)
    mixed = model.infer_programs(toks, styles, speeds, [0, 1, 4, 5])
    assert np.array_equal(mixed[1], whole) and np.array_equal(mixed[0], alone[0]) and np.array_equal(mixed[2], alone[4])
    assert np.array_equal(np.asarray(model.last_limiter(), np.float32)[:, 1], whole_rep[:, 0])
    opts(max_frames=300)
    mixed = model.infer_programs(toks, styles, speeds, [0, 1, 4, 5])
    assert np.array_equal(mixed[1], whole), "program across frame groups"


def test_default_off_and_launch_count(model, opts, weights_path):
    from kokorox_b200.onn import B200Koko, KkxError
    toks, styles, speeds = _batch(seed=90)
    fresh = B200Koko.new(weights_path)
    try:
        want = [a.copy() for a in fresh.infer_batch(toks, styles, speeds)]
        want_launches = fresh.get_stat("launches")
        assert fresh.get_stat("limiter") == 0 and fresh.get_stat("limiter_items") == 0
        with pytest.raises(KkxError) as e:      # limiter off: nothing to report
            fresh.last_limiter()
        assert e.value.code == -5
    finally:
        fresh.close()
    opts(limiter=0)
    got = model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") == want_launches
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    groups = model.get_stat("frame_groups")
    # loudness on: the limiter adds lim_envelope, loud_peak and lim_trim per frame group
    opts(loudness_target=-1400)
    model.infer_batch(toks, styles, speeds)
    loud = model.get_stat("launches")
    opts(limiter=1)
    model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") - loud == 3 * groups
    # loudness off: the three loudness kernels run as well, and at 24 kHz the resampling pass-through
    opts(loudness_target=0)
    model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") - want_launches == 7 * groups
    opts(limiter=0, out_rate=16000)
    model.infer_batch(toks, styles, speeds)
    l16 = model.get_stat("launches")
    opts(limiter=1)
    model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") - l16 == 6 * model.get_stat("frame_groups")


def test_rejected_values_and_report_errors(model, opts):
    from kokorox_b200.onn import KkxError
    opts(limiter=1)
    for v in (2, -1, 100):
        with pytest.raises(KkxError):
            model.set_option("limiter", v)
        assert model.get_stat("limiter") == 1
    toks, styles, speeds = _batch(2, seed=30)
    model.infer_batch(toks, styles, speeds)
    assert model.get_stat("limiter_items") == 2
    red = np.zeros(3, np.float32)
    assert model._lib.kkx_last_limiter(model._ctx, 3, red.ctypes.data_as(C.POINTER(C.c_float)), None) == -1
    assert model._lib.kkx_last_limiter(model._ctx, 2, None, None) == 0
    model.set_option("limiter", 0)
    model.infer_batch(toks, styles, speeds)
    assert model._lib.kkx_last_limiter(model._ctx, 2, None, None) == -5
    assert model.get_stat("limiter_items") == 0
