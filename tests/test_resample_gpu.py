"""GPU tests (-m gpu) of the output-format path: the resampling kernel against float64 scipy.signal.resample_poly, the
"out_rate" option through every waveform entry point (batch invariance included), 16-bit PCM and G.711 output, and
the default rate's bit-for-bit, launch-for-launch equality with a session that never touched the option."""
import ctypes as C
import math
import threading

import numpy as np
import pytest
from scipy.signal import resample_poly

from tests.conftest import synth_case
from tests.test_resample import RATES, alaw_ref, pcm16_ref, ratio, ulaw_ref

pytestmark = pytest.mark.gpu

OP_LENS = (1, 5, 599, 600, 1237, 24000, 180001, 1000003)


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
def rate(model):
    """Sets "out_rate" for one test and restores the default afterwards."""
    def set_rate(r):
        model.set_option("out_rate", r)
    yield set_rate
    model.set_option("out_rate", 24000)


def out_len(n, r):
    U, D = ratio(r)
    return -(-n * U // D)


def op_resample(lib, items, r, law):
    lens = np.asarray([len(x) for x in items], np.int64)
    x = np.ascontiguousarray(np.concatenate(items).astype(np.float32))
    n_out = sum(out_len(int(n), r) for n in lens)
    out = np.zeros(n_out, np.float32)
    pcm = np.zeros(n_out, np.int16)
    codes = np.zeros(n_out, np.uint8)
    rc = lib.kkx_test_resample(0, x.ctypes.data_as(C.POINTER(C.c_float)), len(items),
                               lens.ctypes.data_as(C.POINTER(C.c_int64)), r, law,
                               out.ctypes.data_as(C.POINTER(C.c_float)), pcm.ctypes.data_as(C.POINTER(C.c_int16)),
                               codes.ctypes.data_as(C.POINTER(C.c_uint8)))
    assert rc == 0, lib.kkx_test_last_error()
    offs = np.concatenate([[0], np.cumsum([out_len(int(n), r) for n in lens])])
    return out, pcm, codes, offs


@pytest.mark.parametrize("r", RATES)
def test_resample_kernel_matches_resample_poly(lib, r):
    rng = np.random.default_rng(r)
    # amplitude ~0.6: some samples pass +-1, so the PCM clamp is exercised too
    items = [(rng.standard_normal(n) * 0.6).astype(np.float32) for n in OP_LENS]
    U, D = ratio(r)
    out, pcm, codes_u, offs = op_resample(lib, items, r, 0)
    out_a, pcm_a, codes_a, _ = op_resample(lib, items, r, 1)
    assert np.array_equal(out, out_a) and np.array_equal(pcm, pcm_a)
    for b, x in enumerate(items):
        y = out[offs[b]:offs[b + 1]]
        ref = resample_poly(x.astype(np.float64), U, D)
        assert len(y) == len(ref) == out_len(len(x), r)
        assert np.abs(y - ref).max() <= 1e-5 * np.abs(x).max(), (r, len(x))
        if r == 24000:     # pass-through: the input itself
            assert np.array_equal(y, x)
    # the 16-bit and G.711 twins are conversions of the kernel's own f32 output, bit for bit
    assert np.array_equal(pcm, pcm16_ref(out))
    assert np.array_equal(codes_u, ulaw_ref(pcm))
    assert np.array_equal(codes_a, alaw_ref(pcm))


def _batch(n_items=3, seed=0, lens=(140, 37, 260)):
    cases = [synth_case(int(lens[i % len(lens)]), 9000 + seed + i, 9100 + seed + i) for i in range(n_items)]
    speeds = [1.0, 1.25, 0.85, 1.1, 0.95, 1.2][:n_items]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


@pytest.mark.parametrize("r", (8000, 16000, 22050, 44100, 48000))
def test_model_output_at_rate_matches_resample_poly(model, rate, r):
    toks, styles, speeds = _batch()
    ref24 = [a.copy() for a in model.infer_batch(toks, styles, speeds)]
    rate(r)
    got = model.infer_batch(toks, styles, speeds)
    U, D = ratio(r)
    for b in range(3):
        assert len(got[b]) == out_len(len(ref24[b]), r)
        ref = resample_poly(ref24[b].astype(np.float64), U, D)
        assert np.abs(got[b] - ref).max() <= 1e-5 * np.abs(ref24[b]).max(), (r, b)
    # the device-resident path reports the same lengths as offsets
    model.stage(toks, styles, speeds)
    total, _ = model.run_staged()
    wav, soff, _ = model.fetch_staged(total)
    assert total == sum(len(g) for g in got)
    for b in range(3):
        assert soff[b + 1] - soff[b] == len(got[b])
        assert np.array_equal(wav[soff[b]:soff[b + 1]], got[b])


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


def test_batch_invariance_at_22050(model, rate):
    # 22050 Hz: U / D = 147 / 160, so item offsets at the output rate are not multiples of 4
    toks, styles, speeds = _batch(5, seed=50, lens=(200, 61, 333, 148, 90))
    rate(22050)
    alone = [model.infer_one(t, s, sp).copy() for t, s, sp in zip(toks, styles, speeds)]
    assert any(len(a) % 4 for a in alone)
    batch = model.infer_batch(toks, styles, speeds)
    for b in range(5):
        assert np.array_equal(batch[b], alone[b]), f"item {b}: batch differs from its own call"
    # several passes of one call
    model.set_option("max_tokens", 512)
    try:
        passes = model.infer_batch(toks, styles, speeds)
    finally:
        model.set_option("max_tokens", 40960)
    for b in range(5):
        assert np.array_equal(passes[b], alone[b]), f"item {b}: multi-pass result differs"
    # coalesced concurrent callers
    before = model.get_stat("coalesced_batches")
    model.set_option("coalesce", 5)
    model.set_option("coalesce_wait_us", 500000)
    try:
        res, errs = _run_threads(lambda i: model.infer_one(toks[i], styles[i], speeds[i]), 5)
    finally:
        model.set_option("coalesce", 0)
        model.set_option("coalesce_wait_us", 0)
    assert all(e is None for e in errs), errs
    assert model.get_stat("coalesced_batches") > before
    for b in range(5):
        assert np.array_equal(res[b], alone[b]), f"caller {b}: coalesced result differs"
    # asynchronous submit / wait
    t = model.submit(toks[2], styles[2], speeds[2])
    assert np.array_equal(model.wait(t), alone[2])
    # styles mixed on the device from a voice table whose row len - 2 of voice b is style b
    table = {f"v{b}": np.zeros((511, 256), np.float32) for b in range(5)}
    for b in range(5):
        table[f"v{b}"][len(toks[b]) - 2] = styles[b]
    model.load_voices(table)
    voiced = model.infer_batch_voices(toks, [f"v{b}" for b in range(5)], speeds)
    for b in range(5):
        assert np.array_equal(voiced[b], alone[b]), f"item {b}: device-mixed styles differ"
    # device-resident run + fetch
    model.stage(toks, styles, speeds)
    total, _ = model.run_staged()
    wav, soff, _ = model.fetch_staged(total)
    assert total == sum(len(a) for a in alone)
    for b in range(5):
        assert np.array_equal(wav[soff[b]:soff[b + 1]], alone[b])


def test_pcm16_and_g711_output(model, rate):
    from kokorox_b200.onn import KkxError
    toks, styles, speeds = _batch(seed=70)
    rate(16000)
    f = model.infer_batch(toks, styles, speeds)
    p = model.infer_batch_pcm16(toks, styles, speeds)
    for a, b in zip(f, p):
        assert b.dtype == np.int16 and len(a) == len(b)
        assert np.array_equal(b, pcm16_ref(a))
    rate(8000)
    p8 = model.infer_batch_pcm16(toks, styles, speeds)
    u8, dur = model.infer_batch_g711(toks, styles, speeds, law="ulaw", return_durations=True)
    a8 = model.infer_batch_g711(toks, styles, speeds, law="alaw")
    for b in range(3):
        assert u8[b].dtype == np.uint8 and len(u8[b]) == len(p8[b]) == out_len(600 * int(dur[b].sum()), 8000)
        assert np.array_equal(u8[b], ulaw_ref(p8[b]))
        assert np.array_equal(a8[b], alaw_ref(p8[b]))
    # at 24 kHz the codes are those of today's pcm16 output (pass-through mode)
    rate(24000)
    p24 = model.infer_batch_pcm16(toks, styles, speeds)
    u24 = model.infer_batch_g711(toks, styles, speeds, law="ulaw")
    a24 = model.infer_batch_g711(toks, styles, speeds, law="alaw")
    for b in range(3):
        assert np.array_equal(u24[b], ulaw_ref(p24[b]))
        assert np.array_equal(a24[b], alaw_ref(p24[b]))
    # law outside {0, 1}
    offs = np.asarray([0, len(toks[0])], np.int32)
    tk = np.asarray(toks[0], np.int64)
    st = np.asarray(styles[0], np.float32)
    sp = np.asarray([1.0], np.float32)
    codes = C.POINTER(C.c_uint8)()
    rc = model._lib.kkx_infer_batch_g711(model._ctx, 1, tk.ctypes.data_as(C.POINTER(C.c_int64)),
                                         offs.ctypes.data_as(C.POINTER(C.c_int32)),
                                         st.ctypes.data_as(C.POINTER(C.c_float)),
                                         sp.ctypes.data_as(C.POINTER(C.c_float)), 2, C.byref(codes), None, None)
    assert rc == -1 and not codes
    with pytest.raises(KkxError):
        model.infer_batch_g711(toks, styles, speeds, law="pcmu")


def test_default_rate_is_unchanged(model, weights_path):
    from kokorox_b200.onn import B200Koko
    toks, styles, speeds = _batch(seed=90)
    fresh = B200Koko.new(weights_path)
    try:
        want = [a.copy() for a in fresh.infer_batch(toks, styles, speeds)]
        want_launches = fresh.get_stat("launches")
    finally:
        fresh.close()
    model.set_option("out_rate", 16000)
    model.infer_batch(toks, styles, speeds)
    model.set_option("out_rate", 24000)
    assert model.get_stat("out_rate") == 24000
    got = model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") == want_launches
    for a, b in zip(got, want):
        assert np.array_equal(a, b)


def test_rejected_rates_keep_the_previous_rate(model, rate):
    from kokorox_b200.onn import KkxError
    rate(16000)
    for x in (0, 7999, 44099, 48001):
        with pytest.raises(KkxError) as e:
            model.set_option("out_rate", x)
        if x == 44099:
            g = math.gcd(44099, 24000)
            assert f"{44099 // g}/{24000 // g}" in str(e.value)
        assert model.get_stat("out_rate") == 16000
