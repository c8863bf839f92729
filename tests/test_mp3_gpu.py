"""GPU tests (-m gpu) of MP3 output (kkx_infer_batch_mp3, kkx_infer_programs_mp3, kernels_mp3.cu): the encoder kernel
against the float64 reference encoder of tests/test_mp3.py at every rate, a 2^25-sample item, the model's files
against its own 16-bit PCM, programs (purity, identity, determinism), launch counts, the absence of sticky state and
argument errors."""
import ctypes as C

import numpy as np
import pytest

from tests.conftest import synth_case
from tests.test_mp3 import (DELAY, KBPS_LSF, KBPS_MPEG1, MPEG1_RATES, RATES, Mp3Error, decode_ref, encode_ref,
                            frame_starts, n_frames, parse_header, snr_db, speechlike, square, stream_format)

pytestmark = pytest.mark.gpu


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
    def set_opts(**kw):
        for k, v in kw.items():
            model.set_option(k, v)
    yield set_opts
    for k, v in (("loudness_target", 0), ("true_peak_max", -100), ("out_rate", 24000), ("max_frames", 49152),
                 ("limiter", 0)):
        model.set_option(k, v)


def op_mp3(lib, items, rate, kbps=0):
    lens = np.asarray([len(x) for x in items], np.int64)
    pcm = np.ascontiguousarray(np.concatenate(items).astype(np.int16))
    offs = np.zeros(len(items) + 1, np.int64)
    args = (0, pcm.ctypes.data_as(C.POINTER(C.c_int16)), len(items), lens.ctypes.data_as(C.POINTER(C.c_int64)), rate,
            kbps)
    n = lib.kkx_test_mp3(*args, None, 0, offs.ctypes.data_as(C.POINTER(C.c_int64)))
    assert n > 0, lib.kkx_test_last_error()
    buf = np.zeros(n, np.uint8)
    n2 = lib.kkx_test_mp3(*args, buf.ctypes.data_as(C.POINTER(C.c_uint8)), n, offs.ctypes.data_as(C.POINTER(C.c_int64)))
    assert n2 == n == offs[-1], lib.kkx_test_last_error()
    return [buf[offs[b]:offs[b + 1]].tobytes() for b in range(len(items))]


def _decoded_snr(data, pcm):
    dec, info = decode_ref(data)
    x = np.asarray(pcm, np.float64) / 32768.0
    return snr_db(x, dec[DELAY:DELAY + len(x)]), info


# ------------------------------------------------------------------------------------------------ kernel vs reference
@pytest.mark.parametrize("rate", RATES)
def test_kernel_matches_the_reference_encoder(lib, rate):
    table = KBPS_MPEG1 if rate in MPEG1_RATES else KBPS_LSF
    items = [speechlike(rate // 3, rate, seed=21), square(577, rate), np.zeros(1, np.int16),
             np.random.default_rng(2).integers(-20000, 20000, 3000).astype(np.int16)]
    gg_total = gg_equal = 0
    for kbps in (table[0], 0, table[-1]):
        got = op_mp3(lib, items, rate, kbps)
        fm = stream_format(rate, kbps)
        for pcm, data in zip(items, got):
            info = []
            want = encode_ref(pcm, rate, kbps, info=info)
            assert len(data) == len(want)
            F = n_frames(fm, len(pcm))
            starts = frame_starts(fm, F)
            s_got, dec = _decoded_snr(data, pcm)          # also rejects anything outside the subset
            s_want, _ = _decoded_snr(want, pcm)
            assert len(dec["frames"]) == F
            for f, fr in enumerate(dec["frames"]):
                assert fr["offset"] == starts[f]
                assert data[starts[f]:starts[f] + 4] == want[starts[f]:starts[f] + 4]
                for j, g in enumerate(fr["granules"]):
                    d = g["gg"] - info[f * fm["ngr"] + j]["gg"]
                    assert abs(d) <= 1, (rate, kbps, f, j)
                    gg_total += 1
                    gg_equal += d == 0
            if np.any(pcm):
                assert abs(s_got - s_want) < 0.1, (rate, kbps, s_got, s_want)
    assert gg_equal >= 0.99 * gg_total, (gg_equal, gg_total)


def test_long_item_frames_stand_alone(lib):
    n = 1 << 25
    rate = 24000
    pcm = speechlike(n, rate, seed=31)
    data = op_mp3(lib, [pcm], rate)[0]
    fm = stream_format(rate)
    F = n_frames(fm, n)
    starts = frame_starts(fm, F)
    assert len(data) == starts[-1]
    buf = np.frombuffer(data, np.uint8)
    for f in range(F):          # every header: sync, the stream's fields, the padding of its length
        hd = parse_header(data, starts[f])
        assert hd["length"] == starts[f + 1] - starts[f] and hd["rate"] == rate and hd["kbps"] == 160
    assert buf.size == starts[-1]
    x = pcm / 32768.0
    for f in np.linspace(2, F - 1, 12).astype(int):
        # frames f - 2 .. f decoded alone: frame f's granule is exact (f - 1 feeds the MDCT overlap and the
        # synthesis history)
        dec, _ = decode_ref(data[starts[f - 2]:starts[f + 1]])
        y = dec[2 * 576:3 * 576]
        t0 = 576 * f - DELAY
        ref = x[max(t0, 0):t0 + 576]
        if np.sum(ref ** 2) > 0:
            assert snr_db(ref, y[576 - len(ref):] if t0 < 0 else y[:len(ref)]) > 40, f


# ------------------------------------------------------------------------------------------------ the model
def _batch(n_items, seed=0, lens=(140, 37, 260, 61, 190, 90)):
    cases = [synth_case(int(lens[i % len(lens)]), 9700 + seed + i, 9750 + seed + i) for i in range(n_items)]
    speeds = [(1.0, 1.25, 0.85, 1.1, 0.95, 1.2)[i % 6] for i in range(n_items)]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


@pytest.mark.parametrize("rate", RATES)
def test_model_mp3_is_the_encoding_of_its_pcm16(model, weights_path, lib, opts, rate):
    from kokorox_b200.onn import B200Koko
    toks, styles, speeds = _batch(3, seed=rate % 97)
    fresh = B200Koko.new(weights_path)
    try:
        fresh.set_option("out_rate", rate)
        pcm = [p.copy() for p in fresh.infer_batch_pcm16(toks, styles, speeds)]
    finally:
        fresh.close()
    opts(out_rate=rate)
    files, dur = model.infer_batch_mp3(toks, styles, speeds, return_durations=True)
    assert files == op_mp3(lib, pcm, rate)
    for b in range(3):
        assert isinstance(files[b], bytes)
        s, info = _decoded_snr(files[b], pcm[b])
        assert info["rate"] == rate and s > 30, (rate, b, s)
        assert len(dur[b]) == len(toks[b])


@pytest.mark.parametrize("kw", (dict(loudness_target=-1600), dict(loudness_target=-1000, limiter=1)))
def test_model_mp3_after_loudness_and_limiter(model, lib, opts, kw):
    toks, styles, speeds = _batch(3, seed=50)
    opts(**kw)
    pcm = [p.copy() for p in model.infer_batch_pcm16(toks, styles, speeds)]
    want_report = [np.asarray(a).copy() for a in model.last_loudness()]
    files = model.infer_batch_mp3(toks, styles, speeds)
    assert files == op_mp3(lib, pcm, 24000)
    for a, b in zip(model.last_loudness(), want_report):
        assert np.array_equal(a, b, equal_nan=True)
    if kw.get("limiter"):
        model.last_limiter()


def test_programs_purity_identity_determinism(model, opts):
    toks, styles, speeds = _batch(6, seed=60)
    poffs = [0, 2, 3, 6]
    want = model.infer_programs_mp3(toks, styles, speeds, poffs)
    assert model.infer_programs_mp3(toks, styles, speeds, poffs) == want            # determinism
    # other neighbours and positions
    alone = model.infer_programs_mp3(toks[3:6], styles[3:6], speeds[3:6], [0, 3])
    assert alone[0] == want[2]
    moved = model.infer_programs_mp3(toks[3:6] + toks[0:2], styles[3:6] + styles[0:2], speeds[3:6] + speeds[0:2],
                                     [0, 3, 5])
    assert moved == [want[2], want[0]]
    # frame groups: a max_frames split that cuts programs into several groups
    opts(max_frames=200)
    assert model.infer_programs_mp3(toks, styles, speeds, poffs) == want
    opts(max_frames=49152)
    # identity: a one-item program is the per-item file
    one = model.infer_programs_mp3(toks[2:3], styles[2:3], speeds[2:3], [0, 1])
    assert one == model.infer_batch_mp3(toks[2:3], styles[2:3], speeds[2:3])
    assert one[0] == want[1]
    # at 48 kHz and 192 kbps too
    opts(out_rate=48000)
    per = model.infer_batch_mp3(toks, styles, speeds, kbps=192)
    progs = model.infer_programs_mp3(toks, styles, speeds, list(range(7)), kbps=192)
    assert per == progs


def test_no_sticky_state_and_launch_count(model, weights_path):
    from kokorox_b200.onn import B200Koko
    toks, styles, speeds = _batch(3, seed=70)
    fresh = B200Koko.new(weights_path)
    try:
        want = [a.copy() for a in fresh.infer_batch(toks, styles, speeds)]
        want_launches = fresh.get_stat("launches")
        fresh.infer_batch_pcm16(toks, styles, speeds)
        pcm_launches = fresh.get_stat("launches")
    finally:
        fresh.close()
    model.infer_batch_mp3(toks, styles, speeds)
    assert model.get_stat("launches") == pcm_launches + 1        # the encoder is one launch
    got = model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") == want_launches
    for a, b in zip(got, want):
        assert np.array_equal(a, b)


def test_profile_names_the_encoder_kernel(model):
    import json
    toks, styles, speeds = _batch(2, seed=75)
    model._lib.kkx_profile_enable(model._ctx, 1)
    try:
        model.infer_batch_mp3(toks, styles, speeds)
        n = model._lib.kkx_profile_json(model._ctx, None, 0)
        buf = C.create_string_buffer(int(n) + 1)
        model._lib.kkx_profile_json(model._ctx, buf, n + 1)
    finally:
        model._lib.kkx_profile_enable(model._ctx, 0)
    k = json.loads(buf.value.decode())["kernels"]["mp3_encode"]
    assert k[0] == 1 and k[1] > 0


def _raw(model, toks, styles, speeds, kbps, poffs=None, n_programs=None, null_bytes=False, null_offsets=False):
    B = len(toks)
    offs = np.zeros(B + 1, np.int32)
    offs[1:] = np.cumsum([len(t) for t in toks])
    flat = np.concatenate(toks).astype(np.int64)
    st = np.ascontiguousarray(np.asarray(styles, np.float32).reshape(B, 256))
    sp = np.asarray(speeds, np.float32)
    buf = C.POINTER(C.c_uint8)()
    boff = np.zeros(B + 2, np.int64)
    P = C.POINTER
    common = (model._ctx, B, flat.ctypes.data_as(P(C.c_int64)), offs.ctypes.data_as(P(C.c_int32)),
              st.ctypes.data_as(P(C.c_float)), sp.ctypes.data_as(P(C.c_float)))
    outs = (None if null_bytes else C.byref(buf), None if null_offsets else boff.ctypes.data_as(P(C.c_int64)),
            None, None)
    if poffs is None:
        rc = model._lib.kkx_infer_batch_mp3(*common, kbps, *outs)
    else:
        po = np.ascontiguousarray(np.asarray(poffs, np.int32))
        rc = model._lib.kkx_infer_programs_mp3(*common, n_programs, po.ctypes.data_as(P(C.c_int32)), kbps, *outs)
    if rc == 0:
        model._lib.kkx_release_mp3(model._ctx, buf)
    else:
        assert not buf
    return rc


def test_argument_errors_leave_the_session_unchanged(model, opts):
    from kokorox_b200.onn import KkxError
    toks, styles, speeds = _batch(3, seed=80)
    opts(loudness_target=-2000)
    want = model.infer_batch_mp3(toks, styles, speeds)
    want_rep = np.asarray(model.last_loudness())
    cases = [dict(kbps=192), dict(kbps=7), dict(kbps=-1), dict(kbps=0, null_bytes=True),
             dict(kbps=0, null_offsets=True), dict(kbps=0, poffs=[0, 2, 2], n_programs=2),
             dict(kbps=0, poffs=[1, 3], n_programs=1), dict(kbps=0, poffs=[0, 3], n_programs=0),
             dict(kbps=144, poffs=[0, 1, 3], n_programs=2, null_offsets=True)]
    for case in cases:
        assert _raw(model, toks, styles, speeds, **case) == -1, case
        assert np.array_equal(np.asarray(model.last_loudness()), want_rep, equal_nan=True), case
    msg = model._lib.kkx_last_error(model._ctx).decode()
    assert "is null" in msg
    assert _raw(model, toks, styles, speeds, 192) == -1
    assert "MPEG-2" in model._lib.kkx_last_error(model._ctx).decode()
    opts(out_rate=48000)
    assert _raw(model, toks, styles, speeds, 8) == -1
    assert "MPEG-1" in model._lib.kkx_last_error(model._ctx).decode()
    opts(out_rate=24000)
    assert model.infer_batch_mp3(toks, styles, speeds) == want
    with pytest.raises(KkxError) as e:
        model.infer_programs(toks, styles, speeds, [0, 3], encoding="mp3")
    assert "infer_programs_mp3" in str(e.value)


def test_decoder_rejects_a_corrupted_kernel_file(lib):
    data = bytearray(op_mp3(lib, [speechlike(4000, 24000, seed=90)], 24000)[0])
    data[0] = 0
    with pytest.raises(Mp3Error):
        decode_ref(bytes(data))
