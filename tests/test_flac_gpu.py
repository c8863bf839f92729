"""GPU tests (-m gpu) of FLAC output (kkx_infer_batch_flac, kernels_flac.cu): the encoder kernels byte for byte against
the numpy reference encoder of tests/test_flac.py, the model's FLAC files against its own 16-bit PCM at several
"out_rate" values (batch invariance included), a session's other outputs after a FLAC call, and argument errors."""
import ctypes as C

import numpy as np
import pytest

from tests.conftest import synth_case
from tests.test_flac import RATES, all_cases, flac_decode_ref, flac_encode_ref, rate_case

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


def op_flac(lib, items, rate):
    lens = np.asarray([len(x) for x in items], np.int64)
    pcm = np.ascontiguousarray(np.concatenate(items).astype(np.int16))
    offs = np.zeros(len(items) + 1, np.int64)
    args = (0, pcm.ctypes.data_as(C.POINTER(C.c_int16)), len(items), lens.ctypes.data_as(C.POINTER(C.c_int64)), rate)
    n = lib.kkx_test_flac(*args, None, 0, offs.ctypes.data_as(C.POINTER(C.c_int64)))
    assert n > 0, lib.kkx_test_last_error()
    buf = np.zeros(n, np.uint8)
    n2 = lib.kkx_test_flac(*args, buf.ctypes.data_as(C.POINTER(C.c_uint8)), n, offs.ctypes.data_as(C.POINTER(C.c_int64)))
    assert n2 == n == offs[-1], lib.kkx_test_last_error()
    return [buf[offs[b]:offs[b + 1]].tobytes() for b in range(len(items))]


def test_kernel_matches_reference_encoder(lib):
    cases = all_cases()
    got = op_flac(lib, [c[1] for c in cases], 24000)
    for (name, pcm), data in zip(cases, got):
        assert data == flac_encode_ref(pcm, 24000), name


@pytest.mark.parametrize("rate", RATES)
def test_kernel_at_every_rate(lib, rate):
    items = [rate_case(rate), rate_case(rate)[:4097], rate_case(rate)[:193]]
    for pcm, data in zip(items, op_flac(lib, items, rate)):
        assert data == flac_encode_ref(pcm, rate)


def _batch(n_items=3, seed=0, lens=(140, 37, 260)):
    cases = [synth_case(int(lens[i % len(lens)]), 9000 + seed + i, 9100 + seed + i) for i in range(n_items)]
    speeds = [1.0, 1.25, 0.85, 1.1, 0.95, 1.2][:n_items]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


def _raw_flac(model, toks, styles, speeds, null_bytes=False, null_offsets=False):
    B = len(toks)
    lens = [len(t) for t in toks]
    offs = np.zeros(B + 1, np.int32)
    offs[1:] = np.cumsum(lens)
    flat = np.concatenate(toks).astype(np.int64)
    st = np.ascontiguousarray(np.asarray(styles, np.float32).reshape(B, 256))
    sp = np.asarray(speeds, np.float32)
    buf = C.POINTER(C.c_uint8)()
    boff = np.zeros(B + 1, np.int64)
    soff = np.zeros(B + 1, np.int64)
    dur = np.zeros(int(offs[-1]), np.int32)
    rc = model._lib.kkx_infer_batch_flac(
        model._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)), offs.ctypes.data_as(C.POINTER(C.c_int32)),
        st.ctypes.data_as(C.POINTER(C.c_float)), sp.ctypes.data_as(C.POINTER(C.c_float)),
        None if null_bytes else C.byref(buf), None if null_offsets else boff.ctypes.data_as(C.POINTER(C.c_int64)),
        soff.ctypes.data_as(C.POINTER(C.c_int64)), dur.ctypes.data_as(C.POINTER(C.c_int32)))
    if rc == 0:
        model._lib.kkx_release_flac(model._ctx, buf)
    return rc, soff, [dur[offs[b]:offs[b + 1]] for b in range(B)], bool(buf)


@pytest.mark.parametrize("r", (24000, 8000, 11025))
def test_model_flac_decodes_to_its_pcm16(model, r):
    toks, styles, speeds = _batch(4, seed=20, lens=(140, 37, 260, 61))
    model.set_option("out_rate", r)
    try:
        pcm = [p.copy() for p in model.infer_batch_pcm16(toks, styles, speeds)]
        files, dur = model.infer_batch_flac(toks, styles, speeds, return_durations=True)
        alone = model.infer_batch_flac(toks[1:2], styles[1:2], speeds[1:2])
        rc, soff, dur_raw, _ = _raw_flac(model, toks, styles, speeds)
        _, dur_pcm = model.infer_batch_g711(toks, styles, speeds, return_durations=True)
    finally:
        model.set_option("out_rate", 24000)
    assert rc == 0
    for b in range(4):
        assert isinstance(files[b], bytes)
        dec, info = flac_decode_ref(files[b])
        assert info["rate"] == r and np.array_equal(dec, pcm[b]), f"item {b} at {r} Hz"
        assert files[b] == flac_encode_ref(pcm[b], r)
        assert soff[b + 1] - soff[b] == len(pcm[b])
        assert np.array_equal(dur[b], dur_pcm[b]) and np.array_equal(dur_raw[b], dur_pcm[b])
    assert alone[0] == files[1], "an item encoded alone differs from the same item in the batch"


def test_other_outputs_unchanged_after_flac(model, weights_path):
    from kokorox_b200.onn import B200Koko
    toks, styles, speeds = _batch(seed=40)
    fresh = B200Koko.new(weights_path)
    try:
        want = [a.copy() for a in fresh.infer_batch(toks, styles, speeds)]
        want_launches = fresh.get_stat("launches")
        want_pcm = [a.copy() for a in fresh.infer_batch_pcm16(toks, styles, speeds)]
        want_pcm_launches = fresh.get_stat("launches")
    finally:
        fresh.close()
    model.infer_batch_flac(toks, styles, speeds)
    flac_launches = model.get_stat("launches")
    got = model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") == want_launches
    for a, b in zip(got, want):
        assert np.array_equal(a, b)
    got_pcm = model.infer_batch_pcm16(toks, styles, speeds)
    assert model.get_stat("launches") == want_pcm_launches
    for a, b in zip(got_pcm, want_pcm):
        assert np.array_equal(a, b)
    assert flac_launches == want_pcm_launches + 3   # the encoder's three kernels


def test_profile_names_the_encoder_kernels(model):
    import json
    toks, styles, speeds = _batch(seed=60)
    model._lib.kkx_profile_enable(model._ctx, 1)
    try:
        model.infer_batch_flac(toks, styles, speeds)
        n = model._lib.kkx_profile_json(model._ctx, None, 0)
        buf = C.create_string_buffer(int(n) + 1)
        model._lib.kkx_profile_json(model._ctx, buf, n + 1)
    finally:
        model._lib.kkx_profile_enable(model._ctx, 0)
    kernels = json.loads(buf.value.decode())["kernels"]
    for name in ("flac_analyze", "flac_scan", "flac_pack"):
        assert kernels[name][0] == 1 and kernels[name][1] > 0, name


def test_null_outputs_are_argument_errors(model):
    toks, styles, speeds = _batch(1, seed=80)
    for nb, no in ((True, False), (False, True)):
        rc, _, _, got = _raw_flac(model, toks, styles, speeds, null_bytes=nb, null_offsets=no)
        assert rc == -1 and not got
        msg = model._lib.kkx_last_error(model._ctx).decode()
        assert "is null" in msg
    files = model.infer_batch_flac(toks, styles, speeds)
    pcm = model.infer_batch_pcm16(toks, styles, speeds)
    assert np.array_equal(flac_decode_ref(files[0])[0], pcm[0])
