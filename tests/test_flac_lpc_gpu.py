"""GPU tests (-m gpu) of FLAC linear prediction ("flac_lpc_order", kernels_flac.cu): the encoder kernels byte for byte
against the numpy reference of tests/test_flac_lpc.py at every rate and order, the model's FLAC files and FLAC
programs with the option on against their own 16-bit PCM, the option's off state and its argument errors."""
import ctypes as C
import json

import numpy as np
import pytest

from tests.conftest import synth_case
from tests.test_flac import RATES, all_cases, flac_decode_ref
from tests.test_flac_lpc import ORDERS, flac_lpc_decode_ref, flac_lpc_encode_ref

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
    """Sets session options for one test and restores the defaults afterwards."""
    def set_opts(**kw):
        for k, v in kw.items():
            model.set_option(k, v)
    yield set_opts
    for k, v in (("flac_lpc_order", 0), ("loudness_target", 0), ("limiter", 0), ("out_rate", 24000)):
        model.set_option(k, v)


def op_flac_lpc(lib, items, rate, order):
    lens = np.asarray([len(x) for x in items], np.int64)
    pcm = np.ascontiguousarray(np.concatenate(items).astype(np.int16))
    offs = np.zeros(len(items) + 1, np.int64)
    args = (0, pcm.ctypes.data_as(C.POINTER(C.c_int16)), len(items), lens.ctypes.data_as(C.POINTER(C.c_int64)), rate,
            order)
    n = lib.kkx_test_flac_lpc(*args, None, 0, offs.ctypes.data_as(C.POINTER(C.c_int64)))
    assert n > 0, lib.kkx_test_last_error()
    buf = np.zeros(n, np.uint8)
    n2 = lib.kkx_test_flac_lpc(*args, buf.ctypes.data_as(C.POINTER(C.c_uint8)), n,
                               offs.ctypes.data_as(C.POINTER(C.c_int64)))
    assert n2 == n == offs[-1], lib.kkx_test_last_error()
    return [buf[offs[b]:offs[b + 1]].tobytes() for b in range(len(items))]


@pytest.mark.parametrize("rate", RATES)
@pytest.mark.parametrize("p", ORDERS)
def test_kernel_matches_reference_encoder(lib, p, rate):
    cases = all_cases()
    got = op_flac_lpc(lib, [c[1] for c in cases], rate, p)
    for (name, pcm), data in zip(cases, got):
        assert data == flac_lpc_encode_ref(pcm, rate, p), f"{name} at p = {p}, {rate} Hz"


def _batch(n_items=3, seed=0, lens=(140, 37, 260, 61)):
    cases = [synth_case(int(lens[i % len(lens)]), 9300 + seed + i, 9400 + seed + i) for i in range(n_items)]
    speeds = [(1.0, 1.25, 0.85, 1.1)[i % 4] for i in range(n_items)]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


@pytest.mark.parametrize("r", (24000, 8000, 11025))
def test_model_flac_decodes_to_its_pcm16(model, opts, r):
    toks, styles, speeds = _batch(4, seed=20)
    opts(out_rate=r, flac_lpc_order=8)
    assert model.get_stat("flac_lpc_order") == 8
    pcm = [p.copy() for p in model.infer_batch_pcm16(toks, styles, speeds)]
    files = model.infer_batch_flac(toks, styles, speeds)
    alone = model.infer_batch_flac(toks[1:2], styles[1:2], speeds[1:2])
    for b in range(4):
        dec, info = flac_lpc_decode_ref(files[b])
        assert info["rate"] == r and np.array_equal(dec, pcm[b]), f"item {b} at {r} Hz"
        assert files[b] == flac_lpc_encode_ref(pcm[b], r, 8)
    assert alone[0] == files[1], "an item encoded alone differs from the same item in the batch"


def test_programs(model, opts):
    toks, styles, speeds = _batch(4, seed=30)
    opts(flac_lpc_order=12)
    per_item = model.infer_batch_flac(toks, styles, speeds)
    one = model.infer_programs(toks, styles, speeds, [0, 1, 2, 3, 4], encoding="flac")
    assert one == per_item, "a one-item program differs from the item's own file"
    pcm = [a.copy() for a in model.infer_programs(toks, styles, speeds, [0, 3, 4], encoding="pcm16")]
    files = model.infer_programs(toks, styles, speeds, [0, 3, 4], encoding="flac")
    for k in range(2):
        assert np.array_equal(flac_lpc_decode_ref(files[k])[0], pcm[k]), k
        assert files[k] == flac_lpc_encode_ref(pcm[k], 24000, 12), k
    items = [a.copy() for a in model.infer_batch_pcm16(toks, styles, speeds)]
    assert np.array_equal(pcm[0], np.concatenate(items[:3]))


def test_programs_with_loudness_and_limiter(model, opts):
    toks, styles, speeds = _batch(4, seed=40)
    opts(flac_lpc_order=8, loudness_target=-1600, limiter=1)
    poffs = [0, 2, 4]
    pcm = [a.copy() for a in model.infer_programs(toks, styles, speeds, poffs, encoding="pcm16")]
    files = model.infer_programs(toks, styles, speeds, poffs, encoding="flac")
    for k in range(2):
        assert np.array_equal(flac_lpc_decode_ref(files[k])[0], pcm[k]), k
        assert files[k] == flac_lpc_encode_ref(pcm[k], 24000, 8), k


def _profile_kernels(model, fn):
    model._lib.kkx_profile_enable(model._ctx, 1)
    try:
        fn()
        n = model._lib.kkx_profile_json(model._ctx, None, 0)
        buf = C.create_string_buffer(int(n) + 1)
        model._lib.kkx_profile_json(model._ctx, buf, n + 1)
    finally:
        model._lib.kkx_profile_enable(model._ctx, 0)
    return json.loads(buf.value.decode())["kernels"]


def test_off_again_is_a_fresh_session(model, opts, weights_path):
    from kokorox_b200.onn import B200Koko
    toks, styles, speeds = _batch(3, seed=50)
    fresh = B200Koko.new(weights_path)
    try:
        assert fresh.get_stat("flac_lpc_order") == 0
        fresh.infer_batch_pcm16(toks, styles, speeds)
        pcm_launches = fresh.get_stat("launches")
        want = fresh.infer_batch_flac(toks, styles, speeds)
        want_launches = fresh.get_stat("launches")
    finally:
        fresh.close()
    assert want_launches == pcm_launches + 3
    opts(flac_lpc_order=8)
    on = model.infer_batch_flac(toks, styles, speeds)
    # the LPC variant of flac_analyze: the same three launches
    assert model.get_stat("launches") == pcm_launches + 3
    kernels = _profile_kernels(model, lambda: model.infer_batch_flac(toks, styles, speeds))
    for name in ("flac_analyze", "flac_scan", "flac_pack"):
        assert kernels[name][0] == 1 and kernels[name][1] > 0, name
    assert len(b"".join(on)) <= len(b"".join(want))
    model.set_option("flac_lpc_order", 0)
    assert model.infer_batch_flac(toks, styles, speeds) == want
    assert model.get_stat("launches") == want_launches
    for b in range(3):
        assert np.array_equal(flac_decode_ref(want[b])[0], flac_lpc_decode_ref(on[b])[0])


def test_bad_values_are_argument_errors(model, opts):
    from kokorox_b200.onn import KkxError
    opts(flac_lpc_order=4)
    for v in (-1, 13, 1000):
        with pytest.raises(KkxError) as e:
            model.set_option("flac_lpc_order", v)
        assert e.value.code == -1
        assert "1..12" in model._lib.kkx_last_error(model._ctx).decode()
        assert model.get_stat("flac_lpc_order") == 4
