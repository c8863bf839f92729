"""GPU tests (-m gpu) of programs (kkx_infer_programs): one output per run of consecutive items, computed as if the
program were one utterance whose 24 kHz waveform is the concatenation of its items' waveforms.  Identity with the
per-item entry points for one-item programs, bit-exact concatenation at 24 kHz, resampling, loudness and FLAC over the
whole program against the float64 / reference-encoder references, purity (position, neighbours, frame groups), launch
counts, argument errors and the absence of sticky state; and the kernels at a program length no single item reaches."""
import ctypes as C
import math

import numpy as np
import pytest
from scipy.signal import resample_poly

from tests.conftest import synth_case
from tests.test_flac import flac_decode_ref, flac_encode_ref
from tests.test_loudness import kweight, loudness_ref, true_peak_ref
from tests.test_resample import alaw_ref, pcm16_ref, ratio, ulaw_ref

pytestmark = pytest.mark.gpu

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
    for k, v in (("loudness_target", 0), ("true_peak_max", -100), ("out_rate", 24000), ("max_frames", 49152),
                 ("max_tokens", 40960)):
        model.set_option(k, v)


def out_len(n, r):
    U, D = ratio(r)
    return -(-n * U // D)


def _batch(n_items, seed=0, lens=(140, 37, 260, 61, 190, 90)):
    cases = [synth_case(int(lens[i % len(lens)]), 9800 + seed + i, 9900 + seed + i) for i in range(n_items)]
    speeds = [(1.0, 1.25, 0.85, 1.1, 0.95, 1.2)[i % 6] for i in range(n_items)]
    return [c[0] for c in cases], [c[1] for c in cases], speeds


def per_item(model, enc, toks, styles, speeds):
    """What the existing entry point of `enc` returns, item by item (copied out of the library's buffer)."""
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


def report(model):
    return np.asarray(model.last_loudness(), np.float32)


def raw_programs(model, toks, styles, speeds, n_programs, poffs, encoding, null_bytes=False, null_offsets=False):
    """kkx_infer_programs through ctypes with every argument as given (None = a null pointer); returns the rc."""
    B = len(toks)
    offs = np.zeros(B + 1, np.int32)
    offs[1:] = np.cumsum([len(t) for t in toks])
    flat = np.concatenate(toks).astype(np.int64)
    st = np.ascontiguousarray(np.asarray(styles, np.float32).reshape(B, 256))
    sp = np.asarray(speeds, np.float32)
    po = None if poffs is None else np.ascontiguousarray(np.asarray(poffs, np.int32))
    buf = C.c_void_p()
    boff = np.zeros(max(n_programs, 0) + 2, np.int64)
    rc = model._lib.kkx_infer_programs(
        model._ctx, B, flat.ctypes.data_as(C.POINTER(C.c_int64)), offs.ctypes.data_as(C.POINTER(C.c_int32)),
        st.ctypes.data_as(C.POINTER(C.c_float)), sp.ctypes.data_as(C.POINTER(C.c_float)), n_programs,
        None if po is None else po.ctypes.data_as(C.POINTER(C.c_int32)), encoding,
        None if null_bytes else C.byref(buf), None if null_offsets else boff.ctypes.data_as(C.POINTER(C.c_int64)),
        None, None)
    if rc == 0:
        model._lib.kkx_release_programs(model._ctx, buf)
    else:
        assert not buf.value
    return rc


# ------------------------------------------------------------------------------------------------ 1. identity
@pytest.mark.parametrize("r,target", ((24000, 0), (16000, 0), (22050, -2300)))
@pytest.mark.parametrize("enc", ENCODINGS)
def test_one_item_programs_are_the_per_item_outputs(model, opts, enc, r, target):
    toks, styles, speeds = _batch(3, seed=0)
    opts(out_rate=r, loudness_target=target)
    want = per_item(model, enc, toks, styles, speeds)
    want_launches = model.get_stat("launches")
    want_rep = report(model) if target else None
    got = programs(model, enc, toks, styles, speeds, [0, 1, 2, 3])
    assert model.get_stat("launches") == want_launches
    assert len(got) == 3
    for b in range(3):
        if enc == "flac":
            assert got[b] == want[b], b
        else:
            assert got[b].dtype == want[b].dtype and got[b].tobytes() == want[b].tobytes(), b
    if target:
        assert np.array_equal(report(model), want_rep, equal_nan=True)
        assert model.get_stat("loudness_items") == 3


# ------------------------------------------------------------------------------------------------ 2. concatenation
@pytest.mark.parametrize("enc", ("f32", "pcm16"))
def test_programs_at_24k_are_the_concatenated_items(model, opts, enc):
    toks, styles, speeds = _batch(12, seed=20)
    poffs = [0, 1, 4, 12]                      # programs of 1, 3 and 8 items
    items = per_item(model, enc, toks, styles, speeds)
    got = programs(model, enc, toks, styles, speeds, poffs)
    for k in range(3):
        want = np.concatenate(items[poffs[k]:poffs[k + 1]])
        assert got[k].dtype == want.dtype and got[k].tobytes() == want.tobytes(), k


# ------------------------------------------------------------------------------------------------ 3. resampling
@pytest.mark.parametrize("r", (8000, 22050))
def test_resampled_programs_match_resample_poly(model, opts, r):
    toks, styles, speeds = _batch(7, seed=30)
    poffs = [0, 1, 4, 7]
    items24 = per_item(model, "f32", toks, styles, speeds)
    opts(out_rate=r)
    f32 = programs(model, "f32", toks, styles, speeds, poffs)
    pcm = programs(model, "pcm16", toks, styles, speeds, poffs)
    ul = programs(model, "ulaw", toks, styles, speeds, poffs)
    al = programs(model, "alaw", toks, styles, speeds, poffs)
    U, D = ratio(r)
    for k in range(3):
        x = np.concatenate(items24[poffs[k]:poffs[k + 1]]).astype(np.float64)
        assert len(f32[k]) == out_len(len(x), r), k
        ref = resample_poly(x, U, D)
        assert np.abs(f32[k] - ref).max() <= 1e-5 * np.abs(x).max(), (r, k)
        assert np.array_equal(pcm[k], pcm16_ref(f32[k]))
        assert np.array_equal(ul[k], ulaw_ref(pcm[k])) and np.array_equal(al[k], alaw_ref(pcm[k]))
    # a multi-item program is not the concatenation of its resampled items: the filter runs across the joins
    items_r = per_item(model, "f32", toks, styles, speeds)
    assert not np.array_equal(f32[1], np.concatenate(items_r[1:4]))


# ------------------------------------------------------------------------------------------------ 4. loudness
def _level_pool():
    """Items whose levels differ: the style's scale moves the random-init model's output level a long way."""
    scales = (0.0, 1.0, 3.0, 8.0, 16.0, 32.0)
    toks, styles, speeds = _batch(len(scales), seed=40, lens=(150, 120, 170, 140))
    return toks, [s * np.float32(f) for s, f in zip(styles, scales)], speeds


@pytest.mark.parametrize("r", (24000, 48000))
def test_program_loudness(model, opts, r):
    toks, styles, speeds = _level_pool()
    short_tok, short_style = synth_case(3, 9700, 9701)      # under 400 ms at speed 10
    toks.append(short_tok)
    styles.append(short_style)
    speeds.append(10.0)
    items24 = per_item(model, "f32", toks, styles, speeds)
    lv = [loudness_ref(x.astype(np.float64)) for x in items24]
    S = len(items24) - 1                                      # the short item
    assert len(items24[S]) < 9600 and math.isnan(lv[S])
    # the quietest and the loudest item with a defined level form one program, with the short item between them
    q = int(np.nanargmin(lv[:S]))
    ld = int(np.nanargmax(lv[:S]))
    assert lv[ld] - lv[q] > 10.0, lv
    rest = [b for b in range(S) if b not in (q, ld)]
    order = [q, S, ld] + rest                                 # programs: [q, short, loud], [rest...]
    toks = [toks[b] for b in order]
    styles = [styles[b] for b in order]
    speeds = [speeds[b] for b in order]
    items24 = [items24[b] for b in order]
    poffs = [0, 3, len(order)]
    opts(out_rate=r)
    off = programs(model, "f32", toks, styles, speeds, poffs)
    opts(loudness_target=-2300)
    on = programs(model, "f32", toks, styles, speeds, poffs)
    L, tp, g = model.last_loudness()
    assert len(L) == 2 and model.get_stat("loudness_items") == 2
    for k in range(2):
        x = np.concatenate(items24[poffs[k]:poffs[k + 1]]).astype(np.float64)
        assert abs(L[k] - loudness_ref(x)) <= 0.01, (k, L[k], loudness_ref(x))
        assert abs(tp[k] - 20 * math.log10(true_peak_ref(x))) <= 0.01, k
        # one gain covers the whole program
        assert np.array_equal(on[k], np.float32(off[k] * g[k])), (r, k)
    # the level is no longer equalised per item: the loud and the quiet item keep their distance (K-weighted energy,
    # ungated: after the common gain the quiet item may fall under the absolute gate)
    if r == 24000:
        n0, n2 = len(items24[0]), len(items24[0]) + len(items24[1])
        y_in, y_out = kweight(np.concatenate(items24[:3])), kweight(on[0])
        lvl = lambda y: 10 * math.log10(np.mean(y[n2:] ** 2) / np.mean(y[:n0] ** 2))  # noqa: E731
        assert abs(lvl(y_out) - lvl(y_in)) <= 0.01, (lvl(y_in), lvl(y_out))


# ------------------------------------------------------------------------------------------------ 5. FLAC
@pytest.mark.parametrize("r,target", ((24000, 0), (22050, -1600)))
def test_flac_programs(model, opts, r, target):
    toks, styles, speeds = _batch(6, seed=50)
    poffs = [0, 2, 3, 6]
    opts(out_rate=r, loudness_target=target)
    pcm = programs(model, "pcm16", toks, styles, speeds, poffs)
    files = programs(model, "flac", toks, styles, speeds, poffs)
    assert len(files) == 3
    for k in range(3):
        assert isinstance(files[k], bytes)
        dec, info = flac_decode_ref(files[k])
        assert info["rate"] == r and info["total"] == len(pcm[k])
        assert np.array_equal(dec, pcm[k]), k
        assert files[k] == flac_encode_ref(pcm[k], r), k


# ------------------------------------------------------------------------------------------------ 6. purity
def test_program_bits_do_not_depend_on_neighbours_or_groups(model, opts):
    toks, styles, speeds = _batch(9, seed=60)
    X, A, Bq = [0, 1, 2], [3, 4], [5, 6, 7, 8]
    opts(out_rate=16000, loudness_target=-1600)

    def run(groups, where):
        order = [b for gr in groups for b in gr]
        poffs = list(np.cumsum([0] + [len(gr) for gr in groups]))
        t, s, sp = [toks[b] for b in order], [styles[b] for b in order], [speeds[b] for b in order]
        k = groups.index(X)
        fl = programs(model, "flac", t, s, sp, poffs)[k]
        rep = report(model)[:, k]
        f32, dur = model.infer_programs(t, s, sp, poffs, encoding="f32", return_durations=True)
        assert np.array_equal(report(model)[:, k], rep, equal_nan=True), where
        return fl, f32[k].copy(), rep, [int(d.sum()) for d in dur], poffs[k]

    fl0, f0, rep0, _, _ = run([X], "alone")
    for groups, where in (([X, A, Bq], "first"), ([A, X, Bq], "middle"), ([A, Bq, X], "last")):
        fl, f, rep, _, _ = run(groups, where)
        assert fl == fl0 and f.tobytes() == f0.tobytes(), where
        assert np.array_equal(rep, rep0, equal_nan=True), where
    # frame groups: a budget smaller than the program puts its items into different groups
    _, _, _, T, _ = run([X], "alone")
    opts(max_frames=max(T))
    fl, f, rep, _, p0 = run([A, X, Bq], "frame groups")
    assert model.get_stat("frame_groups") > 1
    firsts = [model.get_stat(f"group_first:{g}") for g in range(model.get_stat("frame_groups"))]
    assert any(p0 < gf < p0 + len(X) for gf in firsts), firsts     # a group starts inside the program
    assert fl == fl0 and f.tobytes() == f0.tobytes() and np.array_equal(rep, rep0, equal_nan=True)


# ------------------------------------------------------------------------------------------------ 7. launches
def test_a_program_across_groups_is_post_processed_once(model, opts):
    toks, styles, speeds = _batch(6, seed=70)
    _, dur = model.infer_batch(toks, styles, speeds, return_durations=True)
    opts(max_frames=max(int(d.sum()) for d in dur))
    model.infer_programs(toks, styles, speeds, [0, 6])
    groups = model.get_stat("frame_groups")
    assert groups > 1
    off = model.get_stat("launches")
    opts(loudness_target=-2300)
    model.infer_programs(toks, styles, speeds, [0, 6])
    assert model.get_stat("frame_groups") == groups
    assert model.get_stat("launches") - off == 4          # 3 loudness kernels + the pass-through, once


# ------------------------------------------------------------------------------------------------ 8. errors
def test_argument_errors_leave_the_session_as_it_was(model, opts, weights_path):
    from kokorox_b200.onn import B200Koko, KkxError
    toks, styles, speeds = _batch(3, seed=80)
    opts(out_rate=16000, loudness_target=-2300)
    fresh = B200Koko.new(weights_path)
    try:
        fresh.set_option("out_rate", 16000)
        fresh.set_option("loudness_target", -2300)
        want = fresh.infer_batch_flac(toks, styles, speeds)
        want_rep = report(fresh)
    finally:
        fresh.close()
    model.infer_programs(toks, styles, speeds, [0, 2, 3], encoding="flac")
    prev = report(model)
    good = dict(n_programs=2, poffs=[0, 2, 3], encoding=4)
    cases = [dict(null_bytes=True), dict(null_offsets=True),
             dict(n_programs=0, poffs=[0]), dict(n_programs=4, poffs=[0, 1, 2, 3, 3]),
             dict(poffs=None), dict(poffs=[1, 2, 3]), dict(poffs=[0, 2, 2]), dict(poffs=[0, 1, 4]),
             dict(n_programs=3, poffs=[0, 2, 2, 3]), dict(n_programs=2, poffs=[0, 3, 2]),
             dict(encoding=-1), dict(encoding=5)]
    for case in cases:
        a = dict(good, **case)
        rc = raw_programs(model, toks, styles, speeds, a["n_programs"], a["poffs"], a["encoding"],
                          a.get("null_bytes", False), a.get("null_offsets", False))
        assert rc == -1, case
        assert np.array_equal(report(model), prev, equal_nan=True), case
        assert model.infer_batch_flac(toks, styles, speeds) == want, case
        prev = report(model)
        assert np.array_equal(prev, want_rep, equal_nan=True), case
    with pytest.raises(KkxError):
        model.infer_programs(toks, styles, speeds, [0, 3], encoding="mp3")


# ------------------------------------------------------------------------------------------------ 9. no sticky state
def test_no_state_carries_over_from_a_program_call(model, opts, weights_path):
    from kokorox_b200.onn import B200Koko
    toks, styles, speeds = _batch(5, seed=90)
    fresh = B200Koko.new(weights_path)
    try:
        for key, v in (("out_rate", 22050), ("loudness_target", -1600)):
            fresh.set_option(key, v)
        want = [a.copy() for a in fresh.infer_batch(toks, styles, speeds)]
        want_launches = fresh.get_stat("launches")
        want_rep = report(fresh)
    finally:
        fresh.close()
    opts(out_rate=22050, loudness_target=-1600)
    model.infer_programs(toks, styles, speeds, [0, 2, 5], encoding="flac")
    assert model.get_stat("loudness_items") == 2
    got = model.infer_batch(toks, styles, speeds)
    assert model.get_stat("launches") == want_launches
    assert model.get_stat("loudness_items") == 5
    assert np.array_equal(report(model), want_rep, equal_nan=True)
    for a, b in zip(got, want):
        assert a.tobytes() == b.tobytes()


# ------------------------------------------------------------------------------------------------ kernels at program length
# One item has at most 65536 frames (39 321 600 samples at 24 kHz); a program of several is longer.  The kernels take
# 64-bit offsets and lengths, so a program longer than any item is measured and resampled like a short one.
LONG = 65536 * 600 + 2400 * 7 + 1


def _speechlike(n, seed, level=0.1):
    rng = np.random.default_rng(seed)
    t = np.arange(n) / 24000.0
    env = np.maximum(np.sin(2 * np.pi * 3.1 * t + seed), 0.0) ** 2 + 0.02
    return (level * env * rng.standard_normal(n)).astype(np.float32)


def test_loudness_kernels_at_program_length(lib):
    items = [_speechlike(24000, 1), _speechlike(LONG, 2), _speechlike(9601, 3)]
    lens = np.asarray([len(x) for x in items], np.int64)
    x = np.ascontiguousarray(np.concatenate(items))
    L, tp, g = (np.zeros(3, np.float32) for _ in range(3))
    fp = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    rc = lib.kkx_test_loudness(0, fp(x), 3, lens.ctypes.data_as(C.POINTER(C.c_int64)), -2300, -100, fp(L), fp(tp),
                               fp(g))
    assert rc == 0, lib.kkx_test_last_error()
    for b, it in enumerate(items):
        xd = it.astype(np.float64)
        assert abs(L[b] - loudness_ref(xd)) <= 0.01, (b, L[b])
        assert abs(tp[b] - 20 * math.log10(true_peak_ref(xd))) <= 0.01, b


def test_resample_kernel_at_program_length(lib):
    rng = np.random.default_rng(5)
    items = [(rng.standard_normal(n) * 0.3).astype(np.float32) for n in (600, LONG, 1237)]
    r = 8000
    U, D = ratio(r)
    lens = np.asarray([len(x) for x in items], np.int64)
    n_out = [out_len(int(n), r) for n in lens]
    x = np.ascontiguousarray(np.concatenate(items))
    out = np.zeros(sum(n_out), np.float32)
    rc = lib.kkx_test_resample(0, x.ctypes.data_as(C.POINTER(C.c_float)), 3, lens.ctypes.data_as(C.POINTER(C.c_int64)),
                               r, -1, out.ctypes.data_as(C.POINTER(C.c_float)), None, None)
    assert rc == 0, lib.kkx_test_last_error()
    offs = np.concatenate([[0], np.cumsum(n_out)])
    for b, it in enumerate(items):
        ref = resample_poly(it.astype(np.float64), U, D)
        y = out[offs[b]:offs[b + 1]]
        assert len(y) == len(ref)
        assert np.abs(y - ref).max() <= 1e-5 * np.abs(it).max(), b
