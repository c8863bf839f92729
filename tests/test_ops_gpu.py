"""GPU tests (-m gpu): each hand-written kernel in isolation against the matching torch op,
through the op-level hooks of include/kkx_test.h."""
import ctypes as C
import ctypes as C_

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def lib():
    from kokorox_b200.onn import load_library
    lib = load_library()
    lib.kkx_test_last_error.restype = C.c_char_p
    return lib


def fp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_float))


def run_conv(lib, x, w_kic, bias, ks, dil, pad, stride, m_len, out_rows, ors=1, oro=0, pscale=None, pshift=None,
             pact=0, pslope=0.0, palpha=None, res=None, res_shift=0, oscale=1.0, eact=0, accumulate=0, out_init=None):
    rows_in, Ci = x.shape
    Co = w_kic.shape[2]
    out = np.zeros((out_rows, Co), np.float32) if out_init is None else out_init.copy()
    rc = lib.kkx_test_conv(0, fp(x), rows_in, Ci, Ci, fp(w_kic), fp(bias), Co, ks, dil, pad, stride, fp(pscale),
                           fp(pshift), pact, C.c_float(pslope), fp(palpha), m_len, ors, oro, out_rows, fp(res),
                           0 if res is None else res.shape[0], res_shift, C.c_float(oscale), eact, accumulate, fp(out))
    assert rc == 0, lib.kkx_test_last_error()
    return out


def rnd(*shape, seed=0, scale=1.0):
    return (np.random.default_rng(seed).standard_normal(shape) * scale).astype(np.float32)


@pytest.mark.parametrize("L,Ci,Co,k,dil", [(300, 128, 128, 3, 1), (777, 256, 256, 7, 3), (513, 128, 128, 11, 5),
                                           (130, 514, 1024, 3, 1), (1000, 128, 22, 7, 1), (40, 768, 2304, 1, 1)])
def test_conv1d_matches_torch(lib, L, Ci, Co, k, dil):
    x, w, b = rnd(L, Ci, seed=1), rnd(Co, Ci, k, seed=2, scale=1 / np.sqrt(Ci * k)), rnd(Co, seed=3)
    pad = dil * (k - 1) // 2
    ref = F.conv1d(torch.from_numpy(x.T)[None], torch.from_numpy(w), torch.from_numpy(b), padding=pad, dilation=dil)[0].T.numpy()
    got = run_conv(lib, x, np.ascontiguousarray(w.transpose(2, 1, 0)), b, k, dil, pad, 1, L, L)
    np.testing.assert_allclose(got, ref, atol=2e-4, rtol=1e-4)


def test_conv_strided_noise_conv(lib):
    # noise_convs[0]: Conv1d(22,256,k12,s6,p3) on 120T+1 rows -> 20T rows
    T = 7
    x, w, b = rnd(120 * T + 1, 22, seed=4), rnd(256, 22, 12, seed=5, scale=0.1), rnd(256, seed=6)
    ref = F.conv1d(torch.from_numpy(x.T)[None], torch.from_numpy(w), torch.from_numpy(b), stride=6, padding=3)[0].T.numpy()
    assert ref.shape[0] == 20 * T
    got = run_conv(lib, x, np.ascontiguousarray(w.transpose(2, 1, 0)), b, 12, 1, 3, 6, 20 * T, 20 * T)
    np.testing.assert_allclose(got, ref, atol=2e-4, rtol=1e-4)


@pytest.mark.parametrize("Ci,Co,k,s", [(512, 256, 20, 10), (256, 128, 12, 6)])
def test_conv_transpose_as_phase_convs(lib, Ci, Co, k, s):
    # generator ups: ConvTranspose1d(k=2s, stride s, padding s/2) as s two-tap phase convs, with the
    # LeakyReLU(0.1) prologue the generator applies first
    L, p = 37, (k - s) // 2
    x, w, b = rnd(L, Ci, seed=7), rnd(Ci, Co, k, seed=8, scale=0.05), rnd(Co, seed=9)
    xin = F.leaky_relu(torch.from_numpy(x.T)[None], 0.1)
    ref = F.conv_transpose1d(xin, torch.from_numpy(w), torch.from_numpy(b), stride=s, padding=p)[0].T.numpy()
    out = np.full((L * s, Co), np.nan, np.float32)
    for r in range(s):
        q0 = 1 if r < p else 0
        ph = np.stack([w[:, :, r], w[:, :, r + s]])  # [2][Ci][Co]
        out = run_conv(lib, x, np.ascontiguousarray(ph), b, 2, -1, -q0, 1, L, L * s, ors=s, oro=q0 * s + r - p,
                       pact=1, pslope=0.1, out_init=out)
    assert not np.isnan(out).any()
    np.testing.assert_allclose(out, ref, atol=2e-4, rtol=1e-4)


def test_conv_prologue_epilogue_fusions(lib):
    # AdaIN scale/shift + Snake on the operand, bias + residual(row>>1) + scale + accumulate on the result
    L, Cc, k = 200, 128, 3
    x, w, b = rnd(L, Cc, seed=10), rnd(Cc, Cc, k, seed=11, scale=0.05), rnd(Cc, seed=12)
    sc, sh = (1 + 0.3 * rnd(Cc, seed=13)), 0.2 * rnd(Cc, seed=14)
    alpha = np.clip(1 + 0.3 * rnd(Cc, seed=15), 0.3, 2).astype(np.float32)
    res = rnd(L // 2, Cc, seed=16)
    init = rnd(L, Cc, seed=17)
    xt = torch.from_numpy(x) * torch.from_numpy(sc) + torch.from_numpy(sh)
    a = torch.from_numpy(alpha)
    xt = xt + (1 / a) * torch.sin(a * xt) ** 2
    y = F.conv1d(xt.T[None], torch.from_numpy(w), torch.from_numpy(b), padding=1)[0].T
    ref = (torch.from_numpy(init) + 0.5 * (y + torch.from_numpy(res).repeat_interleave(2, 0))).numpy()
    got = run_conv(lib, x, np.ascontiguousarray(w.transpose(2, 1, 0)), b, k, 1, 1, 1, L, L, pscale=sc.astype(np.float32),
                   pshift=sh.astype(np.float32), pact=2, palpha=alpha, res=res, res_shift=1, oscale=0.5, accumulate=1,
                   out_init=init)
    np.testing.assert_allclose(got, ref, atol=3e-4, rtol=1e-4)


def test_gemm_gelu_new_epilogue(lib):
    x, w, b = rnd(100, 768, seed=18), rnd(2048, 768, seed=19, scale=0.03), rnd(2048, seed=20)
    f = torch.from_numpy(x) @ torch.from_numpy(w).T + torch.from_numpy(b)
    ref = (0.5 * f * (1 + torch.tanh(np.sqrt(2 / np.pi) * (f + 0.044715 * f ** 3)))).numpy()
    got = run_conv(lib, x, np.ascontiguousarray(w.T[None]), b, 1, 1, 0, 1, 100, 100, eact=3)
    np.testing.assert_allclose(got, ref, atol=2e-4, rtol=1e-4)


@pytest.mark.parametrize("N", [1, 5, 64, 200])
def test_lstm_matches_torch(lib, N):
    torch.manual_seed(N)
    m = torch.nn.LSTM(640, 256, 1, batch_first=True, bidirectional=True).eval()
    x = torch.randn(1, N, 640)
    with torch.no_grad():
        ref = m(x)[0][0].numpy()
        xp = []
        whh = np.zeros((2, 256, 1024), np.float32)
        for d, sfx in enumerate(("", "_reverse")):
            wih, b = getattr(m, "weight_ih_l0" + sfx), getattr(m, "bias_ih_l0" + sfx) + getattr(m, "bias_hh_l0" + sfx)
            xp.append((x[0] @ wih.T + b).numpy())
            whh[d] = getattr(m, "weight_hh_l0" + sfx).numpy().T
    xproj = np.ascontiguousarray(np.concatenate(xp, axis=1), dtype=np.float32)
    out = np.zeros((N, 512), np.float32)
    rc = lib.kkx_test_lstm(0, fp(xproj), fp(whh), N, fp(out))
    assert rc == 0, lib.kkx_test_last_error()
    np.testing.assert_allclose(out, ref, atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("B", [2, 9, 20, 40, 56, 64, 77, 100])
def test_lstm_ragged_batch_groups(lib, B):
    # the persistent cluster kernel processes G = 1/2/4/8/10/12 items per cluster (G chosen so that the clusters
    # of one launch are co-resident: 15 clusters of 8 CTAs fit a B200); ragged lengths
    torch.manual_seed(B)
    m = torch.nn.LSTM(512, 256, 1, batch_first=True, bidirectional=True).eval()
    rng = np.random.default_rng(B)
    lens = rng.integers(1, 90, B).astype(np.int32)
    offs = np.zeros(B, np.int32)
    o = 3
    for b in range(B):
        offs[b] = o
        o += int(lens[b]) + 5
    rows = o
    xproj = np.zeros((rows, 2048), np.float32)
    ref = np.zeros((rows, 512), np.float32)
    whh = np.zeros((2, 256, 1024), np.float32)
    with torch.no_grad():
        for d, sfx in enumerate(("", "_reverse")):
            whh[d] = getattr(m, "weight_hh_l0" + sfx).numpy().T
        for b in range(B):
            x = torch.randn(1, int(lens[b]), 512)
            ref[offs[b]:offs[b] + lens[b]] = m(x)[0][0].numpy()
            for d, sfx in enumerate(("", "_reverse")):
                wih, bb = getattr(m, "weight_ih_l0" + sfx), getattr(m, "bias_ih_l0" + sfx) + getattr(m, "bias_hh_l0" + sfx)
                xproj[offs[b]:offs[b] + lens[b], d * 1024:(d + 1) * 1024] = (x[0] @ wih.T + bb).numpy()
    out = np.zeros((rows, 512), np.float32)
    rc = lib.kkx_test_lstm_batch(0, fp(xproj), fp(whh), B, offs.ctypes.data_as(C.POINTER(C.c_int)),
                                 lens.ctypes.data_as(C.POINTER(C.c_int)), rows, fp(out))
    assert rc == 0, lib.kkx_test_last_error()
    np.testing.assert_allclose(out, ref, atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("B,lo,hi", [(2, 1, 90), (9, 200, 300), (40, 60, 90), (64, 500, 512), (100, 1, 40)])
def test_lstm_kernel_variants_agree(lib, B, lo, hi):
    """The cluster kernel with SFU gate functions (tensor-core configuration) against the one with libm gate functions
    (fp32 configuration; same dot products) and the plain one-CTA-per-item kernel (other summation order), over
    sequences long enough for a recurrent error to build up."""
    rng = np.random.default_rng(100 + B)
    lens = rng.integers(lo, hi, B).astype(np.int32)
    offs = np.zeros(B, np.int32)
    o = 2
    for b in range(B):
        offs[b] = o
        o += int(lens[b]) + 3
    rows = o
    xproj = (rng.standard_normal((rows, 2048)) * 1.5).astype(np.float32)
    whh = (rng.standard_normal((2, 256, 1024)) * 0.06).astype(np.float32)
    outs = []
    for variant in (1, 0, -1):
        out = np.zeros((rows, 512), np.float32)
        ms = C.c_float(0)
        rc = lib.kkx_test_lstm_batch_v(0, fp(xproj), fp(whh), B, offs.ctypes.data_as(C.POINTER(C.c_int)),
                                       lens.ctypes.data_as(C.POINTER(C.c_int)), rows, variant, 0, fp(out), C.byref(ms))
        assert rc == 0, lib.kkx_test_last_error()
        outs.append(out)
    assert np.abs(outs[0]).max() > 0.05
    np.testing.assert_allclose(outs[1], outs[2], atol=2e-5, rtol=1e-4)
    np.testing.assert_allclose(outs[0], outs[1], atol=2e-5, rtol=1e-4)
    rel = np.sqrt(((outs[0] - outs[1]) ** 2).sum() / (outs[1] ** 2).sum())
    assert rel < 2e-6, rel


@pytest.mark.parametrize("lens", [[1], [127], [128], [129], [1000, 5, 260, 384]])
def test_pointwise_conv_with_statistics(lib, lens):
    """noise_convs[1] (22 -> 128, k = 1) as one fp32 pass that also emits the per-128-row column sums: the output
    against numpy fp64, the statistics against the colstats pass over that output, gap rows untouched."""
    rng = np.random.default_rng(len(lens) * 1000 + lens[0])
    B = len(lens)
    lens_a = np.asarray(lens, np.int32)
    offs = np.zeros(B, np.int32)
    o = 32
    for b in range(B):
        offs[b] = o
        o += int(lens_a[b]) + 32
    rows = o
    x = rng.standard_normal((rows, 24)).astype(np.float32) * 3
    x[:, 22:] = np.nan                                   # pad columns must never be read into the result
    w = (rng.standard_normal((22, 128)) * 0.3).astype(np.float32)
    bias = rng.standard_normal(128).astype(np.float32)
    max_len = int(lens_a.max())
    nchunk = (max_len + 127) // 128
    out = np.full((rows, 128), 7.5, np.float32)
    part = np.zeros((B, nchunk, 2, 128), np.float32)
    part_ref = np.zeros_like(part)
    rc = lib.kkx_test_pointwise_conv_stats(0, fp(x), fp(w), fp(bias), B, offs.ctypes.data_as(C.POINTER(C.c_int)),
                                           lens_a.ctypes.data_as(C.POINTER(C.c_int)), rows, max_len, fp(out), fp(part),
                                           fp(part_ref))
    assert rc == 0, lib.kkx_test_last_error()
    ref = x[:, :22].astype(np.float64) @ w.astype(np.float64) + bias
    touched = np.zeros(rows, bool)
    for b in range(B):
        sl = slice(offs[b], offs[b] + lens_a[b])
        touched[sl] = True
        np.testing.assert_allclose(out[sl], ref[sl], atol=2e-5, rtol=2e-6)
        for ch in range((lens_a[b] + 127) // 128):
            blk = out[offs[b] + ch * 128: offs[b] + min(lens_a[b], ch * 128 + 128)].astype(np.float64)
            np.testing.assert_allclose(part[b, ch, 0], blk.sum(0), atol=2e-3, rtol=1e-5)
            np.testing.assert_allclose(part[b, ch, 1], (blk ** 2).sum(0), atol=2e-3, rtol=1e-5)
            np.testing.assert_allclose(part[b, ch], part_ref[b, ch], atol=2e-3, rtol=1e-5)
    assert np.all(out[~touched] == 7.5)


@pytest.mark.parametrize("C,rows,res,affine,ada,slope,planes", [
    (768, 37, True, True, False, 1.0, True),      # ALBERT: LN(x + residual), planes for the next GEMM (vector kernel)
    (768, 5, False, True, False, 1.0, False),
    (512, 64, False, False, True, 1.0, False),    # AdaLayerNorm of the duration encoder
    (512, 9, False, True, False, 0.2, False),     # channel LN + LeakyReLU of the text encoder
    (128, 20, False, True, False, 1.0, True),
    (640, 11, True, True, True, 1.0, True),       # no vector instantiation: scalar kernel
])
def test_layernorm_kernels(lib, C, rows, res, affine, ada, slope, planes):
    """layernorm_vec_kernel (row in registers, 128-bit accesses) and the scalar kernel against torch fp64; the operand
    planes must hold hi + lo = 16 * the fp32 result to fp32 accuracy (what the split-FP16 GEMM reads next)."""
    rng = np.random.default_rng(C + rows)
    x = (rng.standard_normal((rows, C)) * 2 + 0.3).astype(np.float32)
    r = rng.standard_normal((rows, C)).astype(np.float32) if res else None
    w = (1 + 0.2 * rng.standard_normal(C)).astype(np.float32) if affine else None
    b = (0.1 * rng.standard_normal(C)).astype(np.float32) if affine else None
    ad = (0.3 * rng.standard_normal(2 * C)).astype(np.float32) if ada else None
    out = np.zeros((rows, C), np.float32)
    hi = np.zeros((rows, C), np.uint16) if planes else None
    lo = np.zeros((rows, C), np.uint16) if planes else None
    u16 = lambda a: a.ctypes.data_as(C_.POINTER(C_.c_ushort)) if a is not None else None  # noqa: E731
    fpn = lambda a: fp(a) if a is not None else None  # noqa: E731
    rc = lib.kkx_test_layernorm(0, fp(x), fpn(r), fpn(w), fpn(b), fpn(ad), rows, C, C_.c_float(1e-5), C_.c_float(slope),
                                fp(out), u16(hi), u16(lo))
    assert rc == 0, lib.kkx_test_last_error()
    t = torch.from_numpy(x).double() + (torch.from_numpy(r).double() if res else 0)
    ref = torch.nn.functional.layer_norm(t, (C,), eps=1e-5)
    if affine:
        ref = ref * torch.from_numpy(w).double() + torch.from_numpy(b).double()
    if ada:
        ref = (1 + torch.from_numpy(ad[:C]).double()) * ref + torch.from_numpy(ad[C:]).double()
    if slope != 1.0:
        ref = torch.where(ref > 0, ref, ref * slope)
    np.testing.assert_allclose(out, ref.numpy(), atol=3e-6, rtol=3e-6)
    if planes:
        got = hi.view(np.float16).astype(np.float64) + lo.view(np.float16).astype(np.float64)
        np.testing.assert_allclose(got, 16.0 * out.astype(np.float64), atol=2e-6, rtol=2e-7)


@pytest.mark.parametrize("frames", [[1], [7, 40], [33, 2, 100]])
def test_im2col_fast_kernel_is_bit_identical(lib, frames):
    """noise_convs[0] operand gather (k = 12, stride 6, pad 3 over the 120T+1 STFT frames -> 20T rows of 12 x 22 columns):
    the shared-memory kernel against the element-wise one, bit for bit, and against numpy."""
    rng = np.random.default_rng(sum(frames))
    B = len(frames)
    out_len = np.asarray([20 * t for t in frames], np.int32)
    in_len = np.asarray([120 * t + 1 for t in frames], np.int32)
    in_off = np.zeros(B, np.int32); out_off = np.zeros(B, np.int32)
    oi, oo = 32, 32
    for b in range(B):
        in_off[b], out_off[b] = oi, oo
        oi += int(in_len[b]) + 32
        oo += int(out_len[b]) + 32 + 8
    rows_in, rows_out = oi, oo          # 32 + 8 rows behind the last item: what one launch's grid covers (max_len + 72 rows per item)
    x = rng.standard_normal((rows_in, 24)).astype(np.float32)
    Cpad = 320
    ip = lambda a: a.ctypes.data_as(C.POINTER(C.c_int))  # noqa: E731
    outs = []
    for generic in (1, 0):
        out = np.full((rows_out, Cpad), 0x7fc0, np.uint16)           # bf16 NaN bits: untouched rows stay visible
        rc = lib.kkx_test_im2col(0, fp(x), rows_in, B, ip(in_off), ip(in_len), ip(out_off), ip(out_len), rows_out,
                                 int(out_len.max()), Cpad, generic, out.ctypes.data_as(C.POINTER(C.c_ushort)))
        assert rc == 0, lib.kkx_test_last_error()
        outs.append(out)
    assert np.array_equal(outs[0], outs[1])
    got = (outs[1].astype(np.uint32) << 16).view(np.float32)
    for b in range(B):
        for m in (0, 1, int(out_len[b]) // 2, int(out_len[b]) - 1):
            ref = np.zeros(Cpad, np.float32)
            for tap in range(12):
                ir = m * 6 + tap - 3
                if 0 <= ir < in_len[b]:
                    ref[tap * 22:(tap + 1) * 22] = x[in_off[b] + ir, :22]
            ref_bf = (torch.from_numpy(ref).to(torch.bfloat16).to(torch.float32)).numpy()
            assert np.array_equal(got[out_off[b] + m], ref_bf), (b, m)


@pytest.mark.parametrize("N", [3, 52, 130, 512])
def test_attention_matches_torch(lib, N):
    qkv = rnd(N, 2304, seed=N)
    t = torch.from_numpy(qkv)
    q, k, v = (t[:, i * 768:(i + 1) * 768].view(N, 12, 64).transpose(0, 1) for i in range(3))
    p = torch.softmax(q @ k.transpose(1, 2) / 8.0, -1)
    ref = (p @ v).transpose(0, 1).reshape(N, 768).numpy()
    out = np.zeros((N, 768), np.float32)
    rc = lib.kkx_test_attention(0, fp(qkv), N, fp(out))
    assert rc == 0, lib.kkx_test_last_error()
    np.testing.assert_allclose(out, ref, atol=2e-5, rtol=1e-4)


@pytest.mark.parametrize("lens", [[3], [64], [65], [130], [512], [52, 512, 1, 200, 129, 383]])
def test_attention_tcgen05_matches_torch_and_mma_sync(lib, lens):
    """kernels_attn.cu: S and P V on tcgen05 with P in tensor memory, against torch fp32 softmax attention and the
    round-1 mma.sync kernel.  Ragged items packed with gap rows; gap rows carry NaN so that a stale row reaching a
    valid result would show."""
    i32 = C.POINTER(C.c_int32)
    B = len(lens)
    off, o = [], 32
    for n in lens:
        off.append(o)
        o = (o + n + 32 + 7) & ~7
    rows = o
    qkv = np.full((rows, 2304), np.nan, np.float32)
    for b, n in enumerate(lens):
        qkv[off[b]:off[b] + n] = rnd(n, 2304, seed=100 * n + b)
    offa, lena = np.asarray(off, np.int32), np.asarray(lens, np.int32)
    outs = []
    for umma in (1, 0):
        out = np.zeros((rows, 768), np.float32)
        rc = lib.kkx_test_attention_batch(0, fp(qkv), B, offa.ctypes.data_as(i32), lena.ctypes.data_as(i32), rows, umma, fp(out))
        assert rc == 0, lib.kkx_test_last_error()
        outs.append(out)
    for b, n in enumerate(lens):
        t = torch.from_numpy(qkv[off[b]:off[b] + n])
        q, k, v = (t[:, i * 768:(i + 1) * 768].view(n, 12, 64).transpose(0, 1) for i in range(3))
        p = torch.softmax(q.double() @ k.double().transpose(1, 2) / 8.0, -1)
        ref = (p @ v.double()).transpose(0, 1).reshape(n, 768).numpy()
        for name, out in zip(("tcgen05", "mma.sync"), outs):
            got = out[off[b]:off[b] + n]
            assert np.isfinite(got).all(), f"{name}: item {b} has non-finite values"
            err = np.abs(got - ref).max()
            assert err < 2e-5, f"{name}: item {b} (N={n}) max abs error {err}"
    # rows outside the items are never written
    mask = np.ones(rows, bool)
    for b, n in enumerate(lens):
        mask[off[b]:off[b] + n] = False
    assert not outs[0][mask].any()


@pytest.mark.parametrize("L,Cc", [(50, 128), (1000, 256), (20001, 128)])
def test_instance_norm_adain_coefficients(lib, L, Cc):
    x = (rnd(L, Cc, seed=L) * 2 + 3 * rnd(1, Cc, seed=L + 1)).astype(np.float32)
    gb = rnd(2 * Cc, seed=L + 2, scale=0.3)
    sc, sh = np.zeros(Cc, np.float32), np.zeros(Cc, np.float32)
    rc = lib.kkx_test_adain_coef(0, fp(x), L, Cc, fp(gb), fp(sc), fp(sh))
    assert rc == 0, lib.kkx_test_last_error()
    ref = (1 + torch.from_numpy(gb[:Cc]))[None, :, None] * F.instance_norm(torch.from_numpy(x.T.copy())[None], eps=1e-5) \
        + torch.from_numpy(gb[Cc:])[None, :, None]
    got = x * sc + sh
    np.testing.assert_allclose(got, ref[0].T.numpy(), atol=3e-4, rtol=1e-4)


# ---------------------------------------------------------------------------- tensor-core path
def bf16_round(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(torch.bfloat16).to(torch.float32)


def run_conv_tc(lib, x, w_co_ks_ci, bias, dil, pad, m_len, out_rows, ors=1, oro=0, pscale=None, pshift=None, pact=0,
                pslope=0.0, palpha=None, res=None, res_shift=0, oscale=1.0, accumulate=0, out_init=None):
    L, Ci = x.shape
    Co, ks, _ = w_co_ks_ci.shape
    out = np.zeros((out_rows, Co), np.float32) if out_init is None else out_init.copy()
    rc = lib.kkx_test_conv_tc(0, fp(x), L, Ci, fp(w_co_ks_ci), fp(bias), Co, ks, dil, pad, fp(pscale), fp(pshift), pact,
                              C.c_float(pslope), fp(palpha), m_len, ors, oro, out_rows, fp(res),
                              0 if res is None else res.shape[0], res_shift, C.c_float(oscale), accumulate, fp(out))
    assert rc == 0, lib.kkx_test_last_error()
    return out


@pytest.mark.parametrize("L,Ci,Co,k,dil", [(300, 128, 128, 3, 1), (1000, 256, 256, 7, 3), (513, 128, 128, 11, 5),
                                           (130, 514, 1024, 3, 1), (77, 1090, 512, 3, 1), (260, 1090, 1024, 1, 1),
                                           (129, 64, 64, 3, 1)])
def test_tc_conv_matches_torch_on_bf16_operands(lib, L, Ci, Co, k, dil):
    x, w, b = rnd(L, Ci, seed=1), rnd(Co, Ci, k, seed=2, scale=1 / np.sqrt(Ci * k)), rnd(Co, seed=3)
    pad = dil * (k - 1) // 2
    ref = F.conv1d(bf16_round(x).T[None], bf16_round(w), torch.from_numpy(b), padding=pad, dilation=dil)[0].T.numpy()
    got = run_conv_tc(lib, x, np.ascontiguousarray(w.transpose(0, 2, 1)), b, dil, pad, L, L)
    np.testing.assert_allclose(got, ref, atol=3e-4, rtol=1e-4)
    # and against the fp32 conv: the stated bf16-operand tolerance
    ref32 = F.conv1d(torch.from_numpy(x.T)[None], torch.from_numpy(w), torch.from_numpy(b), padding=pad, dilation=dil)[0].T.numpy()
    assert np.sqrt(((got - ref32) ** 2).sum() / (ref32 ** 2).sum()) < 6e-3


@pytest.mark.parametrize("Ci,Co,k,s", [(512, 256, 20, 10), (256, 128, 12, 6)])
def test_tc_conv_transpose_phases(lib, Ci, Co, k, s):
    L, p = 141, (k - s) // 2
    x, w, b = rnd(L, Ci, seed=7), rnd(Ci, Co, k, seed=8, scale=0.05), rnd(Co, seed=9)
    xin = bf16_round(F.leaky_relu(torch.from_numpy(x), 0.1).numpy()).T[None]
    ref = F.conv_transpose1d(xin, bf16_round(w), torch.from_numpy(b), stride=s, padding=p)[0].T.numpy()
    out = np.full((L * s, Co), np.nan, np.float32)
    for r in range(s):
        q0 = 1 if r < p else 0
        ph = np.ascontiguousarray(np.stack([w[:, :, r], w[:, :, r + s]], axis=0).transpose(2, 0, 1))  # [Co][2][Ci]
        out = run_conv_tc(lib, x, ph, b, -1, -q0, L, L * s, ors=s, oro=q0 * s + r - p, pact=1, pslope=0.1, out_init=out)
    assert not np.isnan(out).any()
    np.testing.assert_allclose(out, ref, atol=3e-4, rtol=1e-4)


def test_tc_conv_fused_prologue_epilogue(lib):
    L, Cc, k = 700, 128, 7
    x, w, b = rnd(L, Cc, seed=10), rnd(Cc, Cc, k, seed=11, scale=0.04), rnd(Cc, seed=12)
    sc, sh = (1 + 0.3 * rnd(Cc, seed=13)).astype(np.float32), (0.2 * rnd(Cc, seed=14)).astype(np.float32)
    alpha = np.clip(1 + 0.3 * rnd(Cc, seed=15), 0.3, 2).astype(np.float32)
    res, init = rnd(L, Cc, seed=16), rnd(L, Cc, seed=17)
    xt = torch.from_numpy(x) * torch.from_numpy(sc) + torch.from_numpy(sh)
    a = torch.from_numpy(alpha)
    xt = xt + (1 / a) * torch.sin(a * xt) ** 2
    y = F.conv1d(bf16_round(xt.numpy()).T[None], bf16_round(w), torch.from_numpy(b), padding=3)[0].T
    ref = (torch.from_numpy(init) + (1 / 3) * (y + torch.from_numpy(res))).numpy()
    got = run_conv_tc(lib, x, np.ascontiguousarray(w.transpose(0, 2, 1)), b, 1, 3, L, L, pscale=sc, pshift=sh, pact=2,
                      palpha=alpha, res=res, oscale=1 / 3, accumulate=1, out_init=init)
    np.testing.assert_allclose(got, ref, atol=2e-3, rtol=1e-3)


# ---------------------------------------------------------------------------- split-TF32 tensor-core GEMM
@pytest.mark.parametrize("L,Ci,Co,k", [(512, 768, 2304, 1), (300, 2048, 768, 1), (200, 128, 768, 1), (140, 640, 2048, 1),
                                       (333, 512, 512, 5), (77, 512, 50, 1), (260, 256, 256, 3)])
@pytest.mark.parametrize("nprod", [3, 4])
def test_split_tf32_gemm_is_fp32_grade(lib, L, Ci, Co, k, nprod):
    x, w, b = rnd(L, Ci, seed=21), rnd(Co, Ci, k, seed=22, scale=1 / np.sqrt(Ci * k)), rnd(Co, seed=23)
    pad = (k - 1) // 2
    ref64 = F.conv1d(torch.from_numpy(x.T.astype(np.float64))[None], torch.from_numpy(w.astype(np.float64)),
                     torch.from_numpy(b.astype(np.float64)), padding=pad)[0].T.numpy()
    ref32 = F.conv1d(torch.from_numpy(x.T)[None], torch.from_numpy(w), torch.from_numpy(b), padding=pad)[0].T.numpy()
    out = np.zeros((L, Co), np.float32)
    rc = lib.kkx_test_conv_tf32(0, fp(x), L, Ci, fp(np.ascontiguousarray(w.transpose(0, 2, 1))), fp(b), Co, k, 1, pad,
                                nprod, 0, fp(out))
    assert rc == 0, lib.kkx_test_last_error()
    e_tc = np.abs(out - ref64).max()
    e_32 = np.abs(ref32 - ref64).max()
    rms_tc = np.sqrt(((out - ref64) ** 2).mean())
    rms_32 = np.sqrt(((ref32 - ref64) ** 2).mean())
    print(f"split-TF32 x{nprod}: max err {e_tc:.3e} (torch fp32 {e_32:.3e}), rms err {rms_tc:.3e} (fp32 {rms_32:.3e})")
    assert e_tc < 2e-5 and rms_tc < 8 * max(rms_32, 1e-8)


@pytest.mark.parametrize("L,Ci,Co,k", [(512, 768, 2304, 1), (300, 2048, 768, 1), (200, 128, 768, 1), (140, 640, 2048, 1),
                                       (333, 512, 512, 5), (257, 512, 256, 3), (64, 512, 50, 1), (52, 768, 768, 1),
                                       (20000, 768, 768, 1), (9000, 512, 512, 3)])
def test_split_fp16_gemm_is_fp32_grade(lib, L, Ci, Co, k):
    """"3xFP16": fp16 hi/lo operand planes (the same 22 significand bits as the tf32 pair) on kind::f16 MMAs with the
    power-of-two plane scaling undone in the epilogue -- must be as close to the fp64 result as torch's own fp32.
    The two largest cases take the persistent kernel (>= 148 tiles), the others the single-tile kernel.  Inputs span
    five decades (row scales 1e-3 .. 30) so that small activations and the saturating range are exercised."""
    x = rnd(L, Ci, seed=L + Ci)
    x *= np.exp(np.random.default_rng(7).uniform(np.log(1e-3), np.log(30.0), size=(L, 1))).astype(np.float32)
    w = rnd(Co, Ci, k, seed=L + Co, scale=0.5 / np.sqrt(Ci * k))
    b = rnd(Co, seed=3)
    pad = (k - 1) // 2
    tx, tw, tb = torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(b)
    ref64 = F.conv1d(tx.double().T[None], tw.double(), tb.double(), padding=pad)[0].T.numpy()
    ref32 = F.conv1d(tx.T[None], tw, tb, padding=pad)[0].T.numpy()
    out = np.zeros((L, Co), np.float32)
    rc = lib.kkx_test_conv_f16x3(0, fp(x), L, Ci, fp(np.ascontiguousarray(w.transpose(0, 2, 1))), fp(b), Co, k, 1, pad,
                                 0, fp(out))
    assert rc == 0, lib.kkx_test_last_error()
    scale = np.abs(ref64).max(axis=1, keepdims=True) + 1e-6          # per-row magnitude (rows differ by 4 decades)
    e_tc = (np.abs(out - ref64) / scale).max()
    e_32 = (np.abs(ref32 - ref64) / scale).max()
    rms_tc = np.sqrt((((out - ref64) / scale) ** 2).mean())
    rms_32 = np.sqrt((((ref32 - ref64) / scale) ** 2).mean())
    print(f"split-FP16 x3: max rel err {e_tc:.3e} (torch fp32 {e_32:.3e}), rms {rms_tc:.3e} (fp32 {rms_32:.3e})")
    assert e_tc < 4e-6 and rms_tc < 8 * max(rms_32, 1e-9)


@pytest.mark.parametrize("L,Ci,Co,k,eact,use_res", [(20000, 768, 768, 1, 0, True), (128 * 151 + 5, 768, 2304, 1, 0, False),
                                                     (128 * 37, 2048, 768, 1, 0, True), (9000, 512, 512, 3, 0, False),
                                                     (128 * 75 + 1, 768, 2048, 1, 3, False), (300, 640, 2048, 1, 0, True)])
def test_split_fp16_gemm_kernels_are_bit_identical(lib, L, Ci, Co, k, eact, use_res):
    """The single-tile kernel, the persistent kernel and the persistent CTA-pair kernel (tcgen05 cta_group::2: 256 x 128
    tiles, each CTA holds half of the weight tile) accumulate every output element in the same order: identical bits,
    for odd and even m-tile counts (an odd count ends with a pair whose second CTA stores nothing), ragged tails,
    residual + scale and the GELU epilogue.  Which kernel runs depends on the batch, so this is what keeps results
    independent of the batch composition."""
    x = rnd(L, Ci, seed=L + Ci)
    w = rnd(Co, Ci, k, seed=L + Co, scale=0.5 / np.sqrt(Ci * k))
    b = rnd(Co, seed=3)
    res = rnd(L, Co, seed=5) if use_res else None
    pad = (k - 1) // 2
    outs = []
    for kernel in (1, 2, 3):
        out = np.full((L, Co), np.nan, np.float32)
        rc = lib.kkx_test_conv_f16x3_k(0, fp(x), L, Ci, fp(np.ascontiguousarray(w.transpose(0, 2, 1))), fp(b), Co, k, 1, pad,
                                       eact, kernel, fp(res) if use_res else None, 0.5 if use_res else 1.0, fp(out))
        assert rc == 0, lib.kkx_test_last_error()
        assert np.isfinite(out).all()
        outs.append(out)
    assert np.array_equal(outs[0], outs[1]), "persistent kernel differs from the single-tile kernel"
    assert np.array_equal(outs[0], outs[2]), "CTA-pair kernel differs from the single-tile kernel"
    tx, tw, tb = torch.from_numpy(x), torch.from_numpy(w), torch.from_numpy(b)
    ref = F.conv1d(tx.double().T[None], tw.double(), tb.double(), padding=pad)[0].T
    if eact == 3:
        ref = 0.5 * ref * (1.0 + torch.tanh(0.7978845608028654 * (ref + 0.044715 * ref ** 3)))
    ref = ref.numpy()
    if use_res:
        ref = (ref + res) * 0.5
    assert np.abs(outs[2] - ref).max() < 2e-5 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("Cc,k,dil", [(128, 3, 1), (128, 11, 5), (256, 7, 3)])
def test_tc_conv_large_ragged_fused_epilogue(lib, Cc, k, dil):
    # a large conv (>= 1184 128-row tiles) on the single-tile kernel with a ragged tail (L not a multiple of 128)
    # and residual, scale and accumulate fused in the epilogue
    L = 128 * 4 * 300 + 77 if Cc == 128 else 128 * 4 * 150 + 205
    x, w, b = rnd(L, Cc, seed=31), rnd(Cc, Cc, k, seed=32, scale=1 / np.sqrt(Cc * k)), rnd(Cc, seed=33)
    res, init = rnd(L, Cc, seed=34), rnd(L, Cc, seed=35)
    pad = dil * (k - 1) // 2
    y = F.conv1d(bf16_round(x).T[None], bf16_round(w), torch.from_numpy(b), padding=pad, dilation=dil)[0].T
    ref = (torch.from_numpy(init) + (1 / 3) * (y + torch.from_numpy(res))).numpy()
    got = run_conv_tc(lib, x, np.ascontiguousarray(w.transpose(0, 2, 1)), b, dil, pad, L, L, res=res, oscale=1 / 3,
                      accumulate=1, out_init=init)
    np.testing.assert_allclose(got, ref, atol=5e-4, rtol=1e-4)


@pytest.mark.parametrize("Cc,k,dil,lens", [(128, 3, 1, [300]), (128, 11, 5, [700, 13, 257]), (128, 7, 3, [256, 512, 1]),
                                            (256, 7, 1, [333]), (256, 11, 5, [129, 640]), (256, 3, 3, [128, 127])])
@pytest.mark.parametrize("variant", ["conv1_f32_to_bf16_stats", "conv2_bf16_res_accumulate"])
def test_fused_arb_conv(lib, Cc, k, dil, lens, variant):
    # kernels_arb.cu: AdaIN scale/shift + Snake inside the conv, row-shifted smem views per tap, ragged items
    # separated by NaN gap rows (the hook fills them), epilogue statistics.  Reference: float64 conv of the
    # same bf16-rounded operands (tools/arb_probe.py).
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from arb_probe import run_case
    if variant == "conv1_f32_to_bf16_stats":
        out, ref, sums, rs = run_case(lib, Cc, k, dil, lens, 0, 1, 0, 1.0, 0, 0)
        np.testing.assert_allclose(out, ref, rtol=2 ** -7, atol=1e-3)      # one bf16 ulp of the stored value
    else:
        out, ref, sums, rs = run_case(lib, Cc, k, dil, lens, 1, 0, 1, 1.0 / 3.0, 1, 0)
        np.testing.assert_allclose(out, ref, rtol=1e-4, atol=1e-3)         # fast-sin + bf16 re-rounding flips
    assert not np.isnan(out).any()
    np.testing.assert_allclose(sums, rs, rtol=1e-3, atol=1e-2 * float(np.abs(rs).max()) * 1e-2)


@pytest.mark.parametrize("Cc,k,dil,lens", [(128, 3, 1, [300]), (128, 11, 5, [700, 13, 257]), (128, 7, 3, [256, 512, 1]),
                                            (256, 7, 1, [333]), (256, 11, 5, [129, 640]), (256, 3, 3, [128, 127])])
@pytest.mark.parametrize("variant", ["conv1_bf16_in", "conv2_bf16_stream", "conv2_bf16_res_to_f32"])
def test_fused_arb_conv_bf16_residual_stream(lib, Cc, k, dil, lens, variant):
    # the res-block's residual stream kept in bf16 between iterations (kernels_arb.cu, SB variants): conv1 reads bf16 x;
    # conv2 adds the bf16 residual and writes the next bf16 x, or (last iteration) the fp32 block output.  Statistics
    # come from the fp32 accumulator either way.
    import os
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tools"))
    from arb_probe import run_case_stream
    lib.kkx_test_arb_conv_stream.restype = C.c_int
    if variant == "conv1_bf16_in":
        out, ref, sums, rs = run_case_stream(lib, Cc, k, dil, lens, 0, 1, 1.0, 0)
        np.testing.assert_allclose(out, ref, rtol=2 ** -7, atol=3e-3)
    elif variant == "conv2_bf16_stream":
        out, ref, sums, rs = run_case_stream(lib, Cc, k, dil, lens, 1, 1, 1.0, 0)
        np.testing.assert_allclose(out, ref, rtol=2 ** -7, atol=3e-3)
    else:
        out, ref, sums, rs = run_case_stream(lib, Cc, k, dil, lens, 1, 0, 1.0 / 3.0, 1)
        np.testing.assert_allclose(out, ref, rtol=1e-4, atol=1e-3)
    assert not np.isnan(out).any()
    np.testing.assert_allclose(sums, rs, rtol=1e-3, atol=1e-2 * float(np.abs(rs).max()) * 1e-2)
