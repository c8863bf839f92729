"""The C++ ONNX reader behind kkx_create (kokorox_b200/csrc/onnx_loader.cu): OrtKoko::new is given the downloaded
.onnx file (ort_base.rs:27-33, hf_cache.rs:135-144), so the library must open that file itself.

No real export exists in this environment (no network), so the files are SYNTHETIC EXPORTS of the random-init
model written by the independent protobuf writer of tests/test_onnx_init.py, laid out the way torch.onnx lays a
Kokoro export out: state-dict names only where the exporter keeps them (embeddings, norms, biases, alphas, behind
a "kmodel." wrapper prefix), nn.Linear weights as anonymous transposed "onnx::MatMul_N" operands, weight-normed
conv weights constant-folded into "onnx::Conv_N", nn.LSTM parameters as "onnx::LSTM_N" W/R/B in ONNX gate order,
node names carrying the torch scope path.  CPU tests convert through the host-only kkx_convert_model_file and
compare the recovered state dict bit for bit; the GPU test loads the .onnx through kkx_create and requires audio
bit-identical to the KKXW load.
"""
import numpy as np
import pytest

from kokorox_b200.weightfile import random_weights, read_weights, weight_specs
from tests.test_onnx_init import model, node, tensor, to_onnx_lstm, fld, fvar


@pytest.fixture(scope="module")
def built():
    from kokorox_b200 import build
    build.build()
    from kokorox_b200 import onn
    return onn


@pytest.fixture(scope="module")
def ref():
    return random_weights(1234)


def scope_name(module_path: str, op: str, wrapper: str = "kmodel") -> str:
    """torch.onnx node name of `op` inside `module_path`: one level per called module, each the module's name with
    the parents' atoms dropped but numeric atoms kept with the non-numeric atom before them
    (torch.onnx _unqualified_variable_name): text_encoder.cnn.0.0 -> /text_encoder/cnn.0/cnn.0.0/Conv."""
    atoms = module_path.split(".")
    levels = []
    for i, a in enumerate(atoms):
        nxt_numeric = i + 1 < len(atoms) and atoms[i + 1].isdigit()
        if not a.isdigit():
            if not nxt_numeric:
                levels.append(a)
        else:
            j = i
            while atoms[j].isdigit():
                j -= 1
            levels.append(".".join(atoms[j:i + 1]))
    return "/" + "/".join(([wrapper] if wrapper else []) + levels + [op])


def attr_int(name, v):
    return fld(5, fld(1, name.encode()) + fvar(3, v) + fvar(20, 2))


def node_with_attrs(op, name, inputs, outputs, attrs=b""):
    msg = b"".join(fld(1, i.encode()) for i in inputs) + b"".join(fld(2, o.encode()) for o in outputs)
    return msg + fld(3, name.encode()) + fld(4, op.encode()) + attrs


def quant_u8(w, axis=None):
    """Asymmetric uint8 quantisation (ORT quantize_dynamic style): returns (q, scale, zero_point, dequantised)."""
    w = w.astype(np.float32)
    lo, hi = min(float(w.min()), 0.0), max(float(w.max()), 0.0)
    scale = np.float32((hi - lo) / 255.0) if hi > lo else np.float32(1.0)
    zp = np.uint8(np.clip(round(-lo / float(scale)), 0, 255))
    q = np.clip(np.round(w / scale) + np.float32(zp), 0, 255).astype(np.uint8)
    deq = ((q.astype(np.float32) - np.float32(zp)) * scale).astype(np.float32)
    return q, scale, zp, deq


def quant_q4(w, bs=32):
    """MatMulNBits packing of a torch Linear weight [N, K]: blocks of bs along K, 4-bit codes, zero point 8."""
    N, K = w.shape
    nblk = (K + bs - 1) // bs
    wp = np.zeros((N, nblk * bs), np.float32)
    wp[:, :K] = w
    blocks = wp.reshape(N, nblk, bs)
    amax = np.abs(blocks).max(axis=2)
    scale = np.where(amax > 0, amax / 7.0, 1.0).astype(np.float32)
    q = np.clip(np.round(blocks / scale[:, :, None]) + 8, 0, 15).astype(np.uint8)
    packed = (q[:, :, 0::2] | (q[:, :, 1::2] << 4)).astype(np.uint8)            # low nibble first
    deq = ((q.astype(np.float32) - 8.0) * scale[:, :, None]).astype(np.float32).reshape(N, nblk * bs)[:, :K]
    return packed, scale.reshape(-1), deq


def build_export(ref, mode="fp32", wrapper="kmodel", unfolded_wn=(), no_node_names=False):
    """Returns (file bytes, expected state dict).  mode: fp32 | fp16 | int8 | q4."""
    specs = weight_specs()
    kinds = {n: k for n, _s, k in specs}
    pre = (wrapper + ".") if wrapper else ""
    enc = (lambda a: a.astype(np.float16)) if mode == "fp16" else (lambda a: a)
    rt = (lambda a: a.astype(np.float16).astype(np.float32)) if mode == "fp16" else (lambda a: a)
    inits, nodes, expect = [], [], {}
    counter = [1000]

    def anon(op):
        counter[0] += 1
        return f"onnx::{op}_{counter[0]}"

    def nname(mod, op):
        counter[0] += 1
        return f"{op}_{counter[0]}" if no_node_names else scope_name(mod, op, wrapper)

    lstm_mods = sorted({n.rsplit(".", 1)[0] for n in ref if ".weight_ih_l0" in n and not n.endswith("_reverse")})
    done = set()
    for mod in lstm_mods:
        W, R, B = to_onnx_lstm(ref, mod)
        keys = [k for k in ref if k.startswith(mod + ".") and "_l0" in k]
        done.update(keys)
        if mode == "int8":
            # com.microsoft DynamicQuantizeLSTM: W [D, I, 4H], R [D, H, 4H] quantised per direction
            Wt, Rt = np.transpose(W, (0, 2, 1)), np.transpose(R, (0, 2, 1))
            qs = [[quant_u8(Wt[d]) for d in range(2)], [quant_u8(Rt[d]) for d in range(2)]]
            names = [anon("LSTM") for _ in range(7)]
            Wq = np.stack([qs[0][d][0] for d in range(2)]); Rq = np.stack([qs[1][d][0] for d in range(2)])
            inits += [tensor(names[0], Wq, dtype_code=2), tensor(names[1], Rq, dtype_code=2), tensor(names[2], B),
                      tensor(names[3], np.array([qs[0][d][1] for d in range(2)], np.float32)),
                      tensor(names[4], np.array([qs[0][d][2] for d in range(2)], np.uint8), dtype_code=2),
                      tensor(names[5], np.array([qs[1][d][1] for d in range(2)], np.float32)),
                      tensor(names[6], np.array([qs[1][d][2] for d in range(2)], np.uint8), dtype_code=2)]
            nodes.append(node_with_attrs("DynamicQuantizeLSTM", nname(mod, "LSTM_quant"),
                                         ["x", names[0], names[1], names[2], "", "", "", "", names[3], names[4], names[5], names[6]],
                                         ["y_" + mod]))
            Wd = np.stack([qs[0][d][3] for d in range(2)]).transpose(0, 2, 1)
            Rd = np.stack([qs[1][d][3] for d in range(2)]).transpose(0, 2, 1)
            from kokorox_b200.onnx_init import onnx_lstm_to_torch
            for k, v in onnx_lstm_to_torch(Wd, Rd, B).items():
                expect[f"{mod}.{k}"] = v
        else:
            names = [anon("LSTM") for _ in range(3)]
            inits += [tensor(nm, enc(a)) for nm, a in zip(names, (W, R, B))]
            nodes.append(node("LSTM", nname(mod, "LSTM"), ["x"] + names, ["y_" + mod]))
            for k in keys:
                expect[k] = rt(ref[k])
    for name, shape, kind in specs:
        if name in done:
            continue
        w = ref[name]
        mod = name.rsplit(".", 1)[0]
        is_weight = name.endswith(".weight") and kind not in ("emb", "ln_w")
        if name == "bert.pooler.weight" or name == "bert.pooler.bias":
            inits.append(tensor(pre + name, enc(w)))       # present in the checkpoint, unused by the graph
            continue
        if is_weight and w.ndim == 2:                     # nn.Linear -> MatMul(x, W^T) + Add(bias)
            out_v = "mm_" + mod
            if mode == "int8":
                q, sc, zp, deq = quant_u8(np.ascontiguousarray(w.T))
                base = anon("MatMul")
                inits += [tensor(base + "_quantized", q, dtype_code=2), tensor(base + "_scale", np.float32(sc).reshape(())),
                          tensor(base + "_zero_point", np.uint8(zp).reshape(()), dtype_code=2)]
                nodes.append(node("MatMulInteger", nname(mod, "MatMul_quant"), ["xq", base + "_quantized", "xzp", base + "_zero_point"], [out_v]))
                expect[name] = np.ascontiguousarray(deq.T)
            elif mode == "q4" and w.shape[1] % 32 == 0 and w.shape[0] >= 16:
                packed, scales, deq = quant_q4(w)
                b, s = anon("MatMul") + "_Q4", anon("MatMul") + "_scales"
                inits += [tensor(b, packed, dtype_code=2), tensor(s, scales)]
                attrs = attr_int("K", w.shape[1]) + attr_int("N", w.shape[0]) + attr_int("bits", 4) + attr_int("block_size", 32)
                nodes.append(node_with_attrs("MatMulNBits", nname(mod, "MatMul_Q4"), ["x", b, s], [out_v], attrs))
                expect[name] = deq
            else:
                a = anon("MatMul")
                inits.append(tensor(a, enc(np.ascontiguousarray(w.T))))
                nodes.append(node("MatMul", nname(mod, "MatMul"), ["x", a], [out_v]))
                expect[name] = rt(w)
            if mod + ".bias" in ref:
                nodes.append(node("Add", nname(mod, "Add"), [pre + mod + ".bias", out_v], ["add_" + mod]))
        elif is_weight and w.ndim == 3:                   # Conv1d / ConvTranspose1d
            op = "ConvTranspose" if kind in ("wn_convT", "wn_pool") else "Conv"
            ins = ["x"]
            if name in unfolded_wn:                       # exporter did not fold weight-norm: g, v stay named
                rng = np.random.default_rng(abs(hash(name)) % (2 ** 31))
                v = (w * rng.uniform(0.5, 2.0, size=(w.shape[0], 1, 1))).astype(np.float32)
                g = np.sqrt((w.astype(np.float64) ** 2).sum(axis=(1, 2), keepdims=True)).astype(np.float32)
                inits += [tensor(pre + mod + ".weight_g", enc(g)), tensor(pre + mod + ".weight_v", enc(v))]
                g64, v64 = rt(g).astype(np.float64), rt(v).astype(np.float64)
                nrm = np.sqrt((v64 * v64).sum(axis=(1, 2), keepdims=True))
                expect[name] = (v64 * (g64 / nrm)).astype(np.float32)
                ins.append("wn_" + mod)
            elif mode == "int8" and kind != "wn_pool" and w.size >= 4096:
                q, sc, zp, deq = quant_u8(w)
                base = anon("Conv")
                inits += [tensor(base + "_quantized", q, dtype_code=2), tensor(base + "_scale", np.float32(sc).reshape(())),
                          tensor(base + "_zero_point", np.uint8(zp).reshape(()), dtype_code=2)]
                op = "ConvInteger"
                ins = ["xq", base + "_quantized", "xzp", base + "_zero_point"]
                expect[name] = deq
            else:
                a = anon("Conv") if kind != "conv" else pre + name     # plain convs (noise_convs) keep their names
                inits.append(tensor(a, enc(w)))
                ins.append(a)
                expect[name] = rt(w)
            if mod + ".bias" in ref and op != "ConvInteger":
                ins.append(pre + mod + ".bias")
            nodes.append(node(op, nname(mod, op if op != "ConvInteger" else "Conv_quant"), ins, ["conv_" + mod]))
        else:                                             # everything the exporter keeps by name
            a = w.reshape(-1) if kind == "alpha" and mode == "fp16" else w     # alphas as [C] or [1,C,1]
            inits.append(tensor(pre + name, enc(a)))
            expect[name] = rt(w)
    inits.append(tensor("onnx::Reshape_1", np.array([1, -1], dtype=np.int64)))
    return model(inits, nodes), expect


def check(onn, tmp_path, blob, expect, tag):
    src = tmp_path / f"kokoro_{tag}.onnx"
    src.write_bytes(blob)
    dst = tmp_path / f"kokoro_{tag}.kkxw"
    n = onn.convert_model_file(str(src), str(dst))
    got = read_weights(str(dst))
    assert n == len(got)
    for name, shape, _k in weight_specs():
        if name.startswith("bert.pooler"):
            continue
        assert name in got, name
        assert tuple(got[name].shape) == tuple(shape), name
        np.testing.assert_array_equal(got[name], expect[name].reshape(shape), err_msg=name)
    return str(src)


def test_spec_tables_agree(built):
    lib = dict(built.library_tensor_specs())
    py = {n: tuple(s) for n, s, _k in weight_specs() if not n.startswith("bert.pooler")}
    assert lib == py


def test_scope_names():
    assert scope_name("text_encoder.cnn.0.0", "Conv") == "/kmodel/text_encoder/cnn.0/cnn.0.0/Conv"
    assert scope_name("predictor.F0.1.conv1", "Conv", "") == "/predictor/F0.1/conv1/Conv"
    assert (scope_name("bert.encoder.albert_layer_groups.0.albert_layers.0.attention.query", "MatMul_3") ==
            "/kmodel/bert/encoder/albert_layer_groups.0/albert_layers.0/attention/query/MatMul_3")


def test_fp32_export_resolves_bit_exactly(built, ref, tmp_path):
    blob, expect = build_export(ref, "fp32")
    check(built, tmp_path, blob, expect, "fp32")


def test_fp16_export_without_wrapper_prefix(built, ref, tmp_path):
    blob, expect = build_export(ref, "fp16", wrapper="")
    check(built, tmp_path, blob, expect, "fp16")


def test_unfolded_weight_norm_is_folded(built, ref, tmp_path):
    wn = {n for n, _s, k in weight_specs() if k in ("wn_conv", "wn_convT", "post_w") and ("resblocks.4" in n or "ups.1" in n or "cnn.1" in n)}
    blob, expect = build_export(ref, "fp32", unfolded_wn=wn)
    src = tmp_path / "wn.onnx"
    src.write_bytes(blob)
    dst = tmp_path / "wn.kkxw"
    built.convert_model_file(str(src), str(dst))
    got = read_weights(str(dst))
    for name in wn:
        np.testing.assert_allclose(got[name], expect[name], rtol=2e-7, atol=0, err_msg=name)
    for name in ("decoder.generator.resblocks.0.convs1.0.weight", "bert_encoder.weight"):
        np.testing.assert_array_equal(got[name], expect[name])


def test_int8_dynamic_quantised_export(built, ref, tmp_path):
    blob, expect = build_export(ref, "int8")
    check(built, tmp_path, blob, expect, "int8")


def test_q4_matmulnbits_export(built, ref, tmp_path):
    blob, expect = build_export(ref, "q4")
    check(built, tmp_path, blob, expect, "q4")


def test_bias_fallback_and_unresolved_report(built, ref, tmp_path, weights_path):
    # exporters that do not name nodes by scope ("MatMul_12"): modules are recovered from the bias a Conv consumes or
    # the Add behind a MatMul adds; bias-less convs (conv1x1) and LSTMs cannot be, and the error must list them
    blob, _ = build_export(ref, "fp32", no_node_names=True)
    src = tmp_path / "anon.onnx"
    src.write_bytes(blob)
    with pytest.raises(built.KkxError) as e:
        built.convert_model_file(str(src), str(tmp_path / "anon.kkxw"))
    msg = str(e.value)
    assert "55 tensors missing" in msg and "conv1x1.weight" in msg and "lstm.weight_ih_l0" in msg
    assert "25 weight-sized initialisers were not placed" in msg and "onnx::LSTM_" in msg and "pooler" not in msg
    assert "attention.query.weight" not in msg and "conv_post.weight" not in msg     # resolved through their biases
    # a file that is neither format
    junk = tmp_path / "junk.bin"
    junk.write_bytes(b"\xff" * 4096)
    with pytest.raises(built.KkxError):
        built.convert_model_file(str(junk), str(tmp_path / "junk.kkxw"))
    # a corrupt KKXW header (offset wraps) is an error, not a crash (ADVICE r1)
    with open(weights_path, "rb") as f:
        good = f.read(4096)
    bad = bytearray(good)
    p = 16 + 2 + int.from_bytes(good[16:18], "little") + 8 + 4 * int.from_bytes(good[16 + 2 + int.from_bytes(good[16:18], "little") + 4:][:4], "little")
    bad[p:p + 8] = (2 ** 64 - 64).to_bytes(8, "little")
    (tmp_path / "bad.kkxw").write_bytes(bytes(bad))
    with pytest.raises(built.KkxError):
        built.convert_model_file(str(tmp_path / "bad.kkxw"), str(tmp_path / "bad2.kkxw"))


@pytest.mark.gpu
def test_kkx_create_opens_the_onnx_file(built, ref, tmp_path, weights_path):
    """OrtKoko::new(model_path) with the .onnx path: audio must be bit-identical to the KKXW load, and a second
    session of the same file must share the device weight set."""
    from kokorox_b200.synth import synth_case
    blob, _ = build_export(ref, "fp32")
    src = tmp_path / "kokoro-v1.0.onnx"
    src.write_bytes(blob)
    a = built.B200Koko.new(weights_path)
    b = built.B200Koko.new(str(src))
    c = built.B200Koko.new(str(src))
    try:
        assert b.get_stat("weights_from_onnx") == 1 and a.get_stat("weights_from_onnx") == 0
        assert b.get_stat("weights_sessions") == 2 and c.get_stat("weights_sessions") == 2
        ids, style = synth_case(60, 5, 6)
        for m in (a, b, c):
            m.set_noise(None)
        ya, da = a.infer_batch([ids], [style], [1.0], return_durations=True)
        yb, db = b.infer_batch([ids], [style], [1.0], return_durations=True)
        yc = c.infer_one(ids, style, 1.0)
        assert np.array_equal(da[0], db[0])
        assert np.array_equal(ya[0], yb[0]) and np.array_equal(ya[0], yc)
    finally:
        for m in (a, b, c):
            m.close()
