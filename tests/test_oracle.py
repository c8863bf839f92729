"""CPU tests (-m "not gpu"): the oracle against its pinned vectors, the weight format, and the
ALBERT restatement against transformers.AlbertModel."""
import os

import numpy as np
import pytest
import torch

from tests.conftest import REF_EXAMPLE_IDS, REF_TOKENIZE_IDS, make_noise, synth_case
from tests.test_parity_gpu import avg_spectrum_db_diff

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_param_counts_match_published_totals():
    # SURVEY.md A.12: per-module totals of Kokoro-82M (weight-norm un-folded)
    from kokorox_b200.weightfile import param_count_unfolded
    pc = param_count_unfolded()
    assert pc == {"bert": 6292480, "bert_encoder": 393728, "text_encoder": 5606400,
                  "predictor": 16194612, "decoder": 53276190}
    assert sum(pc.values()) == 81763410


def test_weightfile_roundtrip(tmp_path):
    from kokorox_b200.weightfile import read_weights, write_weights
    from collections import OrderedDict
    rng = np.random.default_rng(0)
    t = OrderedDict(a=rng.standard_normal((3, 5)).astype(np.float32), b=np.arange(7, dtype=np.float32),
                    c=rng.standard_normal((2, 3, 4)).astype(np.float32))
    p = str(tmp_path / "w.kkxw")
    write_weights(p, t)
    r = read_weights(p)
    assert list(r) == list(t)
    for k in t:
        assert r[k].shape == t[k].shape and np.array_equal(r[k], t[k])
    with open(p, "r+b") as f:
        f.write(b"XXXX")
    with pytest.raises(ValueError):
        read_weights(p)


def test_reference_token_vectors_are_in_domain():
    # tokenize.rs:119-129 pins the id<->symbol table; ids 0..177 (vocab.rs:5-20)
    for ids in (REF_EXAMPLE_IDS, REF_TOKENIZE_IDS):
        assert ids[0] == 0 and ids[-1] == 0 and 0 <= min(ids) and max(ids) <= 177
    assert len(REF_EXAMPLE_IDS) == 23 and len(REF_TOKENIZE_IDS) == 17


def test_albert_restatement_matches_transformers(oracle, weights):
    transformers = pytest.importorskip("transformers")
    cfg = transformers.AlbertConfig(vocab_size=178, embedding_size=128, hidden_size=768, num_attention_heads=12,
                                    intermediate_size=2048, max_position_embeddings=512, num_hidden_layers=12,
                                    num_hidden_groups=1, hidden_dropout_prob=0.0, attention_probs_dropout_prob=0.0,
                                    hidden_act="gelu_new", type_vocab_size=2)
    m = transformers.AlbertModel(cfg).eval()
    sd = {k[len("bert."):]: torch.from_numpy(np.array(v)) for k, v in weights.items() if k.startswith("bert.")}
    missing, unexpected = m.load_state_dict(sd, strict=False)
    assert not unexpected, unexpected
    assert all("position_ids" in k for k in missing), missing
    ids, _ = synth_case(40, 11, 12)
    with torch.no_grad():
        ref = m(torch.from_numpy(ids)[None], attention_mask=torch.ones(1, len(ids), dtype=torch.long)).last_hidden_state[0]
        got = oracle.albert(torch.from_numpy(ids))
    assert torch.allclose(ref, got, atol=2e-5, rtol=1e-4), float((ref - got).abs().max())


@pytest.mark.parametrize("name", ["ref_example", "ref_tokenize", "cfg0"])
def test_oracle_reproduces_golden(oracle, name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    noise = make_noise(int(g["noise_frames_max"]), seed=int(g["noise_seed"]))
    r = oracle.forward(g["tokens"], g["style"], float(g["speed"]), noise=noise, stages=True)
    assert np.array_equal(r["pred_dur"], g["pred_dur"])
    assert r["audio"].shape == g["audio"].shape == (600 * int(g["pred_dur"].sum()),)
    np.testing.assert_allclose(r["stages"]["dur_float"], g["stage.dur_float"], rtol=0, atol=2e-5)
    np.testing.assert_allclose(r["stages"]["F0"], g["stage.F0"], rtol=0, atol=2e-3)
    np.testing.assert_allclose(r["stages"]["N"], g["stage.N"], rtol=0, atol=1e-4)
    # torch's CPU reductions follow the thread count: with 16 threads instead of the 8 the vectors were made with, F0
    # moves by 5e-4 and N by 1e-5, and since the harmonic source integrates F0 into a phase of 1e4..1e5 rad the
    # free-running waveform moves by up to 0.08 (test_parity_gpu.py).  So it is compared phase-insensitively (measured
    # 0.07 dB), and the waveform is held sample for sample with the pinned F0 / N curves teacher-forced (2e-7).
    assert avg_spectrum_db_diff(g["audio"], r["audio"]) < 0.5
    t = oracle.forward(g["tokens"], g["style"], float(g["speed"]), noise=noise, stages=True,
                       inject={"pred_dur": g["pred_dur"], "F0": g["stage.F0"], "N": g["stage.N"]})
    np.testing.assert_allclose(t["stages"]["har_source"], g["stage.har_source"], rtol=0, atol=1e-5)
    err = np.abs(t["audio"] - g["audio"]).max()
    assert err < 1e-4, err


def test_oracle_structure_properties(oracle):
    ids, style = synth_case(30, 5, 6)
    r = oracle.forward(ids, style, 1.0, noise_seed=1, stages=True)
    st = r["stages"]
    T = r["T"]
    assert (r["pred_dur"] >= 1).all() and T == int(r["pred_dur"].sum())
    assert st["idx"].shape == (T,) and (np.diff(st["idx"]) >= 0).all()
    assert np.array_equal(np.bincount(st["idx"], minlength=len(ids)), r["pred_dur"])
    assert st["F0"].shape == (2 * T,) and st["har"].shape == (120 * T + 1, 22)
    assert st["gen.stage.0"].shape == (20 * T, 256) and st["gen.stage.1"].shape == (120 * T + 1, 128)
    assert r["audio"].shape == (600 * T,) and np.isfinite(r["audio"]).all()
    # speed divides the duration sum (A.1)
    r2 = oracle.forward(ids, style, 2.0, noise_seed=1, stages=True)
    np.testing.assert_allclose(r2["stages"]["dur_float"], st["dur_float"] / 2.0, rtol=1e-6)


def test_rand_ini_is_a_noop_in_the_source(oracle):
    # SURVEY A.9: the random initial phase is added at time index 0 only and the x1/300 linear
    # down-sampling never reads index 0
    import torch.nn.functional as F
    f0 = torch.rand(1, 2400, 9) * 0.05
    a = F.interpolate(f0.transpose(1, 2), scale_factor=1 / 300, mode="linear")
    f0b = f0.clone()
    f0b[:, 0, :] += torch.rand(1, 9)
    b = F.interpolate(f0b.transpose(1, 2), scale_factor=1 / 300, mode="linear")
    assert torch.equal(a, b)
