"""bench.py --dump-outputs: what the benchmark's timed path computed, written for comparison between two builds."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
from tests.conftest import ROOT


def test_dump_arrays_whole_and_sampled(monkeypatch):
    rng = np.random.default_rng(3)
    audio = rng.standard_normal(50_000).astype(np.float32)
    soff = np.array([0, 20_000, 50_000], np.int64)
    dur = rng.integers(1, 9, 40).astype(np.int32)

    whole = bench.dump_arrays(audio, soff, dur)
    assert set(whole) == {"audio", "sample_offsets", "durations"}
    assert whole["audio"].dtype == np.float32 and np.array_equal(whole["audio"], audio)
    assert whole["sample_offsets"].dtype == np.float64 and np.array_equal(whole["sample_offsets"], soff)
    assert whole["durations"].dtype == np.float64 and np.array_equal(whole["durations"], dur)

    monkeypatch.setattr(bench, "DUMP_BYTES", 4096 + 100_000)
    a = bench.dump_arrays(audio, soff, dur)
    b = bench.dump_arrays(audio.copy(), soff, dur)
    assert sum(x.nbytes for x in a.values()) <= 100_000
    idx = a["audio_index"]
    assert idx.dtype == np.float64 and np.array_equal(idx, b["audio_index"])      # seeded: the same positions
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < audio.size
    assert a["audio"].dtype == np.float32 and np.array_equal(a["audio"], audio[idx.astype(np.int64)])
    assert idx.size > 5000                                                           # the budget is used


@pytest.mark.gpu
def test_dump_outputs_are_what_the_caller_receives(tmp_path, weights_path):
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "2", "--batch", "3", "--tokens",
                        "40", "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["warmup"] == 1
    got = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(got) == {"audio", "sample_offsets", "durations"}
    assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= 64_000_000

    from kokorox_b200.onn import B200Koko, init_ort
    from kokorox_b200.synth import synth_batch
    init_ort()
    m = B200Koko.new(weights_path)
    try:
        m.set_option("precision", 1)
        toks, styles, speeds = synth_batch(3, 40, 0)
        outs, durs = m.infer_batch(toks, styles, speeds, return_durations=True)
        assert np.array_equal(got["sample_offsets"], np.cumsum([0] + [len(o) for o in outs]))
        assert np.array_equal(got["durations"], np.concatenate(durs))
        assert np.array_equal(got["audio"], np.concatenate(outs))
    finally:
        m.close()
