"""Cost of the lookahead true-peak limiter ("limiter"): the benchmark's B = 64 x 510 batch as 16-bit PCM at 24 kHz,
normalised to -14 LUFS, with the limiter off and on.  Both settings alternate over --rounds rounds (warm-up, then a
timed loop of infer_batch_pcm16 calls, each ending in a device synchronise with the result in host memory), so that
drift on a shared host hits both alike.  Afterwards one profiled step per setting (kkx_profile_enable: a CUDA event
after every launch, a run of its own since the events slow the host) gives the device time of the post-processing
kernels -- loudness, limiter, the resampling pass-through that applies the gain -- and of the whole step.

    python tools/limiter_e2e.py [--batch 64] [--tokens 510] [--steps 10] [--warmup 3] [--rounds 3] [--out FILE]
Prints one JSON object with the card's name, power limit and top SM clock, read in the same run.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kokorox_b200.synth import ensure_weights, synth_batch  # noqa: E402

POST_KERNELS = ("loud_energy", "loud_peak", "loud_gain", "lim_envelope", "lim_trim", "resample")


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--tokens", type=int, default=510)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    from kokorox_b200.onn import B200Koko, init_ort
    init_ort()
    toks, styles, speeds = synth_batch(a.batch, a.tokens, 0)
    m = B200Koko.new(ensure_weights())
    m.set_option("loudness_target", -1400)
    res = {s: {"wall_ms_per_step": []} for s in ("off", "on")}
    for _ in range(a.rounds):
        for s in ("off", "on"):
            m.set_option("limiter", 1 if s == "on" else 0)
            outs = None
            for _ in range(a.warmup):      # the previous result stays alive during the next call, as in bench.py
                outs = m.infer_batch_pcm16(toks, styles, speeds)
            t0 = time.perf_counter()
            for _ in range(a.steps):
                outs = m.infer_batch_pcm16(toks, styles, speeds)
            res[s]["wall_ms_per_step"].append(round((time.perf_counter() - t0) / a.steps * 1e3, 3))
            res[s]["samples_per_step"] = sum(len(o) for o in outs)
            res[s]["pcm16_peak"] = int(max(np.abs(o.astype(np.int32)).max() for o in outs))
            del outs
    for s in ("off", "on"):
        m.set_option("limiter", 1 if s == "on" else 0)
        m._lib.kkx_profile_enable(m._ctx, 1)
        m.infer_batch_pcm16(toks, styles, speeds)
        n = m._lib.kkx_profile_json(m._ctx, None, 0)
        buf = ctypes.create_string_buffer(int(n) + 1)
        m._lib.kkx_profile_json(m._ctx, buf, n + 1)
        m._lib.kkx_profile_enable(m._ctx, 0)
        kern = json.loads(buf.value.decode())["kernels"]
        post = {k: [kern[k][0], round(kern[k][1] / 1e3, 4)] for k in POST_KERNELS if k in kern}
        step_ms = sum(v[1] for v in kern.values()) / 1e3
        r = res[s]
        r["profile"] = {"step_kernels_ms": round(step_ms, 3), "post_kernels_launches_ms": post,
                        "post_total_ms": round(sum(v[1] for v in post.values()), 4),
                        "launches": m.get_stat("launches"), "frame_groups": m.get_stat("frame_groups")}
        r["best_wall_ms"] = min(r["wall_ms_per_step"])
        if s == "on":
            red, tp = m.last_limiter()
            r["max_reduction_db_range"] = [round(float(red.min()), 3), round(float(red.max()), 3)]
            r["true_peak_dbtp_max"] = round(float(tp.max()), 4)
    out = {"gpu": gpu_info(), "batch": a.batch, "tokens": a.tokens, "steps": a.steps, "warmup": a.warmup,
           "rounds": a.rounds, "encoding": "pcm16", "out_rate": 24000, "loudness_target_lufs": -14.0,
           "true_peak_max_dbtp": -1.0, "limiter": res}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    m.close()


if __name__ == "__main__":
    main()
