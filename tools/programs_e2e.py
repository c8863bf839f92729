"""Cost of programs (kkx_infer_programs): the benchmark's B = 64 x 510 batch through infer_programs in two layouts,

  * per_item    64 programs of one item (what the per-item entry points compute)
  * programs8x8  8 programs of 8 consecutive items (one output per request of 8 chunks)

for two output configurations,

  * flac_24k          FLAC at 24 kHz, loudness off
  * pcm16_16k_lufs16  PCM16 at 16 kHz with "loudness_target" -1600 (loudness and resampling over whole programs)

Layouts and configurations alternate over --rounds rounds so that drift on a shared host hits all of them alike.  Per
case: the wall time per step through the binding (every call ends in a device synchronise, the result in host memory),
the forward pass's device time per step ("gpu_us", CUDA events; the FLAC encoder runs after it and is not included),
and, from one profiled step of its own (kkx_profile_enable), the per-kernel device time of "resample", "loud_*" and
"flac_*", the sum of all kernels, the launch count and the frame-group count.

    python tools/programs_e2e.py [--batch 64] [--tokens 510] [--steps 10] [--warmup 3] [--rounds 2] [--out FILE]
The random-init checkpoint's audio is not speech: nothing about FLAC sizes follows from it.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kokorox_b200.synth import ensure_weights, synth_batch  # noqa: E402

CONFIGS = (   # name, encoding, out_rate, loudness_target
    ("flac_24k", "flac", 24000, 0),
    ("pcm16_16k_lufs16", "pcm16", 16000, -1600),
)
POST_KERNELS = ("resample", "loud_energy", "loud_peak", "loud_gain", "flac_analyze", "flac_scan", "flac_pack")


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
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if a.batch % 8:
        raise SystemExit("--batch must be a multiple of 8 (8 programs of batch / 8 items)")
    from kokorox_b200.onn import B200Koko, init_ort
    init_ort()
    toks, styles, speeds = synth_batch(a.batch, a.tokens, 0)
    layouts = {"per_item": list(range(a.batch + 1)), "programs8x8": list(range(0, a.batch + 1, a.batch // 8))}
    m = B200Koko.new(ensure_weights())

    def setup(rate, lt):
        m.set_option("out_rate", rate)
        m.set_option("loudness_target", lt)

    res = {c[0]: {lay: {"wall_ms_per_step": [], "gpu_ms_per_step": []} for lay in layouts} for c in CONFIGS}
    for _ in range(a.rounds):
        for name, enc, rate, lt in CONFIGS:
            for lay, poffs in layouts.items():
                setup(rate, lt)
                for _ in range(a.warmup):
                    outs = m.infer_programs(toks, styles, speeds, poffs, encoding=enc)
                gpu = []
                t0 = time.perf_counter()
                for _ in range(a.steps):
                    outs = m.infer_programs(toks, styles, speeds, poffs, encoding=enc)
                    gpu.append(m.get_stat("gpu_us") / 1e3)
                wall = (time.perf_counter() - t0) / a.steps
                r = res[name][lay]
                r["wall_ms_per_step"].append(round(wall * 1e3, 3))
                r["gpu_ms_per_step"].append(round(float(np.mean(gpu)), 3))
                r["outputs"] = len(outs)
                r["bytes_per_step"] = int(sum(len(o) if enc == "flac" else o.nbytes for o in outs))
                del outs
    for name, enc, rate, lt in CONFIGS:   # one profiled step per case, in a run of its own
        for lay, poffs in layouts.items():
            setup(rate, lt)
            m.profile_enable(True)
            m.infer_programs(toks, styles, speeds, poffs, encoding=enc)
            p = m.profile()
            m.profile_enable(False)
            kern = p["kernels"]
            r = res[name][lay]
            r["profile"] = {"kernels_launches_ms": {k: [kern[k][0], round(kern[k][1] / 1e3, 4)]
                                                    for k in POST_KERNELS if k in kern},
                            "post_total_ms": round(sum(kern[k][1] for k in POST_KERNELS if k in kern) / 1e3, 4),
                            "all_kernels_ms": round(sum(v[1] for v in kern.values()) / 1e3, 3),
                            "launches": m.get_stat("launches"), "frame_groups": m.get_stat("frame_groups")}
    setup(24000, 0)
    out = {"gpu": gpu_info(), "batch": a.batch, "tokens": a.tokens, "steps": a.steps, "warmup": a.warmup,
           "rounds": a.rounds, "cases": res,
           "note": "random-init checkpoint: the audio is not speech, so FLAC sizes say nothing about real-model speech"}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    m.close()


if __name__ == "__main__":
    main()
