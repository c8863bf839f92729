"""Cost and size of FLAC linear prediction ("flac_lpc_order"): the benchmark's B = 64 x 510 batch as FLAC
(kkx_infer_batch_flac) at 24 kHz and 48 kHz with the LPC order p = 0 (off), 8 and 12, beside PCM16 at the same rate.
Cases alternate over --rounds rounds so that drift on a shared host hits all of them alike.  Per case: wall time per
step through the binding (every call ends in a device synchronise, the result in host memory), the forward pass's
device time per step ("gpu_us"; the encoder runs after it and is not included), the bytes per step and their ratio to
PCM16, and, from one profiled step of its own, the encoder kernels' device time (with p > 0, flac_analyze is its LPC
variant: the predictor design runs inside it) and the launch count.

    python tools/flac_lpc_e2e.py [--batch 64] [--tokens 510] [--steps 5] [--warmup 2] [--rounds 2] [--out FILE]
The random-init checkpoint's audio is not speech: the sizes say nothing about the compression of real-model speech.
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

RATES = (24000, 48000)
ORDERS = (0, 8, 12)
ENCODER_KERNELS = ("flac_analyze", "flac_scan", "flac_pack")


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
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    from kokorox_b200.onn import B200Koko, init_ort
    init_ort()
    toks, styles, speeds = synth_batch(a.batch, a.tokens, 0)
    m = B200Koko.new(ensure_weights())
    cases = {"pcm16": None, **{f"flac_p{p}": p for p in ORDERS}}

    def call(p):
        if p is None:
            return m.infer_batch_pcm16(toks, styles, speeds)
        m.set_option("flac_lpc_order", p)
        return m.infer_batch_flac(toks, styles, speeds)

    res = {f"{r // 1000}k": {c: {"wall_ms_per_step": [], "gpu_ms_per_step": []} for c in cases} for r in RATES}
    for _ in range(a.rounds):
        for rate in RATES:
            m.set_option("out_rate", rate)
            for c, p in cases.items():
                for _ in range(a.warmup):
                    call(p)
                gpu = []
                t0 = time.perf_counter()
                for _ in range(a.steps):
                    outs = call(p)
                    gpu.append(m.get_stat("gpu_us") / 1e3)
                wall = (time.perf_counter() - t0) / a.steps
                r = res[f"{rate // 1000}k"][c]
                r["wall_ms_per_step"].append(round(wall * 1e3, 3))
                r["gpu_ms_per_step"].append(round(float(np.mean(gpu)), 3))
                r["bytes_per_step"] = int(sum(len(o) if isinstance(o, bytes) else o.nbytes for o in outs))
                del outs
    for rate in RATES:   # one profiled step per case, in a run of its own
        m.set_option("out_rate", rate)
        for c, p in cases.items():
            m.profile_enable(True)
            call(p)
            prof = m.profile()
            m.profile_enable(False)
            kern = prof["kernels"]
            r = res[f"{rate // 1000}k"][c]
            r["profile"] = {"encoder_kernels_launches_ms": {k: [kern[k][0], round(kern[k][1] / 1e3, 4)]
                                                            for k in ENCODER_KERNELS if k in kern},
                            "launches": m.get_stat("launches")}
        pcm = res[f"{rate // 1000}k"]["pcm16"]["bytes_per_step"]
        for c in cases:
            r = res[f"{rate // 1000}k"][c]
            r["bytes_vs_pcm16"] = round(r["bytes_per_step"] / pcm, 4)
    m.set_option("flac_lpc_order", 0)
    m.set_option("out_rate", 24000)
    out = {"gpu": gpu_info(), "batch": a.batch, "tokens": a.tokens, "steps": a.steps, "warmup": a.warmup,
           "rounds": a.rounds, "cases": res,
           "note": "random-init checkpoint: the audio is not speech, so the FLAC sizes say nothing about the "
                   "compression of real-model speech"}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    m.close()


if __name__ == "__main__":
    main()
