"""Cost of MP3 output (kkx_infer_batch_mp3 / kkx_infer_programs_mp3): the benchmark's B = 64 x 510 batch as

  * mp3_24k_160   MP3 at 24 kHz, 160 kbps (MPEG-2 LSF, the model's own rate)
  * mp3_48k_192   MP3 at 48 kHz, 192 kbps (MPEG-1, the reference's LAME bitrate)

in two layouts, per_item (infer_batch_mp3) and programs8x8 (8 programs of 8 items, infer_programs_mp3), against PCM16
and FLAC at the same rate in the same call.  Cases alternate over --rounds rounds so that drift on a shared host hits
all of them alike.  Per case: wall time per step through the binding (every call ends in a device synchronise, the
result in host memory), the forward pass's device time per step ("gpu_us"; the encoders run after it and are not
included), and, from one profiled step of its own, the encoder kernels' device time and the launch count.

    python tools/mp3_e2e.py [--batch 64] [--tokens 510] [--steps 10] [--warmup 3] [--rounds 2] [--out FILE]
The random-init checkpoint's audio is not speech: nothing about MP3 quality follows from it.
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

RATES = ((24000, 160), (48000, 192))
ENCODER_KERNELS = ("mp3_encode", "flac_analyze", "flac_scan", "flac_pack")


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
    poffs = list(range(0, a.batch + 1, a.batch // 8))
    m = B200Koko.new(ensure_weights())
    calls = {
        "pcm16": lambda kb: m.infer_batch_pcm16(toks, styles, speeds),
        "flac": lambda kb: m.infer_batch_flac(toks, styles, speeds),
        "mp3_per_item": lambda kb: m.infer_batch_mp3(toks, styles, speeds, kbps=kb),
        "mp3_programs8x8": lambda kb: m.infer_programs_mp3(toks, styles, speeds, poffs, kbps=kb),
    }
    res = {f"{r // 1000}k_{kb}": {c: {"wall_ms_per_step": [], "gpu_ms_per_step": []} for c in calls} for r, kb in RATES}
    for _ in range(a.rounds):
        for rate, kb in RATES:
            m.set_option("out_rate", rate)
            for c, fn in calls.items():
                for _ in range(a.warmup):
                    fn(kb)
                gpu = []
                t0 = time.perf_counter()
                for _ in range(a.steps):
                    outs = fn(kb)
                    gpu.append(m.get_stat("gpu_us") / 1e3)
                wall = (time.perf_counter() - t0) / a.steps
                r = res[f"{rate // 1000}k_{kb}"][c]
                r["wall_ms_per_step"].append(round(wall * 1e3, 3))
                r["gpu_ms_per_step"].append(round(float(np.mean(gpu)), 3))
                r["bytes_per_step"] = int(sum(len(o) if isinstance(o, bytes) else o.nbytes for o in outs))
                del outs
    for rate, kb in RATES:   # one profiled step per case, in a run of its own
        m.set_option("out_rate", rate)
        for c, fn in calls.items():
            m.profile_enable(True)
            fn(kb)
            p = m.profile()
            m.profile_enable(False)
            kern = p["kernels"]
            res[f"{rate // 1000}k_{kb}"][c]["profile"] = {
                "encoder_kernels_launches_ms": {k: [kern[k][0], round(kern[k][1] / 1e3, 4)]
                                                for k in ENCODER_KERNELS if k in kern},
                "all_kernels_ms": round(sum(v[1] for v in kern.values()) / 1e3, 3),
                "launches": m.get_stat("launches")}
    m.set_option("out_rate", 24000)
    out = {"gpu": gpu_info(), "batch": a.batch, "tokens": a.tokens, "steps": a.steps, "warmup": a.warmup,
           "rounds": a.rounds, "cases": res,
           "note": "random-init checkpoint: the audio is not speech, so MP3 quality and FLAC sizes say nothing about "
                   "real-model speech; MP3 sizes are fixed by the bitrate"}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    m.close()


if __name__ == "__main__":
    main()
