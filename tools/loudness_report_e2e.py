"""Cost of the EBU R128 loudness report ("loudness_report"): the benchmark's B = 64 x 510 batch as 16-bit PCM at
24 kHz in three settings -- report off (plain output), report on with "loudness_target" 0 (measure-only) and report on
with a -16 LUFS target.  The settings alternate over --rounds rounds (warm-up, then a timed loop of
infer_batch_pcm16 calls, each ending in a device synchronise with the result in host memory), so that drift on a
shared host hits all alike.  Afterwards one profiled step per setting (kkx_profile_enable: a CUDA event after every
launch, a run of its own since the events slow the host) gives the device time of loud_short and loud_range, of all
the post-processing kernels (loudness, report, the resampling pass-through) and of the whole step.

    python tools/loudness_report_e2e.py [--batch 64] [--tokens 510] [--steps 10] [--warmup 3] [--rounds 3] [--out FILE]
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

POST_KERNELS = ("loud_energy", "loud_peak", "loud_gain", "loud_short", "loud_range", "resample")
# setting -> (loudness_report, loudness_target in 1/100 LUFS)
SETTINGS = {"off": (0, 0), "measure_only": (1, 0), "report_target_-16": (1, -1600)}


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

    def use(s):
        rep, target = SETTINGS[s]
        m.set_option("loudness_report", rep)
        m.set_option("loudness_target", target)

    res = {s: {"wall_ms_per_step": []} for s in SETTINGS}
    first = {}
    for _ in range(a.rounds):
        for s in SETTINGS:
            use(s)
            outs = None
            for _ in range(a.warmup):      # the previous result stays alive during the next call, as in bench.py
                outs = m.infer_batch_pcm16(toks, styles, speeds)
            t0 = time.perf_counter()
            for _ in range(a.steps):
                outs = m.infer_batch_pcm16(toks, styles, speeds)
            res[s]["wall_ms_per_step"].append(round((time.perf_counter() - t0) / a.steps * 1e3, 3))
            res[s]["samples_per_step"] = sum(len(o) for o in outs)
            first.setdefault(s, np.concatenate(outs).copy())
            del outs
    for s in SETTINGS:
        use(s)
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
                        "report_kernels_ms": round(sum(post[k][1] for k in ("loud_short", "loud_range") if k in post), 4),
                        "launches": m.get_stat("launches"), "frame_groups": m.get_stat("frame_groups")}
        w = r["wall_ms_per_step"]
        r["best_wall_ms"] = min(w)
        r["wall_spread_ms"] = round(max(w) - min(w), 3)
        if SETTINGS[s][0]:
            lra, mm, sm = m.last_loudness_range()
            L, tp, g = m.last_loudness()
            r["lra_lu_range"] = [round(float(np.nanmin(lra)), 3), round(float(np.nanmax(lra)), 3)]
            r["max_momentary_lufs_range"] = [round(float(mm.min()), 3), round(float(mm.max()), 3)]
            r["max_short_term_lufs_range"] = [round(float(sm.min()), 3), round(float(sm.max()), 3)]
            r["gain_range"] = [float(g.min()), float(g.max())]
    out = {"gpu": gpu_info(), "batch": a.batch, "tokens": a.tokens, "steps": a.steps, "warmup": a.warmup,
           "rounds": a.rounds, "encoding": "pcm16", "out_rate": 24000, "settings": SETTINGS,
           "measure_only_output_equals_off": bool(np.array_equal(first["off"], first["measure_only"])),
           "measure_only_post_cost_ms": res["measure_only"]["profile"]["post_total_ms"]
           - res["off"]["profile"]["post_total_ms"],
           "report": res}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    m.close()


if __name__ == "__main__":
    main()
