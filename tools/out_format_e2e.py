"""End-to-end cost of the output formats: the benchmark's B = 64 x 510 batch through the public calls with host
buffers (warm-up, then a timed loop; every call ends in a device synchronise and the result in pinned host memory),
comparing

  * infer_batch        at 24 kHz, f32      (the benchmark's e2e leg)
  * infer_batch_pcm16  at 16 kHz, int16    ("out_rate" 16000)
  * infer_batch_g711   at  8 kHz, mu-law   ("out_rate" 8000)
  * infer_batch_flac   at 24 kHz, FLAC     (lossless, encoded on the device)
  * infer_batch_pcm16  at 24 kHz, int16, without and with loudness normalisation ("loudness_target" -1600)

One session switches "out_rate" before each format's warm-up (a server would hold one session per rate; those share the
device weights), and the formats alternate over --rounds rounds so that drift on a shared host hits all of them alike.

    python tools/out_format_e2e.py [--batch 64] [--tokens 510] [--steps 10] [--warmup 3] [--rounds 2] [--out FILE]
Prints one JSON object: per format the wall time per step (every round), audio seconds per step, audio-s/s and the
device-to-host bytes per step (waveform payload + the per-token durations the call also returns; for FLAC also the
per-item byte offsets, and the payload's bytes per sample against 16-bit PCM).  After the timed rounds, one more
FLAC step runs with kkx_profile_enable (a run of its own, since the per-launch events slow the host) and
"flac_profile" gives the encoder kernels' device time in that step; a profiled normalised PCM16 step at 24 kHz gives
"loudness_profile", the device time of the loudness kernels and of the resampling pass-through that applies the gain.  The compression of the random-init
checkpoint's audio says nothing about the ratio on real-model speech.
"""
import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kokorox_b200.synth import ensure_weights, synth_batch  # noqa: E402

FORMATS = (   # name, out_rate, bytes per sample, per-token durations fetched by the binding, loudness_target
    ("f32_24k", 24000, 4, True, 0),
    ("pcm16_16k", 16000, 2, False, 0),
    ("g711_ulaw_8k", 8000, 1, True, 0),
    ("flac_24k", 24000, None, True, 0),   # variable: the files' byte count
    ("pcm16_24k", 24000, 2, False, 0),
    ("pcm16_24k_lufs16", 24000, 2, False, -1600),
)
FLAC_KERNELS = ("flac_analyze", "flac_scan", "flac_pack")
LOUD_KERNELS = ("loud_energy", "loud_peak", "loud_gain", "resample")


def flac_samples(data: bytes) -> int:
    return int.from_bytes(data[18:26], "big") & ((1 << 36) - 1)   # STREAMINFO total samples


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
    from kokorox_b200.onn import B200Koko, init_ort
    init_ort()
    wp = ensure_weights()
    toks, styles, speeds = synth_batch(a.batch, a.tokens, 0)
    sum_n = sum(len(t) for t in toks)
    m = B200Koko.new(wp)

    def call(name):
        if name.startswith("f32"):
            return m.infer_batch(toks, styles, speeds)
        if name.startswith("pcm16"):
            return m.infer_batch_pcm16(toks, styles, speeds)
        if name.startswith("flac"):
            return m.infer_batch_flac(toks, styles, speeds)
        return m.infer_batch_g711(toks, styles, speeds, law="ulaw")

    res = {name: {"out_rate": rate, "loudness_target": lt, "wall_ms_per_step": []} for name, rate, _, _, lt in FORMATS}
    for _ in range(a.rounds):
        for name, rate, bps, with_dur, lt in FORMATS:
            m.set_option("out_rate", rate)
            m.set_option("loudness_target", lt)
            outs = None
            for _ in range(a.warmup):      # the previous result stays alive during the next call, as in bench.py
                outs = call(name)
            t0 = time.perf_counter()
            for _ in range(a.steps):
                outs = call(name)
            wall = (time.perf_counter() - t0) / a.steps
            r = res[name]
            if bps is None:
                n = sum(flac_samples(o) for o in outs)
                payload = sum(len(o) for o in outs)
                r["payload_bytes_per_step"] = payload
                r["bytes_per_sample"] = round(payload / n, 4)
                r["of_pcm16"] = round(payload / (2 * n), 4)
                payload += 8 * (a.batch + 1)
            else:
                n = sum(len(o) for o in outs)
                payload = n * bps
            del outs
            r["wall_ms_per_step"].append(round(wall * 1e3, 3))
            r["samples_per_step"] = n
            r["audio_s_per_step"] = n / rate
            r["d2h_bytes_per_step"] = payload + (sum_n * 4 if with_dur else 0)
    for name, *_ in FORMATS:
        r = res[name]
        best = min(r["wall_ms_per_step"])
        r["audio_s_per_s_best"] = round(r["audio_s_per_step"] / (best / 1e3), 1)
    def profiled(name):   # one step with per-kernel device time (an event after every launch)
        m._lib.kkx_profile_enable(m._ctx, 1)
        call(name)
        nbuf = m._lib.kkx_profile_json(m._ctx, None, 0)
        buf = ctypes.create_string_buffer(int(nbuf) + 1)
        m._lib.kkx_profile_json(m._ctx, buf, nbuf + 1)
        m._lib.kkx_profile_enable(m._ctx, 0)
        return json.loads(buf.value.decode())

    # one profiled FLAC step: the run and the encoder
    m.set_option("out_rate", 24000)
    m.set_option("loudness_target", 0)
    prof = profiled("flac")
    kern = prof["kernels"]
    enc_ms = {k: round(kern[k][1] / 1e3, 4) for k in FLAC_KERNELS}
    step_ms = sum(v[1] for v in kern.values()) / 1e3
    flac_profile = {"run_gpu_ms": round(prof["gpu_us"] / 1e3, 3), "step_kernels_ms": round(step_ms, 3),
                    "encoder_ms": enc_ms, "encoder_total_ms": round(sum(enc_ms.values()), 4),
                    "encoder_share_of_step": round(sum(enc_ms.values()) / step_ms, 5),
                    "launches": m.get_stat("launches")}
    # one profiled normalised PCM16 step at 24 kHz: the loudness kernels and the pass-through that applies the gain
    m.set_option("loudness_target", -1600)
    prof = profiled("pcm16")
    kern = prof["kernels"]
    loud_ms = {k: [kern[k][0], round(kern[k][1] / 1e3, 4)] for k in LOUD_KERNELS if k in kern}
    step_ms = sum(v[1] for v in kern.values()) / 1e3
    loud_total = sum(v[1] for v in loud_ms.values())
    lufs, tp, gain = m.last_loudness()
    loudness_profile = {"run_gpu_ms": round(prof["gpu_us"] / 1e3, 3), "step_kernels_ms": round(step_ms, 3),
                        "kernels_launches_ms": loud_ms, "total_ms": round(loud_total, 4),
                        "share_of_step": round(loud_total / step_ms, 5), "launches": m.get_stat("launches"),
                        "frame_groups": m.get_stat("frame_groups"),
                        "lufs_range": [float(min(lufs)), float(max(lufs))],
                        "gain_db_range": [round(20 * math.log10(float(min(gain))), 3),
                                          round(20 * math.log10(float(max(gain))), 3)]}
    m.set_option("loudness_target", 0)
    out = {"gpu": gpu_info(), "batch": a.batch, "tokens": a.tokens, "steps": a.steps, "warmup": a.warmup,
           "rounds": a.rounds, "formats": res, "flac_profile": flac_profile, "loudness_profile": loudness_profile,
           "note": "FLAC sizes are those of the random-init checkpoint's audio; they say nothing about the "
                   "compression ratio of real-model speech"}
    print(json.dumps(out, indent=1))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)
    m.close()


if __name__ == "__main__":
    main()
