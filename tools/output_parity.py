"""Digest of everything the output stage returns, over a fixed, seeded matrix, for comparing two builds bit for bit:

  * encodings f32, pcm16, ulaw, alaw, flac, mp3;  out_rate 24000, 16000, 44100;
  * processing: plain, loudness -16 LUFS, limiter at -14 LUFS, report (measure only), report + limiter;
  * layout: per item (infer_batch*) and as programs [0, 2, 5, 6] (infer_programs*);
  * a batch of 6 items (item 0 under 400 ms, item 2 over 3 s, by teacher-forced durations) in frame groups of at
    most 300 frames, so that programs span groups;
  * one f32 infer_batch split into two "max_tokens" passes, and one stage / run_staged / fetch_staged.

Per case: sha256 of every output's bytes and its length (the offsets), the durations where the call returns them, the
three reports (or the error code), "loudness_items", "limiter_items", "launches", and the kernel names with their
launch counts from a profiled repeat of the call.

    python tools/output_parity.py --out FILE
"""
import argparse
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kokorox_b200.synth import ensure_weights, synth_case  # noqa: E402

ENCODINGS = ("f32", "pcm16", "ulaw", "alaw", "flac", "mp3")
RATES = (24000, 16000, 44100)
PROCESSING = {
    "plain": {},
    "loudness": {"loudness_target": -1600},
    "limiter": {"loudness_target": -1400, "limiter": 1},
    "report": {"loudness_report": 1},
    "report_limiter": {"loudness_target": -1400, "limiter": 1, "loudness_report": 1},
}
DEFAULTS = {"loudness_target": 0, "limiter": 0, "loudness_report": 0, "out_rate": 24000, "max_frames": 49152,
            "max_tokens": 40960}
PROGRAMS = [0, 2, 5, 6]
LENS = (6, 140, 260, 61, 190, 90)


def digest(outs):
    return [[len(bytes(o)) if isinstance(o, bytes) else int(o.nbytes),
             hashlib.sha256(o if isinstance(o, bytes) else np.ascontiguousarray(o).tobytes()).hexdigest()]
            for o in outs]


def floats(a):
    return [None if np.isnan(x) else float(x) for x in np.asarray(a, np.float32).reshape(-1)]


def reports(m, KkxError):
    out = {}
    for name, fn in (("loudness", m.last_loudness), ("limiter", m.last_limiter),
                     ("loudness_range", m.last_loudness_range)):
        try:
            out[name] = [floats(c) for c in fn()]
        except KkxError as e:
            out[name] = "error: " + str(e)
    for k in ("loudness_items", "limiter_items", "launches", "frame_groups"):
        out[k] = m.get_stat(k)
    return out


def call(m, enc, layout, toks, styles, speeds):
    """Outputs and durations (None where the entry point returns none) of one case."""
    if layout == "programs":
        if enc == "mp3":
            return m.infer_programs_mp3(toks, styles, speeds, PROGRAMS, return_durations=True)
        outs, dur = m.infer_programs(toks, styles, speeds, PROGRAMS, encoding=enc, return_durations=True)
        return [o if isinstance(o, bytes) else o.copy() for o in outs], dur
    if enc == "f32":
        outs, dur = m.infer_batch(toks, styles, speeds, return_durations=True)
    elif enc == "pcm16":
        outs, dur = m.infer_batch_pcm16(toks, styles, speeds), None
    elif enc in ("ulaw", "alaw"):
        outs, dur = m.infer_batch_g711(toks, styles, speeds, law=enc, return_durations=True)
    elif enc == "flac":
        outs, dur = m.infer_batch_flac(toks, styles, speeds, return_durations=True)
    else:
        outs, dur = m.infer_batch_mp3(toks, styles, speeds, return_durations=True)
    return [o if isinstance(o, bytes) else o.copy() for o in outs], dur


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    from kokorox_b200.onn import B200Koko, KkxError, init_ort
    init_ort()
    cases = [synth_case(n, 7100 + i, 7200 + i) for i, n in enumerate(LENS)]
    toks, styles = [c[0] for c in cases], [c[1] for c in cases]
    speeds = [1.0, 1.25, 0.85, 1.1, 0.95, 1.2]
    m = B200Koko.new(ensure_weights())

    def opts(**kw):
        for k, v in {**DEFAULTS, **kw}.items():
            m.set_option(k, v)

    def inject(on):
        m.set_inject("pred_dur", np.ones(len(toks[0]), np.int32) if on else None, 0)
        m.set_inject("pred_dur", np.full(len(toks[2]), 2, np.int32) if on else None, 2)

    res = {}
    inject(True)
    for rate in RATES:
        for proc, kw in PROCESSING.items():
            for enc in ENCODINGS:
                for layout in ("per_item", "programs"):
                    opts(out_rate=rate, max_frames=300, **kw)
                    outs, dur = call(m, enc, layout, toks, styles, speeds)
                    r = {"outputs": digest(outs), "pred_dur": None if dur is None else [d.tolist() for d in dur]}
                    r.update(reports(m, KkxError))
                    m.profile_enable(True)
                    call(m, enc, layout, toks, styles, speeds)
                    r["profile_kernels"] = {k: v[0] for k, v in sorted(m.profile()["kernels"].items())}
                    r["profile_launches"] = m.get_stat("launches")
                    m.profile_enable(False)
                    res[f"{rate}/{proc}/{enc}/{layout}"] = r
    inject(False)
    opts(max_tokens=512, loudness_report=1)
    outs, dur = m.infer_batch(toks, styles, speeds, return_durations=True)
    r = {"outputs": digest([o.copy() for o in outs]), "pred_dur": [d.tolist() for d in dur]}
    r.update(reports(m, KkxError))
    res["max_tokens_512"] = r
    opts()
    m.stage(toks, styles, speeds)
    n, launches = m.run_staged()
    audio, soff, dur = m.fetch_staged(n)
    res["run_staged"] = {"outputs": digest([audio]), "sample_offsets": soff.tolist(), "pred_dur": dur.tolist(),
                         "launches": launches}
    m.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
    print(f"{len(res)} cases -> {a.out}")


if __name__ == "__main__":
    main()
