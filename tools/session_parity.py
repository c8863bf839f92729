"""Digest of the session-level behaviour of the C boundary that tools/output_parity.py does not reach, for comparing
two builds bit for bit:

  * kkx_infer (one utterance) and kkx_infer_batch_voices (voice table mixed on the device);
  * coalesced callers ("coalesce" > 1): one output digest per caller, the views released in an order different from
    the one they were returned in, one view read after the others have gone back;
  * kkx_submit / kkx_wait / kkx_poll, a wait that releases the result itself, an unknown and a redeemed ticket;
  * release / re-acquire cycles: whether the next result reuses the buffer that came back;
  * the three report accessors after each synchronous path and after coalesced / asynchronous calls;
  * return code and message of bad arguments (one and two at a time) to the six encoded entry points,
    kkx_set_option and the value-returning accessors, and the staged batch and report after them.

    python tools/session_parity.py --out FILE
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import threading

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from kokorox_b200.synth import ensure_weights, synth_case, synth_voice_table  # noqa: E402

LENS = (40, 120, 75, 200)
P = C.POINTER


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def floats(a):
    return [None if np.isnan(x) else float(x) for x in np.asarray(a, np.float32).reshape(-1)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    a = ap.parse_args()
    from kokorox_b200.onn import B200Koko, KkxError, init_ort
    init_ort()
    cases = [synth_case(n, 8100 + i, 8200 + i) for i, n in enumerate(LENS)]
    toks, styles = [c[0] for c in cases], [c[1] for c in cases]
    speeds = [1.0, 1.2, 0.9, 1.05]
    m = B200Koko.new(ensure_weights())
    lib, ctx = m._lib, m._ctx
    res = {}

    def err():
        return (lib.kkx_last_error(ctx) or b"").decode()

    def reports():
        out = {}
        for name, fn in (("loudness", m.last_loudness), ("limiter", m.last_limiter),
                         ("loudness_range", m.last_loudness_range)):
            try:
                out[name] = [floats(c) for c in fn()]
            except KkxError as e:
                out[name] = "error: " + str(e)
        for k in ("loudness_items", "limiter_items"):
            out[k] = m.get_stat(k)
        return out

    m.set_option("loudness_report", 1)
    m.set_option("loudness_target", -1800)
    m.set_option("limiter", 1)
    res["reports_before_any_call"] = reports()

    # kkx_infer without coalescing
    audio, dur = m.infer_one(toks[1], styles[1], speeds[1], return_durations=True)
    res["infer"] = {"audio": sha(audio), "n": int(audio.size), "pred_dur": dur.tolist(), "reports": reports()}

    # kkx_infer_batch_voices
    table = synth_voice_table(3)
    m.load_voices({"v0": table[0], "v1": table[1], "v2": table[2]})
    outs, durs = m.infer_batch_voices(toks, ["v0", "v1.6+v2.4", "v2", "v0.3+v1.7"], speeds, return_durations=True)
    res["voices"] = {"audio": [sha(o) for o in outs], "n": [int(o.size) for o in outs],
                     "pred_dur": [d.tolist() for d in durs], "reports": reports()}

    # f32 batch in two "max_tokens" passes, then the report of a batch after it
    m.set_option("max_tokens", 512)
    outs = m.infer_batch(toks + toks, styles + styles, speeds + speeds)
    res["batch_max_tokens"] = {"audio": [sha(o) for o in outs], "reports": reports()}
    m.set_option("max_tokens", 40960)

    # raw kkx_infer for the coalesced callers, so that the views can be released in a chosen order
    def raw_infer(i, slot):
        tk = np.ascontiguousarray(toks[i], np.int64)
        st = np.ascontiguousarray(styles[i], np.float32)
        ptr, ns = P(C.c_float)(), C.c_int64(0)
        dur = np.zeros(tk.size, np.int32)
        rc = lib.kkx_infer(ctx, tk.ctypes.data_as(P(C.c_int64)), int(tk.size), st.ctypes.data_as(P(C.c_float)),
                           C.c_float(speeds[i]), C.byref(ptr), C.byref(ns), dur.ctypes.data_as(P(C.c_int32)))
        slot[i] = (rc, ptr, ns.value, dur)

    def view(ptr, n):
        return np.ctypeslib.as_array(ptr, shape=(n,)).copy()

    m.set_option("coalesce", len(LENS))
    m.set_option("coalesce_wait_us", 500000)
    r0 = m.get_stat("coalesced_requests")
    slot = {}
    th = [threading.Thread(target=raw_infer, args=(i, slot)) for i in range(len(LENS))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    coal = {"rc": [slot[i][0] for i in range(len(LENS))],
            "audio": [sha(view(slot[i][1], slot[i][2])) for i in range(len(LENS))],
            "pred_dur": [slot[i][3].tolist() for i in range(len(LENS))],
            "requests": m.get_stat("coalesced_requests") - r0, "reports": reports()}
    addrs = [C.cast(slot[i][1], C.c_void_p).value for i in range(len(LENS))]
    coal["distinct_views"] = len(set(addrs)) == len(addrs)
    together = m.get_stat("coalesced_largest") == len(LENS)
    for i in (2, 0, 3):                       # all but caller 1, out of order; one released twice
        lib.kkx_release(ctx, slot[i][1])
    lib.kkx_release(ctx, slot[2][1])
    coal["last_view_intact"] = sha(view(slot[1][1], slot[1][2])) == coal["audio"][1]
    lib.kkx_release(ctx, slot[1][1])
    res["coalesced"] = coal
    # a coalesced batch's shared buffer goes back with its last view: the next batch of that size reuses it
    slot2 = {}
    th = [threading.Thread(target=raw_infer, args=(i, slot2)) for i in range(len(LENS))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    addrs2 = [C.cast(slot2[i][1], C.c_void_p).value for i in range(len(LENS))]
    res["coalesced_again"] = {"rc": [slot2[i][0] for i in range(len(LENS))],
                              "audio": [sha(view(slot2[i][1], slot2[i][2])) for i in range(len(LENS))],
                              "reuses_a_view_address": (not together) or bool(set(addrs) & set(addrs2))}
    for i in range(len(LENS)):
        lib.kkx_release(ctx, slot2[i][1])
    m.set_option("coalesce", 0)
    m.set_option("coalesce_wait_us", 0)

    # asynchronous requests
    a0 = m.get_stat("async_requests")
    tickets = [m.submit(toks[i], styles[i], speeds[i]) for i in range(len(LENS))]
    got = [m.wait(t, return_durations=True) for t in tickets]
    asy = {"audio": [sha(g[0]) for g in got], "pred_dur": [g[1].tolist() for g in got],
           "requests": m.get_stat("async_requests") - a0, "reports": reports()}
    rc = lib.kkx_poll(ctx, 987654)
    asy["poll_unknown"] = [rc, err()]
    rc = lib.kkx_wait(ctx, tickets[0], None, None, None)
    asy["wait_redeemed"] = [rc, err()]
    rc = lib.kkx_poll(ctx, tickets[1])
    asy["poll_redeemed"] = [rc, err()]
    t = m.submit(toks[0], styles[0], speeds[0])
    rc = lib.kkx_wait(ctx, t, None, None, None)           # no out_audio: the library releases the result itself
    asy["wait_without_out_audio"] = rc
    res["async"] = asy
    del got

    # release / re-acquire: a returned buffer is reused by the next result that fits
    def raw_batch(n_items):
        B = n_items
        flat = np.ascontiguousarray(np.concatenate(toks[:B]).astype(np.int64))
        offs = np.zeros(B + 1, np.int32)
        offs[1:] = np.cumsum([len(t) for t in toks[:B]])
        st = np.ascontiguousarray(np.stack(styles[:B]).astype(np.float32))
        sp = np.ascontiguousarray(speeds[:B], np.float32)
        ptr = P(C.c_float)()
        soff = np.zeros(B + 1, np.int64)
        rc = lib.kkx_infer_batch(ctx, B, flat.ctypes.data_as(P(C.c_int64)), offs.ctypes.data_as(P(C.c_int32)),
                                 st.ctypes.data_as(P(C.c_float)), sp.ctypes.data_as(P(C.c_float)), C.byref(ptr),
                                 soff.ctypes.data_as(P(C.c_int64)), None)
        return rc, ptr, int(soff[-1])

    cyc = []
    prev = None
    for n_items in (4, 4, 2, 4, 1, 1):
        rc, ptr, n = raw_batch(n_items)
        addr = C.cast(ptr, C.c_void_p).value
        cyc.append([n_items, rc, sha(view(ptr, n)), prev is not None and addr == prev])
        lib.kkx_release(ctx, ptr)
        prev = addr
    held = [raw_batch(2) for _ in range(3)]                  # three outstanding, released in reverse
    cyc.append(["held", [h[0] for h in held], len({C.cast(h[1], C.c_void_p).value for h in held})])
    for h in reversed(held):
        lib.kkx_release(ctx, h[1])
    res["release_cycles"] = cyc

    # bad arguments: stage a known batch first, so that what follows can show it is still the one staged
    m.stage(toks[:2], styles[:2], speeds[:2])
    B, flat, offs, st, sp = m._pack(toks[:2], styles[:2], speeds[:2])
    tp, op = flat.ctypes.data_as(P(C.c_int64)), offs.ctypes.data_as(P(C.c_int32))
    stp, spp = st.ctypes.data_as(P(C.c_float)), sp.ctypes.data_as(P(C.c_float))
    soff = np.zeros(B + 1, np.int64)
    boff = np.zeros(B + 1, np.int64)
    sop, bop = soff.ctypes.data_as(P(C.c_int64)), boff.ctypes.data_as(P(C.c_int64))
    good_prog = np.array([0, 2], np.int32)
    bad_prog = np.array([0, 0, 2], np.int32)
    pg, pb = good_prog.ctypes.data_as(P(C.c_int32)), bad_prog.ctypes.data_as(P(C.c_int32))
    pcm, u8, vp = P(C.c_int16)(), P(C.c_uint8)(), C.c_void_p()
    pcm_r, u8_r, vp_r = C.byref(pcm), C.byref(u8), C.byref(vp)
    bad = {}

    def call(name, fn, *args):
        rc = fn(*args)
        bad[name] = [rc, err() if rc else ""]

    f = lib.kkx_infer_batch_pcm16
    call("pcm16/out_null", f, ctx, B, tp, op, stp, spp, None, sop, None)
    call("pcm16/batch0", f, ctx, 0, tp, op, stp, spp, pcm_r, sop, None)
    call("pcm16/tokens_null", f, ctx, B, None, op, stp, spp, pcm_r, sop, None)
    call("pcm16/out_null+batch0", f, ctx, 0, tp, op, stp, spp, None, sop, None)
    call("pcm16/null_ctx", f, None, B, tp, op, stp, spp, pcm_r, sop, None)
    f = lib.kkx_infer_batch_g711
    call("g711/out_null", f, ctx, B, tp, op, stp, spp, 0, None, sop, None)
    call("g711/law2", f, ctx, B, tp, op, stp, spp, 2, u8_r, sop, None)
    call("g711/law-1", f, ctx, B, tp, op, stp, spp, -1, u8_r, sop, None)
    call("g711/batch0", f, ctx, 0, tp, op, stp, spp, 1, u8_r, sop, None)
    call("g711/law2+batch0", f, ctx, 0, tp, op, stp, spp, 2, u8_r, sop, None)
    call("g711/out_null+law2", f, ctx, B, tp, op, stp, spp, 2, None, sop, None)
    f = lib.kkx_infer_batch_flac
    call("flac/out_null", f, ctx, B, tp, op, stp, spp, None, bop, sop, None)
    call("flac/offsets_null", f, ctx, B, tp, op, stp, spp, u8_r, None, sop, None)
    call("flac/batch0", f, ctx, 0, tp, op, stp, spp, u8_r, bop, sop, None)
    call("flac/offsets_null+batch0", f, ctx, 0, tp, op, stp, spp, u8_r, None, sop, None)
    call("flac/out_null+offsets_null", f, ctx, B, tp, op, stp, spp, None, None, sop, None)
    f = lib.kkx_infer_programs
    call("programs/out_null", f, ctx, B, tp, op, stp, spp, 1, pg, 0, None, bop, sop, None)
    call("programs/offsets_null", f, ctx, B, tp, op, stp, spp, 1, pg, 0, vp_r, None, sop, None)
    for e in (5, 6, -1):
        call(f"programs/encoding{e}", f, ctx, B, tp, op, stp, spp, 1, pg, e, vp_r, bop, sop, None)
    call("programs/batch0", f, ctx, 0, tp, op, stp, spp, 1, pg, 0, vp_r, bop, sop, None)
    call("programs/n0", f, ctx, B, tp, op, stp, spp, 0, pg, 0, vp_r, bop, sop, None)
    call("programs/n3", f, ctx, B, tp, op, stp, spp, 3, pg, 0, vp_r, bop, sop, None)
    call("programs/table_null", f, ctx, B, tp, op, stp, spp, 1, None, 1, vp_r, bop, sop, None)
    call("programs/table_empty_program", f, ctx, B, tp, op, stp, spp, 2, pb, 4, vp_r, bop, sop, None)
    call("programs/encoding5+bad_table", f, ctx, B, tp, op, stp, spp, 2, pb, 5, vp_r, bop, sop, None)
    call("programs/offsets_null+encoding5", f, ctx, B, tp, op, stp, spp, 1, pg, 5, vp_r, None, sop, None)
    call("programs/batch0+bad_table", f, ctx, 0, tp, op, stp, spp, 2, pb, 0, vp_r, bop, sop, None)
    call("programs/tokens_null", f, ctx, B, None, op, stp, spp, 1, pg, 0, vp_r, bop, sop, None)
    f = lib.kkx_infer_batch_mp3
    call("mp3/out_null", f, ctx, B, tp, op, stp, spp, 0, None, bop, sop, None)
    call("mp3/offsets_null", f, ctx, B, tp, op, stp, spp, 0, u8_r, None, sop, None)
    call("mp3/kbps100", f, ctx, B, tp, op, stp, spp, 100, u8_r, bop, sop, None)
    call("mp3/kbps-8", f, ctx, B, tp, op, stp, spp, -8, u8_r, bop, sop, None)
    call("mp3/batch0", f, ctx, 0, tp, op, stp, spp, 0, u8_r, bop, sop, None)
    call("mp3/kbps100+batch0", f, ctx, 0, tp, op, stp, spp, 100, u8_r, bop, sop, None)
    call("mp3/offsets_null+kbps100", f, ctx, B, tp, op, stp, spp, 100, u8_r, None, sop, None)
    f = lib.kkx_infer_programs_mp3
    call("programs_mp3/out_null", f, ctx, B, tp, op, stp, spp, 1, pg, 0, None, bop, sop, None)
    call("programs_mp3/offsets_null", f, ctx, B, tp, op, stp, spp, 1, pg, 0, u8_r, None, sop, None)
    call("programs_mp3/kbps100", f, ctx, B, tp, op, stp, spp, 1, pg, 100, u8_r, bop, sop, None)
    call("programs_mp3/batch0", f, ctx, 0, tp, op, stp, spp, 1, pg, 0, u8_r, bop, sop, None)
    call("programs_mp3/bad_table", f, ctx, B, tp, op, stp, spp, 2, pb, 0, u8_r, bop, sop, None)
    call("programs_mp3/kbps100+bad_table", f, ctx, B, tp, op, stp, spp, 2, pb, 100, u8_r, bop, sop, None)
    call("programs_mp3/batch0+bad_table", f, ctx, 0, tp, op, stp, spp, 2, pb, 0, u8_r, bop, sop, None)
    call("programs_mp3/offsets_null+kbps100", f, ctx, B, tp, op, stp, spp, 1, pg, 100, u8_r, None, sop, None)
    f = lib.kkx_set_option
    call("set_option/null_key", f, ctx, None, 1)
    call("set_option/null_ctx", f, None, b"precision", 1)
    for k, v in (("nonsense", 1), ("precision", 2), ("max_frames", 0), ("fork_max_batch", 513), ("max_tokens", 100),
                 ("coalesce", 513), ("coalesce_wait_us", -1), ("async_batch", 0), ("out_rate", 7000),
                 ("out_rate", 23000), ("loudness_target", -100), ("true_peak_max", 1), ("limiter", 2),
                 ("loudness_report", 2), ("flac_lpc_order", 13)):
        call(f"set_option/{k}={v}", f, ctx, k.encode(), v)
    for name, fn, args in (("get_stat/null_key", lib.kkx_get_stat, (ctx, None)),
                           ("get_stat/unknown", lib.kkx_get_stat, (ctx, b"nonsense")),
                           ("get_stat/null_ctx", lib.kkx_get_stat, (None, b"launches")),
                           ("profile_json/null_ctx", lib.kkx_profile_json, (None, None, 0)),
                           ("debug_stage/null_name", lib.kkx_debug_stage, (ctx, None, 0, None, 0, None, None)),
                           ("debug_stage/unknown", lib.kkx_debug_stage, (ctx, b"nonsense", 0, None, 0, None, None)),
                           ("debug_stage/null_ctx", lib.kkx_debug_stage, (None, b"F0", 0, None, 0, None, None))):
        rc = fn(*args)
        bad[name] = [rc, err() if rc < 0 else ""]
    call("profile_enable/null_ctx", lib.kkx_profile_enable, None, 1)
    call("debug_enable/null_ctx", lib.kkx_debug_enable, None, 1)
    call("debug_select/null_ctx", lib.kkx_debug_select, None, 1, 0)
    call("last_loudness/batch_mismatch", lib.kkx_last_loudness, ctx, 7, None, None, None)
    res["bad_arguments"] = bad
    res["after_bad_arguments"] = {"reports": reports(), "out_rate": m.get_stat("out_rate"),
                                  "precision": m.get_stat("precision")}
    n, _ = m.run_staged()                    # still the batch staged before the rejected calls
    audio, so, dur = m.fetch_staged(n)
    res["after_bad_arguments"].update({"staged_audio": sha(audio), "sample_offsets": so.tolist(),
                                       "pred_dur": dur.tolist(), "run_staged_reports": reports()})
    # a run without the report options: the accessors say so
    m.set_option("loudness_report", 0)
    m.set_option("loudness_target", 0)
    m.set_option("limiter", 0)
    outs = m.infer_batch(toks[:2], styles[:2], speeds[:2])
    res["no_report"] = {"audio": [sha(o) for o in outs], "reports": reports()}
    m.close()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as fo:
        json.dump(res, fo, indent=1, sort_keys=True)
    print(f"{len(res)} sections, {len(bad)} bad-argument cases -> {a.out}")


if __name__ == "__main__":
    main()
