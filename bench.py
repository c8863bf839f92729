#!/usr/bin/env python
"""bench.py -- benchmark of the B200-native Kokoro-82M backend (BASELINE.json metric and configs).

    python bench.py --gpus N --steps K --warmup W            # our arm (default: every config below)
    python bench.py --impl reference --gpus N --steps K ...  # CPU reference arm (rank 0 only)
    python bench.py --config 2|3|4 ...                       # one config only
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as .npy

Headline (BASELINE configs[2]): audio-seconds generated per second at B = 64 x 510 tokens per GPU.  A "step" is one
pass of the whole forward over one batch of 64 synthetic utterances (kokorox_b200.synth.synth_batch: 510 ids ~
U{1..177} seeds 1000+b, styles N(0,0.15^2) seeds 2000+b, speed 1.0 -- SURVEY.md 8d).
  `value`  times kkx_run_staged (inputs resident in HBM, CUDA events on the library's stream);
  `e2e`    times B200Koko.infer_batch (host numpy in, pinned host audio out, copies in the timed region).
Extra keys of the same JSON line, so that the driver's run measures them too:
  `latency`  configs[1]: B = 1 latency at 510 tokens (mixed style 0.4*A + 0.5*B, koko.rs:1283) and at 50 tokens;
  `cfg3`     configs[3]: 128-token segments, closed loop at c = 1/4/16/64 clients, first-audio p50/p95 -- driven by
             the NATIVE load generator kokorox_b200/lib/kkx_loadgen (C++ threads calling kkx_infer / kkx_submit);
  `cfg4`     configs[4]: 4096 mixed requests (length, voice, speed, 10 % to a second model) sharded by request
             over the N ranks with kokorox_b200.sharding.shard_requests;
  `per_rank` step time, frames and clocks of every rank (N > 1), so a scaling loss can be attributed;
  `ort`      the reference's ORT CPU path when onnxruntime + a model file exist, else "absent".
Multi-GPU: one process per GPU, each with its own requests (weak scaling); there is NO collective on the data path
(utterances are independent, koko.rs:947-1191).  torch.distributed is initialised as the driver's launch contract
asks (NCCL, one rank per GPU) and is used only for the barrier around the timed region and for reducing scalars.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark leaves the tree as it found it (it may be read-only)

from kokorox_b200.synth import (ensure_weights, synth_batch, synth_case, synth_requests_cfg4,  # noqa: E402
                                synth_voice_table)

# SURVEY.md 8d work model: MACs per token (attention term scaled by N/512) and per frame
MAC_TOKEN_FIXED = 88.86e6 - 9.44e6
MAC_TOKEN_ATTN = 9.44e6
MAC_FRAME = 658.55e6
REF_SUBSET = (0, 1)      # utterances of the batch the reference arm runs every step (fixed, stated)
DUMP_BYTES = 64_000_000  # --dump-outputs writes at most this many bytes in all
DUMP_SEED = 0            # fixed sample of a waveform too large to dump whole

_checkpoint_dir = None


def checkpoint(seed: int = 1234) -> str:
    """The random-init checkpoint of `seed` (kokorox_b200.synth), generated on first use.  None ships with the project
    and the tree may be read-only, so it goes to a temporary directory of this process, removed at exit.  A file named
    by $KKX_WEIGHTS stands in for the seed-1234 one."""
    global _checkpoint_dir
    if seed == 1234 and "KKX_WEIGHTS" in os.environ:
        return ensure_weights()
    if _checkpoint_dir is None:
        _checkpoint_dir = tempfile.mkdtemp(prefix="kkx_bench_")
        atexit.register(shutil.rmtree, _checkpoint_dir, True)
    return ensure_weights(os.path.join(_checkpoint_dir, f"kokoro_random_{seed}.kkxw"), seed=seed)


def dump_arrays(audio: np.ndarray, sample_offsets: np.ndarray, durations: np.ndarray) -> dict:
    """What --dump-outputs writes for one staged step: the flat waveform of the batch, where each utterance starts in
    it, and the integer frame durations of every token.  A waveform too large for what DUMP_BYTES leaves after the
    other arrays is replaced by a seeded, sorted sample of its positions (`audio_index`), the same for the same
    length, so that two builds can be compared array for array."""
    out = {"sample_offsets": sample_offsets.astype(np.float64), "durations": durations.astype(np.float64)}
    room = DUMP_BYTES - 4096 - sum(a.nbytes for a in out.values())     # 4 KB for the .npy headers
    audio = np.asarray(audio, dtype=np.float32)
    if audio.nbytes > room:
        n = room // (4 + 8)                               # f32 sample + f64 index per kept position
        idx = np.sort(np.random.default_rng(DUMP_SEED).choice(audio.size, n, replace=False))
        out["audio_index"] = idx.astype(np.float64)
        audio = audio[idx]
    out["audio"] = audio
    return out


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING a timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu: int):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        ok = [r for r in self.rows if len(r) >= 7]
        sm = [float(r[0]) for r in ok if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in ok if r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in ok if r[2].replace(".", "").isdigit()]
        reasons, capped = set(), 0
        for r in ok:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
                    capped += name == "sw_power_cap"
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(pw) if pw else None,
                "sw_power_cap_samples": capped}


# ------------------------------------------------------------------------------------------- reference arm
def make_cpu_reference(threads: int):
    """(callable(tokens, style) -> waveform, kind, description).  ORT CPU EP on the real model when it can be had
    (oracle/ort_ref.py), else the torch fp32 restatement of the published algorithm (kind "port")."""
    from oracle import ort_ref
    ok, why = ort_ref.available()
    if ok:
        ref = ort_ref.OrtReference(why, threads=threads)
        return (lambda t, s: ref.infer(t, s, 1.0)), "ort", f"ONNX Runtime CPU EP on {os.path.basename(why)}"
    from kokorox_b200.weightfile import read_weights
    from oracle.kokoro_ref import KokoroOracle
    o = KokoroOracle(read_weights(checkpoint()), threads=threads)
    k = [0]

    def run(t, s):
        k[0] += 1
        return o.forward(t, s, 1.0, noise_seed=k[0])["audio"]
    return run, "port", "torch fp32 CPU restatement of the ONNX graph (oracle/kokoro_ref.py); ORT absent: " + why


def cpu_reference_rate(utts, threads: int, n_tokens: int):
    """Times the CPU reference (B = 1 sequential, like the reference's chunk loop koko.rs:947-1191) on `utts`."""
    run, kind, desc = make_cpu_reference(threads)
    toks, styles, _ = synth_batch(max(utts) + 1, n_tokens)
    run(toks[0][:60], styles[0])  # warm-up (lazy init, thread pools)
    t0 = time.perf_counter()
    audio_s = 0.0
    for b in utts:
        audio_s += len(run(toks[b], styles[b])) / 24000.0
    dt = time.perf_counter() - t0
    return audio_s / dt, audio_s, dt, kind, desc


def run_reference(args, rank: int):
    """The reference's CPU implementation of the path on this box's cores: every step runs the SAME fixed subset of
    the benched batch (utterances REF_SUBSET of synth_batch(64, 510)), B = 1 sequentially like koko.rs:947-1191."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    run, kind, desc = make_cpu_reference(threads)
    toks, styles, _ = synth_batch(args.batch, args.tokens)
    times, audio = [], []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        a = 0.0
        for b in REF_SUBSET:
            a += len(run(toks[b], styles[b])) / 24000.0
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
            audio.append(a)
    value = sum(audio) / sum(times)
    sample = (f"utterances {list(REF_SUBSET)} of the {args.batch} of the benched batch, every step (same seeds as the "
              f"GPU arm), B=1 sequential (koko.rs:947-1191); {desc}")
    import torch
    print(json.dumps({
        "impl": "reference", "metric": "audio-seconds per second", "value": value, "unit": "audio-s/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"B={args.batch} x {args.tokens} tokens, ragged durations (BASELINE configs[2]); "
                               f"bounded sample: {len(REF_SUBSET)} fixed utterances per step",
                   "weights": "random-init seed 1234 (no checkpoint, no network)" if kind == "port" else "kokoro-v1.0.onnx",
                   "subset": list(REF_SUBSET), "audio_s_per_step": sum(audio) / len(audio)},
        "cpu_baseline": {"value": value, "unit": "audio-s/s", "cores": threads, "kind": kind, "sample": sample,
                         "threads": {"os_cpu_count": os.cpu_count(), "torch_num_threads": torch.get_num_threads(),
                                     "torch_interop_threads": torch.get_num_interop_threads()}},
        "e2e": {"value": value, "unit": "audio-s/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


# ------------------------------------------------------------------------------------------- helpers
def all_gather_floats(vals, world):
    """[world][len(vals)] floats from every rank (local values at N = 1)."""
    import torch
    import torch.distributed as dist
    if world == 1:
        return [list(map(float, vals))]
    t = torch.tensor(list(vals), dtype=torch.float64, device="cuda")
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t)
    return [[float(x) for x in o.tolist()] for o in out]


def pack_requests(idx, lens, token_budget=64 * 512, max_items=512):
    """Ragged batches under the token budget, longest first so a batch's items have similar length."""
    out, cur, tok = [], [], 0
    for i in sorted(idx, key=lambda i: (-lens[i], i)):
        if cur and (tok + lens[i] > token_budget or len(cur) >= max_items):
            out.append(cur)
            cur, tok = [], 0
        cur.append(i)
        tok += lens[i]
    if cur:
        out.append(cur)
    return out


# ------------------------------------------------------------------------------------------- configs[3]
def run_cfg3(local_rank: int, conc="1,4,16,64", requests=8, tokens=128):
    """Closed-loop clients on ONE GPU through the native load generator (kokorox_b200/csrc/loadgen.cpp)."""
    from kokorox_b200 import build
    exe = build.LOADGEN
    if not os.path.exists(exe):
        return {"error": "kkx_loadgen not built"}
    sampler = ClockSampler(local_rank).start()
    t0 = time.perf_counter()
    r = subprocess.run([exe, checkpoint(), "--device", str(local_rank), "--tokens", str(tokens), "--requests",
                        str(requests), "--conc", conc, "--modes", "serial,coalesce,async"],
                       capture_output=True, text=True, timeout=900)
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    if r.returncode != 0:
        return {"error": f"kkx_loadgen rc={r.returncode}: {r.stderr[-300:]}"}
    rows = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    best = max((x for x in rows if x["mode"] != "serial"), key=lambda x: (x["concurrency"], x["audio_s_per_s"]), default=None)
    return {"workload": f"BASELINE configs[3]: {tokens}-token segments, closed loop, {requests} segments per client, "
                        "native load generator (C++ threads on the C ABI)",
            "first_audio": "submit -> the segment's complete waveform in host memory",
            "rows": rows, "headline": best, "clocks": clocks, "wall_s": round(wall, 2)}


# ------------------------------------------------------------------------------------------- configs[4]
def run_cfg4(rank, local_rank, world, barrier, passes=1, n_req=4096):
    """4096 mixed requests sharded over the ranks; 10 % go to a second session holding a DIFFERENT weight set."""
    import torch
    from kokorox_b200.onn import B200Koko
    from kokorox_b200.sharding import reduce_step, shard_requests
    toks, voices, speeds, zh = synth_requests_cfg4(n_req)
    lens = [len(t) for t in toks]
    mine = shard_requests(lens, world)[rank]
    table = synth_voice_table(54)
    vt = {f"v{v:02d}": table[v] for v in range(54)}
    sessions = {}
    for lang, wp in (("en", checkpoint()), ("zh", checkpoint(4321))):
        m = B200Koko.new(wp, device=local_rank)
        m.load_voices(vt)
        sessions[lang] = m
    work = [(lang, b) for lang in ("en", "zh")
            for b in pack_requests([i for i in mine if bool(zh[i]) == (lang == "zh")], lens)]
    launches = [0]

    def run_all():
        audio = 0.0
        for lang, b in work:
            outs = sessions[lang].infer_batch_voices([toks[i] for i in b], [f"v{voices[i]:02d}" for i in b],
                                                     [float(speeds[i]) for i in b])
            audio += sum(len(o) for o in outs) / 24000.0
            launches[0] += sessions[lang].get_stat("launches")
        return audio

    barrier()
    t0 = time.perf_counter()
    run_all()                      # cold pass: device arenas and the pinned pool grow to their working size
    torch.cuda.synchronize()
    cold = time.perf_counter() - t0
    sampler = ClockSampler(local_rank).start()
    barrier()
    launches[0] = 0
    t0 = time.perf_counter()
    audio = 0.0
    for _ in range(passes):
        audio += run_all()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    barrier()
    clocks = sampler.stop()
    wall_max, (audio_all, req_all, tok_all, launches_all) = reduce_step(
        wall, [audio, float(len(mine) * passes), float(sum(lens[i] for i in mine) * passes), float(launches[0])],
        torch.device("cuda", local_rank))
    per_rank = all_gather_floats([wall, audio, len(mine)], world)
    for m in sessions.values():
        m.close()
    return {"workload": f"BASELINE configs[4]: {n_req} requests, N~U{{10..510}} tokens, 54 device-resident voices, "
                        "speed~U[0.8,1.3], 10% routed to a second model (different weight set), sharded by request "
                        f"over {world} GPU(s) with shard_requests, ragged batches <= 64x512 tokens",
            "n_gpus": world, "requests": int(req_all), "tokens": int(tok_all), "audio_s": round(audio_all, 1),
            "wall_s": round(wall_max, 3), "audio_s_per_s": round(audio_all / wall_max, 1),
            "requests_per_s": round(req_all / wall_max, 1), "cold_first_pass_wall_s_rank0": round(cold, 3),
            "gpu_launches": int(launches_all), "batches_rank0": len(work), "clocks_rank0": clocks,
            "per_rank": [{"rank": r, "wall_s": round(v[0], 3), "audio_s": round(v[1], 1), "requests": int(v[2])}
                         for r, v in enumerate(per_rank)],
            "timing": "host wall clock around the public host-buffer calls (kkx_infer_batch_voices), max over ranks"}


# ------------------------------------------------------------------------------------------- ORT leg
def ort_leg(local_rank: int):
    """SURVEY 8c / BASELINE.md 2: when onnxruntime and a model file exist, run ORT CPU EP and the CUDA path loaded
    from the SAME file on the cfg0 input and report sum(dur) equality + waveform distances.  Otherwise "absent"."""
    try:
        from oracle import ort_ref
        ok, why = ort_ref.available()
        if not ok:
            return "absent", why
        from kokorox_b200.onn import B200Koko
        ids, style = synth_case(50, 0, 100)
        ref = ort_ref.OrtReference(why, threads=os.cpu_count())
        t0 = time.perf_counter()
        want = ref.infer(ids, style, 1.0)
        dt = time.perf_counter() - t0
        m = B200Koko.new(why, device=local_rank)          # kkx_create reads the .onnx itself
        got = m.infer_one(ids, style, 1.0).copy()
        m.close()
        out = ort_ref.compare(got, want)
        out.update({"model": os.path.basename(why), "ort_audio_s_per_s": len(want) / 24000.0 / dt})
        return out, why
    except Exception as e:  # noqa: BLE001 -- the bench line must survive a broken optional leg
        return {"error": f"{type(e).__name__}: {e}"}, ""


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="all", choices=["all", "2", "3", "4"],
                    help="all = headline configs[2] + latency + cfg3 + cfg4 as extra keys; 2/3/4 = that config only")
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--tokens", type=int, default=510)
    ap.add_argument("--precision", type=int, default=int(os.environ.get("KKX_PRECISION", "1")),
                    help="1 = tensor-core configuration (the library default), 0 = fp32 SIMT everywhere")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-out", default=None, help="write the per-kernel timing table of one step here")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step of the headline path computed to DIR/<name>.npy "
                         "(waveform, utterance offsets, token durations; at most 64 MB, a seeded sample of the waveform)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.config in ("3", "4")):
        ap.error("--dump-outputs writes the headline path's results: it needs --impl ours and --config all or 2")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the B200 backend has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from kokorox_b200 import build
    from kokorox_b200.onn import B200Koko, init_ort
    from kokorox_b200.sharding import reduce_step
    build.build()
    init_ort()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # every process generates the synthetic checkpoints it reads, in its own temporary directory, before any timing
    checkpoint()
    if args.config in ("all", "4"):
        checkpoint(4321)

    if args.config == "3":
        if rank == 0:
            c3 = run_cfg3(local_rank)
            h = c3.get("headline") or {}
            print(json.dumps({"metric": "audio-seconds per second", "value": h.get("audio_s_per_s"), "unit": "audio-s/s",
                              "n_gpus": 1, "steps": 1, "warmup": 1, "ms_per_step": None, "higher_is_better": True,
                              "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                              "config": {"workload": c3.get("workload")}, "clocks": c3.get("clocks"), "cfg3": c3}))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return
    if args.config == "4":
        c4 = run_cfg4(rank, local_rank, world, barrier, passes=max(1, args.steps // 3))
        if rank == 0:
            print(json.dumps({"metric": "audio-seconds per second", "value": c4["audio_s_per_s"], "unit": "audio-s/s",
                              "n_gpus": world, "steps": max(1, args.steps // 3), "warmup": 1,
                              "ms_per_step": c4["wall_s"] * 1e3 / max(1, args.steps // 3), "higher_is_better": True,
                              "scaling": "strong", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                              "config": {"workload": c4["workload"]}, "clocks": c4["clocks_rank0"],
                              "gpu_launches": c4["gpu_launches"], "cfg4": c4}))
        if world > 1:
            dist.destroy_process_group()
        return

    m = B200Koko.new(checkpoint(), device=local_rank)
    default_precision = m.get_stat("precision")          # what an unconfigured session runs (ADVICE r1: stated)
    m.set_option("precision", args.precision)
    # weak scaling: every rank runs the SAME 64 utterances (per-GPU work fixed; rank-dependent seeds made the ranks'
    # frame counts differ by ~5 %, which showed up as a scaling loss that was really load imbalance -- VERDICT r1).
    # The mixed, sharded workload is cfg4.
    toks, styles, speeds = synth_batch(args.batch, args.tokens, 0)
    sum_n = sum(len(t) for t in toks)

    # ---------------- value: inputs resident in HBM, device-timed
    m.stage(toks, styles, speeds)
    launches = 0
    for _ in range(args.warmup):
        total, launches = m.run_staged()
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    t0 = time.perf_counter()
    gpu_us, totals = [], []
    for _ in range(args.steps):
        total, launches = m.run_staged()
        gpu_us.append(m.get_stat("gpu_us"))
        totals.append(total)
    barrier()
    wall = time.perf_counter() - t0
    clocks = sampler.stop()
    dev_s = sum(gpu_us) * 1e-6
    frames = m.get_stat("last_frames")
    groups = m.get_stat("frame_groups")
    audio_s_step = totals[-1] / 24000.0
    if args.dump_outputs and rank == 0:          # every rank runs the same batch
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dump_arrays(*m.fetch_staged(totals[-1])).items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)

    # one profiled step (not part of the timed region) for the roofline of the dominant kernel
    m.profile_enable(True)
    m.run_staged()
    prof = m.profile()
    m.profile_enable(False)
    if args.profile_out and rank == 0:
        with open(args.profile_out, "w") as f:
            json.dump(prof, f, indent=1)

    # ---------------- e2e: host buffers through the public call, copies inside the timed region
    outs = None
    for _ in range(max(args.warmup, 3)):   # same call pattern as the timed loop: the previous result is still alive
        outs = m.infer_batch(toks, styles, speeds)   # during the next call, so the library cycles two pinned buffers
    barrier()
    t1 = time.perf_counter()
    e2e_audio = 0.0
    for _ in range(args.steps):
        outs = m.infer_batch(toks, styles, speeds)
        e2e_audio += sum(len(o) for o in outs) / 24000.0
    barrier()
    e2e_wall = time.perf_counter() - t1
    del outs
    h2d = sum_n * 8 + styles.nbytes + speeds.nbytes
    d2h = int(totals[-1]) * 4 + sum_n * 4

    # ---------------- B=1 latency (configs[1]): 510 tokens with the mixed style 0.4*A + 0.5*B (koko.rs:1283); 50 tokens
    latency = None
    if rank == 0:
        mix = (0.4 * styles[0] + 0.5 * styles[1]).astype(np.float32)
        short = synth_case(50, 0, 100)
        latency = {}
        for name, ids, st in (("b1_510tok", toks[0], mix), ("b1_50tok", short[0], short[1])):
            lat, gpu = [], []
            for i in range(12):
                ta = time.perf_counter()
                y = m.infer_one(ids, st, 1.0)
                lat.append((time.perf_counter() - ta) * 1e3)
                gpu.append(m.get_stat("gpu_us") / 1e3)
                del y
            lat, gpu = lat[4:], gpu[4:]
            latency[name] = {"p50_ms": statistics.median(lat), "min_ms": min(lat), "max_ms": max(lat),
                             "gpu_ms_p50": statistics.median(gpu), "launches": m.get_stat("launches"),
                             "graph_replays": m.get_stat("graph_replays")}
        latency["call"] = "kkx_infer (host buffers in, pinned host waveform out), wall clock around the call, 8 timed calls after 4 warm-up"

    # ---------------- reductions over ranks (max time, summed work) + per-rank record
    step_s = dev_s / args.steps
    dev = torch.device("cuda", local_rank)
    my_step_s = step_s
    step_s, (audio_all, frames_all, tokens_all) = reduce_step(step_s, [audio_s_step, float(frames), float(sum_n)], dev)
    wall_step_s, _ = reduce_step(wall / args.steps, [0.0], dev)
    e2e_step_s, (e2e_audio_all,) = reduce_step(e2e_wall / args.steps, [e2e_audio / args.steps], dev)
    per_rank = all_gather_floats([my_step_s * 1e3, frames, audio_s_step, e2e_wall / args.steps * 1e3,
                                  clocks["sm_mhz"] or 0.0, clocks["sw_power_cap_samples"], clocks["samples"],
                                  clocks["power_w_max"] or 0.0], world)
    m.close()

    # ---------------- the other configs, measured in the same run
    cfg3 = cfg4 = None
    if args.config == "all":
        if rank == 0 and world == 1:
            try:
                cfg3 = run_cfg3(local_rank)
            except Exception as e:  # noqa: BLE001
                cfg3 = {"error": f"{type(e).__name__}: {e}"}
        cfg4 = run_cfg4(rank, local_rank, world, barrier)

    if rank == 0:
        peaks, peaks_src = load_peaks()
        # whole-step algorithmic work (SURVEY.md 8d), per rank
        flops_step = 2.0 * (MAC_TOKEN_FIXED * sum_n + MAC_TOKEN_ATTN * sum(len(t) ** 2 for t in toks) / 512.0
                            + MAC_FRAME * frames)
        kern = prof.get("kernels", {})
        top = max(kern.items(), key=lambda kv: kv[1][1]) if kern else ("none", [0, 0.0])
        total_us = sum(v[1] for v in kern.values()) or 1.0
        # roofline of the dominant kernel family.  The generator res-block convs (kernels_arb.cu, "arb_conv")
        # dominate the step; they are tensor-pipe work whose activations (GBs per launch) stream through HBM, so
        # both fractions are reported: algorithmic FLOPs and algorithmic bytes (every tensor once) over the summed,
        # event-timed launch durations of that kernel.
        conv_names = [k for k in kern if k.startswith("conv") or k == "arb_conv"]
        conv_us = sum(kern[k][1] for k in conv_names) or 1.0
        peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
        peak_gbs = peaks.get("hbm_gbs", 6650.0)
        dom = "arb_conv" if "arb_conv" in kern else (top[0] if top[0].startswith("conv") else "conv")
        if dom == "arb_conv":
            dn, dus = kern[dom]
            dflops, dbytes = prof.get("arb_flops", 0.0), prof.get("arb_bytes", 0.0)
        else:
            dn = sum(kern[k][0] for k in conv_names) or 1
            dus, dflops, dbytes = conv_us, prof.get("conv_flops", 0.0), 0.0
        achieved_tf = dflops / (dus * 1e-6) / 1e12
        # DRAM traffic per launch: the ncu --set full capture of this kernel (profiles/) measured
        # dram read+write = 1.00 x the algorithmic bytes; scale this run's per-launch algorithmic bytes by that ratio
        traffic, traffic_src = None, None
        try:
            with open(os.path.join(ROOT, "profiles", "r1_arb_conv_traffic.json")) as f:
                tj = json.load(f)
            if dom == "arb_conv" and dbytes > 0:
                traffic = tj["traffic_over_algorithmic"] * dbytes / max(dn, 1)
                traffic_src = "ncu dram__bytes_read+write / algorithmic bytes = %.4f (%s)" % (tj["traffic_over_algorithmic"], "profiles/r1_arb_conv_traffic.json")
        except Exception:
            pass
        roofline = {
            "bound": "tensor", "kernel": dom,
            "achieved": achieved_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved_tf / peak_tf,
            "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": f"{peaks_src} (sustained bf16; kernel timed inside a long step)",
            "launches_per_step": dn, "avg_launch_us": dus / max(dn, 1),
            "alg_flops_per_launch": dflops / max(dn, 1),
            "alg_bytes_per_launch": dbytes / max(dn, 1),
            "hbm_achieved_gbs": dbytes / (dus * 1e-6) / 1e9, "hbm_peak_gbs": peak_gbs,
            "hbm_frac": dbytes / (dus * 1e-6) / 1e9 / peak_gbs,
            "share_of_step": dus / total_us, "top_kernel": top[0], "top_kernel_share": top[1][1] / total_us,
            "all_conv_share_of_step": conv_us / total_us,
            "all_conv_tflops": prof.get("conv_flops", 0.0) / (conv_us * 1e-6) / 1e12,
            "step_alg_tflops": flops_step / step_s / 1e12,
            "kernel_ms": {k: round(v[1] / 1e3, 3) for k, v in sorted(kern.items(), key=lambda kv: -kv[1][1])[:14]},
        }
        line = {
            "metric": "audio-seconds per second", "value": audio_all / step_s, "unit": "audio-s/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_s * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == 0 else "bf16", "data": "synthetic",
            "config": {"workload": f"B={args.batch} x {args.tokens} tokens per GPU, ragged durations (BASELINE configs[2])",
                       "frames_per_step": frames_all, "tokens_per_step": tokens_all,
                       "audio_s_per_step": audio_all, "frame_groups_per_step": groups,
                       "weights": "random-init seed 1234 (no checkpoint, no network)",
                       "precision": args.precision, "library_default_precision": default_precision,
                       "parallelism": f"one process + one session per GPU x{world}, every rank the same batch, no collective on the data path",
                       "l2": "working set per step (GBs of activations) is larger than the 126 MB L2; no flush needed"},
            "clocks": clocks,
            "e2e": {"value": e2e_audio_all / e2e_step_s, "unit": "audio-s/s", "h2d_bytes_per_step": h2d * world,
                    "d2h_bytes_per_step": d2h * world},
            "gpu_launches": int(launches) * args.steps,
            "wall_ms_per_step": wall_step_s * 1e3,
            "roofline": roofline,
            "realtime_factor": audio_all / step_s,
            "latency": latency,
            "latency_b1_510tok_ms_p50": latency["b1_510tok"]["p50_ms"] if latency else None,
            "per_rank": [{"rank": r, "ms_per_step": round(v[0], 3), "frames": int(v[1]), "audio_s": round(v[2], 2),
                          "e2e_ms_per_step": round(v[3], 3), "sm_mhz": v[4], "sw_power_cap_samples": int(v[5]),
                          "clock_samples": int(v[6]), "power_w_max": v[7]} for r, v in enumerate(per_rank)],
            "cfg3": cfg3, "cfg4": cfg4,
        }
        ort, _ = ort_leg(local_rank) if world == 1 else ("not run at N > 1", "")
        line["ort"] = ort
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            utts = (0, 1, 2)
            v, a_s, dt, kind, desc = cpu_reference_rate(utts, threads, args.tokens)
            line["cpu_baseline"] = {"value": v, "unit": "audio-s/s", "cores": threads, "kind": kind,
                                    "sample": f"utterances {list(utts)} of the {args.batch} ({a_s:.1f} audio-s in {dt:.1f} s), "
                                              f"B=1 sequential like koko.rs:947-1191; {desc}"}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
