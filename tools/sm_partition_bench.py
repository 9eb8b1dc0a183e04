#!/usr/bin/env python
"""Two encoders on one GPU: contexts on SM groups (fo_create_on_sms) against whole-device contexts.

    python tools/sm_partition_bench.py [--chunks 200] [--runs 5] [--out profiles/r03_sm_partition.json]

Shipped model, bf16, random-init weights ("user" seed 0, "system" seed 1), device-resident int16 PCM.  Legs, alternated
within each run:
  (a) one whole-device context alone;
  (b) one context on half of the SMs (split 2, group 0) alone;
  (c) two half contexts (groups 0 and 1) streaming at once, one host thread and stream each;
  (d) two whole-device contexts streaming at once, the same way.
Per leg: 1 session, per-chunk latency (enqueue -> stream synchronised) p50 / p99; 64 sessions, step time p50 and the
aggregate audio-s/s of every context of the leg.  Best and spread (max - min) of each figure over the runs; the card's name,
power limit and SM clock are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402

CHUNK_SEC = 0.16


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True).stdout
        return dict(zip(q.split(","), [v.strip() for v in out.splitlines()[0].split(",")]))
    except Exception as e:      # the figures are still measured; the record says the card was not identified
        return {"error": str(e)}


def stream(eng, ids, pcm, times, st):
    """Every chunk of pcm (k, n, samples) through eng on stream st, each timed from enqueue to completion."""
    with torch.cuda.stream(st):
        for x in pcm:
            t0 = time.perf_counter()
            eng.stream_step(ids, x, 1.0)
            st.synchronize()
            times.append(time.perf_counter() - t0)


def leg(pairs):
    """pairs: [(engine, ids, pcm)], each streamed from its own host thread and stream; per-context chunk times and wall."""
    times = [[] for _ in pairs]
    streams = [torch.cuda.Stream() for _ in pairs]
    th = [threading.Thread(target=stream, args=(e, i, p, times[k], streams[k])) for k, (e, i, p) in enumerate(pairs)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for t in th:
        t.start()
    for t in th:
        t.join()
    torch.cuda.synchronize()
    return times, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--chunks", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_sm_partition.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a B200"
    info = card()
    cfg = load_path_config("shipped")
    states = [(make_encoder_state(cfg, s), make_adapter_state(cfg, s)) for s in (0, 1)]

    def make(seed, part):
        return Engine(cfg, *states[seed], dtype=torch.bfloat16, max_sessions=64, sm_partition=part)

    whole = [make(0, None), make(1, None)]
    half = [make(0, (2, 0)), make(1, (2, 1))]
    legs = {"a_whole_alone": [whole[0]], "b_half_alone": [half[0]], "c_two_halves": half, "d_two_wholes": whole}
    g = torch.Generator().manual_seed(7)
    res = {}
    for n in (1, 64):
        k = a.chunks if n == 1 else max(20, a.chunks // 4)
        pcm = [torch.randint(-3000, 3000, (k, n, cfg.samples_per_chunk), generator=g, dtype=torch.int32).to(torch.int16).cuda()
               for _ in range(2)]
        ids = {id(e): e.alloc(n) for e in whole + half}
        for name, engs in legs.items():                     # warm-up: graphs captured, workspaces sized
            leg([(e, ids[id(e)], pcm[j][:a.warmup]) for j, e in enumerate(engs)])
        runs = {name: [] for name in legs}
        for r in range(a.runs):
            order = list(legs) if r % 2 == 0 else list(legs)[::-1]
            for name in order:
                engs = legs[name]
                times, wall = leg([(e, ids[id(e)], pcm[j]) for j, e in enumerate(engs)])
                ms = [1e3 * np.asarray(t) for t in times]
                runs[name].append({"p50_ms": [float(np.percentile(m, 50)) for m in ms],
                                   "p99_ms": [float(np.percentile(m, 99)) for m in ms],
                                   "audio_s_per_s": len(engs) * n * k * CHUNK_SEC / wall})
        for e in whole + half:
            e.free(ids[id(e)])
        for name, rs in runs.items():
            out = {}
            for key in ("p50_ms", "p99_ms"):
                worst = [max(r[key]) for r in rs]              # the slower context of the leg
                out[key] = {"best": min(worst), "spread": max(worst) - min(worst), "per_context_runs": [r[key] for r in rs]}
            agg = [r["audio_s_per_s"] for r in rs]
            out["audio_s_per_s"] = {"best": max(agg), "spread": max(agg) - min(agg)}
            res["%d_sessions/%s" % (n, name)] = out
            print("%2d sessions %-14s p50 %.3f ms (spread %.3f)  p99 %.3f ms  aggregate %.0f audio-s/s"
                  % (n, name, out["p50_ms"]["best"], out["p50_ms"]["spread"], out["p99_ms"]["best"], out["audio_s_per_s"]["best"]))
    rec = {"card": info, "sm_count": {"whole": whole[0].sm_count, "half": half[0].sm_count}, "chunks": a.chunks,
           "runs": a.runs, "model": "shipped, bf16, random-init weights, device-resident int16 PCM", "results": res}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    for e in whole + half:
        e.close()


if __name__ == "__main__":
    main()
