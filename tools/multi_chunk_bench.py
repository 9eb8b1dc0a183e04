"""Multi-chunk streaming steps (Engine.encode_stream_chunks) on the shipped model in bf16: what they buy the scheduler's
speech-onset ticks and exact-streaming encoding of whole files, and whether the single-chunk step moved.

  * ticks: 64 sessions through StreamScheduler, m of them at a speech onset (1 + onset_chunks blocks) and the rest with one
    block, max_chunks 1 and 7 alternated in one process on twin session sets fed identical audio: ms per tick, encode calls
    per tick and the max-abs difference of the two schedulers' encoder frames.
  * whole-file exact streaming: 188 chunks (30 s) per session at k = 1 and k = 16, for 1 and 16 sessions, audio-s per s.
  * --bench-ab TREE: `bench.py --gpus 1` of TREE (the parent commit, built) and of this tree, alternated twice.

Writes one JSON file (--out) that names the GPU and its power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.scheduler import StreamScheduler  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, r


def bench_ticks(eng, cfg, sessions, onsets, reps):
    scheds = {mc: StreamScheduler(eng, history_chunks=10, onset_chunks=6, bucket=16, max_sessions=sessions, max_chunks=mc)
              for mc in (1, 7)}
    for s in scheds.values():
        for i in range(sessions):
            s.open(i)
    g = torch.Generator().manual_seed(7)
    res = []
    for m in onsets:
        ms = {1: [], 7: []}
        calls = {1: [], 7: []}
        diff = 0.0
        for r in range(reps + 2):                                  # the first two ticks of a shape warm up and capture graphs
            pcm = (0.05 * torch.randn(sessions, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16).cuda()
            outs = {}
            for mc in ((1, 7) if r % 2 == 0 else (7, 1)):
                s = scheds[mc]
                for i in range(sessions):
                    s.push(i, pcm[i], "ipu_sl" if i < m else "ipu_cl")
                c0 = s.stats["encode_calls"]
                t, outs[mc] = timed(s.tick)
                if r >= 2:
                    ms[mc].append(t)
                    calls[mc].append(s.stats["encode_calls"] - c0)
            for i in range(sessions):
                for b1, b7 in zip(outs[1][i], outs[7][i]):
                    diff = max(diff, float((b1.enc - b7.enc).abs().max()))
        res.append({"onset_sessions": m,
                    "ms_per_tick": {str(mc): float(np.median(ms[mc])) for mc in ms},
                    "encode_calls_per_tick": {str(mc): float(np.mean(calls[mc])) for mc in calls},
                    "max_abs_enc_diff": diff})
        print(json.dumps(res[-1]), flush=True)
    for s in scheds.values():
        for i in range(sessions):
            s.close(i)
        eng.free(s.scratch)
    return res


def bench_exact_streaming(eng, cfg, chunks=188):
    res = []
    for n in (1, 16):
        ids = eng.alloc(n)
        g = torch.Generator().manual_seed(9)
        feats = (9.0 + 3.0 * torch.randn(n, chunks, cfg.chunk_feat_frames, cfg.feat_dim, generator=g)).cuda()
        for k in (1, 16):
            def run():
                for c0 in range(0, chunks, k):
                    kk = min(k, chunks - c0)
                    if k == 1:
                        eng.encode_stream(ids, feats[:, c0].contiguous())
                    else:
                        eng.encode_stream_chunks(ids, feats[:, c0:c0 + kk].contiguous())
            best = None
            for _ in range(3):                                     # pass 1 warms up and captures the graphs
                eng.reset(ids)
                ms, _ = timed(run)
                best = ms if best is None else min(best, ms)
            res.append({"sessions": n, "k": k, "ms": best, "audio_s_per_s": n * chunks * 0.16 / (best * 1e-3)})
            print(json.dumps(res[-1]), flush=True)
        eng.free(ids)
    return res


def bench_ab(parent_tree, steps, warmup):
    """bench.py of `parent_tree` (a checkout of the parent commit with its library built) against this tree's, alternated."""
    out = []
    for rep in range(2):
        for name, tree in (("parent", parent_tree), ("this", ROOT)):
            p = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup",
                                str(warmup)], capture_output=True, text=True, cwd=tree)
            lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
            if not lines:
                raise RuntimeError("bench.py of %s failed:\n%s" % (tree, p.stderr[-3000:]))
            line = json.loads(lines[-1])
            out.append({"build": name, "rep": rep, "value": line.get("value"), "unit": line.get("unit"),
                        "latency1": line.get("latency1")})
            print(json.dumps(out[-1]), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--bench-ab", default="", help="built checkout of another commit to compare bench.py against")
    ap.add_argument("--bench-steps", type=int, default=100)
    ap.add_argument("--bench-warmup", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    result = {"gpu": gpu_info()}
    cfg = load_path_config("shipped")
    eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=2 * (64 + 15))
    result["ticks_64_sessions"] = bench_ticks(eng, cfg, 64, (0, 1, 2, 8), args.reps)
    result["exact_streaming_188_chunks"] = bench_exact_streaming(eng, cfg)
    eng.close()
    if args.bench_ab:
        result["bench_ab"] = bench_ab(os.path.abspath(args.bench_ab), args.bench_steps, args.bench_warmup)
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
