"""Multi-chunk streaming steps (Engine.encode_stream_chunks) on the shipped model in bf16: what they buy the scheduler's
speech-onset ticks and exact-streaming encoding of whole files, and whether the single-chunk step moved.

  * ticks: 64 sessions through StreamScheduler, m of them at a speech onset (1 + onset_chunks blocks) and the rest with one
    block; max_chunks 1, max_chunks 7 (one call per chunk count) and max_chunks 7 with mixed_calls (one call per round)
    alternated in one process on three session sets fed identical audio: ms per tick, encode calls per tick, the distinct
    call shapes (= graph keys) the run used, and the max-abs difference of each scheduler's encoder frames against
    max_chunks 1.
  * adapter share: a 64-session mixed call (1 or 8 sessions at 7 chunks) with and without the adapter, against the same for
    one single-chunk call over as many blocks (the adapter without the per-session padding of the mixed call's conv grid).
  * whole-file exact streaming: 188 chunks (30 s) per session at k = 1 and k = 16, for 1 and 16 sessions, audio-s per s.
  * --bench-ab TREE: `bench.py --gpus 1` of TREE (the parent commit, built) and of this tree, alternated --ab-reps times,
    which of the two goes first swapping every rep.

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


class ShapeLog:
    """Wraps the engine's streaming entries and records the shape of every call: (entry, sessions, blocks, largest count,
    leading one-chunk run) -- the totals a captured step graph is keyed by."""

    def __init__(self, eng):
        self.eng, self.shapes = eng, set()

    def __getattr__(self, name):
        return getattr(self.eng, name)

    def encode_stream(self, ids, feats, **kw):
        self.shapes.add(("stream", len(ids), len(ids), 1, len(ids)))
        return self.eng.encode_stream(ids, feats, **kw)

    def encode_stream_chunks(self, ids, feats, **kw):
        self.shapes.add(("chunks", len(ids), len(ids) * feats.shape[1], feats.shape[1], 0))
        return self.eng.encode_stream_chunks(ids, feats, **kw)

    def encode_stream_chunks_v(self, ids, chunks, feats, **kw):
        c = list(chunks)
        n1 = next((i for i, k in enumerate(c) if k > 1), len(c))
        self.shapes.add(("chunks_v", len(c), sum(c), max(c), n1))
        return self.eng.encode_stream_chunks_v(ids, chunks, feats, **kw)


SCHEDULERS = {"1": dict(max_chunks=1), "7": dict(max_chunks=7), "7_mixed": dict(max_chunks=7, mixed_calls=True)}


def bench_ticks(eng, cfg, sessions, onsets, reps):
    logs = {name: ShapeLog(eng) for name in SCHEDULERS}
    scheds = {name: StreamScheduler(logs[name], history_chunks=10, onset_chunks=6, bucket=16, max_sessions=sessions, **kw)
              for name, kw in SCHEDULERS.items()}
    for s in scheds.values():
        for i in range(sessions):
            s.open(i)
    g = torch.Generator().manual_seed(7)
    res = []
    names = list(SCHEDULERS)
    for m in onsets:
        ms = {name: [] for name in names}
        calls = {name: [] for name in names}
        diff = {name: 0.0 for name in names[1:]}
        for lg in logs.values():
            lg.shapes = set()
        for r in range(reps + 2):                                  # the first two ticks of a shape warm up and capture graphs
            pcm = (0.05 * torch.randn(sessions, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16).cuda()
            outs = {}
            for name in names[r % 3:] + names[:r % 3]:             # rotate which scheduler goes first
                s = scheds[name]
                for i in range(sessions):
                    s.push(i, pcm[i], "ipu_sl" if i < m else "ipu_cl")
                c0 = s.stats["encode_calls"]
                t, outs[name] = timed(s.tick)
                if r >= 2:
                    ms[name].append(t)
                    calls[name].append(s.stats["encode_calls"] - c0)
            for name in names[1:]:
                for i in range(sessions):
                    assert len(outs["1"][i]) == len(outs[name][i])
                    for b1, bk in zip(outs["1"][i], outs[name][i]):
                        diff[name] = max(diff[name], float((b1.enc - bk.enc).abs().max()))
        res.append({"onset_sessions": m,
                    "ms_per_tick": {name: float(np.median(ms[name])) for name in names},
                    "encode_calls_per_tick": {name: float(np.mean(calls[name])) for name in names},
                    "call_shapes": {name: len(logs[name].shapes) for name in names},
                    "max_abs_enc_diff_vs_1": diff})
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


def bench_adapter_share(eng, cfg, sessions, onsets, reps):
    """ms of a mixed call with and without the adapter, and of a single-chunk call over as many blocks, alternated."""
    res = []
    g = torch.Generator().manual_seed(11)
    for m in onsets:
        chunks = np.array([1] * (sessions - m) + [7] * m, np.int32)
        B = int(chunks.sum())
        mixed, single = eng.alloc(sessions), eng.alloc(B)
        feats = (9.0 + 3.0 * torch.randn(B, cfg.chunk_feat_frames, cfg.feat_dim, generator=g)).cuda()
        runs = {"mixed_with_adapter": lambda: eng.encode_stream_chunks_v(mixed, chunks, feats, want_adapter=True),
                "mixed_encoder_only": lambda: eng.encode_stream_chunks_v(mixed, chunks, feats, want_adapter=False),
                "single_with_adapter": lambda: eng.encode_stream(single, feats, want_adapter=True),
                "single_encoder_only": lambda: eng.encode_stream(single, feats, want_adapter=False)}
        ms = {k: [] for k in runs}
        for r in range(reps + 2):                                  # two passes warm up and capture the graphs
            for k in (list(runs) if r % 2 == 0 else list(runs)[::-1]):
                t, _ = timed(runs[k])
                if r >= 2:
                    ms[k].append(t)
        med = {k: float(np.median(v)) for k, v in ms.items()}
        ad_mixed = med["mixed_with_adapter"] - med["mixed_encoder_only"]
        ad_single = med["single_with_adapter"] - med["single_encoder_only"]
        res.append({"sessions": sessions, "onset_sessions": m, "blocks": B, "ms": med,
                    "adapter_ms_mixed": ad_mixed, "adapter_ms_single_call_same_blocks": ad_single,
                    "adapter_share_of_mixed_call": ad_mixed / med["mixed_with_adapter"],
                    "padding_ms": ad_mixed - ad_single,
                    "padding_share_of_mixed_call": (ad_mixed - ad_single) / med["mixed_with_adapter"]})
        print(json.dumps(res[-1]), flush=True)
        eng.free(mixed)
        eng.free(single)
    return res


def bench_ab(parent_tree, steps, warmup, reps):
    """bench.py of `parent_tree` (a checkout of the parent commit with its library built) against this tree's, alternated;
    the build that runs first swaps every rep, so that a drift over the run does not favour one of them."""
    out = []
    for rep in range(reps):
        order = (("parent", parent_tree), ("this", ROOT))
        for name, tree in (order if rep % 2 == 0 else order[::-1]):
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
    ap.add_argument("--ab-reps", type=int, default=4)
    ap.add_argument("--ticks-only", action="store_true", help="skip the adapter-share and whole-file exact-streaming runs")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    result = {"gpu": gpu_info()}
    cfg = load_path_config("shipped")
    eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=3 * (64 + 15))
    result["ticks_64_sessions"] = bench_ticks(eng, cfg, 64, (0, 1, 2, 8, 32), args.reps)
    if not args.ticks_only:
        result["adapter_share_64_sessions"] = bench_adapter_share(eng, cfg, 64, (1, 8), 4 * args.reps)
        result["exact_streaming_188_chunks"] = bench_exact_streaming(eng, cfg)
    eng.close()
    if args.bench_ab:
        result["bench_ab"] = bench_ab(os.path.abspath(args.bench_ab), args.bench_steps, args.bench_warmup, args.ab_reps)
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
