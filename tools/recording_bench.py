"""Exact-streaming encoding of recorded audio (Engine.stream_steps_v) on the shipped model in bf16, against the two ways the
project had before: the k = 16 loop of multi_chunk_bench's bench_exact_streaming (encode_stream_chunks over features, 12
calls per 30 s) and fo_encode_offline of the same audio (the ceiling; its rel-pos offsets differ from streaming after chunk
16, SURVEY 2.4-1, so its outputs are not comparable).

  * 1 and 16 sessions x 188 chunks (30 s) of seeded int16 audio, device buffers; the three legs alternated --reps times in
    one process after one warm-up round each (best and median ms, audio-s per s).  stream_steps_v includes the fbank; the
    k = 16 loop and offline start from features computed beforehand.
  * --profile: a separate run with torch.profiler around one stream_steps_v call per session count, programmatic dependent
    launch off: device time per kernel name, and the share of the pass attention (attention_chunks*) and its separate ring append
    (chunks_append_ring*, launched when a session spreads over several CTAs of a head).

Writes one JSON file (--out) that names the GPU, its power limit and its clocks."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402

CHUNKS = 188                      # 30 s of 160 ms chunks


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3


def legs(eng, cfg, n):
    ids = eng.alloc(n)
    g = torch.Generator().manual_seed(17 + n)
    pcm = torch.randint(-3000, 3000, (n, CHUNKS, cfg.samples_per_chunk), generator=g, dtype=torch.int32).to(torch.int16)
    pcm = pcm.cuda()
    flat = pcm.view(n * CHUNKS, -1)
    feats_off = eng.fbank_offline(pcm.view(n, -1))                           # (n, frames, F)
    ilens = torch.full((n,), feats_off.shape[1], dtype=torch.int32)
    gf = torch.Generator().manual_seed(9)
    feats = (9.0 + 3.0 * torch.randn(n, CHUNKS, cfg.chunk_feat_frames, cfg.feat_dim, generator=gf)).cuda()
    t, t_out = eng.out_frames(cfg.chunk_feat_frames)
    enc = torch.empty(n * CHUNKS, t, cfg.d_model, device="cuda")
    y = torch.empty(n * CHUNKS, t_out, cfg.llm_dim, device="cuda")

    def steps_v():
        eng.reset(ids)
        eng.stream_steps_v(ids, [CHUNKS] * n, flat, enc_out=enc, adapter_out=y)

    def k16():
        eng.reset(ids)
        for c0 in range(0, CHUNKS, 16):
            eng.encode_stream_chunks(ids, feats[:, c0:c0 + 16].contiguous())

    def offline():
        eng.encode_offline(feats_off, ilens)

    return ids, {"stream_steps_v": steps_v, "k16_loop": k16, "offline": offline}


def bench(eng, cfg, n, reps):
    ids, fns = legs(eng, cfg, n)
    times = {k: [] for k in fns}
    for k, fn in fns.items():                                                  # warm-up: workspaces, graphs
        fn()
        fn()
    for _ in range(reps):
        for k, fn in fns.items():
            times[k].append(timed(fn))
    out = {"sessions": n, "chunks": CHUNKS, "audio_s": n * CHUNKS * 0.16}
    for k, v in times.items():
        best, med = min(v), statistics.median(v)
        out[k] = {"ms_best": best, "ms_median": med, "audio_s_per_s": out["audio_s"] / (best * 1e-3), "ms_all": v}
    eng.free(ids)
    print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "ms_all"}) for k, v in out.items()}),
          flush=True)
    return out


def profile(eng, cfg, n):
    from torch.profiler import ProfilerActivity, profile as tprofile
    ids, fns = legs(eng, cfg, n)
    eng.set_option("pdl", 0)          # a kernel's device time then excludes its wait for the one before it
    fns["stream_steps_v"]()
    torch.cuda.synchronize()
    with tprofile(activities=[ProfilerActivity.CUDA]) as prof:
        fns["stream_steps_v"]()
        torch.cuda.synchronize()
    per = {}
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and e.device_time_total > 0:
            per[e.name] = per.get(e.name, 0.0) + e.device_time_total
    total = sum(per.values())
    attn = sum(v for k, v in per.items() if "attention_chunks" in k)
    append = sum(v for k, v in per.items() if "chunks_append_ring" in k)
    top = sorted(per.items(), key=lambda kv: -kv[1])[:15]
    eng.set_option("pdl", 1)
    eng.free(ids)
    out = {"sessions": n, "kernel_us_total": total, "attention_steps_us": attn, "attention_steps_share": attn / total if total else 0.0,
           "ring_append_us": append, "top_kernels_us": [[k[:120], v] for k, v in top]}
    print(json.dumps({k: v for k, v in out.items() if k != "top_kernels_us"}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sessions", type=int, nargs="+", default=[1, 16])
    ap.add_argument("--profile", action="store_true", help="torch.profiler kernel split of one call instead of the timing legs")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    result = {"gpu": gpu_info()}
    cfg = load_path_config("shipped")
    eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=2 * max(args.sessions))
    result["pass_blocks"] = eng.get_option("steps_pass_blocks")
    if args.profile:
        result["profile"] = [profile(eng, cfg, n) for n in args.sessions]
    else:
        result["runs"] = [bench(eng, cfg, n, args.reps) for n in args.sessions]
    eng.close()
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
