"""Replaying recorded, VAD-annotated conversations through the gated scheduler (StreamScheduler.replay) on the shipped model in
bf16, against the two ways the project had before:

  * the push / tick loop, one tick per 160 ms chunk, with StreamScheduler(max_chunks=7, mixed_calls=True) -- the only exact
    path before replay: same blocks, labels and session state;
  * Engine.stream_steps_v of the same PCM -- every chunk encoded, no gating, no labels: the ungated ceiling.

1 and 16 sessions x 188 chunks (30 s) of seeded int16 audio on the device, with about half of the chunks speech and a speech
onset ('ipu_sl', which replays 6 history blocks) every 1-7 s.  Every leg starts from freshly reset sessions; the legs alternate
--reps times in one process after two warm-up rounds each (best and median ms, audio-s per s).  Writes one JSON file (--out)
that names the GPU, its power limit and its clocks, read in the same run."""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.scheduler import IPU_CONT, IPU_START, StreamScheduler  # noqa: E402
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


def conversation(rng, n):
    """Silences of 5-20 chunks and speech turns of 5-25 chunks opening with 'ipu_sl': about half speech."""
    out, speaking = [], rng.random() < 0.5
    while len(out) < n:
        out += [IPU_START] + [IPU_CONT] * rng.randint(4, 24) if speaking else [None] * rng.randint(5, 20)
        speaking = not speaking
    return out[:n]


def legs(eng, cfg, sch, n):
    keys = list(range(n))
    for k in keys:
        sch.open(k)
    ids = eng.alloc(n)
    g = torch.Generator().manual_seed(23 + n)
    pcm = torch.randint(-3000, 3000, (n, CHUNKS, cfg.samples_per_chunk), generator=g, dtype=torch.int32).to(torch.int16).cuda()
    rng = random.Random(n)
    statuses = [conversation(rng, CHUNKS) for _ in keys]
    blocks = {}

    def reset():
        for k in keys:
            sch.reset(k)

    def replay():
        reset()
        out = sch.replay({k: (pcm[k], statuses[k]) for k in keys})
        blocks["replay"] = sum(len(v) for v in out.values())

    def tick_loop():
        reset()
        count = 0
        for j in range(CHUNKS):
            for k in keys:
                sch.push(k, pcm[k, j], statuses[k][j])
            count += sum(len(v) for v in sch.tick().values())
        blocks["tick_loop"] = count

    def steps_v():
        eng.reset(ids)
        eng.stream_steps_v(ids, [CHUNKS] * n, pcm.view(n * CHUNKS, -1))
        blocks["stream_steps_v"] = n * CHUNKS

    def close():
        for k in keys:
            sch.close(k)
        eng.free(ids)

    speech = sum(s is not None for st in statuses for s in st) / (n * CHUNKS)
    onsets = sum(s == IPU_START for st in statuses for s in st)
    return {"replay": replay, "tick_loop": tick_loop, "stream_steps_v": steps_v}, blocks, close, speech, onsets


def bench(eng, cfg, sch, n, reps):
    fns, blocks, close, speech, onsets = legs(eng, cfg, sch, n)
    times = {k: [] for k in fns}
    for fn in fns.values():                                                   # warm-up: workspaces, graphs
        fn()
        fn()
    assert blocks["replay"] == blocks["tick_loop"], blocks
    for _ in range(reps):
        for k, fn in fns.items():
            times[k].append(timed(fn))
    out = {"sessions": n, "chunks": CHUNKS, "audio_s": n * CHUNKS * 0.16, "speech_share": speech, "onsets": onsets,
           "encoded_blocks": dict(blocks)}
    for k, v in times.items():
        best, med = min(v), statistics.median(v)
        out[k] = {"ms_best": best, "ms_median": med, "audio_s_per_s": out["audio_s"] / (best * 1e-3), "ms_all": v}
    close()
    print(json.dumps({k: (v if not isinstance(v, dict) or k == "encoded_blocks" else
                          {kk: vv for kk, vv in v.items() if kk != "ms_all"}) for k, v in out.items()}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_gated_replay.json"), help="JSON file to write")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sessions", type=int, nargs="+", default=[1, 16])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    result = {"gpu": gpu_info()}
    cfg = load_path_config("shipped")
    n_max = max(args.sessions)
    eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=2 * n_max + 16)
    sch = StreamScheduler(eng, history_chunks=10, onset_chunks=6, max_chunks=7, mixed_calls=True, max_sessions=n_max)
    result["pass_blocks"] = eng.get_option("steps_pass_blocks_in_use")
    result["runs"] = [bench(eng, cfg, sch, n, args.reps) for n in args.sessions]
    eng.close()
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
