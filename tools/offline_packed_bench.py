"""Ragged full-utterance encoding: padded fo_encode_offline against fo_encode_offline_packed on the same utterances, shipped
model in bf16 (SURVEY 8d config 4 and its ragged variant).

  * ragged: 256 utterances of seeded U[10, 30] s int16 audio; equal: 256 x 30 s, where the two entries do the same rows.
  * Each leg is fbank + encoder + adapter over the 256 utterances (audio on the device before timing):
    padded = per slice of --slice (as bench.py slices the padded batch), fbank_offline of the slice padded to its longest
    utterance, then encode_offline; packed = per slice, fbank_offline per utterance into one packed feature buffer, then
    encode_offline_packed; packed_pcm = per slice, one encode_offline_packed_pcm (fbank written onto the packed grid);
    corpus_pcm = ONE encode_offline_packed_pcm over all utterances, in passes at the default packed_pass_frames budget.
  * Every leg has an engine of its own (same weights), so fo_stats.device_bytes after a leg is that leg's footprint:
    weights plus the workspaces it grew (`device_bytes` per workload, read after its timed runs; the equal set runs second).
  * The legs alternate --reps times in one process after a warm-up each; best and median, audio-s per s of real audio.
  * rows: encoder rows each entry computes (padded B x T'_max per slice, packed sum T'_i); their ratio bounds the gain.

Writes one JSON file (--out) that names the GPU, its power limit and its clocks."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402


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


def legs(engs, cfg, seconds, slice_):
    sr = cfg.sample_rate
    g = torch.Generator().manual_seed(11)
    pcm = [(0.05 * torch.randn(int(s * sr), generator=g) * 32768).round().clamp(-32768, 32767).to(torch.int16).cuda() for s in seconds]
    slices = [list(range(i, min(i + slice_, len(pcm)))) for i in range(0, len(pcm), slice_)]
    # padded: each slice zero-padded to its longest utterance (ilens = the real frames)
    pad = []
    for sl in slices:
        n = max(pcm[i].numel() for i in sl)
        x = torch.zeros(len(sl), n, dtype=torch.int16, device="cuda")
        for j, i in enumerate(sl):
            x[j, :pcm[i].numel()] = pcm[i]
        il = np.array([1 + (pcm[i].numel() - cfg.frame_len) // cfg.frame_shift for i in sl], dtype=np.int32)
        pad.append((x, il))
    rows = {"padded": 0, "packed": 0}
    for x, il in pad:
        rows["padded"] += len(il) * cfg.sub_len(int(il.max()))
        rows["packed"] += int(sum(cfg.sub_len(int(t)) for t in il))

    def padded(eng=engs["padded"]):
        for x, il in pad:
            feats = eng.fbank_offline(x, 1.0)
            eng.encode_offline(feats, il, cfg.chunk_size, cfg.left_chunks)

    def packed(eng=engs["packed"]):
        for (x, il), sl in zip(pad, slices):
            feats = torch.cat([eng.fbank_offline(pcm[i][None], 1.0)[0] for i in sl])
            eng.encode_offline_packed(feats, il, cfg.chunk_size, cfg.left_chunks)

    flat = [torch.cat([pcm[i] for i in sl]) for sl in slices]
    counts = [np.array([pcm[i].numel() for i in sl], dtype=np.int64) for sl in slices]

    def packed_pcm(eng=engs["packed_pcm"]):
        for x, n in zip(flat, counts):
            eng.encode_offline_packed_pcm(x, cfg.chunk_size, cfg.left_chunks, 1.0, n_samples=n)

    corpus, corpus_n = torch.cat(flat), np.concatenate(counts)

    def corpus_pcm(eng=engs["corpus_pcm"]):
        eng.encode_offline_packed_pcm(corpus, cfg.chunk_size, cfg.left_chunks, 1.0, n_samples=corpus_n)

    return {"padded": padded, "packed": packed, "packed_pcm": packed_pcm, "corpus_pcm": corpus_pcm}, rows


def bench(engs, cfg, name, seconds, slice_, reps):
    fns, rows = legs(engs, cfg, seconds, slice_)
    times = {k: [] for k in fns}
    for fn in fns.values():
        fn()
    for _ in range(reps):
        for k, fn in fns.items():
            times[k].append(timed(fn))
    audio = float(sum(seconds))
    out = {"workload": name, "utterances": len(seconds), "audio_s": audio, "slice": slice_, "encoder_rows": rows,
           "row_ratio": rows["padded"] / rows["packed"]}
    for k, v in times.items():
        best = min(v)
        out[k] = {"ms_best": best, "ms_median": statistics.median(v), "audio_s_per_s": audio / (best * 1e-3), "ms_all": v,
                  "device_bytes": engs[k].stats()["device_bytes"]}
    out["speedup_best"] = out["padded"]["ms_best"] / out["packed"]["ms_best"]
    out["packed_pcm_vs_packed_best"] = out["packed"]["ms_best"] / out["packed_pcm"]["ms_best"]
    out["corpus_pcm_vs_packed_best"] = out["packed"]["ms_best"] / out["corpus_pcm"]["ms_best"]
    print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "ms_all"}) for k, v in out.items()}),
          flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--utterances", type=int, default=256)
    ap.add_argument("--slice", type=int, default=32)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    result = {"gpu": gpu_info()}
    cfg = load_path_config("shipped")
    esd, asd = make_encoder_state(cfg, 0), make_adapter_state(cfg, 0)
    engs = {k: Engine(cfg, esd, asd, dtype=torch.bfloat16, max_sessions=2) for k in ("padded", "packed", "packed_pcm", "corpus_pcm")}
    result["packed_pass_frames"] = engs["corpus_pcm"].get_option("packed_pass_frames")
    result["device_bytes_weights"] = {k: e.stats()["device_bytes"] for k, e in engs.items()}
    rng = np.random.default_rng(2024)
    ragged = [round(float(s), 2) for s in rng.uniform(10.0, 30.0, size=args.utterances)]
    result["runs"] = [bench(engs, cfg, "ragged_U10_30s", ragged, args.slice, args.reps),
                      bench(engs, cfg, "equal_30s", [30.0] * args.utterances, args.slice, args.reps)]
    for e in engs.values():
        e.close()
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
