"""The LLM hand-off of a gated replay (StreamScheduler.replay(handoff=)) on the shipped model in bf16, against what a caller had
to do before it:

  * replay(handoff=ho): every window's encoder call writes the blocks' fp16 LLM rows, mask rows and start rows on the device;
  * replay() followed by the torch hand-off per block into the same kind of buffers -- the reference's
    cat(prefix, y) / .half() / mask sequence (models/audioLLM.py:404-411), one block at a time;
  * replay() alone: the floor.

1 and 16 sessions x 188 chunks (30 s) of the seeded recordings tools/gated_replay_bench.py generates (about half speech, an
onset every few seconds).  Every leg starts from freshly reset sessions; the legs alternate --reps times in one process after
two warm-up rounds each (best and median ms).  The two hand-off legs must leave bit-identical buffers.  Writes one JSON file
(--out) that names the GPU, its power limit and its clocks, read in the same run."""
import argparse
import json
import os
import random
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from gated_replay_bench import CHUNKS, conversation, gpu_info, timed  # noqa: E402
from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.scheduler import IPU_START, Handoff, StreamScheduler, plan_gated_replay  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402

PREFIX = 8                        # chat-prefix rows in front of an onset block


def bench(eng, cfg, sch, n, reps):
    keys = list(range(n))
    for k in keys:
        sch.open(k)
    # the recordings of gated_replay_bench.legs(n): same seeds, same generator
    g = torch.Generator().manual_seed(23 + n)
    pcm = torch.randint(-3000, 3000, (n, CHUNKS, cfg.samples_per_chunk), generator=g, dtype=torch.int32).to(torch.int16).cuda()
    rng = random.Random(n)
    statuses = [conversation(rng, CHUNKS) for _ in keys]
    rec = {k: (pcm[k], statuses[k]) for k in keys}
    total = sum(len(plan_gated_replay(s, sch.history_chunks, sch.onset_chunks).blocks) for s in statuses)
    gp = torch.Generator().manual_seed(5)
    prefix = torch.randn(1, PREFIX, cfg.llm_dim, generator=gp)
    pmask = (torch.rand(PREFIX, generator=gp) > 0.2).to(torch.uint8)
    fused, manual = Handoff(eng, total, prefix, pmask), Handoff(eng, total, prefix, pmask)
    t_out = fused.rows - PREFIX
    dev = eng.torch_device
    prefix16, pmask_d = prefix[0].to(dev).half(), pmask.to(dev)
    ones = torch.ones(t_out, dtype=torch.uint8, device=dev)

    def reset():
        for k in keys:
            sch.reset(k)

    def replay_handoff():
        reset()
        sch.replay(rec, handoff=fused)

    def replay_torch_handoff():
        reset()
        out = sch.replay(rec)
        b, starts = 0, []
        for k in keys:                      # any block order will do; the fused leg's is window by window
            for blk in out.get(k, []):
                y16 = blk.emb.half()                                              # audioLLM.py:410
                if blk.status == IPU_START:                                       # audioLLM.py:404-406
                    manual.embeds[b].copy_(torch.cat((prefix16, y16), 0))
                    manual.attn_mask[b].copy_(torch.cat((pmask_d, ones), 0))
                    starts.append(0)
                else:
                    manual.embeds[b, PREFIX:].copy_(y16)
                    manual.attn_mask[b].copy_(torch.cat((torch.zeros_like(pmask_d), ones), 0))
                    starts.append(PREFIX)
                b += 1
        manual.row_start[:b].copy_(torch.tensor(starts, dtype=torch.int32))

    def replay_only():
        reset()
        sch.replay(rec)

    fns = {"replay_handoff": replay_handoff, "replay_torch_handoff": replay_torch_handoff, "replay": replay_only}
    for fn in fns.values():                                                   # warm-up: workspaces, pinned tables
        fn()
        fn()
    # same rows, masks and starts, up to the block order: sort both by (embeds, mask) bytes of each block
    torch.cuda.synchronize()

    def canon(h):
        e, m, r = h.embeds.cpu().view(torch.int16).numpy(), h.attn_mask.cpu().numpy(), h.row_start.cpu().tolist()
        return sorted((e[b].tobytes() + m[b].tobytes(), r[b]) for b in range(total))
    identical = canon(fused) == canon(manual)
    assert identical, "the fused hand-off differs from the torch sequence"
    times = {k: [] for k in fns}
    for _ in range(reps):
        for k, fn in fns.items():
            times[k].append(timed(fn))
    out = {"sessions": n, "chunks": CHUNKS, "audio_s": n * CHUNKS * 0.16, "blocks": total, "prefix_rows": PREFIX,
           "handoff_bytes": total * t_out * cfg.llm_dim * (4 + 2), "bit_identical": identical}
    for k, v in times.items():
        out[k] = {"ms_best": min(v), "ms_median": statistics.median(v), "ms_all": v}
    for k in keys:
        sch.close(k)
    print(json.dumps({k: (v if not isinstance(v, dict) else {kk: vv for kk, vv in v.items() if kk != "ms_all"})
                      for k, v in out.items()}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_replay_handoff.json"), help="JSON file to write")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sessions", type=int, nargs="+", default=[1, 16])
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    result = {"gpu": gpu_info()}
    cfg = load_path_config("shipped")
    n_max = max(args.sessions)
    eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=torch.bfloat16, max_sessions=n_max + 16)
    sch = StreamScheduler(eng, history_chunks=10, onset_chunks=6, max_sessions=n_max)
    result["pass_blocks"] = eng.get_option("steps_pass_blocks_in_use")
    result["runs"] = [bench(eng, cfg, sch, n, args.reps) for n in args.sessions]
    eng.close()
    result["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
