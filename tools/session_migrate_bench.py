"""Session snapshots (Engine.save_sessions / restore_sessions) on the shipped model in bf16: what moving a conversation costs.

For n = 1, 16 and 64 sessions, each saturated (n_frames past the KV window, the window wrapping the ring's end, so every
record row is a real ring row):
  * save and restore device to device, CUDA events around `--reps` calls after warm-up;
  * save into and restore from pinned host memory (the staged path), CUDA events likewise; the rate reported is that of the
    host link, which carries each record once;
  * with two visible GPUs: save on device 0, peer copy, restore on device 1, host clock around the synchronised sequence.
A restore's time includes its header read-back and stream sync; a save into host memory its stream sync.
Bytes: a save reads the KV window + fp32 sections and writes the record, a restore the reverse, so 2 x n x record bytes of HBM
traffic each (the header and zero rows past a short window are a rounding error here).  GB/s over that, and its fraction of
the HBM figure bench.py's load_peaks() uses (named in the output).  The n = 1 and 16 working sets (6 and 100 MB) fit the
126 MB L2; n = 64 (400 MB) does not.
For comparison, one session through the per-layer reference-layout calls (24 x fo_session_export_kv + 24 x
fo_session_import_kv, adapter cache, n_frames, pe_index), host clock.
Writes one JSON file (--out) that names the GPU and its power limit (nvidia-smi, read-only query, same run)."""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import load_peaks  # noqa: E402
from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.engine import Engine  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402

SIZES = (1, 16, 64)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def event_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def saturate(eng, ids, frames):
    """Sessions with `frames` encoder frames behind them (ring contents as left by the engine; the copy moves them all)."""
    for s in ids:
        eng.set_frames(int(s), frames)


def case(n, path, ms, rec_bytes, peak):
    if "host" in path:    # bound by the host link, which carries the records once: its rate, not a share of HBM
        return {"n": n, "path": path, "ms": round(ms, 4), "host_link_gbs": round(n * rec_bytes / (ms * 1e-3) / 1e9, 1)}
    gbs = 2.0 * n * rec_bytes / (ms * 1e-3) / 1e9
    return {"n": n, "path": path, "ms": round(ms, 4), "hbm_gbs": round(gbs, 1), "frac_hbm_peak": round(gbs / peak, 3)}


def legacy_one_session(eng, cfg, src, dst, reps):
    """The per-layer reference-layout export / import loop, one session."""
    def once():
        nf, pe = eng.state(int(src))
        eng.set_frames(int(dst), nf)
        for li in range(cfg.n_layers):
            k, v = eng.export_kv(int(src), li)
            eng.import_kv(int(dst), li, k, v)
        eng.import_adapter_cache(int(dst), eng.export_adapter_cache(int(src)))
        eng.set_pe_index([int(dst)], pe)
    once()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="JSON file to write")
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    hbm, _, _, peak_src = load_peaks()
    result = {"gpu": gpu_info(), "model": "shipped, bf16", "hbm_peak_gbs": hbm,
              "hbm_peak_figure": "bench.py load_peaks() hbm_gbs (%s)" % peak_src, "cases": []}
    cfg = load_path_config("shipped")
    esd, asd = make_encoder_state(cfg, 0), make_adapter_state(cfg, 0)
    cap_n = max(SIZES)
    src = Engine(cfg, esd, asd, dtype=torch.bfloat16, max_sessions=cap_n + 1)
    dst = Engine(cfg, esd, asd, dtype=torch.bfloat16, max_sessions=cap_n + 3)
    B = src.snapshot_bytes
    result["bytes_per_session"] = B
    result["ring_cap"] = src.get_option("ring_cap")
    frames = cfg.kv_window + 36                       # (frames - window) % ring_cap + window > ring_cap: two runs per unit
    a, b = src.alloc(cap_n), dst.alloc(cap_n)
    saturate(src, a, frames)
    pinned = torch.empty(cap_n, B, dtype=torch.uint8).pin_memory()
    for n in SIZES:
        blob = src.save_sessions(a[:n])
        result["cases"].append(case(n, "save_device", event_ms(lambda: src.save_sessions(a[:n], out=blob), args.reps), B, hbm))
        result["cases"].append(case(n, "restore_device", event_ms(lambda: dst.restore_sessions(b[:n], blob), args.reps), B, hbm))
        host = pinned[:n]
        result["cases"].append(case(n, "save_pinned_host", event_ms(lambda: src.save_sessions(a[:n], out=host), args.reps), B, hbm))
        result["cases"].append(case(n, "restore_pinned_host", event_ms(lambda: dst.restore_sessions(b[:n], host), args.reps), B, hbm))
        print(json.dumps(result["cases"][-4:]), flush=True)
    if torch.cuda.device_count() >= 2:
        far = Engine(cfg, esd, asd, dtype=torch.bfloat16, device=1, max_sessions=cap_n + 3)
        c = far.alloc(cap_n)
        for n in SIZES:
            def move():
                far.restore_sessions(c[:n], src.save_sessions(a[:n]).to(far.torch_device))
            move()
            torch.cuda.synchronize(0)
            torch.cuda.synchronize(1)
            t0 = time.perf_counter()
            for _ in range(args.reps):
                move()
            torch.cuda.synchronize(0)
            torch.cuda.synchronize(1)
            ms = (time.perf_counter() - t0) * 1e3 / args.reps
            result["cases"].append({"n": n, "path": "save_peer_copy_restore_gpu0_to_gpu1", "ms": round(ms, 4),
                                    "mb_per_s_moved": round(n * B / (ms * 1e-3) / 1e6, 1)})
        far.close()
    else:
        result["across_gpus"] = "not measured: one GPU visible"
    result["legacy_per_layer_one_session_ms"] = round(legacy_one_session(src, cfg, a[0], a[1], 5), 3)
    src.close()
    dst.close()
    result["gpu_after"] = gpu_info()
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
