#!/usr/bin/env python
"""Benchmark of the hot path: streamed audio-seconds per second through fbank -> CMVN -> encoder -> adapter.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload stream|latency|offline]
                    [--dump-outputs DIR]

One "step" = every session of the batch advances one 160 ms chunk (int16 PCM in, LLM-space embeddings out).
Workload at N=1 is BASELINE.json configs[1]: 64 concurrent sessions, synthetic 16 kHz audio, streaming chunks with
KV/CNN caches, bf16 context, shipped config with random-init weights.  With N>1 (torchrun, one rank per GPU) every
rank owns its own 64 sessions -- sessions are independent, so there is no collective on the data path (weak
scaling); NCCL only carries the barrier and the max-over-ranks timing reduction.
Other workloads (BASELINE.json configs 4 and 5) are selectable for the record: `--workload latency` (1 session,
p50/p99 per chunk) and `--workload offline` (full-utterance encode, batch x 30 s).

Output: ONE JSON line on rank 0: value (inputs resident in HBM), e2e (pinned-host PCM in, embeddings back to host,
through the C ABI), roofline of the dominant kernel class (the tcgen05 GEMM launches, timed with CUDA events on the
launching stream inside the library), cpu_baseline (the oracle port of the reference modules on the host cores,
bounded sample), clocks, gpu_launches.  `--impl reference` times the reference's CPU implementation of the same
step (oracle port; the reference is pure Python/PyTorch and cannot travel to the GPU box, see DESIGN.md section 8).
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from freeze_omni_b200.config import load_path_config  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402

METRIC = "streamed audio-sec/sec (encoder+adapter)"
UNIT = "audio-s/s"
CHUNK_SEC = 0.16
# SURVEY 8d: algorithmic FLOPs per session-chunk (2*M*N*K of the data-dependent contractions)
GFLOP_PER_CHUNK = 4.136
GFLOP_GEMM_PER_CHUNK = 4.136 - 0.0065 - 0.0401     # minus conv1 and the attention core (not GEMM launches)
DTYPE = "bf16w_x_fp16act_f32acc"          # what the tensor cores multiply (VERDICT r1 weak 7), not a precision claim
DTYPE_NOTE = ("weights rounded to bf16 (held in fp16 containers) x fp16 activations, fp32 accumulate (tcgen05 kind::f16); "
              "LayerNorm/softmax/residual fp32; fp16-range saturations are counted (fo_stats.act_saturations)")


def synth_pcm(n_sessions, n_chunks, samples_per_chunk, seed0=1000):
    """SURVEY 8d config 2: 0.1*N(0,1), band-limited, 200 ms silent gaps, int16-quantised."""
    out = np.empty((n_chunks, n_sessions, samples_per_chunk), dtype=np.int16)
    n = n_chunks * samples_per_chunk
    for s in range(n_sessions):
        g = torch.Generator().manual_seed(seed0 + s)
        x = 0.1 * torch.randn(n + 8, generator=g)
        x = torch.nn.functional.avg_pool1d(x.view(1, 1, -1), 5, 1).view(-1)[:n] * 2.0
        t = torch.arange(n)
        x = x * ((t // 3200) % 5 != 4).float()
        out[:, s, :] = torch.clamp((x * 32768.0).round(), -32768, 32767).to(torch.int16).view(n_chunks, -1).numpy()
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons sampled DURING the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                r = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if r.returncode == 0 and r.stdout.strip():
                    self.rows.append([c.strip() for c in r.stdout.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows)}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1400.0, 1590.0, "fallback"


def cpu_reference_step_rate(cfg, n_sessions, steps, warmup, threads=None, budget_s=None):
    """The reference's CPU implementation of one step (oracle port, fp32, torch CPU ops on all host threads):
    n_sessions lock-step sessions, fbank per session then batched encoder.infer + adapter -- the most favourable way
    to run the reference's modules (it batches when sessions are in lock step, SURVEY 8c).  With a time budget the run
    stops early (at least one timed step).  Returns (audio-s/s, seconds per step, threads, timed steps, warm-up steps)."""
    from oracle import freeze_omni_oracle as O
    if threads:
        torch.set_num_threads(threads)
    esd, asd = make_encoder_state(cfg, 0), make_adapter_state(cfg, 0)
    n_pcm = min(steps + warmup, 32)
    pcm = synth_pcm(n_sessions, n_pcm, cfg.samples_per_chunk)
    fronts = [O.StreamingFrontend(cfg.sample_rate, cfg.frame_length_ms, cfg.frame_shift_ms, cfg.frames_per_chunk,
                                  cfg.context_frames, cfg.feat_dim) for _ in range(n_sessions)]
    enc = O.EncoderOracle(cfg, esd)
    buf, cache, pe = enc.new_buffer(), None, 0
    times = []
    t_start = time.perf_counter()
    with torch.no_grad():
        for i in range(steps + warmup):
            t0 = time.perf_counter()
            j = i % n_pcm
            feats = torch.cat([fronts[s].process(torch.from_numpy(pcm[j, s].astype(np.float32)), 1.0) for s in range(n_sessions)])
            eo, buf, pe = enc.infer(feats, buf, pe)
            mask = torch.ones(n_sessions, 1, eo.size(1), dtype=torch.bool)
            y, _, cache = O.adapter_forward(cfg, asd, eo, mask, cache)
            times.append(time.perf_counter() - t0)
            if budget_s and len(times) > warmup and time.perf_counter() - t_start > budget_s:
                break
    warm = min(warmup, len(times) - 1)
    t = float(np.mean(times[warm:]))
    return n_sessions * CHUNK_SEC / t, t, torch.get_num_threads(), len(times) - warm, warm


def gpu_torch_reference_latency(cfg, steps, warmup):
    """The reference's GPU PyTorch path for one session (BASELINE.md 2b): the oracle port of its modules moved to the
    GPU, eager, under torch.autocast(bf16) as models/pipeline.py:67-68 runs them, batch 1 per call, including the
    per-chunk CPU sin/cos table + H2D copy of transformer.py:278-279.  CUDA-event time per chunk (ms)."""
    from oracle import freeze_omni_oracle as O
    dev = torch.device("cuda")
    esd = {k: v.to(dev) for k, v in make_encoder_state(cfg, 0).items()}
    asd = {k: v.to(dev) for k, v in make_adapter_state(cfg, 0).items()}
    enc = O.EncoderOracle(cfg, esd)
    g = torch.Generator().manual_seed(3)
    buf, cache, pe = enc.new_buffer(), None, 0
    lat = []
    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
        for i in range(steps + warmup):
            feats = (9.0 + 3.0 * torch.randn(1, cfg.chunk_feat_frames, cfg.feat_dim, generator=g)).to(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            eo, buf, pe = enc.infer(feats, buf, pe)
            mask = torch.ones(1, 1, eo.size(1), dtype=torch.bool, device=dev)
            y, _, cache = O.adapter_forward(cfg, asd, eo.float(), mask, cache)
            b.record()
            b.synchronize()
            if i >= warmup:
                lat.append(a.elapsed_time(b))
    lat = np.asarray(lat)
    return {"p50_ms": float(np.percentile(lat, 50)), "p99_ms": float(np.percentile(lat, 99)), "chunks": int(len(lat)),
            "what": "oracle port of the reference modules on the GPU, eager, autocast bf16, 1 session per call"}


def workload_text(S):
    return ("%d concurrent sessions per GPU, streaming 160 ms chunks with KV/CNN caches (windows full), shipped config "
            "(24x1024, adapter 3584), random-init weights" % S)


def run_reference(args, rank, world):
    if rank != 0:
        return
    cfg = load_path_config(args.config)
    n = min(args.sessions, args.ref_sessions)
    # the arm's own --steps / --warmup, cut short only by the time budget (a 64-session step is ~0.25 s on 16 cores)
    # all the host threads the box has (torchrun exports OMP_NUM_THREADS=1, which would starve the reference)
    v, t, th, steps, warm = cpu_reference_step_rate(cfg, n, max(1, args.steps), max(0, args.warmup), threads=os.cpu_count(),
                                                    budget_s=args.ref_budget)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warm, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload_text(n), "sessions_per_gpu": n,
                       "note": "reference CPU path: oracle port of the reference modules, torch CPU fp32, %d timed steps after %d warm-up "
                               "(requested %d / %d, time budget %d s)" % (steps, warm, args.steps, args.warmup, args.ref_budget)},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": th, "kind": "port",
                             "sample": "%d sessions x %d chunks (oracle port of the reference modules, fp32, torch CPU)" % (n, steps)},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def bench_offline(args, eng, cfg, rank, world, with_shapes=True):
    """BASELINE.json config 4: full-utterance encode, batch x 30 s synthetic audio, processed in slices (every rank its own
    batch).  Returns the result dict (rank 0 prints it or folds it into the line)."""
    B, sl = args.offline_batch, args.offline_slice
    n_samples = 30 * cfg.sample_rate
    g = torch.Generator().manual_seed(7 + rank)
    pcm = (0.05 * torch.randn(sl, n_samples, generator=g) * 32768).round().clamp(-32768, 32767).to(torch.int16).cuda()

    def one_pass(slices=B // sl):
        for _ in range(slices):
            feats = eng.fbank_offline(pcm, 1.0)
            il = np.full((sl,), feats.shape[1], dtype=np.int32)
            eng.encode_offline(feats, il, cfg.chunk_size, cfg.left_chunks)

    one_pass(2)                                               # warm-up: sizes the workspaces, first-use costs
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(1, args.offline_passes)
    e0.record()
    for _ in range(reps):
        one_pass()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    shapes = []
    if with_shapes:
        try:
            eng.set_option("profile_gemm", 1)
            one_pass(1)
            torch.cuda.synchronize()
            rows = eng.profile_dump()
            eng.set_option("profile_gemm", 0)
            for (m, n, k, cnt, us) in sorted(rows, key=lambda r: -r[4]):
                shapes.append({"M": m, "N": n, "K": k, "launches": cnt, "ms_total": us / 1e3, "tflops": 2.0 * m * n * k * cnt / us / 1e6})
        except Exception:
            pass
    _, tf_sus, _, _ = load_peaks()
    gflop = 773.0 * B                                         # SURVEY 8d: ~773 GFLOP per 30 s utterance (banded attention)
    out = {"workload": "offline full-utterance encode, batch %d x 30 s in slices of %d (BASELINE config 4)" % (B, sl),
           "metric": "offline audio-sec/sec (fbank+encoder+adapter)", "value": world * B * 30.0 / (ms * 1e-3),
           "unit": UNIT, "ms_per_pass": ms, "tflops": gflop / ms, "frac_of_sustained_bf16": gflop / ms / tf_sus,
           "n_gpus": world, "dtype": DTYPE}
    if shapes:
        out["gemm_ms_per_slice"] = sum(x["ms_total"] for x in shapes)
        out["gemm_shapes"] = shapes[:8]
    return out


def ragged_trace(total, seed=7):
    """SURVEY 8d config 3: ONE seeded trace of `total` sessions, lengths U[5 s, 120 s] rounded to chunks, arrivals spread over
    the first 16 s.  (arrive, end) in chunk steps."""
    rng = np.random.RandomState(seed)
    length = np.maximum(1, np.round(rng.uniform(5.0, 120.0, total) / CHUNK_SEC).astype(np.int64))
    arrive = rng.randint(0, 100, total)
    return arrive, arrive + length


def bench_ragged(args, eng, cfg, rank, world, dist, total=None, max_steps=None):
    """BASELINE.json config 3: the sessions of ONE trace are partitioned `id % world` over the ranks (pool.py:79-83 places
    sessions round-robin); every rank steps through the trace advancing ITS active sessions, the active set padded to a
    multiple of 16 with scratch sessions so that one captured graph serves each batch-size bucket.  Strong scaling: the
    same `total` sessions at every N; time = the slowest rank's CUDA-event time."""
    total = total or args.ragged_total
    bucket = 16
    arrive_all, end_all = ragged_trace(total)
    mine = np.arange(rank, total, world)
    arrive, end = arrive_all[mine], end_all[mine]
    S = len(mine)
    total_steps = int(end_all.max()) if max_steps is None else min(int(end_all.max()), max_steps)
    ids_all = eng.alloc(S + bucket)
    real, scratch = ids_all[:S], ids_all[S:]
    n_pcm = 16
    pcm_dev = torch.from_numpy(synth_pcm(min(S, 128) + bucket, n_pcm, cfg.samples_per_chunk, seed0=5000 + 4096 * rank)).cuda()
    P = pcm_dev.shape[1]
    t_enc, t_out = eng.out_frames(cfg.chunk_feat_frames)
    y_dev = torch.empty(S + bucket, t_out, cfg.llm_dim, device="cuda")
    # the per-step batches (ids, audio rows) are a function of the trace alone: build them before the clock starts
    plan = []
    for k in range(total_steps):
        act = np.nonzero((arrive <= k) & (k < end))[0]
        if len(act) == 0:
            plan.append(None)
            continue
        pad = (-len(act)) % bucket
        ids = np.concatenate([real[act], scratch[:pad]]).astype(np.int32)
        rows = torch.from_numpy(np.concatenate([act % (P - bucket), np.arange(P - bucket, P - bucket + pad)])).cuda()
        plan.append((ids, rows, len(act)))

    def step(k):
        if plan[k] is None:
            return 0
        ids, rows, n_act = plan[k]
        eng.stream_step(ids, pcm_dev[k % n_pcm].index_select(0, rows), 1.0, adapter_out=y_dev[:len(ids)], want_enc=False)
        return n_act

    # warm every bucket that occurs (eager + capture + replay), then reset the sessions and time the whole trace
    for n in sorted({len(p[0]) for p in plan if p is not None}):
        ids = np.concatenate([real[:min(n, S)], scratch[:n - min(n, S)]]).astype(np.int32)
        rows = torch.arange(n, device="cuda") % P
        for _ in range(3):
            eng.stream_step(ids, pcm_dev[0].index_select(0, rows), 1.0, adapter_out=y_dev[:n], want_enc=False)
    eng.reset(ids_all)
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    chunks = 0
    for k in range(total_steps):
        chunks += step(k)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
    tot = torch.tensor([float(chunks)], device="cuda")
    if dist is not None:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    eng.free(ids_all)
    return {"workload": "ragged: ONE trace of %d sessions (lengths U[5,120] s, seed 7, arrivals over the first 16 s) partitioned id %% world "
                        "= %d per GPU; active set padded to multiples of %d (BASELINE config 3)" % (total, S, bucket),
            "metric": METRIC, "value": float(tot.item()) * CHUNK_SEC / (float(ms.item()) * 1e-3), "unit": UNIT,
            "n_gpus": world, "steps": total_steps, "session_chunks": float(tot.item()), "ms_total": float(ms.item()),
            "mean_active_per_gpu": float(tot.item()) / world / max(1, total_steps), "scaling": "strong",
            "sessions_total": total, "dtype": DTYPE}


def bench_latency1(args, eng, cfg, chunks=300, warm=40, with_gpu_ref=True):
    """BASELINE.json config 5: ONE session, smallest chunk (19 fbank frames -> 4 encoder frames), warm caches, CUDA-event
    time from "chunk PCM resident on the device" to "adapter output written", p50 / p99; next to it the reference's GPU
    PyTorch path (oracle port of its modules on the GPU, eager, autocast bf16) on the same box."""
    ids = eng.alloc(1)
    pcm = torch.from_numpy(synth_pcm(1, 32, cfg.samples_per_chunk, seed0=900)).cuda()
    t_enc, t_out = eng.out_frames(cfg.chunk_feat_frames)
    y = torch.empty(1, t_out, cfg.llm_dim, device="cuda")
    st = torch.cuda.current_stream()
    lat = []
    for i in range(chunks + warm):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(st)
        eng.stream_step(ids, pcm[i % 32], 1.0, adapter_out=y, want_enc=False)
        b.record(st)
        b.synchronize()
        if i >= warm:
            lat.append(a.elapsed_time(b))
    # back to back (no host synchronisation between chunks): what the device needs per chunk
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for i in range(chunks):
        eng.stream_step(ids, pcm[i % 32], 1.0, adapter_out=y, want_enc=False)
    e1.record(st)
    torch.cuda.synchronize()
    eng.free(ids)
    lat = np.asarray(lat)
    hbm_peak, _, _, _ = load_peaks()
    floor_ms = (751.6e6 + 6.7e6) / (hbm_peak * 1e9) * 1e3
    out = {"workload": "1 session, 160 ms chunks, warm caches (BASELINE config 5)", "p50_ms": float(np.percentile(lat, 50)),
           "p99_ms": float(np.percentile(lat, 99)), "chunks": int(len(lat)), "back_to_back_ms": e0.elapsed_time(e1) / chunks,
           "hbm_floor_ms": floor_ms, "frac_of_hbm": floor_ms / float(np.percentile(lat, 50))}
    if with_gpu_ref:
        try:
            out["gpu_torch_baseline"] = gpu_torch_reference_latency(cfg, 120, 20)
        except Exception as ex:
            out["gpu_torch_baseline"] = {"error": str(ex)[:200]}
    return out


def parity_spot_check(eng, cfg, n_sessions, steps=3, sampled=(0, 1)):
    """The exact timed configuration (same context, n_sessions per step, same synthetic audio, graph replay) checked
    against the oracle OUTSIDE the timed region: `sampled` sessions run through per-session oracle sessions on the same
    bf16-rounded weights; returns the worst max-abs difference of encoder and adapter outputs."""
    from oracle import freeze_omni_oracle as O

    def bf16w(sd):
        keep = ("pos_bias", "conv.0.weight")
        return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}
    esd, asd = make_encoder_state(cfg, 0), make_adapter_state(cfg, 0)
    if eng.dtype == torch.bfloat16:
        esd, asd = bf16w(esd), bf16w(asd)
    torch.set_num_threads(os.cpu_count() or 8)
    ids = eng.alloc(n_sessions)
    pcm = synth_pcm(n_sessions, steps, cfg.samples_per_chunk, seed0=1000)
    oracle = {s: O.StreamSession(cfg, esd, asd) for s in sampled if s < n_sessions}
    we = wy = 0.0
    for i in range(steps):
        enc, y = eng.stream_step(ids, torch.from_numpy(pcm[i]).cuda(), 1.0)
        for s, o in oracle.items():
            _, eo, yo = o.step_pcm(torch.from_numpy(pcm[i, s].astype(np.float32)), 1.0)
            we = max(we, float((enc[s].cpu() - eo[0]).abs().max()))
            wy = max(wy, float((y[s].cpu() - yo[0]).abs().max()))
    eng.free(ids)
    return {"parity_maxabs": max(we, wy), "encoder": we, "adapter": wy, "tolerance": 2e-2 if eng.dtype == torch.bfloat16 else 1e-4,
            "what": "%d-session stream steps x %d (the timed configuration), sessions %s vs per-session oracle on the same "
                    "%s weights" % (n_sessions, steps, list(oracle), "bf16-rounded" if eng.dtype == torch.bfloat16 else "fp32")}


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each (sessions, ...) output as out_dir/<name>.npy in float32 so that two builds can be compared output for
    output.  Past DUMP_LIMIT bytes in all, the same seeded sample of session rows is kept of every array and its row
    numbers are written as out_dir/session_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    host = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    n = len(next(iter(host.values())))
    row_bytes = sum(a[0].nbytes for a in host.values())
    if n * row_bytes > DUMP_LIMIT:
        rows = np.sort(np.random.RandomState(0).choice(n, DUMP_LIMIT // row_bytes, replace=False))
        host = {k: a[rows] for k, a in host.items()}
        np.save(os.path.join(out_dir, "session_index.npy"), rows.astype(np.float64))
    for k, a in host.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def ncu_traffic():
    """dram__bytes_read+write per GEMM launch of a 64-session step from the committed ncu capture of THIS round's build
    (profiles/r02_ncu_gemm_dram_traffic_stream64.json written by tools/ncu_summary.py); None when absent."""
    p = os.path.join(ROOT, "profiles", "r02_ncu_gemm_dram_traffic_stream64.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p))
    return d.get("bytes_per_launch"), d.get("source")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="stream", choices=["stream", "latency", "offline", "ragged"])
    ap.add_argument("--sessions", type=int, default=64, help="concurrent sessions per GPU")
    ap.add_argument("--ref-sessions", type=int, default=64)
    ap.add_argument("--ref-budget", type=int, default=150, help="--impl reference: stop after this many seconds")
    ap.add_argument("--no-extras", action="store_true", help="skip the ragged1024 / latency1 / offline256 / parity legs of the line")
    ap.add_argument("--ragged-total", type=int, default=1024, help="sessions of the ONE ragged trace shared by all ranks")
    ap.add_argument("--offline-passes", type=int, default=1)
    ap.add_argument("--offline-batch", type=int, default=256)
    ap.add_argument("--offline-slice", type=int, default=32)
    ap.add_argument("--config", default="shipped")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"])
    ap.add_argument("--cpu-steps", type=int, default=6, help="bounded CPU sample (steps of the same workload)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--graph", type=int, default=-1, help="override the library's use_graph option")
    ap.add_argument("--backend", type=int, default=-1, help="override gemm_backend (0 FFMA, 1 tcgen05)")
    ap.add_argument("--groups", type=int, default=-1, help="override session_groups (parallel layer streams)")
    ap.add_argument("--debug-skip", type=int, default=0, help="timing attribution only: bitmask of kernel classes to skip")
    ap.add_argument("--quick", action="store_true", help="device-resident timing only")
    ap.add_argument("--opt", action="append", default=[], help="library option name=value (fo_set_option), repeatable")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (adapter_out, float32) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload in ("ragged", "offline")):
        ap.error("--dump-outputs covers the streaming path (--impl ours, --workload stream or latency)")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.workload == "latency":
        args.sessions = 1

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: freeze_omni_b200 has no CPU fallback")
    from freeze_omni_b200.engine import Engine
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    cfg = load_path_config(args.config)
    dtype = torch.bfloat16 if args.dtype == "bf16" else torch.float32
    S, K, W = args.sessions, args.steps, args.warmup
    extras = args.workload == "stream" and not args.no_extras and not args.quick and args.dtype == "bf16" and args.config == "shipped"
    per_rank_ragged = (args.ragged_total + world - 1) // world
    need = S + 1
    if extras or args.workload == "ragged":
        need = max(need, per_rank_ragged + 16 + 1)
    eng = Engine(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0), dtype=dtype, device=local_rank,
                 max_sessions=need, max_stream_frames=cfg.chunk_feat_frames)
    if args.graph >= 0:
        eng.set_option("use_graph", args.graph)
    if args.backend >= 0:
        eng.set_option("gemm_backend", args.backend)
    if args.groups >= 1:
        eng.set_option("session_groups", args.groups)
    if args.debug_skip:
        eng.set_option("debug_skip", args.debug_skip)
    for kv in args.opt:
        k, v = kv.split("=")
        eng.set_option(k, int(v))
    if args.workload == "ragged":
        res = bench_ragged(args, eng, cfg, rank, world, dist)
        if rank == 0:
            print(json.dumps(res))
        eng.close()
        if dist is not None:
            dist.destroy_process_group()
        return
    if args.workload == "offline":
        res = bench_offline(args, eng, cfg, rank, world)
        if rank == 0:
            print(json.dumps(res))
        eng.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    ids = eng.alloc(S)
    n_pcm = 64                                               # synthetic audio is cycled after 64 chunks
    pcm_host = torch.from_numpy(synth_pcm(S, n_pcm, cfg.samples_per_chunk, seed0=1000 + 4096 * rank)).pin_memory()
    pcm_dev = pcm_host.cuda(non_blocking=True)
    t_enc, t_out = eng.out_frames(cfg.chunk_feat_frames)
    y_dev = torch.empty(S, t_out, cfg.llm_dim, device="cuda")
    y_host = torch.empty(S, t_out, cfg.llm_dim).pin_memory()
    stream = torch.cuda.current_stream()

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(n_steps, host_io, first):
        for i in range(n_steps):
            j = (first + i) % n_pcm
            if host_io:
                eng.stream_step(ids, pcm_host[j], 1.0, adapter_out=y_host, want_enc=False)
                stream.synchronize()                         # a server needs the embeddings every chunk
            else:
                eng.stream_step(ids, pcm_dev[j], 1.0, adapter_out=y_dev, want_enc=False)

    y_host2 = torch.empty(S, t_out, cfg.llm_dim).pin_memory()

    def run_steps_pipelined(n_steps, first):
        """fo_stream_step_async: the upload of chunk i+1 and the read-back of chunk i overlap the kernels in between; the
        host still takes delivery of every chunk's embeddings, one step behind the launch."""
        prev = None
        for i in range(n_steps):
            j = (first + i) % n_pcm
            tk = eng.stream_step_async(ids, pcm_host[j], y_host if i & 1 else y_host2, 1.0)
            if prev is not None:
                eng.stream_wait(prev)
            prev = tk
        if prev is not None:
            eng.stream_wait(prev)

    def timed_pipelined(n_steps, first):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_steps_pipelined(n_steps, first)                  # returns after the last read-back has landed
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    def timed(n_steps, host_io, first):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        run_steps(n_steps, host_io, first)
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    # ---- device-resident throughput ------------------------------------------------------------
    run_steps(max(0, 17 - W), False, 0)                      # untimed: fill the 64-row KV windows (steady state)
    run_steps(W, False, 0)
    sampler = ClockSampler(local_rank)
    sampler.start()
    l0 = eng.stats()["kernel_launches"]
    ms = timed(K, False, W)
    launches = eng.stats()["kernel_launches"] - l0
    value = world * S * CHUNK_SEC * K / (ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"adapter_out": y_dev})      # y_dev holds the last timed step's embeddings
    if args.quick:
        sampler.stop_flag = True
        if rank == 0:
            print(json.dumps({"quick": True, "ms_per_step": ms / K, "value": value, "sessions": S, "debug_skip": args.debug_skip,
                              "groups": eng.get_option("session_groups")}))
        eng.free(ids)
        eng.close()
        if dist is not None:
            dist.destroy_process_group()
        return

    # ---- end to end through the C ABI with host buffers -------------------------------------------
    run_steps(W, True, 0)
    ms_e2e_sync = timed(K, True, W)                          # every step: upload, kernels, read-back, host synchronisation
    run_steps_pipelined(max(W, 6), 0)                        # both staging-buffer parities warmed and captured
    ms_e2e = timed_pipelined(K, W)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    e2e = world * S * CHUNK_SEC * K / (ms_e2e * 1e-3)
    e2e_sync = world * S * CHUNK_SEC * K / (ms_e2e_sync * 1e-3)

    # ---- per-step latency distribution (device timed, one event pair per step) --------------------
    lat = []
    for i in range(min(K, 200)):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        run_steps(1, False, i)
        b.record(stream)
        b.synchronize()
        lat.append(a.elapsed_time(b))
    lat = np.asarray(lat)

    # ---- roofline of the dominant kernel class (the tcgen05 GEMM launches).  Their time inside a step is measured
    # differentially with CUDA events on the launching stream: K graph-replayed steps with every kernel, minus K steps
    # with exactly the GEMM launches dropped (library option debug_skip=32; outputs of that pass are discarded).
    # Per-shape rates come from event pairs around each eager launch (they include ~3 us of event/launch overhead per
    # launch, so they are lower bounds on the rates).
    hbm_peak, tf_sustained, tf_burst, peak_kind = load_peaks()
    step_ms = ms / K
    roof, shapes = None, []
    try:
        eng.set_option("debug_skip", 32)
        run_steps(3, False, 0)
        ms_nogemm = timed(K, False, 3) / K
        eng.set_option("debug_skip", args.debug_skip)
        eng.reset(ids)                                               # the skipped pass left garbage in the session state
        run_steps(18, False, 0)
        gemm_ms = max(step_ms - ms_nogemm, 1e-6)
        steps_prof = min(K, 10)
        eng.set_option("profile_gemm", 1)
        run_steps(steps_prof, False, 0)
        torch.cuda.synchronize()
        rows = eng.profile_dump()
        eng.set_option("profile_gemm", 0)
        gemm_n = sum(r[3] for r in rows)
        gflop = GFLOP_GEMM_PER_CHUNK * S
        achieved = gflop / gemm_ms                                  # GFLOP / ms == TFLOP/s
        roof = {"bound": "tensor", "achieved": achieved, "peak": tf_sustained, "unit": "TFLOP/s",
                "frac": achieved / tf_sustained,
                # M = 256 rows sits on the ridge: both bounds reported (VERDICT r1 item 3)
                "frac_tensor": achieved / tf_sustained, "frac_hbm": 751.6e-3 / gemm_ms * 1e3 / hbm_peak,
                "algorithmic_bytes_per_launch": 751.6e6 / max(1, gemm_n // steps_prof),
                # dram__bytes_read+write per GEMM launch of a 64-session step from the committed ncu capture of this round's
                # build (None when the capture is absent or the shape differs)
                "traffic": (ncu_traffic()[0] if S == 64 else None), "traffic_source": (ncu_traffic()[1] if S == 64 else None),
                "traffic_unit": "bytes per launch (ncu)",
                "peak_source": peak_kind + " (sustained bf16 cuBLAS)",
                "kernel": "gemm_tc_kernel (all %d GEMM launches of a step; algorithmic %.2f GFLOP per session-chunk)"
                          % (gemm_n // steps_prof, GFLOP_GEMM_PER_CHUNK),
                "launches_per_step": gemm_n / steps_prof, "gemm_ms_per_step": gemm_ms, "ms_per_step_without_gemms": ms_nogemm,
                "share_of_step": gemm_ms / step_ms,
                "weights_GBs": 751.6e-3 / gemm_ms * 1e3, "weights_frac_of_hbm": 751.6e-3 / gemm_ms * 1e3 / hbm_peak,
                "note": "M = 4 rows per session puts the layer GEMMs on the weight-streaming / latency side of the ridge "
                        "(each launch is 6-12 us of pipeline fill, L2->SM ingest and epilogue, two CTAs per SM overlapping each other; the "
                        "split-K sums of out-proj / FFN2 are finished by the LayerNorm that follows); gemm_shapes gives per-shape "
                        "rates, conv2 (M = sessions*80 padded rows) is the tensor-bound one; ncu capture in profiles/"}
        for (m, n, k, cnt, us) in sorted(rows, key=lambda r: -r[4]):
            shapes.append({"M": m, "N": n, "K": k, "launches_per_step": cnt / steps_prof, "us_per_launch_eager_events": us / cnt,
                           "tflops": 2.0 * m * n * k * cnt / us / 1e6, "weight_GBs": 2.0 * n * k * cnt / us / 1e3})
    except Exception as ex:  # library built without the profiling options
        roof = {"bound": "tensor", "achieved": None, "peak": tf_sustained, "unit": "TFLOP/s", "frac": None,
                "traffic": None, "note": "gemm profiling unavailable: %s" % ex}
    step_bytes = 751.6e6 + S * 6.7e6
    whole = {"tflops": GFLOP_PER_CHUNK * S / step_ms, "frac_of_sustained_bf16": GFLOP_PER_CHUNK * S / step_ms / tf_sustained,
             "algorithmic_GB_per_step": step_bytes / 1e9, "hbm_gbs": step_bytes / 1e6 / step_ms,
             "frac_of_hbm": step_bytes / 1e6 / step_ms / hbm_peak}

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload ----------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, t, th, _, _ = cpu_reference_step_rate(cfg, S, args.cpu_steps, 1, threads=os.cpu_count())
        cpu = {"value": v, "unit": UNIT, "cores": th, "kind": "port",
               "sample": "%d sessions x %d chunks, oracle port of the reference modules (fp32 torch CPU), %.2f s/step" % (S, args.cpu_steps, t)}

    gpu_ref = None
    if rank == 0 and world == 1 and args.workload == "latency":
        try:
            gpu_ref = gpu_torch_reference_latency(cfg, 200, 30)
        except Exception as ex:
            gpu_ref = {"error": str(ex)[:200]}
    # ---- the other BASELINE.json configs, same context, outside the timed region of `value` (VERDICT r1 item 4) ----------
    eng.free(ids)
    ids = np.zeros(0, np.int32)
    parity = latency1 = offline256 = ragged1024 = None
    if extras:
        def guarded(fn):
            try:
                return fn()
            except Exception as ex:
                return {"error": str(ex)[:300]}
        if world == 1:
            parity = guarded(lambda: parity_spot_check(eng, cfg, S))
            latency1 = guarded(lambda: bench_latency1(args, eng, cfg))
            offline256 = guarded(lambda: bench_offline(args, eng, cfg, rank, world, with_shapes=False))
        ragged1024 = bench_ragged(args, eng, cfg, rank, world, dist)       # collective inside: every rank, no guard
    if rank == 0:
        h2d = S * cfg.samples_per_chunk * 2 + S * 4
        d2h = S * t_out * cfg.llm_dim * 4
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": DTYPE if args.dtype == "bf16" else "f32",
                "dtype_note": DTYPE_NOTE if args.dtype == "bf16" else "fp32 FFMA",
                "data": "synthetic",
                "config": {"workload": workload_text(S), "sessions_per_gpu": S,
                           "parallelism": "sessions sharded over ranks, no collective",
                           "l2": "inputs larger than L2: each step streams 752 MB of weights + %.0f MB of KV rings (L2 is 126 MB)" % (S * 6.3)},
                "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / K,
                        "how": "fo_stream_step_async + fo_stream_wait: pinned-host int16 PCM in, fp32 embeddings back to the host "
                               "every step; uploads and read-backs on the library's own two copy streams, overlapping the neighbouring steps' kernels (this loop therefore hides the staging copies that the device-resident loop of `value` runs in-stream)",
                        "sync_each_step": {"value": e2e_sync, "ms_per_step": ms_e2e_sync / K,
                                           "how": "fo_stream_step with host buffers + stream synchronisation after every step"}},
                "gpu_launches": int(launches),
                "latency_ms": {"p50": float(np.percentile(lat, 50)), "p99": float(np.percentile(lat, 99)), "sessions": S},
                "roofline": roof, "gemm_shapes": shapes[:12], "step_roofline": whole, "cpu_baseline": cpu,
                "gpu_torch_baseline": gpu_ref if gpu_ref is not None else (latency1 or {}).get("gpu_torch_baseline"),
                "parity": parity, "parity_maxabs": (parity or {}).get("parity_maxabs"),
                "latency1": latency1, "offline256": offline256, "ragged1024": ragged1024,
                "clocks": sampler.summary(),
                "options": {"gemm_backend": eng.get_option("gemm_backend"), "use_graph": eng.get_option("use_graph"),
                            "session_groups": eng.get_option("session_groups")}}
        print(json.dumps(line))
    if len(ids):
        eng.free(ids)
    eng.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
