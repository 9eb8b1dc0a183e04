"""Contexts on a group of the GPU's SMs (fo_create_on_sms, Engine(sm_partition=(split, group))): where their work runs,
launched directly and replayed from a captured graph as a streaming step is; that every path is within the oracle's bar
(the streaming step, the multi-chunk and recording calls with the hand-off, packed offline PCM; the scheduler's tick and
replay against a whole-device twin); that two contexts streaming at once on one GPU give bit for bit what each gives
alone; and that sessions move between partitioned and whole-device contexts."""
import threading

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config
from freeze_omni_b200.scheduler import IPU_CONT, IPU_START, StreamScheduler
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
from oracle import freeze_omni_oracle as O

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
BF16_TOL = 2e-2
TWIN_BF16_TOL = 4e-3            # bf16 twins that differ in GEMM plans (split-K order): the bar of the multi-chunk tests


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def engine(name, seed, dtype, sm_partition=None, max_sessions=8):
    from freeze_omni_b200.engine import Engine
    cfg = load_path_config(name)
    return cfg, Engine(cfg, make_encoder_state(cfg, seed), make_adapter_state(cfg, seed), dtype=dtype, max_sessions=max_sessions,
                       sm_partition=sm_partition)


def bf16_weights(sd):
    keep = ("pos_bias", "conv.0.weight")
    return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}


def pcm_chunks(cfg, n, k, seed):
    g = torch.Generator().manual_seed(seed)
    return [(0.05 * torch.randn(n, cfg.samples_per_chunk, generator=g) * 32768).round().clamp(-32768, 32767).to(torch.int16)
            for _ in range(k)]


@pytest.fixture(scope="module")
def user():
    cfg, eng = engine("shipped", 0, torch.bfloat16, (2, 0), max_sessions=130)
    yield cfg, eng
    eng.close()


@pytest.fixture(scope="module")
def system():
    cfg, eng = engine("shipped", 1, torch.bfloat16, (2, 1), max_sessions=130)
    yield cfg, eng
    eng.close()


@pytest.fixture(scope="module")
def whole():
    cfg, eng = engine("shipped", 0, torch.bfloat16, None, max_sessions=130)
    yield cfg, eng
    eng.close()


# ---- 1. where the work runs --------------------------------------------------------------------------------------------------
def test_groups_are_disjoint_and_smaller_than_the_device(user, system, whole):
    """Direct launches, and launches captured on the capture stream and replayed on the execution stream (the form every
    streaming step takes after its first calls), run inside the context's group; the groups are disjoint."""
    a, b, w = user[1], system[1], whole[1]
    assert a.sm_count % 8 == 0 and b.sm_count % 8 == 0 and 8 <= a.sm_count <= 74 and 8 <= b.sm_count <= 74
    assert w.sm_count == torch.cuda.get_device_properties(0).multi_processor_count
    n = 4 * w.sm_count
    sa, sb, sw = (set(e.debug_sm_ids(n).cpu().tolist()) for e in (a, b, w))
    ga, gb, gw = (set(e.debug_sm_ids(n, graph=True).cpu().tolist()) for e in (a, b, w))
    print("SM ids seen: group 0 %d (%d..%d), group 1 %d (%d..%d), whole device %d; replayed graphs: %d, %d, %d"
          % (len(sa), min(sa), max(sa), len(sb), min(sb), max(sb), len(sw), len(ga), len(gb), len(gw)))
    assert not (sa & sb)
    assert len(sa) <= a.sm_count and len(sb) <= b.sm_count
    assert len(sw) > max(len(sa), len(sb))
    assert ga <= sa and gb <= sb and not (ga & gb)
    assert len(gw) > max(len(ga), len(gb))


# ---- 2. accuracy ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2])
def test_tiny_fp32_stream_step_vs_oracle(n):
    cfg, eng = engine("tiny", 3, torch.float32, (2, 1))
    try:
        esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
        ses = [O.StreamSession(cfg, esd, asd) for _ in range(n)]
        ids = eng.alloc(n)
        worst = 0.0
        for i, pcm in enumerate(pcm_chunks(cfg, n, 20, 50 + n)):
            enc, y = eng.stream_step(ids, pcm, 1.0)
            for j in range(n):
                _, eo, yo = ses[j].step_pcm(pcm[j].float(), 1.0)
                worst = max(worst, maxabs(enc[j].cpu(), eo[0]), maxabs(y[j].cpu(), yo[0]))
        print("tiny fp32 on SM group, %d sessions x 20 chunks: max-abs vs oracle %.3g" % (n, worst))
        assert worst < FP32_TOL
    finally:
        eng.close()


@pytest.mark.parametrize("n", [1, 2, 64])
def test_shipped_bf16_stream_step_vs_oracle(user, whole, n):
    """n sessions x 20 chunks of PCM on the group-0 context; the first two sessions against the oracle on bf16-rounded weights
    (bar 2e-2), every session against the whole-device twin; positions bit-exact."""
    cfg, eng = user
    _, weng = whole
    esd, asd = bf16_weights(make_encoder_state(cfg, 0)), bf16_weights(make_adapter_state(cfg, 0))
    k = min(n, 2)
    ses = [O.StreamSession(cfg, esd, asd) for _ in range(k)]
    ids, wids = eng.alloc(n), weng.alloc(n)
    we = wt = 0.0
    try:
        for pcm in pcm_chunks(cfg, n, 20, 60 + n):
            enc, y = eng.stream_step(ids, pcm, 1.0)
            wenc, wy = weng.stream_step(wids, pcm, 1.0)
            for j in range(k):
                _, eo, yo = ses[j].step_pcm(pcm[j].float(), 1.0)
                we = max(we, maxabs(enc[j].cpu(), eo[0]), maxabs(y[j].cpu(), yo[0]))
            wt = max(wt, maxabs(enc.cpu(), wenc.cpu()), maxabs(y.cpu(), wy.cpu()))
        print("shipped bf16 on SM group (%d SMs), %d sessions x 20 chunks: max-abs vs oracle on bf16 weights %.4g, vs whole device %.4g"
              % (eng.sm_count, n, we, wt))
        assert we < BF16_TOL and wt < BF16_TOL
        for a, b in zip(ids, wids):
            assert eng.state(int(a)) == weng.state(int(b))
        assert eng.stats()["act_saturations"] == 0
    finally:
        eng.free(ids)
        weng.free(wids)


def test_chunks_v_and_recording_with_handoff(user, whole):
    cfg, eng = user
    _, weng = whole
    counts = [1, 3, 2, 4]
    B = sum(counts)
    g = torch.Generator().manual_seed(70)
    feats = 9.0 + 3.0 * torch.randn(B, cfg.chunk_feat_frames, cfg.feat_dim, generator=g)
    ids, wids = eng.alloc(4), weng.alloc(4)
    esd, asd = bf16_weights(make_encoder_state(cfg, 0)), bf16_weights(make_adapter_state(cfg, 0))
    off = np.concatenate([[0], np.cumsum(counts)])
    try:
        e, y = eng.encode_stream_chunks_v(ids, counts, feats)
        we, wy = weng.encode_stream_chunks_v(wids, counts, feats)
        assert maxabs(e.cpu(), we.cpu()) < TWIN_BF16_TOL and maxabs(y.cpu(), wy.cpu()) < TWIN_BF16_TOL
        worst = 0.0
        for j in (1, 3):                              # sessions of 3 and 4 chunks against the oracle
            ses = O.StreamSession(cfg, esd, asd)
            for b in range(off[j], off[j + 1]):
                eo, yo = ses.step_feats(feats[b:b + 1])
                worst = max(worst, maxabs(e[b].cpu(), eo[0]), maxabs(y[b].cpu(), yo[0]))
        print("encode_stream_chunks_v on an SM group: max-abs vs oracle on bf16 weights %.4g" % worst)
        assert worst < BF16_TOL
        pcm = torch.randint(-3000, 3000, (B, cfg.samples_per_chunk), generator=g, dtype=torch.int32).to(torch.int16)
        t_out = eng.out_frames(cfg.chunk_feat_frames)[1]
        P = 3
        outs = []
        for en, i in ((eng, ids), (weng, wids)):
            embeds = torch.zeros(B, P + t_out, cfg.llm_dim, dtype=torch.float16, device=en.torch_device)
            mask = torch.zeros(B, P + t_out, dtype=torch.uint8, device=en.torch_device)
            start = torch.zeros(B, dtype=torch.int32, device=en.torch_device)
            pm = torch.tensor([1, 0, 1], dtype=torch.uint8, device=en.torch_device)
            en.handoff_arm(B, embeds, P, [1, 0] * (B // 2), pm, mask, start)
            ea, _ = en.stream_steps_v(i, counts, pcm, want_adapter=False)
            torch.cuda.synchronize()
            outs.append((ea.cpu(), embeds.float().cpu(), mask.cpu(), start.cpu()))
        (ea, ya, ma, sa), (eb, yb, mb, sb) = outs
        assert maxabs(ea, eb) < TWIN_BF16_TOL and maxabs(ya, yb) < TWIN_BF16_TOL
        assert torch.equal(ma, mb) and torch.equal(sa, sb)
        # sessions 0 and 2 (the first continues from the chunks above) against the oracle: encoder rows and hand-off rows
        worst = 0.0
        for j in (0, 2):
            ses = O.StreamSession(cfg, esd, asd)
            for b in range(off[j], off[j + 1]):
                ses.step_feats(feats[b:b + 1])
            for b in range(off[j], off[j + 1]):
                _, eo, yo = ses.step_pcm(pcm[b].float(), 1.0)
                worst = max(worst, maxabs(ea[b], eo[0]), maxabs(ya[b, P:P + t_out], yo[0]))
        print("stream_steps_v + hand-off on an SM group: max-abs vs oracle on bf16 weights %.4g" % worst)
        assert worst < BF16_TOL
        for a, b in zip(ids, wids):
            assert eng.state(int(a)) == weng.state(int(b))
    finally:
        eng.free(ids)
        weng.free(wids)


def test_offline_packed_pcm(user, whole):
    cfg, eng = user
    _, weng = whole
    g = torch.Generator().manual_seed(71)
    pcms = [torch.randint(-3000, 3000, (n,), generator=g, dtype=torch.int32).to(torch.int16) for n in (16000, 40000, 7000)]
    e, y, eo, ao, feats = eng.encode_offline_packed_pcm(pcms, scale=1.0, want_feats=True)
    we, wy, weo, wao = weng.encode_offline_packed_pcm(pcms, scale=1.0)
    assert np.array_equal(np.asarray(eo), np.asarray(weo)) and np.array_equal(np.asarray(ao), np.asarray(wao))
    assert maxabs(e.cpu(), we.cpu()) < TWIN_BF16_TOL and maxabs(y.cpu(), wy.cpu()) < TWIN_BF16_TOL
    # every utterance against the oracle fed the call's own features
    esd, asd = bf16_weights(make_encoder_state(cfg, 0)), bf16_weights(make_adapter_state(cfg, 0))
    frames, _, _ = cfg.packed_audio_offsets([len(p) for p in pcms])
    fo = np.concatenate([[0], np.cumsum(frames)])
    e, y, feats = e.cpu(), y.cpu(), feats.cpu()
    worst = 0.0
    for i in range(len(pcms)):
        f = feats[fo[i]:fo[i + 1]]
        xo, _, yo, _ = O.offline_path(cfg, esd, asd, f[None], torch.tensor([f.shape[0]]), cfg.chunk_size, cfg.left_chunks)
        worst = max(worst, maxabs(e[eo[i]:eo[i + 1]], xo[0]), maxabs(y[ao[i]:ao[i + 1]], yo[0]))
    print("packed offline PCM on an SM group: max-abs vs oracle on bf16 weights %.4g" % worst)
    assert worst < BF16_TOL


def test_scheduler_tick_and_replay(user, whole):
    """Ticks and one replay on an SM group against the same on a whole-device twin: the same blocks with the same statuses,
    rows within 4e-3.  The twin's ticks are held to the oracle within 2e-2 (test_gpu_parity.test_scheduler_vad_gating_vs_oracle),
    so the group's are within 2.4e-2 of it; its stream steps are within 2e-2 directly (test_shipped_bf16_stream_step_vs_oracle)."""
    cfg, eng = user
    _, weng = whole
    statuses = [[None, IPU_START, IPU_CONT, IPU_CONT, None], [IPU_START, IPU_CONT, None]]
    pcm = [pcm_chunks(cfg, len(s), 1, 80 + i)[0] for i, s in enumerate(statuses)]
    res = []
    for en in (eng, weng):
        sch = StreamScheduler(en, history_chunks=10, onset_chunks=6, bucket=1, max_sessions=4)
        for i in range(2):
            sch.open(("t", i))
            sch.open(("r", i))
        ticks = {}
        for j in range(5):
            for i, s in enumerate(statuses):
                if j < len(s):
                    sch.push(("t", i), pcm[i][j], s[j])
            for k, bl in sch.tick().items():
                ticks.setdefault(k[1], []).extend(bl)
        rep = sch.replay({("r", i): (pcm[i], s) for i, s in enumerate(statuses)})
        res.append((ticks, rep, [en.state(sch.keys[("r", i)]) for i in range(2)]))
        for key in list(sch.keys):
            sch.close(key)
    (ta, ra, sa), (tb, rb, sb) = res
    assert sa == sb
    pairs = [(ta.get(i, []), tb.get(i, [])) for i in range(2)] + [(ra.get(("r", i), []), rb.get(("r", i), [])) for i in range(2)]
    assert sum(len(x) for x, _ in pairs) > 0
    for xs, zs in pairs:
        assert len(xs) == len(zs)
        for x, z in zip(xs, zs):
            assert x.status == z.status
            assert maxabs(x.enc.cpu(), z.enc.cpu()) < TWIN_BF16_TOL
            assert (x.emb is None) == (z.emb is None)
            if x.emb is not None:
                assert maxabs(x.emb.float().cpu(), z.emb.float().cpu()) < TWIN_BF16_TOL


# ---- 3. the layer stack on a group ---------------------------------------------------------------------------------------------
def test_stack_kernel_on_a_group():
    """Toy widths fit the stack's plan at 72 SMs: the one-session step takes it, within 4e-4 of the chain on the same context."""
    import ctypes as C
    cfg, eng = engine("tiny", 3, torch.bfloat16, (2, 0))
    try:
        out = [C.c_int() for _ in range(5)]
        smem = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
        t = eng.out_frames(cfg.chunk_feat_frames)[0]
        fits = eng.lib.fo_debug_stack_plan(cfg.d_model, cfg.ffn_dim, cfg.n_heads, 1, t, cfg.chunk_size * cfg.left_chunks,
                                           cfg.n_layers, eng.sm_count, smem, *[C.byref(o) for o in out]) == 0
        assert fits
        ia, ib = eng.alloc(1), eng.alloc(1)
        l0 = eng.get_option("stack_launches")
        worst = 0.0
        for pcm in pcm_chunks(cfg, 1, 20, 90):
            eng.set_option("stack_rows", 8)
            e1, y1 = eng.stream_step(ia, pcm, 1.0)
            eng.set_option("stack_rows", 0)
            e0, y0 = eng.stream_step(ib, pcm, 1.0)
            worst = max(worst, maxabs(e1.cpu(), e0.cpu()), maxabs(y1.cpu(), y0.cpu()))
        eng.set_option("stack_rows", 8)
        print("stack kernel on %d SMs vs chain: %.3g" % (eng.sm_count, worst))
        assert eng.get_option("stack_launches") - l0 == 20
        assert worst < 4e-4
    finally:
        eng.close()


# ---- 4. two contexts at once -----------------------------------------------------------------------------------------------
def _run(eng, n, chunks, stream=None):
    ids = eng.alloc(n)
    outs = []
    ctx = torch.cuda.stream(stream) if stream is not None else torch.cuda.stream(torch.cuda.current_stream())
    with ctx:
        for pcm in chunks:
            e, y = eng.stream_step(ids, pcm, 1.0)
            outs.append((e.clone(), y.clone()))
    return ids, outs


def _snap(eng, ids):
    blob = eng.save_sessions(ids)
    torch.cuda.synchronize()
    return blob.cpu()


@pytest.mark.parametrize("n", [1, 64])
def test_two_contexts_concurrently_bit_identical_to_alone(user, system, n):
    (cfg, a), (_, b) = user, system
    ca, cb = pcm_chunks(cfg, n, 20, 100 + n), pcm_chunks(cfg, n, 20, 200 + n)
    alone = []
    for eng, ch in ((a, ca), (b, cb)):
        ids, outs = _run(eng, n, ch)
        torch.cuda.synchronize()
        alone.append(([(e.cpu(), y.cpu()) for e, y in outs], _snap(eng, ids)))
        eng.free(ids)

    def check(eng, ids, outs, ref):
        torch.cuda.synchronize()
        for (e, y), (re, ry) in zip(outs, ref[0]):
            assert torch.equal(e.cpu(), re) and torch.equal(y.cpu(), ry)
        assert torch.equal(_snap(eng, ids), ref[1])
        eng.free(ids)

    # alternating on two streams, no synchronisation in between
    sa, sb = torch.cuda.Stream(), torch.cuda.Stream()
    ia, ib = a.alloc(n), b.alloc(n)
    oa, ob = [], []
    for k in range(20):
        with torch.cuda.stream(sa):
            e, y = a.stream_step(ia, ca[k], 1.0)
            oa.append((e, y))
        with torch.cuda.stream(sb):
            e, y = b.stream_step(ib, cb[k], 1.0)
            ob.append((e, y))
    check(a, ia, oa, alone[0])
    check(b, ib, ob, alone[1])

    # from two host threads
    res = {}

    def worker(key, eng, ch):
        res[key] = _run(eng, n, ch, torch.cuda.Stream())
        torch.cuda.synchronize()

    th = [threading.Thread(target=worker, args=("a", a, ca)), threading.Thread(target=worker, args=("b", b, cb))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    check(a, *res["a"], alone[0])
    check(b, *res["b"], alone[1])


# ---- 5. sessions move between partitioned and whole-device contexts --------------------------------------------------------------
def test_session_moves_between_group_and_whole_device(user, whole):
    """A session moved from an SM group to the whole device and back (and the reverse) continues bit for bit as the session
    that never left: restoring into the other context and saving from it changes no state.  On the other context it
    continues within the twin bar of the context it came from."""
    cfg, eng = user
    _, weng = whole
    ch = pcm_chunks(cfg, 2, 16, 300)
    for home, away in ((eng, weng), (weng, eng)):
        stay = home.alloc(2)
        for p in ch[:8]:
            home.stream_step(stay, p, 1.0)
        blob = home.save_sessions(stay)
        there = away.alloc(2)
        away.restore_sessions(there, blob)
        back = home.alloc(2)
        home.restore_sessions(back, away.save_sessions(there))
        for p in ch[8:]:
            e0, y0 = home.stream_step(stay, p, 1.0)
            e1, y1 = home.stream_step(back, p, 1.0)
            e2, y2 = away.stream_step(there, p, 1.0)
            assert torch.equal(e0.cpu(), e1.cpu()) and torch.equal(y0.cpu(), y1.cpu())
            assert maxabs(e2.cpu(), e0.cpu()) < TWIN_BF16_TOL and maxabs(y2.cpu(), y0.cpu()) < TWIN_BF16_TOL
        torch.cuda.synchronize()
        assert torch.equal(home.save_sessions(back).cpu(), home.save_sessions(stay).cpu())
        assert [away.state(int(x)) for x in there] == [home.state(int(x)) for x in stay]
        for ids, en in ((stay, home), (there, away), (back, home)):
            en.free(ids)


# ---- 6. refusals ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("part,msg", [((0, 0), "sm_split must be >= 1"), ((2, 2), "outside [0, sm_split = 2)"),
                                      ((2, -1), "outside [0, sm_split = 2)"), ((32, 0), "below the 8-SM granularity")])
def test_refusals_name_the_cause(part, msg):
    with pytest.raises(RuntimeError, match=msg.replace("[", r"\[").replace("(", r"\(").replace(")", r"\)")):
        engine("tiny", 3, torch.float32, part)
