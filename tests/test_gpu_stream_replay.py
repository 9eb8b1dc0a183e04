"""Gated replay of recorded conversations: fo_fbank_stream_v / Engine.fbank_stream_v, fo_encode_stream_steps_v /
Engine.encode_stream_steps_v and StreamScheduler.replay.  The two halves must be bit-identical to the calls they split
(per-chunk fbank_stream, stream_steps_v), and a replay must leave every session as pushing the recording one chunk per
tick does: labels, history ring and (n_frames, pe_index) exactly, encoder and adapter rows within the twin-session bars."""
import dataclasses
import random

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config, load_yaml, path_config_from_dict
from freeze_omni_b200.scheduler import IPU_CONT, IPU_START, StreamScheduler
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
# bf16 twin sessions encoded at other batchings (the bar of the multi-chunk and recording tests)
TWIN_BF16_TOL = 4e-3


def maxabs(a, b):
    return float((a.detach().double().cpu() - b.detach().double().cpu()).abs().max())


def pcm_blocks(cfg, n, seed, dtype=torch.int16):
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(-3000, 3000, (n, cfg.samples_per_chunk), generator=g, dtype=torch.int32).to(torch.int16)
    return x if dtype == torch.int16 else (x.float() / 32768.0)


def fork_cfg():
    y = load_yaml("tiny")
    y["frontend"] = dict(y["frontend"], frame_length_ms=16, frame_shift_ms=8, frames_per_chunk=28, context_frames=4)
    return path_config_from_dict(y)


def config(name):
    if name == "fork_t7":
        return fork_cfg()
    if name == "cnn":
        return dataclasses.replace(path_config_from_dict(load_yaml("tiny_bn")), adapter_type="cnn")
    return load_path_config(name)


def engine(cfg, **kw):
    from freeze_omni_b200.engine import Engine
    return Engine(cfg, make_encoder_state(cfg, 3), make_adapter_state(cfg, 5), **kw)


def conversation(rng, n, speech_from_start=False):
    """VAD statuses of n chunks: silences of 2-20 chunks and speech turns of 3-25 opening with 'ipu_sl' (about half speech)."""
    out, speaking = [], speech_from_start
    while len(out) < n:
        if speaking:
            out += [IPU_START] + [IPU_CONT] * rng.randint(2, 24)
        else:
            out += [None] * rng.randint(2, 20)
        speaking = not speaking
    return out[:n]


# ---- 1. fbank_stream_v == per-chunk fbank_stream ---------------------------------------------------------------------------
@pytest.mark.parametrize("on_device", [False, True], ids=["host", "device"])
@pytest.mark.parametrize("pcm_dtype", [torch.int16, torch.float32], ids=["i16", "f32"])
@pytest.mark.parametrize("name", ["tiny", "fork_t7"])
def test_fbank_stream_v_bit_identical(name, pcm_dtype, on_device):
    """Counts 5, 1, 13 in passes of 4 blocks against twins fed one fbank_stream per chunk: features bit for bit, and the next
    fbank_stream of both gives bit-identical features (sample carry and feature ring)."""
    cfg = config(name)
    eng = engine(cfg, max_sessions=8)
    try:
        eng.set_option("steps_pass_blocks", 4)
        counts = [5, 1, 13]
        a, b = eng.alloc(3), eng.alloc(3)
        eng.fbank_stream(a, pcm_blocks(cfg, 3, 1, pcm_dtype))             # a non-zero carry and ring before the call
        eng.fbank_stream(b, pcm_blocks(cfg, 3, 1, pcm_dtype))
        pcm = pcm_blocks(cfg, sum(counts), 2, pcm_dtype)
        got = eng.fbank_stream_v(a, counts, pcm.cuda() if on_device else pcm).cpu()
        off = np.concatenate([[0], np.cumsum(counts)])
        for j in range(max(counts)):
            sel = [i for i in range(3) if j < counts[i]]
            want = eng.fbank_stream(b[sel], pcm[[off[i] + j for i in sel]].contiguous()).cpu()
            for r, i in enumerate(sel):
                assert torch.equal(got[off[i] + j], want[r]), (i, j)
        nxt = pcm_blocks(cfg, 3, 3, pcm_dtype)
        assert torch.equal(eng.fbank_stream(a, nxt).cpu(), eng.fbank_stream(b, nxt).cpu())
        for i in range(3):
            assert eng.state(int(a[i])) == eng.state(int(b[i])) == (0, 0)      # the encoder state did not move
    finally:
        eng.close()


# ---- 2. encode_stream_steps_v == stream_steps_v on the features fbank_stream_v gave ------------------------------------------
@pytest.mark.parametrize("name,dtype", [("tiny", torch.float32), ("fork_t7", torch.float32), ("cnn", torch.float32),
                                        ("tiny", torch.bfloat16), ("fork_t7", torch.bfloat16)])
def test_encode_stream_steps_v_bit_identical(name, dtype):
    cfg = config(name)
    eng = engine(cfg, dtype=dtype, max_sessions=8)
    try:
        eng.set_option("steps_pass_blocks", 7)
        counts = [9, 1, 30]
        a, b = eng.alloc(3), eng.alloc(3)
        pcm = pcm_blocks(cfg, sum(counts), 4)
        for k in range(2):                         # the second round continues from the state the first left
            p = pcm if k == 0 else pcm_blocks(cfg, sum(counts), 5)
            ea, ya = eng.stream_steps_v(a, counts, p)
            feats = eng.fbank_stream_v(b, counts, p)
            eb, yb = eng.encode_stream_steps_v(b, counts, feats)
            assert torch.equal(ea.cpu(), eb.cpu()) and torch.equal(ya.cpu(), yb.cpu()), k
            for i in range(3):
                assert eng.state(int(a[i])) == eng.state(int(b[i]))
        nxt = pcm_blocks(cfg, 3, 6)
        ea, ya = eng.stream_step(a, nxt)
        eb, yb = eng.stream_step(b, nxt)
        assert torch.equal(ea.cpu(), eb.cpu()) and torch.equal(ya.cpu(), yb.cpu())
    finally:
        eng.close()


# ---- 3. replay == the tick loop, then live ticks -----------------------------------------------------------------------------
def compare_blocks(got, want, tol, tag):
    assert [b.status for b in got] == [b.status for b in want], tag
    worst = 0.0
    for g, w in zip(got, want):
        worst = max(worst, maxabs(g.enc, w.enc), maxabs(g.emb, w.emb) if w.emb is not None else 0.0)
    assert worst < tol, (tag, worst)
    return worst


def replay_vs_ticks(eng, cfg, statuses, tol, seed, live_ticks=10, roundtrip=0):
    """Sessions ('t', i) fed by push/tick one chunk at a time and twins ('r', i) by one replay, on one scheduler; then
    `live_ticks` ticks of the same chunks for both, after a detach / attach of ('r', roundtrip).  An extra open session
    ('idle',) is left out of the replay and must stay untouched."""
    sch = StreamScheduler(eng, history_chunks=10, onset_chunks=6, bucket=1, max_sessions=2 * len(statuses) + 1)
    n = len(statuses)
    for i in range(n):
        sch.open(("t", i))
        sch.open(("r", i))
    sch.open(("idle",))
    pcm = [pcm_blocks(cfg, len(s), seed + i) for i, s in enumerate(statuses)]
    want = {}
    for j in range(max(len(s) for s in statuses)):
        for i, s in enumerate(statuses):
            if j < len(s):
                sch.push(("t", i), pcm[i][j], s[j])
        for k, bl in sch.tick().items():
            want.setdefault(k[1], []).extend(bl)
    got = sch.replay({("r", i): (pcm[i], s) for i, s in enumerate(statuses)})
    worst = 0.0
    for i in range(n):
        worst = max(worst, compare_blocks(got.get(("r", i), []), want.get(i, []), tol, ("replay", i)))
        assert torch.equal(sch.history(("r", i)), sch.history(("t", i))), i
        assert eng.state(sch.keys[("r", i)]) == eng.state(sch.keys[("t", i)]), i
    assert eng.state(sch.keys[("idle",)]) == (0, 0) and not sch.history(("idle",)).any()
    snap = sch.detach(("r", roundtrip))
    sch.attach(("r", roundtrip), snap)
    rng = random.Random(seed)
    for k in range(live_ticks):
        x = pcm_blocks(cfg, n, seed + 100 + k)
        for i in range(n):
            st = rng.choice([None, IPU_START, IPU_CONT])
            sch.push(("t", i), x[i], st)
            sch.push(("r", i), x[i], st)
        out = sch.tick()
        for i in range(n):
            worst = max(worst, compare_blocks(out.get(("r", i), []), out.get(("t", i), []), tol, ("live", k, i)))
            assert torch.equal(sch.history(("r", i)), sch.history(("t", i)))
            assert eng.state(sch.keys[("r", i)]) == eng.state(sch.keys[("t", i)])
    return worst


@pytest.mark.parametrize("name", ["tiny", "fork_t7", "cnn"])
def test_replay_vs_tick_loop_fp32(name):
    """Edge sessions: speech from chunk 0, all silent, a short one with an onset before any silence, a long conversation;
    windows forced small, so sessions leave the window calls at different points."""
    cfg = config(name)
    eng = engine(cfg, max_sessions=16)
    try:
        eng.set_option("steps_pass_blocks", 24)
        rng = random.Random(7)
        statuses = [conversation(rng, 60, speech_from_start=True), [None] * 25, [IPU_START, IPU_CONT, IPU_START],
                    conversation(rng, 90)]
        worst = replay_vs_ticks(eng, cfg, statuses, FP32_TOL, seed=50)
        print("%s fp32 replay vs tick loop: max abs %.3g" % (name, worst))
    finally:
        eng.close()


def test_replay_vs_tick_loop_bf16_shipped():
    """The shipped model in bf16, 4 sessions x 188 chunks (30 s each, about half speech) against the tick loop."""
    cfg = load_path_config("shipped")
    eng = engine(cfg, dtype=torch.bfloat16, max_sessions=12)
    try:
        rng = random.Random(11)
        statuses = [conversation(rng, 188, speech_from_start=(i == 0)) for i in range(4)]
        worst = replay_vs_ticks(eng, cfg, statuses, TWIN_BF16_TOL, seed=70, roundtrip=2)
        print("bf16 shipped replay vs tick loop: max abs %.3g" % worst)
        assert eng.stats()["act_saturations"] == 0
    finally:
        eng.close()


# ---- 4. refusals ---------------------------------------------------------------------------------------------------------
def _snapshot(eng, ids):
    return [(eng.state(int(s)), eng.save_sessions([int(s)]).cpu()) for s in ids]


def test_refusals_touch_nothing():
    from freeze_omni_b200 import _lib
    from freeze_omni_b200.engine import _i32p
    cfg = load_path_config("tiny")
    eng = engine(cfg, max_sessions=6)
    try:
        ids = eng.alloc(2)
        eng.stream_steps_v(ids, [3, 2], pcm_blocks(cfg, 5, 1))
        before = _snapshot(eng, ids)
        l0 = eng.stats()["kernel_launches"]
        feats = torch.zeros(2, cfg.chunk_feat_frames, cfg.feat_dim, device=eng.torch_device)
        bad = [(ids, [0, 2]), (np.array([ids[0], ids[0]]), [1, 1]), (np.array([ids[0], 5]), [1, 1])]
        for bid, ch in bad:
            with pytest.raises(RuntimeError):
                eng.fbank_stream_v(bid, ch, pcm_blocks(cfg, max(1, int(np.sum(ch))), 2))
            with pytest.raises(RuntimeError):
                eng.encode_stream_steps_v(bid, ch, feats[:max(1, int(np.sum(ch)))].contiguous())
        pcm = pcm_blocks(cfg, 2, 3)
        with pytest.raises(RuntimeError, match="FO_F32 or FO_I16"):
            _lib.check(eng.lib.fo_fbank_stream_v(eng._h, _i32p(ids), _i32p(np.array([1, 1], np.int32)), 2, pcm.data_ptr(), 99, 1.0,
                                                 None, eng._stream()))
        torch.cuda.synchronize()
        assert eng.stats()["kernel_launches"] == l0
        after = _snapshot(eng, ids)
        for (sa, ra), (sb, rb) in zip(before, after):
            assert sa == sb and torch.equal(ra, rb)
        # the scheduler: a session with a pushed chunk refuses the whole replay before anything runs
        sch = StreamScheduler(eng, bucket=1, max_sessions=3)
        sch.open("a")
        sch.open("b")
        sch.push("b", pcm[0], IPU_CONT)
        keep = _snapshot(eng, [sch.keys["a"], sch.keys["b"]])
        with pytest.raises(RuntimeError, match="tick first"):
            sch.replay({"a": (pcm, [None, IPU_START]), "b": (pcm, [IPU_CONT, IPU_CONT])})
        for (sa, ra), (sb, rb) in zip(keep, _snapshot(eng, [sch.keys["a"], sch.keys["b"]])):
            assert sa == sb and torch.equal(ra, rb)
        assert not sch.history("a").any()
    finally:
        eng.close()


def test_encode_refuses_while_handoff_armed_and_keeps_it():
    cfg = load_path_config("shipped")
    eng = engine(cfg, dtype=torch.bfloat16, max_sessions=2)
    try:
        ids = eng.alloc(1)
        t, t_out = eng.out_frames(cfg.chunk_feat_frames)
        embeds = torch.zeros(1, 8 + t_out, cfg.llm_dim, dtype=torch.float16, device=eng.torch_device)
        eng.handoff_arm(1, embeds, 8, [1])
        feats = torch.zeros(2, cfg.chunk_feat_frames, cfg.feat_dim, device=eng.torch_device)
        with pytest.raises(RuntimeError, match="armed"):
            eng.encode_stream_steps_v(ids, [2], feats)
        assert eng.state(int(ids[0])) == (0, 0)
        eng.encode_stream(ids, feats[:1].contiguous(), want_adapter=False)      # the arm is still there, and this step takes it
        torch.cuda.synchronize()
        assert embeds[0, 8:].abs().sum().item() > 0
    finally:
        eng.close()


def test_encode_refuses_multilayered_conv1d_and_long_windows():
    for cfg, match in ((load_path_config("tiny_mlconv"), "MultiLayeredConv1d"),
                       (dataclasses.replace(load_path_config("tiny"), chunk_size=4, left_chunks=32, frames_per_chunk=16,
                                            context_frames=3), "128")):
        eng = engine(cfg, max_sessions=2)
        try:
            ids = eng.alloc(1)
            feats = torch.zeros(3, cfg.chunk_feat_frames, cfg.feat_dim, device=eng.torch_device)
            with pytest.raises(RuntimeError, match=match):
                eng.encode_stream_steps_v(ids, [3], feats)
            assert eng.state(int(ids[0])) == (0, 0)
        finally:
            eng.close()
