"""fo_encode_stream_chunks / Engine.encode_stream_chunks: k consecutive chunks of every session in one streaming step must
give what k single-chunk steps give -- against the CPU oracle run one chunk at a time, and against sequential single-chunk
calls on the same engine (which the other GPU tests pin to the reference's goldens)."""
import dataclasses

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config, load_yaml, path_config_from_dict
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
from oracle import freeze_omni_oracle as O

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
BF16_TOL = 2e-2


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def bf16_weights(sd):
    keep = ("pos_bias", "conv.0.weight")
    return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}


def feats_for(cfg, n, chunks, seed, t_in=None):
    g = torch.Generator().manual_seed(seed)
    return 9.0 + 3.0 * torch.randn(n, chunks, t_in or cfg.chunk_feat_frames, cfg.feat_dim, generator=g)


def engine(cfg, seed=3, adapter_seed=3, **kw):
    from freeze_omni_b200.engine import Engine
    return Engine(cfg, make_encoder_state(cfg, seed), make_adapter_state(cfg, adapter_seed), **kw)


@pytest.fixture(scope="module")
def tiny32():
    cfg = load_path_config("tiny")
    eng = engine(cfg, max_sessions=8)
    yield cfg, eng
    eng.close()


@pytest.fixture(scope="module")
def shipped16():
    cfg = load_path_config("shipped")
    eng = engine(cfg, seed=0, adapter_seed=0, dtype=torch.bfloat16, max_sessions=4)
    yield cfg, eng
    eng.close()


def test_tiny_fp32_vs_oracle_chunk_by_chunk(tiny32):
    """2 fresh sessions, 40 chunks in calls of k = 1, 3, 7, 2, 16, 11 (crossing the 17-chunk ring saturation): every chunk
    against the oracle run one chunk at a time; bookkeeping and exported caches after every call."""
    cfg, eng = tiny32
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    sessions = [O.StreamSession(cfg, esd, asd) for _ in range(2)]
    ids = eng.alloc(2)
    feats = feats_for(cfg, 2, 40, 11)
    try:
        c0 = 0
        for k in (1, 3, 7, 2, 16, 11):
            enc, y = eng.encode_stream_chunks(ids, feats[:, c0:c0 + k].contiguous())
            assert tuple(enc.shape) == (2, k, 4, cfg.d_model) and tuple(y.shape) == (2, k, 2, cfg.llm_dim)
            for b, s in enumerate(sessions):
                for j in range(k):
                    eo, yo = s.step_feats(feats[b, c0 + j].unsqueeze(0))
                    assert maxabs(enc[b, j].cpu(), eo[0]) < FP32_TOL, (k, b, j)
                    assert maxabs(y[b, j].cpu(), yo[0]) < FP32_TOL, (k, b, j)
                assert eng.state(int(ids[b])) == (4 * (c0 + k), s.pe_index)
                for li in range(cfg.n_layers):
                    kk, vv = eng.export_kv(int(ids[b]), li)
                    assert maxabs(kk, s.buffer[li][0]) < FP32_TOL and maxabs(vv, s.buffer[li][1]) < FP32_TOL
                assert maxabs(eng.export_adapter_cache(int(ids[b])), s.cache[0]) < FP32_TOL
            c0 += k
    finally:
        eng.free(ids)


@pytest.mark.parametrize("which", ["tiny32", "shipped16"])
def test_one_chunk_is_bit_identical_to_encode_stream(which, request):
    cfg, eng = request.getfixturevalue(which)
    a, b = eng.alloc(2), eng.alloc(2)
    feats = feats_for(cfg, 2, 5, 12)
    try:
        for i in range(5):
            e1, y1 = eng.encode_stream(a, feats[:, i].contiguous())
            e2, y2 = eng.encode_stream_chunks(b, feats[:, i:i + 1].contiguous())
            assert torch.equal(e1, e2[:, 0]) and torch.equal(y1, y2[:, 0]), i
    finally:
        eng.free(a)
        eng.free(b)


def test_pe_index_wraps_inside_one_call(tiny32):
    cfg, eng = tiny32
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    sess = O.StreamSession(cfg, esd, asd)
    sess.pe_index = cfg.pe_wrap - 8
    ids = eng.alloc(1)
    feats = feats_for(cfg, 1, 14, 13)
    try:
        eng.set_pe_index(ids, cfg.pe_wrap - 8)
        for c0 in (0, 7):
            enc, y = eng.encode_stream_chunks(ids, feats[:, c0:c0 + 7].contiguous())
            for j in range(7):
                eo, yo = sess.step_feats(feats[:, c0 + j])
                assert maxabs(enc[0, j].cpu(), eo[0]) < FP32_TOL and maxabs(y[0, j].cpu(), yo[0]) < FP32_TOL, (c0, j)
            assert eng.state(int(ids[0]))[1] == sess.pe_index
    finally:
        eng.free(ids)


def _variant(name):
    if name in ("cnn", "two"):
        base = path_config_from_dict(load_yaml("tiny_bn"))
        return dataclasses.replace(base, adapter_type="cnn") if name == "cnn" else dataclasses.replace(base, llm_dim=base.d_model * 4 + 64)
    if name == "fork_t7":
        return load_path_config("tiny")
    return load_path_config(name)


@pytest.mark.parametrize("name", ["tiny_linear", "cnn", "two", "tiny_bn", "tiny_conv1d", "tiny_postnorm_concat", "fork_t7"])
def test_variants_vs_sequential_single_chunk_calls(name):
    """Every adapter / layer variant, k = 3 then 7, against single-chunk calls of twin sessions on the same engine.
    fork_t7: 32 feature frames per chunk -> t = 7, odd, so the CNNSubsampling adapter runs its convolutions at stride 1 over
    each session's frames and picks every chunk's output rows."""
    cfg = _variant(name)
    t_in = 32 if name == "fork_t7" else cfg.chunk_feat_frames
    eng = engine(cfg, adapter_seed=5 if name in ("cnn", "two") else 3, max_sessions=6)
    try:
        a, b = eng.alloc(2), eng.alloc(2)
        feats = feats_for(cfg, 2, 12, 14, t_in)
        c0 = 0
        for k in (1, 3, 7):
            enc, y = eng.encode_stream_chunks(a, feats[:, c0:c0 + k].contiguous())
            for j in range(k):
                eo, yo = eng.encode_stream(b, feats[:, c0 + j].contiguous())
                assert maxabs(enc[:, j].cpu(), eo.cpu()) < FP32_TOL, (k, j)
                assert maxabs(y[:, j].cpu(), yo.cpu()) < FP32_TOL, (k, j)
            for s, r in zip(a, b):
                assert eng.state(int(s)) == eng.state(int(r))
            c0 += k
        if name == "tiny_conv1d":
            for s, r in zip(a, b):
                assert maxabs(eng.export_ffn_cache(int(s), 0), eng.export_ffn_cache(int(r), 0)) < FP32_TOL
    finally:
        eng.close()


@pytest.mark.parametrize("name", ["tiny_linear", "cnn", "two", "tiny_bn", "fork_t7"])
def test_handoff_through_every_adapter_variant(name):
    """The fp16 LLM hand-off of every adapter variant on a bf16 engine, k = 1 then 3: an armed call writes, behind the prefix of
    each (session, chunk) block, the adapter rows that twin sessions get as fp32, rounded to fp16 bit for bit; the prefix and
    trailing rows keep what they held; both sets of sessions end in the same state.  fork_t7 (t = 7): the CNNSubsampling adapter
    picks every chunk's rows from a stride-1 pass, and its later chunks land in blocks j0 > 0 of a session."""
    cfg = _variant(name)
    t_in = 32 if name == "fork_t7" else cfg.chunk_feat_frames
    eng = engine(cfg, adapter_seed=5 if name in ("cnn", "two") else 3, dtype=torch.bfloat16, max_sessions=4)
    try:
        a, b = eng.alloc(2), eng.alloc(2)
        feats = feats_for(cfg, 2, 4, 21, t_in)
        _, t_out = eng.out_frames(t_in)
        P = 3
        g = torch.Generator().manual_seed(22)
        c0 = 0
        for k in (1, 3):
            f = feats[:, c0:c0 + k].contiguous()
            emb = torch.randn(2 * k, P + t_out + 2, cfg.llm_dim, generator=g).half().cuda()
            before = emb.clone()
            eng.handoff_arm(2 * k, emb, P, [1, 0] * k)
            eng.encode_stream_chunks(a, f, want_adapter=False)
            _, y = eng.encode_stream_chunks(b, f)
            torch.cuda.synchronize()
            assert torch.equal(emb[:, P:P + t_out], y.reshape(2 * k, t_out, cfg.llm_dim).half()), k
            assert torch.equal(emb[:, :P], before[:, :P]) and torch.equal(emb[:, P + t_out:], before[:, P + t_out:]), k
            for s, r in zip(a, b):
                assert eng.state(int(s)) == eng.state(int(r))
                if cfg.adapter_type == "subsampling":
                    for w in range(2 if cfg.adapter_two_conv else 1):
                        assert torch.equal(eng.export_adapter_cache(int(s), w), eng.export_adapter_cache(int(r), w)), (k, w)
            c0 += k
    finally:
        eng.close()


def test_shipped_bf16_vs_oracle_on_bf16_weights(shipped16):
    cfg, eng = shipped16
    esd, asd = bf16_weights(make_encoder_state(cfg, 0)), bf16_weights(make_adapter_state(cfg, 0))
    we = wy = 0.0
    # 2 sessions: 20 single-chunk steps, then one k = 7 call
    ses = [O.StreamSession(cfg, esd, asd) for _ in range(2)]
    ids = eng.alloc(2)
    feats = feats_for(cfg, 2, 27, 15)
    try:
        for i in range(20):
            eng.encode_stream(ids, feats[:, i].contiguous())
            for b in range(2):
                ses[b].step_feats(feats[b:b + 1, i])
        enc, y = eng.encode_stream_chunks(ids, feats[:, 20:27].contiguous())
        for b in range(2):
            for j in range(7):
                eo, yo = ses[b].step_feats(feats[b:b + 1, 20 + j])
                we, wy = max(we, maxabs(enc[b, j].cpu(), eo[0])), max(wy, maxabs(y[b, j].cpu(), yo[0]))
            assert eng.state(int(ids[b])) == (4 * 27, ses[b].pe_index)
    finally:
        eng.free(ids)
    # 1 session: 12 calls of k = 16 (192 chunks, 30.7 s of audio)
    ses = O.StreamSession(cfg, esd, asd)
    ids = eng.alloc(1)
    feats = feats_for(cfg, 1, 192, 16)
    try:
        for c in range(12):
            enc, y = eng.encode_stream_chunks(ids, feats[:, 16 * c:16 * (c + 1)].contiguous())
            for j in range(16):
                eo, yo = ses.step_feats(feats[:, 16 * c + j])
                we, wy = max(we, maxabs(enc[0, j].cpu(), eo[0])), max(wy, maxabs(y[0, j].cpu(), yo[0]))
        assert eng.state(int(ids[0])) == (4 * 192, ses.pe_index)
    finally:
        eng.free(ids)
    print("multi-chunk bf16 max-abs vs oracle on bf16 weights: encoder %.4g adapter %.4g" % (we, wy))
    assert we < BF16_TOL and wy < BF16_TOL


def test_graph_replay_and_no_stack_kernel(shipped16):
    cfg, eng = shipped16
    a, b = eng.alloc(1), eng.alloc(1)
    feats = feats_for(cfg, 1, 6, 17)
    try:
        stacks0 = eng.get_option("stack_launches")
        outs = []
        for i in range(3):
            r0 = eng.stats()["graph_replays"]
            outs.append(eng.encode_stream_chunks(a, feats[:, 2 * i:2 * i + 2].contiguous()))
            torch.cuda.synchronize()
            if i == 2:
                assert eng.stats()["graph_replays"] == r0 + 1
        assert eng.get_option("stack_launches") == stacks0          # 1 session x 2 chunks = 8 rows: still the chain
        eng.set_option("use_graph", 0)
        try:
            for i in range(3):
                e, y = eng.encode_stream_chunks(b, feats[:, 2 * i:2 * i + 2].contiguous())
                assert torch.equal(e, outs[i][0]) and torch.equal(y, outs[i][1]), i
        finally:
            eng.set_option("use_graph", 1)
        s = eng.stats()
        assert s["session_chunks"] >= 12
    finally:
        eng.free(a)
        eng.free(b)


def test_refusals(tiny32, shipped16):
    from freeze_omni_b200 import _lib
    cfg, eng = tiny32
    ids = eng.alloc(1)
    try:
        with pytest.raises(_lib.FoError, match="largest k is 16"):
            eng.encode_stream_chunks(ids, feats_for(cfg, 1, 17, 18))
        rc = eng.lib.fo_encode_stream_chunks(eng._h, ids.ctypes.data_as(_lib._I32P), 1, 2, None, cfg.chunk_feat_frames, None, None,
                                             eng._stream())
        assert rc == -1                                               # FO_ERR_ARG
        assert b"feats" in eng.lib.fo_last_error()
        assert eng.state(int(ids[0])) == (0, 0)                       # nothing advanced
    finally:
        eng.free(ids)
    mcfg = load_path_config("tiny_mlconv")
    meng = engine(mcfg, max_sessions=2)
    try:
        with pytest.raises(_lib.FoError, match="MultiLayeredConv1d"):
            meng.encode_stream_chunks(meng.alloc(1), feats_for(mcfg, 1, 2, 19))
    finally:
        meng.close()
    scfg, seng = shipped16
    sids = seng.alloc(2)
    try:
        emb = torch.zeros(4, 2 + 2, scfg.llm_dim, dtype=torch.float16, device="cuda")
        seng.handoff_arm(2, emb, 2, [0, 1])
        with pytest.raises(_lib.FoError, match="armed for 2 blocks"):
            seng.encode_stream_chunks(sids, feats_for(scfg, 2, 2, 20), want_adapter=False)
    finally:
        seng.free(sids)


def _gating_run(eng, g, max_chunks, handoff=None):
    from freeze_omni_b200.scheduler import StreamScheduler
    sch = StreamScheduler(eng, history_chunks=10, onset_chunks=6, bucket=4, max_sessions=2, max_chunks=max_chunks)
    sch.open("u")
    sch.open("v")
    sch.block_log = []
    blocks, calls = [], []
    try:
        for i, st in enumerate(g["statuses"]):
            a = g["pcm"][i * 2560:(i + 1) * 2560].astype(np.float32) / 32768.0
            sch.push("u", a, str(st) if str(st) else None)
            sch.push("v", a[::-1].copy(), "ipu_cl")                   # a second session that speaks throughout
            c0 = sch.stats["encode_calls"]
            out = sch.tick(float(g["scale"]), handoff=handoff)
            calls.append((len(out.get("u", [])), sch.stats["encode_calls"] - c0))
            for s in ("u", "v"):
                for blk in out.get(s, []):
                    start = None
                    if handoff is not None:                           # row_start of the hand-off block this Block views
                        row = (blk.emb.data_ptr() - handoff.embeds.data_ptr()) // (handoff.embeds.stride(0) * 2)
                        start = int(handoff.row_start[row])
                    blocks.append((s, blk.status, blk.enc.cpu().clone(), None if blk.emb is None else blk.emb.float().cpu().clone(),
                                   None if blk.mask is None else blk.mask.cpu().clone(), start))
        return blocks, calls, [lab for _, _, lab in sch.block_log]
    finally:
        for s in list(sch.keys):
            sch.close(s)
        eng.free(sch.scratch)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_scheduler_max_chunks_on_gating_golden(golden, dtype):
    """max_chunks = 7 against max_chunks = 1 on the gating golden's stream: same blocks, statuses and order, frames within the
    bf16 bar; an onset tick is exactly 2 encode calls.  bf16 adds the fused LLM hand-off: fp16 rows within the bar, masks and
    row_start bit-exact."""
    from freeze_omni_b200.scheduler import Handoff
    cfg = load_path_config("tiny")
    g = golden("gating")
    eng = engine(cfg, dtype=dtype, max_sessions=12)
    try:
        ho1 = ho7 = None
        if dtype == torch.bfloat16:
            prefix = torch.randn(1, 3, cfg.llm_dim, generator=torch.Generator().manual_seed(3))
            ho1, ho7 = Handoff(eng, 64, prefix), Handoff(eng, 64, prefix)
        ref, calls1, labels1 = _gating_run(eng, g, 1, ho1)
        got, calls7, labels7 = _gating_run(eng, g, 7, ho7)
        assert labels1 == labels7
        assert [b[:2] for b in ref] == [b[:2] for b in got]
        for r, q in zip(ref, got):
            assert maxabs(r[2], q[2]) < BF16_TOL and r[5] == q[5]
            if r[3] is not None:
                assert maxabs(r[3], q[3]) < BF16_TOL
            if r[4] is not None:
                assert torch.equal(r[4], q[4])
        onset_ticks = [c for c in calls7 if c[0] == 7]
        assert onset_ticks and all(c[1] == 2 for c in onset_ticks)
        assert all(c1[1] == 7 for c1, c7 in zip(calls1, calls7) if c7[0] == 7)
    finally:
        eng.close()
