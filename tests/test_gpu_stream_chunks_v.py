"""fo_encode_stream_chunks_v / Engine.encode_stream_chunks_v: every session of one streaming step advances by its own number
of consecutive chunks.  Each chunk must be what that many single-chunk steps give -- against the CPU oracle run one chunk at
a time, and against twin sessions advanced by uniform calls on the same engine -- and equal counts must be the old call."""
import dataclasses

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config, load_yaml, path_config_from_dict
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
from oracle import freeze_omni_oracle as O

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
TWIN_BF16_TOL = 4e-3          # a batched bf16 call against differently batched twins (the k-chunk tests' bar)
BF16_TOL = 2e-2
MAX_KEYS = 128


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def bf16_weights(sd):
    keep = ("pos_bias", "conv.0.weight")
    return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}


def rand_feats(cfg, shape, seed):
    g = torch.Generator().manual_seed(seed)
    return 9.0 + 3.0 * torch.randn(*shape, cfg.feat_dim, generator=g)


def engine(cfg, seed=3, adapter_seed=3, **kw):
    from freeze_omni_b200.engine import Engine
    return Engine(cfg, make_encoder_state(cfg, seed), make_adapter_state(cfg, adapter_seed), **kw)


def pack(per_session):
    """[(k_i, t_in, F)] -> (sum k_i, t_in, F) in (session, chunk) order"""
    return torch.cat(per_session, 0).contiguous()


def offsets(chunks):
    return np.concatenate([[0], np.cumsum(chunks)]).astype(int)


# ---- 1. fp32 against the oracle -------------------------------------------------------------------------------------------
CHUNKINGS = [(4, 16), (3, 5), (2, 8), (8, 8)]


def _sat_chunks(cfg, t, ring_cap):
    """Single-chunk steps after which the saturated ring window [n - window, n) wraps around the ring's end."""
    w = cfg.kv_window
    for p in range(1, 4 * ring_cap):
        n = p * t
        if n >= w and (w == 1 or (n - w) % ring_cap + w > ring_cap):
            return p
    return 1


@pytest.mark.parametrize("cap", ["tight", "default"])
@pytest.mark.parametrize("c,left", CHUNKINGS)
def test_fp32_vs_oracle_mixed_counts(c, left, cap):
    """Five sessions, per call a different count each: fresh; one that saturates its window inside the call; one whose ring
    window wraps past the ring's end; one whose pe_index wraps inside the call; a second fresh one.  Every chunk against
    the oracle run one chunk at a time; (n_frames, pe_index) exact and exported K/V, adapter and caches after every call."""
    from freeze_omni_b200.engine import Engine
    cfg = dataclasses.replace(load_path_config("tiny"), chunk_size=c, left_chunks=left)
    t_in, t = 4 * c + 3, c
    eng = Engine(cfg, make_encoder_state(cfg, 3), make_adapter_state(cfg, 3), max_sessions=8,
                 max_stream_frames=t_in if cap == "tight" else None)
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    kcap = max(1, (MAX_KEYS - cfg.kv_window) // t)
    ring_cap = eng.get_option("ring_cap")
    try:
        ids = eng.alloc(5)
        ses = [O.StreamSession(cfg, esd, asd) for _ in range(5)]
        nf = [0] * 5
        gen = torch.Generator().manual_seed(100 + c)
        # priming, single-chunk steps: session 1 just below its window, session 2 at the ring-wrap phase, session 3 two
        # chunks in, then moved to pe_index = pe_wrap - C, so that its second chunk of the first mixed call (count 7) wraps
        prime = [0, max(0, cfg.kv_window - t) // t, _sat_chunks(cfg, t, ring_cap), 2, 0]
        for i, p in enumerate(prime):
            for _ in range(p):
                f = 9.0 + 3.0 * torch.randn(1, t_in, cfg.feat_dim, generator=gen)
                eng.encode_stream(ids[i:i + 1], f)
                ses[i].step_feats(f)
                nf[i] += t
        eng.set_pe_index(ids[3:4], cfg.pe_wrap - c)
        ses[3].pe_index = cfg.pe_wrap - c
        assert eng.state(int(ids[3]))[1] == cfg.pe_wrap - c
        rng = np.random.default_rng(c * 31 + left)
        mixes = [[1, 4, 1, 7, 2], [3, 1, 16, 1, 1]] + [list(rng.integers(1, 8, 5)) for _ in range(3)]
        for call, mix in enumerate(mixes):
            chunks = np.minimum(np.array(mix, np.int32), kcap)
            feats = 9.0 + 3.0 * torch.randn(int(chunks.sum()), t_in, cfg.feat_dim, generator=gen)
            pe_before = ses[3].pe_index
            enc, y = eng.encode_stream_chunks_v(ids, chunks, feats)
            enc, y = enc.cpu(), y.cpu()
            off = offsets(chunks)
            for i, s in enumerate(ses):
                for j in range(chunks[i]):
                    eo, yo = s.step_feats(feats[off[i] + j].unsqueeze(0))
                    assert maxabs(enc[off[i] + j], eo[0]) < FP32_TOL and maxabs(y[off[i] + j], yo[0]) < FP32_TOL, (call, i, j)
                nf[i] += int(chunks[i]) * t
                sid = int(ids[i])
                assert eng.state(sid) == (nf[i], s.pe_index), (call, i)
                for li in range(cfg.n_layers):
                    k, v = eng.export_kv(sid, li)
                    assert maxabs(k, s.buffer[li][0]) < FP32_TOL and maxabs(v, s.buffer[li][1]) < FP32_TOL, (call, i, li)
                assert maxabs(eng.export_adapter_cache(sid), s.cache[0]) < FP32_TOL, (call, i)
            if call == 0:                         # session 3's pe_index wrapped inside this call
                assert chunks[3] >= 2 and ses[3].pe_index < pe_before
    finally:
        eng.close()


# ---- 2. every variant against uniform calls of twin sessions --------------------------------------------------------------
def _variant(name):
    if name in ("cnn", "two"):
        base = path_config_from_dict(load_yaml("tiny_bn"))
        return dataclasses.replace(base, adapter_type="cnn") if name == "cnn" else dataclasses.replace(base, llm_dim=base.d_model * 4 + 64)
    if name == "fork_t7":
        return load_path_config("tiny")
    return load_path_config(name)


VARIANTS = ["tiny_linear", "cnn", "two", "tiny_bn", "tiny_conv1d", "tiny_postnorm_concat", "fork_t7"]
MIXES = [[1, 3, 1, 7], [2, 1, 5, 1], [1, 1, 1, 4], [6, 2, 2, 3]]


def _twin_run(eng, cfg, t_in, a, b, feats_fn, mixes=MIXES):
    """Sessions a by mixed calls, twins b by one uniform encode_stream_chunks(k_i) call per session; yields per call."""
    for call, mix in enumerate(mixes):
        chunks = np.array(mix, np.int32)
        per = [feats_fn(call, i, k) for i, k in enumerate(chunks)]
        enc, y = eng.encode_stream_chunks_v(a, chunks, pack(per))
        off = offsets(chunks)
        twins = [eng.encode_stream_chunks(b[i:i + 1], per[i].unsqueeze(0)) for i in range(len(chunks))]
        yield call, chunks, off, enc, y, twins


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name", VARIANTS)
def test_variants_vs_uniform_twin_calls(name, dtype):
    cfg = _variant(name)
    t_in = 32 if name == "fork_t7" else cfg.chunk_feat_frames
    eng = engine(cfg, adapter_seed=5 if name in ("cnn", "two") else 3, dtype=dtype, max_sessions=8)
    tol = FP32_TOL if dtype == torch.float32 else TWIN_BF16_TOL
    try:
        a, b = eng.alloc(4), eng.alloc(4)
        feats = rand_feats(cfg, (4, 20, t_in), 14)
        pos = [0] * 4

        def feats_fn(call, i, k):
            f = feats[i, pos[i]:pos[i] + k]
            pos[i] += k
            return f
        worst, exact = 0.0, True
        for call, chunks, off, enc, y, twins in _twin_run(eng, cfg, t_in, a, b, feats_fn):
            for i, (te, ty) in enumerate(twins):
                ge, gy = enc[off[i]:off[i + 1]], y[off[i]:off[i + 1]]
                worst = max(worst, maxabs(ge.cpu(), te[0].cpu()), maxabs(gy.cpu(), ty[0].cpu()))
                exact = exact and torch.equal(ge, te[0]) and torch.equal(gy, ty[0])
                assert eng.state(int(a[i])) == eng.state(int(b[i])), (call, i)
                if cfg.adapter_type == "subsampling":
                    for w in range(2 if cfg.adapter_two_conv else 1):
                        assert maxabs(eng.export_adapter_cache(int(a[i]), w), eng.export_adapter_cache(int(b[i]), w)) < tol, (call, i, w)
                if name == "tiny_conv1d":
                    assert maxabs(eng.export_ffn_cache(int(a[i]), 0), eng.export_ffn_cache(int(b[i]), 0)) < tol
            assert worst < tol, (call, worst)
        print("%s %s: mixed vs uniform twins max-abs %.3g, bit-identical: %s" % (name, dtype, worst, exact))
    finally:
        eng.close()


# ---- 3. equal counts are the old call --------------------------------------------------------------------------------------
@pytest.mark.parametrize("which", ["tiny", "shipped"])
def test_uniform_counts_are_the_old_calls(which):
    cfg = load_path_config(which)
    kw = dict(dtype=torch.bfloat16, seed=0, adapter_seed=0) if which == "shipped" else {}
    eng = engine(cfg, max_sessions=8, **kw)
    try:
        for n in (1, 2, 3):                         # shipped bf16 at 1-2 sessions: the single-chunk calls take the stack kernel
            a, b = eng.alloc(n), eng.alloc(n)
            feats = rand_feats(cfg, (n, 12, cfg.chunk_feat_frames), 30 + n)
            c0 = 0
            for k in (1, 3, 1, 7):
                f = feats[:, c0:c0 + k].contiguous()
                e1, y1 = eng.encode_stream_chunks_v(a, np.full(n, k, np.int32), f.reshape(n * k, *f.shape[2:]))
                if k == 1:
                    e2, y2 = eng.encode_stream(b, f[:, 0].contiguous())
                else:
                    e2, y2 = eng.encode_stream_chunks(b, f)
                assert torch.equal(e1, e2.reshape(e1.shape)) and torch.equal(y1, y2.reshape(y1.shape)), (n, k)
                c0 += k
            eng.free(a)
            eng.free(b)
    finally:
        eng.close()


# ---- 4. hand-off ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["tiny_linear", "cnn", "two", "tiny_bn", "fork_t7"])
def test_handoff_mixed_counts(name):
    """An armed mixed call writes, behind the prefix of block off_i + j, the fp32 adapter rows of a twin mixed call rounded to
    fp16 bit for bit; prefix and trailing rows untouched; mask rows and row_start exact."""
    cfg = _variant(name)
    t_in = 32 if name == "fork_t7" else cfg.chunk_feat_frames
    eng = engine(cfg, adapter_seed=5 if name in ("cnn", "two") else 3, dtype=torch.bfloat16, max_sessions=8)
    try:
        a, b = eng.alloc(3), eng.alloc(3)
        _, t_out = eng.out_frames(t_in)
        P, R = 3, 3 + t_out + 2
        g = torch.Generator().manual_seed(22)
        for call, mix in enumerate([[1, 4, 2], [3, 1, 1], [1, 1, 6]]):
            chunks = np.array(mix, np.int32)
            B = int(chunks.sum())
            f = rand_feats(cfg, (B, t_in), 40 + call)
            emb = torch.randn(B, R, cfg.llm_dim, generator=g).half().cuda()
            before = emb.clone()
            mask = torch.full((B, R), 7, dtype=torch.uint8, device="cuda")
            start = torch.full((B,), -1, dtype=torch.int32, device="cuda")
            onset = [(i + call) % 3 == 0 for i in range(B)]
            eng.handoff_arm(B, emb, P, onset, None, mask, start)
            eng.encode_stream_chunks_v(a, chunks, f, want_adapter=False)
            _, y = eng.encode_stream_chunks_v(b, chunks, f)
            torch.cuda.synchronize()
            assert torch.equal(emb[:, P:P + t_out], y.half()), call
            assert torch.equal(emb[:, :P], before[:, :P]) and torch.equal(emb[:, P + t_out:], before[:, P + t_out:]), call
            for r in range(B):
                want = [1 if onset[r] else 0] * P + [1] * t_out + [0] * (R - P - t_out)
                assert mask[r].tolist() == want and int(start[r]) == (0 if onset[r] else P), (call, r)
            for s, r in zip(a, b):
                assert eng.state(int(s)) == eng.state(int(r))
                if cfg.adapter_type == "subsampling":
                    for w in range(2 if cfg.adapter_two_conv else 1):
                        assert torch.equal(eng.export_adapter_cache(int(s), w), eng.export_adapter_cache(int(r), w)), (call, w)
    finally:
        eng.close()


# ---- 5. graphs ------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def shipped16():
    cfg = load_path_config("shipped")
    eng = engine(cfg, seed=0, adapter_seed=0, dtype=torch.bfloat16, max_sessions=160)
    yield cfg, eng
    eng.close()


def test_new_mix_with_the_same_totals_replays_the_graph(shipped16):
    cfg, eng = shipped16
    a, b = eng.alloc(4), eng.alloc(4)
    mix_a, mix_b = np.array([1, 1, 3, 2], np.int32), np.array([1, 1, 2, 3], np.int32)    # 4 sessions, 7 blocks, kmax 3, n1 2
    feats = rand_feats(cfg, (4 * 7, cfg.chunk_feat_frames), 50)
    try:
        outs = []
        for call, mix in enumerate([mix_a, mix_a, mix_b]):
            r0 = eng.stats()["graph_replays"]
            outs.append(eng.encode_stream_chunks_v(a, mix, feats[7 * call:7 * call + 7].contiguous()))
            torch.cuda.synchronize()
            if call == 2:                         # first call of mix_b: a replay of mix_a's graph, not an eager first run
                assert eng.stats()["graph_replays"] == r0 + 1
        eng.set_option("use_graph", 0)
        try:
            for call, mix in enumerate([mix_a, mix_a, mix_b]):
                e, y = eng.encode_stream_chunks_v(b, mix, feats[7 * call:7 * call + 7].contiguous())
                assert torch.equal(e, outs[call][0]) and torch.equal(y, outs[call][1]), call
        finally:
            eng.set_option("use_graph", 1)
    finally:
        eng.free(a)
        eng.free(b)


# ---- 6. shipped bf16 at the benchmarked size -------------------------------------------------------------------------------
@pytest.mark.parametrize("n_onset", [1, 8])
def test_shipped_64_sessions_onset_mix(shipped16, n_onset):
    """64 sessions, n_onset of them at 7 chunks: one sampled session of each kind against the oracle on bf16-rounded weights,
    and all of them against twins run with the grouped two-call plan (encode_stream + encode_stream_chunks(7))."""
    cfg, eng = shipped16
    n = 64
    chunks = np.array([1] * (n - n_onset) + [7] * n_onset, np.int32)
    a, b = eng.alloc(n), eng.alloc(n)
    esd, asd = bf16_weights(make_encoder_state(cfg, 0)), bf16_weights(make_adapter_state(cfg, 0))
    sample = [0, n - 1]
    ses = [O.StreamSession(cfg, esd, asd) for _ in sample]
    try:
        warm = rand_feats(cfg, (2, n, cfg.chunk_feat_frames), 60 + n_onset)
        for i in range(2):
            eng.encode_stream(a, warm[i])
            eng.encode_stream(b, warm[i])
            for s, q in zip(ses, sample):
                s.step_feats(warm[i, q:q + 1])
        B = int(chunks.sum())
        f = rand_feats(cfg, (B, cfg.chunk_feat_frames), 70 + n_onset)
        enc, y = eng.encode_stream_chunks_v(a, chunks, f)
        n1 = n - n_onset
        e1, y1 = eng.encode_stream(b[:n1], f[:n1].contiguous())
        e7, y7 = eng.encode_stream_chunks(b[n1:], f[n1:].reshape(n_onset, 7, *f.shape[1:]).contiguous())
        tw = max(maxabs(enc[:n1].cpu(), e1.cpu()), maxabs(y[:n1].cpu(), y1.cpu()),
                 maxabs(enc[n1:].cpu(), e7.reshape(-1, *e7.shape[2:]).cpu()), maxabs(y[n1:].cpu(), y7.reshape(-1, *y7.shape[2:]).cpu()))
        off = offsets(chunks)
        wo = 0.0
        for s, q in zip(ses, sample):
            for j in range(chunks[q]):
                eo, yo = s.step_feats(f[off[q] + j].unsqueeze(0))
                wo = max(wo, maxabs(enc[off[q] + j].cpu(), eo[0]), maxabs(y[off[q] + j].cpu(), yo[0]))
        for s, r in zip(a, b):
            assert eng.state(int(s)) == eng.state(int(r))
        print("64 sessions, %d at 7 chunks: vs oracle on bf16 weights %.3g, vs grouped twins %.3g" % (n_onset, wo, tw))
        assert wo < BF16_TOL and tw < TWIN_BF16_TOL
    finally:
        eng.free(a)
        eng.free(b)


# ---- 7. refusals ----------------------------------------------------------------------------------------------------------
def test_refusals_enqueue_nothing():
    from freeze_omni_b200 import _lib
    cfg = load_path_config("tiny")
    eng = engine(cfg, dtype=torch.bfloat16, max_sessions=8)
    t_in = cfg.chunk_feat_frames
    try:
        a, b = eng.alloc(2), eng.alloc(2)
        f = rand_feats(cfg, (40, t_in), 80)
        eng.encode_stream_chunks_v(a, [1, 2], f[:3])
        eng.encode_stream_chunks_v(b, [1, 2], f[:3])
        before = [eng.state(int(s)) for s in a]
        with pytest.raises(_lib.FoError, match="counts must be >= 1"):
            _lib.check(eng.lib.fo_encode_stream_chunks_v(eng._h, a.ctypes.data_as(_lib._I32P),
                                                         np.array([0, 2], np.int32).ctypes.data_as(_lib._I32P), 2,
                                                         f.data_ptr(), t_in, None, None, eng._stream()))
        with pytest.raises(_lib.FoError, match=r"session 1 \(id %d\).*largest count is 16" % int(a[1])):
            eng.encode_stream_chunks_v(a, [1, 17], f[:18])
        with pytest.raises(_lib.FoError, match="not allocated"):
            eng.encode_stream_chunks_v(np.array([int(a[0]), 7], np.int32), [1, 1], f[:2])
        with pytest.raises(_lib.FoError, match="context allows"):
            eng.encode_stream_chunks_v(a, [1, 1], rand_feats(cfg, (2, 4 * 40 + 3), 81))
        rc = eng.lib.fo_encode_stream_chunks_v(eng._h, a.ctypes.data_as(_lib._I32P), np.array([1, 1], np.int32).ctypes.data_as(_lib._I32P),
                                               2, None, t_in, None, None, eng._stream())
        assert rc == -1 and b"feats" in eng.lib.fo_last_error()
        emb = torch.zeros(8, 3 + 2, cfg.llm_dim, dtype=torch.float16, device="cuda")
        eng.handoff_arm(2, emb, 3, [0, 1])
        with pytest.raises(_lib.FoError, match="armed for 2 blocks"):
            eng.encode_stream_chunks_v(a, [1, 2], f[3:6], want_adapter=False)
        assert [eng.state(int(s)) for s in a] == before
        e1, y1 = eng.encode_stream_chunks_v(a, [2, 1], f[6:9])
        e2, y2 = eng.encode_stream_chunks_v(b, [2, 1], f[6:9])
        assert torch.equal(e1, e2) and torch.equal(y1, y2)
    finally:
        eng.close()


# ---- 8. the scheduler on the gating golden ---------------------------------------------------------------------------------
def _gating_run(eng, g, max_chunks, mixed, handoff=None):
    from freeze_omni_b200.scheduler import StreamScheduler
    sch = StreamScheduler(eng, history_chunks=10, onset_chunks=6, bucket=4, max_sessions=2, max_chunks=max_chunks, mixed_calls=mixed)
    sch.open("u")
    sch.open("v")
    sch.block_log = []
    blocks, calls = [], []
    try:
        for i, st in enumerate(g["statuses"]):
            x = g["pcm"][i * 2560:(i + 1) * 2560].astype(np.float32) / 32768.0
            sch.push("u", x, str(st) if str(st) else None)
            sch.push("v", x[::-1].copy(), "ipu_cl")
            c0 = sch.stats["encode_calls"]
            out = sch.tick(float(g["scale"]), handoff=handoff)
            calls.append((len(out.get("u", [])), sch.stats["encode_calls"] - c0))
            for s in ("u", "v"):
                for blk in out.get(s, []):
                    start = None
                    if handoff is not None:
                        row = (blk.emb.data_ptr() - handoff.embeds.data_ptr()) // (handoff.embeds.stride(0) * 2)
                        start = int(handoff.row_start[row])
                    blocks.append((s, blk.status, blk.enc.cpu().clone(), None if blk.emb is None else blk.emb.float().cpu().clone(),
                                   None if blk.mask is None else blk.mask.cpu().clone(), start))
        return blocks, calls, [lab for _, _, lab in sch.block_log]
    finally:
        for s in list(sch.keys):
            sch.close(s)
        eng.free(sch.scratch)


@pytest.mark.parametrize("with_handoff", [False, True])
def test_scheduler_mixed_calls_on_gating_golden(golden, with_handoff):
    from freeze_omni_b200.scheduler import Handoff
    cfg = load_path_config("tiny")
    g = golden("gating")
    eng = engine(cfg, dtype=torch.bfloat16, max_sessions=12)
    try:
        ho1 = hom = None
        if with_handoff:
            prefix = torch.randn(1, 3, cfg.llm_dim, generator=torch.Generator().manual_seed(3))
            ho1, hom = Handoff(eng, 64, prefix), Handoff(eng, 64, prefix)
        ref, calls1, labels1 = _gating_run(eng, g, 1, False, ho1)
        got, callsm, labelsm = _gating_run(eng, g, 7, True, hom)
        assert labels1 == labelsm
        assert [r[:2] for r in ref] == [q[:2] for q in got]
        for r, q in zip(ref, got):
            assert maxabs(r[2], q[2]) < BF16_TOL and r[5] == q[5]
            if r[3] is not None:
                assert maxabs(r[3], q[3]) < BF16_TOL
            if r[4] is not None:
                assert torch.equal(r[4], q[4])
        onset_ticks = [c for c in callsm if c[0] == 7]
        assert onset_ticks and all(c[1] == 1 for c in onset_ticks)
    finally:
        eng.close()
