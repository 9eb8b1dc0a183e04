"""The LLM hand-off of the recording entries (fo_stream_steps_v, fo_encode_stream_steps_v armed by fo_handoff_arm) and of
StreamScheduler.replay(handoff=).  Every block's fp16 rows must be .half() of the fp32 adapter rows the same call returns
without an arm, bit for bit; its mask row and row_start the torch sequence of models/audioLLM.py:404-420; nothing else in the
caller's buffers may change, and a refused call must leave the sessions and the arm as they were."""
import dataclasses
import random

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config, load_yaml, path_config_from_dict
from freeze_omni_b200.scheduler import IPU_CONT, IPU_START, Handoff, StreamScheduler, plan_gated_replay
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state

pytestmark = pytest.mark.gpu

# bf16 twin sessions encoded at other batchings (the bar of the multi-chunk, recording and replay tests)
TWIN_BF16_TOL = 4e-3
PREFIX_MASK = [1, 0, 1, 1, 0]


def pcm_blocks(cfg, n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(-3000, 3000, (n, cfg.samples_per_chunk), generator=g, dtype=torch.int32).to(torch.int16)


def config(name):
    if name == "fork_t7":                       # odd t: 28 + 4 frames per chunk give 7 encoder frames
        y = load_yaml("tiny")
        y["frontend"] = dict(y["frontend"], frame_length_ms=16, frame_shift_ms=8, frames_per_chunk=28, context_frames=4)
        return path_config_from_dict(y)
    if name in ("cnn", "two"):
        base = path_config_from_dict(load_yaml("tiny_bn"))
        return dataclasses.replace(base, adapter_type="cnn") if name == "cnn" else dataclasses.replace(base, llm_dim=base.d_model * 4 + 64)
    return load_path_config(name)


def engine(cfg, **kw):
    from freeze_omni_b200.engine import Engine
    return Engine(cfg, make_encoder_state(cfg, 3), make_adapter_state(cfg, 5), dtype=torch.bfloat16, **kw)


class Buffers:
    """Hand-off buffers of B blocks with `tail` spare rows past prefix + t_out, every entry pre-filled with sentinels."""

    def __init__(self, eng, B, P=len(PREFIX_MASK), tail=2, seed=0):
        g = torch.Generator().manual_seed(seed)
        dev = eng.torch_device
        self.P, self.t_out = P, eng.out_frames(eng.cfg.chunk_feat_frames)[1]
        self.rows = P + self.t_out + tail
        self.embeds = torch.randn(B, self.rows, eng.cfg.llm_dim, generator=g).half().to(dev)
        self.attn_mask = torch.full((B, self.rows), 7, dtype=torch.uint8, device=dev)
        self.row_start = torch.full((B,), -1, dtype=torch.int32, device=dev)
        self.prefix_mask = torch.tensor(PREFIX_MASK[:P], dtype=torch.uint8, device=dev)
        self.before = self.embeds.clone()

    def arm(self, eng, onset, n=None):
        eng.handoff_arm(len(onset) if n is None else n, self.embeds, self.P, onset, self.prefix_mask, self.attn_mask, self.row_start)

    def check(self, y, onset, tag):
        """Blocks [0, len(y)) against the fp32 adapter rows y of a twin call; the rest of the buffers untouched."""
        B, P, t_out = len(onset), self.P, self.t_out
        e = self.embeds.cpu()
        assert torch.equal(e[:B, P:P + t_out], y.cpu().half()), tag                  # audioLLM.py:410
        assert torch.equal(e[:B, :P], self.before[:B, :P].cpu()), tag                 # the chat prefix stays the caller's
        assert torch.equal(e[:B, P + t_out:], self.before[:B, P + t_out:].cpu()), tag
        assert torch.equal(e[B:], self.before[B:].cpu()), tag
        # audioLLM.py:404-406,418-420: attention_mask = cat(prefix_mask, ones) on an onset block, else ones behind zeros
        on = torch.tensor([bool(o) for o in onset])
        pm = self.prefix_mask.cpu()
        want = torch.zeros(B, self.rows, dtype=torch.uint8)
        want[:, :P] = torch.where(on[:, None], pm[None, :], torch.zeros_like(pm)[None, :])
        want[:, P:P + t_out] = 1
        assert torch.equal(self.attn_mask[:B].cpu(), want), tag
        assert torch.equal(self.row_start[:B].cpu(), torch.where(on, 0, P).to(torch.int32)), tag
        assert (self.attn_mask[B:] == 7).all() and (self.row_start[B:] == -1).all(), tag


def onset_pattern(B, seed):
    rng = random.Random(seed)
    return [int(rng.random() < 0.3) for _ in range(B)]


def records(eng, ids):
    torch.cuda.synchronize()
    return eng.save_sessions([int(s) for s in ids]).cpu()


@pytest.fixture(scope="module")
def shipped():
    cfg = load_path_config("shipped")
    eng = engine(cfg, max_sessions=12)
    yield cfg, eng
    eng.close()


# ---- 1. fo_stream_steps_v with an arm for sum(chunks) blocks ---------------------------------------------------------------
def test_stream_steps_v_handoff_shipped(shipped):
    """Passes of 6 blocks over counts [1, 7, 13, 3]: sessions split across passes; twins take adapter_out and no arm."""
    cfg, eng = shipped
    a, b = eng.alloc(4), eng.alloc(4)
    try:
        eng.set_option("steps_pass_blocks", 6)
        counts = [1, 7, 13, 3]
        B = sum(counts)
        for rnd in range(2):                          # the second call continues from the state the first left
            pcm = pcm_blocks(cfg, B, 10 + rnd)
            onset = onset_pattern(B, rnd)
            buf = Buffers(eng, B + 3, seed=rnd)
            sat0 = eng.stats()["act_saturations"]
            buf.arm(eng, onset)
            ea, ya = eng.stream_steps_v(a, counts, pcm, want_adapter=False)
            assert ya is None
            eb, yb = eng.stream_steps_v(b, counts, pcm)
            torch.cuda.synchronize()
            assert torch.equal(ea.cpu(), eb.cpu()), rnd
            buf.check(yb, onset, rnd)
            assert torch.equal(records(eng, a), records(eng, b)), rnd
            assert eng.stats()["act_saturations"] == sat0 == 0
    finally:
        eng.set_option("steps_pass_blocks", 0)
        eng.free(a)
        eng.free(b)


# ---- 2. fo_encode_stream_steps_v on fbank_stream_v features, every adapter variant -------------------------------------------
def _encode_vs_twin(cfg, eng, counts, pass_blocks, seed):
    eng.set_option("steps_pass_blocks", pass_blocks)
    a, b = eng.alloc(len(counts)), eng.alloc(len(counts))
    B = sum(counts)
    feats = eng.fbank_stream_v(a, counts, pcm_blocks(cfg, B, seed))
    onset = onset_pattern(B, seed)
    buf = Buffers(eng, B, seed=seed)
    buf.arm(eng, onset)
    ea, _ = eng.encode_stream_steps_v(a, counts, feats, want_adapter=False)
    eb, yb = eng.encode_stream_steps_v(b, counts, feats)
    torch.cuda.synchronize()
    assert torch.equal(ea.cpu(), eb.cpu())
    buf.check(yb, onset, (cfg.adapter_type, seed))
    # the features session a's fbank moved are not in b; the encoder state is compared through the next armed call
    feats2 = torch.randn(B, cfg.chunk_feat_frames, cfg.feat_dim, generator=torch.Generator().manual_seed(seed), device="cpu").cuda() * 3 + 9
    buf2 = Buffers(eng, B, seed=seed + 1)
    buf2.arm(eng, onset)
    eng.encode_stream_steps_v(a, counts, feats2, want_adapter=False)
    _, yb2 = eng.encode_stream_steps_v(b, counts, feats2)
    torch.cuda.synchronize()
    buf2.check(yb2, onset, (cfg.adapter_type, seed, 2))
    for s, t in zip(a, b):
        assert eng.state(int(s)) == eng.state(int(t))
    eng.free(a)
    eng.free(b)


def test_encode_stream_steps_v_handoff_shipped(shipped):
    cfg, eng = shipped
    try:
        _encode_vs_twin(cfg, eng, [1, 7, 13, 3], 6, 20)
        assert eng.stats()["act_saturations"] == 0
    finally:
        eng.set_option("steps_pass_blocks", 0)


@pytest.mark.parametrize("name", ["tiny", "tiny_linear", "cnn", "two", "tiny_bn", "tiny_conv1d", "tiny_postnorm_concat", "fork_t7"])
def test_encode_stream_steps_v_handoff_variants(name):
    cfg = config(name)
    eng = engine(cfg, max_sessions=8)
    try:
        _encode_vs_twin(cfg, eng, [5, 1, 17], 4, 30)
        assert eng.stats()["act_saturations"] == 0
    finally:
        eng.close()


# ---- 3. refusals keep the sessions and the arm ------------------------------------------------------------------------------
def test_refusals_keep_the_arm():
    cfg = load_path_config("tiny")
    eng = engine(cfg, max_sessions=6)
    try:
        ids, twin = eng.alloc(2), eng.alloc(2)
        counts = [3, 2]
        B = sum(counts)
        pcm = pcm_blocks(cfg, B, 1)
        feats = torch.zeros(B, cfg.chunk_feat_frames, cfg.feat_dim, device=eng.torch_device)
        onset = onset_pattern(B, 2)
        for wrong in (B - 1, B + 1):
            buf = Buffers(eng, B + 1)
            buf.arm(eng, (onset + [1])[:wrong], n=wrong)
            before, l0 = records(eng, ids), eng.stats()["kernel_launches"]
            with pytest.raises(RuntimeError, match="armed"):
                eng.stream_steps_v(ids, counts, pcm, want_adapter=False)
            with pytest.raises(RuntimeError, match="armed"):
                eng.encode_stream_steps_v(ids, counts, feats, want_adapter=False)
            assert eng.stats()["kernel_launches"] == l0 and torch.equal(records(eng, ids), before), wrong
            assert torch.equal(buf.embeds, buf.before), wrong
            # the arm is still there: a call of `wrong` blocks takes it (and the twins follow, to keep the states equal)
            c2 = [wrong - 1, 1]
            eng.stream_steps_v(ids, c2, pcm_blocks(cfg, wrong, 3), want_adapter=False)
            _, y = eng.stream_steps_v(twin, c2, pcm_blocks(cfg, wrong, 3))
            torch.cuda.synchronize()
            buf.check(y, (onset + [1])[:wrong], wrong)
        # adapter_out with an arm
        buf = Buffers(eng, B)
        buf.arm(eng, onset)
        before, l0 = records(eng, ids), eng.stats()["kernel_launches"]
        with pytest.raises(RuntimeError, match="armed"):
            eng.stream_steps_v(ids, counts, pcm)
        with pytest.raises(RuntimeError, match="armed"):
            eng.encode_stream_steps_v(ids, counts, feats)
        assert eng.stats()["kernel_launches"] == l0 and torch.equal(records(eng, ids), before)
        assert torch.equal(buf.embeds, buf.before)
        eng.stream_steps_v(ids, counts, pcm, want_adapter=False)
        _, y = eng.stream_steps_v(twin, counts, pcm)
        torch.cuda.synchronize()
        buf.check(y, onset, "adapter_out")
        assert torch.equal(records(eng, ids), records(eng, twin))
    finally:
        eng.close()


def test_two_slots_take_an_arm_for_800_blocks():
    """fo_handoff_arm admits the block count of any recording call: 2 sessions x 400 chunks on a 2-slot context."""
    cfg = load_path_config("tiny")
    eng = engine(cfg, max_sessions=2)
    try:
        ids = eng.alloc(2)
        counts = [400, 400]
        B = sum(counts)
        feats = 9.0 + 3.0 * torch.randn(B, cfg.chunk_feat_frames, cfg.feat_dim, generator=torch.Generator().manual_seed(4))
        feats = feats.cuda()
        onset = onset_pattern(B, 5)
        buf = Buffers(eng, B)
        buf.arm(eng, onset)
        eng.encode_stream_steps_v(ids, counts, feats, want_adapter=False)
        after = eng.state(int(ids[0])), eng.state(int(ids[1]))
        eng.reset(ids)                                # the same call again from fresh sessions, with adapter_out
        _, y = eng.encode_stream_steps_v(ids, counts, feats)
        torch.cuda.synchronize()
        assert (eng.state(int(ids[0])), eng.state(int(ids[1]))) == after
        buf.check(y, onset, "800")
    finally:
        eng.close()


# ---- 4. StreamScheduler.replay(handoff=) ------------------------------------------------------------------------------------
def conversations(rng, lengths):
    """Silence before the first onset in most sessions; onsets land inside and across the small windows."""
    out = []
    for i, n in enumerate(lengths):
        s, speaking = [], i == 0
        while len(s) < n:
            s += [IPU_START] + [IPU_CONT] * rng.randint(0, 9) if speaking else [None] * rng.randint(1, 12)
            speaking = not speaking
        out.append(s[:n])
    return out


def _prefix(cfg, P, seed):
    return torch.randn(1, P, cfg.llm_dim, generator=torch.Generator().manual_seed(seed))


def test_replay_handoff_vs_replay_and_ticks(shipped):
    cfg, eng = shipped
    P = len(PREFIX_MASK)
    prefix, pmask = _prefix(cfg, P, 1), torch.tensor(PREFIX_MASK, dtype=torch.uint8)
    rng = random.Random(3)
    statuses = conversations(rng, [41, 60, 23])
    n = len(statuses)
    pcm = [pcm_blocks(cfg, len(s), 40 + i) for i, s in enumerate(statuses)]
    H, O = 10, 6
    total = sum(len(plan_gated_replay(s, H, O).blocks) for s in statuses)
    sch = StreamScheduler(eng, history_chunks=H, onset_chunks=O, bucket=1, max_sessions=3 * n)
    try:
        eng.set_option("steps_pass_blocks", 12)           # windows of 12 chunks: several per recording
        for i in range(n):
            for tag in "hrt":
                sch.open((tag, i))
        ho = Handoff(eng, total + 4, prefix, pmask)
        before = ho.embeds.clone()
        got = sch.replay({("h", i): (pcm[i], s) for i, s in enumerate(statuses)}, handoff=ho)
        ref = sch.replay({("r", i): (pcm[i], s) for i, s in enumerate(statuses)})
        torch.cuda.synchronize()
        # ticks with max_chunks=1, their hand-off copied out after every tick (the next one reuses the buffers)
        ho_t = Handoff(eng, n * (1 + O), prefix, pmask)
        ticks = {}
        for j in range(max(len(s) for s in statuses)):
            for i, s in enumerate(statuses):
                if j < len(s):
                    sch.push(("t", i), pcm[i][j], s[j])
            for k, bl in sch.tick(handoff=ho_t).items():
                ticks.setdefault(k[1], []).extend(b._replace(emb=b.emb.clone(), mask=b.mask.clone()) for b in bl)
        seen = []
        t_out = ho.rows - P
        for i in range(n):
            g, r, t = got.get(("h", i), []), ref.get(("r", i), []), ticks.get(i, [])
            assert [b.status for b in g] == [b.status for b in r] == [b.status for b in t], i
            for blk, rb, tb in zip(g, r, t):
                on = blk.status == IPU_START
                idx = (blk.mask.data_ptr() - ho.attn_mask.data_ptr()) // ho.rows
                seen.append(idx)
                assert blk.emb.data_ptr() == ho.embeds[idx, 0 if on else P:].data_ptr()
                assert torch.equal(blk.enc, rb.enc)
                assert torch.equal(blk.emb[-t_out:], rb.emb.half())                         # .half() of the twin's rows
                assert torch.equal(blk.mask, tb.mask) and blk.emb.shape == tb.emb.shape
                assert int(ho.row_start[idx]) == (0 if on else P)
                if on:
                    assert torch.equal(blk.emb[:P], tb.emb[:P])                              # the chat prefix
                w = tb.emb[-t_out:].float()
                assert ((blk.emb[-t_out:].float() - w).abs() <= TWIN_BF16_TOL + w.abs() * 2.0 ** -10).all(), (i, blk.status)
        assert sorted(seen) == list(range(total))
        assert torch.equal(ho.embeds[total:], before[total:]) and (ho.attn_mask[total:] == 0).all()
        for i in range(n):
            for other in "rt":
                assert torch.equal(sch.history(("h", i)), sch.history((other, i))), (i, other)
            assert torch.equal(records(eng, [sch.keys[("h", i)]]), records(eng, [sch.keys[("r", i)]])), i
        assert eng.stats()["act_saturations"] == 0
    finally:
        eng.set_option("steps_pass_blocks", 0)
        for k in list(sch.keys):
            sch.close(k)


# ---- 5. a replay over the Handoff capacity runs nothing -----------------------------------------------------------------------
def test_replay_over_capacity_touches_nothing(shipped):
    cfg, eng = shipped
    P = len(PREFIX_MASK)
    statuses = [[None, None, IPU_START, IPU_CONT, None], [IPU_CONT, None, IPU_START]]
    total = sum(len(plan_gated_replay(s, 4, 2).blocks) for s in statuses)
    sch = StreamScheduler(eng, history_chunks=4, onset_chunks=2, bucket=1, max_sessions=2)
    try:
        for i in range(2):
            sch.open(i)
        sch.replay({i: (pcm_blocks(cfg, 3, 60 + i), [None, IPU_START, None]) for i in range(2)})   # non-zero history and state
        ho = Handoff(eng, total - 1, _prefix(cfg, P, 2), torch.tensor(PREFIX_MASK, dtype=torch.uint8))
        keep = [t.clone() for t in (ho.embeds, ho.attn_mask, ho.row_start)]
        recs, hist = records(eng, [sch.keys[i] for i in range(2)]), [sch.history(i).clone() for i in range(2)]
        stats = dict(sch.stats)
        with pytest.raises(RuntimeError, match="capacity"):
            sch.replay({i: (pcm_blocks(cfg, len(s), 70 + i), s) for i, s in enumerate(statuses)}, handoff=ho)
        assert sch.stats == stats
        assert torch.equal(records(eng, [sch.keys[i] for i in range(2)]), recs)
        for i in range(2):
            assert torch.equal(sch.history(i), hist[i])
        for a, b in zip((ho.embeds, ho.attn_mask, ho.row_start), keep):
            assert torch.equal(a, b)
    finally:
        for k in list(sch.keys):
            sch.close(k)
