"""Host logic of the gated replay (no GPU): plan_gated_replay against `tick`'s gating rule run chunk by chunk, against the
reference's blocks of tests/golden/gating.npz, and StreamScheduler.replay driven through a fake engine against a tick loop."""
import random

import numpy as np
import pytest
import torch

from freeze_omni_b200.scheduler import IPU_CONT, IPU_START, ReplaySource, StreamScheduler, plan_gated_replay

T_IN, F, SPC = 19, 80, 2560


class FakeCfg:
    chunk_feat_frames, feat_dim, samples_per_chunk = T_IN, F, SPC


class TagEngine:
    """Fake engine whose fbank blocks carry the slot's running chunk number (1, 2, ...) in every element, so a block's value
    names the chunk it came from; the encoder returns slices of its input.  Offers both the tick and the replay calls."""

    def __init__(self, pass_blocks=5):
        self.cfg, self.torch_device, self.max_sessions = FakeCfg(), torch.device("cpu"), 64
        self.next_slot, self.pass_blocks, self.seen = 0, pass_blocks, {}
        self.calls = []

    def stats(self):
        return {"sessions_in_use": self.next_slot}

    def alloc(self, n):
        ids = np.arange(self.next_slot, self.next_slot + n, dtype=np.int32)
        self.next_slot += n
        return ids

    def free(self, ids):
        pass

    def get_option(self, name):
        assert name == "steps_pass_blocks_in_use"
        return self.pass_blocks

    def _tags(self, ids, counts):
        out = []
        for s, c in zip(ids, counts):
            for _ in range(c):
                self.seen[int(s)] = self.seen.get(int(s), 0) + 1
                out.append(float(self.seen[int(s)]))
        return torch.tensor(out).view(-1, 1, 1).expand(len(out), T_IN, F).clone()

    def fbank_stream(self, ids, pcm, scale=None):
        return self._tags(ids, [1] * len(ids))

    def fbank_stream_v(self, ids, chunks, pcm, scale=None):
        assert pcm.shape == (sum(chunks), SPC) and all(c >= 1 for c in chunks)
        self.calls.append(("fbank", list(ids), list(chunks)))
        return self._tags(ids, chunks)

    def encode_stream(self, ids, feats):
        return feats[:, :4, :8].clone(), feats[:, :2, :4].clone()

    def encode_stream_steps_v(self, ids, chunks, feats):
        assert feats.shape[0] == sum(chunks) and all(c >= 1 for c in chunks)
        self.calls.append(("encode", list(ids), list(chunks)))
        return feats[:, :4, :8].clone(), feats[:, :2, :4].clone()


def tick_reference(statuses, H, O):
    """`tick` itself, one chunk per tick, on a TagEngine: history slot h pre-filled with -(h + 1) so that every queued block
    and every history row names its source.  Returns ([(source, label)], [history sources])."""
    eng = TagEngine()
    sch = StreamScheduler(eng, history_chunks=H, onset_chunks=O, bucket=1, max_sessions=2)
    sch.open("s")
    sch.history("s")[:] = -torch.arange(1, H + 1, dtype=torch.float32).view(H, 1, 1)
    sch.block_log = []
    for st in statuses:
        sch.push("s", np.zeros(SPC, np.int16), st)
        sch.tick()

    def source(v):
        v = int(v)
        return ReplaySource("history", -v - 1) if v < 0 else ReplaySource("chunk", v - 1)

    blocks = [(source(b[0, 0]), lab) for _, b, lab in sch.block_log]
    return blocks, [source(h[0, 0]) for h in sch.history("s")]


def random_statuses(rng, n):
    # runs of silence and speech, onsets at run starts and a few mid-speech; other labels pass through as the reference's do
    out, speaking = [], False
    while len(out) < n:
        run = rng.randint(1, 9)
        if speaking:
            out += [IPU_CONT if rng.random() < 0.9 else rng.choice([IPU_START, "ipu_end"]) for _ in range(run)]
        else:
            out += [None] * run
            out.append(IPU_START)
        speaking = not speaking
    return out[:n]


@pytest.mark.parametrize("H,O", [(10, 6), (4, 4), (5, 0), (3, 1), (1, 1)])
def test_plan_matches_tick_on_random_statuses(H, O):
    rng = random.Random(100 * H + O)
    for trial in range(40):
        statuses = random_statuses(rng, rng.randint(0, 60))
        plan = plan_gated_replay(statuses, H, O)
        blocks, hist = tick_reference(statuses, H, O)
        assert plan.blocks == blocks, (trial, statuses)
        assert plan.history == hist, (trial, statuses)


def test_plan_edge_cases():
    H, O = 4, 2
    # an onset before any silence replays the still-zero history slots
    p = plan_gated_replay([IPU_START, IPU_CONT], H, O)
    assert p.blocks == [(ReplaySource("history", 2), IPU_START), (ReplaySource("history", 3), IPU_CONT),
                        (ReplaySource("chunk", 0), IPU_CONT), (ReplaySource("chunk", 1), IPU_CONT)]
    assert p.history == [ReplaySource("history", h) for h in range(H)]
    # two onsets with no silence between them replay the same history blocks
    p = plan_gated_replay([None, None, None, IPU_START, IPU_CONT, IPU_START], H, O)
    replayed = [s for s, lab in p.blocks if s.kind == "chunk" and s.index < 3]
    assert replayed == [ReplaySource("chunk", 1), ReplaySource("chunk", 2)] * 2
    assert [lab for _, lab in p.blocks] == [IPU_START, IPU_CONT, IPU_CONT, IPU_CONT, IPU_START, IPU_CONT, IPU_CONT]
    assert p.history == [ReplaySource("history", 3), ReplaySource("chunk", 0), ReplaySource("chunk", 1), ReplaySource("chunk", 2)]
    # all silent: no block, the ring holds the last H chunks; onset_chunks 0: the onset keeps its own label
    p = plan_gated_replay([None] * 7, H, O)
    assert p.blocks == [] and p.history == [ReplaySource("chunk", j) for j in range(3, 7)]
    assert plan_gated_replay([IPU_START], H, 0).blocks == [(ReplaySource("chunk", 0), IPU_START)]
    assert plan_gated_replay([], H, O) == (([], [ReplaySource("history", h) for h in range(H)]))


def test_plan_reproduces_reference_gating_golden():
    """tests/golden/gating.npz: the blocks, order and labels that models/AudioFeatureGating.process_and_gate + the relabelling
    loop of bin/dialog_state_pred.py:626-670 queued for a seeded stream, and its history ring; the plan resolved on the oracle
    frontend's per-chunk features (history zero before the stream) gives them."""
    from conftest import load_golden
    from oracle import freeze_omni_oracle as O
    g = load_golden("gating")
    fr = O.StreamingFrontend()
    feats = torch.cat([fr.process(torch.as_tensor(g["pcm"][i * SPC:(i + 1) * SPC].astype(np.float32) / 32768.0),
                                  float(g["scale"])) for i in range(len(g["statuses"]))]).numpy()
    plan = plan_gated_replay([str(s) if str(s) else None for s in g["statuses"]], 10, 6)

    def value(s):
        return np.zeros((T_IN, F), np.float32) if s.kind == "history" else feats[s.index]

    assert [lab for _, lab in plan.blocks] == [str(x) for x in g["labels"]]
    got = np.stack([value(s) for s, _ in plan.blocks])
    assert np.abs(got - g["blocks"]).max() / max(1.0, np.abs(g["blocks"]).max()) < 1e-5
    hist = np.stack([value(s) for s in plan.history])
    assert np.abs(hist - g["history"]).max() / max(1.0, np.abs(g["history"]).max()) < 1e-5


def _run(sched_kw, recordings, mode, pass_blocks, prime=()):
    """A TagEngine scheduler with sessions opened in key order, primed by ticks of `prime` [(key, status)], then the
    recordings by replay or by a tick loop; returns (blocks per key as (value, label), history per key, block log, scheduler,
    engine)."""
    eng = TagEngine(pass_blocks)
    sch = StreamScheduler(eng, bucket=1, max_sessions=8, **sched_kw)
    for key in sorted(recordings):
        sch.open(key)
    for key, st in prime:
        sch.push(key, np.zeros(SPC, np.int16), st)
        sch.tick()
    sch.block_log = []
    out = {}
    if mode == "replay":
        res = sch.replay({k: (np.zeros((len(s), SPC), np.int16), s) for k, s in recordings.items()})
        for k, bl in res.items():
            out[k] = [(float(b.enc[0, 0]), b.status) for b in bl]
    else:
        for j in range(max(len(s) for s in recordings.values())):
            for k, s in recordings.items():
                if j < len(s):
                    sch.push(k, np.zeros(SPC, np.int16), s[j])
            for k, bl in sch.tick().items():
                out.setdefault(k, []).extend((float(b.enc[0, 0]), b.status) for b in bl)
    log = [(k, float(b[0, 0]), lab) for k, b, lab in sch.block_log]
    hist = {k: sch.history(k)[:, 0, 0].tolist() for k in recordings}
    return out, hist, log, sch, eng


@pytest.mark.parametrize("pass_blocks", [1, 5, 1000])
def test_replay_equals_tick_loop_on_fake_engine(pass_blocks):
    rng = random.Random(pass_blocks)
    recordings = {"a": random_statuses(rng, 47), "b": [None] * 13, "c": [IPU_START] + [IPU_CONT] * 9, "d": [],
                  "e": random_statuses(rng, 30)}
    prime = [("a", None), ("a", None), ("e", IPU_CONT)]
    kw = dict(history_chunks=6, onset_chunks=4)
    want, whist, wlog, _, _ = _run(kw, recordings, "tick", pass_blocks, prime)
    got, ghist, glog, sch, eng = _run(kw, recordings, "replay", pass_blocks, prime)
    assert got == want and ghist == whist
    assert sorted(glog, key=lambda r: r[0]) == sorted(wlog, key=lambda r: r[0])     # per session in stream order
    assert "d" not in got and "b" not in got
    fb = [c for c in eng.calls if c[0] == "fbank"]
    enc = [c for c in eng.calls if c[0] == "encode"]
    assert len(fb) == sch.stats["fbank_calls"] - len(prime) and len(enc) == sch.stats["encode_calls"] - 1   # priming ticks
    for call in fb:                                        # windows bounded like the engine's recording passes
        assert sum(call[2]) <= max(pass_blocks, len(call[1]))
    assert all(sch.keys["d"] not in ids for _, ids, _ in eng.calls)
    for (_, fids, _), (_, eids, _) in zip(fb, enc):
        assert set(eids) <= set(fids)
    # a window in which "b" (all silent) has chunks sends it to the fbank but not to the encoder
    assert any(sch.keys["b"] in ids for _, ids, _ in fb) and all(sch.keys["b"] not in ids for _, ids, _ in enc)


def test_replay_refusals_touch_nothing():
    eng = TagEngine()
    sch = StreamScheduler(eng, history_chunks=4, onset_chunks=2, bucket=1, max_sessions=4)
    sch.open("a")
    sch.open("b")
    sch.push("b", np.zeros(SPC, np.int16), IPU_CONT)
    ok = (np.zeros((3, SPC), np.int16), [None, IPU_START, IPU_CONT])
    with pytest.raises(RuntimeError, match="tick first"):
        sch.replay({"a": ok, "b": ok})
    sch.tick()
    sch.queues["b"].append((torch.zeros(T_IN, F), IPU_CONT))
    with pytest.raises(RuntimeError, match="tick first"):
        sch.replay({"a": ok, "b": ok})
    sch.queues["b"].clear()
    bad = [
        {"zz": ok},                                                        # not open
        {"a": (np.zeros((3, SPC), np.int16), [None, None])},               # statuses do not match the chunks
        {"a": (np.zeros((3, SPC - 1), np.int16), [None] * 3)},             # not whole chunks
        {"a": (np.zeros((3, SPC), np.float64), [None] * 3)},               # dtype
        {"a": (np.zeros((1, SPC), np.int16), [1])},                        # status neither None nor str
        {"a": ok, "b": (np.zeros((3, SPC), np.float32), ok[1])},           # mixed dtypes
    ]
    for rec in bad:
        with pytest.raises((KeyError, ValueError, TypeError)):
            sch.replay(rec)
    assert eng.calls == [] and sch.stats["fbank_calls"] == 1
    assert torch.equal(sch.history("a"), torch.zeros(4, T_IN, F))
