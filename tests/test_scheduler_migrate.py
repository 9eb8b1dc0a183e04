"""StreamScheduler.detach / attach without a GPU: a session moved between two schedulers in the middle of the gating golden's
stream gives the blocks, labels and history of the unsplit run, including an onset after the move that replays history
recorded before it.  The engine is a fake whose frontend is the CPU oracle's stateful fbank, one per slot; its snapshot record
carries that frontend."""
import copy

import numpy as np
import pytest
import torch

from freeze_omni_b200.scheduler import SessionSnapshot, StreamScheduler


class FakeCfg:
    chunk_feat_frames, feat_dim, samples_per_chunk = 19, 80, 2560


class MigratingEngine:
    """Slots numbered from `first_slot` (so that the two engines of a move differ); `save_sessions` returns one uint8 row per
    session whose first 8 bytes index a copy of that slot's frontend in a registry shared by all fake engines."""
    saved = {}

    def __init__(self, first_slot=0):
        from oracle import freeze_omni_oracle as O
        self.O, self.front = O, {}
        self.cfg, self.torch_device, self.max_sessions = FakeCfg(), torch.device("cpu"), 64
        self.next_slot = self.first_slot = first_slot

    def stats(self):
        return {"sessions_in_use": self.next_slot - self.first_slot}

    def alloc(self, n):
        ids = np.arange(self.next_slot, self.next_slot + n, dtype=np.int32)
        self.next_slot += n
        return ids

    def free(self, ids):
        for s in ids:
            self.front.pop(int(s), None)

    def fbank_stream(self, ids, pcm, scale=None):
        out = []
        for i, s in enumerate(ids):
            fr = self.front.setdefault(int(s), self.O.StreamingFrontend())
            out.append(fr.process(torch.as_tensor(pcm[i]).float(), 1.0 if scale is None else scale))
        return torch.cat(out, 0)

    def encode_stream(self, ids, feats):
        return feats[:, :4, :8].clone(), feats[:, :2, :4].clone()

    def save_sessions(self, ids):
        rows = []
        for s in ids:
            key = len(MigratingEngine.saved)
            MigratingEngine.saved[key] = copy.deepcopy(self.front.get(int(s), self.O.StreamingFrontend()))
            rows.append(torch.tensor(np.array([key], np.int64).view(np.uint8)))
        return torch.stack(rows)

    def restore_sessions(self, ids, blob):
        for s, row in zip(ids, blob):
            self.front[int(s)] = copy.deepcopy(MigratingEngine.saved[int(row.numpy().view(np.int64)[0])])


def _run(g, move_at=None):
    """The golden's stream through one scheduler, or moved to a second one after `move_at` ticks.  Returns the queued blocks
    with their labels, the blocks each tick returned, and the final history ring."""
    a = StreamScheduler(MigratingEngine(0), history_chunks=10, onset_chunks=6, bucket=1, max_sessions=4)
    b = StreamScheduler(MigratingEngine(20), history_chunks=10, onset_chunks=6, bucket=1, max_sessions=4)
    a.open("other")                               # the moved session lands in a different slot and history row
    a.open("u")
    sch, log, outs = a, [], []
    a.block_log = b.block_log = log
    for i, st in enumerate(g["statuses"]):
        if i == move_at:
            b.open("x")
            b.open("y")
            b.attach("u", a.detach("u").to("cpu"))
            assert (b.keys["u"], b.rows["u"]) == (22, 2) and "u" not in a.keys
            sch = b
        pcm = g["pcm"][i * 2560:(i + 1) * 2560].astype(np.float32) / 32768.0
        sch.push("u", pcm, str(st) if str(st) else None)
        outs.append([(blk.enc, blk.emb, blk.status) for blk in sch.tick(float(g["scale"])).get("u", [])])
    return log, outs, sch.history("u").clone()


def test_detach_attach_mid_stream_matches_the_unsplit_run():
    from conftest import load_golden
    g = load_golden("gating")
    statuses = [str(s) for s in g["statuses"]]
    log0, outs0, hist0 = _run(g)
    # the unsplit run is the reference's (test_scheduler_logic pins it to the golden)
    assert [lab for _, _, lab in log0] == [str(x) for x in g["labels"]]
    move_at = 10
    # the first onset after the move replays history rows recorded before it
    onset = statuses.index("ipu_sl", move_at)
    assert onset - 6 < move_at and all(s == "" for s in statuses[onset - 6:move_at])
    log1, outs1, hist1 = _run(g, move_at)
    assert len(log1) == len(log0)
    for (k0, b0, l0), (k1, b1, l1) in zip(log0, log1):
        assert k0 == k1 and l0 == l1 and torch.equal(b0, b1)
    assert len(outs1) == len(outs0)
    for t0, t1 in zip(outs0, outs1):
        assert len(t0) == len(t1)
        for (e0, y0, s0), (e1, y1, s1) in zip(t0, t1):
            assert s0 == s1 and torch.equal(e0, e1) and torch.equal(y0, y1)
    assert torch.equal(hist0, hist1)


def test_detach_refuses_an_unticked_chunk_and_attach_checks_the_history_shape():
    a = StreamScheduler(MigratingEngine(0), history_chunks=10, onset_chunks=6, bucket=1, max_sessions=4)
    a.open("u")
    a.push("u", np.zeros(2560, np.float32), None)
    with pytest.raises(RuntimeError, match="not ticked"):
        a.detach("u")
    a.tick()
    snap = a.detach("u")
    assert isinstance(snap, SessionSnapshot) and "u" not in a.keys
    short = StreamScheduler(MigratingEngine(0), history_chunks=4, onset_chunks=2, bucket=1, max_sessions=4)
    with pytest.raises(ValueError, match="history"):
        short.attach("u", snap)
    assert "u" not in short.keys
