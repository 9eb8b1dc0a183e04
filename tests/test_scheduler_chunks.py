"""Host logic of the scheduler's multi-chunk drain (StreamScheduler(max_chunks > 1)), no GPU: the grouping function and the
call sequence a fake engine records."""
import numpy as np
import torch

from freeze_omni_b200.scheduler import StreamScheduler, chunk_bucket_size, plan_chunk_calls, plan_rounds
from test_scheduler_logic import FakeEngine


def test_plan_chunk_calls_groups_sessions_by_chunk_count():
    # an onset tick: "a" replays 6 history blocks in front of its current one, everyone else has one block
    assert plan_chunk_calls({"a": 7, "b": 1, "c": 1}, max_chunks=7, max_batch=8) == [(1, ["b", "c"]), (7, ["a"])]
    # fewer chunks per call than queued: the rest drains in later rounds, in order
    assert plan_chunk_calls({"a": 7, "b": 1}, max_chunks=4, max_batch=8) == [(1, ["b"]), (4, ["a"]), (3, ["a"])]
    assert plan_chunk_calls({"a": 3, "b": 3, "c": 0}, max_chunks=7, max_batch=1) == [(3, ["a"]), (3, ["b"])]
    assert plan_chunk_calls({}, 7, 4) == [] and plan_chunk_calls({"x": 0}, 7, 4) == []
    # max_chunks = 1 is plan_rounds
    q = {"a": 1, "b": 7, "c": 0, "d": 2}
    assert plan_chunk_calls(q, 1, 2) == [(1, r) for r in plan_rounds(q, 2)]


def test_chunk_bucket_size_pads_by_blocks():
    assert [chunk_bucket_size(n, 1, 16) for n in (1, 16, 17)] == [16, 16, 32]          # single-chunk calls: as before
    assert [chunk_bucket_size(n, 7, 16) for n in (1, 2, 3)] == [2, 2, 4]               # granule 2 sessions = 14 blocks
    assert chunk_bucket_size(2, 16, 16) == 2 and chunk_bucket_size(5, 3, 4) == 5


class ChunkFakeEngine(FakeEngine):
    def encode_stream_chunks(self, ids, feats, want_adapter=None):
        self.encode_calls.append((list(ids), feats[:, :, 0, 0].tolist()))
        return feats[:, :, :4, :8].clone(), feats[:, :, :2, :4].clone()


def test_fake_engine_run_with_max_chunks():
    eng = ChunkFakeEngine()
    sch = StreamScheduler(eng, history_chunks=4, onset_chunks=2, bucket=4, max_sessions=8, max_chunks=7)
    a, b = sch.open("a"), sch.open("b")
    pcm = np.zeros(2560, np.int16)
    for _ in range(3):
        sch.push("a", pcm, None)
        sch.push("b", pcm, "ipu_cl")
        out = sch.tick()
        assert list(out) == ["b"] and len(out["b"]) == 1
    n_calls = len(eng.encode_calls)
    sch.push("a", pcm, "ipu_sl")
    sch.push("b", pcm, "ipu_cl")
    out = sch.tick()
    # onset tick: one single-chunk call (b, padded to the bucket) and one 3-chunk call (a, padded by blocks: 4 // 3 = 1 session)
    calls = eng.encode_calls[n_calls:]
    assert len(calls) == 2
    assert calls[0][0][0] == b and len(calls[0][0]) == 4 and set(calls[0][0][1:]) <= set(sch.scratch.tolist())
    assert calls[1][0] == [a] and calls[1][1] == [[100.0 * a + 2, 100.0 * a + 3, 100.0 * a + 4]]
    assert [float(e.enc[0, 0]) for e in out["a"]] == [100.0 * a + 2, 100.0 * a + 3, 100.0 * a + 4]
    assert [e.status for e in out["a"]] == ["ipu_sl", "ipu_cl", "ipu_cl"]
    assert len(out["b"]) == 1 and out["b"][0].status == "ipu_cl" and tuple(out["b"][0].enc.shape) == (4, 8)
    assert sch.stats["encode_calls"] == 3 + 2 and sch.stats["session_steps"] == 3 + 4
    assert sch.history("a")[-1, 0, 0].item() == 100.0 * a + 3


def test_default_max_chunks_keeps_the_single_chunk_calls():
    eng = FakeEngine()                                    # no encode_stream_chunks: the default never asks for it
    sch = StreamScheduler(eng, history_chunks=4, onset_chunks=2, bucket=4, max_sessions=8)
    assert sch.max_chunks == 1
    sch.open("a")
    for st in (None, None, "ipu_sl"):
        sch.push("a", np.zeros(2560, np.int16), st)
        sch.tick()
    assert len(eng.encode_calls) == 3 and all(torch.tensor(f).numel() == 4 for _, f in eng.encode_calls)
