"""Host logic of the scheduler's mixed-count drain (StreamScheduler(max_chunks > 1, mixed_calls=True)), no GPU: the plan,
the padding rule and the blocks a fake engine run hands out."""
import numpy as np

from freeze_omni_b200.scheduler import StreamScheduler, mixed_padding, plan_mixed_calls
from test_scheduler_chunks import ChunkFakeEngine


def test_plan_mixed_calls_one_call_per_round_one_chunk_sessions_first():
    # an onset tick: "a" replays 6 history blocks in front of its current one, everyone else has one block -> ONE call
    assert plan_mixed_calls({"a": 7, "b": 1, "c": 1}, max_chunks=7, max_batch=8) == [[("b", 1), ("c", 1), ("a", 7)]]
    # more queued than max_chunks: the rest drains in the next round
    assert plan_mixed_calls({"a": 9, "b": 1, "c": 2}, max_chunks=7, max_batch=8) == [[("b", 1), ("a", 7), ("c", 2)], [("a", 2)]]
    # max_batch splits a round (sessions, in the reordered sequence)
    assert plan_mixed_calls({"a": 3, "b": 1, "c": 1}, max_chunks=7, max_batch=2) == [[("b", 1), ("c", 1)], [("a", 3)]]
    assert plan_mixed_calls({}, 7, 4) == [] and plan_mixed_calls({"x": 0}, 7, 4) == []
    # a session appears at most once per call and its blocks add up to its queue
    q = {i: (i * 5) % 11 for i in range(9)}
    calls = plan_mixed_calls(q, 4, 3)
    for call in calls:
        assert len({s for s, _ in call}) == len(call) <= 3
        ks = [k for _, k in call]
        assert ks == sorted(ks, key=lambda k: k > 1) and all(1 <= k <= 4 for k in ks)
    assert {s: sum(k for c in calls for t, k in c if t == s) for s in q if q[s]} == {s: n for s, n in q.items() if n}


def test_mixed_padding_adds_fewer_than_a_bucket_of_blocks():
    assert mixed_padding([1, 1, 7], 16) == 7                    # 9 blocks -> 16
    assert mixed_padding([1] * 63 + [7], 16) == 10              # 70 -> 80
    assert mixed_padding([8, 8], 16) == 0 and mixed_padding([3, 2], 1) == 0
    for counts in ([1, 2], [7] * 5, [1] * 17 + [3]):
        pad = mixed_padding(counts, 16)
        assert 0 <= pad < 16 and (sum(counts) + pad) % 16 == 0


class MixedFakeEngine(ChunkFakeEngine):
    def encode_stream_chunks_v(self, ids, chunks, feats, want_adapter=None):
        self.encode_calls.append((list(ids), list(chunks), feats[:, 0, 0].tolist()))
        return feats[:, :4, :8].clone(), feats[:, :2, :4].clone()


def _run(max_chunks, mixed):
    eng = MixedFakeEngine()
    sch = StreamScheduler(eng, history_chunks=4, onset_chunks=2, bucket=4, max_sessions=8, max_chunks=max_chunks,
                          mixed_calls=mixed)
    for key in "abc":
        sch.open(key)
    pcm = np.zeros(2560, np.int16)
    script = [{"a": None, "b": "ipu_cl", "c": None}, {"a": None, "b": "ipu_cl", "c": None},
              {"a": "ipu_sl", "b": "ipu_cl", "c": None}, {"a": "ipu_cl", "b": "ipu_cl", "c": "ipu_sl"},
              {"a": "ipu_cl", "b": None, "c": "ipu_cl"}]
    ticks = []
    for step in script:
        n0 = len(eng.encode_calls)
        for key, status in step.items():
            sch.push(key, pcm, status)
        out = sch.tick()
        ticks.append(({k: [(float(b.enc[0, 0]), b.status) for b in v] for k, v in out.items()}, eng.encode_calls[n0:]))
    return sch, eng, ticks


def test_fake_engine_mixed_run_yields_the_blocks_of_max_chunks_1():
    _, _, ref = _run(1, False)
    sch, eng, got = _run(7, True)
    assert [t[0] for t in got] == [t[0] for t in ref]
    # the onset ticks are one call each, with the one-chunk sessions first and the scratch padding behind them
    ids, chunks, _ = got[2][1][0]
    assert len(got[2][1]) == 1 and chunks[0] == 1 and chunks[-1] == 3 and sum(chunks) % 4 == 0
    assert set(ids[1:-1]) <= set(sch.scratch.tolist()) and all(k == 1 for k in chunks[:-1])
    assert len(got[3][1]) == 1 and sorted(got[3][1][0][1])[-1] == 3
    # no onset: the uniform single-chunk call
    assert got[0][1] == [(got[0][1][0][0], got[0][1][0][1])] and len(got[0][1][0]) == 2
    assert sch.stats["encode_calls"] == 5


def test_mixed_calls_default_off():
    eng = MixedFakeEngine()
    sch = StreamScheduler(eng, max_sessions=8, bucket=4, max_chunks=7)
    assert sch.mixed_calls is False
