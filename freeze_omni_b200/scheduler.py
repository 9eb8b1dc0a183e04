"""Batched session scheduler with the VAD-gated streaming frontend (SURVEY 8 f1 + f3).

The reference runs one feature-gating thread and one predictor thread PER SESSION, hands fbank blocks between them
as Python lists and calls the encoder with batch 1 (bin/dialog_state_pred.py:600-684 feature gating, :719-775 the
processing loop, :793-814 the encoder call; bin/pool.py:61-91 the pipeline pool).  Here one scheduler per GPU gathers
the chunks that arrived during a tick (<= 160 ms), runs ONE batched fbank call for all of them, applies the gating rule
on the device and drains the per-session feature queues with batched encoder+adapter steps:

  gating rule (models/AudioFeatureGating.py:77-109, process_and_gate):
    * features are ALWAYS extracted, so the sample carry / context ring stay continuous;
    * status None (no speech):       the block only enters the session's history ring (last `history_chunks` blocks);
    * status 'ipu_sl' (speech onset): the last `onset_chunks` history blocks are queued in front of the current one
      (dialog_state_pred.py:639-670), each of them is one encoder step;
    * any other status:              the block is queued.
  Each queued block is one `encoder.infer` + adapter step of that session (dialog_state_pred.py:793-814).

Per drain round the head block of every session with a non-empty queue forms one batch; the batch is padded to a
multiple of `bucket` with scratch sessions so that a handful of captured CUDA graphs serve every active-set size.
With `max_chunks` > 1 a round takes up to that many queued blocks of a session at once (Engine.encode_stream_chunks, same
results as one block per call): an onset tick then costs one call for the sessions with one block and one for those
replaying their history, instead of 1 + onset_chunks calls.  With `mixed_calls` as well, a round is ONE call in which every
session brings its own number of blocks (Engine.encode_stream_chunks_v), so an onset tick costs one encoder step.
State (KV rings, adapter cache, sample carry, feature ring, history ring, queued blocks) never leaves the device, unless a
session is moved: `detach` / `attach` carry it, history rows included, to another scheduler on any GPU.
A recorded, VAD-annotated conversation goes through `replay` in one call: `plan_gated_replay` applies the same rule on the host,
and windows of recorded chunks run as one fbank call (Engine.fbank_stream_v) and one encoder call (Engine.encode_stream_steps_v)
each, with the blocks and history rows gathered on the device; the sessions end as one tick per chunk would leave them.  With a
Handoff, the encoder call of each window writes the blocks' LLM inputs (fp16 rows, mask rows, start rows) as a tick's does.
"""
from collections import deque
from typing import Any, Deque, Dict, Hashable, List, NamedTuple, Optional, Tuple

import numpy as np
import torch

IPU_START = "ipu_sl"
IPU_CONT = "ipu_cl"


class Block(NamedTuple):
    """One encoder + adapter step of one session, as `tick` hands it to the LLM stage.  `status` is the label the reference's
    feature-gating thread gives the block (bin/dialog_state_pred.py:639-670): the FIRST block of a speech onset carries
    'ipu_sl' -- which is where AudioLLM.recognize puts the chat prefix (models/audioLLM.py:404-406) -- every other one 'ipu_cl'."""
    enc: torch.Tensor                 # (t, D) encoder frames
    emb: Optional[torch.Tensor]       # (t_out, E) adapter embeddings; with a Handoff: the fp16 LLM input rows, chat prefix included
    status: str                       # when status == 'ipu_sl' (views of the Handoff buffers)
    mask: Optional[torch.Tensor] = None   # with a Handoff: the attention-mask entries of those rows


class Handoff:
    """Pre-allocated LLM-side buffers for `StreamScheduler.tick(handoff=...)` and `StreamScheduler.replay(..., handoff=...)`
    (models/audioLLM.py:383-411): `embeds` (capacity, prefix_len + t_out, E) fp16 whose first prefix_len rows of every block hold
    the chat-prefix embeddings, `attn_mask` (capacity, prefix_len + t_out) uint8 and `row_start` (capacity) int32.  One block per
    encoder step of a tick or a replay."""

    def __init__(self, engine, capacity: int, prefix_embeds: torch.Tensor, prefix_mask: Optional[torch.Tensor] = None):
        dev = engine.torch_device
        self.prefix_len = int(prefix_embeds.shape[-2])
        _, t_out = engine.out_frames(engine.cfg.chunk_feat_frames)
        self.rows = self.prefix_len + t_out
        self.embeds = torch.zeros(capacity, self.rows, engine.cfg.llm_dim, dtype=torch.float16, device=dev)
        self.embeds[:, :self.prefix_len] = prefix_embeds.reshape(self.prefix_len, -1).to(dev, torch.float16)
        self.prefix_mask = None if prefix_mask is None else prefix_mask.reshape(-1).to(dev, torch.uint8).contiguous()
        self.attn_mask = torch.zeros(capacity, self.rows, dtype=torch.uint8, device=dev)
        self.row_start = torch.zeros(capacity, dtype=torch.int32, device=dev)


class SessionSnapshot(NamedTuple):
    """A session taken out of a scheduler (`StreamScheduler.detach`): the engine's snapshot record and the session's rows of
    the history ring, which a speech onset after the move replays.  `to(device)` moves both, e.g. to another GPU's scheduler."""
    record: torch.Tensor              # (snapshot_bytes,) uint8, Engine.save_sessions
    history: torch.Tensor             # (history_chunks, t_in, F) fp32

    def to(self, device) -> "SessionSnapshot":
        return SessionSnapshot(self.record.to(device), self.history.to(device))


def onset_statuses(n_history: int, status: str) -> List[str]:
    """Labels of the blocks one pushed chunk turns into (bin/dialog_state_pred.py:639-670): the replayed history blocks are
    'ipu_sl', 'ipu_cl', 'ipu_cl', ... and the current block is 'ipu_cl' when history was replayed, else keeps its status."""
    if status != IPU_START or n_history == 0:
        return [status]
    return [IPU_START] + [IPU_CONT] * n_history


class ReplaySource(NamedTuple):
    """Where a block of a gated replay comes from: recorded chunk `index` of the replayed statuses (kind 'chunk'), or slot
    `index` of the session's history ring as it stood before them (kind 'history', oldest slot 0)."""
    kind: str
    index: int


class GatedPlan(NamedTuple):
    blocks: List[Tuple[ReplaySource, str]]    # the encoder blocks in stream order, with their labels
    history: List[ReplaySource]               # the history ring afterwards, oldest first


def plan_gated_replay(statuses, history_chunks: int, onset_chunks: int) -> GatedPlan:
    """What `tick`'s gating rule makes of a session's chunks pushed one per tick with these statuses: a silent chunk (None) only
    enters the history ring, an 'ipu_sl' onset queues the last `onset_chunks` history slots in front of its own chunk (slots
    still zero when no silence came before, and the same slots again for a second onset with no silence in between), any other
    status queues its chunk.  Pure function of the statuses -> testable without a GPU."""
    assert 0 <= onset_chunks <= history_chunks
    ring = [ReplaySource("history", h) for h in range(history_chunks)]
    blocks: List[Tuple[ReplaySource, str]] = []
    for j, status in enumerate(statuses):
        cur = ReplaySource("chunk", j)
        if status is None:
            ring = (ring + [cur])[1:]
            continue
        replayed = ring[history_chunks - onset_chunks:] if status == IPU_START and onset_chunks > 0 else []
        blocks.extend(zip(replayed + [cur], onset_statuses(len(replayed), status)))
    return GatedPlan(blocks, ring)


def gated_block_count(statuses, onset_chunks: int) -> int:
    """len(plan_gated_replay(statuses, history_chunks, onset_chunks).blocks) without building the plan: every non-silent chunk is
    one block, and an 'ipu_sl' chunk brings `onset_chunks` history slots in front of it (the ring always holds history_chunks)."""
    statuses = list(statuses)
    return sum(st is not None for st in statuses) + onset_chunks * statuses.count(IPU_START)


def plan_rounds(queue_lens: Dict[Hashable, int], max_batch: int) -> List[List[Hashable]]:
    """Drain order for per-session FIFO queues: every round takes the head block of each session that still has one
    (a session's blocks must run in order, so it appears at most once per round), `max_batch` sessions per batch.
    Pure function of the queue lengths -> testable without a GPU."""
    left = dict(queue_lens)
    rounds: List[List[Hashable]] = []
    while True:
        ready = [k for k, n in left.items() if n > 0]
        if not ready:
            return rounds
        for i in range(0, len(ready), max_batch):
            rounds.append(ready[i:i + max_batch])
        for k in ready:
            left[k] -= 1


def plan_chunk_calls(queue_lens: Dict[Hashable, int], max_chunks: int, max_batch: int) -> List[Tuple[int, List[Hashable]]]:
    """Drain order when one call may advance a session by up to `max_chunks` consecutive queued blocks: every round takes
    k = min(blocks left, max_chunks) blocks of each session that still has some; sessions with the same k share a call
    (smaller k first, sessions in queue order, `max_batch` sessions per call).  A session appears at most once per round and
    rounds run in order, so its blocks stay in stream order.  Returns [(k, sessions)]; max_chunks = 1 is plan_rounds.
    Pure function of the queue lengths -> testable without a GPU."""
    assert max_chunks >= 1
    left = dict(queue_lens)
    calls: List[Tuple[int, List[Hashable]]] = []
    while True:
        ready = [key for key, n in left.items() if n > 0]
        if not ready:
            return calls
        by_k: Dict[int, List[Hashable]] = {}
        for key in ready:
            by_k.setdefault(min(left[key], max_chunks), []).append(key)
        for k in sorted(by_k):
            group = by_k[k]
            for i in range(0, len(group), max_batch):
                calls.append((k, group[i:i + max_batch]))
        for key in ready:
            left[key] -= min(left[key], max_chunks)


def plan_mixed_calls(queue_lens: Dict[Hashable, int], max_chunks: int, max_batch: int) -> List[List[Tuple[Hashable, int]]]:
    """Drain order when one call may advance each of its sessions by its own number of queued blocks (up to `max_chunks`):
    every round takes k = min(blocks left, max_chunks) blocks of each session that still has some, all in one call (split
    only by `max_batch` sessions).  Within a call the sessions with k = 1 come first, in queue order, so that they form the
    leading one-chunk run the encoder attends with its single-chunk kernel; the others follow in queue order.  Returns the
    calls as [(session, k)].  Pure function of the queue lengths -> testable without a GPU."""
    assert max_chunks >= 1
    left = dict(queue_lens)
    calls: List[List[Tuple[Hashable, int]]] = []
    while True:
        ready = [(key, min(n, max_chunks)) for key, n in left.items() if n > 0]
        if not ready:
            return calls
        ordered = [r for r in ready if r[1] == 1] + [r for r in ready if r[1] > 1]
        for i in range(0, len(ordered), max_batch):
            calls.append(ordered[i:i + max_batch])
        for key, k in ready:
            left[key] -= k


def mixed_padding(counts: List[int], bucket: int) -> int:
    """Scratch sessions, one block each, that pad a call with these per-session block counts to a multiple of `bucket`
    blocks (fewer than `bucket` of them).  They join the leading one-chunk run."""
    blocks = sum(counts)
    return bucket_size(blocks, bucket) - blocks


def bucket_size(n: int, bucket: int) -> int:
    return (n + bucket - 1) // bucket * bucket


def chunk_bucket_size(n: int, k: int, bucket: int) -> int:
    """Sessions of a call of n sessions x k chunks after padding.  The padding is counted in blocks (token rows), not in
    sessions: sessions are padded to a multiple of max(1, bucket // k), so it adds fewer than `bucket` blocks, as the padding
    of a single-chunk call does (2 onset sessions x 7 chunks stay 2 sessions with bucket 16, not 16 x 7 blocks)."""
    return bucket_size(n, max(1, bucket // k))


class StreamScheduler:
    def __init__(self, engine, history_chunks: int = 10, onset_chunks: int = 6, bucket: int = 16,
                 max_batch: Optional[int] = None, max_sessions: Optional[int] = None, max_chunks: int = 1,
                 mixed_calls: bool = False):
        assert 0 <= onset_chunks <= history_chunks and max_chunks >= 1
        self.max_chunks = int(max_chunks)
        self.mixed_calls = bool(mixed_calls)
        self.eng, self.cfg = engine, engine.cfg
        self.history_chunks, self.onset_chunks, self.bucket = history_chunks, onset_chunks, max(1, bucket)
        self.max_batch = max_batch or 1 << 30
        self.keys: Dict[Hashable, int] = {}                    # session key -> slot
        self.rows: Dict[Hashable, int] = {}                    # session key -> row of the history tensor
        self.free_rows: List[int] = []
        self.pending: Dict[Hashable, Tuple[Any, Optional[str]]] = {}
        self.queues: Dict[Hashable, Deque[Tuple[torch.Tensor, str]]] = {}
        # the scratch sessions that pad a batch to its bucket come out of the engine's slot pool: the scheduler can only
        # promise what is left of it
        free = engine.max_sessions - engine.stats()["sessions_in_use"] - (self.bucket - 1)
        if free < 1:
            raise ValueError("engine has %d session slots, %d in use: no room for bucket=%d (needs bucket-1 scratch sessions + 1)"
                             % (engine.max_sessions, engine.stats()["sessions_in_use"], self.bucket))
        cap = free if max_sessions is None else int(max_sessions)
        if cap > free:
            raise ValueError("max_sessions=%d exceeds the engine's free slots (%d of %d) minus %d scratch sessions"
                             % (cap, free + self.bucket - 1, engine.max_sessions, self.bucket - 1))
        self.scratch = engine.alloc(self.bucket - 1) if self.bucket > 1 else np.zeros(0, np.int32)
        self._hist = torch.zeros(cap, history_chunks, self.cfg.chunk_feat_frames, self.cfg.feat_dim, device=engine.torch_device)
        self.free_rows = list(range(cap - 1, -1, -1))
        self.stats = {"ticks": 0, "fbank_calls": 0, "encode_calls": 0, "session_steps": 0, "padded_steps": 0}
        # tests: when a list, every block the gating rule queues is appended as (key, feature block, status)
        self.block_log: Optional[List[Tuple[Hashable, torch.Tensor, str]]] = None

    # ---- sessions ---------------------------------------------------------------------------------
    def open(self, key: Hashable) -> int:
        """New session == encoder_cache None, adapter_cache None, pe_index 0 (dialog_state_pred.py:221-232) and a
        zeroed frontend (AudioFeatureGating.reset)."""
        assert key not in self.keys, "session already open"
        if not self.free_rows:
            raise RuntimeError("scheduler is full (max_sessions=%d)" % self._hist.shape[0])
        slot = int(self.eng.alloc(1)[0])
        self.keys[key], self.rows[key] = slot, self.free_rows.pop()
        self._hist[self.rows[key]].zero_()
        self.queues[key] = deque()
        return slot

    def close(self, key: Hashable) -> None:
        self.eng.free([self.keys.pop(key)])
        self.free_rows.append(self.rows.pop(key))
        self.queues.pop(key)
        self.pending.pop(key, None)

    def reset(self, key: Hashable) -> None:
        self.eng.reset([self.keys[key]])
        self._hist[self.rows[key]].zero_()
        self.queues[key].clear()
        self.pending.pop(key, None)

    def detach(self, key: Hashable) -> SessionSnapshot:
        """Take a session out of this scheduler between ticks (to rebalance GPUs, drain one, or restart a server): its whole
        state as a SessionSnapshot, then the session is closed here.  `attach` continues it in any scheduler of the same model,
        on any GPU, exactly as if it had stayed.  A chunk pushed since the last tick must be ticked first."""
        if key in self.pending:
            raise RuntimeError("session %r has a pushed chunk that was not ticked yet: tick before detaching it" % (key,))
        snap = SessionSnapshot(self.eng.save_sessions([self.keys[key]])[0], self._hist[self.rows[key]].clone())
        self.close(key)
        return snap

    def attach(self, key: Hashable, snap: SessionSnapshot) -> int:
        """Open `key` with the state of a detached session; returns its slot in this scheduler's engine."""
        if tuple(snap.history.shape) != tuple(self._hist.shape[1:]):
            raise ValueError("history rows %s do not fit this scheduler's %s (history_chunks differ)"
                             % (tuple(snap.history.shape), tuple(self._hist.shape[1:])))
        slot = self.open(key)
        try:
            self.eng.restore_sessions([slot], snap.record.to(self.eng.torch_device).view(1, -1))
        except Exception:
            self.close(key)
            raise
        self._hist[self.rows[key]].copy_(snap.history)
        return slot

    # ---- data path ----------------------------------------------------------------------------------
    def push(self, key: Hashable, pcm, status: Optional[str]) -> None:
        """One chunk of `samples_per_chunk` samples (int16 or float32, host or device) with its VAD annotation."""
        assert key in self.keys and key not in self.pending, "one chunk per session per tick"
        self.pending[key] = (pcm, status)

    def tick(self, scale: Optional[float] = None, handoff: Optional[Handoff] = None) -> Dict[Hashable, List[Block]]:
        """Process everything pushed since the last tick.  Returns, per session that produced output, the list of
        Block(encoder frames (t, D), adapter embeddings (t_out, E), status) in stream order (one entry per queued block).
        `scale` None = the engine's rule: 1.0 for int16 PCM, cfg.pcm_scale for float audio in [-1, 1]."""
        self.stats["ticks"] += 1
        out: Dict[Hashable, List[Block]] = {}
        if self.pending:
            keys = list(self.pending)
            dev = self.eng.torch_device
            pcm = torch.stack([torch.as_tensor(self.pending[k][0]).to(dev, non_blocking=True) for k in keys])
            ids = np.array([self.keys[k] for k in keys], np.int32)
            feats = self.eng.fbank_stream(ids, pcm, scale)                       # carry + context ring advance for everyone
            self.stats["fbank_calls"] += 1
            silent = [i for i, k in enumerate(keys) if self.pending[k][1] is None]
            if silent:                                                           # history ring: drop the oldest, append
                rows = torch.tensor([self.rows[keys[i]] for i in silent], device=dev)
                h = self._hist.index_select(0, rows)
                h = torch.cat([h[:, 1:], feats.index_select(0, torch.tensor(silent, device=dev)).unsqueeze(1)], dim=1)
                self._hist.index_copy_(0, rows, h)
            for i, k in enumerate(keys):
                status = self.pending[k][1]
                if status is None:
                    continue
                blocks = [feats[i]]
                if status == IPU_START and self.onset_chunks > 0:
                    hist = self._hist[self.rows[k], self.history_chunks - self.onset_chunks:].clone()
                    blocks = list(hist.unbind(0)) + blocks
                labelled = list(zip(blocks, onset_statuses(len(blocks) - 1, status)))
                self.queues[k].extend(labelled)
                if self.block_log is not None:
                    self.block_log.extend((k, b, lab) for b, lab in labelled)
            self.pending.clear()
        cursor = 0
        if self.mixed_calls:
            return self._drain_mixed(out, handoff)
        if self.max_chunks > 1:
            return self._drain_chunks(out, handoff)
        for batch in plan_rounds({k: len(q) for k, q in self.queues.items()}, self.max_batch):
            heads = [self.queues[k].popleft() for k in batch]
            blocks = [h[0] for h in heads]
            n = len(batch)
            pad = bucket_size(n, self.bucket) - n
            ids = np.concatenate([np.array([self.keys[k] for k in batch], np.int32), self.scratch[:pad]]).astype(np.int32)
            x = torch.stack(blocks + [blocks[0]] * pad)
            if handoff is not None:
                # fused hand-off: rows of this batch land in the next free blocks of the caller's buffers (audioLLM.py:404-411)
                n_all = n + pad
                if cursor + n_all > handoff.embeds.shape[0]:
                    raise RuntimeError("Handoff capacity %d exceeded in one tick" % handoff.embeds.shape[0])
                onset = [h[1] == IPU_START for h in heads] + [False] * pad
                self.eng.handoff_arm(n_all, handoff.embeds[cursor:], handoff.prefix_len, onset, handoff.prefix_mask,
                                     handoff.attn_mask[cursor:], handoff.row_start[cursor:])
                enc, _ = self.eng.encode_stream(ids, x, want_adapter=False)
                self.stats["encode_calls"] += 1
                self.stats["session_steps"] += n
                self.stats["padded_steps"] += pad
                for i, k in enumerate(batch):
                    st0 = 0 if heads[i][1] == IPU_START else handoff.prefix_len
                    out.setdefault(k, []).append(Block(enc[i], handoff.embeds[cursor + i, st0:], heads[i][1],
                                                       handoff.attn_mask[cursor + i, st0:]))
                cursor += n_all
                continue
            enc, emb = self.eng.encode_stream(ids, x)
            self.stats["encode_calls"] += 1
            self.stats["session_steps"] += n
            self.stats["padded_steps"] += pad
            for i, k in enumerate(batch):
                out.setdefault(k, []).append(Block(enc[i], emb[i] if emb is not None else None, heads[i][1]))
        return out

    def _drain_chunks(self, out: Dict[Hashable, List[Block]], handoff: Optional[Handoff]) -> Dict[Hashable, List[Block]]:
        """The drain of tick() with up to max_chunks blocks of a session per call (plan_chunk_calls)."""
        cursor = 0
        for k, batch in plan_chunk_calls({s: len(q) for s, q in self.queues.items()}, self.max_chunks, self.max_batch):
            cursor = self._chunk_call(k, batch, out, handoff, cursor)
        return out

    def _drain_mixed(self, out: Dict[Hashable, List[Block]], handoff: Optional[Handoff]) -> Dict[Hashable, List[Block]]:
        """The drain of tick() with one call per round, each session bringing up to max_chunks blocks (plan_mixed_calls).
        A round whose sessions all bring the same number of blocks keeps the uniform call."""
        cursor = 0
        for call in plan_mixed_calls({s: len(q) for s, q in self.queues.items()}, self.max_chunks, self.max_batch):
            counts = [k for _, k in call]
            batch = [s for s, _ in call]
            if len(set(counts)) == 1:
                cursor = self._chunk_call(counts[0], batch, out, handoff, cursor)
                continue
            heads = [[self.queues[s].popleft() for _ in range(k)] for s, k in call]
            n1 = counts.index(next(k for k in counts if k > 1))           # the leading one-chunk run
            pad = mixed_padding(counts, self.bucket)
            order = list(range(n1)) + [-1] * pad + list(range(n1, len(call)))   # -1: a scratch session
            ids = np.concatenate([np.array([self.keys[s] for s in batch[:n1]], np.int32), self.scratch[:pad],
                                  np.array([self.keys[s] for s in batch[n1:]], np.int32)]).astype(np.int32)
            chunks = np.array([counts[i] if i >= 0 else 1 for i in order], np.int32)
            x = torch.stack([h[0] for i in order for h in (heads[i] if i >= 0 else heads[0][:1])])      # (sum(chunks), t_in, F)
            first = np.concatenate([[0], np.cumsum(chunks)[:-1]])        # block of each session's first chunk
            self.stats["encode_calls"] += 1
            self.stats["session_steps"] += sum(counts)
            self.stats["padded_steps"] += pad
            if handoff is not None:
                n_blocks = int(chunks.sum())
                if cursor + n_blocks > handoff.embeds.shape[0]:
                    raise RuntimeError("Handoff capacity %d exceeded in one tick" % handoff.embeds.shape[0])
                onset = [h[1] == IPU_START for i in order for h in (heads[i] if i >= 0 else [(None, None)])]
                self.eng.handoff_arm(n_blocks, handoff.embeds[cursor:], handoff.prefix_len, onset, handoff.prefix_mask,
                                     handoff.attn_mask[cursor:], handoff.row_start[cursor:])
                enc, _ = self.eng.encode_stream_chunks_v(ids, chunks, x, want_adapter=False)
            else:
                enc, emb = self.eng.encode_stream_chunks_v(ids, chunks, x)
            for p, i in enumerate(order):
                if i < 0:
                    continue
                for j, h in enumerate(heads[i]):
                    b = int(first[p]) + j
                    if handoff is not None:
                        st0 = 0 if h[1] == IPU_START else handoff.prefix_len
                        out.setdefault(batch[i], []).append(Block(enc[b], handoff.embeds[cursor + b, st0:], h[1],
                                                                  handoff.attn_mask[cursor + b, st0:]))
                    else:
                        out.setdefault(batch[i], []).append(Block(enc[b], emb[b] if emb is not None else None, h[1]))
            if handoff is not None:
                cursor += int(chunks.sum())
        return out

    def _chunk_call(self, k: int, batch: List[Hashable], out: Dict[Hashable, List[Block]], handoff: Optional[Handoff],
                    cursor: int) -> int:
        """One call advancing every session of `batch` by k queued blocks; returns the next free hand-off block."""
        heads = [[self.queues[s].popleft() for _ in range(k)] for s in batch]
        n = len(batch)
        pad = chunk_bucket_size(n, k, self.bucket) - n
        ids = np.concatenate([np.array([self.keys[s] for s in batch], np.int32), self.scratch[:pad]]).astype(np.int32)
        x = torch.stack([h[0] for hs in heads + [heads[0]] * pad for h in hs])
        x = x.view(n + pad, k, *x.shape[1:])                                                  # (n + pad, k, t_in, F)
        self.stats["encode_calls"] += 1
        self.stats["session_steps"] += n * k
        self.stats["padded_steps"] += pad * k
        if handoff is not None:
            # block i*k + j of the armed call is chunk j of session i
            n_blocks = (n + pad) * k
            if cursor + n_blocks > handoff.embeds.shape[0]:
                raise RuntimeError("Handoff capacity %d exceeded in one tick" % handoff.embeds.shape[0])
            onset = [h[1] == IPU_START for hs in heads for h in hs] + [False] * (pad * k)
            self.eng.handoff_arm(n_blocks, handoff.embeds[cursor:], handoff.prefix_len, onset, handoff.prefix_mask,
                                 handoff.attn_mask[cursor:], handoff.row_start[cursor:])
            enc, _ = self._encode(ids, x, k, want_adapter=False)
            for i, s in enumerate(batch):
                for j, h in enumerate(heads[i]):
                    row = cursor + i * k + j
                    st0 = 0 if h[1] == IPU_START else handoff.prefix_len
                    out.setdefault(s, []).append(Block(enc[i, j], handoff.embeds[row, st0:], h[1], handoff.attn_mask[row, st0:]))
            return cursor + n_blocks
        enc, emb = self._encode(ids, x, k)
        for i, s in enumerate(batch):
            for j, h in enumerate(heads[i]):
                out.setdefault(s, []).append(Block(enc[i, j], emb[i, j] if emb is not None else None, h[1]))
        return cursor

    def _encode(self, ids, x, k, **kw):
        """(n, k, ...) results of one call: a single-chunk call keeps the engine's one-chunk entry point."""
        if k == 1:
            enc, emb = self.eng.encode_stream(ids, x[:, 0], **kw)
            return enc.unsqueeze(1), (emb.unsqueeze(1) if emb is not None else None)
        return self.eng.encode_stream_chunks(ids, x, **kw)

    def replay(self, recordings: Dict[Hashable, Tuple[Any, Any]], scale: Optional[float] = None,
               handoff: Optional[Handoff] = None) -> Dict[Hashable, List[Block]]:
        """Recorded, VAD-annotated audio of open sessions in one call, with the blocks, labels and session state that pushing
        it one chunk per tick would give (plan_gated_replay).  `recordings` maps a key to (pcm (c, samples_per_chunk) int16 or
        float32, host or device, statuses (c,) of None or str); every recording has the same PCM dtype.  Returns, per session
        that produced output, its Blocks in stream order, and logs them in `block_log` as tick does.  The recordings run in
        windows of at most max(P, sessions) chunks, P the engine's "steps_pass_blocks_in_use": per window one fbank_stream_v
        over every session, the encoder blocks and the new history rows gathered on the device from the window's features and
        the history rows, and one encode_stream_steps_v over the sessions with a block in the window.  A session with a
        pushed chunk or queued blocks is refused before anything runs: tick first.
        With a Handoff (bf16 engines), every block's LLM input is written as tick(handoff=) writes it: Block.emb and Block.mask
        are views of `handoff.embeds` / `handoff.attn_mask` (chat prefix included for 'ipu_sl' blocks), the fp16 rows being
        .half() of the adapter rows the replay returns without one.  Hand-off block b is the replay's b-th block: window by
        window, and within a window session by session in stream order.  A replay with more blocks than the Handoff holds
        is refused before anything runs."""
        recs: Dict[Hashable, Tuple[torch.Tensor, List[Optional[str]]]] = {}
        for key, (pcm, statuses) in recordings.items():
            if key not in self.keys:
                raise KeyError("session %r is not open" % (key,))
            if key in self.pending or self.queues[key]:
                raise RuntimeError("session %r has a pushed chunk or queued blocks: tick first, then replay" % (key,))
            pcm, statuses = torch.as_tensor(pcm), list(statuses)
            if pcm.dtype not in (torch.int16, torch.float32):
                raise TypeError("session %r: PCM must be int16 or float32, got %s" % (key, pcm.dtype))
            if pcm.ndim != 2 or pcm.shape[1] != self.cfg.samples_per_chunk or pcm.shape[0] != len(statuses):
                raise ValueError("session %r: pcm %s and %d statuses do not form (c, %d) chunks with one status each"
                                 % (key, tuple(pcm.shape), len(statuses), self.cfg.samples_per_chunk))
            if any(st is not None and not isinstance(st, str) for st in statuses):
                raise TypeError("session %r: statuses must be None or str" % (key,))
            if len(statuses):
                recs[key] = (pcm, statuses)
        if len({p.dtype for p, _ in recs.values()}) > 1:
            raise TypeError("the recordings of one replay must share one PCM dtype")
        out: Dict[Hashable, List[Block]] = {}
        dev, H = self.eng.torch_device, self.history_chunks
        if handoff is not None:
            # the windows split no block count: a chunk gives its blocks (onset history included) in whichever window it falls
            total = sum(gated_block_count(st, self.onset_chunks) for _, st in recs.values())
            if total > handoff.embeds.shape[0]:
                raise RuntimeError("the replay gives %d blocks, more than the Handoff capacity %d" % (total, handoff.embeds.shape[0]))
        cursor = 0
        P = self.eng.get_option("steps_pass_blocks_in_use")
        done = {key: 0 for key in recs}
        while True:
            active = [key for key in recs if done[key] < len(recs[key][1])]
            if not active:
                return out
            q = max(1, P // len(active))
            counts = [min(q, len(recs[key][1]) - done[key]) for key in active]
            pcm = torch.cat([recs[key][0][done[key]:done[key] + c].to(dev) for key, c in zip(active, counts)])
            feats = self.eng.fbank_stream_v([self.keys[key] for key in active], counts, pcm, scale)
            self.stats["fbank_calls"] += 1
            # gather table: the history rows of every window session (H each), then the window's feature blocks
            rows = torch.tensor([self.rows[key] for key in active], device=dev)
            table = torch.cat([self._hist.index_select(0, rows).flatten(0, 1), feats])
            src: List[int] = []
            hist_src: List[int] = []
            labels: List[str] = []
            enc_keys: List[Hashable] = []
            enc_counts: List[int] = []
            first = len(active) * H
            for i, (key, c) in enumerate(zip(active, counts)):
                plan = plan_gated_replay(recs[key][1][done[key]:done[key] + c], H, self.onset_chunks)
                row = [i * H + h for h in range(H)] + list(range(first, first + c))     # table row of history slot / chunk
                hist_src.extend(row[s.index if s.kind == "history" else H + s.index] for s in plan.history)
                if plan.blocks:
                    enc_keys.append(key)
                    enc_counts.append(len(plan.blocks))
                    src.extend(row[s.index if s.kind == "history" else H + s.index] for s, _ in plan.blocks)
                    labels.extend(lab for _, lab in plan.blocks)
                first += c
            if H:
                self._hist.index_copy_(0, rows, table.index_select(0, torch.tensor(hist_src, device=dev)).view(len(active), H,
                                                                                                              *feats.shape[1:]))
            if enc_keys:
                x = table.index_select(0, torch.tensor(src, device=dev))
                ids = [self.keys[key] for key in enc_keys]
                if handoff is not None:
                    # the window's blocks land in the next free blocks of the caller's buffers, as in tick's drains
                    self.eng.handoff_arm(len(src), handoff.embeds[cursor:], handoff.prefix_len, [lab == IPU_START for lab in labels],
                                         handoff.prefix_mask, handoff.attn_mask[cursor:], handoff.row_start[cursor:])
                    enc, emb = self.eng.encode_stream_steps_v(ids, enc_counts, x, want_adapter=False)
                else:
                    enc, emb = self.eng.encode_stream_steps_v(ids, enc_counts, x)
                self.stats["encode_calls"] += 1
                self.stats["session_steps"] += len(src)
                owners = [key for key, c in zip(enc_keys, enc_counts) for _ in range(c)]
                if handoff is not None:
                    # the views tick(handoff=) returns, cut in four calls rather than two per block: [st0:] of every
                    # block, st0 = 0 for 'ipu_sl' (chat prefix included) and prefix_len otherwise
                    win = slice(cursor, cursor + len(src))
                    views = {st0: (handoff.embeds[win, st0:].unbind(0), handoff.attn_mask[win, st0:].unbind(0))
                             for st0 in (0, handoff.prefix_len)}
                for b, (key, lab) in enumerate(zip(owners, labels)):
                    if handoff is not None:
                        e, m = views[0 if lab == IPU_START else handoff.prefix_len]
                        blk = Block(enc[b], e[b], lab, m[b])
                    else:
                        blk = Block(enc[b], emb[b] if emb is not None else None, lab)
                    out.setdefault(key, []).append(blk)
                    if self.block_log is not None:
                        self.block_log.append((key, x[b], lab))
                cursor += len(src)
            for key, c in zip(active, counts):
                done[key] += c

    def history(self, key: Hashable) -> torch.Tensor:
        return self._hist[self.rows[key]]
