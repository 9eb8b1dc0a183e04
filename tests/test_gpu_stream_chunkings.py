"""The streaming encoder against the CPU oracle at attention geometries other than the shipped one (chunk_size 4,
left_chunks 16).  Window (chunk_size * left_chunks), frames per chunk t, ring capacity, full_chunk and pe_wrap are runtime
values of the attention kernels, and each steers indexing: the ring copy split, the fp16 chunk swizzle, key tiles padded to
16, the 4-keys-per-lane softmax, the multi-chunk ring append of more rows than the ring holds, rel-pos positions past the
sinusoid table's pos_max_len rows.  Every chunking runs at two ring capacities (max_stream_frames = t_in, and the Engine
default), with sessions at different fill levels and pe_index phases sharing calls, as a server's calls mix them.

  C   L   t_in  window  keys/call  largest k  reaches
  4   16  19    64      68         16         control (shipped geometry)
  4   2   19    8       12         30         k*t = 120 > ring_cap 16: the ring append keeps only the last ring_cap rows
  3   1   15    3       6          41         odd t (adapter: stride-1 grid + row pick)
  3   5   15    15      18         37         window not a multiple of 8
  2   8   11    16      18         56
  1   16  7     16      17         112        t = 1
  8   8   35    64      72         8          t = 8: full MMA N; stack kernel at 2 x 8 rows
  4   31  19    124     128        1          every key lane; k = 2 refused naming k = 1
  4   -1  19    1       5          31         the reference's buffersize 1; positions up to 5000 (pe_wrap = pos_max_len)
"""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
from oracle import freeze_omni_oracle as O

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
# bf16 bars, calibrated on a B200 (see the docstrings of the tests that use them)
BF16_ORACLE_TOL = 7.5e-3
BF16_CHUNKS_TOL = 4e-3
STACK_TOL = 4e-4
MAX_KEYS = 128

ROWS = [(4, 16), (4, 2), (3, 1), (3, 5), (2, 8), (1, 16), (8, 8), (4, 31), (4, -1)]
ROW_IDS = ["c%d_l%d" % r for r in ROWS]
CAPS = ["tight", "default"]


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def bf16_weights(sd):
    keep = ("pos_bias", "conv.0.weight")
    return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}


def chunk_cfg(c, left):
    return dataclasses.replace(load_path_config("tiny"), chunk_size=c, left_chunks=left)


def t_in_of(c):
    return 4 * c + 3                 # ((t_in - 1) // 2 - 1) // 2 == c encoder frames


def largest_k(cfg, t):
    return max(1, (MAX_KEYS - cfg.kv_window) // t)


_STATES = {}


def states(cfg, bf16=False):
    """Oracle weights (the same seeds as the engines; the chunking does not change the shapes)."""
    if bf16 not in _STATES:
        esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
        _STATES[bf16] = (bf16_weights(esd), bf16_weights(asd)) if bf16 else (esd, asd)
    return _STATES[bf16]


@pytest.fixture(scope="module")
def engines():
    from freeze_omni_b200.engine import Engine
    made = {}

    def get(c, left, dtype=torch.float32, cap="default"):
        key = (c, left, dtype, cap)
        if key not in made:
            cfg = chunk_cfg(c, left)
            msf = t_in_of(c) if cap == "tight" else None
            made[key] = (cfg, Engine(cfg, make_encoder_state(cfg, 3), make_adapter_state(cfg, 3), dtype=dtype, max_sessions=8,
                                     max_stream_frames=msf))
        return made[key]
    yield get
    for _, eng in made.values():
        eng.close()


def feats_for(cfg, shape, gen):
    return 9.0 + 3.0 * torch.randn(*shape, cfg.feat_dim, generator=gen)


def check_state(eng, cfg, sid, s, n_frames, tag):
    """Bookkeeping bit-exact; every layer's exported K/V cache (cache_len = min(n_frames, window)) and the adapter cache
    against the oracle session."""
    assert eng.state(sid) == (n_frames, s.pe_index), tag
    for li in range(cfg.n_layers):
        k, v = eng.export_kv(sid, li)
        assert k.shape[2] == min(n_frames, cfg.kv_window), tag
        assert maxabs(k, s.buffer[li][0]) < FP32_TOL and maxabs(v, s.buffer[li][1]) < FP32_TOL, (tag, li)
    assert maxabs(eng.export_adapter_cache(sid), s.cache[0]) < FP32_TOL, tag


def chunks_call(eng, cfg, ids, sessions, n_frames, feats, tag):
    """One encode_stream_chunks call of len(ids) sessions x k chunks, every chunk against the oracle run chunk by chunk."""
    k = feats.shape[1]
    t = cfg.chunk_size
    enc, y = eng.encode_stream_chunks(ids, feats.contiguous())
    enc, y = enc.cpu(), y.cpu()
    for row, (sid, s) in enumerate(zip(ids, sessions)):
        for j in range(k):
            eo, yo = s.step_feats(feats[row, j].unsqueeze(0))
            assert maxabs(enc[row, j], eo[0]) < FP32_TOL and maxabs(y[row, j], yo[0]) < FP32_TOL, (tag, row, j)
        n_frames[int(sid)] += k * t
        check_state(eng, cfg, int(sid), s, n_frames[int(sid)], (tag, row))


@pytest.mark.parametrize("cap", CAPS)
@pytest.mark.parametrize("c,left", ROWS, ids=ROW_IDS)
def test_fp32_single_chunk_calls(engines, c, left, cap):
    """Four sessions joining at steps 0, 1, 3 and 5, in a different order in every call, until the first one has wrapped
    its ring twice; the third starts at pe_index = pe_wrap - 2C, so it wraps pe_index on its third call (with left_chunks
    -1 that call reads position pe_wrap = pos_max_len)."""
    cfg, eng = engines(c, left, cap=cap)
    t_in, t = t_in_of(c), c
    assert eng.max_t == min(8, t) if cap == "tight" else eng.max_t == 8
    ring_cap = eng.get_option("ring_cap")
    assert ring_cap == (cfg.kv_window + eng.max_t + 7) // 8 * 8
    esd, asd = states(cfg)
    sessions = [O.StreamSession(cfg, esd, asd) for _ in range(4)]
    ids = eng.alloc(4)
    joins = (0, 1, 3, 5)
    sessions[2].pe_index = cfg.pe_wrap - 2 * c
    eng.set_pe_index(ids[2:3], cfg.pe_wrap - 2 * c)
    n_frames = {int(i): 0 for i in ids}
    gen = torch.Generator().manual_seed(1000 + 10 * c + left)
    rng = np.random.default_rng(c * 100 + left)
    try:
        for step in range(2 * ring_cap // t + 2):
            order = rng.permutation([j for j in range(4) if joins[j] <= step])
            feats = feats_for(cfg, (len(order), t_in), gen)
            enc, y = eng.encode_stream(ids[order], feats)
            enc, y = enc.cpu(), y.cpu()
            for row, j in enumerate(order):
                eo, yo = sessions[j].step_feats(feats[row:row + 1])
                assert maxabs(enc[row], eo[0]) < FP32_TOL and maxabs(y[row], yo[0]) < FP32_TOL, (step, j)
                n_frames[int(ids[j])] += t
                check_state(eng, cfg, int(ids[j]), sessions[j], n_frames[int(ids[j])], (step, j))
        assert n_frames[int(ids[0])] >= 2 * ring_cap
    finally:
        eng.free(ids)


def _sat_chunks(cfg, t, ring_cap):
    """Chunks after which the saturated ring window [n - window, n) wraps around the ring's end."""
    w = cfg.kv_window
    for p in range(1, 4 * ring_cap):
        n = p * t
        if n >= w and (w == 1 or (n - w) % ring_cap + w > ring_cap):
            return p
    raise AssertionError("no wrapping phase")


@pytest.mark.parametrize("cap", CAPS)
@pytest.mark.parametrize("c,left", ROWS, ids=ROW_IDS)
def test_fp32_k_chunk_calls_mixed_states(engines, c, left, cap):
    """One multi-chunk call over four sessions primed to different states: fresh; window - t frames (saturates inside the
    call); saturated with its ring window wrapping around the ring's end; pe_index = pe_wrap - C (wraps inside the call).
    Then calls of k = the largest allowed, 1 and a middle value; every chunk, the bookkeeping and the caches after each."""
    cfg, eng = engines(c, left, cap=cap)
    t_in, t, w = t_in_of(c), c, cfg.kv_window
    ring_cap = eng.get_option("ring_cap")
    kmax = largest_k(cfg, t)
    esd, asd = states(cfg)
    sessions = [O.StreamSession(cfg, esd, asd) for _ in range(4)]
    ids = eng.alloc(4)
    n_frames = {int(i): 0 for i in ids}
    gen = torch.Generator().manual_seed(2000 + 10 * c + left)
    prime = (0, max(0, w - t) // t, _sat_chunks(cfg, t, ring_cap), 2)
    try:
        for j, p in enumerate(prime):
            while n_frames[int(ids[j])] < p * t:
                k = min(kmax, p - n_frames[int(ids[j])] // t)
                chunks_call(eng, cfg, ids[j:j + 1], sessions[j:j + 1], n_frames, feats_for(cfg, (1, k, t_in), gen), ("prime", j))
        sessions[3].pe_index = cfg.pe_wrap - c
        eng.set_pe_index(ids[3:4], cfg.pe_wrap - c)
        nf2 = n_frames[int(ids[2])]
        assert nf2 >= w and (w == 1 or (nf2 - w) % ring_cap + w > ring_cap)
        order = np.array([2, 0, 3, 1])
        for k in (kmax, 1, max(1, kmax // 2)):
            chunks_call(eng, cfg, ids[order], [sessions[j] for j in order], n_frames, feats_for(cfg, (4, k, t_in), gen), ("k", k))
        if kmax == 1:
            from freeze_omni_b200 import _lib
            with pytest.raises(_lib.FoError, match="the largest k is 1"):
                eng.encode_stream_chunks(ids[:1], feats_for(cfg, (1, 2, t_in), gen))
            check_state(eng, cfg, int(ids[0]), sessions[0], n_frames[int(ids[0])], "refused k = 2")
    finally:
        eng.free(ids)


@pytest.mark.parametrize("c,left", ROWS, ids=ROW_IDS)
def test_bf16_vs_oracle_on_bf16_weights(engines, c, left):
    """bf16 context against the oracle on the same bf16-rounded weights: two sessions, single-chunk calls past saturation
    on the per-kernel chain, then one call of the largest k.  Measured on an NVIDIA B200 at a 1000 W power limit: 2.5e-3 /
    7.4e-4 (encoder / adapter) at the control (4, 16), at most 2.5e-3 / 8.5e-4 at every chunking; the bar is 3 x the
    control."""
    cfg, eng = engines(c, left, dtype=torch.bfloat16)
    t_in, t = t_in_of(c), c
    esd, asd = states(cfg, bf16=True)
    sessions = [O.StreamSession(cfg, esd, asd) for _ in range(2)]
    ids = eng.alloc(2)
    gen = torch.Generator().manual_seed(3000 + 10 * c + left)
    we = wy = 0.0
    eng.set_option("stack_rows", 0)               # the per-kernel chain (the stack kernel is held to it below)
    try:
        for i in range(max(cfg.left_chunks, 1) + 4):
            feats = feats_for(cfg, (2, t_in), gen)
            enc, y = eng.encode_stream(ids, feats)
            for b in range(2):
                eo, yo = sessions[b].step_feats(feats[b:b + 1])
                we, wy = max(we, maxabs(enc[b].cpu(), eo[0])), max(wy, maxabs(y[b].cpu(), yo[0]))
        k = largest_k(cfg, t)
        feats = feats_for(cfg, (2, k, t_in), gen)
        enc, y = eng.encode_stream_chunks(ids, feats)
        for b in range(2):
            for j in range(k):
                eo, yo = sessions[b].step_feats(feats[b, j].unsqueeze(0))
                we, wy = max(we, maxabs(enc[b, j].cpu(), eo[0])), max(wy, maxabs(y[b, j].cpu(), yo[0]))
            assert eng.state(int(ids[b]))[1] == sessions[b].pe_index
    finally:
        eng.set_option("stack_rows", 8)
        eng.free(ids)
    print("bf16 vs oracle c%d l%d: encoder %.4g adapter %.4g" % (c, left, we, wy))
    assert eng.stats()["act_saturations"] == 0
    assert we < BF16_ORACLE_TOL and wy < BF16_ORACLE_TOL


@pytest.mark.parametrize("c,left", ROWS, ids=ROW_IDS)
def test_bf16_k_chunk_vs_single_chunk_calls(engines, c, left):
    """Twin sessions on one bf16 engine, the same features: calls of k = largest, 1, middle against single-chunk calls.
    Both run the same GEMMs on the same bf16 weights; the fp16 attention kernels (multi-chunk vs single-chunk) and the
    GEMM tile plans for n*k*t vs n*t rows differ, and with them the fp16 rounding of the staged activations.  Measured on
    an NVIDIA B200 at a 1000 W power limit: at most 1.4e-3 over the chunkings (1.1e-3 at the control); bar 4e-3."""
    cfg, eng = engines(c, left, dtype=torch.bfloat16)
    t_in, t = t_in_of(c), c
    kmax = largest_k(cfg, t)
    a, b = eng.alloc(2), eng.alloc(2)
    gen = torch.Generator().manual_seed(4000 + 10 * c + left)
    worst = 0.0
    eng.set_option("stack_rows", 0)
    try:
        for k in (kmax, 1, max(1, kmax // 2), kmax):
            feats = feats_for(cfg, (2, k, t_in), gen)
            enc, y = eng.encode_stream_chunks(a, feats)
            for j in range(k):
                e1, y1 = eng.encode_stream(b, feats[:, j].contiguous())
                worst = max(worst, maxabs(enc[:, j].cpu(), e1.cpu()), maxabs(y[:, j].cpu(), y1.cpu()))
            for s, r in zip(a, b):
                assert eng.state(int(s)) == eng.state(int(r)), k
    finally:
        eng.set_option("stack_rows", 8)
        eng.free(a)
        eng.free(b)
    print("bf16 k-chunk vs single-chunk c%d l%d: %.4g" % (c, left, worst))
    assert worst < BF16_CHUNKS_TOL


def _stack_plan_ok(cfg, n, t):
    from freeze_omni_b200 import _lib
    prop = torch.cuda.get_device_properties(0)
    smem = getattr(prop, "shared_memory_per_block_optin", 232448)
    out = [C.c_int() for _ in range(5)]
    rc = _lib.load().fo_debug_stack_plan(cfg.d_model, cfg.ffn_dim, cfg.n_heads, n, t, cfg.kv_window, cfg.n_layers,
                                         prop.multi_processor_count, smem, *[C.byref(o) for o in out])
    return rc == 0


@pytest.mark.parametrize("c,left", ROWS, ids=ROW_IDS)
def test_bf16_stack_kernel_vs_chain(engines, c, left):
    """Two sessions per call (2 x t <= 16 token rows): the one-launch layer stack (stack_rows 16) against the per-kernel
    chain (stack_rows 0) on twin sessions, past saturation.  Where fo_debug_stack_plan says the step does not qualify,
    the stack kernel must not run.  Measured on an NVIDIA B200 at a 1000 W power limit: at most 3.6e-4 (control)."""
    cfg, eng = engines(c, left, dtype=torch.bfloat16)
    t_in, t = t_in_of(c), c
    qualifies = _stack_plan_ok(cfg, 2, t)
    a, b = eng.alloc(2), eng.alloc(2)
    gen = torch.Generator().manual_seed(5000 + 10 * c + left)
    steps = max(cfg.left_chunks, 1) + 4
    worst = 0.0
    try:
        l0 = eng.get_option("stack_launches")
        for i in range(steps):
            feats = feats_for(cfg, (2, t_in), gen)
            eng.set_option("stack_rows", 16)
            e1, y1 = eng.encode_stream(a, feats)
            eng.set_option("stack_rows", 0)
            e0, y0 = eng.encode_stream(b, feats)
            worst = max(worst, maxabs(e1.cpu(), e0.cpu()), maxabs(y1.cpu(), y0.cpu()))
        assert eng.get_option("stack_launches") - l0 == (steps if qualifies else 0)
        for s, r in zip(a, b):
            assert eng.state(int(s)) == eng.state(int(r))
    finally:
        eng.set_option("stack_rows", 8)
        eng.free(a)
        eng.free(b)
    print("stack kernel vs chain c%d l%d (qualifies %d): %.4g" % (c, left, qualifies, worst))
    assert worst < STACK_TOL


def _refused(eng, cfg, ids, call, match, sessions, n_frames):
    """A refused call enqueues no kernel and leaves every session as it was."""
    from freeze_omni_b200 import _lib
    torch.cuda.synchronize()
    before = [eng.state(int(i)) for i in ids]
    launches = eng.stats()["kernel_launches"]
    with pytest.raises(_lib.FoError, match=match):
        call()
    torch.cuda.synchronize()
    assert eng.stats()["kernel_launches"] == launches
    assert [eng.state(int(i)) for i in ids] == before
    for i, s in zip(ids, sessions):
        if n_frames[int(i)]:
            check_state(eng, cfg, int(i), s, n_frames[int(i)], match)


def test_refuses_nine_frames_per_chunk(engines):
    """39 feature frames give 9 encoder frames; the streaming attention takes 8.  The Engine's default max_stream_frames
    (39) caps max_t at 8, so the call is refused before anything is enqueued, and the next valid call still matches."""
    cfg, eng = engines(4, 16)
    assert eng.max_t == 8 and eng.get_option("ring_cap") == 72
    esd, asd = states(cfg)
    s = O.StreamSession(cfg, esd, asd)
    ids = eng.alloc(1)
    n_frames = {int(ids[0]): 0}
    gen = torch.Generator().manual_seed(6000)
    try:
        chunks_call(eng, cfg, ids, [s], n_frames, feats_for(cfg, (1, 2, 19), gen), "before")
        nine = feats_for(cfg, (1, 39), gen)
        _refused(eng, cfg, ids, lambda: eng.encode_stream(ids, nine), "context allows 1..8", [s], n_frames)
        _refused(eng, cfg, ids, lambda: eng.encode_stream_chunks(ids, nine.unsqueeze(1)), "context allows 1..8", [s], n_frames)
        eight = feats_for(cfg, (1, 35), gen)                  # 8 frames: the largest chunk, still accepted
        e, y = eng.encode_stream(ids, eight)
        eo, yo = s.step_feats(eight)
        n_frames[int(ids[0])] += 8
        assert maxabs(e[0].cpu(), eo[0]) < FP32_TOL and maxabs(y[0].cpu(), yo[0]) < FP32_TOL
        chunks_call(eng, cfg, ids, [s], n_frames, feats_for(cfg, (1, 3, 19), gen), "after")
    finally:
        eng.free(ids)


def test_refuses_window_past_128_keys_offline_still_works(engines):
    """left_chunks 32: window 128 + 4 new frames exceed the 128 keys of the streaming attention.  Streaming is refused up
    front; the full-utterance path of the same context (chunk 4, left 32) still matches the oracle."""
    cfg, eng = engines(4, 32)
    esd, asd = states(cfg)
    ids = eng.alloc(1)
    gen = torch.Generator().manual_seed(7000)
    try:
        f = feats_for(cfg, (1, 19), gen)
        _refused(eng, cfg, ids, lambda: eng.encode_stream(ids, f), "exceeds the 128 keys", [], {int(ids[0]): 0})
        _refused(eng, cfg, ids, lambda: eng.encode_stream_chunks(ids, f.unsqueeze(1)), "exceeds the 128 keys", [], {int(ids[0]): 0})
    finally:
        eng.free(ids)
    feats = feats_for(cfg, (2, 4 * 4 * 40 + 3), gen)
    ilens = torch.tensor([feats.shape[1], feats.shape[1] - 200], dtype=torch.int32)
    xs, m, y, ym = eng.encode_offline(feats, ilens)
    xo, mo, yo, ymo = O.offline_path(cfg, esd, asd, feats, ilens, 4, 32)
    assert torch.equal(m.cpu(), mo) and torch.equal(ym.cpu(), ymo)
    valid = mo[:, 0]
    assert maxabs(xs.cpu()[valid], xo[valid]) < FP32_TOL
    assert maxabs(y.cpu()[ymo[:, 0]], yo[ymo[:, 0]]) < FP32_TOL


def test_refuses_streaming_without_chunk_size(engines):
    """transformer-chunk_size <= 0 (the reference's default when the yaml omits it) is full attention: pe_index would step
    backwards into negative values, where C's % and Python's % disagree.  Streaming is refused with a message; offline
    full attention still matches the oracle."""
    cfg, eng = engines(-1, -1)
    esd, asd = states(cfg)
    ids = eng.alloc(1)
    gen = torch.Generator().manual_seed(8000)
    try:
        f = feats_for(cfg, (1, 19), gen)
        _refused(eng, cfg, ids, lambda: eng.encode_stream(ids, f), "chunk_size > 0", [], {int(ids[0]): 0})
        _refused(eng, cfg, ids, lambda: eng.encode_stream_chunks(ids, f.unsqueeze(1)), "chunk_size > 0", [], {int(ids[0]): 0})
    finally:
        eng.free(ids)
    feats = feats_for(cfg, (1, 203), gen)
    ilens = torch.tensor([203], dtype=torch.int32)
    xs, _, y, _ = eng.encode_offline(feats, ilens)
    xo, _, yo, _ = O.offline_path(cfg, esd, asd, feats, ilens, -1, -1)
    assert maxabs(xs.cpu(), xo) < FP32_TOL and maxabs(y.cpu(), yo) < FP32_TOL
