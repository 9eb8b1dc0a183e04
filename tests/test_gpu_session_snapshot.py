"""Session snapshots (fo_session_save / fo_session_restore, Engine.save_sessions / restore_sessions, StreamScheduler.detach /
attach): a session restored from a record continues bit for bit as a twin session that never moved and runs the same calls --
in a fresh engine with other capacities and slot ids, at another ring capacity, in a second slot of the same engine (fork), and
on another GPU.  Every comparison is torch.equal."""
import dataclasses

import numpy as np
import pytest
import torch

from freeze_omni_b200._lib import FoError
from freeze_omni_b200.config import load_path_config, load_yaml, path_config_from_dict
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state

pytestmark = pytest.mark.gpu


def engine(cfg, seed=3, adapter_seed=3, **kw):
    from freeze_omni_b200.engine import Engine
    return Engine(cfg, make_encoder_state(cfg, seed), make_adapter_state(cfg, adapter_seed), **kw)


def variant(name):
    if name in ("cnn", "two"):
        base = path_config_from_dict(load_yaml("tiny_bn"))
        return dataclasses.replace(base, adapter_type="cnn") if name == "cnn" else dataclasses.replace(base, llm_dim=base.d_model * 4 + 64)
    return load_path_config("tiny" if name == "fork_t7" else name)


def pcm_chunks(cfg, n, chunks, seed):
    g = torch.Generator().manual_seed(seed)
    x = (3000.0 * torch.randn(n, chunks, cfg.samples_per_chunk, generator=g)).clamp(-32768, 32767)
    return x.to(torch.int16)


def feats_for(cfg, n, chunks, t_in, seed):
    g = torch.Generator().manual_seed(seed)
    return 9.0 + 3.0 * torch.randn(n, chunks, t_in, cfg.feat_dim, generator=g)


def assert_same_state(ea, a, eb, b, tag=""):
    """(n_frames, pe_index), every layer's exported K/V, the adapter caches and the Conv1dLinear contexts of session a of
    engine ea and session b of engine eb are identical."""
    cfg = ea.cfg
    for sa, sb in zip(np.atleast_1d(a), np.atleast_1d(b)):
        sa, sb = int(sa), int(sb)
        if ea.has_encoder:
            assert ea.state(sa) == eb.state(sb), tag
            for li in range(cfg.n_layers):
                ka, va = ea.export_kv(sa, li)
                kb, vb = eb.export_kv(sb, li)
                assert torch.equal(ka, kb) and torch.equal(va, vb), (tag, li)
                if cfg.ffn_type == "conv1d-linear":
                    assert torch.equal(ea.export_ffn_cache(sa, li), eb.export_ffn_cache(sb, li)), (tag, li)
        if ea.has_adapter and cfg.adapter_type == "subsampling":
            for w in range(2 if cfg.adapter_two_conv else 1):
                ca, cb = ea.export_adapter_cache(sa, w), eb.export_adapter_cache(sb, w)
                assert (ca is None) == (cb is None) and (ca is None or torch.equal(ca, cb)), (tag, w)


def same_outputs(x, y, tag):
    for u, v in zip(x, y):
        assert (u is None) == (v is None) and (u is None or torch.equal(u, v)), tag


def continue_both(ea, a, eb, b, calls, tag):
    """Run the same calls on session(s) a of ea and b of eb; outputs and state identical after every call.  calls: list of
    ("pcm", int16 (n, samples)) | ("chunks", feats (n, k, t_in, F)) | ("feats", feats (n, t_in, F))."""
    for i, (kind, x) in enumerate(calls):
        if kind == "pcm":
            ra, rb = ea.stream_step(a, x), eb.stream_step(b, x)
        elif kind == "chunks":
            ra, rb = ea.encode_stream_chunks(a, x), eb.encode_stream_chunks(b, x)
        else:
            ra, rb = ea.encode_stream(a, x), eb.encode_stream(b, x)
        torch.cuda.synchronize()
        same_outputs(ra, rb, (tag, i, kind))
        assert_same_state(ea, a, eb, b, (tag, i, kind))


def mixed_calls(cfg, n, seed):
    """PCM steps and multi-chunk calls, 1 + 3 + 1 + 2 = 7 chunks."""
    pcm = pcm_chunks(cfg, n, 2, seed).cuda()
    f = feats_for(cfg, n, 5, cfg.chunk_feat_frames, seed + 1).cuda()
    return [("pcm", pcm[:, 0].contiguous()), ("chunks", f[:, :3].contiguous()), ("pcm", pcm[:, 1].contiguous()),
            ("chunks", f[:, 3:5].contiguous())]


def move(src, ids, dst, dst_ids, via="device"):
    if via == "device":
        blob = src.save_sessions(ids)
    else:
        blob = src.save_sessions(ids, out=torch.empty(len(ids), src.snapshot_bytes, dtype=torch.uint8).pin_memory())
    dst.restore_sessions(dst_ids, blob.to(dst.torch_device) if via == "device" else blob)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_pcm_fed_sessions_continue_bit_for_bit_in_a_fresh_engine(dtype):
    """Saved fresh, mid-window, with the ring window wrapping the ring's end, and with pe_index just before its wrap; each
    restored into a fresh slot of another engine (other max_sessions, other slot ids) through a device or a pinned host
    buffer, then both copies run PCM steps and multi-chunk calls."""
    cfg = load_path_config("tiny")
    e1, e2 = engine(cfg, dtype=dtype, max_sessions=3), engine(cfg, dtype=dtype, max_sessions=7)
    try:
        assert e1.snapshot_bytes == e2.snapshot_bytes and e1.snapshot_bytes % 256 == 0
        e1.alloc(1)
        s = e1.alloc(1)
        e2.alloc(2)
        cap = e1.get_option("ring_cap")
        for p, (advance, pe) in enumerate([(0, None), (0, None), (5, None), (0, cfg.pe_wrap - 8)]):
            for c in range(advance):
                e1.stream_step(s, pcm_chunks(cfg, 1, 1, 100 + 10 * p + c)[:, 0].cuda())
            if pe is not None:
                e1.set_pe_index(s, pe)
            nf, _ = e1.state(int(s[0]))
            if p == 2:   # saturated: the window's frames run past the ring's end
                assert nf >= cfg.kv_window and (nf - cfg.kv_window) % cap + cfg.kv_window > cap, nf
            m = e2.alloc(1)
            assert int(m[0]) != int(s[0])
            move(e1, s, e2, m, via="device" if p % 2 == 0 else "host")
            torch.cuda.synchronize()
            assert_same_state(e1, s, e2, m, ("restored", p))
            continue_both(e1, s, e2, m, mixed_calls(cfg, 1, 40 + p), p)
            e2.free(m)
        assert e1.state(int(s[0]))[1] < 8 * cfg.chunk_size      # pe_index wrapped after the last restore
    finally:
        e1.close()
        e2.close()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_across_ring_capacities(dtype):
    """Chunking (3, 1): the ring holds 8 rows with max_stream_frames 15 and 16 with the default.  Saved at one capacity with
    the window wrapping the ring's end, restored at the other, in both directions."""
    cfg = dataclasses.replace(load_path_config("tiny"), chunk_size=3, left_chunks=1)
    tight, wide = engine(cfg, dtype=dtype, max_sessions=2, max_stream_frames=15), engine(cfg, dtype=dtype, max_sessions=3)
    try:
        assert (tight.get_option("ring_cap"), wide.get_option("ring_cap")) == (8, 16)
        f = feats_for(cfg, 1, 40, 15, 7).cuda()
        c0 = 0
        for src, dst in ((tight, wide), (wide, tight)):
            a, b = src.alloc(1), dst.alloc(1)
            for k in (1, 2):                                        # 9 frames: (9 - 3) % 8 + 3 > 8 on the tight ring
                src.encode_stream_chunks(a, f[:, c0:c0 + k].contiguous())
                c0 += k
            move(src, a, dst, b)
            calls = [("feats", f[:, c0].contiguous()), ("chunks", f[:, c0 + 1:c0 + 6].contiguous()), ("feats", f[:, c0 + 6].contiguous())]
            continue_both(src, a, dst, b, calls, (src.get_option("ring_cap"), dst.get_option("ring_cap")))
            c0 = 0
            src.free(a)
            dst.free(b)
    finally:
        tight.close()
        wide.close()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name", ["tiny_linear", "cnn", "two", "tiny_bn", "fork_t7", "tiny_conv1d"])
def test_adapter_and_layer_variants(name, dtype):
    """Every adapter variant (LinearAdapter, CNNAdapter, two-conv CNNSubsampling, BatchNorm, t = 7 through the stride-1 grid and row pick) and the
    Conv1dLinear layers, whose left context the record carries."""
    cfg = variant(name)
    t_in = 32 if name == "fork_t7" else cfg.chunk_feat_frames
    seed = 5 if name in ("cnn", "two") else 3
    e1, e2 = engine(cfg, adapter_seed=seed, dtype=dtype, max_sessions=3), engine(cfg, adapter_seed=seed, dtype=dtype, max_sessions=5)
    try:
        a, _, b = e1.alloc(2), e2.alloc(2), e2.alloc(2)
        f = feats_for(cfg, 2, 12, t_in, 21).cuda()
        e1.encode_stream_chunks(a, f[:, :3].contiguous())
        e1.encode_stream(a, f[:, 3].contiguous())
        move(e1, a, e2, b)
        calls = [("feats", f[:, 4].contiguous()), ("chunks", f[:, 5:8].contiguous()), ("feats", f[:, 8].contiguous())]
        continue_both(e1, a, e2, b, calls, name)
    finally:
        e1.close()
        e2.close()


@pytest.mark.parametrize("n", [1, 2, 16])
def test_shipped_bf16_keeps_the_step_graphs(n):
    """Shipped model, bf16, use_graph on: 1 and 2 sessions take the layer-stack kernel, 16 the per-kernel chain.  A save
    between two graph-replayed steps does not force a re-capture on the source engine, nor a restore on the target: the next
    step of each is one more graph replay."""
    cfg = load_path_config("shipped")
    e1, e2 = engine(cfg, seed=0, adapter_seed=0, dtype=torch.bfloat16, max_sessions=n + 1), \
        engine(cfg, seed=0, adapter_seed=0, dtype=torch.bfloat16, max_sessions=n + 3)
    try:
        assert e1.get_option("use_graph") == 1
        a = e1.alloc(n)
        e2.alloc(2)
        b = e2.alloc(n)
        pcm = pcm_chunks(cfg, n, 6, 77).cuda()
        for c in range(3):                       # eager, capture, replay
            e1.stream_step(a, pcm[:, c].contiguous())
            e2.stream_step(b, pcm[:, c].contiguous())    # warms e2's graph of this shape; the restore overwrites b
        r1, r2 = e1.stats()["graph_replays"], e2.stats()["graph_replays"]
        move(e1, a, e2, b)
        calls = [("pcm", pcm[:, c].contiguous()) for c in range(3, 6)]
        continue_both(e1, a, e2, b, calls[:1], ("shipped", n))
        assert e1.stats()["graph_replays"] == r1 + 1 and e2.stats()["graph_replays"] == r2 + 1
        continue_both(e1, a, e2, b, calls[1:], ("shipped", n))
        if n <= 2:
            assert e1.get_option("stack_launches") > 0
    finally:
        e1.close()
        e2.close()


def test_fork_into_a_second_slot_of_the_same_engine():
    cfg = load_path_config("tiny")
    eng = engine(cfg, dtype=torch.bfloat16, max_sessions=4)
    try:
        a = eng.alloc(2)
        pcm = pcm_chunks(cfg, 2, 4, 5).cuda()
        for c in range(4):
            eng.stream_step(a, pcm[:, c].contiguous())
        b = eng.alloc(2)
        eng.restore_sessions(b[::-1].copy(), eng.save_sessions(a)[[1, 0]].contiguous())      # rows reordered: b[i] from a[i]
        continue_both(eng, a, eng, b, mixed_calls(cfg, 2, 9), "fork")
    finally:
        eng.close()


def test_host_and_device_buffers_give_identical_records():
    cfg = load_path_config("tiny_conv1d")
    eng = engine(cfg, max_sessions=3)
    try:
        a = eng.alloc(3)
        for c, x in enumerate(pcm_chunks(cfg, 3, 3, 8).cuda().unbind(1)):
            eng.stream_step(a, x.contiguous())
        dev = eng.save_sessions(a)
        pinned = eng.save_sessions(a, out=torch.empty_like(dev, device="cpu").pin_memory())
        pageable = eng.save_sessions(a, out=torch.empty_like(dev, device="cpu"))
        assert torch.equal(dev.cpu(), pinned) and torch.equal(pinned, pageable)
        one = eng.save_sessions(a[1:2])
        assert torch.equal(one[0], dev[1])          # a record does not depend on its neighbours in the call
        eng.restore_sessions(a, pageable)            # host restore through the staging buffer, then byte-identical again
        assert torch.equal(eng.save_sessions(a), dev)
    finally:
        eng.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_across_gpus():
    from freeze_omni_b200.engine import Engine
    cfg = load_path_config("shipped")
    esd, asd = make_encoder_state(cfg, 0), make_adapter_state(cfg, 0)
    e0 = Engine(cfg, esd, asd, dtype=torch.bfloat16, device=0, max_sessions=4)
    e1 = Engine(cfg, esd, asd, dtype=torch.bfloat16, device=1, max_sessions=6)
    try:
        a = e0.alloc(2)
        e1.alloc(3)
        b = e1.alloc(2)
        pcm = pcm_chunks(cfg, 2, 6, 31)
        for c in range(3):
            e0.stream_step(a, pcm[:, c].contiguous().cuda(0))
        blob = e0.save_sessions(a)
        with pytest.raises(ValueError, match="copy it over"):
            e1.restore_sessions(b, blob)
        with torch.cuda.device(1):
            e1.restore_sessions(b, blob.to(e1.torch_device))
        for c in range(3, 6):
            r0 = e0.stream_step(a, pcm[:, c].contiguous().cuda(0))
            with torch.cuda.device(1):
                r1 = e1.stream_step(b, pcm[:, c].contiguous().cuda(1))
            torch.cuda.synchronize(0)
            torch.cuda.synchronize(1)
            same_outputs([x.cpu() for x in r0], [x.cpu() for x in r1], ("gpus", c))
            for s0, s1 in zip(a, b):
                assert e0.state(int(s0)) == e1.state(int(s1))
    finally:
        e0.close()
        e1.close()


def test_refusals_name_the_field_and_touch_no_slot():
    cfg = load_path_config("tiny")
    eng = engine(cfg, dtype=torch.bfloat16, max_sessions=6)
    others = {
        "chunk_size": engine(dataclasses.replace(cfg, chunk_size=3, left_chunks=5), dtype=torch.bfloat16, max_sessions=1),
        "n_layers": engine(dataclasses.replace(cfg, n_layers=1), dtype=torch.bfloat16, max_sessions=1),
        "dtype": engine(cfg, dtype=torch.float32, max_sessions=1),
    }
    try:
        t, twin = eng.alloc(2), eng.alloc(2)
        pcm = pcm_chunks(cfg, 2, 3, 3).cuda()
        for c in range(3):
            eng.stream_step(t, pcm[:, c].contiguous())
            eng.stream_step(twin, pcm[:, c].contiguous())
        good = eng.save_sessions(twin)
        B = eng.snapshot_bytes

        def refused(blob, match, ids=t):
            with pytest.raises(FoError, match="error -1: .*" + match):
                eng.restore_sessions(ids, blob)

        for field, other in others.items():
            o = other.save_sessions(other.alloc(1))
            bad = good.clone()
            bad[1, :256] = o[0, :256]                                # record 1 of 2 is foreign: neither slot is written
            refused(bad, "record 1: %s is" % field)
        for word, value, match in ((0, 0x12345678, "bad magic"), (1, 2, "format version 2"), (2, B - 256, "record size")):
            bad = good.clone()
            bad.view(torch.int32).view(2, -1)[0, word] = value
            refused(bad, "record 0: " + match)
        free_id = np.setdiff1d(np.arange(6), np.concatenate([t, twin]))[:1].astype(np.int32)
        refused(good, "not allocated", ids=np.array([t[0], free_id[0]], np.int32))
        refused(good, "twice", ids=np.array([t[0], t[0]], np.int32))
        with pytest.raises(ValueError):
            eng.restore_sessions(t, good[:, :-256].contiguous())   # a truncated buffer never reaches the library
        continue_both(eng, t, eng, twin, mixed_calls(cfg, 2, 4), "refused")
    finally:
        eng.close()
        for o in others.values():
            o.close()


def test_scheduler_detach_attach_on_the_gpu():
    """The gating golden's stream (speech onsets replaying history) with a detach from one engine and an attach to a second
    engine in the middle gives the Block outputs of the unsplit run."""
    from conftest import load_golden
    from freeze_omni_b200.scheduler import StreamScheduler
    g = load_golden("gating")
    cfg = load_path_config("tiny")
    engines = [engine(cfg, max_sessions=4) for _ in range(3)]
    try:
        def run(move_at):
            sch = StreamScheduler(engines[0] if move_at is None else engines[1], bucket=1, max_sessions=2)
            dst = StreamScheduler(engines[2], bucket=1, max_sessions=2)
            dst.open("other")
            sch.open("u")
            outs = []
            for i, st in enumerate(g["statuses"]):
                if i == move_at:
                    dst.attach("u", sch.detach("u"))
                    sch = dst
                pcm = torch.from_numpy(g["pcm"][i * 2560:(i + 1) * 2560].astype(np.float32) / 32768.0)
                sch.push("u", pcm, str(st) if str(st) else None)
                outs.append([(b.enc.clone(), b.emb.clone(), b.status) for b in sch.tick(float(g["scale"])).get("u", [])])
            return outs
        ref, moved = run(None), run(10)
        assert sum(len(o) for o in ref) == len(g["labels"])
        for i, (x, y) in enumerate(zip(ref, moved)):
            assert len(x) == len(y), i
            for (e0, y0, s0), (e1, y1, s1) in zip(x, y):
                assert s0 == s1 and torch.equal(e0, e1) and torch.equal(y0, y1), i
    finally:
        for e in engines:
            e.close()
