"""fo_fbank_offline_packed / fo_encode_offline_packed_pcm: recordings of different lengths, PCM in, features or embeddings out.

  1. the packed fbank equals fo_fbank_offline of each utterance alone, bit for bit (int16 / fp32, host / device PCM, odd sample
     offsets, both frontend constant sets);
  2. the PCM encode equals per-utterance fbank + fo_encode_offline_packed, bit for bit, on every toy variant;
  3. a call that runs in several passes equals the features path pass by pass, and the memory it adds follows the pass budget;
  4. per utterance against the oracle fed the call's own features;
  5. refused calls enqueue nothing and leave the outputs untouched."""
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
CHUNKINGS = [(4, 16), (4, -1), (-1, -1)]
VARIANTS = ["tiny", "tiny_linear", "tiny_bn", "tiny_conv1d", "tiny_mlconv", "tiny_postnorm_concat", "cnn", "two"]


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def bf16_weights(sd):
    keep = ("pos_bias", "conv.0.weight")
    return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}


def fork_cfg():
    y = load_yaml("tiny")
    y["frontend"] = dict(y["frontend"], frame_length_ms=16, frame_shift_ms=8, frames_per_chunk=28, context_frames=4)
    return path_config_from_dict(y)


def variant(name):
    """cnn: CNNAdapter; two: the two-conv CNNSubsampling (llm_dim > 4 * d_model); the rest are configs/<name>.yaml."""
    if name in ("cnn", "two"):
        base = path_config_from_dict(load_yaml("tiny_bn"))
        return dataclasses.replace(base, adapter_type="cnn") if name == "cnn" else dataclasses.replace(base, llm_dim=base.d_model * 4 + 64)
    return load_path_config(name)


def seeds(name):
    return 3, 5 if name in ("cnn", "two") else 3


def engine(cfg, seed=3, adapter_seed=3, encoder=True, adapter=True, **kw):
    from freeze_omni_b200.engine import Engine
    return Engine(cfg, make_encoder_state(cfg, seed) if encoder else None, make_adapter_state(cfg, adapter_seed) if adapter else None,
                  max_sessions=2, **kw)


def signals(n_samples, seed, dtype=torch.int16):
    """Seeded speech-like levels: int16 PCM, or the same values as float32 in [-1, 1)."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for n in n_samples:
        x = (0.05 * torch.randn(int(n), generator=g) * 32768).round().clamp(-32768, 32767)
        out.append(x.to(torch.int16) if dtype == torch.int16 else (x / 32768.0).float())
    return out


def sample_counts(cfg, frames, seed):
    """n_samples for the given frame counts, each with a random remainder of 0 .. frame_shift - 1 trailing samples."""
    rng = np.random.default_rng(seed)
    return [cfg.frame_len + (m - 1) * cfg.frame_shift + int(rng.integers(0, cfg.frame_shift)) for m in frames]


def ref_feats(eng, pcms, scale=None):
    return [eng.fbank_offline(p.reshape(1, -1), scale)[0] for p in pcms]


def grid_frames(m):
    return (int(m) + 3) // 4 * 4


def pass_split(frames, budget):
    """The documented pass rule: consecutive utterances while their grid frames (ceil(m / 4) * 4 each) fit the budget; an
    utterance larger than the budget alone."""
    passes, i = [], 0
    while i < len(frames):
        j, g = i + 1, grid_frames(frames[i])
        while j < len(frames) and g + grid_frames(frames[j]) <= budget:
            g += grid_frames(frames[j])
            j += 1
        passes.append((i, j))
        i = j
    return passes


# ---- 1. packed fbank, bit for bit -------------------------------------------------------------------------------------------
def fbank_lengths(cfg, B):
    L, S = cfg.frame_len, cfg.frame_shift
    base = [L, L + 1, L + S - 1, L + S, 2 * L + 1, 3 * cfg.sample_rate + 1, 5 * cfg.sample_rate]
    if B == 1:
        return [3 * cfg.sample_rate + 7]
    rng = np.random.default_rng(B)
    odd = [int(v) | 1 for v in rng.integers(L, 40 * S, size=B - len(base))]     # odd counts: int16 signals start at odd offsets
    out = base + odd
    rng.shuffle(out)
    return out


@pytest.mark.parametrize("frontend", ["shipped", "fork"])
@pytest.mark.parametrize("B", [1, 37])
def test_packed_fbank_bit_exact(frontend, B):
    cfg = load_path_config("tiny") if frontend == "shipped" else fork_cfg()
    eng = engine(cfg)
    try:
        lens = fbank_lengths(cfg, B)
        for dtype in (torch.int16, torch.float32):
            pcms = signals(lens, 17 + B, dtype)
            ref = ref_feats(eng, [p.cuda() for p in pcms])
            for where in ("host", "device"):
                src = [p.cuda() for p in pcms] if where == "device" else [p.numpy() for p in pcms]
                feats, off = eng.fbank_offline_packed(src)
                assert feats.shape[0] == off[-1] == sum(r.shape[0] for r in ref)
                for i, r in enumerate(ref):
                    assert torch.equal(feats[off[i]:off[i + 1]], r), (dtype, where, i, lens[i])
            # a packed 1-D tensor plus n_samples, explicit scale
            feats, off = eng.fbank_offline_packed(torch.cat(pcms).cuda(), scale=0.5, n_samples=lens)
            ref = ref_feats(eng, [p.cuda() for p in pcms], 0.5)
            assert all(torch.equal(feats[off[i]:off[i + 1]], r) for i, r in enumerate(ref))
    finally:
        eng.close()


# ---- 2. PCM encode == per-utterance fbank + packed encode, bit for bit ---------------------------------------------------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name", VARIANTS)
def test_pcm_encode_bit_exact_with_features_path(name, dtype):
    from freeze_omni_b200 import _lib
    cfg = variant(name)
    eng = engine(cfg, *seeds(name), dtype=dtype)
    frames = [7, 8, 19, 67, 203, 1003]
    lens = sample_counts(cfg, frames, 5)
    pcms = [p.cuda() for p in signals(lens, 23)]
    try:
        fb = ref_feats(eng, pcms)
        assert [f.shape[0] for f in fb] == frames
        for c, L in CHUNKINGS:
            pe, py, peo, pao = eng.encode_offline_packed(torch.cat(fb), frames, c, L)
            before = eng.stats()["offline_calls"]
            enc, y, eo, ao, feats = eng.encode_offline_packed_pcm(pcms, c, L, want_feats=True)
            assert eng.stats()["offline_calls"] == before + 1
            assert np.array_equal(eo, peo) and np.array_equal(ao, pao)
            assert torch.equal(enc, pe) and torch.equal(y, py), (c, L)
            assert torch.equal(feats, torch.cat(fb))
        # host PCM and host outputs take the staging paths: same rows
        enc_h = torch.empty_like(enc).cpu()
        host_pcm, ns = torch.cat(pcms).cpu(), np.array(lens, np.int64)
        rc = eng.lib.fo_encode_offline_packed_pcm(eng._h, host_pcm.data_ptr(), _lib.FO_I16, ns.ctypes.data, len(lens), 1.0, 4, 16,
                                                  enc_h.data_ptr(), None, None, eng._stream())
        assert rc == 0
        torch.cuda.synchronize()
        pe, _, _, _ = eng.encode_offline_packed(torch.cat(fb), frames, 4, 16)
        assert torch.equal(enc_h, pe.cpu())
    finally:
        eng.close()


# ---- 3. passes -------------------------------------------------------------------------------------------------------------
BUDGET = 1024


def pass_corpus(cfg):
    """20 utterances: the first longer than the budget (a pass of its own, and the largest in every workspace), then 19 of
    200 .. 400 frames that fill several passes."""
    rng = np.random.default_rng(31)
    frames = [2400] + [int(v) for v in rng.integers(200, 401, size=19)]
    return frames, sample_counts(cfg, frames, 32)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_passes_equal_features_path_per_pass(dtype):
    cfg = load_path_config("tiny")
    eng = engine(cfg, dtype=dtype)
    frames, lens = pass_corpus(cfg)
    pcms = signals(lens, 33)
    try:
        eng.set_option("packed_pass_frames", BUDGET)
        assert eng.get_option("packed_pass_frames") == BUDGET
        passes = pass_split(frames, BUDGET)
        assert len(passes) >= 4 and passes[0] == (0, 1)
        enc, y, eo, ao, feats = eng.encode_offline_packed_pcm([p.numpy() for p in pcms], want_feats=True)
        fb = ref_feats(eng, [p.cuda() for p in pcms])
        for i, j in passes:
            pe, py, _, _ = eng.encode_offline_packed(torch.cat(fb[i:j]), frames[i:j])
            assert torch.equal(enc[eo[i]:eo[j]], pe) and torch.equal(y[ao[i]:ao[j]], py), (i, j)
        assert torch.equal(feats, torch.cat(fb))
    finally:
        eng.close()


def test_pass_memory_follows_the_budget():
    """Fresh engines: the 20-utterance call ends with the device bytes of its largest pass alone, and a one-pass call of the
    same utterances needs more."""
    cfg = load_path_config("tiny")
    frames, lens = pass_corpus(cfg)
    pcm = [p.numpy() for p in signals(lens, 34)]

    def bytes_after(utts, budget):
        eng = engine(cfg)
        try:
            eng.set_option("packed_pass_frames", budget)
            eng.encode_offline_packed_pcm(utts)
            torch.cuda.synchronize()
            return eng.stats()["device_bytes"]
        finally:
            eng.close()

    corpus, largest = bytes_after(pcm, BUDGET), bytes_after(pcm[:1], BUDGET)
    one_pass = bytes_after(pcm, 1 << 20)
    print("device bytes: 20 utterances in passes of %d grid frames %d, largest pass alone %d, one pass %d"
          % (BUDGET, corpus, largest, one_pass))
    assert corpus == largest
    assert one_pass > corpus


def test_default_budget_holds_a_slice_of_32_x_30s():
    """The default pass budget keeps one slice of 32 utterances of 30 s of the shipped bf16 model in one pass, and no setting
    goes past the grid frames the conv2 GEMM of one pass can take."""
    cfg = load_path_config("shipped")
    eng = engine(cfg, 0, 0, dtype=torch.bfloat16)
    try:
        m = 1 + (30 * cfg.sample_rate - cfg.frame_len) // cfg.frame_shift
        P = eng.get_option("packed_pass_frames")
        eng.set_option("packed_pass_frames", 1 << 26)
        cap = eng.get_option("packed_pass_frames")
        print("default packed_pass_frames (shipped, bf16): %d grid frames; largest setting in force: %d" % (P, cap))
        assert len(pass_split([m] * 32, P)) == 1 and P <= cap < 1 << 26
    finally:
        eng.close()


# ---- 4. against the oracle -------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["tiny", "two", "tiny_mlconv", "tiny_conv1d"])
def test_pcm_encode_vs_oracle_fp32(name):
    cfg = variant(name)
    es, as_ = seeds(name)
    eng = engine(cfg, es, as_)
    esd, asd = make_encoder_state(cfg, es), make_adapter_state(cfg, as_)
    frames = [7, 19, 203, 1003]
    lens = sample_counts(cfg, frames, 6)
    try:
        enc, y, eo, ao, feats = eng.encode_offline_packed_pcm([p.numpy() for p in signals(lens, 24)], 4, 16, want_feats=True)
        enc, y, feats = enc.cpu(), y.cpu(), feats.cpu()
        fo = np.concatenate([[0], np.cumsum(frames)])
        for i in range(len(frames)):
            f = feats[fo[i]:fo[i + 1]]
            xo, _, yo, _ = O.offline_path(cfg, esd, asd, f[None], torch.tensor([f.shape[0]]), 4, 16)
            assert maxabs(enc[eo[i]:eo[i + 1]], xo[0]) < FP32_TOL and maxabs(y[ao[i]:ao[i + 1]], yo[0]) < FP32_TOL, i
    finally:
        eng.close()


def test_shipped_bf16_pcm_vs_oracle():
    """Shipped model, bf16: 16 recordings of U[10, 30] s in one call, each against the oracle on bf16-rounded weights fed the
    features the call returned."""
    cfg = load_path_config("shipped")
    eng = engine(cfg, 0, 0, dtype=torch.bfloat16)
    rng = np.random.default_rng(8)
    lens = [int(s * cfg.sample_rate) + int(rng.integers(0, cfg.frame_shift)) for s in rng.uniform(10.0, 30.0, size=16)]
    esd, asd = bf16_weights(make_encoder_state(cfg, 0)), bf16_weights(make_adapter_state(cfg, 0))
    try:
        enc, y, eo, ao, feats = eng.encode_offline_packed_pcm([p.cuda() for p in signals(lens, 25)], want_feats=True)
        enc, y, feats = enc.cpu(), y.cpu(), feats.cpu()
        frames, _, _ = cfg.packed_audio_offsets(lens)
        fo = np.concatenate([[0], np.cumsum(frames)])
        we = wy = 0.0
        for i in range(len(lens)):
            f = feats[fo[i]:fo[i + 1]]
            xo, _, yo, _ = O.offline_path(cfg, esd, asd, f[None], torch.tensor([f.shape[0]]), cfg.chunk_size, cfg.left_chunks)
            we, wy = max(we, maxabs(enc[eo[i]:eo[i + 1]], xo[0])), max(wy, maxabs(y[ao[i]:ao[i + 1]], yo[0]))
        print("shipped bf16 packed PCM, 16 x U[10,30] s, max-abs vs oracle on bf16 weights: encoder %.4g adapter %.4g" % (we, wy))
        assert we < BF16_TOL and wy < BF16_TOL
    finally:
        eng.close()


# ---- 5. refusals -----------------------------------------------------------------------------------------------------------
def test_refusals_enqueue_nothing():
    from freeze_omni_b200 import _lib
    cfg = load_path_config("tiny")
    L, S = cfg.frame_len, cfg.frame_shift
    full = engine(cfg)
    enc_only = engine(cfg, adapter=False)
    adp_only = engine(cfg, encoder=False)
    pcm = torch.zeros(L + (4 * (cfg.pos_max_len + 1) + 7) * S, dtype=torch.int16)      # long enough for every case
    sent = torch.full((4096, 256), 7.0, device="cuda")

    def untouched():
        return bool((sent == 7.0).all())

    def fbank(eng, ns, dtype=_lib.FO_I16):
        ns = np.array(ns, np.int64)
        return eng.lib.fo_fbank_offline_packed(eng._h, pcm.data_ptr(), dtype, ns.ctypes.data, len(ns), 1.0, sent.data_ptr(), eng._stream())

    def encode(eng, ns, y=True):
        ns = np.array(ns, np.int64)
        return eng.lib.fo_encode_offline_packed_pcm(eng._h, pcm.data_ptr(), _lib.FO_I16, ns.ctypes.data, len(ns), 1.0, 4, 16,
                                                    sent.data_ptr(), sent.data_ptr() if y else None, sent.data_ptr(), eng._stream())
    ok = L + 40 * S
    past_pos = L + (4 * (cfg.pos_max_len + 1) + 6) * S          # T' = pos_max_len + 1
    cases = [
        ("fbank B = 0", lambda: fbank(full, []), None),
        ("fbank short utterance", lambda: fbank(full, [ok, L - 1]), "utterance 1"),
        ("fbank bad dtype", lambda: fbank(full, [ok], 7), None),
        ("encode without encoder", lambda: encode(adp_only, [ok]), "no finalized encoder"),
        ("adapter_out without adapter", lambda: encode(enc_only, [ok]), "no adapter"),
        ("encode B = 0", lambda: encode(full, []), None),
        ("encode m < 7", lambda: encode(full, [ok, ok, L + 5 * S]), "utterance 2"),
        ("encode past the positional table", lambda: encode(full, [ok, past_pos]), "utterance 1"),
    ]
    try:
        for what, fn, msg in cases:
            engs = (full, enc_only, adp_only)
            before = [e.stats()["kernel_launches"] for e in engs]
            assert fn() == -1, what
            if msg:
                assert msg in full.lib.fo_last_error().decode(), what
            torch.cuda.synchronize()
            assert [e.stats()["kernel_launches"] for e in engs] == before, what
            assert untouched(), what
        # the encoder-only context still encodes without adapter rows
        enc, y, _, _ = enc_only.encode_offline_packed_pcm([pcm[:ok].numpy()])
        assert y is None and enc.shape[0] > 0
    finally:
        for e in (full, enc_only, adp_only):
            e.close()
