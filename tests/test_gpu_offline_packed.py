"""fo_encode_offline_packed / Engine.encode_offline_packed: utterances of different lengths packed end to end, no padding rows.
Every utterance's rows must be what the reference's full-utterance forward returns for it alone -- against the CPU oracle run
per utterance, against the padded fo_encode_offline (bit for bit for a one-utterance call; the valid rows of a ragged padded
batch for every variant without a two-sided time convolution), and on the shipped model in bf16.  Refused calls enqueue
nothing."""
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
BF16_RAGGED_TOL = 4e-3         # bf16 packed vs padded valid rows: the split-K plans of the GEMMs differ with the row count
LENS = [7, 8, 19, 67, 203, 1003]
CHUNKINGS = [(4, 16), (4, -1), (-1, -1), (1, 16), (8, 8)]
VARIANTS = ["tiny", "tiny_bn", "tiny_linear", "cnn", "two", "tiny_conv1d", "tiny_concat", "tiny_postnorm_concat", "tiny_mlconv"]


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def bf16_weights(sd):
    keep = ("pos_bias", "conv.0.weight")
    return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}


def variant(name):
    """cnn: CNNAdapter; two: the two-conv CNNSubsampling (llm_dim > 4 * d_model); the rest are configs/<name>.yaml."""
    if name in ("cnn", "two"):
        base = path_config_from_dict(load_yaml("tiny_bn"))
        return dataclasses.replace(base, adapter_type="cnn") if name == "cnn" else dataclasses.replace(base, llm_dim=base.d_model * 4 + 64)
    return load_path_config(name)


def seeds(name):
    return 3, 5 if name in ("cnn", "two") else 3


def engine(cfg, seed, adapter_seed, **kw):
    from freeze_omni_b200.engine import Engine
    return Engine(cfg, make_encoder_state(cfg, seed), make_adapter_state(cfg, adapter_seed), **kw)


def packed_feats(cfg, lens, seed):
    g = torch.Generator().manual_seed(seed)
    return [9.0 + 3.0 * torch.randn(t, cfg.feat_dim, generator=g) for t in lens]


def padded(feats):
    T = max(f.shape[0] for f in feats)
    x = torch.zeros(len(feats), T, feats[0].shape[1])
    for i, f in enumerate(feats):
        x[i, :f.shape[0]] = f
    return x, np.array([f.shape[0] for f in feats], dtype=np.int32)


@pytest.mark.parametrize("name", VARIANTS)
def test_packed_vs_oracle_per_utterance(name):
    """Lengths 7 .. 1003 in one call, every chunking: each utterance against the oracle's forward of it alone, 1e-4."""
    cfg = variant(name)
    es, as_ = seeds(name)
    eng = engine(cfg, es, as_, max_sessions=2)
    esd, asd = make_encoder_state(cfg, es), make_adapter_state(cfg, as_)
    feats = packed_feats(cfg, LENS, 40)
    try:
        for c, L in CHUNKINGS:
            enc, y, eo, ao = eng.encode_offline_packed(torch.cat(feats), LENS, c, L)
            assert enc.shape[0] == eo[-1] and y.shape[0] == ao[-1]
            enc, y = enc.cpu(), y.cpu()
            for i, f in enumerate(feats):
                xo, _, yo, _ = O.offline_path(cfg, esd, asd, f[None], torch.tensor([f.shape[0]]), c, L)
                assert xo.shape[1] == eo[i + 1] - eo[i] and yo.shape[1] == ao[i + 1] - ao[i], (c, L, i)
                assert maxabs(enc[eo[i]:eo[i + 1]], xo[0]) < FP32_TOL, (c, L, i)
                assert maxabs(y[ao[i]:ao[i + 1]], yo[0]) < FP32_TOL, (c, L, i)
    finally:
        eng.close()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("name", VARIANTS)
def test_one_utterance_bit_exact_with_padded(name, dtype):
    """A packed call of one utterance runs the padded call's arithmetic: equal bit for bit, encoder and adapter rows."""
    cfg = variant(name)
    eng = engine(cfg, *seeds(name), dtype=dtype, max_sessions=2)
    try:
        for t, (c, L) in ((203, (4, 16)), (1003, (-1, -1)), (67, (8, 8))):
            f = packed_feats(cfg, [t], t)[0]
            enc, y, _, _ = eng.encode_offline_packed(f, [t], c, L)
            pe, _, py, _ = eng.encode_offline(f[None], np.array([t], dtype=np.int32), c, L)
            assert torch.equal(enc, pe[0]) and torch.equal(y, py[0]), (t, c, L)
    finally:
        eng.close()


@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_RAGGED_TOL)])
@pytest.mark.parametrize("name", [v for v in VARIANTS if v != "tiny_mlconv"])
def test_ragged_packed_matches_padded_valid_rows(name, dtype, tol):
    """Without a two-sided time convolution every receptive field stays inside the valid frames, so the packed rows equal
    the valid rows of the padded call: fp32 1e-4; bf16 differs only by the GEMM plans of another row count."""
    cfg = variant(name)
    eng = engine(cfg, *seeds(name), dtype=dtype, max_sessions=2)
    feats = packed_feats(cfg, LENS, 41)
    x, il = padded(feats)
    try:
        worst = 0.0
        for c, L in ((4, 16), (-1, -1)):
            enc, y, eo, ao = eng.encode_offline_packed(torch.cat(feats), LENS, c, L)
            pe, _, py, _ = eng.encode_offline(x, il, c, L)
            for i in range(len(LENS)):
                worst = max(worst, maxabs(enc[eo[i]:eo[i + 1]].cpu(), pe[i, :eo[i + 1] - eo[i]].cpu()),
                            maxabs(y[ao[i]:ao[i + 1]].cpu(), py[i, :ao[i + 1] - ao[i]].cpu()))
        print("%s %s packed vs padded valid rows: max-abs %.3g" % (name, dtype, worst))
        assert worst < tol
    finally:
        eng.close()


def test_multilayered_conv1d_packed_vs_padded_rows():
    """MultiLayeredConv1d pads (k-1)/2 rows on both sides, so in a padded batch the last valid rows of a shorter utterance see
    pad-row content; the packed call gives each utterance its own zero padding (the per-utterance forward, checked against the
    oracle above).  The longest utterance of the padded batch has no pad rows and agrees; the others are reported."""
    cfg = load_path_config("tiny_mlconv")
    eng = engine(cfg, 3, 3, max_sessions=2)
    feats = packed_feats(cfg, LENS, 42)
    x, il = padded(feats)
    try:
        enc, _, eo, _ = eng.encode_offline_packed(torch.cat(feats), LENS, 4, 16)
        pe, _, _, _ = eng.encode_offline(x, il, 4, 16)
        d = [maxabs(enc[eo[i]:eo[i + 1]].cpu(), pe[i, :eo[i + 1] - eo[i]].cpu()) for i in range(len(LENS))]
        print("tiny_mlconv packed vs padded valid rows per utterance: " + " ".join("%.3g" % v for v in d))
        assert d[-1] < FP32_TOL
    finally:
        eng.close()


def test_shipped_bf16_ragged_vs_oracle():
    """Shipped model, bf16: 16 utterances of U[10, 30] s (seeded) in one call, each against the oracle on bf16-rounded weights."""
    cfg = load_path_config("shipped")
    eng = engine(cfg, 0, 0, dtype=torch.bfloat16, max_sessions=2)
    rng = np.random.default_rng(7)
    lens = [int(v) for v in rng.integers(1000, 3001, size=16)]      # 10 ms frames
    feats = packed_feats(cfg, lens, 43)
    esd, asd = bf16_weights(make_encoder_state(cfg, 0)), bf16_weights(make_adapter_state(cfg, 0))
    try:
        enc, y, eo, ao = eng.encode_offline_packed(torch.cat(feats), lens)
        enc, y = enc.cpu(), y.cpu()
        we = wy = 0.0
        for i, f in enumerate(feats):
            xo, _, yo, _ = O.offline_path(cfg, esd, asd, f[None], torch.tensor([f.shape[0]]), cfg.chunk_size, cfg.left_chunks)
            we, wy = max(we, maxabs(enc[eo[i]:eo[i + 1]], xo[0])), max(wy, maxabs(y[ao[i]:ao[i + 1]], yo[0]))
        print("shipped bf16 packed, 16 x U[10,30] s, max-abs vs oracle on bf16 weights: encoder %.4g adapter %.4g" % (we, wy))
        assert we < BF16_TOL and wy < BF16_TOL
    finally:
        eng.close()


def test_refusals_enqueue_nothing():
    from freeze_omni_b200.engine import Engine
    from freeze_omni_b200 import _lib
    cfg = load_path_config("tiny")
    eng = engine(cfg, 3, 3, max_sessions=2)
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    feats = packed_feats(cfg, [40, 9], 44)
    try:
        long_t = 4 * cfg.pos_max_len + 7                  # T' = pos_max_len + 1
        cases = [
            (torch.zeros(0, cfg.feat_dim), np.zeros(0, np.int32)),                   # B = 0
            (torch.cat(feats[:1] + [feats[1][:6]]), np.array([40, 6], np.int32)),     # T_i < 7
            (torch.zeros(long_t, cfg.feat_dim), np.array([long_t], np.int32)),        # past the rel-pos table
        ]
        for f, ln in cases:
            before = eng.stats()["kernel_launches"]
            rc = eng.lib.fo_encode_offline_packed(eng._h, f.data_ptr(), ln.ctypes.data, len(ln), 4, 16, None, None, eng._stream())
            assert rc == -1, len(ln)
            assert eng.stats()["kernel_launches"] == before
        enc, y, eo, ao = eng.encode_offline_packed(torch.cat(feats), [40, 9])
        for i, f in enumerate(feats):
            xo, _, yo, _ = O.offline_path(cfg, esd, asd, f[None], torch.tensor([f.shape[0]]), cfg.chunk_size, cfg.left_chunks)
            assert maxabs(enc[eo[i]:eo[i + 1]].cpu(), xo[0]) < FP32_TOL and maxabs(y[ao[i]:ao[i + 1]].cpu(), yo[0]) < FP32_TOL
    finally:
        eng.close()
    adp = Engine(cfg, None, asd, max_sessions=2)            # a context without an encoder
    try:
        before = adp.stats()["kernel_launches"]
        f = torch.cat(feats)
        ln = np.array([40, 9], np.int32)
        assert adp.lib.fo_encode_offline_packed(adp._h, f.data_ptr(), ln.ctypes.data, 2, 4, 16, None, None, adp._stream()) == -1
        assert adp.stats()["kernel_launches"] == before
        with pytest.raises(_lib.FoError, match="no finalized encoder"):
            adp.encode_offline_packed(f, ln)
    finally:
        adp.close()
