"""Pin the CPU oracle to the vectors produced by the reference modules (tests/golden/make_golden.py).
These run without a GPU."""
import dataclasses

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
from oracle import freeze_omni_oracle as O

FP32_TOL = 1e-4      # north_star: encoder and adapter outputs within 1e-4 max-abs in fp32


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1.0)))


def test_fbank_known_answers_from_survey(golden):
    g = golden("fbank")
    wav = torch.cat([torch.zeros(240), torch.from_numpy(g["question_pcm"].astype(np.float32))])
    pad = (-(len(g["question_pcm"])) % 2560)
    wav = torch.cat([wav, torch.zeros(pad)])
    out = O.fbank(wav)
    assert out.shape == (208, 80)
    assert abs(float(out.sum()) - 156308.2261) < 0.5
    assert abs(float(out.min()) - (-15.9424)) < 1e-3 and int((out < -15.94).sum()) == 2400
    np.testing.assert_allclose(out[100, :6].numpy(), [11.3679, 13.1892, 12.8945, 19.0391, 20.4948, 21.0801], atol=2e-4)
    np.testing.assert_allclose(out[150, 40:44].numpy(), [8.4979, 8.0307, 8.7213, 8.4356], atol=2e-4)


def test_fbank_matches_reference_vectors(golden):
    g = golden("fbank")
    assert torch.equal(O.povey_window(400), torch.from_numpy(g["window"]))
    assert torch.equal(O.mel_banks(80, 512, 16000.0)[:, :256], torch.from_numpy(g["mel"]))
    wav = torch.cat([torch.zeros(240), torch.from_numpy(g["synth_pcm"].astype(np.float32))])
    assert rel_err(O.fbank(wav).numpy(), g["synth_offline"]) < 1e-5


def test_streaming_frontend_default_and_fork(golden):
    g = golden("fbank")
    pcm = g["question_pcm"]
    n = -(-len(pcm) // 2560) * 2560
    x = np.zeros(n, np.float32)
    x[:len(pcm)] = pcm
    fe = O.StreamingFrontend()
    outs = [fe.process(torch.from_numpy(x[i:i + 2560] / 32768.0), 32767.0) for i in range(0, n, 2560)]
    assert rel_err(torch.cat(outs, 0).numpy(), g["question_gating_default"]) < 1e-5
    fe = O.StreamingFrontend(16000, 16, 8, 28, 4, 80)
    nf = (n // 3584) * 3584
    outs = [fe.process(torch.from_numpy(x[i:i + 3584] / 32768.0), 32767.0) for i in range(0, nf, 3584)]
    assert outs[0].shape == (1, 32, 80)
    assert rel_err(torch.cat(outs, 0).numpy(), g["question_gating_fork"]) < 1e-5


def test_streaming_fbank_equals_offline(golden):
    """SURVEY 2.4-10: per-frame DC removal and pre-emphasis make the streamed frames equal the
    offline frames of [240 zeros | signal]."""
    g = golden("fbank")
    pcm = g["synth_pcm"].astype(np.float32)[:2560 * 10]
    fe = O.StreamingFrontend()
    st = torch.cat([fe.process(torch.from_numpy(pcm[i:i + 2560]), 1.0)[0, 3:] for i in range(0, len(pcm), 2560)])
    off = O.fbank(torch.cat([torch.zeros(240), torch.from_numpy(pcm)]))
    assert torch.equal(st, off)


def test_masks_bit_exact(golden):
    g = golden("masks")
    for key, packed in g.items():
        T, c, L = (int(s[1:]) for s in key.split("_"))
        want = np.unpackbits(packed)[:T * T].reshape(T, T).astype(bool)
        got = O.subsequent_chunk_mask(T, c, L).numpy()
        assert np.array_equal(got, want), key
        for i in range(T):
            s, e = O.chunk_window(i, T, c, L)
            assert np.array_equal(np.flatnonzero(want[i]), np.arange(s, e)), key


def test_subsampled_lengths():
    cfg = load_path_config("tiny")
    x = torch.zeros(2, 67, 80)
    _, m = O.EncoderOracle(cfg, make_encoder_state(cfg, 3)).forward(x, torch.tensor([67, 40]), 4, 16)
    assert m.squeeze(1).sum(1).tolist() == [16, 9]       # SURVEY 8c probed values


@pytest.fixture(scope="module")
def tiny():
    cfg = load_path_config("tiny")
    return cfg, make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)


def _run_stream(cfg, esd, asd, feats_seq):
    enc = O.EncoderOracle(cfg, esd)
    buf, cache, pe = enc.new_buffer(), None, 0
    eos, ys, pes = [], [], []
    for f in feats_seq:
        eo, buf, pe = enc.infer(torch.from_numpy(f), buf, pe)
        y, _, cache = O.adapter_forward(cfg, asd, eo, torch.ones(eo.size(0), 1, eo.size(1), dtype=torch.bool), cache)
        eos.append(eo)
        ys.append(y)
        pes.append(pe)
    return torch.stack(eos).numpy(), torch.stack(ys).numpy(), pes, buf, cache


def test_tiny_stream(golden, tiny):
    cfg, esd, asd = tiny
    g = golden("tiny")
    eo, y, pes, buf, cache = _run_stream(cfg, esd, asd, g["stream_feats"])
    assert np.abs(eo - g["stream_enc_out"]).max() < FP32_TOL
    assert np.abs(y - g["stream_adapter_out"]).max() < FP32_TOL
    assert pes == g["stream_pe_index"].tolist()
    for li in (0, 1):                                                # the golden keeps a sample of the head dimension
        assert np.abs(buf[li][0].numpy()[..., g["kv_cols"]] - g["stream_k_cache_l%d" % li]).max() < FP32_TOL
        assert np.abs(buf[li][1].numpy()[..., g["kv_cols"]] - g["stream_v_cache_l%d" % li]).max() < FP32_TOL
    assert buf[0][0].shape[2] == cfg.kv_window
    assert np.abs(cache[0].numpy() - g["stream_adapter_cache"]).max() < FP32_TOL


def test_tiny_stream_from_pcm(golden, tiny):
    cfg, esd, asd = tiny
    g = golden("tiny")
    sess = O.StreamSession(cfg, esd, asd)
    pcm = g["stream_pcm"][1].astype(np.float32) / 32768.0
    for i in range(4):
        feats, eo, y = sess.step_pcm(torch.from_numpy(pcm[i * 2560:(i + 1) * 2560]))
        assert rel_err(feats.numpy(), g["stream_feats"][i, 1:2]) < 1e-5
        assert np.abs(eo.numpy() - g["stream_enc_out"][i, 1:2]).max() < FP32_TOL


def test_tiny_stream_seven_frames_per_call(golden, tiny):
    """The fork feeds 32 fbank frames -> 7 encoder frames while pe_index still advances by 4
    (SURVEY 2.4-2): reproduce, don't repair."""
    cfg, esd, asd = tiny
    g = golden("tiny")
    eo, y, pes, buf, cache = _run_stream(cfg, esd, asd, g["t7_feats"])
    assert eo.shape[2] == 7
    assert np.abs(eo - g["t7_enc_out"]).max() < FP32_TOL
    assert np.abs(y - g["t7_adapter_out"]).max() < FP32_TOL
    assert pes == g["t7_pe_index"].tolist()


@pytest.mark.parametrize("c,L", [(4, 16), (4, 2), (-1, -1), (4, -1), (3, 1)])
def test_tiny_offline(golden, tiny, c, L):
    cfg, esd, asd = tiny
    g = golden("tiny")
    xs, m, y, ym = O.offline_path(cfg, esd, asd, torch.from_numpy(g["off_feats"]), torch.from_numpy(g["off_ilens"]), c, L)
    tag = "c%d_L%d" % (c, L)
    assert np.array_equal(m.numpy(), g["off_mask_" + tag])
    assert np.array_equal(ym.numpy(), g["off_amask_" + tag])
    assert np.abs(xs.numpy() - g["off_enc_" + tag]).max() < FP32_TOL
    assert np.abs(y.numpy() - g["off_adp_" + tag]).max() < FP32_TOL


def test_tiny_stream_equals_offline_until_saturation(golden, tiny):
    """SURVEY 2.4-1: chunks 0..16 match offline(chunk 4, left 16); later ones drift by the
    one-chunk positional offset of attention.py:112-114."""
    cfg, esd, asd = tiny
    g = golden("tiny")
    pcm = g["stream_pcm"][0].astype(np.float32)
    off_feats = O.fbank(torch.cat([torch.zeros(240), torch.from_numpy(pcm)])).unsqueeze(0)
    off_feats = torch.cat([torch.zeros(1, 3, 80), off_feats], 1)     # the ring starts as zeros
    xs, _ = O.EncoderOracle(cfg, esd).forward(off_feats, torch.tensor([off_feats.size(1)]), 4, 16)
    st = torch.from_numpy(g["stream_enc_out"][:, 0])                 # (24, 4, D)
    n = st.shape[0] * 4
    diff = (xs[0, :n].reshape(-1, 4, cfg.d_model) - st).abs().amax(dim=(1, 2))
    assert float(diff[:17].max()) < 1e-4
    assert float(diff[17:].max()) > 1e-4


@pytest.mark.parametrize("C,L", [(4, 16), (4, 2), (3, 1), (3, 5), (2, 8), (1, 16), (8, 8), (4, 31)])
def test_tiny_stream_equals_offline_until_saturation_other_chunkings(tiny, C, L):
    """The property above at every chunking the streaming GPU tests run, on seeded features: chunk i is the block
    F[4C*i : 4C*i + 4C + 3] (t_in = 4C + 3 gives t = C frames, offline frames [C*i, C*i + C)).  Streaming equals
    forward(C, L) for chunks 0..L, while the cache fills; from chunk L+1 on the rel-pos rows start one chunk behind the
    keys (SURVEY 2.4-1) and every chunk differs."""
    base, esd, _ = tiny
    cfg = dataclasses.replace(base, chunk_size=C, left_chunks=L)
    n_chunks = L + 4
    g = torch.Generator().manual_seed(100 * C + L)
    feats = 9.0 + 3.0 * torch.randn(1, 4 * C * n_chunks + 3, cfg.feat_dim, generator=g)
    enc = O.EncoderOracle(cfg, esd)
    xs, _ = enc.forward(feats, torch.tensor([feats.size(1)]), C, L)
    assert xs.size(1) >= C * n_chunks
    buf, pe = enc.new_buffer(), 0
    diff = []
    for i in range(n_chunks):
        out, buf, pe = enc.infer(feats[:, 4 * C * i:4 * C * i + 4 * C + 3], buf, pe)
        assert out.shape == (1, C, cfg.d_model)
        diff.append(float((out[0] - xs[0, C * i:C * (i + 1)]).abs().max()))
    assert max(diff[:L + 1]) < 1e-4, diff
    assert min(diff[L + 1:]) > 1e-4, diff


# ---- conv1d-linear positionwise variant (Conv1dLinear, attention.py:198-266) -------------------------------------
@pytest.fixture(scope="module")
def tiny_conv1d():
    cfg = load_path_config("tiny_conv1d")
    return cfg, make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)


@pytest.mark.parametrize("c,L", [(4, 16), (-1, -1)])
def test_conv1d_linear_offline(golden, tiny_conv1d, c, L):
    """The reference can only run `forward` for this variant; its outputs pin the oracle's Conv1dLinear."""
    cfg, esd, asd = tiny_conv1d
    g = golden("tiny_conv1d")
    xs, m, y, ym = O.offline_path(cfg, esd, asd, torch.from_numpy(g["off_feats"]), torch.from_numpy(g["off_ilens"]), c, L)
    tag = "c%d_L%d" % (c, L)
    assert np.array_equal(m.numpy(), g["off_mask_" + tag])
    assert np.abs(xs.numpy() - g["off_enc_" + tag]).max() < FP32_TOL
    assert np.abs(y.numpy() - g["off_adp_" + tag]).max() < FP32_TOL


def test_conv1d_linear_stream_equals_offline(golden, tiny_conv1d):
    """Streaming carry of the depthwise conv (last k-1 frames per layer): chunked evaluation must equal `forward`
    on the whole signal until the KV window saturates (then the positional offset of SURVEY 2.4-1 applies)."""
    cfg, esd, asd = tiny_conv1d
    pcm = golden("tiny")["stream_pcm"][0].astype(np.float32)
    off_feats = O.fbank(torch.cat([torch.zeros(240), torch.from_numpy(pcm)])).unsqueeze(0)
    off_feats = torch.cat([torch.zeros(1, 3, 80), off_feats], 1)
    xs, _ = O.EncoderOracle(cfg, esd).forward(off_feats, torch.tensor([off_feats.size(1)]), 4, 16)
    sess = O.StreamSession(cfg, esd, asd)
    outs = []
    for i in range(20):
        _, eo, _ = sess.step_pcm(torch.from_numpy(pcm[i * 2560:(i + 1) * 2560]), 1.0)
        outs.append(eo[0])
    st = torch.stack(outs)
    diff = (xs[0, :80].reshape(-1, 4, cfg.d_model) - st).abs().amax(dim=(1, 2))
    assert float(diff[:17].max()) < 1e-4
    assert sess.buffer[0][2].shape == (1, cfg.d_model, cfg.ffn_conv_kernel - 1)


@pytest.fixture(scope="module")
def shipped():
    cfg = load_path_config("shipped")
    return cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0)


def test_shipped_question_stream(golden, shipped):
    """BASELINE.json config 1: question.wav, 13 chunks, 1 session, fp32 (the golden keeps a seeded sample of the
    feature columns of each output)."""
    cfg, esd, asd = shipped
    g = golden("shipped_question")
    sess = O.StreamSession(cfg, esd, asd)
    pcm = g["pcm"].astype(np.float32) / 32768.0
    for i in range(13):
        feats, eo, y = sess.step_pcm(torch.from_numpy(pcm[i * 2560:(i + 1) * 2560]))
        assert rel_err(feats.numpy(), g["feats"][i]) < 1e-5
        assert np.abs(eo.numpy()[..., g["enc_cols"]] - g["enc_out"][i]).max() < FP32_TOL, i
        assert np.abs(y.numpy()[..., g["adp_cols"]] - g["adapter_out"][i]).max() < FP32_TOL, i
        assert sess.pe_index == int(g["pe_index"][i])
    for li in (0, 23):
        assert np.abs(sess.buffer[li][0].numpy()[..., g["kv_cols"]] - g["k_cache_l%d" % li]).max() < FP32_TOL
    assert np.abs(sess.cache[0].numpy() - g["adapter_cache"]).max() < FP32_TOL


def test_shipped_offline(golden, shipped):
    cfg, esd, asd = shipped
    g = golden("shipped_offline")
    xs, m, y, ym = O.offline_path(cfg, esd, asd, torch.from_numpy(g["feats"]), torch.from_numpy(g["ilens"]), 4, 16)
    assert np.array_equal(m.numpy(), g["mask"]) and np.array_equal(ym.numpy(), g["adapter_mask"])
    assert np.abs(xs.numpy() - g["enc_out"]).max() < FP32_TOL
    assert np.abs(y.numpy() - g["adapter_out"]).max() < FP32_TOL


def test_adapter_batchnorm_relu_vs_reference(golden):
    """CNNSubsampling(norm='batch', activation_func='relu') in eval mode (adapter.py:100-101,106-107): the oracle's folded
    running-statistics BatchNorm against outputs of the reference module (tests/golden/tiny_bn.npz), streaming with the
    conv cache and full-sequence with a ragged pad mask."""
    cfg = load_path_config("tiny_bn")
    asd = make_adapter_state(cfg, 3)
    g = golden("tiny_bn")
    cache = None
    for i in range(g["stream_x"].shape[0]):
        y, _, cache = O.adapter_forward(cfg, asd, torch.from_numpy(g["stream_x"][i]), torch.ones(2, 1, 4, dtype=torch.bool), cache)
        assert float((y - torch.from_numpy(g["stream_y"][i])).abs().max()) < 1e-5, i
    assert float((cache[0] - torch.from_numpy(g["stream_cache"])).abs().max()) == 0.0
    y, m, _ = O.adapter_forward(cfg, asd, torch.from_numpy(g["off_x"]), torch.from_numpy(g["off_mask"]))
    assert float((y - torch.from_numpy(g["off_y"])).abs().max()) < 1e-5
    assert torch.equal(m, torch.from_numpy(g["off_mask_out"]))


def test_linear_adapter_vs_reference(golden):
    """LinearAdapter (adapter.py:59-70, adpter_type 'linear'): oracle against the reference module's output; the mask passes
    through unchanged and the padded frames are NOT zeroed (the reference applies no mask fill here)."""
    cfg = load_path_config("tiny_linear")
    asd = make_adapter_state(cfg, 3)
    g = golden("tiny_linear")
    y, m, cache = O.adapter_forward(cfg, asd, torch.from_numpy(g["x"]), torch.from_numpy(g["mask"]))
    assert cache is None and torch.equal(m, torch.from_numpy(g["mask_out"]))
    assert float((y - torch.from_numpy(g["y"])).abs().max()) < 1e-5


def test_oracle_covers_cnn_adapter_and_two_conv_subsampling(golden):
    """The two adapter variants the GPU path does not build yet (config.validate refuses them): the oracle's restatement is
    already pinned to the reference modules (CNNAdapter adapter.py:10-57; CNNSubsampling two-conv branch :84-96,123-143 with
    its two caches), so the next round starts from a checked checker."""
    import dataclasses
    g = golden("tiny_adapter_variants")
    base = load_path_config("tiny_bn")
    cfg = dataclasses.replace(base, adapter_type="cnn")
    y, m, cache = O.adapter_forward(cfg, make_adapter_state(cfg, 5), torch.from_numpy(g["cnn_x"]), torch.from_numpy(g["cnn_mask"]))
    assert cache is None and float((y - torch.from_numpy(g["cnn_y"])).abs().max()) < 1e-5
    cfg2 = dataclasses.replace(base, llm_dim=int(g["two_llm_dim"]))
    asd = make_adapter_state(cfg2, 5)
    cache = None
    for i in range(g["two_stream_x"].shape[0]):
        y, _, cache = O.adapter_forward(cfg2, asd, torch.from_numpy(g["two_stream_x"][i]), torch.ones(2, 1, 4, dtype=torch.bool), cache)
        assert float((y - torch.from_numpy(g["two_stream_y"][i])).abs().max()) < 1e-5, i
    assert float((cache[0] - torch.from_numpy(g["two_cache0"])).abs().max()) < 1e-6
    assert float((cache[1] - torch.from_numpy(g["two_cache1"])).abs().max()) == 0.0
    y, m, _ = O.adapter_forward(cfg2, asd, torch.from_numpy(g["two_off_x"]), torch.from_numpy(g["two_off_mask"]))
    assert float((y - torch.from_numpy(g["two_off_y"])).abs().max()) < 1e-5
    assert torch.equal(m, torch.from_numpy(g["two_off_mask_out"]))


@pytest.mark.parametrize("name", ["tiny_postnorm_concat", "tiny_concat"])
def test_oracle_layer_variants_match_reference(golden, name):
    """transformer-normalize-before: false (post-norm layers, no after_norm) and transformer-concat-after: true
    (models/encoder/transformer.py:56-70,85-98,108-128,232-233): the oracle against the reference modules' outputs."""
    from freeze_omni_b200.config import load_path_config
    from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
    cfg = load_path_config(name)
    g = golden("tiny_layer_variants")
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    assert ("enc.1.after_norm.weight" in esd) == cfg.normalize_before
    assert ("enc.1.encoders.0.concat_linear.weight" in esd) == cfg.concat_after
    ses = O.StreamSession(cfg, esd, asd)
    for i in range(g[name + "_feats"].shape[0]):
        eo, yo = ses.step_feats(torch.from_numpy(g[name + "_feats"][i]))
        assert float((eo - torch.from_numpy(g[name + "_enc_out"][i])).abs().max()) < 2e-5, i
        assert float((yo - torch.from_numpy(g[name + "_adapter_out"][i])).abs().max()) < 2e-5, i
        assert ses.pe_index == int(g[name + "_pe_index"][i])
    xo, mo = O.EncoderOracle(cfg, esd).forward(torch.from_numpy(g[name + "_off_feats"]), torch.from_numpy(g[name + "_off_ilens"]), 4, 16)
    assert np.array_equal(mo.numpy(), g[name + "_off_mask"])
    assert float((xo - torch.from_numpy(g[name + "_off_enc"])).abs().max()) < 2e-5


def test_oracle_multilayered_conv1d_matches_reference(golden):
    """transformer-positionwise-layer-type: conv1d (MultiLayeredConv1d, attention.py:145-196), full-utterance forward."""
    cfg = load_path_config("tiny_mlconv")
    g = golden("tiny_mlconv")
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    assert tuple(esd["enc.1.encoders.0.feed_forward.w_1.weight"].shape) == (cfg.ffn_dim, cfg.d_model, 3)
    for (c_, L_) in ((4, 16), (-1, -1)):
        xo, mo, yo, _ = O.offline_path(cfg, esd, asd, torch.from_numpy(g["feats"]), torch.from_numpy(g["ilens"]), c_, L_)
        m = torch.from_numpy(g["mask_c%d_L%d" % (c_, L_)])[:, 0, :].unsqueeze(-1).float()
        assert np.array_equal(mo.numpy(), g["mask_c%d_L%d" % (c_, L_)])
        assert float(((xo - torch.from_numpy(g["enc_c%d_L%d" % (c_, L_)])) * m).abs().max()) < 2e-5
