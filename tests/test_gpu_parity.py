"""GPU parity tests proper: the CUDA path, called through the C ABI (freeze_omni_b200.engine / .modules),
against the golden vectors produced by the reference modules and against the CPU oracle on seeded inputs.
Tolerances are the north star's: fbank 1e-5 relative (fp32), encoder/adapter 1e-4 max-abs in fp32 and
2e-2 max-abs in bf16, masks / cache indexing / position bookkeeping bit-exact."""
import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config, load_yaml
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state
from oracle import freeze_omni_oracle as O

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-4
BF16_TOL = 2e-2
FBANK_REL = 1e-5


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b) / np.maximum(np.abs(b), 1.0)


def maxabs(a, b):
    return float(np.abs(np.asarray(a, np.float64) - np.asarray(b, np.float64)).max())


def make_engine(name, seed, dtype=torch.float32, max_sessions=8, **kw):
    from freeze_omni_b200.engine import Engine
    cfg = load_path_config(name)
    return cfg, Engine(cfg, make_encoder_state(cfg, seed), make_adapter_state(cfg, seed), dtype=dtype,
                       max_sessions=max_sessions, **kw)


@pytest.fixture(scope="module")
def tiny32():
    cfg, eng = make_engine("tiny", 3)
    yield cfg, eng
    eng.close()


@pytest.fixture(scope="module")
def shipped32():
    cfg, eng = make_engine("shipped", 0, max_sessions=4)
    yield cfg, eng
    eng.close()


@pytest.fixture(scope="module")
def shipped16():
    cfg, eng = make_engine("shipped", 0, dtype=torch.bfloat16, max_sessions=4)
    yield cfg, eng
    eng.close()


# ------------------------------------------------------------------------------------------------
# frontend
# ------------------------------------------------------------------------------------------------
def exact_fbank(wave_f32, cfg):
    """Exact-arithmetic (fp64) evaluation of the kaldi recipe on the fp32-windowed frames: the yardstick
    for entries where torchaudio's own fp32 FFT is further than 1e-5 from the true value."""
    win, shift = cfg.frame_len, cfg.frame_shift
    m = 1 + (len(wave_f32) - win) // shift
    fr = torch.from_numpy(wave_f32).as_strided((m, win), (shift, 1)).clone()
    fr = fr - fr.mean(dim=1, keepdim=True)
    fr = fr - 0.97 * torch.cat([fr[:, :1], fr[:, :-1]], 1)
    fr = (fr * O.povey_window(win)).numpy().astype(np.float64)
    P = 1 << (win - 1).bit_length()
    power = np.abs(np.fft.rfft(fr, n=P)) ** 2
    mel = O.mel_banks(cfg.feat_dim, P, float(cfg.sample_rate)).numpy().astype(np.float64)
    return np.log(np.maximum((power @ mel.T).astype(np.float32), np.float32(O.FLT_EPSILON)))


def test_fbank_offline(golden, tiny32):
    cfg, eng = tiny32
    g = golden("fbank")
    for name in ("synth", "question"):
        pcm = g[name + "_pcm"]
        if name == "question":
            pcm = np.concatenate([pcm, np.zeros((-len(pcm)) % 2560, np.int16)])
        wave = np.concatenate([np.zeros(240, np.float32), pcm.astype(np.float32)])
        got = eng.fbank_offline(torch.from_numpy(wave).unsqueeze(0), 1.0)[0].cpu().numpy()
        ref = g[name + "_offline"]
        assert got.shape == ref.shape
        exact = exact_fbank(wave, cfg)
        assert rel_err(got, exact).max() < FBANK_REL, name          # vs exact arithmetic: everywhere
        r = rel_err(got, ref)
        trusted = rel_err(ref, exact) < FBANK_REL                   # where torchaudio itself is within 1e-5
        assert trusted.mean() > 0.99
        assert r[trusted].max() < 2 * FBANK_REL, name
        assert r.max() < 5e-4, name
        if name == "synth":
            assert r.max() < FBANK_REL
    # int16 ingest gives the same bits as float ingest of the same samples
    pcm = g["synth_pcm"][:16000]
    a = eng.fbank_offline(torch.from_numpy(pcm.copy()).unsqueeze(0), 1.0)
    b = eng.fbank_offline(torch.from_numpy(pcm.astype(np.float32)).unsqueeze(0), 1.0)
    assert torch.equal(a, b)
    # digital silence hits the log floor exactly (SURVEY appendix A-7)
    z = eng.fbank_offline(torch.zeros(1, 4000), 1.0)
    assert float(z.max()) == float(z.min()) == pytest.approx(-15.942385, abs=1e-5)


def test_fbank_stream_matches_reference_frontend(golden, tiny32):
    cfg, eng = tiny32
    g = golden("tiny")
    ids = eng.alloc(3)
    try:
        pcm = g["stream_pcm"].astype(np.float32) / 32768.0          # what bin/inference.py feeds (x 32768 inside)
        for i in range(6):
            feats = eng.fbank_stream(ids, torch.from_numpy(pcm[:, i * 2560:(i + 1) * 2560].copy()), 32768.0)
            assert rel_err(feats.cpu().numpy(), g["stream_feats"][i]).max() < FBANK_REL, i
        # int16 ingest, different session order, same result for the next chunk
        i = 6
        perm = np.array([2, 0, 1])
        feats = eng.fbank_stream(ids[perm], torch.from_numpy(g["stream_pcm"][perm, i * 2560:(i + 1) * 2560].copy()), 1.0)
        assert rel_err(feats.cpu().numpy(), g["stream_feats"][i][perm]).max() < FBANK_REL
    finally:
        eng.free(ids)


# ------------------------------------------------------------------------------------------------
# tiny config, fp32
# ------------------------------------------------------------------------------------------------
def test_tiny_stream_fp32(golden, tiny32):
    cfg, eng = tiny32
    g = golden("tiny")
    ids = eng.alloc(3)
    try:
        for i in range(24):
            enc, y = eng.encode_stream(ids, torch.from_numpy(g["stream_feats"][i]))
            assert maxabs(enc.cpu(), g["stream_enc_out"][i]) < FP32_TOL, i
            assert maxabs(y.cpu(), g["stream_adapter_out"][i]) < FP32_TOL, i
            for b in range(3):
                nf, pe = eng.state(int(ids[b]))
                assert nf == 4 * (i + 1) and pe == int(g["stream_pe_index"][i])       # bit-exact bookkeeping
        kv = g["kv_cols"]                                          # the golden keeps a sample of the head dimension
        for li in (0, 1):
            k = torch.cat([eng.export_kv(int(s), li)[0] for s in ids])
            v = torch.cat([eng.export_kv(int(s), li)[1] for s in ids])
            assert k.shape == g["stream_k_cache_l%d" % li].shape[:-1] + (cfg.d_k,)
            assert maxabs(k[..., kv], g["stream_k_cache_l%d" % li]) < FP32_TOL
            assert maxabs(v[..., kv], g["stream_v_cache_l%d" % li]) < FP32_TOL
        ac = torch.cat([eng.export_adapter_cache(int(s)) for s in ids])
        assert maxabs(ac, g["stream_adapter_cache"]) < FP32_TOL
    finally:
        eng.free(ids)


def test_tiny_stream_from_pcm_one_call(golden, tiny32):
    cfg, eng = tiny32
    g = golden("tiny")
    ids = eng.alloc(3)
    try:
        for i in range(5):
            enc, y = eng.stream_step(ids, torch.from_numpy(g["stream_pcm"][:, i * 2560:(i + 1) * 2560].copy()), 1.0)
            assert maxabs(enc.cpu(), g["stream_enc_out"][i]) < FP32_TOL, i
            assert maxabs(y.cpu(), g["stream_adapter_out"][i]) < FP32_TOL, i
    finally:
        eng.free(ids)


def test_tiny_stream_seven_frames(golden, tiny32):
    cfg, eng = tiny32
    g = golden("tiny")
    ids = eng.alloc(1)
    try:
        for i in range(12):
            enc, y = eng.encode_stream(ids, torch.from_numpy(g["t7_feats"][i]))
            assert enc.shape[1] == 7
            assert maxabs(enc.cpu(), g["t7_enc_out"][i]) < FP32_TOL, i
            assert maxabs(y.cpu(), g["t7_adapter_out"][i]) < FP32_TOL, i
            assert eng.state(int(ids[0])) == (7 * (i + 1), int(g["t7_pe_index"][i]))
    finally:
        eng.free(ids)


@pytest.mark.parametrize("c,L", [(4, 16), (4, 2), (-1, -1), (4, -1), (3, 1)])
def test_tiny_offline_fp32(golden, tiny32, c, L):
    cfg, eng = tiny32
    g = golden("tiny")
    enc, mask, y, ymask = eng.encode_offline(torch.from_numpy(g["off_feats"]), g["off_ilens"], c, L)
    tag = "c%d_L%d" % (c, L)
    assert np.array_equal(mask.cpu().numpy(), g["off_mask_" + tag])                 # bit-exact masks
    assert np.array_equal(ymask.cpu().numpy(), g["off_amask_" + tag])
    assert maxabs(enc.cpu(), g["off_enc_" + tag]) < FP32_TOL
    assert maxabs(y.cpu(), g["off_adp_" + tag]) < FP32_TOL


def test_tiny_ragged_sessions_vs_oracle(tiny32):
    """Sessions join and leave at different steps and are batched in changing orders (config 3's shape):
    each must equal its own single-session oracle run."""
    cfg, eng = tiny32
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    g = torch.Generator().manual_seed(77)
    n_sess, n_steps = 5, 22
    start = [0, 0, 3, 7, 12]
    length = [22, 9, 19, 15, 10]
    feats = [9.0 + 3.0 * torch.randn(length[s], 19, 80, generator=g) for s in range(n_sess)]
    oracle = [O.StreamSession(cfg, esd, asd) for _ in range(n_sess)]
    ids = {}
    for step in range(n_steps):
        active = [s for s in range(n_sess) if start[s] <= step < start[s] + length[s]]
        if not active:
            continue
        for s in active:
            if s not in ids:
                ids[s] = int(eng.alloc(1)[0])
        order = active[::-1] if step % 2 else active
        batch = torch.stack([feats[s][step - start[s]] for s in order])
        enc, y = eng.encode_stream(np.array([ids[s] for s in order], np.int32), batch)
        for j, s in enumerate(order):
            eo, yo = oracle[s].step_feats(feats[s][step - start[s]].unsqueeze(0))
            assert maxabs(enc[j].cpu(), eo[0]) < FP32_TOL, (step, s)
            assert maxabs(y[j].cpu(), yo[0]) < FP32_TOL, (step, s)
        for s in list(ids):
            if step + 1 == start[s] + length[s]:
                eng.free([ids.pop(s)])
    assert eng.stats()["sessions_in_use"] == 0


def test_tiny_session_reset_and_cache_roundtrip(golden, tiny32):
    cfg, eng = tiny32
    g = golden("tiny")
    a, b = eng.alloc(1), eng.alloc(1)
    try:
        for i in range(20):
            eng.encode_stream(a, torch.from_numpy(g["stream_feats"][i][:1]))
        # export session a in the reference layout, import into b, continue both: identical
        nf, pe = eng.state(int(a[0]))
        eng.set_frames(int(b[0]), nf)
        for li in range(cfg.n_layers):
            k, v = eng.export_kv(int(a[0]), li)
            eng.import_kv(int(b[0]), li, k, v)
        eng.set_pe_index(b, pe)
        eng.import_adapter_cache(int(b[0]), eng.export_adapter_cache(int(a[0])))
        x = torch.from_numpy(g["stream_feats"][20][:1])
        ea, ya = eng.encode_stream(a, x)
        eb, yb = eng.encode_stream(b, x)
        assert torch.equal(ea, eb) and torch.equal(ya, yb)
        assert maxabs(ea.cpu(), g["stream_enc_out"][20][:1]) < FP32_TOL
        # reset == fresh session
        eng.reset(a)
        e0, y0 = eng.encode_stream(a, torch.from_numpy(g["stream_feats"][0][:1]))
        assert maxabs(e0.cpu(), g["stream_enc_out"][0][:1]) < FP32_TOL
        assert maxabs(y0.cpu(), g["stream_adapter_out"][0][:1]) < FP32_TOL
    finally:
        eng.free(a)
        eng.free(b)


def test_tiny_pe_index_wraps(tiny32):
    """pe_index % 4932 bookkeeping (attention.py:107): start a session near the wrap point."""
    cfg, eng = tiny32
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    sess = O.StreamSession(cfg, esd, asd)
    sess.pe_index = cfg.pe_wrap - 8
    ids = eng.alloc(1)
    try:
        eng.set_pe_index(ids, cfg.pe_wrap - 8)
        g = torch.Generator().manual_seed(5)
        for i in range(5):
            x = 9.0 + 3.0 * torch.randn(1, 19, 80, generator=g)
            eo, _ = sess.step_feats(x)
            enc, _ = eng.encode_stream(ids, x)
            assert maxabs(enc.cpu(), eo) < FP32_TOL, i
            assert eng.state(int(ids[0]))[1] == sess.pe_index
    finally:
        eng.free(ids)


def test_dropin_modules_tiny(golden):
    """The nn.Module surface models/audioLLM.py:377-387 drives: infer() with an opaque buffer + adapter with
    an explicit cache list, same state-dict keys."""
    from freeze_omni_b200.modules import CNNSubsampling, GlobalCMVN, speechEncoder
    y = load_yaml("tiny")
    cfg = load_path_config("tiny")
    g = golden("tiny")
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    enc = speechEncoder(80, global_cmvn=GlobalCMVN(esd["global_cmvn.mean"], esd["global_cmvn.istd"]), **y["encoder_conf"])
    enc.load_state_dict(esd, strict=True)
    mc = y["model_conf"]
    adp = CNNSubsampling(mc["enc_out_dim"], mc["llm_embed_dim"], mc["kernel_size"], mc["activation_func"], mc["norm"])
    adp.load_state_dict(asd, strict=True)
    enc, adp = enc.cuda().eval(), adp.cuda().eval()
    buffer, cache, pe = [None] * enc.enc[1].num_blocks, None, 0
    for i in range(19):
        speech = torch.from_numpy(g["stream_feats"][i][:1]).cuda()
        eo, buffer, _, _, pe = enc.infer(speech, buffer, 0, None, pe)
        mask = torch.full(eo.shape[:2], True).unsqueeze(1).to(eo.device)
        emb, mask, cache = adp(eo, mask, cache=cache, return_cache=True)
        assert maxabs(eo.cpu(), g["stream_enc_out"][i][:1]) < FP32_TOL, i
        assert maxabs(emb.cpu(), g["stream_adapter_out"][i][:1]) < FP32_TOL, i
        assert pe == int(g["stream_pe_index"][i])
    assert buffer[0][0].size(2) == cfg.kv_window                   # what transformer.py:277 reads
    # offline forward through the same module
    xs, m = enc(torch.from_numpy(g["off_feats"]).cuda(), torch.from_numpy(g["off_ilens"]), 4, 16)
    assert np.array_equal(m.cpu().numpy(), g["off_mask_c4_L16"])
    assert maxabs(xs.cpu(), g["off_enc_c4_L16"]) < FP32_TOL
    yy, ym = adp(xs, m)
    assert maxabs(yy.cpu(), g["off_adp_c4_L16"]) < FP32_TOL
    assert np.array_equal(ym.cpu().numpy(), g["off_amask_c4_L16"])
    del buffer
    enc.invalidate()
    adp.invalidate()


def test_gemm_simt_vs_torch(tiny32):
    cfg, eng = tiny32
    g = torch.Generator().manual_seed(1)
    for (M, N, K) in ((4, 128, 128), (76, 128, 1152), (300, 384, 256), (130, 256, 640)):
        A = torch.randn(M, K, generator=g).cuda()
        W = torch.randn(N, K, generator=g).cuda() / K ** 0.5
        b = torch.randn(N, generator=g).cuda()
        out, _ = eng.debug_gemm(A, W, b, backend=0, relu=True)
        ref = torch.relu(A.double() @ W.double().T + b.double()).float()
        assert maxabs(out.cpu(), ref.cpu()) < 1e-4, (M, N, K)


# ------------------------------------------------------------------------------------------------
# shipped config
# ------------------------------------------------------------------------------------------------
def test_shipped_question_fp32(golden, shipped32):
    """BASELINE.json config 1 on the GPU path: question.wav, 13 chunks, PCM in.  Against the reference on the seeded
    sample of feature columns the golden keeps, and against the oracle on every column."""
    cfg, eng = shipped32
    g = golden("shipped_question")
    sess = O.StreamSession(cfg, make_encoder_state(cfg, 0), make_adapter_state(cfg, 0))
    ids = eng.alloc(1)
    try:
        pcm = (g["pcm"].astype(np.float32) / 32768.0).reshape(13, 1, 2560)
        for i in range(13):
            enc, y = eng.stream_step(ids, torch.from_numpy(pcm[i]), 32768.0)
            _, eo, yo = sess.step_pcm(torch.from_numpy(pcm[i, 0]), 32768.0)
            assert maxabs(enc.cpu(), eo) < FP32_TOL and maxabs(y.cpu(), yo) < FP32_TOL, i
            assert maxabs(enc.cpu()[..., g["enc_cols"]], g["enc_out"][i]) < FP32_TOL, i
            assert maxabs(y.cpu()[..., g["adp_cols"]], g["adapter_out"][i]) < FP32_TOL, i
            assert eng.state(int(ids[0]))[1] == int(g["pe_index"][i])
        kv = g["kv_cols"]
        for li in (0, 23):
            k, v = eng.export_kv(int(ids[0]), li)
            assert maxabs(k, sess.buffer[li][0]) < FP32_TOL and maxabs(v, sess.buffer[li][1]) < FP32_TOL
            assert maxabs(k[..., kv], g["k_cache_l%d" % li]) < FP32_TOL and maxabs(v[..., kv], g["v_cache_l%d" % li]) < FP32_TOL
        assert maxabs(eng.export_adapter_cache(int(ids[0])), g["adapter_cache"]) < FP32_TOL
    finally:
        eng.free(ids)


def test_shipped_two_sessions_past_saturation_fp32(golden, shipped32):
    """Against the reference on the seeded sample of feature columns the golden keeps, and against the oracle on every
    column."""
    cfg, eng = shipped32
    g = golden("shipped_b2")
    asd = make_adapter_state(cfg, 0)
    orc = O.EncoderOracle(cfg, make_encoder_state(cfg, 0))
    buf, cache, pe = orc.new_buffer(), None, 0
    ids = eng.alloc(2)
    try:
        for i in range(20):
            x = torch.from_numpy(g["feats"][i])
            enc, y = eng.encode_stream(ids, x)
            eo, buf, pe = orc.infer(x, buf, pe)
            yo, _, cache = O.adapter_forward(cfg, asd, eo, torch.ones(2, 1, 4, dtype=torch.bool), cache)
            assert maxabs(enc.cpu(), eo) < FP32_TOL and maxabs(y.cpu(), yo) < FP32_TOL, i
            assert maxabs(enc.cpu()[..., g["enc_cols"]], g["enc_out"][i]) < FP32_TOL, i
            assert maxabs(y.cpu()[..., g["adp_cols"]], g["adapter_out"][i]) < FP32_TOL, i
        k, _ = eng.export_kv(int(ids[1]), 23)
        assert maxabs(k, buf[23][0][1:2]) < FP32_TOL
        assert maxabs(k[..., g["kv_cols"]], g["k_cache_l23"][1:2]) < FP32_TOL
    finally:
        eng.free(ids)


def test_shipped_offline_fp32(golden, shipped32):
    cfg, eng = shipped32
    g = golden("shipped_offline")
    enc, mask, y, ymask = eng.encode_offline(torch.from_numpy(g["feats"]), g["ilens"], 4, 16)
    assert np.array_equal(mask.cpu().numpy(), g["mask"]) and np.array_equal(ymask.cpu().numpy(), g["adapter_mask"])
    assert maxabs(enc.cpu(), g["enc_out"]) < FP32_TOL
    assert maxabs(y.cpu(), g["adapter_out"]) < FP32_TOL


# ---- conv1d-linear positionwise variant (Conv1dLinear, attention.py:198-266; SURVEY 8a row a12) ------------------
@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)])
def test_conv1d_linear_offline(golden, dtype, tol):
    cfg, eng = make_engine("tiny_conv1d", 3, dtype=dtype, max_sessions=4)
    g = golden("tiny_conv1d")
    try:
        for (c, L) in ((4, 16), (-1, -1)):
            enc, mask, y, ymask = eng.encode_offline(torch.from_numpy(g["off_feats"]), g["off_ilens"], c, L)
            tag = "c%d_L%d" % (c, L)
            assert np.array_equal(mask.cpu().numpy(), g["off_mask_" + tag])
            valid = torch.from_numpy(g["off_mask_" + tag]).squeeze(1).unsqueeze(-1)
            assert maxabs((enc.cpu() * valid).numpy(), g["off_enc_" + tag] * valid.numpy()) < tol, tag
    finally:
        eng.close()


def test_conv1d_linear_stream_vs_oracle():
    """Streaming with the per-session, per-layer left context of the depthwise conv: against the oracle's
    StreamSession (whose carry is pinned by chunked == forward in tests/test_oracle_golden.py)."""
    cfg, eng = make_engine("tiny_conv1d", 3, max_sessions=4)
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    g = torch.Generator().manual_seed(41)
    sessions = [O.StreamSession(cfg, esd, asd) for _ in range(3)]
    ids = eng.alloc(3)
    try:
        for i in range(6):
            n = 3 if i != 2 else 2                       # session 2 skips a step: ragged
            pcm = (0.05 * torch.randn(n, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16)
            enc, y = eng.stream_step(ids[:n], pcm, 1.0)
            for b in range(n):
                _, eo, yo = sessions[b].step_pcm(pcm[b].float(), 1.0)
                assert maxabs(enc[b].cpu(), eo[0]) < FP32_TOL and maxabs(y[b].cpu(), yo[0]) < FP32_TOL, (i, b)
        for li in (0, 1):
            assert maxabs(eng.export_ffn_cache(int(ids[1]), li), sessions[1].buffer[li][2]) < FP32_TOL
        eng.reset(ids[:1])
        assert float(eng.export_ffn_cache(int(ids[0]), 0).abs().max()) == 0.0
    finally:
        eng.close()


def _bf16_weights(sd):
    """What a bf16 context computes with: matrices rounded to bf16, vectors (biases, LayerNorm, pos_bias,
    CMVN, first conv) left in fp32 -- the split autocast applies to the reference (SURVEY 2.4-11)."""
    keep = ("pos_bias", "conv.0.weight")
    return {k: (v.bfloat16().float() if v.dim() >= 2 and not any(t in k for t in keep) else v) for k, v in sd.items()}


def test_shipped_stream_bf16(golden, shipped16):
    """bf16 mode.  Two yardsticks: (1) the oracle evaluated in fp32 on the SAME bf16-rounded weights --
    this isolates the implementation from the quantisation of the weights and carries the north-star
    bound of 2e-2; (2) the reference's fp32 outputs, where bf16 weight rounding alone costs 2.5e-2 and
    the reference's own autocast-bf16 run is 0.28 away (tests/golden/shipped_bf16_floor.npz)."""
    cfg, eng = shipped16
    g = golden("shipped_b2")
    floor = golden("shipped_bf16_floor")
    esd, asd = _bf16_weights(make_encoder_state(cfg, 0)), _bf16_weights(make_adapter_state(cfg, 0))
    orc = O.EncoderOracle(cfg, esd)
    buf, cache, pe = orc.new_buffer(), None, 0
    ids = eng.alloc(2)
    we = wy = fe = fy = 0.0
    try:
        for i in range(20):
            x = torch.from_numpy(g["feats"][i])
            enc, y = eng.encode_stream(ids, x)
            eo, buf, pe = orc.infer(x, buf, pe)
            yo, _, cache = O.adapter_forward(cfg, asd, eo, torch.ones(2, 1, 4, dtype=torch.bool), cache)
            we, wy = max(we, maxabs(enc.cpu(), eo)), max(wy, maxabs(y.cpu(), yo))
            fe = max(fe, maxabs(enc.cpu()[..., g["enc_cols"]], g["enc_out"][i]))
            fy = max(fy, maxabs(y.cpu()[..., g["adp_cols"]], g["adapter_out"][i]))
        print("bf16 max-abs vs oracle on bf16 weights: encoder %.4g adapter %.4g; vs fp32 reference: %.4g / %.4g "
              "(reference autocast floor %.4g / %.4g)" % (we, wy, fe, fy, float(floor["ref_autocast_vs_fp32_encoder"]),
                                                          float(floor["ref_autocast_vs_fp32_adapter"])))
        assert we < BF16_TOL and wy < BF16_TOL
        assert fe < float(floor["ref_autocast_vs_fp32_encoder"]) and fy < float(floor["ref_autocast_vs_fp32_adapter"])
    finally:
        eng.free(ids)


def test_shipped_offline_bf16(golden, shipped16):
    cfg, eng = shipped16
    g = golden("shipped_offline")
    floor = golden("shipped_bf16_floor")
    enc, mask, y, ymask = eng.encode_offline(torch.from_numpy(g["feats"]), g["ilens"], 4, 16)
    assert np.array_equal(mask.cpu().numpy(), g["mask"])
    esd, asd = _bf16_weights(make_encoder_state(cfg, 0)), _bf16_weights(make_adapter_state(cfg, 0))
    xo, mo, yo, _ = O.offline_path(cfg, esd, asd, torch.from_numpy(g["feats"]), torch.from_numpy(g["ilens"]), 4, 16)
    print("bf16 offline max-abs vs oracle on bf16 weights: encoder %.4g adapter %.4g; vs fp32 reference %.4g / %.4g"
          % (maxabs(enc.cpu(), xo), maxabs(y.cpu(), yo), maxabs(enc.cpu(), g["enc_out"]), maxabs(y.cpu(), g["adapter_out"])))
    assert maxabs(enc.cpu(), xo) < BF16_TOL and maxabs(y.cpu(), yo) < BF16_TOL
    assert maxabs(enc.cpu(), g["enc_out"]) < float(floor["ref_autocast_vs_fp32_encoder"])


@pytest.mark.parametrize("which", ["tiny32", "shipped16"])
def test_graph_replay_matches_eager(which, request):
    """The captured CUDA graph of a step must be bit-identical to the eager launch sequence, across the
    first (eager), second (capture) and later (replay) calls of a shape."""
    cfg, eng = request.getfixturevalue(which)
    g = torch.Generator().manual_seed(11)
    ids = eng.alloc(2)
    try:
        r0 = eng.stats()["graph_replays"]
        for i in range(6):
            pcm = (0.05 * torch.randn(1, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16)
            eng.set_option("use_graph", 1)
            e1, y1 = eng.stream_step(ids[:1], pcm, 1.0)
            eng.set_option("use_graph", 0)
            e0, y0 = eng.stream_step(ids[1:], pcm, 1.0)
            assert torch.equal(e1, e0) and torch.equal(y1, y0), i
        assert eng.stats()["graph_replays"] - r0 >= 4
        assert eng.state(int(ids[0])) == eng.state(int(ids[1]))
    finally:
        eng.set_option("use_graph", 1)
        eng.free(ids)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_session_groups_match_single_group(dtype):
    """Layer kernels of different session groups run on parallel streams; the result must not depend on the
    grouping (bit-identical in fp32, where the GEMM summation order does not depend on the row count)."""
    cfg, eng = make_engine("tiny", 3, dtype=dtype, max_sessions=48)
    g = torch.Generator().manual_seed(21)
    try:
        ids_a, ids_b = eng.alloc(24), eng.alloc(24)
        for i in range(4):
            pcm = (0.05 * torch.randn(24, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16)
            eng.set_option("session_groups", 1)
            e1, y1 = eng.stream_step(ids_a, pcm, 1.0)
            eng.set_option("session_groups", 3)
            e3, y3 = eng.stream_step(ids_b, pcm, 1.0)
            if dtype == torch.float32:
                assert torch.equal(e1, e3) and torch.equal(y1, y3), i
            else:
                assert maxabs(e1.cpu(), e3.cpu()) < 1e-3 and maxabs(y1.cpu(), y3.cpu()) < 1e-3, i
        assert eng.state(int(ids_a[5])) == eng.state(int(ids_b[5]))
    finally:
        eng.close()


def test_fused_layernorm_matches_standalone(shipped16):
    """LayerNorm fused into the epilogue of the GEMM that completes the residual rows (last-arriving CTA of a row
    block) against the default path (split-K reduction deferred to a LayerNorm that reduces a row with two warps): the
    residual stream is bit-identical by construction (same association of the split-K sum), the row statistics are summed
    in a different order -> agreement to fp32 rounding of the normalised rows."""
    cfg, eng = shipped16
    g = torch.Generator().manual_seed(31)
    ids = eng.alloc(2)
    try:
        for i in range(3):
            pcm = (0.05 * torch.randn(1, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16)
            eng.set_option("fuse_ln", 1)
            e1, y1 = eng.stream_step(ids[:1], pcm, 1.0)
            eng.set_option("fuse_ln", 0)
            e0, y0 = eng.stream_step(ids[1:], pcm, 1.0)
            assert maxabs(e1.cpu(), e0.cpu()) < 2e-3 and maxabs(y1.cpu(), y0.cpu()) < 2e-3, i   # fp16 re-rounding of h over 24 layers
    finally:
        eng.set_option("fuse_ln", 0)
        eng.free(ids)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)])
def test_adapter_batchnorm_relu(golden, dtype, tol):
    """Adapter variant norm='batch' + ReLU (adapter.py:100-101,106-107; BatchNorm1d eval = per-channel affine of the running
    statistics, folded at fo_finalize_weights) against the reference module's outputs: streaming with the conv cache passed
    in and out, and a full sequence with a ragged pad mask."""
    from freeze_omni_b200.engine import Engine
    cfg = load_path_config("tiny_bn")
    asd = make_adapter_state(cfg, 3)
    eng = Engine(cfg, None, asd, dtype=dtype, max_sessions=1)
    g = golden("tiny_bn")
    try:
        cache = None
        for i in range(g["stream_x"].shape[0]):
            y, cache = eng.adapter_forward(torch.from_numpy(g["stream_x"][i]).cuda(), None, cache)
            assert maxabs(y.cpu(), g["stream_y"][i]) < tol, i
        assert maxabs(cache.cpu(), g["stream_cache"]) < 1e-6
        y, _ = eng.adapter_forward(torch.from_numpy(g["off_x"]).cuda(), torch.from_numpy(g["off_mask"]).cuda(), None)
        assert maxabs(y.cpu(), g["off_y"]) < tol
    finally:
        eng.close()


@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)])
def test_linear_adapter(golden, dtype, tol):
    """adpter_type 'linear' (LinearAdapter, adapter.py:59-70): stateless call against the reference module's output, then
    the whole streaming path (t_out == t, no adapter cache) against per-session oracle runs."""
    cfg, eng = make_engine("tiny_linear", 3, dtype=dtype, max_sessions=4)
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    g = golden("tiny_linear")
    try:
        y, cache = eng.adapter_forward(torch.from_numpy(g["x"]).cuda(), torch.from_numpy(g["mask"]).cuda(), None)
        assert cache is None and maxabs(y.cpu(), g["y"]) < tol
        gen = torch.Generator().manual_seed(59)
        sessions = [O.StreamSession(cfg, esd, asd) for _ in range(2)]
        ids = eng.alloc(2)
        for i in range(4):
            pcm = (0.05 * torch.randn(2, cfg.samples_per_chunk, generator=gen) * 32768).round().to(torch.int16)
            enc, emb = eng.stream_step(ids, pcm, 1.0)
            assert emb.shape[1] == enc.shape[1] == 4
            for b in range(2):
                _, eo, yo = sessions[b].step_pcm(pcm[b].float(), 1.0)
                assert maxabs(enc[b].cpu(), eo[0]) < tol * (1 if dtype == torch.float32 else 4) and maxabs(emb[b].cpu(), yo[0]) < tol * (1 if dtype == torch.float32 else 4), (i, b)
    finally:
        eng.close()


def test_persistent_gemm_matches_tile_per_cta(shipped16):
    """Fat short-K GEMMs run on the persistent tcgen05 kernel (tile loop per SM, double-buffered TMEM accumulator,
    epilogue straight from TMEM registers).  Same k order and same fp32 epilogue arithmetic as the one-tile-per-CTA
    kernel -> bit-identical outputs: plain GEMMs against an fp64 product, and a whole offline pass (bias, ReLU,
    residual, fp32|fp16 split of the QKV output, ragged lengths) with the option off and on."""
    cfg, eng = shipped16
    g = torch.Generator().manual_seed(71)
    try:
        for (M, N, K) in [(5000, 4096, 1024), (4100, 3584, 2048), (12000, 1024, 4096)]:
            A = torch.randn(M, K, generator=g).cuda()
            W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
            b = torch.randn(N, generator=g).cuda()
            ref = (A.half().double() @ W.bfloat16().double().T + b.double()).float().cpu()
            eng.set_option("tc_persist", 1)
            n0 = eng.get_option("tc_persist_launches")
            o1, _ = eng.debug_gemm(A, W, b, backend=1)
            assert eng.get_option("tc_persist_launches") == n0 + 1, "persistent kernel did not launch"
            eng.set_option("tc_persist", 0)
            o0, _ = eng.debug_gemm(A, W, b, backend=1)
            assert eng.get_option("tc_persist_launches") == n0 + 1
            assert maxabs(o1.cpu(), ref) < 2e-3, (M, N, K)
            assert torch.equal(o1, o0), (M, N, K)
        B, T = 5, 2998
        feats = 9.0 + 3.0 * torch.randn(B, T, cfg.feat_dim, generator=g)
        ilens = torch.tensor([2998, 2500, 2998, 1203, 2998])
        eng.set_option("tc_persist", 1)
        n0 = eng.get_option("tc_persist_launches")
        e1, m1, y1, _ = eng.encode_offline(feats.cuda(), ilens, 4, 16)
        assert eng.get_option("tc_persist_launches") > n0
        eng.set_option("tc_persist", 0)
        e0, m0, y0, _ = eng.encode_offline(feats.cuda(), ilens, 4, 16)
        assert torch.equal(m1, m0) and torch.equal(e1, e0) and torch.equal(y1, y0)
    finally:
        eng.set_option("tc_persist", 1)


def test_async_pipelined_step_matches_sync(shipped16):
    """fo_stream_step_async / fo_stream_wait (copies on the library's copy stream, double-buffered staging) must deliver the
    bits of the synchronous call, step after step, with two steps in flight."""
    cfg, eng = shipped16
    g = torch.Generator().manual_seed(83)
    ids = eng.alloc(4)
    t, t_out = eng.out_frames(cfg.chunk_feat_frames)
    try:
        pcm = [(0.05 * torch.randn(2, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16).pin_memory() for _ in range(7)]
        ref = [eng.stream_step(ids[:2], p, 1.0) for p in pcm]
        ref = [(e.cpu(), y.cpu()) for e, y in ref]
        ys = [torch.empty(2, t_out, cfg.llm_dim).pin_memory() for _ in range(7)]
        es = [torch.empty(2, t, cfg.d_model).pin_memory() for _ in range(7)]
        prev = None
        for i in range(7):
            tk = eng.stream_step_async(ids[2:], pcm[i], ys[i], 1.0, enc_out=es[i])
            if prev is not None:
                eng.stream_wait(prev)
                assert torch.equal(ys[i - 1], ref[i - 1][1]) and torch.equal(es[i - 1], ref[i - 1][0]), i - 1
            prev = tk
        eng.stream_wait(prev)
        assert torch.equal(ys[6], ref[6][1]) and torch.equal(es[6], ref[6][0])
        with pytest.raises(Exception):
            eng.stream_wait(prev - 3)                                   # older than the two steps in flight
        # a synchronous call right behind pipelined ones (same staging buffers) without waiting for the last ticket
        tk = eng.stream_step_async(ids[2:], pcm[0], ys[0], 1.0, enc_out=es[0])
        e_s, y_s = eng.stream_step(ids[2:], pcm[1], 1.0)
        eng.stream_wait(tk)
        e_a = eng.stream_step(ids[:2], pcm[0], 1.0)
        e_b, y_b = eng.stream_step(ids[:2], pcm[1], 1.0)
        assert torch.equal(ys[0], e_a[1].cpu()) and torch.equal(y_s, y_b) and torch.equal(e_s, e_b)
        assert eng.state(int(ids[0])) == eng.state(int(ids[2]))
    finally:
        eng.free(ids)


def test_llm_handoff_fp16_embeds(shipped16):
    """fo_stream_step_embeds writes the adapter rows as fp16 straight into the caller's inputs_embeds block behind the
    chat prefix (audioLLM.py:404-411: cat(prefix, embeds).half()): same bits as .half() of the fp32 output, prefix and
    the rows behind untouched, adapter cache advanced as usual."""
    cfg, eng = shipped16
    g = torch.Generator().manual_seed(61)
    ids = eng.alloc(4)
    P, R = 5, 9                                                   # 5 prefix rows, 2 adapter rows, 2 spare rows
    try:
        buf = torch.full((2, R, cfg.llm_dim), 7.0, dtype=torch.float16, device="cuda")
        for i in range(4):
            pcm = (0.05 * torch.randn(2, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16)
            e0, y0 = eng.stream_step(ids[:2], pcm, 1.0)
            e1, _ = eng.stream_step_embeds(ids[2:], pcm, buf, row_offset=P, scale=1.0, want_enc=True)
            assert torch.equal(e0, e1), i
            assert torch.equal(buf[:, P:P + 2], y0.half()), i
            assert bool((buf[:, :P] == 7.0).all()) and bool((buf[:, P + 2:] == 7.0).all())
        with pytest.raises(Exception):
            eng.stream_step_embeds(ids[2:], pcm, buf, row_offset=R - 1, scale=1.0)      # rows would not fit
    finally:
        eng.free(ids)


def test_scheduler_vad_gating_vs_oracle():
    """Batched scheduler + VAD-gated frontend (freeze_omni_b200/scheduler.py) against per-session oracle runs that
    restate the reference flow: features always extracted (AudioFeatureGating.py:92-93), silent blocks only enter the
    10-deep history ring (:96-99), speech onset replays the last 6 history blocks before the current one
    (:109-112, dialog_state_pred.py:639-670), every queued block is one encoder + adapter step (:793-814)."""
    from freeze_omni_b200.scheduler import StreamScheduler
    cfg, eng = make_engine("tiny", 3, max_sessions=24)
    esd, asd = make_encoder_state(cfg, 3), make_adapter_state(cfg, 3)
    g = torch.Generator().manual_seed(53)
    S, T = 4, 16
    pattern = [
        ["ipu_cl"] * T,                                                                   # always speaking
        [None] * 8 + ["ipu_sl"] + ["ipu_cl"] * 3 + [None] * 2 + ["ipu_sl", "ipu_cl"],     # two onsets, full history at the first
        [None] * 3 + ["ipu_sl"] + ["ipu_cl"] * 12,                                        # onset before the history ring is full
        [None] * T,                                                                       # never speaks
    ]
    try:
        sch = StreamScheduler(eng, history_chunks=10, onset_chunks=6, bucket=4, max_sessions=8)
        oracle = [O.StreamSession(cfg, esd, asd) for _ in range(S)]
        hist = [torch.zeros(10, cfg.chunk_feat_frames, cfg.feat_dim) for _ in range(S)]
        for s in range(S):
            sch.open(s)
        expected_steps = 0
        for tck in range(T):
            pcm = (0.05 * torch.randn(S, cfg.samples_per_chunk, generator=g) * 32768).round().to(torch.int16)
            active = [s for s in range(S) if not (s == 0 and tck % 5 == 4)]              # session 0 misses some ticks
            for s in active:
                sch.push(s, pcm[s], pattern[s][tck])
            out = sch.tick(1.0)
            for s in active:
                feats = oracle[s].front.process(pcm[s].float(), 1.0)                      # (1, 19, 80)
                status = pattern[s][tck]
                if status is None:
                    hist[s] = torch.cat([hist[s][1:], feats])
                    assert s not in out
                    continue
                blocks = list(hist[s][-6:].unsqueeze(1)) + [feats] if status == "ipu_sl" else [feats]
                assert len(out[s]) == len(blocks), (tck, s)
                expected_steps += len(blocks)
                want_lab = ["ipu_sl"] + ["ipu_cl"] * 6 if status == "ipu_sl" else [status]
                assert [b.status for b in out[s]] == want_lab
                for ob, blk in zip(out[s], blocks):
                    enc, emb = ob.enc, ob.emb
                    eo, yo = oracle[s].step_feats(blk)
                    assert maxabs(enc.cpu(), eo[0]) < FP32_TOL and maxabs(emb.cpu(), yo[0]) < FP32_TOL, (tck, s)
            assert maxabs(sch.history(1).cpu(), hist[1]) < 1e-4 * 20
        st = sch.stats
        assert st["fbank_calls"] == T and st["session_steps"] == expected_steps
        assert st["encode_calls"] < st["session_steps"]                                   # steps were batched
        for s in range(S):
            assert eng.state(sch.keys[s])[1] == oracle[s].pe_index
    finally:
        eng.close()


def test_tcgen05_gemm_tile_plans(shipped16):
    """Every orientation / UMMA-N / split-K plan of the tcgen05 kernel against an fp64 product of the
    same bf16 operands; checks the kernel really launched (no silent FFMA fallback)."""
    cfg, eng = shipped16
    g = torch.Generator().manual_seed(5)
    plans = [(0, 256, 1), (0, 128, 1), (0, 64, 2), (0, 16, 1), (0, 208, 4), (1, 256, 1), (1, 144, 2), (1, 64, 1),
             (1, 16, 4), (1, 32, 8), (-1, -1, -1)]
    shapes = [(256, 1024, 1024), (76, 1024, 9216), (4, 3072, 1024), (300, 3584, 2048), (1000, 1024, 4096), (128, 2048, 5120)]
    try:
        for (M, N, K) in shapes:
            A = torch.randn(M, K, generator=g).cuda()
            W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
            b = torch.randn(N, generator=g).cuda()
            ref = (A.half().double() @ W.bfloat16().double().T + b.double()).float().cpu()   # fp16 activations x bf16 weights
            for (swap, bn, split) in plans:
                eng.set_option("tc_swap", swap)
                eng.set_option("tc_bn", bn)
                eng.set_option("tc_split", split)
                n0 = eng.get_option("tc_launches")
                o, _ = eng.debug_gemm(A, W, b, backend=1)
                assert eng.get_option("tc_launches") == n0 + 1, "tcgen05 kernel did not launch"
                err = maxabs(o.cpu(), ref)
                assert err < 2e-3, ((M, N, K), (swap, bn, split), err)
    finally:
        eng.set_option("tc_swap", -1)
        eng.set_option("tc_bn", -1)
        eng.set_option("tc_split", -1)


def test_gemm_backends_agree_bf16(shipped16):
    """tcgen05 kernel vs the FFMA kernel on the same bf16 operands (both accumulate in fp32)."""
    cfg, eng = shipped16
    g = torch.Generator().manual_seed(2)
    for (M, N, K) in ((256, 1024, 1024), (256, 4096, 1024), (256, 1024, 4096), (128, 3584, 2048), (100, 3072, 1024),
                      (4, 1024, 1024), (1000, 1024, 1024)):
        A = torch.randn(M, K, generator=g).cuda()
        W = (torch.randn(N, K, generator=g) / K ** 0.5).cuda()
        b = torch.randn(N, generator=g).cuda()
        o0, _ = eng.debug_gemm(A, W, b, backend=0)
        o1, _ = eng.debug_gemm(A, W, b, backend=1)
        ref = (A.half().double() @ W.bfloat16().double().T + b.double()).float()
        assert maxabs(o0.cpu(), ref.cpu()) < 2e-3, (M, N, K)
        assert maxabs(o1.cpu(), ref.cpu()) < 2e-3, (M, N, K)


# ------------------------------------------------------------------------------------------------
# weight-streaming layer stack (csrc/fo_stack.cu): all layers of a step of <= 16 token rows in one cooperative launch
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2])
def test_stack_kernel_matches_chain_shipped(shipped16, n):
    """Same PCM through two groups of sessions, one per execution form (option stack_rows): the persistent stack kernel
    against the per-kernel chain over 22 chunks (past the 17-chunk ring saturation).  Both multiply fp16-staged
    activations with the same bf16-rounded weights; only the order of summation inside a dot product differs."""
    cfg, eng = shipped16
    g = torch.Generator().manual_seed(41)
    ia, ib = eng.alloc(n), eng.alloc(n)
    try:
        l0 = eng.get_option("stack_launches")
        for i in range(22):
            pcm = (0.05 * torch.randn(n, cfg.samples_per_chunk, generator=g) * 32768).round().clamp(-32768, 32767).to(torch.int16)
            eng.set_option("stack_rows", 16)
            e1, y1 = eng.stream_step(ia, pcm, 1.0)
            eng.set_option("stack_rows", 0)
            e0, y0 = eng.stream_step(ib, pcm, 1.0)
            assert torch.isfinite(e1).all() and torch.isfinite(y1).all(), i
            assert maxabs(e1.cpu(), e0.cpu()) < 2e-3 and maxabs(y1.cpu(), y0.cpu()) < 2e-3, i
        assert eng.get_option("stack_launches") - l0 == 22
        assert eng.state(int(ia[0])) == eng.state(int(ib[0]))
        assert eng.stats()["act_saturations"] == 0
    finally:
        eng.set_option("stack_rows", 8)
        eng.free(ia)
        eng.free(ib)


def test_stack_kernel_vs_oracle_one_session(shipped16):
    """One session (the latency configuration, BASELINE config 5) through the stack kernel against the oracle on the same
    bf16-rounded weights, 20 chunks of PCM through fo_stream_step; bar 2e-2."""
    cfg, eng = shipped16
    esd, asd = _bf16_weights(make_encoder_state(cfg, 0)), _bf16_weights(make_adapter_state(cfg, 0))
    ses = O.StreamSession(cfg, esd, asd)
    g = torch.Generator().manual_seed(43)
    ids = eng.alloc(1)
    we = wy = 0.0
    try:
        l0 = eng.get_option("stack_launches")
        for i in range(20):
            pcm = (0.05 * torch.randn(1, cfg.samples_per_chunk, generator=g) * 32768).round().clamp(-32768, 32767).to(torch.int16)
            enc, y = eng.stream_step(ids, pcm, 1.0)
            _, eo, yo = ses.step_pcm(pcm[0].float(), 1.0)
            we, wy = max(we, maxabs(enc[0].cpu(), eo[0])), max(wy, maxabs(y[0].cpu(), yo[0]))
        print("stack kernel, 1 session x 20 chunks, max-abs vs oracle on bf16 weights: encoder %.4g adapter %.4g" % (we, wy))
        assert eng.get_option("stack_launches") - l0 == 20, "the one-session step must run the stack kernel"
        assert we < BF16_TOL and wy < BF16_TOL
    finally:
        eng.free(ids)


def test_stack_kernel_tiny_rows_and_frames(golden):
    """Toy widths (D = 128, FF = 256, 2 heads: CTAs with zero, one or two weight rows per phase), 12 and 16 token rows
    (two activation rows per warp pair, FFN2 activations in K chunks) and 7 encoder frames per call (fork frontend)."""
    cfg, eng = make_engine("tiny", 3, dtype=torch.bfloat16, max_sessions=16)
    g = torch.Generator().manual_seed(47)
    try:
        for n in (3, 4):
            ia, ib = eng.alloc(n), eng.alloc(n)
            l0 = eng.get_option("stack_launches")
            for i in range(20):
                pcm = (0.05 * torch.randn(n, cfg.samples_per_chunk, generator=g) * 32768).round().clamp(-32768, 32767).to(torch.int16)
                eng.set_option("stack_rows", 16)
                e1, y1 = eng.stream_step(ia, pcm, 1.0)
                eng.set_option("stack_rows", 0)
                e0, y0 = eng.stream_step(ib, pcm, 1.0)
                assert maxabs(e1.cpu(), e0.cpu()) < 2e-3 and maxabs(y1.cpu(), y0.cpu()) < 2e-3, (n, i)
            assert eng.get_option("stack_launches") - l0 == 20
            eng.free(ia)
            eng.free(ib)
        golden7 = golden("tiny")
        ia, ib = eng.alloc(2), eng.alloc(2)
        l0 = eng.get_option("stack_launches")
        for i in range(12):
            x = torch.from_numpy(golden7["t7_feats"][i]).repeat(2, 1, 1)
            eng.set_option("stack_rows", 16)
            e1, y1 = eng.encode_stream(ia, x)
            eng.set_option("stack_rows", 0)
            e0, y0 = eng.encode_stream(ib, x)
            assert e1.shape[1] == 7
            assert maxabs(e1.cpu(), e0.cpu()) < 2e-3 and maxabs(y1.cpu(), y0.cpu()) < 2e-3, i
        assert eng.get_option("stack_launches") - l0 == 12
        assert eng.state(int(ia[1])) == eng.state(int(ib[1]))
    finally:
        eng.close()
