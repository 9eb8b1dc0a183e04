#!/usr/bin/env python
"""Generate tests/golden/*.npz by EXECUTING THE REFERENCE MODULES (authoring container only).

Run:  PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py [--ref /root/reference]

The reference (TheDoctor-JI/Freeze-Omni) ships no tests or golden vectors (SURVEY 4), so the
pins for the oracle and the CUDA path are the outputs of its own modules
(models.encoder.encoder.speechEncoder, models.encoder.cmvn.GlobalCMVN, models.adapter.CNNSubsampling,
models.AudioFeatureGating, models.masks) imported unmodified from /root/reference, with the
harness shims of SURVEY 8c:
  1. models.encoder.encoder.make_pad_mask is injected (encoder.py:142 calls an un-imported name);
  2. Tensor.to('cuda') is mapped to a no-op on this GPU-less host (transformer.py:279);
  3. sys.argv is cleared before construction (encoder.py:54-56 parses the process argv).
Weights are the seeded state dict of freeze_omni_b200/weights.py loaded with strict=True.
Nothing in the test suite imports this file: it needs a checkout of the reference.

Every stored file stays under 1 MB.  Inputs that are a function of a seed (synthetic audio, random features) are not
stored: tests/conftest.py rebuilds them with the same seeds.  The streaming fbank features of those streams are stored
only as the SHA-256 of the reference's values, which the features rebuilt from the audio must match bit for bit.  The
widest outputs keep a seeded sample of their last axis, with the sampled indices stored as <name>_cols.
"""
import argparse
import hashlib
import os
import sys
import wave

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

from conftest import synth_audio  # noqa: E402
from freeze_omni_b200.config import load_yaml, path_config_from_dict  # noqa: E402
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state  # noqa: E402


def feats_digest(feats):
    return np.array(hashlib.sha256(np.ascontiguousarray(feats, np.float32).tobytes()).hexdigest())


def sample_last_axis(arrs, name, n, keys):
    """Keep the same seeded n indices of the last axis of every array in keys; store them as <name>_cols."""
    cols = np.sort(np.random.RandomState(0).choice(arrs[keys[0]].shape[-1], n, replace=False))
    arrs[name + "_cols"] = cols
    for k in keys:
        arrs[k] = arrs[k][..., cols]


def import_reference(ref_root):
    sys.path.insert(0, ref_root)
    sys.dont_write_bytecode = True
    saved_argv = sys.argv
    sys.argv = ["x"]
    import models.encoder.encoder as ref_encoder
    import models.encoder.cmvn as ref_cmvn
    import models.adapter as ref_adapter
    import models.masks as ref_masks
    import models.AudioFeatureGating as ref_gating
    ref_encoder.make_pad_mask = lambda lengths, max_len: (
        torch.arange(max_len).unsqueeze(0) >= lengths.reshape(-1, 1))
    orig_to = torch.Tensor.to

    def to_shim(self, *a, **k):
        if a and isinstance(a[0], str) and a[0].startswith("cuda") and not torch.cuda.is_available():
            return self
        return orig_to(self, *a, **k)
    torch.Tensor.to = to_shim
    sys.argv = saved_argv
    return ref_encoder, ref_cmvn, ref_adapter, ref_masks, ref_gating


def build_reference(mods, yaml_cfg, cfg, seed):
    ref_encoder, ref_cmvn, ref_adapter, _, _ = mods
    enc_sd = make_encoder_state(cfg, seed)
    adp_sd = make_adapter_state(cfg, seed)
    argv = sys.argv
    sys.argv = ["x"]
    cm = ref_cmvn.GlobalCMVN(enc_sd["global_cmvn.mean"].clone(), enc_sd["global_cmvn.istd"].clone())
    enc = ref_encoder.speechEncoder(cfg.feat_dim, global_cmvn=cm, **yaml_cfg["encoder_conf"])
    sys.argv = argv
    enc.load_state_dict(enc_sd, strict=True)
    mc = yaml_cfg["model_conf"]
    adp = ref_adapter.CNNSubsampling(mc["enc_out_dim"], mc["llm_embed_dim"], mc["kernel_size"],
                                     mc["activation_func"], mc["norm"])
    adp.load_state_dict(adp_sd, strict=True)
    return enc.eval(), adp.eval()


def stream_reference(enc, adp, feats_seq, layers_to_keep=(0,)):
    """AudioLLM.recognize's encoder/adapter calls (audioLLM.py:377-387), chunk by chunk."""
    buffer, cache, pe = [None] * enc.enc[1].num_blocks, None, 0
    enc_outs, adp_outs, pes = [], [], []
    with torch.no_grad():
        for feats in feats_seq:
            eo, buffer, _, _, pe = enc.infer(feats, buffer, 0, None, pe)
            enc_outs.append(eo.clone())      # the adapter zero-fills through a view of eo
            mask = torch.full(eo.shape[:2], True).unsqueeze(1)
            y, _, cache = adp(eo, mask, cache=cache, return_cache=True)
            adp_outs.append(y.clone())
            pes.append(pe)
    out = {"enc_out": torch.stack(enc_outs).numpy(), "adapter_out": torch.stack(adp_outs).numpy(),
           "pe_index": np.asarray(pes, dtype=np.int64), "adapter_cache": cache[0].contiguous().numpy()}
    for li in layers_to_keep:
        out["k_cache_l%d" % li] = buffer[li][0].contiguous().numpy()
        out["v_cache_l%d" % li] = buffer[li][1].contiguous().numpy()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", default="/root/reference")
    ap.add_argument("--only", default="")
    args = ap.parse_args()
    mods = import_reference(args.ref)
    ref_encoder, ref_cmvn, ref_adapter, ref_masks, ref_gating = mods
    import torchaudio.compliance.kaldi as kaldi
    torch.manual_seed(0)
    torch.set_num_threads(8)

    def want(name):
        return not args.only or name in args.only.split(",")

    def save(name, **arrs):
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **arrs)
        print("wrote", path, "%.1f KB" % (os.path.getsize(path) / 1024))

    with wave.open(os.path.join(args.ref, "assets", "question.wav"), "rb") as w:
        assert w.getframerate() == 16000 and w.getnchannels() == 1 and w.getsampwidth() == 2
        pcm = np.frombuffer(w.readframes(w.getnframes()), dtype=np.int16).copy()
    n_chunks = -(-len(pcm) // 2560)
    pcm_pad = np.zeros(n_chunks * 2560, dtype=np.int16)
    pcm_pad[:len(pcm)] = pcm

    # ---------------- cmvn statistics files (models/encoder/cmvn.py:37-107) -------------------
    if want("cmvn"):
        import json
        import tempfile
        rs = np.random.RandomState(11)
        d, count = 80, 123457.0
        x_mean = rs.uniform(-3, 12, d)
        x_std = rs.uniform(0.5, 4, d)
        x_std[7] = 0.0                                       # degenerate channel -> variance floor 1e-20
        sums = (x_mean * count).tolist()
        sqs = ((x_std ** 2 + x_mean ** 2) * count).tolist()
        js = json.dumps({"mean_stat": sums, "var_stat": sqs, "frame_num": count})
        kaldi_txt = " [\n  " + " ".join(repr(v) for v in sums) + " " + repr(count) + "\n  " + \
            " ".join(repr(v) for v in sqs) + " 0 ]\n"
        with tempfile.TemporaryDirectory() as td:
            pj, pk = os.path.join(td, "c.json"), os.path.join(td, "c.txt")
            open(pj, "w").write(js)
            open(pk, "w").write(kaldi_txt)
            mj, ij = ref_cmvn.load_cmvn(pj, True)
            mk, ik = ref_cmvn.load_cmvn(pk, False)
        save("cmvn", json_text=np.frombuffer(js.encode(), np.uint8), kaldi_text=np.frombuffer(kaldi_txt.encode(), np.uint8),
             json_mean=mj, json_istd=ij, kaldi_mean=mk, kaldi_istd=ik)

    # ---------------- fbank ----------------------------------------------------------------
    def gating_stream(int16_pcm, fbank_config, chunk):
        g = ref_gating.AudioFeatureGating(16000, fbank_config=fbank_config)
        outs = []
        for i in range(len(int16_pcm) // chunk):
            a = int16_pcm[i * chunk:(i + 1) * chunk].astype(np.float32) / 32768.0
            outs.append(g._extract_fbank(a).clone())
        return torch.cat(outs, 0).numpy()

    if want("fbank"):
        # (a) the survey's known-answer case: offline kaldi.fbank over [240 zeros | signal], scale 1
        wav = torch.cat([torch.zeros(240), torch.from_numpy(pcm_pad.astype(np.float32))]).unsqueeze(0)
        off = kaldi.fbank(wav, dither=0, frame_length=25, frame_shift=10, num_mel_bins=80)
        assert off.shape == (208, 80) and abs(float(off.sum()) - 156308.2261) < 0.5, float(off.sum())
        # (b) reference's own stateful frontend, default constants (scale 32767, 16+3 frames)
        g_def = gating_stream(pcm_pad, None, 2560)
        # (c) the fork's constants (configs/dialog_state_pred_config.yaml:23-30): 16 ms / 8 ms
        fork = {"feat_dim": 80, "expected_audio_chunk_duration_in_sec": 0.224,
                "audio_to_proc_per_step_in_sec": 0.016, "step_size_in_sec": 0.008,
                "context_duration_in_sec": 0.032}
        n_fork = len(pcm_pad) // 3584
        g_fork = gating_stream(pcm_pad[:n_fork * 3584], fork, 3584)
        syn = synth_audio(1000, 16000 * 2).numpy()
        wav2 = torch.cat([torch.zeros(240), torch.from_numpy(syn.astype(np.float32))]).unsqueeze(0)
        off2 = kaldi.fbank(wav2, dither=0, frame_length=25, frame_shift=10, num_mel_bins=80)
        save("fbank", question_pcm=pcm, question_offline=off.numpy(), question_gating_default=g_def,
             question_gating_fork=g_fork, synth_pcm=syn, synth_offline=off2.numpy(),
             window=kaldi._feature_window_function("povey", 400, 0.42, torch.device("cpu"), torch.float32).numpy(),
             mel=kaldi.get_mel_banks(80, 512, 16000.0, 20.0, 0.0, 100.0, -500.0, 1.0)[0].numpy())

    # ---------------- VAD gating rule (models/AudioFeatureGating.py:77-109 + the relabelling loop of
    # bin/dialog_state_pred.py:626-670, restated here because that file imports the service stack) ----------
    if want("gating"):
        statuses = [None] * 3 + ["ipu_sl"] + ["ipu_cl"] * 2 + [None] * 9 + ["ipu_sl", "ipu_cl", None, "ipu_sl"]
        audio = synth_audio(77, 2560 * len(statuses)).numpy()
        g = ref_gating.AudioFeatureGating(16000)                       # defaults: history 10, onset 6, 25/10 ms, 16+3 frames
        blocks, labels, owner = [], [], []
        for i, st_ in enumerate(statuses):
            a = audio[i * 2560:(i + 1) * 2560].astype(np.float32) / 32768.0
            res = g.process_and_gate({"audio": a, "status": st_, "ipu_id": 0})
            if not res:
                continue
            if res["status"] == "ipu_sl":                              # dialog_state_pred.py:639-663
                for j, feat in enumerate(res["feature_last_chunk"]):
                    blocks.append(np.asarray(feat, np.float32).reshape(19, 80))
                    labels.append("ipu_sl" if j == 0 else "ipu_cl")
                    owner.append(i)
                blocks.append(np.asarray(res["feature"], np.float32).reshape(19, 80))
                labels.append("ipu_cl" if len(res["feature_last_chunk"]) > 0 else "ipu_sl")
                owner.append(i)
            else:                                                      # :665-670
                blocks.append(np.asarray(res["feature"], np.float32).reshape(19, 80))
                labels.append(res["status"])
                owner.append(i)
        save("gating", pcm=audio, statuses=np.array(["" if s_ is None else s_ for s_ in statuses]),
             blocks=np.stack(blocks), labels=np.array(labels), owner=np.asarray(owner, np.int64),
             history=g.history.numpy().copy(), scale=np.float64(32767.0))

    # ---------------- masks ----------------------------------------------------------------
    if want("masks"):
        arrs = {}
        for T in (1, 3, 4, 5, 17, 68, 69, 100):
            for c in (1, 4, 7):
                for L in (-1, 0, 1, 16):
                    m = ref_masks.subsequent_chunk_mask(T, c, L).numpy()
                    arrs["T%d_c%d_L%d" % (T, c, L)] = np.packbits(m.reshape(-1))
        save("masks", **arrs)

    def feats_from_pcm(int16_pcm):
        """bin/inference.py:57-80 (audioEncoderProcessor; not importable: the file needs soundfile
        and web.*) restated with the reference's own kaldi call, scale 32768."""
        samples, ring, out = torch.zeros(1, 2800), torch.zeros(1, 19, 80), []
        for i in range(len(int16_pcm) // 2560):
            a = torch.from_numpy(int16_pcm[i * 2560:(i + 1) * 2560].astype(np.float32) / 32768.0) * 32768
            samples = torch.cat([samples[:, -240:], a.view(1, -1)], 1)
            xs = kaldi.fbank(waveform=samples, dither=0, frame_length=25, frame_shift=10, num_mel_bins=80)
            ring = torch.cat([ring[:, -3:], xs.unsqueeze(0)], 1)
            out.append(ring.clone())
        return out

    # ---------------- tiny config ----------------------------------------------------------
    if want("tiny"):
        ycfg = load_yaml("tiny")
        cfg = path_config_from_dict(ycfg)
        enc, adp = build_reference(mods, ycfg, cfg, seed=3)
        B = 3
        pcm_b = [synth_audio(2000 + b, 2560 * 24).numpy() for b in range(B)]
        per = [feats_from_pcm(p) for p in pcm_b]
        feats_seq = [torch.cat([per[b][i] for b in range(B)], 0) for i in range(24)]
        st = stream_reference(enc, adp, feats_seq, layers_to_keep=(0, 1))
        # t = 7 frames per call (the fork's 32-frame inputs; SURVEY 2.4-2): position stride 4 != 7
        g = torch.Generator().manual_seed(5)
        feats32 = [9.0 + 3.0 * torch.randn(1, 32, 80, generator=g) for _ in range(12)]
        st7 = stream_reference(enc, adp, feats32, layers_to_keep=(0,))
        # offline ragged
        T = 150
        xs = 9.0 + 3.0 * torch.randn(B, T, 80, generator=g)
        ilens = torch.tensor([150, 97, 40])
        off = {}
        with torch.no_grad():
            for (c, L) in ((4, 16), (4, 2), (-1, -1), (4, -1), (3, 1)):
                eo, m = enc(xs, ilens, c, L)
                eo = eo.clone()
                y, ym = adp(eo.clone(), m)
                off["enc_c%d_L%d" % (c, L)] = eo.numpy()
                off["adp_c%d_L%d" % (c, L)] = y.numpy()
                off["mask_c%d_L%d" % (c, L)] = m.numpy()
                off["amask_c%d_L%d" % (c, L)] = ym.numpy()
        arrs = dict(seed=np.int64(3), stream_feats_sha256=feats_digest(torch.stack(feats_seq).numpy()),
                    **{"stream_" + k: v for k, v in st.items()},
                    **{"t7_" + k: st7[k] for k in ("enc_out", "adapter_out", "pe_index")},
                    off_ilens=ilens.numpy(), **{"off_" + k: v for k, v in off.items()})
        sample_last_axis(arrs, "kv", 16, ["stream_k_cache_l0", "stream_v_cache_l0", "stream_k_cache_l1", "stream_v_cache_l1"])
        save("tiny", **arrs)

    # ---------------- conv1d-linear positionwise variant (Conv1dLinear, attention.py:198-266) ----------
    # Only `forward` can be executed in the reference for this variant (its streaming wiring is broken, SURVEY 2.3):
    # offline goldens here; the streaming carry is pinned by the property "chunked == forward" in the tests.
    if want("tiny_conv1d"):
        ycfg = load_yaml("tiny_conv1d")
        cfg = path_config_from_dict(ycfg)
        enc, adp = build_reference(mods, ycfg, cfg, seed=3)
        g = torch.Generator().manual_seed(17)
        xs = 9.0 + 3.0 * torch.randn(3, 150, 80, generator=g)
        ilens = torch.tensor([150, 97, 40])
        off = {}
        with torch.no_grad():
            for (c, L) in ((4, 16), (-1, -1)):
                eo, m = enc(xs, ilens, c, L)
                eo = eo.clone()
                y, ym = adp(eo.clone(), m)
                off["enc_c%d_L%d" % (c, L)] = eo.numpy()
                off["adp_c%d_L%d" % (c, L)] = y.numpy()
                off["mask_c%d_L%d" % (c, L)] = m.numpy()
        save("tiny_conv1d", seed=np.int64(3), off_feats=xs.numpy(), off_ilens=ilens.numpy(), **{"off_" + k: v for k, v in off.items()})

    # ---------------- adapter with BatchNorm1d + ReLU (adapter.py:100-101,106-107), eval mode ----------------
    if want("tiny_bn"):
        ycfg = load_yaml("tiny_bn")
        cfg = path_config_from_dict(ycfg)
        mc = ycfg["model_conf"]
        adp = ref_adapter.CNNSubsampling(mc["enc_out_dim"], mc["llm_embed_dim"], mc["kernel_size"], mc["activation_func"], mc["norm"])
        sd = make_adapter_state(cfg, 3)
        missing = adp.load_state_dict(sd, strict=False)
        assert set(missing.missing_keys) <= {"bn2.num_batches_tracked"} and not missing.unexpected_keys, missing
        adp.eval()
        g = torch.Generator().manual_seed(23)
        xs = [torch.randn(2, 4, cfg.d_model, generator=g) for _ in range(5)]
        ys, cache = [], None
        with torch.no_grad():
            for x in xs:
                y, _, cache = adp(x.clone(), torch.ones(2, 1, 4, dtype=torch.bool), cache=cache, return_cache=True)
                ys.append(y.clone())
            xo = torch.randn(2, 37, cfg.d_model, generator=g)
            mo = torch.arange(37)[None, None, :] < torch.tensor([37, 20])[:, None, None]
            yo, mo2 = adp(xo.clone(), mo)
        save("tiny_bn", seed=np.int64(3), stream_x=torch.stack(xs).numpy(), stream_y=torch.stack(ys).numpy(),
             stream_cache=cache[0].contiguous().numpy(), off_x=xo.numpy(), off_mask=mo.numpy(), off_y=yo.numpy(),
             off_mask_out=mo2.numpy())

    # ---------------- LinearAdapter (adapter.py:59-70) ------------------------------------------------------
    if want("tiny_linear"):
        ycfg = load_yaml("tiny_linear")
        cfg = path_config_from_dict(ycfg)
        mc = ycfg["model_conf"]
        adp = ref_adapter.LinearAdapter(mc["enc_out_dim"], mc["llm_embed_dim"])
        adp.load_state_dict(make_adapter_state(cfg, 3), strict=True)
        adp.eval()
        g = torch.Generator().manual_seed(29)
        x = torch.randn(3, 11, cfg.d_model, generator=g)
        m = torch.arange(11)[None, None, :] < torch.tensor([11, 7, 2])[:, None, None]
        with torch.no_grad():
            y, m2 = adp(x.clone(), m)
        save("tiny_linear", seed=np.int64(3), x=x.numpy(), mask=m.numpy(), y=y.numpy(), mask_out=m2.numpy())

    # ---------------- adapter variants that only the ORACLE covers so far: CNNAdapter, two-conv CNNSubsampling ----------
    if want("tiny_adapter_variants"):
        import dataclasses
        base = path_config_from_dict(load_yaml("tiny_bn"))
        g = torch.Generator().manual_seed(37)
        out = {}
        # CNNAdapter (adapter.py:10-57)
        cfg = dataclasses.replace(base, adapter_type="cnn")
        adp = ref_adapter.CNNAdapter(cfg.d_model, cfg.llm_dim, cfg.adapter_kernel)
        miss = adp.load_state_dict(make_adapter_state(cfg, 5), strict=False)
        assert not miss.unexpected_keys and all(k.endswith("num_batches_tracked") for k in miss.missing_keys), miss
        adp.eval()
        x = torch.randn(2, 23, cfg.d_model, generator=g)
        m = torch.arange(23)[None, None, :] < torch.tensor([23, 9])[:, None, None]
        with torch.no_grad():
            y, _ = adp(x.clone(), m)
        out.update(cnn_x=x.numpy(), cnn_mask=m.numpy(), cnn_y=y.numpy())
        # CNNSubsampling with 4 * enc_out_dim < llm_embed_dim (adapter.py:84-96): streaming with both caches, then offline
        cfg2 = dataclasses.replace(base, llm_dim=cfg.d_model * 4 + 64)
        adp2 = ref_adapter.CNNSubsampling(cfg2.d_model, cfg2.llm_dim, cfg2.adapter_kernel, "relu", "batch")
        assert adp2.cnn_num == 2
        miss = adp2.load_state_dict(make_adapter_state(cfg2, 5), strict=False)
        assert not miss.unexpected_keys and all(k.endswith("num_batches_tracked") for k in miss.missing_keys), miss
        adp2.eval()
        xs = [torch.randn(2, 4, cfg2.d_model, generator=g) for _ in range(5)]
        ys, cache = [], None
        with torch.no_grad():
            for xx in xs:
                yy, _, cache = adp2(xx.clone(), torch.ones(2, 1, 4, dtype=torch.bool), cache=cache, return_cache=True)
                ys.append(yy.clone())
            xo = torch.randn(2, 31, cfg2.d_model, generator=g)
            mo = torch.arange(31)[None, None, :] < torch.tensor([31, 12])[:, None, None]
            yo, mo2 = adp2(xo.clone(), mo)
        out.update(two_llm_dim=np.int64(cfg2.llm_dim), two_stream_x=torch.stack(xs).numpy(), two_stream_y=torch.stack(ys).numpy(),
                   two_cache0=cache[0].contiguous().numpy(), two_cache1=cache[1].contiguous().numpy(),
                   two_off_x=xo.numpy(), two_off_mask=mo.numpy(), two_off_y=yo.numpy(), two_off_mask_out=mo2.numpy())
        save("tiny_adapter_variants", seed=np.int64(5), **out)

    # ---------------- TransformerLayer options: post-norm (transformer.py:89-90,97-98) and concat_after (:85-87) ------------
    if want("tiny_layer_variants"):
        out = {}
        for name in ("tiny_postnorm_concat", "tiny_concat"):
            ycfg = load_yaml(name)
            cfg = path_config_from_dict(ycfg)
            enc, adp = build_reference(mods, ycfg, cfg, seed=3)
            g = torch.Generator().manual_seed(59)
            feats_seq = [9.0 + 3.0 * torch.randn(2, 19, cfg.feat_dim, generator=g) for _ in range(19)]    # past the window saturation
            st_ = stream_reference(enc, adp, feats_seq, layers_to_keep=(0,))
            xs = 9.0 + 3.0 * torch.randn(2, 131, cfg.feat_dim, generator=g)
            ilens = torch.tensor([131, 70])
            with torch.no_grad():
                eo, m = enc(xs, ilens, 4, 16)
            out.update({name + "_feats": torch.stack(feats_seq).numpy(), name + "_enc_out": st_["enc_out"], name + "_adapter_out": st_["adapter_out"],
                        name + "_pe_index": st_["pe_index"], name + "_off_feats": xs.numpy(), name + "_off_ilens": ilens.numpy(),
                        name + "_off_enc": eo.numpy(), name + "_off_mask": m.numpy()})
        save("tiny_layer_variants", seed=np.int64(3), **out)

    # ---------------- MultiLayeredConv1d feed-forward (attention.py:145-196): full-utterance forward only ------------------
    if want("tiny_mlconv"):
        ycfg = load_yaml("tiny_mlconv")
        cfg = path_config_from_dict(ycfg)
        enc, adp = build_reference(mods, ycfg, cfg, seed=3)
        g = torch.Generator().manual_seed(61)
        xs = 9.0 + 3.0 * torch.randn(3, 163, cfg.feat_dim, generator=g)
        ilens = torch.tensor([163, 100, 41])
        out = {}
        with torch.no_grad():
            for (c_, L_) in ((4, 16), (-1, -1)):
                eo, m = enc(xs, ilens, c_, L_)
                eo = eo.clone()
                y, ym = adp(eo.clone(), m)
                out["enc_c%d_L%d" % (c_, L_)] = eo.numpy()
                out["adp_c%d_L%d" % (c_, L_)] = y.numpy()
                out["mask_c%d_L%d" % (c_, L_)] = m.numpy()
        save("tiny_mlconv", seed=np.int64(3), feats=xs.numpy(), ilens=ilens.numpy(), **out)

    # ---------------- shipped config -------------------------------------------------------
    if want("shipped"):
        ycfg = load_yaml("shipped")
        cfg = path_config_from_dict(ycfg)
        enc, adp = build_reference(mods, ycfg, cfg, seed=0)
        # config 1: question.wav, 13 chunks, 1 session
        fq = feats_from_pcm(pcm_pad)
        st = stream_reference(enc, adp, fq, layers_to_keep=(0, 23))
        arrs = dict(seed=np.int64(0), pcm=pcm_pad, feats_sha256=feats_digest(torch.stack(fq).numpy()), **st)
        sample_last_axis(arrs, "enc", 512, ["enc_out"])
        sample_last_axis(arrs, "adp", 1024, ["adapter_out"])
        sample_last_axis(arrs, "kv", 32, ["k_cache_l0", "v_cache_l0", "k_cache_l23", "v_cache_l23"])
        save("shipped_question", **arrs)
        # 2 lock-step sessions x 20 chunks: crosses the 17-chunk cache saturation (SURVEY 2.4-1)
        pcm_b = [synth_audio(1000 + b, 2560 * 20).numpy() for b in range(2)]
        per = [feats_from_pcm(p) for p in pcm_b]
        feats_seq = [torch.cat([per[b][i] for b in range(2)], 0) for i in range(20)]
        st2 = stream_reference(enc, adp, feats_seq, layers_to_keep=(0, 23))
        arrs = dict(seed=np.int64(0), feats_sha256=feats_digest(torch.stack(feats_seq).numpy()),
                    enc_out=st2["enc_out"], adapter_out=st2["adapter_out"], k_cache_l23=st2["k_cache_l23"])
        sample_last_axis(arrs, "enc", 512, ["enc_out"])
        sample_last_axis(arrs, "adp", 1024, ["adapter_out"])
        sample_last_axis(arrs, "kv", 32, ["k_cache_l23"])
        save("shipped_b2", **arrs)
        # the reference's own bf16 regime (models/pipeline.py:67-68 runs it under autocast bf16; on this
        # GPU-less host the CPU autocast is the executable stand-in): its distance from its fp32 outputs
        # is the noise floor quoted next to the bf16 parity numbers.
        eo_l, y_l = [], []
        with torch.no_grad(), torch.autocast("cpu", dtype=torch.bfloat16):
            buffer, cache, pe = [None] * 24, None, 0
            for f in feats_seq:
                eo, buffer, _, _, pe = enc.infer(f, buffer, 0, None, pe)
                eo_l.append(eo.float().clone())
                y, _, cache = adp(eo, torch.ones(2, 1, 4, dtype=torch.bool), cache=cache, return_cache=True)
                y_l.append(y.float().clone())
        fe = float(np.abs(torch.stack(eo_l).numpy() - st2["enc_out"]).max())
        fy = float(np.abs(torch.stack(y_l).numpy() - st2["adapter_out"]).max())
        print("reference autocast-bf16 vs fp32: encoder %.4f adapter %.4f" % (fe, fy))
        save("shipped_bf16_floor", ref_autocast_vs_fp32_encoder=np.float64(fe), ref_autocast_vs_fp32_adapter=np.float64(fy))
        # offline ragged pair
        g = torch.Generator().manual_seed(11)
        xs = 9.0 + 3.0 * torch.randn(2, 131, 80, generator=g)
        ilens = torch.tensor([131, 90])
        with torch.no_grad():
            eo, m = enc(xs, ilens, 4, 16)
            eo = eo.clone()
            y, ym = adp(eo.clone(), m)
        save("shipped_offline", seed=np.int64(0), feats=xs.numpy(), ilens=ilens.numpy(), enc_out=eo.numpy(),
             mask=m.numpy(), adapter_out=y.numpy(), adapter_mask=ym.numpy())


if __name__ == "__main__":
    main()
