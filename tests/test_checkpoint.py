"""Trained-weights ingest: CMVN statistics parsers pinned to the outputs of the reference's own load_cmvn
(tests/golden/cmvn.npz, made by tests/golden/make_golden.py --only cmvn), checkpoint splitting and the strict audit."""
import os

import numpy as np
import pytest
import torch

from freeze_omni_b200.checkpoint import load_cmvn, load_trained, split_checkpoint
from freeze_omni_b200.config import load_path_config
from freeze_omni_b200.weights import make_adapter_state, make_encoder_state

GOLD = os.path.join(os.path.dirname(__file__), "golden", "cmvn.npz")


def test_cmvn_parsers_bit_exact_against_reference(tmp_path):
    g = np.load(GOLD)
    pj, pk = tmp_path / "c.json", tmp_path / "c.txt"
    pj.write_bytes(g["json_text"].tobytes())
    pk.write_bytes(g["kaldi_text"].tobytes())
    mj, ij = load_cmvn(str(pj), True)
    mk, ik = load_cmvn(str(pk), False)
    assert np.array_equal(mj, g["json_mean"]) and np.array_equal(ij, g["json_istd"])          # float64, bit-exact
    assert np.array_equal(mk, g["kaldi_mean"]) and np.array_equal(ik, g["kaldi_istd"])
    assert ij[7] == 1.0 / np.sqrt(1.0e-20)                                                     # variance floor (cmvn.py:55-56)
    bad = tmp_path / "bin"
    bad.write_bytes(b"\0B junk")
    with pytest.raises(ValueError):
        load_cmvn(str(bad), False)


def test_checkpoint_split_and_audit(tmp_path):
    cfg = load_path_config("tiny")
    enc, adp = make_encoder_state(cfg, 1), make_adapter_state(cfg, 1)
    ckpt = {}
    for role, scale in (("user", 1.0), ("system", 2.0)):                  # audioLLM.py:67-68,160-166: both roles in one file
        ckpt.update({"encoder_%s.%s" % (role, k): v * scale for k, v in enc.items()})
        ckpt.update({"adpter_%s._orig_mod.%s" % (role, k): v * scale for k, v in adp.items()})
    ckpt["llm_decoder.lm_head.weight"] = torch.zeros(3, 3)                # unrelated tensors are ignored
    e_u, a_u = split_checkpoint(ckpt, "user")
    e_s, a_s = split_checkpoint(ckpt, "system")
    assert set(e_u) == set(enc) and set(a_u) == set(adp)
    k = "enc.1.encoders.0.self_attn.linear_q.weight"
    assert torch.equal(e_u[k], enc[k]) and torch.equal(e_s[k], enc[k] * 2.0)
    # end to end through files, yaml found next to the checkpoint
    import shutil
    import yaml
    from freeze_omni_b200.config import load_yaml
    shutil.copyfile(os.path.join(os.path.dirname(__file__), "..", "configs", "tiny.yaml"), tmp_path / "final.yaml")
    torch.save(ckpt, tmp_path / "final.pt")
    cfg2, e2, a2 = load_trained(str(tmp_path), role="system")
    assert cfg2.d_model == cfg.d_model and torch.equal(e2[k], enc[k] * 2.0) and set(a2) == set(adp)
    # a renamed key must be reported, not silently dropped (utils.py:20 loads with strict=False)
    broken = dict(ckpt)
    broken["encoder_user.enc.1.encoders.0.self_attn.linear_Q.weight"] = broken.pop("encoder_user." + k)
    torch.save(broken, tmp_path / "final.pt")
    with pytest.raises(KeyError):
        load_trained(str(tmp_path), role="user")
    assert load_yaml(str(tmp_path / "final.yaml")) and yaml is not None


def test_absent_model_conf_keys_take_the_reference_defaults(tmp_path):
    """AudioLLM.__init__ defaults (models/audioLLM.py:27-52): kernel_size 3, activation_func 'relu', norm 'batch',
    llm_embed_dim 4096, enc_out_dim 512, adpter_type 'cnn' -- NOT the shipped values (ADVICE r1): a train.yaml that omits
    activation_func / norm describes a BatchNorm + ReLU adapter."""
    import copy
    from freeze_omni_b200.config import load_yaml, path_config_from_dict
    y = load_yaml("tiny")
    y2 = copy.deepcopy(y)
    for k in ("activation_func", "norm", "kernel_size"):
        y2["model_conf"].pop(k)
    cfg = path_config_from_dict(y2)
    assert (cfg.adapter_act, cfg.adapter_norm, cfg.adapter_kernel) == ("relu", "batch", 3)
    y3 = copy.deepcopy(y)
    y3["model_conf"].pop("enc_out_dim")                                    # default 512 != tiny's 128
    with pytest.raises(ValueError, match="enc_out_dim"):
        path_config_from_dict(y3)
    # a LayerNorm yaml on a BatchNorm checkpoint (extra bn2.running_*) is refused, not silently mis-loaded
    cfg_ln = load_path_config("tiny")
    cfg_bn = load_path_config("tiny_bn")
    enc, adp_bn = make_encoder_state(cfg_ln, 1), make_adapter_state(cfg_bn, 1)
    ckpt = {"encoder.%s" % k: v for k, v in enc.items()}
    ckpt.update({"adpter.%s" % k: v for k, v in adp_bn.items()})
    ckpt["adpter.bn2.num_batches_tracked"] = torch.tensor(7)
    import shutil
    torch.save(ckpt, tmp_path / "final.pt")
    shutil.copyfile(os.path.join(os.path.dirname(__file__), "..", "configs", "tiny.yaml"), tmp_path / "final.yaml")
    with pytest.raises(ValueError, match="does not use"):
        load_trained(str(tmp_path))
    shutil.copyfile(os.path.join(os.path.dirname(__file__), "..", "configs", "tiny_bn.yaml"), tmp_path / "final.yaml")
    cfg2, _, a2 = load_trained(str(tmp_path))                              # num_batches_tracked rides along with a BatchNorm
    assert cfg2.adapter_norm == "batch" and "bn2.running_var" in a2
