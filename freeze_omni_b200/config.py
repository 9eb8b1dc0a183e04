"""Configuration of the streaming speech encoder + adapter path.

The yaml schema is the reference's own (``models/utils.py:30-49`` reads ``input_dim``,
``encoder_conf = {overview_conf, para_conf}`` and ``model_conf``; the dashed option names are the
argparse flags of ``models/encoder/encoder.py:12-34``, ``models/encoder/transformer.py:134-154``
and ``models/encoder/subsampling.py:77-84``).  ``PathConfig`` flattens it into the handful of
integers the C-ABI (``include/fo_b200.h: fo_config``) and the oracle need.
"""
from __future__ import annotations

import dataclasses
import os
from typing import Any, Dict, Optional

import yaml

_HERE = os.path.dirname(os.path.abspath(__file__))
CONFIG_DIR = os.path.join(os.path.dirname(_HERE), "configs")

# argparse defaults of the reference (transformer.py:136-153, subsampling.py:80-83)
_TRANSFORMER_DEFAULTS = {
    "transformer-input-dim": 256, "transformer-output-dim": 4, "transformer-attention-dim": 256,
    "transformer-attention-heads": 4, "transformer-linear-units": 1024, "transformer-num-blocks": 6,
    "transformer-input-layer": "linear", "transformer-pos-enc-class": "abs-enc",
    "transformer-normalize-before": True, "transformer-concat-after": False,
    "transformer-positionwise-layer-type": "linear", "transformer-positionwise-conv-kernel_size": 1,
    "transformer-chunk_size": -1, "transformer-left_chunks": -1, "transformer-dynamic-chunks": True,
}
# AudioLLM.__init__ defaults (audioLLM.py:27-52) for the model_conf keys this path reads
_MODEL_CONF_DEFAULTS = {
    "enc_out_dim": 512, "llm_embed_dim": 4096, "kernel_size": 3, "adpter_type": "cnn",
    "activation_func": "relu", "norm": "batch",
}
_SUBSAMPLING_DEFAULTS = {
    "subsampling-rate": 4, "subsampling-input-dim": 256, "subsampling-output-dim": 256,
}


@dataclasses.dataclass
class PathConfig:
    feat_dim: int = 80            # fbank bins == encoder-input-dim
    d_model: int = 1024           # subsampling-output-dim == transformer-attention-dim
    n_heads: int = 16
    ffn_dim: int = 4096
    n_layers: int = 24
    chunk_size: int = 4           # transformer-chunk_size (encoder frames)
    left_chunks: int = 16         # transformer-left_chunks
    input_layer: str = "linear"   # transformer-input-layer: linear | none
    normalize_before: bool = True  # False: post-norm layers (transformer.py:89-90,97-98), no after_norm (:232-233)
    concat_after: bool = False     # x + concat_linear(cat(layer input, att)) instead of x + att (transformer.py:85-87)
    dynamic_chunks: bool = False
    # positionwise layer (transformer.py:205-217): "linear" = PositionwiseFeedForward (attention.py:122-143);
    # "conv1d-linear" = Conv1dLinear (attention.py:198-266): causal depthwise Conv1d(k) + 1x1 Conv1d + ReLU + Linear
    ffn_type: str = "linear"
    ffn_conv_kernel: int = 1
    pos_max_len: int = 5000       # RelPositionalEncoding max_len default (attention.py:78)
    # adapter (models/adapter.py:73-110, single-conv branch)
    llm_dim: int = 3584
    adapter_kernel: int = 5
    adapter_act: str = "gelu"
    adapter_norm: str = "layer"
    adapter_type: str = "subsampling"       # 'subsampling' (CNNSubsampling, adapter.py:72-157) | 'linear' (LinearAdapter, :59-70) | 'cnn' (CNNAdapter, :10-57)
    # streaming frontend (bin/inference.py:43-56)
    sample_rate: int = 16000
    frame_length_ms: int = 25
    frame_shift_ms: int = 10
    frames_per_chunk: int = 16
    context_frames: int = 3
    pcm_scale: float = 32768.0

    # ---- derived quantities (attention.py:83,88,291; subsampling.py:34) -----------------------
    @property
    def adapter_two_conv(self) -> bool:
        """CNNAdapter (adapter.py:10-57) and CNNSubsampling with enc_out_dim * 4 < llm_embed_dim (adapter.py:83-96) run two
        convolutions (C -> 2C -> 4C) with BatchNorm1d + ReLU each, whatever activation_func / norm say."""
        return self.adapter_type == "cnn" or (self.adapter_type == "subsampling" and self.d_model * 4 < self.llm_dim)

    @property
    def d_k(self) -> int:
        return self.d_model // self.n_heads

    @property
    def kv_window(self) -> int:          # MultiHeadedAttention.buffersize
        return self.chunk_size * self.left_chunks if (self.chunk_size > 0 and self.left_chunks > 0) else 1

    @property
    def full_chunk_size(self) -> int:    # RelPositionalEncoding.full_chunk_size
        return (self.left_chunks + 1) * self.chunk_size

    @property
    def pe_wrap(self) -> int:            # RelPositionalEncoding.max_len after __init__
        return self.chunk_size * (self.pos_max_len // self.chunk_size) - self.full_chunk_size

    @property
    def sub_freq(self) -> int:           # ((idim - 1) // 2 - 1) // 2
        return ((self.feat_dim - 1) // 2 - 1) // 2

    @property
    def frame_len(self) -> int:
        return self.sample_rate * self.frame_length_ms // 1000

    @property
    def frame_shift(self) -> int:
        return self.sample_rate * self.frame_shift_ms // 1000

    @property
    def samples_per_chunk(self) -> int:
        return self.frame_shift * self.frames_per_chunk

    @property
    def sample_carry(self) -> int:
        return self.frame_len - self.frame_shift

    @property
    def chunk_feat_frames(self) -> int:
        return self.frames_per_chunk + self.context_frames

    @staticmethod
    def sub_len(t: int) -> int:
        """Frames after Conv2dSubsampling4: ((T-1)//2 - 1)//2 (subsampling.py:28-34)."""
        return ((t - 1) // 2 - 1) // 2

    def adapter_len(self, t: int) -> int:
        """Adapter frames for t encoder frames: CNNSubsampling's stride-2 conv over k-1 left frames gives (t-1)//2 + 1
        (adapter.py:137-144); LinearAdapter and CNNAdapter keep the rate."""
        return t if self.adapter_type in ("linear", "cnn") else (t - 1) // 2 + 1

    def packed_offsets(self, lens):
        """Row offsets of a packed offline call (fo_encode_offline_packed) for feature lengths ``lens``: (enc_offsets,
        adapter_offsets), int64 arrays of B + 1 prefix sums of the per-utterance encoder / adapter rows."""
        import numpy as np
        t = np.asarray(lens, dtype=np.int64).reshape(-1)
        if t.size == 0 or (t < 7).any():
            raise ValueError("every utterance needs >= 7 feature frames")
        t2 = ((t - 1) // 2 - 1) // 2
        t3 = t2 if self.adapter_type in ("linear", "cnn") else (t2 - 1) // 2 + 1
        return np.concatenate([[0], np.cumsum(t2)]), np.concatenate([[0], np.cumsum(t3)])

    def packed_audio_offsets(self, n_samples):
        """Offsets of a packed PCM call (fo_encode_offline_packed_pcm) for utterances of ``n_samples`` samples: (frames,
        enc_offsets, adapter_offsets), int64 arrays.  frames[i] = 1 + (n_samples[i] - frame_len) // frame_shift (kaldi
        snip_edges: trailing samples that fill no frame are dropped); the offsets are packed_offsets(frames)."""
        import numpy as np
        n = np.asarray(n_samples, dtype=np.int64).reshape(-1)
        m = np.where(n >= self.frame_len, 1 + (n - self.frame_len) // self.frame_shift, 0)
        if m.size == 0 or (m < 7).any():
            raise ValueError("every utterance needs >= 7 feature frames (%d samples)" % (self.frame_len + 6 * self.frame_shift))
        eoff, aoff = self.packed_offsets(m)
        return m, eoff, aoff

    def validate(self) -> None:
        """The reference exits on an inconsistent config (encoder.py:74-75,86-87,94); here a
        ValueError.  Variants whose streaming path is broken upstream are refused loudly
        (SURVEY 2.3): abs-enc has no ``infer``; conv1d FFNs cannot stream."""
        if self.d_model % self.n_heads:
            raise ValueError("attention dim must be divisible by heads (attention.py:279)")
        if self.d_k != 64:
            raise ValueError("the sm_100a attention kernel is built for d_k == 64 (got %d)" % self.d_k)
        if self.d_model % 64 or self.ffn_dim % 64 or self.llm_dim % 64:
            raise ValueError("d_model, ffn_dim and llm_dim must be multiples of 64")
        if self.input_layer not in ("linear", "none"):
            raise ValueError("unsupported transformer-input-layer: %s" % self.input_layer)
        if self.adapter_norm not in ("layer", "batch") or self.adapter_act not in ("gelu", "relu"):
            raise ValueError("adapter: norm must be layer|batch and activation gelu|relu (adapter.py:100-107)")
        if self.adapter_kernel < 2:
            raise ValueError("adapter kernel_size must be >= 2")
        if self.adapter_type not in ("subsampling", "linear", "cnn"):
            raise ValueError("adpter_type must be cnn | linear | subsampling (audioLLM.py:159-165); got %r" % self.adapter_type)
        if self.adapter_two_conv and self.d_model * 4 > 4096:
            raise ValueError("the two-conv adapters normalise 4 * d_model channels; d_model must be <= 1024")
        if self.ffn_type not in ("linear", "conv1d-linear", "conv1d"):
            raise ValueError("positionwise-layer-type %r: support only linear, conv1d or conv1d-linear" % self.ffn_type)
        if self.ffn_type == "conv1d" and not (self.ffn_conv_kernel % 2 == 1 and 3 <= self.ffn_conv_kernel <= 9):
            raise ValueError("conv1d (MultiLayeredConv1d, attention.py:158-196; full-utterance forward only) needs an odd "
                             "positionwise-conv-kernel_size in 3..9")
        if self.ffn_type == "conv1d-linear" and not (2 <= self.ffn_conv_kernel <= 16):
            raise ValueError("conv1d-linear needs 2 <= positionwise-conv-kernel_size <= 16")


def load_yaml(name_or_path: str) -> Dict[str, Any]:
    path = name_or_path
    if not os.path.exists(path):
        path = os.path.join(CONFIG_DIR, name_or_path if name_or_path.endswith(".yaml") else name_or_path + ".yaml")
    with open(path, "r") as fin:
        return yaml.safe_load(fin)


def path_config_from_dict(configs: Dict[str, Any], encoder_only: bool = False) -> PathConfig:
    enc = configs.get("encoder_conf", {})
    over = enc.get("overview_conf", {})
    para = enc.get("para_conf", {})
    layer_cfg = over.get("encoder-layer-config", "subsampling-transformer")
    if layer_cfg != "subsampling-transformer":
        raise ValueError("only encoder-layer-config 'subsampling-transformer' is supported "
                         "(audioLLM.py:378 reads enc[1].num_blocks); got %r" % layer_cfg)
    tr = dict(_TRANSFORMER_DEFAULTS)
    tr.update(para.get("transformer", {}))
    sub = dict(_SUBSAMPLING_DEFAULTS)
    sub.update(para.get("subsampling", {}))
    if tr["transformer-pos-enc-class"] != "rel-enc":
        raise ValueError("only transformer-pos-enc-class 'rel-enc' can stream (attention.py:105)")
    if tr["transformer-positionwise-layer-type"] not in ("linear", "conv1d-linear", "conv1d"):
        raise ValueError("positionwise-layer-type %r: support only linear, conv1d or conv1d-linear (transformer.py:205-219)"
                         % tr["transformer-positionwise-layer-type"])
    if sub["subsampling-rate"] != 4:
        raise ValueError("only subsampling-rate 4 exists (subsampling.py:93-96)")
    feat = int(over.get("encoder-input-dim", configs.get("input_dim", 80)))
    d = int(tr["transformer-attention-dim"])
    dims = {int(sub["subsampling-output-dim"]), int(tr["transformer-input-dim"]), d,
            int(tr["transformer-output-dim"]), int(over.get("encoder-output-dim", d))}
    if len(dims) != 1 or int(sub["subsampling-input-dim"]) != feat:
        raise ValueError("WRONG CONFIG: component input/output dims do not chain (encoder.py:82-96)")
    # absent model_conf keys take the REFERENCE's constructor defaults (AudioLLM.__init__, audioLLM.py:27-52: enc_out_dim 512,
    # llm_embed_dim 4096, kernel_size 3, adpter_type 'cnn', activation_func 'relu', norm 'batch'), not the shipped values:
    # a train.yaml that omits activation_func / norm describes a BatchNorm + ReLU checkpoint
    mc = dict(_MODEL_CONF_DEFAULTS)
    mc.update(configs.get("model_conf", {}) or {})
    if encoder_only:
        mc.update({"enc_out_dim": d, "llm_embed_dim": d, "adpter_type": "linear"})
    adpter_type = str(mc["adpter_type"])
    if adpter_type not in ("subsampling", "linear", "cnn"):
        raise ValueError("adpter_type must be cnn | linear | subsampling (audioLLM.py:159-165); got %r" % adpter_type)
    if int(mc["enc_out_dim"]) != d:
        raise ValueError("model_conf.enc_out_dim (%d; the reference's default is 512) must equal the encoder output dim %d"
                         % (int(mc["enc_out_dim"]), d))
    fe = configs.get("frontend", {})
    cfg = PathConfig(
        feat_dim=feat, d_model=d, n_heads=int(tr["transformer-attention-heads"]),
        ffn_dim=int(tr["transformer-linear-units"]), n_layers=int(tr["transformer-num-blocks"]),
        chunk_size=int(tr["transformer-chunk_size"]), left_chunks=int(tr["transformer-left_chunks"]),
        input_layer=str(tr["transformer-input-layer"]),
        normalize_before=bool(tr["transformer-normalize-before"]), concat_after=bool(tr["transformer-concat-after"]),
        dynamic_chunks=bool(tr["transformer-dynamic-chunks"]),
        ffn_type=str(tr["transformer-positionwise-layer-type"]),
        ffn_conv_kernel=int(tr["transformer-positionwise-conv-kernel_size"]) if tr["transformer-positionwise-layer-type"] != "linear" else 1,
        llm_dim=int(mc["llm_embed_dim"]), adapter_kernel=int(mc["kernel_size"]),
        adapter_act=str(mc["activation_func"]), adapter_norm=str(mc["norm"]),
        adapter_type=adpter_type,
        sample_rate=int(fe.get("sample_rate", 16000)), frame_length_ms=int(fe.get("frame_length_ms", 25)),
        frame_shift_ms=int(fe.get("frame_shift_ms", 10)), frames_per_chunk=int(fe.get("frames_per_chunk", 16)),
        context_frames=int(fe.get("context_frames", 3)), pcm_scale=float(fe.get("pcm_scale", 32768.0)),
    )
    cfg.validate()
    return cfg


def load_path_config(name_or_path: str = "shipped") -> PathConfig:
    return path_config_from_dict(load_yaml(name_or_path))
