"""Python owner of one fo_ctx: loads weights through the C ABI and exposes the batched session API
("model as a server": many sessions advance one chunk per step).  PyTorch is used for device memory and
streams only; all compute happens inside libfo_b200.so."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from . import host_constants as hc
from .config import PathConfig
from .weights import adapter_param_shapes, audit_state_dict, encoder_param_shapes

ArrayLike = Union[torch.Tensor, np.ndarray]


def _ptr(x: Optional[ArrayLike]) -> Optional[int]:
    if x is None:
        return None
    if isinstance(x, torch.Tensor):
        assert x.is_contiguous(), "tensors crossing the C ABI must be contiguous"
        return x.data_ptr()
    assert x.flags["C_CONTIGUOUS"]
    return x.ctypes.data


def _ids(ids) -> np.ndarray:
    if isinstance(ids, torch.Tensor):
        ids = ids.cpu().numpy()
    return np.ascontiguousarray(np.asarray(ids, dtype=np.int32).reshape(-1))


def _i32p(a: np.ndarray):
    return a.ctypes.data_as(C.POINTER(C.c_int32))


class Engine:
    """One context on one GPU.  ``enc_state`` / ``adp_state`` are state dicts under the reference's key
    names (SURVEY 3.4); either may be None to build an encoder-only or adapter-only context."""

    def __init__(self, cfg: PathConfig, enc_state: Optional[Dict[str, torch.Tensor]] = None,
                 adp_state: Optional[Dict[str, torch.Tensor]] = None, dtype: torch.dtype = torch.float32,
                 device: int = 0, max_sessions: int = 64, max_stream_frames: Optional[int] = None,
                 use_cmvn: bool = True, sm_partition: Optional[Tuple[int, int]] = None):
        """``sm_partition``: None runs the context on the whole device; ``(split, group)`` runs it on group ``group`` of
        ``split`` equal groups of the device's SMs (fo_create_on_sms), so that contexts on other groups of the same split
        (another encoder, an LLM beside it) run on disjoint SMs."""
        if not torch.cuda.is_available():
            raise RuntimeError("freeze_omni_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
        if dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("compute dtype must be float32 or bfloat16")
        cfg.validate()
        self.lib = _lib.load()
        self.cfg, self.dtype, self.device = cfg, dtype, int(device)
        self.torch_device = torch.device("cuda", self.device)
        self.has_encoder, self.has_adapter = enc_state is not None, adp_state is not None
        self.max_sessions = int(max_sessions)
        msf = max_stream_frames or max(cfg.chunk_feat_frames, 39)
        c = _lib.FoConfig(
            feat_dim=cfg.feat_dim, d_model=cfg.d_model, n_heads=cfg.n_heads, ffn_dim=cfg.ffn_dim,
            n_layers=cfg.n_layers, chunk_size=cfg.chunk_size, left_chunks=cfg.left_chunks,
            input_layer_linear=int(cfg.input_layer == "linear"), pos_max_len=cfg.pos_max_len, llm_dim=cfg.llm_dim,
            adapter_kernel=cfg.adapter_kernel, adapter_gelu=int(cfg.adapter_act == "gelu"),
            has_encoder=int(self.has_encoder), has_adapter=int(self.has_adapter), sample_rate=cfg.sample_rate,
            frame_len=cfg.frame_len, frame_shift=cfg.frame_shift, frames_per_chunk=cfg.frames_per_chunk,
            context_frames=cfg.context_frames, max_sessions=int(max_sessions), max_stream_frames=int(msf),
            ffn_conv_kernel=int(cfg.ffn_conv_kernel) if cfg.ffn_type in ("conv1d-linear", "conv1d") else 0,
            adapter_batchnorm=int(cfg.adapter_norm == "batch"),
            adapter_type={"subsampling": 0, "linear": 1, "cnn": 2}[cfg.adapter_type],
            post_norm=int(not cfg.normalize_before), concat_after=int(cfg.concat_after),
            ffn_multi_conv=int(cfg.ffn_type == "conv1d"))
        h = C.c_void_p()
        fo_dtype = _lib.FO_BF16 if dtype == torch.bfloat16 else _lib.FO_F32
        if sm_partition is None:
            _lib.check(self.lib.fo_create(C.byref(c), self.device, fo_dtype, C.byref(h)))
        else:
            split, group = sm_partition
            _lib.check(self.lib.fo_create_on_sms(C.byref(c), self.device, fo_dtype, int(split), int(group), C.byref(h)))
        self._h = h
        self.sm_count = self.get_option("sm_count")   # SMs the context's grids spread over: its group's, or the device's
        self.max_t = self.get_option("max_t")      # encoder frames per streaming chunk, capped at 8 by the library
        try:
            if self.has_encoder:
                exp = encoder_param_shapes(cfg)
                if not use_cmvn or "global_cmvn.mean" not in enc_state:
                    exp = [e for e in exp if not e[0].startswith("global_cmvn.")]
                audit_state_dict(exp, enc_state)
                for k, _, _ in exp:
                    self._load(k, enc_state[k])
                self._load("pos.table", hc.pos_table(cfg.pos_max_len, cfg.d_model))
                self._load("fbank.window", hc.fbank_window(cfg.frame_len))
                self._load("fbank.mel", hc.fbank_mel(cfg.feat_dim, cfg.frame_len, cfg.sample_rate))
            if self.has_adapter:
                exp = adapter_param_shapes(cfg)
                audit_state_dict(exp, adp_state)
                for k, _, _ in exp:
                    self._load("adapter." + k, adp_state[k])
            _lib.check(self.lib.fo_finalize_weights(self._h))
        except Exception:
            self.close()
            raise

    # ---- plumbing ---------------------------------------------------------------------------------
    def _load(self, name: str, t: torch.Tensor) -> None:
        t = t.detach().to(torch.float32).contiguous()
        shape = (C.c_int64 * t.dim())(*t.shape)
        _lib.check(self.lib.fo_load_tensor(self._h, name.encode(), t.data_ptr(), shape, t.dim()))

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.torch_device).cuda_stream

    def _out(self, out: Optional[torch.Tensor], shape, dtype=torch.float32) -> torch.Tensor:
        if out is None:
            return torch.empty(shape, dtype=dtype, device=self.torch_device)
        assert tuple(out.shape) == tuple(shape) and out.dtype == dtype and out.is_contiguous()
        return out

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.fo_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_option(self, name: str, value: int) -> None:
        _lib.check(self.lib.fo_set_option(self._h, name.encode(), int(value)))

    def get_option(self, name: str) -> int:
        v = C.c_int64()
        _lib.check(self.lib.fo_get_option(self._h, name.encode(), C.byref(v)))
        return int(v.value)

    def profile_dump(self):
        """[(M, N, K, launches, microseconds)] of the GEMM launches timed under option profile_gemm."""
        buf = C.create_string_buffer(1 << 16)
        _lib.check(self.lib.fo_profile_dump(self._h, buf, len(buf)))
        rows = []
        for line in buf.value.decode().splitlines():
            m, n, k, cnt, us = line.split()
            rows.append((int(m), int(n), int(k), int(cnt), float(us)))
        return rows

    def stats(self) -> Dict[str, int]:
        s = _lib.FoStats()
        _lib.check(self.lib.fo_stats(self._h, C.byref(s)))
        return {n: int(getattr(s, n)) for n, _ in s._fields_}

    # ---- sessions ---------------------------------------------------------------------------------
    def alloc(self, n: int) -> np.ndarray:
        ids = np.zeros(n, dtype=np.int32)
        _lib.check(self.lib.fo_session_alloc(self._h, n, _i32p(ids)))
        return ids

    def free(self, ids) -> None:
        ids = _ids(ids)
        if self._h:
            _lib.check(self.lib.fo_session_free(self._h, len(ids), _i32p(ids)))

    def reset(self, ids) -> None:
        ids = _ids(ids)
        _lib.check(self.lib.fo_session_reset(self._h, len(ids), _i32p(ids)))

    def state(self, sid: int) -> Tuple[int, int]:
        """(encoder frames appended so far, pe_index)."""
        a, b = C.c_int64(), C.c_int64()
        _lib.check(self.lib.fo_session_get_state(self._h, int(sid), C.byref(a), C.byref(b)))
        return int(a.value), int(b.value)

    def set_pe_index(self, ids, pe_index) -> None:
        ids = _ids(ids)
        pe = np.ascontiguousarray(np.broadcast_to(np.asarray(pe_index, dtype=np.int64), ids.shape))
        _lib.check(self.lib.fo_session_set_pe_index(self._h, len(ids), _i32p(ids), pe.ctypes.data_as(C.POINTER(C.c_int64))))

    def export_kv(self, sid: int, layer: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """One layer's cache in the reference layout (1, H, cache_len, d_k) (attention.py:415-428)."""
        n_frames, _ = self.state(sid)
        cl = min(n_frames, self.cfg.kv_window)
        k = torch.empty(1, self.cfg.n_heads, cl, self.cfg.d_k)
        v = torch.empty_like(k)
        got = C.c_int32()
        _lib.check(self.lib.fo_session_export_kv(self._h, int(sid), int(layer), k.data_ptr(), v.data_ptr(), C.byref(got)))
        assert got.value == cl
        return k, v

    def import_kv(self, sid: int, layer: int, k: torch.Tensor, v: torch.Tensor) -> None:
        k = k.detach().float().cpu().contiguous().view(self.cfg.n_heads, -1, self.cfg.d_k)
        v = v.detach().float().cpu().contiguous().view(self.cfg.n_heads, -1, self.cfg.d_k)
        _lib.check(self.lib.fo_session_import_kv(self._h, int(sid), int(layer), k.data_ptr(), v.data_ptr(), k.shape[1]))

    def set_frames(self, sid: int, n_frames: int) -> None:
        _lib.check(self.lib.fo_session_set_frames(self._h, int(sid), int(n_frames)))

    def export_ffn_cache(self, sid: int, layer: int) -> torch.Tensor:
        """Conv1dLinear left context of one layer, reference layout (1, d_model, k-1) (attention.py:258)."""
        buf = torch.empty(1, self.cfg.d_model, self.cfg.ffn_conv_kernel - 1)
        _lib.check(self.lib.fo_session_export_ffn_cache(self._h, int(sid), int(layer), buf.data_ptr()))
        return buf

    def _adapter_cache_channels(self, which: int) -> int:
        if self.cfg.adapter_two_conv:
            return 2 * self.cfg.d_model if which == 0 else self.cfg.d_model
        return self.cfg.d_model

    def export_adapter_cache(self, sid: int, which: int = 0) -> Optional[torch.Tensor]:
        """Entry `which` of the reference's adapter cache list (adapter.py:123-143), (1, channels, k-1); None == not set.
        The two-conv CNNSubsampling has entries 0 (second conv's input, 2 * d_model) and 1 (first conv's input, d_model)."""
        buf = torch.empty(1, self._adapter_cache_channels(which), self.cfg.adapter_kernel - 1)
        valid = C.c_int32()
        _lib.check(self.lib.fo_session_export_adapter_cache_n(self._h, int(sid), int(which), buf.data_ptr(), C.byref(valid)))
        return buf if valid.value else None

    def import_adapter_cache(self, sid: int, cache: Optional[torch.Tensor], which: int = 0) -> None:
        if cache is None:
            _lib.check(self.lib.fo_session_import_adapter_cache_n(self._h, int(sid), int(which), None, 0))
        else:
            c = cache.detach().float().cpu().contiguous()
            assert c.numel() == self._adapter_cache_channels(which) * (self.cfg.adapter_kernel - 1)
            _lib.check(self.lib.fo_session_import_adapter_cache_n(self._h, int(sid), int(which), c.data_ptr(), 1))

    # ---- session snapshots ------------------------------------------------------------------------
    @property
    def snapshot_bytes(self) -> int:
        """Size of one session's snapshot record (fo_session_snapshot_bytes); depends on the model, not on the capacities."""
        b = C.c_int64()
        _lib.check(self.lib.fo_session_snapshot_bytes(self._h, C.byref(b)))
        return int(b.value)

    def save_sessions(self, ids, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The whole state of sessions `ids` as a uint8 tensor (n, snapshot_bytes), one record per row, on this engine's device
        and stream; or into `out` (device, or host -- pinned keeps the copy asynchronous; a host `out` is complete on return).
        Rows restore with restore_sessions here, on another engine of the same model, or on another GPU after
        `blob.to(other.torch_device)`."""
        ids = _ids(ids)
        out = self._out(out, (len(ids), self.snapshot_bytes), torch.uint8)
        _lib.check(self.lib.fo_session_save(self._h, _i32p(ids), len(ids), _ptr(out), self._stream()))
        if not out.is_cuda:
            torch.cuda.current_stream(self.torch_device).synchronize()
        return out

    def restore_sessions(self, ids, blob: torch.Tensor) -> None:
        """Write records (n, snapshot_bytes) -- host, or on this engine's device -- into the allocated sessions `ids`; they
        continue bit for bit as the saved sessions would have.  A record of another model configuration is refused (FoError
        naming the field) before any session is touched."""
        ids = _ids(ids)
        if blob.dtype != torch.uint8 or not blob.is_contiguous() or tuple(blob.shape) != (len(ids), self.snapshot_bytes):
            raise ValueError("blob must be a contiguous uint8 tensor (%d, %d), got %s %s"
                             % (len(ids), self.snapshot_bytes, blob.dtype, tuple(blob.shape)))
        if blob.is_cuda and blob.device != self.torch_device:
            raise ValueError("blob is on %s, the engine on %s: copy it over first (blob.to(engine.torch_device))"
                             % (blob.device, self.torch_device))
        _lib.check(self.lib.fo_session_restore(self._h, _i32p(ids), len(ids), _ptr(blob), self._stream()))

    # ---- frontend ---------------------------------------------------------------------------------
    @staticmethod
    def _pcm_dtype(pcm: ArrayLike) -> int:
        dt = pcm.dtype
        if dt in (torch.int16, np.dtype(np.int16)):
            return _lib.FO_I16
        if dt in (torch.float32, np.dtype(np.float32)):
            return _lib.FO_F32
        raise TypeError("PCM must be int16 or float32")

    def _scale(self, pcm: ArrayLike, scale: Optional[float]) -> float:
        """Factor applied to the samples before the fbank ("value used = sample * scale", fo_b200.h).  The reference feeds
        kaldi.fbank audio in the int16 RANGE: float audio in [-1, 1] is multiplied by 32768 / 32767 (bin/inference.py:74,
        AudioFeatureGating.py:58), i.e. `cfg.pcm_scale`; int16 PCM is already in that range, so its default is 1.0."""
        if scale is not None:
            return float(scale)
        return 1.0 if self._pcm_dtype(pcm) == _lib.FO_I16 else float(self.cfg.pcm_scale)

    def fbank_stream(self, ids, pcm: ArrayLike, scale: Optional[float] = None,
                     out: Optional[torch.Tensor] = None) -> torch.Tensor:
        ids = _ids(ids)
        n = len(ids)
        assert tuple(pcm.shape) == (n, self.cfg.samples_per_chunk), "pcm must be (n, samples_per_chunk)"
        out = self._out(out, (n, self.cfg.chunk_feat_frames, self.cfg.feat_dim))
        _lib.check(self.lib.fo_fbank_stream(self._h, _i32p(ids), n, _ptr(pcm), self._pcm_dtype(pcm),
                                            self._scale(pcm, scale), _ptr(out),
                                            self._stream()))
        return out

    def fbank_offline(self, pcm: ArrayLike, scale: Optional[float] = None) -> torch.Tensor:
        B, N = pcm.shape
        m = 1 + (N - self.cfg.frame_len) // self.cfg.frame_shift
        out = torch.empty(B, m, self.cfg.feat_dim, device=self.torch_device)
        _lib.check(self.lib.fo_fbank_offline(self._h, _ptr(pcm), self._pcm_dtype(pcm), B, N, self._scale(pcm, scale), _ptr(out),
                                             self._stream()))
        return out

    def _packed_pcm(self, pcms, n_samples):
        """(packed 1-D PCM, n_samples int64) from a list of 1-D int16 / float32 tensors or arrays, or a packed 1-D one plus
        n_samples.  A list with a CUDA tensor is packed on the engine's device, else on the host."""
        if n_samples is not None:
            ns = np.ascontiguousarray(np.asarray(n_samples.cpu() if isinstance(n_samples, torch.Tensor) else n_samples,
                                                 dtype=np.int64).reshape(-1))
            assert pcms.ndim == 1 and int(ns.sum()) == pcms.shape[0], "packed pcm must be 1-D with sum(n_samples) samples"
            return pcms, ns
        pcms = list(pcms)
        assert pcms and all(p.ndim == 1 for p in pcms), "pcms must be a non-empty list of 1-D signals"
        dts = {self._pcm_dtype(p) for p in pcms}
        assert len(dts) == 1, "all signals must share one dtype (int16 or float32)"
        ns = np.array([p.shape[0] for p in pcms], dtype=np.int64)
        if any(isinstance(p, torch.Tensor) for p in pcms):
            ts = [p if isinstance(p, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(p)) for p in pcms]
            dev = self.torch_device if any(t.is_cuda for t in ts) else torch.device("cpu")
            return torch.cat([t.to(dev) for t in ts]), ns
        return np.ascontiguousarray(np.concatenate(pcms)), ns

    def fbank_offline_packed(self, pcms, scale: Optional[float] = None, n_samples=None):
        """Filterbank of utterances of different lengths in one call.  Returns (feats (sum m_i, F), frame_offsets int64 (B + 1)):
        utterance i's frames are rows [off[i], off[i+1]), each bit-identical to fbank_offline of it alone."""
        pcm, ns = self._packed_pcm(pcms, n_samples)
        m = np.where(ns >= self.cfg.frame_len, 1 + (ns - self.cfg.frame_len) // self.cfg.frame_shift, 0)
        off = np.concatenate([[0], np.cumsum(m)]).astype(np.int64)
        out = torch.empty(int(off[-1]), self.cfg.feat_dim, device=self.torch_device)
        _lib.check(self.lib.fo_fbank_offline_packed(self._h, _ptr(pcm), self._pcm_dtype(pcm), ns.ctypes.data, len(ns),
                                                    self._scale(pcm, scale), _ptr(out), self._stream()))
        return out, off

    # ---- streaming --------------------------------------------------------------------------------
    def out_frames(self, t_in: int) -> Tuple[int, int]:
        t = PathConfig.sub_len(t_in)
        return t, self.adapter_frames(t)

    def adapter_frames(self, t: int) -> int:
        """Frames the adapter emits for t encoder frames: CNNSubsampling halves (stride-2 conv over k-1 cached frames),
        LinearAdapter keeps the rate."""
        if self.cfg.adapter_type in ("linear", "cnn"):
            return t
        k = self.cfg.adapter_kernel
        return (t + k - 1 - k) // 2 + 1

    def encode_stream(self, ids, feats: Optional[ArrayLike], want_adapter: Optional[bool] = None,
                      enc_out: Optional[torch.Tensor] = None, adapter_out: Optional[torch.Tensor] = None):
        """n sessions advance one chunk.  feats (n, t_in, F) or None (use the block left by fbank_stream)."""
        ids = _ids(ids)
        n = len(ids)
        t_in = self.cfg.chunk_feat_frames if feats is None else int(feats.shape[1])
        if feats is not None:
            assert tuple(feats.shape) == (n, t_in, self.cfg.feat_dim) and feats.dtype in (torch.float32, np.dtype(np.float32))
        t, t_out = self.out_frames(t_in)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc_out = self._out(enc_out, (n, t, self.cfg.d_model))
        if want_adapter:
            adapter_out = self._out(adapter_out, (n, t_out, self.cfg.llm_dim))
        _lib.check(self.lib.fo_encode_stream(self._h, _i32p(ids), n, _ptr(feats), t_in, _ptr(enc_out),
                                             _ptr(adapter_out) if want_adapter else None, self._stream()))
        return enc_out, (adapter_out if want_adapter else None)

    def encode_stream_chunks(self, ids, feats: ArrayLike, want_adapter: Optional[bool] = None,
                             enc_out: Optional[torch.Tensor] = None, adapter_out: Optional[torch.Tensor] = None):
        """n sessions advance k consecutive chunks in one step, with the results of k single-chunk encode_stream calls.
        feats (n, k, t_in, F): every block with its own context frames.  Returns enc (n, k, t, D) and adapter (n, k, t_out, E)."""
        ids = _ids(ids)
        n = len(ids)
        assert feats is not None and feats.ndim == 4, "feats must be (n, k, t_in, F)"
        k, t_in = int(feats.shape[1]), int(feats.shape[2])
        assert tuple(feats.shape) == (n, k, t_in, self.cfg.feat_dim) and feats.dtype in (torch.float32, np.dtype(np.float32))
        t, t_out = self.out_frames(t_in)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc_out = self._out(enc_out, (n, k, t, self.cfg.d_model))
        if want_adapter:
            adapter_out = self._out(adapter_out, (n, k, t_out, self.cfg.llm_dim))
        _lib.check(self.lib.fo_encode_stream_chunks(self._h, _i32p(ids), n, k, _ptr(feats), t_in, _ptr(enc_out),
                                                    _ptr(adapter_out) if want_adapter else None, self._stream()))
        return enc_out, (adapter_out if want_adapter else None)

    def encode_stream_chunks_v(self, ids, chunks, feats: ArrayLike, want_adapter: Optional[bool] = None,
                               enc_out: Optional[torch.Tensor] = None, adapter_out: Optional[torch.Tensor] = None):
        """Session ids[i] advances chunks[i] >= 1 consecutive chunks, all in one step, with the results of chunks[i]
        single-chunk encode_stream calls.  feats (B, t_in, F), B = sum(chunks), blocks in (session, chunk) order: session i's
        blocks start at chunks[0] + ... + chunks[i-1].  Returns enc (B, t, D) and adapter (B, t_out, E) in the same order."""
        ids = _ids(ids)
        n = len(ids)
        cnt = _ids(chunks)
        assert len(cnt) == n, "one chunk count per session"
        assert feats is not None and feats.ndim == 3, "feats must be (sum(chunks), t_in, F)"
        B, t_in = int(feats.shape[0]), int(feats.shape[1])
        assert B == int(cnt.sum()) and tuple(feats.shape) == (B, t_in, self.cfg.feat_dim)
        assert feats.dtype in (torch.float32, np.dtype(np.float32))
        t, t_out = self.out_frames(t_in)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc_out = self._out(enc_out, (B, t, self.cfg.d_model))
        if want_adapter:
            adapter_out = self._out(adapter_out, (B, t_out, self.cfg.llm_dim))
        _lib.check(self.lib.fo_encode_stream_chunks_v(self._h, _i32p(ids), _i32p(cnt), n, _ptr(feats), t_in, _ptr(enc_out),
                                                      _ptr(adapter_out) if want_adapter else None, self._stream()))
        return enc_out, (adapter_out if want_adapter else None)

    def stream_step(self, ids, pcm: ArrayLike, scale: Optional[float] = None, enc_out: Optional[torch.Tensor] = None,
                    adapter_out: Optional[torch.Tensor] = None, want_enc: bool = True):
        """PCM in, encoder frames + LLM-space embeddings out, one library call."""
        ids = _ids(ids)
        n = len(ids)
        assert tuple(pcm.shape) == (n, self.cfg.samples_per_chunk)
        t, t_out = self.out_frames(self.cfg.chunk_feat_frames)
        if want_enc:
            enc_out = self._out(enc_out, (n, t, self.cfg.d_model))
        if self.has_adapter:
            adapter_out = self._out(adapter_out, (n, t_out, self.cfg.llm_dim))
        _lib.check(self.lib.fo_stream_step(self._h, _i32p(ids), n, _ptr(pcm), self._pcm_dtype(pcm),
                                           self._scale(pcm, scale),
                                           _ptr(enc_out) if want_enc else None,
                                           _ptr(adapter_out) if self.has_adapter else None, self._stream()))
        return (enc_out if want_enc else None), (adapter_out if self.has_adapter else None)

    def stream_steps_v(self, ids, chunks, pcm: ArrayLike, scale: Optional[float] = None, want_adapter: Optional[bool] = None,
                       enc_out: Optional[torch.Tensor] = None, adapter_out: Optional[torch.Tensor] = None):
        """Recorded audio of any length: session ids[i] takes chunks[i] >= 1 consecutive chunks of PCM in one call, with the
        results and the session state of chunks[i] stream_step calls.  pcm (B, samples_per_chunk), B = sum(chunks), blocks in
        (session, chunk) order as in encode_stream_chunks_v.  Returns enc (B, t, D) and adapter (B, t_out, E) in that order."""
        ids = _ids(ids)
        n = len(ids)
        cnt = _ids(chunks)
        assert len(cnt) == n, "one chunk count per session"
        B = int(cnt.sum())
        assert tuple(pcm.shape) == (B, self.cfg.samples_per_chunk), "pcm must be (sum(chunks), samples_per_chunk)"
        t, t_out = self.out_frames(self.cfg.chunk_feat_frames)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc_out = self._out(enc_out, (B, t, self.cfg.d_model))
        if want_adapter:
            adapter_out = self._out(adapter_out, (B, t_out, self.cfg.llm_dim))
        _lib.check(self.lib.fo_stream_steps_v(self._h, _i32p(ids), _i32p(cnt), n, _ptr(pcm), self._pcm_dtype(pcm),
                                              self._scale(pcm, scale), _ptr(enc_out),
                                              _ptr(adapter_out) if want_adapter else None, self._stream()))
        return enc_out, (adapter_out if want_adapter else None)

    def fbank_stream_v(self, ids, chunks, pcm: ArrayLike, scale: Optional[float] = None,
                       out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The fbank half of stream_steps_v: session ids[i] takes chunks[i] >= 1 consecutive chunks of PCM (B, samples_per_chunk),
        B = sum(chunks), in (session, chunk) order.  Returns feats (B, t_in, F) in that order, every block with its context
        frames, and leaves sample carry and feature ring bit-identical to chunks[i] fbank_stream calls."""
        ids = _ids(ids)
        n = len(ids)
        cnt = _ids(chunks)
        assert len(cnt) == n, "one chunk count per session"
        B = int(cnt.sum())
        assert tuple(pcm.shape) == (B, self.cfg.samples_per_chunk), "pcm must be (sum(chunks), samples_per_chunk)"
        out = self._out(out, (B, self.cfg.chunk_feat_frames, self.cfg.feat_dim))
        _lib.check(self.lib.fo_fbank_stream_v(self._h, _i32p(ids), _i32p(cnt), n, _ptr(pcm), self._pcm_dtype(pcm),
                                              self._scale(pcm, scale), _ptr(out), self._stream()))
        return out

    def encode_stream_steps_v(self, ids, chunks, feats: ArrayLike, want_adapter: Optional[bool] = None,
                              enc_out: Optional[torch.Tensor] = None, adapter_out: Optional[torch.Tensor] = None):
        """The encoder half of stream_steps_v: session ids[i] advances by chunks[i] >= 1 blocks of feats (B, t_in, F), B =
        sum(chunks), in (session, chunk) order, with no cap on the counts (encode_stream_chunks_v stops at 128 keys).  On the
        features fbank_stream_v gave it is bit-identical to stream_steps_v.  Returns enc (B, t, D) and adapter (B, t_out, E)."""
        ids = _ids(ids)
        n = len(ids)
        cnt = _ids(chunks)
        assert len(cnt) == n, "one chunk count per session"
        assert feats is not None and feats.ndim == 3, "feats must be (sum(chunks), t_in, F)"
        B, t_in = int(feats.shape[0]), int(feats.shape[1])
        assert B == int(cnt.sum()) and tuple(feats.shape) == (B, t_in, self.cfg.feat_dim)
        assert feats.dtype in (torch.float32, np.dtype(np.float32))
        t, t_out = self.out_frames(t_in)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc_out = self._out(enc_out, (B, t, self.cfg.d_model))
        if want_adapter:
            adapter_out = self._out(adapter_out, (B, t_out, self.cfg.llm_dim))
        _lib.check(self.lib.fo_encode_stream_steps_v(self._h, _i32p(ids), _i32p(cnt), n, _ptr(feats), t_in, _ptr(enc_out),
                                                     _ptr(adapter_out) if want_adapter else None, self._stream()))
        return enc_out, (adapter_out if want_adapter else None)

    def stream_step_async(self, ids, pcm: ArrayLike, adapter_out: torch.Tensor, scale: Optional[float] = None,
                          enc_out: Optional[torch.Tensor] = None) -> int:
        """Pipelined stream_step for pinned HOST buffers: returns a ticket; `adapter_out` (and `enc_out`) are valid after
        stream_wait(ticket).  Copies of step i overlap the kernels of step i+1 (at most two steps outstanding)."""
        ids = _ids(ids)
        n = len(ids)
        assert tuple(pcm.shape) == (n, self.cfg.samples_per_chunk)
        t, t_out = self.out_frames(self.cfg.chunk_feat_frames)
        assert tuple(adapter_out.shape) == (n, t_out, self.cfg.llm_dim) and adapter_out.dtype == torch.float32 and adapter_out.is_contiguous()
        if enc_out is not None:
            assert tuple(enc_out.shape) == (n, t, self.cfg.d_model) and enc_out.dtype == torch.float32 and enc_out.is_contiguous()
        ticket = C.c_int64()
        _lib.check(self.lib.fo_stream_step_async(self._h, _i32p(ids), n, _ptr(pcm), self._pcm_dtype(pcm),
                                                 self._scale(pcm, scale), _ptr(enc_out),
                                                 _ptr(adapter_out), self._stream(), C.byref(ticket)))
        return int(ticket.value)

    def stream_wait(self, ticket: int) -> None:
        _lib.check(self.lib.fo_stream_wait(self._h, int(ticket)))

    def stream_step_embeds(self, ids, pcm: ArrayLike, embeds: torch.Tensor, row_offset: int = 0,
                           scale: Optional[float] = None, enc_out: Optional[torch.Tensor] = None, want_enc: bool = False):
        """stream_step whose adapter rows land, as fp16, in rows [row_offset, row_offset + t_out) of each session's block
        of `embeds` (n, rows, llm_dim) -- the pre-allocated inputs_embeds of the LLM step (audioLLM.py:404-411)."""
        ids = _ids(ids)
        n = len(ids)
        assert tuple(pcm.shape) == (n, self.cfg.samples_per_chunk)
        assert embeds.is_cuda and embeds.dtype == torch.float16 and embeds.is_contiguous()
        assert embeds.dim() == 3 and embeds.shape[0] >= n and embeds.shape[2] == self.cfg.llm_dim
        t, _ = self.out_frames(self.cfg.chunk_feat_frames)
        if want_enc:
            enc_out = self._out(enc_out, (n, t, self.cfg.d_model))
        _lib.check(self.lib.fo_stream_step_embeds(self._h, _i32p(ids), n, _ptr(pcm), self._pcm_dtype(pcm),
                                                  self._scale(pcm, scale),
                                                  _ptr(enc_out) if want_enc else None, embeds.data_ptr(),
                                                  int(embeds.shape[1]), int(row_offset), self._stream()))
        return (enc_out if want_enc else None), embeds

    def handoff_arm(self, n: int, embeds: torch.Tensor, prefix_len: int, onset, prefix_mask: Optional[torch.Tensor] = None,
                    attn_mask: Optional[torch.Tensor] = None, row_start: Optional[torch.Tensor] = None) -> None:
        """Arm the NEXT streaming call of n blocks (want_adapter=False) with the LLM hand-off of models/audioLLM.py:383-411:
        adapter rows as fp16 behind the chat prefix of each block of `embeds` (>= n, rows, llm_dim), attention-mask rows and
        input start rows on the device.  `onset`: n flags, status == 'ipu_sl'.  The call is encode_stream / stream_step (a block
        per session), encode_stream_chunks[_v], or one of the recording entries stream_steps_v / encode_stream_steps_v (block
        b is the b-th block of the call's (session, chunk) order, for any number of blocks).  encode_stream & co. consume the arm
        whatever their outcome; a recording entry that refuses the call (another block count, adapter_out given) leaves it armed."""
        assert embeds.is_cuda and embeds.dtype == torch.float16 and embeds.is_contiguous() and embeds.dim() == 3
        assert embeds.shape[0] >= n and embeds.shape[2] == self.cfg.llm_dim
        on = np.ascontiguousarray(np.asarray(onset, dtype=np.uint8).reshape(-1))
        assert len(on) == n
        R = int(embeds.shape[1])
        if attn_mask is not None:
            assert attn_mask.is_cuda and attn_mask.dtype == torch.uint8 and attn_mask.is_contiguous() and tuple(attn_mask.shape[-1:]) == (R,)
            assert attn_mask.numel() >= n * R
        if row_start is not None:
            assert row_start.is_cuda and row_start.dtype == torch.int32 and row_start.numel() >= n
        if prefix_mask is not None:
            assert prefix_mask.is_cuda and prefix_mask.dtype == torch.uint8 and prefix_mask.numel() == prefix_len
        _lib.check(self.lib.fo_handoff_arm(self._h, n, embeds.data_ptr(), R, int(prefix_len), on.ctypes.data, _ptr(prefix_mask),
                                           _ptr(attn_mask), _ptr(row_start)))

    # ---- offline ----------------------------------------------------------------------------------
    def encode_offline(self, feats: ArrayLike, ilens, chunk: Optional[int] = None, left: Optional[int] = None,
                       want_adapter: Optional[bool] = None):
        B, T, F = feats.shape
        assert F == self.cfg.feat_dim
        il = np.ascontiguousarray(np.asarray(ilens.cpu() if isinstance(ilens, torch.Tensor) else ilens, dtype=np.int32))
        chunk = self.cfg.chunk_size if chunk is None else int(chunk)
        left = self.cfg.left_chunks if left is None else int(left)
        t2, t3 = self.out_frames(T)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc = torch.empty(B, t2, self.cfg.d_model, device=self.torch_device)
        mask = torch.empty(B, t2, dtype=torch.uint8, device=self.torch_device)
        y = torch.empty(B, t3, self.cfg.llm_dim, device=self.torch_device) if want_adapter else None
        ymask = torch.empty(B, t3, dtype=torch.uint8, device=self.torch_device) if want_adapter else None
        _lib.check(self.lib.fo_encode_offline(self._h, _ptr(feats), il.ctypes.data, B, T, chunk, left, _ptr(enc),
                                              _ptr(mask), _ptr(y), _ptr(ymask), self._stream()))
        return enc, mask.bool().unsqueeze(1), y, (ymask.bool().unsqueeze(1) if want_adapter else None)

    def encode_offline_packed(self, feats: ArrayLike, lens, chunk: Optional[int] = None, left: Optional[int] = None,
                              want_adapter: Optional[bool] = None):
        """Utterances of different lengths packed end to end, no padding rows.  feats (sum T_i, F), lens (B) the T_i.
        Returns (enc (sum T'_i, D), adapter rows (sum T''_i, E) or None, enc_offsets, adapter_offsets); the offsets are
        int64 (B + 1) prefix sums, utterance i's rows being [off[i], off[i+1]).  Each utterance's rows equal the padded
        forward of it alone."""
        N, F = feats.shape
        assert F == self.cfg.feat_dim
        ln = np.ascontiguousarray(np.asarray(lens.cpu() if isinstance(lens, torch.Tensor) else lens, dtype=np.int32).reshape(-1))
        assert int(ln.sum()) == N, "lens must sum to the feature rows"
        chunk = self.cfg.chunk_size if chunk is None else int(chunk)
        left = self.cfg.left_chunks if left is None else int(left)
        eoff, aoff = self.cfg.packed_offsets(ln)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc = torch.empty(int(eoff[-1]), self.cfg.d_model, device=self.torch_device)
        y = torch.empty(int(aoff[-1]), self.cfg.llm_dim, device=self.torch_device) if want_adapter else None
        _lib.check(self.lib.fo_encode_offline_packed(self._h, _ptr(feats), ln.ctypes.data, len(ln), chunk, left, _ptr(enc), _ptr(y),
                                                     self._stream()))
        return enc, y, eoff, aoff

    def encode_offline_packed_pcm(self, pcms, chunk: Optional[int] = None, left: Optional[int] = None, scale: Optional[float] = None,
                                  want_adapter: Optional[bool] = None, want_feats: bool = False, n_samples=None):
        """PCM -> embeddings for utterances of different lengths, fbank included, in one call that runs in passes of bounded
        memory (option packed_pass_frames).  pcms as for fbank_offline_packed.  Returns (enc, adapter rows or None, enc_offsets,
        adapter_offsets[, feats]) as encode_offline_packed does, feats (sum m_i, F) being fbank_offline_packed's features."""
        pcm, ns = self._packed_pcm(pcms, n_samples)
        chunk = self.cfg.chunk_size if chunk is None else int(chunk)
        left = self.cfg.left_chunks if left is None else int(left)
        m, eoff, aoff = self.cfg.packed_audio_offsets(ns)
        want_adapter = self.has_adapter if want_adapter is None else want_adapter
        enc = torch.empty(int(eoff[-1]), self.cfg.d_model, device=self.torch_device)
        y = torch.empty(int(aoff[-1]), self.cfg.llm_dim, device=self.torch_device) if want_adapter else None
        feats = torch.empty(int(m.sum()), self.cfg.feat_dim, device=self.torch_device) if want_feats else None
        _lib.check(self.lib.fo_encode_offline_packed_pcm(self._h, _ptr(pcm), self._pcm_dtype(pcm), ns.ctypes.data, len(ns),
                                                         self._scale(pcm, scale), chunk, left, _ptr(enc), _ptr(y), _ptr(feats),
                                                         self._stream()))
        return (enc, y, eoff, aoff, feats) if want_feats else (enc, y, eoff, aoff)

    def adapter_forward(self, x: torch.Tensor, mask: Optional[torch.Tensor], cache):
        """Stateless adapter: x (B,T,D), mask (B,1,T)|(B,T) bool or None.  `cache`: None, a tensor (B,D,k-1) (single-conv
        CNNSubsampling), or the reference's list [c0 (B,2D,k-1), c1 (B,D,k-1)] for the two-conv branch (entries may be None
        on the first call, adapter.py:123-143).  Returns (y, new cache in the same form; None for cache-less adapters)."""
        B, T, D = x.shape
        k = self.cfg.adapter_kernel
        t_out = self.adapter_frames(T)
        x = x.detach().float().contiguous()
        m8 = None
        if mask is not None:
            m8 = mask.reshape(B, T).to(torch.uint8).contiguous()
        y = torch.empty(B, t_out, self.cfg.llm_dim, device=self.torch_device)
        if self.cfg.adapter_type in ("linear", "cnn"):         # no cache to carry
            assert cache is None
            _lib.check(self.lib.fo_adapter_forward2(self._h, _ptr(x), _ptr(m8), B, T, None, None, None, None, _ptr(y), self._stream()))
            return y, None
        if self.cfg.adapter_two_conv:
            c0, c1 = (None, None) if cache is None else (cache[0], cache[1])
            c0 = None if c0 is None else c0.detach().float().contiguous()
            c1 = None if c1 is None else c1.detach().float().contiguous()
            assert (c0 is None) == (c1 is None), "the two cache entries are set together (adapter.py:128-141)"
            o0 = torch.empty(B, 2 * D, k - 1, device=self.torch_device)
            o1 = torch.empty(B, D, k - 1, device=self.torch_device)
            _lib.check(self.lib.fo_adapter_forward2(self._h, _ptr(x), _ptr(m8), B, T, _ptr(c0), _ptr(c1), _ptr(o0), _ptr(o1), _ptr(y),
                                                    self._stream()))
            return y, [o0, o1]
        ci = None if cache is None else cache.detach().float().contiguous()
        co = torch.empty(B, D, k - 1, device=self.torch_device)
        _lib.check(self.lib.fo_adapter_forward(self._h, _ptr(x), _ptr(m8), B, T, _ptr(ci), _ptr(co), _ptr(y), self._stream()))
        return y, co

    def debug_gemm(self, A: torch.Tensor, W: torch.Tensor, bias: Optional[torch.Tensor] = None, backend: int = 0,
                   relu: bool = False, iters: int = 0):
        M, K = A.shape
        N = W.shape[0]
        out = torch.empty(M, N, device=self.torch_device)
        ms = C.c_float()
        _lib.check(self.lib.fo_debug_gemm(self._h, _ptr(A), _ptr(W), _ptr(bias), _ptr(out), M, N, K, backend, int(relu),
                                          iters, C.byref(ms), self._stream()))
        return out, float(ms.value)

    def debug_sm_ids(self, n_ctas: int, graph: bool = False) -> torch.Tensor:
        """The SM ids that n_ctas CTAs launched as this context launches its kernels ran on (int32, on the device); with
        `graph` the launch is captured into a graph on the context's capture stream and replayed, as a streaming step is."""
        out = torch.empty(n_ctas, dtype=torch.int32, device=self.torch_device)
        _lib.check(self.lib.fo_debug_sm_ids(self._h, int(n_ctas), int(graph), _ptr(out), self._stream()))
        return out

    def debug_attention(self, mode: str, qkv: Optional[torch.Tensor], ptab: torch.Tensor, pos_u: torch.Tensor,
                        pos_v: torch.Tensor, *, seq=None, T: int = 0, gap: int = 0, chunk: int = 0, left: int = -1, t: int = 0,
                        layer: int = 0, cnt=None, off0: int = 0, group: int = 1, part: Optional[torch.Tensor] = None,
                        part_bias: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One attention launcher of the library (fo_debug_attention) on fp32 device tensors; returns out (rows, D) fp32.
        mode "offline" (seq = ilens, T), "packed" (seq = lens, gap), "stream" (seq = session ids, t, layer; optional split-K
        partials `part` (nsplit, rows, 3D) with `part_bias`), "chunks" (seq = ids, cnt, off0 = off[0], t, layer, group).
        chunk / left: the offline band."""
        m = {"offline": _lib.FO_ATT_OFFLINE, "packed": _lib.FO_ATT_PACKED, "stream": _lib.FO_ATT_STREAM,
             "chunks": _lib.FO_ATT_CHUNKS}[mode]
        s = _ids(seq)
        n = len(s)
        cn = offs = None
        if mode == "offline":
            rows = n * T
        elif mode == "packed":
            rows = int(s.sum()) + (n - 1) * gap
        elif mode == "stream":
            rows = n * t
        else:
            cn = _ids(cnt)
            offs = np.ascontiguousarray(off0 + np.concatenate([[0], np.cumsum(cn)[:-1]]).astype(np.int32))
            rows = int(cn.sum()) * t
        for x in (qkv, ptab, pos_u, pos_v, part, part_bias):
            assert x is None or (x.is_cuda and x.dtype == torch.float32 and x.is_contiguous())
        nsplit = 0 if part is None else int(part.shape[0])
        out = torch.empty(max(rows, 1), self.cfg.d_model, device=self.torch_device)[:rows]
        _lib.check(self.lib.fo_debug_attention(
            self._h, m, n, _i32p(s), None if cn is None else _i32p(cn), None if offs is None else _i32p(offs), int(T), int(gap),
            int(chunk), int(left), int(t), int(layer), int(group), _ptr(qkv), _ptr(part), nsplit, _ptr(part_bias), _ptr(ptab),
            int(ptab.shape[0]), _ptr(pos_u), _ptr(pos_v), _ptr(out), self._stream()))
        return out
