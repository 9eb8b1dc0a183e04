"""Each attention kernel of the library, fp32 and bf16 contexts, against an exact fp64 reference of its own inputs
(fo_debug_attention: one launcher on caller-given tensors).

Reference.  The masks are O.chunk_window / O.offline_attention_mask (band and pad mask; a row whose keys are all masked
gives zeros), the scores O.attention_scores: ((q+u).k_j + (q+v).p_pos(j)) / 8, softmax, sum_j p_j v_j.  Streaming keys are
the last min(n_frames, window) frames plus the chunk's t, rel-pos rows from start = max(0, pe % pe_wrap - full_chunk), pe
stepping by chunk_size per chunk (EncoderOracle.infer).  The reference applies the kernels' deterministic input roundings
and nothing else: in bf16 contexts (fp16 activations) K, V and P are rounded to fp16, (q+u) and (q+v) are summed in fp32
and then rounded to fp16; the split-K route sums its partials in fp32 in the kernel's order (0..n-1, then the bias).
Everything after that is fp64.  test_reference_matches_oracle pins it, roundings off, to the oracle's own functions.

Error bound, per output element o_id of query row i (derivation; first order in the unit roundoffs):
  - scores: every score is an fp32 dot product of 128 terms (64 for K, 64 for P) accumulated in fp32 (FFMA chain or
    mma.sync accumulator): |ds_j| <= 128 * 2^-24 * S_ij = 2^-17 * S_ij with S_ij = sum_d |(q+u)_d k_jd| + |(q+v)_d p_jd|, / 8.
    The exponentials (__expf, ex2.approx of the exp2-domain score) add about 2^-22 relative plus the argument's rounding,
    2^-23 |s|; each online-softmax tile adds one more rescale exponential.  So ds = 2^-17 max_j S_ij
    + 2^-21 (2 + nk / 64) + 2^-22 max_j |s_ij|.  A perturbation e_j of the scores moves p_j by p_j (e_j - sum_k p_k e_k), so
    |d o| <= sum_j p_j |e_j - e_mean| |v_j - o| <= 2 ds sqrt(sum_j p_j (v_j - o)^2)  (Cauchy-Schwarz, sum_j p_j = 1).
  - fp32 accumulation of sum_j p_j v_j and of the normaliser over nk keys: (nk + 8) 2^-24 (A + |o|), A = max |v| over
    the row's keys.
  - fp16 only: every probability is rounded to fp16 before the PV product (relative 2^-11, or 2^-25 absolute below the
    normal range): 2^-11 A + nk 2^-25 A; the output is rounded to fp16: 2^-11 |o| + 2^-25.
  - fp32 only: the output's last rounding 2^-24 |o|.
A row with no key outputs exactly 0 (bound 0).  The worst err / bound ratio per mode and precision is printed; in the
ordinary regime the bound stays below 2.5e-3 max|V| (fp16) and 1e-3 max|V| (fp32; this bound is worst case: 128-term fp32
score chains and up to pos_max_len-term PV sums, DESIGN 2).

Exact checks where the code says the arithmetic is the same: a packed utterance equals a padded call of it alone; a
chunks call of k chunks equals k stream calls (outputs and ring); several groups per session (plus the ring-append
kernel) equal one group; the split-K partials route equals the finished-rows route given the same sums.
"""
import dataclasses
import math

import numpy as np
import pytest
import torch

from freeze_omni_b200.config import load_path_config
from oracle import freeze_omni_oracle as O

ROWS = [(4, 16), (4, 2), (3, 1), (3, 5), (2, 8), (1, 16), (8, 8), (4, 31), (4, -1)]     # test_gpu_stream_chunkings.ROWS
CAPS = ["tight", "default"]
OFF_T = [1, 7, 31, 32, 33, 63, 64, 65, 129, 748]
BANDS = [(4, 16), (4, -1), (-1, -1), (1, 0), (3, 1), (7, 3), (8, 8), (64, 1), (100, 2)]
REGIMES = ["ordinary", "peaked", "ramp", "voffset"]
BOUND_CAP = {True: 2.5e-3, False: 1e-3}          # ordinary regime: max bound / max|V|, fp16 / fp32
MAX_KEYS = 128
DK = 64

WORST = {}                                       # (mode, precision) -> [worst err / bound, worst ordinary bound / max|V|]


def note(mode, f16, ratio, bnd):
    w = WORST.setdefault((mode, "bf16" if f16 else "fp32"), [0.0, 0.0])
    w[0] = max(w[0], ratio)
    w[1] = max(w[1], bnd)


# ---- reference ------------------------------------------------------------------------------------------------------------
def r16(x, f16):
    """The kernels' rounding of an fp32 operand: fp16 round-to-nearest in 16-bit contexts (as from_f<__half>), else as is."""
    x = x.float()
    return (x.clamp(-65504, 65504).half() if f16 else x).double()


def biased(q, bias, f16):
    """(q + bias) summed in fp32, then rounded as the kernels round it."""
    return r16(q.float() + bias.float(), f16)


def ref_attend(qu, qv, k, v, p, allowed, f16, rounded=True):
    """softmax(((q+u) K^T + (q+v) P^T) / 8) V in fp64 over (..., Nq, Nk); allowed (..., Nq, Nk) bool or None (every key).
    Returns (out, bound) with the bound of the module docstring (f16 selects the fp16 terms); rows without keys give 0."""
    s = (qu @ k.mT + qv @ p.mT) / 8
    al = torch.ones_like(s, dtype=torch.bool) if allowed is None else allowed.expand(s.shape)
    s = s.masked_fill(~al, -math.inf)
    live = al.any(-1, keepdim=True)
    pr = torch.softmax(s.masked_fill(~live, 0.0), -1) * live
    o = pr @ v
    if not rounded:
        return o, None
    terms = (qu.abs() @ k.abs().mT + qv.abs() @ p.abs().mT) / 8
    nk = al.sum(-1, keepdim=True).double()
    A = torch.where(al, v.abs().amax(-1).unsqueeze(-2), 0.0).amax(-1, keepdim=True)
    smax = torch.where(al, s.abs(), 0.0).amax(-1, keepdim=True)
    tmax = torch.where(al, terms, 0.0).amax(-1, keepdim=True)
    ds = 2.0 ** -17 * tmax + 2.0 ** -21 * (2 + nk / 64) + 2.0 ** -22 * smax
    dev = (pr @ (v * v) - o * o).clamp(min=0).sqrt()
    b = 2 * ds * dev + (nk + 8) * 2.0 ** -24 * (A + o.abs())
    if f16:
        b = b + 2.0 ** -11 * (A + o.abs()) + nk * 2.0 ** -25 * A + 2.0 ** -25
    else:
        b = b + 2.0 ** -24 * o.abs()
    return o, torch.where(live, b, 0.0)


def heads(x, H):
    """(rows, H*64) -> (H, rows, 64)"""
    return x.view(x.shape[0], H, DK).transpose(0, 1)


def ref_offline(qkv, ptab, pos_u, pos_v, H, T, ilen, chunk, left, f16, rounded=True):
    """One utterance of T rows (qkv (T, 3D) fp32) with ilen valid keys: (out (T, D), bound (T, D))."""
    D = H * DK
    q, k, v = heads(qkv[:, :D], H), heads(qkv[:, D:2 * D], H), heads(qkv[:, 2 * D:], H)
    u, w = pos_u.view(H, 1, DK), pos_v.view(H, 1, DK)
    p = heads(ptab[:T], H)
    if rounded:
        qu, qv, k, v, p = biased(q, u, f16), biased(q, w, f16), r16(k, f16), r16(v, f16), r16(p, f16)
    else:
        qu, qv, k, v, p = q.double() + u.double(), q.double() + w.double(), k.double(), v.double(), p.double()
    valid = (torch.arange(T) < ilen).view(1, 1, T)
    mask = O.offline_attention_mask(valid, chunk, left).to(qkv.device)                       # (1, T, T) or (1, 1, T)
    o, b = ref_attend(qu, qv, k, v, p, mask, f16, rounded)
    o = o.transpose(0, 1).reshape(T, D)
    return o, (None if b is None else b.transpose(0, 1).reshape(T, D))


@dataclasses.dataclass
class Geo:
    """Streaming geometry of a context (fo_create)."""
    window: int
    full_chunk: int
    pe_wrap: int
    chunk_size: int

    @staticmethod
    def of(cfg):
        return Geo(cfg.kv_window, cfg.full_chunk_size, cfg.pe_wrap, cfg.chunk_size)


def ref_chunks(qkv, kw, vw, nf, pe, ptab, pos_u, pos_v, H, t, geo, f16, rounded=True):
    """k = rows / t consecutive chunks of one session: qkv (k*t, 3D) fp32; kw, vw (H, cl, 64) the ring window (the last
    cl = min(nf, window) frames, values as stored); pe its pe_index.  Returns (out, bound, K and V of every frame the call
    saw, (H, cl + k*t, 64), as stored)."""
    D = H * DK
    rnd = (lambda x: r16(x, f16)) if rounded else (lambda x: x.double())
    hk = torch.cat([kw.double(), rnd(heads(qkv[:, D:2 * D], H))], 1)
    hv = torch.cat([vw.double(), rnd(heads(qkv[:, 2 * D:], H))], 1)
    base = nf - kw.shape[1]                                                 # frame number of hk[:, 0]
    outs, bnds = [], []
    for j in range(qkv.shape[0] // t):
        pe = pe % geo.pe_wrap                                               # EncoderOracle.infer
        start = max(0, pe - geo.full_chunk)
        pe += geo.chunk_size
        nfj = nf + j * t
        f0 = nfj - min(nfj, geo.window)
        nk = nfj + t - f0
        q = heads(qkv[j * t:(j + 1) * t, :D], H)
        u, w = pos_u.view(H, 1, DK), pos_v.view(H, 1, DK)
        qu, qv = (biased(q, u, f16), biased(q, w, f16)) if rounded else (q.double() + u.double(), q.double() + w.double())
        p = rnd(heads(ptab[start:start + nk], H))
        o, b = ref_attend(qu, qv, hk[:, f0 - base:f0 - base + nk], hv[:, f0 - base:f0 - base + nk], p, None, f16, rounded)
        outs.append(o.transpose(0, 1).reshape(t, D))
        bnds.append(None if b is None else b.transpose(0, 1).reshape(t, D))
    return torch.cat(outs), (None if rounded is False else torch.cat(bnds)), hk, hv


# ---- inputs ---------------------------------------------------------------------------------------------------------------
def make_inputs(regime, rows, H, prow, gen, device):
    """qkv (rows, 3D), ptab (prow, D), pos_u, pos_v (D), fp32 on `device`.  ordinary: scores of std ~3; peaked: std ~15;
    ramp: the rel-pos term rises 0.1 per position (mod 256), so every later key tile raises the running max; voffset: V =
    50 + N(0, 1)."""
    D = H * DK
    sig = {"ordinary": 1.45, "peaked": 3.26, "ramp": 1.45, "voffset": 1.45}[regime]
    qkv = torch.randn(rows, 3 * D, generator=gen) * sig
    qkv[:, 2 * D:] /= sig
    ptab = torch.randn(prow, D, generator=gen) * sig
    pu, pv = 0.3 * torch.randn(D, generator=gen), 0.3 * torch.randn(D, generator=gen)
    if regime == "ramp":
        qkv[:, 0:D:DK] = 0.0
        pv[0::DK] = 8.0
        ptab[:, 0::DK] = 0.1 * (torch.arange(prow) % 256).float().unsqueeze(1)
    if regime == "voffset":
        qkv[:, 2 * D:] += 50.0
    return [x.contiguous().to(device) for x in (qkv, ptab, pu, pv)]


def window_kv(regime, H, cl, gen, f16):
    """Ring contents of a session (H, cl, 64) K and V, exactly representable in the context's type."""
    sig = {"ordinary": 1.45, "peaked": 3.26, "ramp": 1.45, "voffset": 1.45}[regime]
    k = torch.randn(H, cl, DK, generator=gen) * sig
    v = torch.randn(H, cl, DK, generator=gen) + (50.0 if regime == "voffset" else 0.0)
    if f16:
        k, v = k.half().float(), v.half().float()
    return k, v


def pos_rows_of(cfg, max_t):
    """Rows of the context's rel-pos tables (fo_create)."""
    r = cfg.pos_max_len
    if cfg.chunk_size > 0:
        r = max(r, max(0, cfg.pe_wrap - 1 - cfg.full_chunk_size) + cfg.kv_window + max_t)
    return r


def check(mode, f16, got, want, bound, maxv, regime, tag):
    err = (got.double() - want).abs()
    ratio = float((err / bound.clamp(min=1e-300)).max()) if err.numel() else 0.0
    bad = err > bound
    assert not bool(bad.any()), (tag, "worst err / bound %.3g" % ratio, float(err.max()), torch.nonzero(bad)[:4].tolist())
    nb = float(bound.max() / maxv) if regime == "ordinary" and bound.numel() else 0.0
    note(mode, f16, ratio, nb)
    if regime == "ordinary":
        assert nb < BOUND_CAP[f16], (tag, nb)


# ---- CPU: the reference is the oracle's arithmetic ------------------------------------------------------------------------
def _oracle_attention(q, k, v, pos_emb, u, w, mask):
    """The oracle's attention of one call (heads split): O.attention_scores with an identity linear_pos, then the masked
    softmax of layer_offline (masked_fill(MIN_VALUE) -> softmax -> masked_fill(0))."""
    H, D = u.shape[0], u.shape[0] * DK
    sd = {"a.linear_pos.weight": torch.eye(D, dtype=torch.float64), "a.pos_bias_u": u, "a.pos_bias_v": w}
    s = O.attention_scores(sd, "a.", q, k, pos_emb, H)
    if mask is None:
        return torch.softmax(s, -1) @ v
    dead = mask.unsqueeze(1).eq(0)
    return torch.softmax(s.masked_fill(dead, O.MIN_VALUE), -1).masked_fill(dead, 0.0) @ v


def test_reference_matches_oracle():
    """With the roundings off, ref_offline / ref_chunks compute the oracle's functions: masks, scores, softmax, the streaming
    key window and rel-pos rows across a pe wrap inside a multi-chunk call."""
    gen = torch.Generator().manual_seed(11)
    H, D = 2, 128
    for T, ilen, (chunk, left) in ((33, 20, (4, 2)), (70, 70, (-1, -1)), (40, 1, (8, 0)), (65, 64, (3, -1))):
        qkv, ptab, u, w = make_inputs("ordinary", T, H, T, gen, "cpu")
        got, _ = ref_offline(qkv, ptab, u, w, H, T, ilen, chunk, left, False, rounded=False)
        x = qkv.double().unsqueeze(0)
        valid = (torch.arange(T) < ilen).view(1, 1, T)
        want = _oracle_attention(O._split_heads(x[..., :D], H), O._split_heads(x[..., D:2 * D], H), O._split_heads(x[..., 2 * D:], H),
                                 ptab.double().unsqueeze(0), u.double().view(H, DK), w.double().view(H, DK),
                                 O.offline_attention_mask(valid, chunk, left))
        assert torch.allclose(got, want[0].transpose(0, 1).reshape(T, D), rtol=0, atol=1e-12), (T, chunk, left)
    cfg = dataclasses.replace(load_path_config("tiny"), chunk_size=4, left_chunks=2, pos_max_len=60)
    geo = Geo.of(cfg)
    t = 4
    for nf, pe, k in ((0, 0, 3), (5, geo.pe_wrap - 4, 4), (30, geo.pe_wrap - 1, 2)):
        cl = min(nf, geo.window)
        qkv, ptab, u, w = make_inputs("ordinary", k * t, H, pos_rows_of(cfg, t), gen, "cpu")
        kw, vw = window_kv("ordinary", H, cl, gen, False)
        got, _, _, _ = ref_chunks(qkv, kw, vw, nf, pe, ptab, u, w, H, t, geo, False, rounded=False)
        # the oracle's loop: one infer-style step per chunk, cache trimmed to the window after each (layer_stream)
        x = qkv.double().unsqueeze(0)
        kv = [kw.double().unsqueeze(0), vw.double().unsqueeze(0)] if cl else None
        p = pe
        for j in range(k):
            p = p % cfg.pe_wrap
            start = max(0, p - cfg.full_chunk_size)
            n_cache = 0 if kv is None else kv[0].shape[2]
            pos = ptab[start:start + n_cache + t].double().unsqueeze(0)
            p += cfg.chunk_size
            xs = x[:, j * t:(j + 1) * t]
            kk, vv = O._split_heads(xs[..., D:2 * D], H), O._split_heads(xs[..., 2 * D:], H)
            if kv is not None:
                kk, vv = torch.cat([kv[0], kk], 2), torch.cat([kv[1], vv], 2)
            o = _oracle_attention(O._split_heads(xs[..., :D], H), kk, vv, pos, u.double().view(H, DK), w.double().view(H, DK), None)
            kv = [kk[:, :, -geo.window:], vv[:, :, -geo.window:]]
            assert torch.allclose(got[j * t:(j + 1) * t], o[0].transpose(0, 1).reshape(t, D), rtol=0, atol=1e-12), (nf, pe, j)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
_ENGINES = {}


@pytest.fixture(scope="module")
def engines():
    from freeze_omni_b200.engine import Engine
    from freeze_omni_b200.weights import make_encoder_state

    def get(name, f16, c=4, left=16, cap="default"):
        key = (name, f16, c, left, cap)
        if key not in _ENGINES:
            if name == "shipped":                # shipped attention geometry, one layer, small FFN: cheap to build
                cfg = dataclasses.replace(load_path_config("shipped"), n_layers=1, ffn_dim=256)
            else:
                cfg = dataclasses.replace(load_path_config("tiny"), chunk_size=c, left_chunks=left)
            msf = 4 * min(c, 8) + 3 if cap == "tight" else 35      # t = 8 needs max_stream_frames 35
            eng = Engine(cfg, make_encoder_state(cfg, 3), None, dtype=torch.bfloat16 if f16 else torch.float32,
                         max_sessions=12, max_stream_frames=msf)
            _ENGINES[key] = (cfg, eng)
        return _ENGINES[key]
    yield get
    for _, eng in _ENGINES.values():
        eng.close()
    _ENGINES.clear()
    if WORST:
        print("\nworst err/bound and ordinary-regime bound/max|V| per mode and precision:")
        for (mode, prec), (r, b) in sorted(WORST.items()):
            print("  %-8s %-5s err/bound %.3g  bound/max|V| %.3g" % (mode, prec, r, b))


def _gen(*key):
    return torch.Generator().manual_seed(hash(key) % (2 ** 31))


@pytest.mark.gpu
@pytest.mark.parametrize("f16", [False, True], ids=["fp32", "bf16"])
@pytest.mark.parametrize("name", ["tiny", "shipped"])
def test_offline_padded(engines, name, f16):
    """Padded batches: utterances of T' rows with ragged ilens (T', 1, a middle length), every row checked (padded query
    rows too: masks.py gives them the band of their position over the valid keys)."""
    cfg, eng = engines(name, f16)
    H, D = cfg.n_heads, cfg.d_model
    prow = pos_rows_of(cfg, eng.max_t)
    Ts = OFF_T + ([cfg.pos_max_len] if name == "tiny" else [])
    for T in Ts:
        bands = BANDS if T < 1000 else [(4, 16), (-1, -1), (64, 1)]
        for chunk, left in bands:
            for regime in REGIMES:
                gen = _gen("off", name, T, chunk, left, regime)
                ilens = [T, 1, max(1, (T * 5) // 9)] if T < 1000 else [T, T // 3]
                B = len(ilens)
                qkv, ptab, u, w = make_inputs(regime, B * T, H, prow, gen, "cuda")
                out = eng.debug_attention("offline", qkv, ptab, u, w, seq=ilens, T=T, chunk=chunk, left=left)
                maxv = float(qkv[:, 2 * D:].abs().max())
                for b, il in enumerate(ilens):
                    want, bnd = ref_offline(qkv[b * T:(b + 1) * T], ptab, u, w, H, T, il, chunk, left, f16)
                    check("offline", f16, out[b * T:(b + 1) * T], want, bnd, maxv, regime, (name, T, il, chunk, left, regime))


@pytest.mark.gpu
@pytest.mark.parametrize("f16", [False, True], ids=["fp32", "bf16"])
@pytest.mark.parametrize("name", ["tiny", "shipped"])
def test_offline_packed(engines, name, f16):
    """Packed calls: many utterances of lengths straddling the 32- and 64-query tiles, one long one among short ones, gap
    rows of large finite values between them.  Every utterance against the reference and, bit for bit, against a padded call
    of it alone."""
    cfg, eng = engines(name, f16)
    H, D = cfg.n_heads, cfg.d_model
    prow = pos_rows_of(cfg, eng.max_t)
    sets = [[1, 31, 32, 33, 63, 64, 65, 96, 97, 129], [7, 748, 2, 65, 33], [200, 1, 1, 64]]
    for li, lens in enumerate(sets):
        for gap in (0, 3):
            for chunk, left in ((4, 16), (-1, -1), (3, 1), (64, 1), (1, 0)):
                for regime in ("ordinary", "ramp") if (gap, chunk) != (0, 4) else REGIMES:
                    gen = _gen("pk", name, li, gap, chunk, left, regime)
                    rows = sum(lens) + gap * (len(lens) - 1)
                    qkv, ptab, u, w = make_inputs(regime, rows, H, prow, gen, "cuda")
                    offs = np.concatenate([[0], np.cumsum(np.asarray(lens) + gap)])[:-1]
                    for b, L in enumerate(lens[:-1]):
                        qkv[offs[b] + L:offs[b] + L + gap] = 1.0e4                   # gap rows: never a key or a query
                    out = eng.debug_attention("packed", qkv, ptab, u, w, seq=lens, gap=gap, chunk=chunk, left=left)
                    maxv = float(qkv[:, 2 * D:].abs().max()) if gap == 0 else 60.0
                    for b, L in enumerate(lens):
                        r0 = int(offs[b])
                        want, bnd = ref_offline(qkv[r0:r0 + L], ptab, u, w, H, L, L, chunk, left, f16)
                        check("packed", f16, out[r0:r0 + L], want, bnd, max(maxv, 1e-30), regime if gap == 0 else "x",
                              (name, lens, b, gap, chunk, left, regime))
                        alone = eng.debug_attention("offline", qkv[r0:r0 + L].contiguous(), ptab, u, w, seq=[L], T=L, chunk=chunk,
                                                    left=left)
                        assert torch.equal(out[r0:r0 + L], alone), ("packed != padded alone", name, lens, b, chunk, left)
                        if b + 1 < len(lens) and gap:
                            assert not out[r0 + L:r0 + L + gap].any(), "gap rows are written by no query"


# ---- streaming ------------------------------------------------------------------------------------------------------------
class Streamer:
    """Sessions of one engine placed at chosen (n_frames, pe_index, ring window) and checked after debug calls."""

    def __init__(self, cfg, eng, f16, layer=0):
        self.cfg, self.eng, self.f16, self.layer = cfg, eng, f16, layer
        self.geo = Geo.of(cfg)
        self.H, self.D = cfg.n_heads, cfg.d_model
        self.cap = eng.get_option("ring_cap")
        self.ids = eng.alloc(10)
        self.state = {}

    def place(self, sid, nf, pe, regime, gen):
        cl = min(nf, self.geo.window)
        kw, vw = window_kv(regime, self.H, cl, gen, self.f16)
        self.put(sid, nf, pe, kw, vw)
        return kw, vw

    def put(self, sid, nf, pe, kw, vw):
        sid = int(sid)
        self.eng.set_frames(sid, nf)
        self.eng.set_pe_index([sid], pe)
        if kw.shape[1]:
            self.eng.import_kv(sid, self.layer, kw.unsqueeze(0), vw.unsqueeze(0))
        self.state[sid] = (nf, pe, kw, vw)

    def ring(self, sid):
        k, v = self.eng.export_kv(int(sid), self.layer)
        return k[0], v[0]

    def advance(self, sid, frames, hk, hv):
        """n_frames += frames (pe_index is not read by the checks that follow); the exported window must be the last
        frames the call saw, exactly."""
        nf = self.state[int(sid)][0] + frames
        self.eng.set_frames(int(sid), nf)
        cl = min(nf, self.geo.window)
        k, v = self.ring(sid)
        assert k.shape[1] == cl
        assert torch.equal(k.double(), hk[:, hk.shape[1] - cl:].cpu()) and torch.equal(v.double(), hv[:, hv.shape[1] - cl:].cpu()), \
            ("ring after the call", sid)

    def ref(self, sid, qkv, t):
        nf, pe, kw, vw = self.state[int(sid)]
        g = qkv.device
        return ref_chunks(qkv, kw.to(g), vw.to(g), nf, pe, self.ptab, self.u, self.w, self.H, t, self.geo, self.f16)


def placements(geo, cap, t, k=1):
    """(n_frames, pe_index) of four sessions: empty ring, below the window, at the window, past it with the window copy
    split in two runs of the ring; pe_index 0, below full_chunk, at pe_wrap - 1 (and its wrap inside a multi-chunk call)."""
    w = geo.window
    split = w + (cap - max(1, min(w, cap) // 2)) + 3 * cap if w > 1 else 3 * cap + 1
    return [(0, 0), (max(1, w // 2), max(0, geo.full_chunk // 2)), (w, geo.pe_wrap - 1), (split, geo.pe_wrap - geo.chunk_size * max(1, k - 1))]


def _setup(st, regime, t, rows, gen):
    qkv, ptab, u, w = make_inputs(regime, rows, st.H, pos_rows_of(st.cfg, st.eng.max_t), gen, "cuda")
    st.ptab, st.u, st.w = ptab, u, w
    return qkv


def run_stream(st, regime, t, tag):
    """One stream call of four non-contiguous sessions (a fifth, outside ids, must keep its ring), each against the
    reference; ring checks; then each session again as a chunks call of one chunk on a twin slot, bit for bit."""
    geo, f16, eng = st.geo, st.f16, st.eng
    gen = _gen("st", tag, regime, t)
    sids = [st.ids[5], st.ids[1], st.ids[8], st.ids[3]]
    other = st.ids[0]
    st.place(other, 2 * geo.window + 5, 7, regime, gen)
    before = st.ring(other)
    for sid, (nf, pe) in zip(sids, placements(geo, st.cap, t)):
        st.place(sid, nf, pe, regime, gen)
    qkv = _setup(st, regime, t, 4 * t, gen)
    out = eng.debug_attention("stream", qkv, st.ptab, st.u, st.w, seq=sids, t=t, layer=st.layer)
    maxv = max(float(qkv[:, 2 * st.D:].abs().max()), max(float(st.state[int(s)][3].abs().max()) if st.state[int(s)][3].numel() else 0.0
                                                          for s in sids))
    saved = {}
    for i, sid in enumerate(sids):
        want, bnd, hk, hv = st.ref(sid, qkv[i * t:(i + 1) * t], t)
        check("stream", f16, out[i * t:(i + 1) * t], want, bnd, maxv, regime, (tag, regime, t, i))
        saved[int(sid)] = st.state[int(sid)]
        st.advance(sid, t, hk, hv)
    k, v = st.ring(other)
    assert torch.equal(k, before[0]) and torch.equal(v, before[1]), "a slot outside ids is unchanged"
    # the same chunks through the multi-chunk kernel (one chunk each, off[0] != 0): the same core on the same staged values
    for sid in sids:
        nf, pe, kw, vw = saved[int(sid)]
        st.put(sid, nf, pe, kw, vw)
    out2 = eng.debug_attention("chunks", qkv, st.ptab, st.u, st.w, seq=sids, cnt=[1] * 4, off0=5, t=t, layer=st.layer, group=1)
    assert torch.equal(out, out2), ("stream != chunks of one", tag, regime, t)
    if f16:
        run_partials(st, sids, saved, qkv, out, regime, t, tag)


def run_partials(st, sids, saved, qkv, out_ref, regime, t, tag):
    """The split-K route: partials summed in the kernel's order give bit for bit the finished-rows route's output and ring."""
    gen = _gen("part", tag, regime, t)
    rows, D3 = qkv.shape[0], qkv.shape[1]
    for nsplit in (2, 4):
        part = (torch.randn(nsplit, rows, D3, generator=gen) * 0.7).cuda()
        part[0] += qkv
        bias = (0.1 * torch.randn(D3, generator=gen)).cuda()
        s = part[0].clone()
        for i in range(1, nsplit):
            s = s + part[i]
        s = s + bias
        for sid in sids:
            st.put(sid, *saved[int(sid)])
        got = st.eng.debug_attention("stream", None, st.ptab, st.u, st.w, seq=sids, t=t, layer=st.layer, part=part.contiguous(),
                                     part_bias=bias)
        rings = []
        for sid in sids:
            st.eng.set_frames(int(sid), saved[int(sid)][0] + t)
            rings.append(st.ring(sid))
            st.put(sid, *saved[int(sid)])
        fin = st.eng.debug_attention("stream", s.contiguous(), st.ptab, st.u, st.w, seq=sids, t=t, layer=st.layer)
        for sid in sids:
            st.eng.set_frames(int(sid), saved[int(sid)][0] + t)
        assert torch.equal(got, fin), ("partials != finished rows", nsplit, tag, t)
        maxv = float(s[:, 2 * st.D:].abs().max()) + 60.0
        for i, sid in enumerate(sids):
            want, bnd, _, _ = st.ref(sid, s[i * t:(i + 1) * t], t)
            check("partials", True, got[i * t:(i + 1) * t], want, bnd, maxv, "x", (tag, nsplit, t, i))
            k, v = st.ring(sid)
            assert torch.equal(k, rings[i][0]) and torch.equal(v, rings[i][1]), "ring of the partials route"


def run_chunks(st, regime, t, tag):
    """Mixed counts up to the 128-key limit (k*t past ring_cap where the window is small), a pe wrap inside the call,
    G = k_max and G < k_max (several groups + the ring-append kernel), against the reference and each other; then one
    session's k chunks against k stream calls, outputs and ring bit for bit."""
    geo, f16, eng = st.geo, st.f16, st.eng
    kmax = max(1, (MAX_KEYS - geo.window) // t)
    gen = _gen("ch", tag, regime, t)
    sids = [st.ids[7], st.ids[2], st.ids[9], st.ids[4]]
    cnt = [kmax, 1, min(3, kmax), max(1, kmax - 1)]
    places = placements(geo, st.cap, t, k=kmax)
    saved = {}
    for sid, (nf, pe) in zip(sids, places):
        st.place(sid, nf, pe, regime, gen)
        saved[int(sid)] = st.state[int(sid)]
    rows = sum(cnt) * t
    qkv = _setup(st, regime, t, rows, gen)
    offs = np.concatenate([[0], np.cumsum(cnt)]) * t
    maxv = max(float(qkv[:, 2 * st.D:].abs().max()), 1e-30)
    results = {}
    for G in sorted({kmax, max(1, kmax // 3), 1}, reverse=True):
        for sid in sids:
            st.put(sid, *saved[int(sid)])
        out = eng.debug_attention("chunks", qkv, st.ptab, st.u, st.w, seq=sids, cnt=cnt, off0=3, t=t, layer=st.layer, group=G)
        rings = []
        for i, sid in enumerate(sids):
            seg = qkv[offs[i]:offs[i + 1]]
            want, bnd, hk, hv = st.ref(sid, seg, t)
            check("chunks", f16, out[offs[i]:offs[i + 1]], want, bnd, maxv, regime, (tag, regime, t, G, i))
            st.advance(sid, cnt[i] * t, hk, hv)
            rings.append(st.ring(sid))
        results[G] = (out, rings)
    o0, r0 = results[kmax]
    for G, (o, r) in results.items():
        assert torch.equal(o, o0), ("G < k_max != G = k_max", G, kmax, tag, t)
        for a, b in zip(r, r0):
            assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]), ("ring, G", G)
    # session 0's kmax chunks against kmax stream calls, stepping n_frames / pe_index between them
    sid, k = sids[3], cnt[3]
    nf, pe = saved[int(sid)][:2]
    seq_out = []
    st.put(sid, *saved[int(sid)])
    for j in range(k):
        seq_out.append(eng.debug_attention("stream", qkv[offs[3] + j * t:offs[3] + (j + 1) * t].contiguous(), st.ptab, st.u, st.w,
                                           seq=[sid], t=t, layer=st.layer))
        eng.set_frames(int(sid), nf + (j + 1) * t)
        pe = pe % geo.pe_wrap + geo.chunk_size
        eng.set_pe_index([int(sid)], pe)
    assert torch.equal(torch.cat(seq_out), o0[offs[3]:offs[4]]), ("chunks != stream calls", tag, t)
    k_, v_ = st.ring(sid)
    assert torch.equal(k_, r0[3][0]) and torch.equal(v_, r0[3][1]), ("ring: chunks != stream calls", tag, t)


STREAM_CFGS = [("shipped", 4, 16, "default")] + [("tiny", c, l, cap) for c, l in ROWS for cap in CAPS]


@pytest.mark.gpu
@pytest.mark.parametrize("f16", [False, True], ids=["fp32", "bf16"])
@pytest.mark.parametrize("name,c,left,cap", STREAM_CFGS, ids=["%s_c%d_l%d_%s" % x for x in STREAM_CFGS])
def test_streaming(engines, name, c, left, cap, f16):
    cfg, eng = engines(name, f16, c, left, cap)
    st = Streamer(cfg, eng, f16)
    try:
        ts = [t for t in (1, 3, 4, 7, 8) if t <= eng.max_t]
        if name == "tiny" and (c, left) != (4, 16):
            ts = sorted({min(c, eng.max_t), 1, eng.max_t})
        regimes = REGIMES if (name, c, left) in (("tiny", 4, 16), ("shipped", 4, 16)) else ["ordinary", "ramp"]
        tag = (name, c, left, cap)
        for t in ts:
            if cfg.kv_window + t > MAX_KEYS:               # every streaming entry refuses it
                continue
            for regime in regimes:
                run_stream(st, regime, t, tag)
                run_chunks(st, regime, t, tag)
    finally:
        eng.free(st.ids)


@pytest.mark.gpu
@pytest.mark.parametrize("f16", [False, True], ids=["fp32", "bf16"])
def test_refusals_launch_nothing(engines, f16):
    """Bad geometry is FO_ERR_ARG with no kernel enqueued."""
    from freeze_omni_b200 import _lib
    cfg, eng = engines("tiny", f16, 4, 16, "tight")           # max_t 4
    ids = eng.alloc(2)
    try:
        prow = pos_rows_of(cfg, eng.max_t)
        qkv, ptab, u, w = make_inputs("ordinary", 64, cfg.n_heads, prow, _gen("ref"), "cuda")
        eng.debug_attention("stream", qkv[:8], ptab, u, w, seq=ids, t=4)                 # accepted
        cases = [
            dict(mode="stream", seq=ids, t=5),                                            # t > max_t
            dict(mode="stream", seq=ids, t=0),
            dict(mode="chunks", seq=ids, cnt=[2, 2], t=4, group=(MAX_KEYS - cfg.kv_window) // 4 + 1),   # window + G t > 128
            dict(mode="chunks", seq=ids, cnt=[0, 2], t=4, group=2),
            dict(mode="offline", seq=[3], T=prow + 1),
            dict(mode="stream", seq=[int(ids[0]), int(ids[0])], t=1),                    # duplicate session
        ]
        for kw in cases:
            mode = kw.pop("mode")
            n0 = eng.stats()["kernel_launches"]
            with pytest.raises(_lib.FoError):
                eng.debug_attention(mode, qkv, ptab, u, w, **kw)
            assert eng.stats()["kernel_launches"] == n0, (mode, kw)
        n0 = eng.stats()["kernel_launches"]
        with pytest.raises(_lib.FoError, match="rel-pos table"):
            eng.debug_attention("stream", qkv[:8], ptab[:prow - 1].contiguous(), u, w, seq=ids, t=4)
        assert eng.stats()["kernel_launches"] == n0
    finally:
        eng.free(ids)


@pytest.mark.gpu
@pytest.mark.parametrize("f16", [False, True], ids=["fp32", "bf16"])
def test_graph_step_after_debug_calls(engines, f16):
    """Debug calls between graph-replayed steps of the same sessions leave the step's own id tables alone: the steps equal
    those of an untouched twin pair, bit for bit."""
    cfg, eng = engines("tiny", f16)
    ids = eng.alloc(5)
    try:
        g = torch.Generator().manual_seed(70)
        pcm = (3000 * torch.randn(2, cfg.samples_per_chunk * 4, generator=g)).round().to(torch.int16).numpy()
        chunks = [torch.from_numpy(np.ascontiguousarray(pcm[:, i * cfg.samples_per_chunk:(i + 1) * cfg.samples_per_chunk]))
                  for i in range(4)]
        qkv, ptab, u, w = make_inputs("ordinary", 64, cfg.n_heads, pos_rows_of(cfg, eng.max_t), _gen("graph"), "cuda")
        subj, twin, other = ids[:2], ids[2:4], ids[4:5]
        outs = []
        for i, x in enumerate(chunks):
            outs.append(eng.stream_step(subj, x)[0].clone())
            if i >= 1:                                        # between replays with unchanged ids
                eng.debug_attention("stream", qkv[:4], ptab, u, w, seq=other, t=4)
                eng.debug_attention("chunks", qkv, ptab, u, w, seq=other, cnt=[3], off0=1, t=4, group=1)
        for i, x in enumerate(chunks):           # an overwritten id table would attend other sessions: O(1) differences
            assert float((eng.stream_step(twin, x)[0] - outs[i]).abs().max()) <= (1e-3 if f16 else 1e-6), i
    finally:
        eng.free(ids)
