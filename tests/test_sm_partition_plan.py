"""Host logic of contexts on a group of the device's SMs (fo_create_on_sms), no GPU needed: the layer-stack plan at the SM
counts of a B200 split 2, 2 (at 64), 4 and 8 ways, and the refusals that are decided before a device is touched."""
import ctypes as C

import pytest

from freeze_omni_b200 import _lib

FO_ERR_ARG = -1                                       # include/fo_b200.h
SMEM = 232448                                         # opt-in shared memory per CTA on a B200 (227 KB)


def plan(sms, n, t=4, d=1024, ff=4096, h=16, window=64, layers=24):
    lib = _lib.load()
    out = [C.c_int() for _ in range(5)]
    rc = lib.fo_debug_stack_plan(d, ff, h, n, t, window, layers, sms, SMEM, *[C.byref(o) for o in out])
    return rc, [o.value for o in out]


@pytest.mark.parametrize("sms", [72, 64, 32, 16])
@pytest.mark.parametrize("n", [1, 2])
def test_shipped_model_takes_the_chain_on_a_group(sms, n):
    """The shipped model (D 1024, FF 4096, 16 heads): a CTA's weight slice of one phase is at most 32 rows (MAXG groups of 8),
    and FFN1's 4096 rows over 72 SMs are 57 (QKV 43), so no group of a split B200 runs the layer stack: the step takes the
    per-kernel chain.  148 SMs (fo_create) keep it."""
    assert plan(sms, n)[0] == 1
    assert plan(148, n)[0] == 0


@pytest.mark.parametrize("sms,rows", [(72, (6, 4, 2)), (64, (6, 4, 2)), (32, (12, 8, 4)), (16, (24, 16, 8))])
@pytest.mark.parametrize("n", [1, 2])
def test_toy_widths_fit_every_group(sms, rows, n):
    """D 128, FF 256, 2 heads: the slices grow as the group shrinks (rows per CTA of QKV / FFN1 / out-proj and FFN2 =
    3D / FF / D over the group's SMs, rounded up) and still fit, with the same shared memory at every group size but 16,
    where the 24-row QKV slice outgrows the shared buffer of the 148-SM plan."""
    rc, (smem, kc, rq, rf, ro) = plan(sms, n, d=128, ff=256, h=2, layers=2)
    assert rc == 0
    assert (rq, rf, ro) == rows
    assert kc == 256 and smem <= SMEM
    rc148, (smem148, _, _, _, _) = plan(148, n, d=128, ff=256, h=2, layers=2)
    assert rc148 == 0 and smem >= smem148


@pytest.mark.parametrize("sms,fits", [(72, True), (64, True), (32, False), (16, False)])
def test_mid_width_plan_by_group_size(sms, fits):
    """D 512, FF 1024, 8 heads: QKV's 1536 rows fit a 32-row slice down to 48 SMs: 24 rows per CTA at 64, 48 at 32."""
    rc, (smem, kc, rq, rf, ro) = plan(sms, 1, d=512, ff=1024, h=8, layers=4)
    assert (rc == 0) == fits
    if fits:
        assert rf == -(-1024 // sms) and rq == -(-1536 // sms) and ro == -(-512 // sms) and smem <= SMEM


def _cfg():
    return _lib.FoConfig(feat_dim=80, d_model=128, n_heads=2, ffn_dim=256, n_layers=1, chunk_size=4, left_chunks=16,
                         input_layer_linear=1, pos_max_len=5000, llm_dim=256, adapter_kernel=5, adapter_gelu=1,
                         has_encoder=1, has_adapter=1, sample_rate=16000, frame_len=400, frame_shift=160,
                         frames_per_chunk=16, context_frames=3, max_sessions=2, max_stream_frames=19)


@pytest.mark.parametrize("split,group,msg", [(0, 0, b"sm_split must be >= 1"), (-2, 0, b"sm_split must be >= 1"),
                                             (2, 2, b"sm_group 2 is outside [0, sm_split = 2)"),
                                             (4, -1, b"sm_group -1 is outside [0, sm_split = 4)")])
def test_create_on_sms_refuses_bad_split_or_group(split, group, msg):
    """Refused before any device is touched, so the same on a machine without a GPU."""
    lib = _lib.load()
    h = C.c_void_p()
    cfg = _cfg()
    assert lib.fo_create_on_sms(C.byref(cfg), 0, _lib.FO_BF16, split, group, C.byref(h)) == FO_ERR_ARG
    assert msg in lib.fo_last_error()
    assert not h.value


def test_create_on_sms_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("checks the no-GPU failure mode")
    lib = _lib.load()
    h = C.c_void_p()
    cfg = _cfg()
    assert lib.fo_create_on_sms(C.byref(cfg), 0, _lib.FO_BF16, 2, 0, C.byref(h)) != 0
    assert b"no CUDA device" in lib.fo_last_error()
