"""CPU side of the low-res output mode (the CE-only fused loss of the base step and `predict_bilinear`): the oracles the
GPU tests compare against, the exported symbols, and the argument checks that run before any launch."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import ucd_oracle as O


def argmax_restated(v):
    """torch.argmax over dim 1 written out: channels in order, a strictly larger value or the first NaN takes over."""
    best = v[:, 0].clone()
    idx = torch.zeros(best.shape, dtype=torch.int64)
    for c in range(1, v.shape[1]):
        x = v[:, c]
        take = (x > best) | (torch.isnan(x) & ~torch.isnan(best))
        best = torch.where(take, x, best)
        idx = torch.where(take, torch.full_like(idx, c), idx)
    return idx


@pytest.mark.parametrize("reduction", ["none", "sum", "mean"])
def test_plain_ce_is_unbiased_ce_with_one_old_class(reduction):
    """The step-0 loss the GPU tests check against: fp64 F.cross_entropy (ignore 255) is O.unbiased_ce with old_cl=1
    on labels in [0, C) and 255 (its background branch, lse_all - lse over channel 0, is then the plain CE of class 0)."""
    g = torch.Generator().manual_seed(3)
    B, C, H, W = 2, 7, 19, 23
    x = torch.randn(B, C, H, W, generator=g, dtype=torch.float64) * 3
    y = torch.randint(0, C, (B, H, W), generator=g)
    y[:, 4:7] = 255
    y[1, :, 2] = 255
    ref = F.cross_entropy(x, y, ignore_index=255, reduction=reduction)
    y1 = y.clone()
    mine = O.unbiased_ce(x, y1, 1, 255, reduction)
    assert torch.equal(y1, y)   # no label below old_cl = 1 except 0 itself: nothing is remapped
    torch.testing.assert_close(mine, ref, rtol=1e-12, atol=1e-12)


@pytest.mark.parametrize("case", ["random", "ties", "constant", "nan"])
def test_argmax_restatement_matches_aten(case):
    """The CPU argmax restatement over O.upsample_bilinear equals F.interpolate(...).argmax(1): first maximal channel
    on ties, NaN maximal.  In fp32, as the kernel: for a fp64 input O.upsample_bilinear computes its taps in fp64 and
    ATen does not, and where the source coordinate lands on a cell boundary the two pick different neighbours (one at
    weight 0), which moves the footprint of a NaN."""
    g = torch.Generator().manual_seed(11)
    B, C, h, w, H, W = 2, 6, 5, 7, 65, 97
    lr = torch.randn(B, C, h, w, generator=g) * 3
    if case == "ties":
        lr[:, 4] = lr[:, 1] = lr[:, 1] + 10.0     # channels 1 and 4 tie everywhere: 1 wins
        lr[1, 2] = lr[1, 1]                         # image 1: channels 1, 2 and 4 tie: 1 wins
    elif case == "constant":
        lr[:] = 0.25                                # every channel ties: 0 wins
    elif case == "nan":
        lr[0, 3, 2, 4] = float("nan")               # every pixel whose taps touch the cell predicts 3
        lr[1, 5, 0, 0] = lr[1, 2, 0, 0] = float("nan")   # two NaN channels: the first one, 2, wins
    ref = F.interpolate(lr, size=(H, W), mode="bilinear", align_corners=False).argmax(1)
    mine = argmax_restated(O.upsample_bilinear(lr, H, W))
    assert torch.equal(mine, ref)
    if case == "nan":
        assert bool((ref[0] == 3).any()) and bool((ref[1] == 2).any())


@pytest.mark.parametrize("shape", [(7, 5, 40, 24), (16, 16, 40, 24), (5, 7, 65, 97), (32, 32, 512, 512)], ids=str)
def test_aten_single_plane_is_the_restated_order(shape):
    """The CPU reference of the prediction tests: F.interpolate called on one plane at a time equals the bit-exact
    restatement O._bilinear_eval_f32 (the order ucd_upsample_bilinear_fwd implements) at small (H + W <= 128) and
    generic sizes, with many planes, exact ties and a NaN."""
    h, w, H, W = shape
    g = torch.Generator().manual_seed(7)
    lr = torch.randn(3, 21, h, w, generator=g) * 3
    lr[0, 9] = lr[0, 4]
    lr[1] = 0.5
    lr[2, 6, h // 2, w // 2] = float("nan")
    one = torch.cat([F.interpolate(p, size=(H, W), mode="bilinear", align_corners=False)
                     for p in lr.reshape(63, 1, 1, h, w)]).reshape(3, 21, H, W)
    ref = torch.from_numpy(O._bilinear_eval_f32(lr.numpy(), H, W))
    assert torch.equal(one.isnan(), ref.isnan()) and torch.equal(one.nan_to_num(0.0), ref.nan_to_num(0.0))


@pytest.fixture(scope="module")
def L():
    from ucd_b200 import _lib, build
    build.build()
    return _lib


def test_new_symbols_exported(L):
    h = ctypes.CDLL(L.LIB_PATH)
    assert hasattr(h, "ucd_upsample_argmax") and "ucd_upsample_argmax" in L.EXPORTED
    import ucd_b200
    assert callable(ucd_b200.predict_bilinear) and "predict_bilinear" in ucd_b200.__all__


def test_ce_only_workspace_and_argument_checks(L):
    """C_old == 0 is the CE-only form: its workspace holds one gradient term per cell instead of two.  Null pointers
    and bad shapes are refused with UCD_EINVAL before anything is launched (the pointers below are never
    dereferenced)."""
    lib = L.lib()
    ws0 = lib.ucd_seg_fused_workspace_floats(2, 16, 0, 32, 32, 512, 512)
    ws1 = lib.ucd_seg_fused_workspace_floats(2, 16, 1, 32, 32, 512, 512)
    assert 0 < ws0 < ws1
    assert lib.ucd_seg_fused_workspace_floats(2, 16, -1, 32, 32, 512, 512) == 0
    fake = ctypes.c_void_p(256)

    def fwd(lr, lr_old, g_ce, g_kd, C_old, need_grad, ws=fake, labels=fake):
        return lib.ucd_seg_fused_fwd(lr, lr_old, labels, g_ce, g_kd, fake, ws, 1, 2, 16, C_old, 32, 32, 512, 512, 0,
                                     255, 1.0, need_grad, None)

    assert fwd(None, None, fake, None, 0, 1) == -1 and b"null pointer" in lib.ucd_last_error()
    assert fwd(fake, None, fake, fake, 0, 1, labels=None) == -1 and b"null pointer" in lib.ucd_last_error()
    assert fwd(fake, None, fake, fake, 1, 1) == -1 and b"null pointer" in lib.ucd_last_error()   # KD needs lr_old
    assert fwd(fake, None, None, None, 0, 1) == -1 and b"gradient buffers" in lib.ucd_last_error()
    assert fwd(fake, fake, fake, None, 1, 1) == -1 and b"gradient buffers" in lib.ucd_last_error()
    assert fwd(fake, None, fake, None, -1, 1) == -1 and b"bad shape" in lib.ucd_last_error()
    # CE-only and well formed, but the 1-float workspace is too small: refused, nothing launched
    assert fwd(fake, None, fake, None, 0, 1) == -1 and b"workspace too small" in lib.ucd_last_error()


@pytest.mark.parametrize("shape", [(33, 33, 32, 33), (32, 32, 512, 16), (513, 513, 33, 33), (2, 3, 1, 3)])
def test_upsample_argmax_refuses_downscaling_and_nulls(L, shape):
    lib = L.lib()
    h, w, H, W = shape
    fake = ctypes.c_void_p(256)
    assert lib.ucd_upsample_argmax(fake, fake, 1, 4, h, w, H, W, None) == -1
    assert b"upsampling only" in lib.ucd_last_error()
    assert lib.ucd_upsample_argmax(None, fake, 1, 4, 32, 32, 512, 512, None) == -1
    assert b"null pointer" in lib.ucd_last_error()
    assert lib.ucd_upsample_argmax(fake, None, 1, 4, 32, 32, 512, 512, None) == -1
    assert lib.ucd_upsample_argmax(fake, fake, 1, 0, 32, 32, 512, 512, None) == -1   # C = 0: no argmax
    assert b"bad shape" in lib.ucd_last_error()


def test_predict_bilinear_refuses_cpu_tensors():
    import ucd_b200
    with pytest.raises(RuntimeError, match="no CPU"):
        ucd_b200.predict_bilinear(torch.randn(1, 3, 4, 4), (8, 8))
