"""GPU tests of the low-res output mode: the CE-only form of FusedUnbiasedLosses (the base step, no old model) against
the fp64 oracle chain O.upsample_bilinear -> autograd, and predict_bilinear against the argmax of the materialised
upsample on the GPU and on the CPU."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ucd_oracle as O

pytestmark = pytest.mark.gpu

# (B, C, h, w, H, W, old_cl of a real split)
SHAPES = {
    "32to512": (2, 16, 32, 32, 512, 512, 11),       # VOC 15-5 at step 1 has 16 old of 21 classes; here 11 of 16
    "33to513": (2, 21, 33, 33, 513, 513, 16),       # VOC 15-5, crop 513
    "city32x64": (2, 14, 32, 64, 512, 1024, 13),    # Cityscapes 13-6: 13 old classes + background at step 1
    "ragged19x23": (2, 21, 19, 23, 304, 368, 16),
}


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ucd_b200
    from ucd_b200 import _lib
    assert _lib.lib().ucd_device_ok() == 1, "ucd_b200 needs a compute-capability 10.x device"
    return ucd_b200


def cos(a, b):
    a, b = a.double().reshape(-1).cpu(), b.double().reshape(-1).cpu()
    return float(a @ b / (a.norm() * b.norm()).clamp_min(1e-300))


def make_case(B, C, h, w, H, W, seed=0):
    """Low-res logits and blob labels in [0, C) (nearest-upsampled low-res classes) with an ignore strip."""
    g = torch.Generator().manual_seed(100 + seed)
    lr = torch.randn(B, C, h, w, generator=g) * 3
    cls = torch.randint(0, C, (B, 1, max(h // 4, 1), max(w // 4, 1)), generator=g).float()
    y = F.interpolate(cls, size=(H, W), mode="nearest")[:, 0].long()
    y[:, H // 3:H // 3 + 7] = 255
    y[-1, :, : W // 10] = 255
    return lr, y


def oracle(lr, y, old_cl, reduction):
    """fp64 loss, d loss / d lr and the remapped labels; image by image (bounds the fp64 temporaries at ADE size)."""
    B, H, W = y.shape
    y = y.clone()
    denom = float(B * H * W) if reduction == "mean" else float((y != 255).sum())
    total, grad = 0.0, torch.zeros(lr.shape, dtype=torch.float64)
    for b in range(B):
        x_lr = lr[b:b + 1].double().requires_grad_(True)
        x = O.upsample_bilinear(x_lr, H, W)
        if old_cl == 0:
            s = F.cross_entropy(x, y[b:b + 1], ignore_index=255, reduction="sum")
        else:
            s = O.unbiased_ce(x, y[b:b + 1], old_cl, 255, "sum")    # remaps y[b] in place
        (s / denom).backward()
        total += s.item() / denom
        grad[b] = x_lr.grad[0]
    return total, grad, y


def check_against_oracle(U, lr, y, old_cl, reduction):
    ce_ref, g_ref, y_ref = oracle(lr, y, old_cl, reduction)
    x = lr.cuda().requires_grad_(True)
    lab = y.cuda()
    ce, kd = U.FusedUnbiasedLosses(old_cl, ignore_index=255, ce_reduction=reduction)(x, None, lab)
    assert kd is None
    ce.backward()
    assert abs(ce.item() - ce_ref) <= 1e-5 * abs(ce_ref), (ce.item(), ce_ref)
    assert torch.equal(lab.cpu(), y_ref)
    assert cos(x.grad, g_ref) >= 0.999
    torch.testing.assert_close(x.grad.cpu().double(), g_ref, rtol=2e-3, atol=2e-5 * float(g_ref.abs().max()))


@pytest.mark.parametrize("reduction", ["mean", "valid"])
@pytest.mark.parametrize("old_cl", ["0", "1", "split"])
@pytest.mark.parametrize("shape", list(SHAPES))
def test_ce_only_against_fp64_chain(U, shape, old_cl, reduction):
    B, C, h, w, H, W, split = SHAPES[shape]
    lr, y = make_case(B, C, h, w, H, W)
    check_against_oracle(U, lr, y, {"0": 0, "1": 1, "split": split}[old_cl], reduction)


def test_ce_only_ade_step0_real_size(U):
    """ADE 100-50 step 0 at its real per-GPU size: 3 images, 101 classes, 32x32 -> 512x512."""
    lr, y = make_case(3, 101, 32, 32, 512, 512, seed=1)
    check_against_oracle(U, lr, y, 0, "mean")


def test_ce_only_bit_identical_reruns_and_no_grad(U, monkeypatch):
    from ucd_b200 import _lib
    B, C, h, w, H, W, _ = SHAPES["33to513"]
    lr, y = make_case(B, C, h, w, H, W, seed=2)
    runs = []
    for _ in range(5):
        x = lr.cuda().requires_grad_(True)
        ce, _ = U.FusedUnbiasedLosses(0)(x, None, y.cuda())
        ce.backward()
        runs.append((ce.detach().clone(), x.grad.clone()))
    for ce, g in runs[1:]:
        assert torch.equal(ce, runs[0][0]) and torch.equal(g, runs[0][1])

    calls = []

    class Spy:
        def __init__(self, h):
            self.h = h

        def __getattr__(self, name):
            fn = getattr(self.h, name)
            if name != "ucd_seg_fused_fwd":
                return fn

            def rec(*args):
                calls.append(args)
                return fn(*args)
            return rec

    monkeypatch.setattr(_lib, "_lib", Spy(_lib.lib()))
    x = lr.cuda().requires_grad_(True)
    with torch.no_grad():
        ce, kd = U.FusedUnbiasedLosses(0)(x, None, y.cuda())
    assert kd is None and ce.grad_fn is None and ce.item() == runs[0][0].item()
    (args,) = calls
    assert args[1] is None and args[3] is None and args[4] is None and args[-2] == 0   # no old model, no gradient


def test_ce_only_cuda_graph_replay(U):
    """Forward + backward of the CE-only form captured once and replayed on new data: equal to eager."""
    B, C, h, w, H, W, _ = SHAPES["32to512"]
    lr_a, y_a = make_case(B, C, h, w, H, W, seed=3)
    lr_b, y_b = make_case(B, C, h, w, H, W, seed=4)
    fused = U.FusedUnbiasedLosses(0, ce_reduction="valid")
    x = lr_a.cuda().requires_grad_(True)
    lab = y_a.cuda()

    def step():
        ce, _ = fused(x, None, lab)
        ce.backward()
        return ce

    if hasattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch"):
        torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            x.grad = None
            step()
    torch.cuda.current_stream().wait_stream(side)
    x.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        ce_s = step()
    for lr_n, y_n in ((lr_b, y_b), (lr_a, y_a)):
        with torch.no_grad():
            x.copy_(lr_n.cuda())
            lab.copy_(y_n.cuda())
            x.grad.zero_()
        graph.replay()
        torch.cuda.synchronize()
        x2 = lr_n.cuda().requires_grad_(True)
        ce2, _ = U.FusedUnbiasedLosses(0, ce_reduction="valid")(x2, None, y_n.cuda())
        ce2.backward()
        assert ce_s.item() == ce2.item()
        assert torch.equal(x.grad, x2.grad)


# ------------------------------------------------------------------------------------------------
# predict_bilinear
# the 14 shapes of test_oracle.py::test_bilinear_restatement_bit_exact_vs_aten, taken in the upsampling direction
PRED_SHAPES = [(513, 513, 33, 33), (512, 512, 32, 32), (321, 321, 21, 21), (500, 375, 32, 24), (65, 97, 5, 7),
               (512, 1024, 32, 64), (562, 618, 65, 65), (562, 618, 32, 128), (700, 300, 140, 20), (33, 33, 513, 513),
               (9, 13, 144, 208), (16, 16, 40, 24), (32, 64, 512, 1024), (7, 5, 7, 5)]
PRED_BATCH = {1: 24, 2: 8, 16: 3, 21: 2, 151: 1}


def up_dir(s):
    a, b, c, d = s
    return min(a, c), min(b, d), max(a, c), max(b, d)


def aten_per_plane(lr, H, W):
    """CPU F.interpolate, one plane per call.  For small outputs (H + W <= 128) ATen's CPU kernel runs the planes of a
    batched call in SIMD groups with a scalar remainder whose last bits differ, so identical channels can come out
    different there and an exact tie is decided by plane position.  A single plane always takes the remainder path,
    the operation order that ucd_upsample_bilinear_fwd restates (tests/test_lowres_only_cpu.py pins this)."""
    B, C, h, w = lr.shape
    planes = lr.float().reshape(B * C, 1, 1, h, w)
    out = [F.interpolate(p, size=(H, W), mode="bilinear", align_corners=False) for p in planes]
    return torch.cat(out).reshape(B, C, H, W)


def check_prediction(U, lr, H, W):
    pred = U.predict_bilinear(lr.cuda(), (H, W))
    assert pred.dtype == torch.int64 and pred.shape == (lr.shape[0], H, W)
    ref_gpu = U.interpolate_bilinear(lr.cuda(), (H, W)).argmax(1)
    assert torch.equal(pred, ref_gpu)
    assert torch.equal(pred.cpu(), aten_per_plane(lr, H, W).argmax(1))
    if H + W > 128:   # the generic CPU kernel computes every plane alike: the batched call is the same reference
        ref_cpu = F.interpolate(lr.float(), size=(H, W), mode="bilinear", align_corners=False).argmax(1)
        assert torch.equal(pred.cpu(), ref_cpu)
    return pred


@pytest.mark.parametrize("C", list(PRED_BATCH))
@pytest.mark.parametrize("shape", PRED_SHAPES, ids=lambda s: "%dx%d-%dx%d" % up_dir(s))
def test_predict_bilinear_equals_materialised_argmax(U, shape, C):
    h, w, H, W = up_dir(shape)
    g = torch.Generator().manual_seed(h * 1000 + W + C)
    lr = torch.randn(PRED_BATCH[C], C, h, w, generator=g) * 3
    check_prediction(U, lr, H, W)


@pytest.mark.parametrize("shape", [(32, 32, 512, 512), (5, 7, 65, 97), (7, 5, 40, 24)], ids=str)
def test_predict_bilinear_ties_and_nan(U, shape):
    h, w, H, W = shape
    g = torch.Generator().manual_seed(7)
    lr = torch.randn(3, 21, h, w, generator=g) * 3
    lr[0, 9] = lr[0, 4] = lr[0, 4] + 30.0         # duplicated dominant channels: 4 everywhere
    lr[1] = 0.5                                    # constant maps: every channel ties, 0 everywhere
    lr[2, 6, h // 2, w // 2] = float("nan")        # one NaN cell: 6 wherever its taps reach
    pred = check_prediction(U, lr, H, W)
    assert bool((pred[0] == 4).all()) and bool((pred[1] == 0).all()) and bool((pred[2] == 6).any())


@pytest.mark.parametrize("shape", [(24, 16, 32, 32, 512, 512), (3, 151, 32, 32, 512, 512), (3, 19, 32, 64, 512, 1024)],
                         ids=["voc", "ade", "city"])
def test_predict_bilinear_allocates_only_the_prediction(U, shape):
    B, C, h, w, H, W = shape
    lr = (torch.randn(B, C, h, w) * 3).cuda()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    pred = U.predict_bilinear(lr, (H, W))
    torch.cuda.synchronize()
    growth = torch.cuda.max_memory_allocated() - base
    assert growth <= pred.numel() * 8 + (1 << 20), growth
    assert np.array_equal(pred.cpu().numpy(), U.interpolate_bilinear(lr, (H, W)).argmax(1).cpu().numpy())
