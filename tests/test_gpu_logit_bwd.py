"""GPU tests of the logit backward that folds the bilinear adjoint into the UNCE + UNKD backward
(``ucd_unce_unkd_bwd_lowres``, routed by ucd_b200/losses.py::_Route): the gradient of the low-res logits against the
fp64 oracle and against the two-step path (dx, then the upsample adjoint), in every usage pattern of the drop-in
modules, and which C-ABI calls each pattern makes."""
import pytest
import torch

from oracle import ucd_oracle as O

pytestmark = pytest.mark.gpu

C_OLD = {17: 16, 9: 6, 20: 14, 151: 101}


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ucd_b200
    from ucd_b200 import _lib
    assert _lib.lib().ucd_device_ok() == 1
    return ucd_b200


class _Counter:
    """Counts the C-ABI calls made through ucd_b200._lib while active."""

    def __init__(self, handle):
        self._h, self.counts = handle, {}

    def __getattr__(self, name):
        fn = getattr(self._h, name)

        def wrapped(*args):
            self.counts[name] = self.counts.get(name, 0) + 1
            return fn(*args)
        return wrapped


@pytest.fixture
def calls(U):
    from ucd_b200 import _lib
    h = _lib.lib()
    c = _Counter(h)
    _lib._lib = c
    yield c.counts
    _lib._lib = h


def _case(B, C, h, w, H, W, seed=5):
    g = torch.Generator().manual_seed(seed)
    lr = torch.randn(B, C, h, w, generator=g) * 3
    lpo = torch.randn(B, C_OLD[C], h, w, generator=g) * 3
    y = torch.randint(0, C, (B, H, W), generator=g)
    y[:, : H // 20] = 255
    return lr, lpo, y


def _rell2(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


def _cos(a, b):
    a, b = a.double().reshape(-1).cpu(), b.double().reshape(-1).cpu()
    return float(a @ b / (a.norm() * b.norm()).clamp_min(1e-300))


def _step(U, lr0, lpo, y, H, W, terms=("ce", "kd"), order="ce_first", leaf=True, extra=False, observe=None,
          passes=1, in_place=False, plain=False):
    """One step of the drop-in modules (train.py:115-116,133).  plain=True: the losses see a view of `outputs` - no
    upsample record - which is the two-step path (dx for `outputs`, then the upsample adjoint)."""
    C_old = lpo.shape[1]
    p = lr0.cuda().requires_grad_(True)
    lr = p if leaf else p * 1.0
    out = U.interpolate_bilinear(lr, (H, W))
    with torch.no_grad():
        old = U.interpolate_bilinear(lpo.cuda(), (H, W))
    if in_place:
        out.mul_(1.0)
    x = out.view_as(out) if plain else out
    ce_m = U.UnbiasedCrossEntropy(old_cl=C_old, ignore_index=255, reduction="none")
    kd_m = U.UnbiasedKnowledgeDistillationLoss(alpha=1.0)
    fns = [("ce", lambda: ce_m(x, y.cuda()).mean()), ("kd", lambda: 10 * kd_m(x, old))]
    if order != "ce_first":
        fns.reverse()
    vals = {k: f() for k, f in fns}
    loss = sum(vals[k] for k in terms)
    if extra:
        loss = loss + (out * 0.01).sum()
    if observe == "retain":
        out.retain_grad()
    elif observe == "hook":
        seen = []
        out.register_hook(lambda g: seen.append(g.norm()))
    if observe == "grad_out":
        (g_out,) = torch.autograd.grad(loss, out)
        return g_out, {k: v.item() for k, v in vals.items()}
    if observe == "grad_out_lr":
        g_out, g_lr = torch.autograd.grad(loss, [out, lr])
        return (g_out, g_lr), {k: v.item() for k, v in vals.items()}
    if observe == "inputs_out":
        loss.backward(inputs=[out])
        return out.grad, {k: v.item() for k, v in vals.items()}
    for i in range(passes):
        loss.backward(retain_graph=i + 1 < passes)
    if observe == "retain":
        assert out.grad is not None and out.grad.shape == out.shape
    if observe == "hook":
        assert len(seen) == passes
    return p.grad / passes, {k: v.item() for k, v in vals.items()}


def _oracle(lr0, lpo, y, H, W, terms=("ce", "kd"), extra=False):
    C_old = lpo.shape[1]
    lr = lr0.double().requires_grad_(True)
    x = O.upsample_bilinear(lr, H, W)
    t = O.upsample_bilinear(lpo.double(), H, W)
    n_px = float(y.numel())
    vals = {"ce": O.unbiased_ce(x, y.clone(), C_old, 255, "none").sum() / n_px,
            "kd": 10 * O.unbiased_kd(x, t, 1.0, "sum") / n_px}
    loss = sum(vals[k] for k in terms)
    if extra:
        loss = loss + (x * 0.01).sum()
    loss.backward()
    return lr.grad, {k: v.item() for k, v in vals.items()}


SHAPES = {  # (B, C, h, w, H, W)
    "voc512": (2, 17, 32, 32, 512, 512),
    "scale16": (2, 9, 16, 16, 256, 256),
    "voc513": (2, 17, 33, 33, 513, 513),       # not an integer scale: the two-step path
    "city": (1, 20, 32, 64, 512, 1024),
}
FUSED = {"voc512": True, "scale16": True, "voc513": False, "city": True}


@pytest.mark.parametrize("shape", sorted(SHAPES))
@pytest.mark.parametrize("leaf", [True, False])
def test_pair_against_oracle_and_two_step_path(U, calls, shape, leaf):
    B, C, h, w, H, W = SHAPES[shape]
    lr0, lpo, y = _case(B, C, h, w, H, W)
    want, ref_vals = _oracle(lr0, lpo, y, H, W)
    two_step, _ = _step(U, lr0, lpo, y, H, W, leaf=leaf, plain=True)
    calls.clear()
    got, vals = _step(U, lr0, lpo, y, H, W, leaf=leaf)
    torch.cuda.synchronize()
    for k in ("ce", "kd"):
        assert vals[k] == pytest.approx(ref_vals[k], rel=1e-3)
    assert _cos(got, want) >= 0.999
    assert _rell2(got, two_step) <= 1e-5
    if FUSED[shape]:
        assert calls.get("ucd_unce_unkd_bwd_lowres") == 1
        assert "ucd_unce_unkd_bwd" not in calls and "ucd_upsample_bilinear_bwd" not in calls, calls
    else:
        assert calls.get("ucd_unce_unkd_bwd") == 1 and calls.get("ucd_upsample_bilinear_bwd") == 1, calls
    # deterministic: a second run gives the same bits
    again, _ = _step(U, lr0, lpo, y, H, W, leaf=leaf)
    assert torch.equal(again, got)


CASES = {  # name: _step keyword arguments
    "ce_only": dict(terms=("ce",)),
    "kd_only": dict(terms=("kd",)),
    "kd_first": dict(order="kd_first"),
    "third_consumer": dict(extra=True),
    "retain_graph_two_passes": dict(passes=2),
    "retains_grad": dict(observe="retain"),
    "hook": dict(observe="hook"),
    "in_place_after_upsample": dict(in_place=True),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("leaf", [True, False])
def test_usage_patterns(U, calls, case, leaf):
    B, C, h, w, H, W = SHAPES["scale16"]
    kw = CASES[case]
    lr0, lpo, y = _case(B, C, h, w, H, W, seed=7)
    terms, extra = kw.get("terms", ("ce", "kd")), kw.get("extra", False)
    want, ref_vals = _oracle(lr0, lpo, y, H, W, terms=terms, extra=extra)
    two_step, _ = _step(U, lr0, lpo, y, H, W, leaf=leaf, plain=True, **kw)
    calls.clear()
    got, vals = _step(U, lr0, lpo, y, H, W, leaf=leaf, **kw)
    torch.cuda.synchronize()
    for k in terms:
        assert vals[k] == pytest.approx(ref_vals[k], rel=1e-3)
    assert _cos(got, want) >= 0.999
    assert _rell2(got, two_step) <= 1e-5
    fused = case in ("kd_first", "third_consumer", "retain_graph_two_passes")
    assert (calls.get("ucd_unce_unkd_bwd_lowres", 0) > 0) == fused, calls
    if case in ("retains_grad", "hook"):   # an observer of `outputs`' gradient gets it exactly as before
        assert calls.get("ucd_unce_unkd_bwd") == 1 and calls.get("ucd_upsample_bilinear_bwd") == 1, calls


@pytest.mark.parametrize("leaf", [True, False])
@pytest.mark.parametrize("how", ["grad_out", "inputs_out", "grad_out_lr"])
def test_captured_outputs_get_their_gradient(U, calls, leaf, how):
    """autograd.grad / backward(inputs=...) naming `outputs`: the full-size gradient, identical to the two-step path."""
    B, C, h, w, H, W = SHAPES["scale16"]
    lr0, lpo, y = _case(B, C, h, w, H, W, seed=9)
    want, _ = _step(U, lr0, lpo, y, H, W, leaf=leaf, plain=True, observe=how)
    calls.clear()
    got, _ = _step(U, lr0, lpo, y, H, W, leaf=leaf, observe=how)
    assert "ucd_unce_unkd_bwd_lowres" not in calls, calls
    if how == "grad_out_lr":
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    else:
        assert torch.equal(got, want)


def test_ade_shape(U, calls):
    """ADE 100-50 (151 / 101 classes) at 512x512: the fused path, one image (fp64 oracle memory)."""
    B, C, h, w, H, W = 1, 151, 32, 32, 512, 512
    lr0, lpo, y = _case(B, C, h, w, H, W, seed=3)
    want, ref_vals = _oracle(lr0, lpo, y, H, W)
    two_step, _ = _step(U, lr0, lpo, y, H, W, plain=True)
    calls.clear()
    got, vals = _step(U, lr0, lpo, y, H, W, leaf=False)
    assert calls.get("ucd_unce_unkd_bwd_lowres") == 1 and "ucd_upsample_bilinear_bwd" not in calls, calls
    for k in ("ce", "kd"):
        assert vals[k] == pytest.approx(ref_vals[k], rel=1e-3)
    assert _cos(got, want) >= 0.999
    assert _rell2(got, two_step) <= 1e-5


@pytest.mark.parametrize("variant,rows", [("0", "3"), ("1", "5"), ("0", "32"), ("2", "2"), ("3", "4")])
def test_row_ranges_and_channel_groups(U, monkeypatch, variant, rows):
    """Ranges of several low-res rows (interval hand-over inside a block, plain stores between two ranges' shared rows,
    a short last range) and channel groups of several channels, forced through the debug library's knobs, at the
    bench shape (B=24, 17 / 16 classes) against the two-step path."""
    from ucd_b200 import _lib
    B, C, h, w, H, W = 24, 17, 32, 32, 512, 512
    lr0, lpo, y = _case(B, C, h, w, H, W, seed=13)
    two_step, _ = _step(U, lr0, lpo, y, H, W, plain=True)
    prod = _lib.lib()
    monkeypatch.setenv("UCD_LRB_VARIANT", variant)
    monkeypatch.setenv("UCD_LRB_ROWS", rows)
    try:
        counter = _Counter(_lib.debug_lib())
        _lib._lib = counter
        got, _ = _step(U, lr0, lpo, y, H, W, leaf=False)
        again, _ = _step(U, lr0, lpo, y, H, W, leaf=False)
    finally:
        _lib._lib = prod
    assert counter.counts.get("ucd_unce_unkd_bwd_lowres") == 2, counter.counts
    assert _rell2(got, two_step) <= 1e-5
    assert torch.equal(again, got)


def test_odd_vertical_scale(U, calls):
    """3x along y (odd tap-table lengths) and 8x along x: the sweep form, against the two-step path and the oracle."""
    B, C, h, w, H, W = 1, 17, 32, 64, 96, 512
    lr0, lpo, y = _case(B, C, h, w, H, W, seed=17)
    want, _ = _oracle(lr0, lpo, y, H, W)
    two_step, _ = _step(U, lr0, lpo, y, H, W, plain=True)
    calls.clear()
    got, _ = _step(U, lr0, lpo, y, H, W)
    assert calls.get("ucd_unce_unkd_bwd_lowres") == 1, calls
    assert _cos(got, want) >= 0.999
    assert _rell2(got, two_step) <= 1e-5
