"""GPU tests of the shared CE + KD logit backward (csrc/ce_kd.cu ``pair_args`` / ``pair_coef`` / ``pair_dx``) in every
configuration the loss modules hand it, element by element against the closed-form fp64 oracle of
oracle/logit_pair.py.

Every case of ``logit_pair.GRID`` (a covering array over CE reduction and use, KD module, KD reduction, alpha, mask,
ignore_index, CE old_cl against KD C_old, call order and loss weights) runs the drop-in modules on the same `outputs`
and a backward, on three routes: full-res logits at HW = 33 x 35 (``unce_unkd_bwd_kernel<1, ...>``) and 64 x 96
(``<4, ...>``), and ``outputs = interpolate_bilinear(lr)`` at a 16x upsample (``unce_unkd_bwd_lowres_kernel``).  Each
case asserts that exactly one pair call ran - ``ucd_unce_unkd_bwd`` or ``ucd_unce_unkd_bwd_lowres`` - and none of the
single-loss backward calls or the upsample adjoint.

Bar, per full-res element or per low-res cell (``logit_pair.bar``): |g - g_ref| <= REL * mag + FLOOR * median(mag)
with REL = 3e-5 and FLOOR = 1e-7; the oracle's operands are the fp32 values the kernel reads (for the low-res route the
upsampled logits, read back).  Observed on an NVIDIA B200 (1000 W power limit), max over the grid of
|g - g_ref| / (mag + FLOOR / REL * median(mag)): full-res VEC 1 2.6e-6, VEC 4 2.4e-6, low-res 4.1e-7, low-res with
forced row ranges and channel groups 4.1e-7 (ex2.approx and the fp32 log-sum-exps of the forward; the adjoint's
non-negative weights average the per-element errors of a low-res cell).  Loss values: within 1e-5 of the sum of the
magnitudes of their terms (observed 1.5e-7); the CE valid count and the in-place label remap exact.
tests/test_logit_pair_cpu.py shows every listed kernel slip misses this bar by >= 10x (by >= 2.5e3x at the grid's
inputs).
"""
import pytest
import torch

from oracle import logit_pair as LP

pytestmark = pytest.mark.gpu

PAIR = {"fr33x35": "ucd_unce_unkd_bwd", "fr64x96": "ucd_unce_unkd_bwd", "lr": "ucd_unce_unkd_bwd_lowres"}
OTHER_BWD = ("ucd_unce_unkd_bwd", "ucd_unce_unkd_bwd_lowres", "ucd_unce_bwd", "ucd_kd_bwd", "ucd_upsample_bilinear_bwd")
LR_CASES = [c for c in LP.CASES if c[0] == "lr"]


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ucd_b200
    from ucd_b200 import _lib
    assert _lib.lib().ucd_device_ok() == 1
    return ucd_b200


class _Counter:
    """Counts the C-ABI calls made through ucd_b200._lib while installed as its handle."""

    def __init__(self, handle):
        self._h, self.counts = handle, {}

    def __getattr__(self, name):
        fn = getattr(self._h, name)

        def wrapped(*args):
            self.counts[name] = self.counts.get(name, 0) + 1
            return fn(*args)
        return wrapped


def run(U, route, i, handle=None, plain=False):
    """One forward + backward of case i of `route` through the drop-in modules, with the C-ABI calls counted.
    handle: the library to run on (default the product one); plain=True (low-res route): the losses see a view of
    `outputs`, which has no upsample record - the two-step path (dx, then the upsample adjoint)."""
    from ucd_b200 import _lib
    B, C, C_old, h, w, H, W = LP.SHAPES[route]
    cfg = LP.GRID[route][i]
    d = LP.make_inputs(route, i)
    old_cl = LP.old_cl_of(cfg, C, C_old)
    n = float(B * H * W)
    y = d["y"].cuda()
    mask = None if d["mask"] is None else d["mask"].cuda()
    w_ce, w_kd = d["w_ce"].cuda(), d["w_kd"].cuda()
    prod = _lib.lib()
    counter = _Counter(handle if handle is not None else prod)
    _lib._lib = counter
    try:
        leaf = d["logits"].cuda().requires_grad_(True)
        if route == "lr":
            outputs = U.interpolate_bilinear(leaf, (H, W))
            with torch.no_grad():
                old = U.interpolate_bilinear(d["old"].cuda(), (H, W))
        else:
            outputs, old = leaf * 1.0, d["old"].cuda()
        x = outputs.view_as(outputs) if plain else outputs
        ce_m = U.UnbiasedCrossEntropy(old_cl=old_cl, reduction=cfg.ce if cfg.ce in ("mean", "sum") else "none",
                                      ignore_index=cfg.ign)
        kd_cls = U.UnbiasedKnowledgeDistillationLoss if cfg.kd == "unbiased" else U.MaskKnowledgeDistillationLoss
        kd_m = kd_cls(reduction="none" if cfg.kd_red == "none_w" else cfg.kd_red, alpha=cfg.alpha)
        raw = {}

        def ce():
            v = raw["ce"] = ce_m(x, y)
            return {"none_mean": lambda: v.mean(), "none_w": lambda: (w_ce * v).sum() / n, "mean": lambda: v,
                    "sum": lambda: v / n}[cfg.ce]()

        def kd():
            v = kd_m(x, old, mask)
            return {"mean": lambda: v, "sum": lambda: v / n, "none_w": lambda: (w_kd * v).sum() / n}[cfg.kd_red]()
        vals = {"ce": ce(), "kd": kd()} if cfg.order == "ce" else {"kd": kd(), "ce": ce()}
        # the CE forward's statistics (loss sum, valid count) are saved on its node
        stats = raw["ce"].grad_fn.saved_tensors[3] if cfg.ce in ("mean", "sum") else None
        a, b = LP.loss_weights(cfg)
        (a * vals["ce"] + b * vals["kd"]).backward()
        torch.cuda.synchronize()
    finally:
        _lib._lib = prod
    return dict(grad=leaf.grad.double().cpu(), ce=vals["ce"].item(), kd=vals["kd"].item(),
                n_valid=None if stats is None else float(stats[1]), y=y.cpu(), calls=counter.counts,
                x=outputs.detach().double().cpu(), t=old.double().cpu())


def reference(route, i, r):
    """(g_ref, mag) where the test compares: per element, or per low-res cell through the adjoint.  The operands are the
    fp32 values the kernel read: the inputs, or for the low-res route the upsampled logits."""
    B, C, C_old, h, w, H, W = LP.SHAPES[route]
    dx, mag = LP.oracle(route, i, r["x"], r["t"])
    if route == "lr":
        return LP.adjoint(dx, h, w), LP.adjoint(mag, h, w)
    return dx, mag


def measure(U, route, i, handle=None):
    """Run case i of `route` and compare it with the oracle: (gradient error in units of the bar, run result)."""
    r = run(U, route, i, handle=handle)
    want, mag = reference(route, i, r)
    return LP.excess(r["grad"] - want, mag), r


@pytest.mark.parametrize("route,i", LP.CASES, ids=[LP.case_id(*c) for c in LP.CASES])
def test_pair_against_closed_form(U, route, i):
    B, C, C_old, h, w, H, W = LP.SHAPES[route]
    cfg = LP.GRID[route][i]
    d = LP.make_inputs(route, i)
    err, r = measure(U, route, i)
    # which backward ran: one pair call, nothing else.  Any other call is a configuration that left the pair kernel.
    ran = {k: r["calls"][k] for k in OTHER_BWD if k in r["calls"]}
    assert ran == {PAIR[route]: 1}, ran
    assert err <= 1.0, "gradient off by %.3g x the bar (REL %g, FLOOR %g)" % (err, LP.REL, LP.FLOOR)
    # loss values, the CE valid count, the in-place label remap
    old_cl = LP.old_cl_of(cfg, C, C_old)
    ce, kd, ce_scale, kd_scale = LP.module_losses(cfg, r["x"], d["y"], r["t"], d["mask"], d["w_ce"], d["w_kd"], C_old)
    assert abs(r["ce"] - float(ce)) <= 1e-5 * ce_scale, (r["ce"], float(ce), ce_scale)
    assert abs(r["kd"] - float(kd)) <= 1e-5 * kd_scale, (r["kd"], float(kd), kd_scale)
    if r["n_valid"] is not None:
        assert r["n_valid"] == float((~LP.dead_pixels(d["y"], old_cl, cfg.ign, C)).sum())
    assert torch.equal(r["y"], LP.remap_labels(d["y"], old_cl))


def _rell2(a, b):
    return float((a - b).norm() / b.norm().clamp_min(1e-300))


@pytest.mark.parametrize("route,i", LR_CASES, ids=[LP.case_id(*c) for c in LR_CASES])
def test_lowres_reruns_and_two_step_path(U, route, i):
    """The low-res kernel gives the same bits on a rerun (range boundary rows: two atomicAdds onto zero), and agrees
    with the two-step path (full-res dx, then the upsample adjoint)."""
    a = run(U, route, i)
    b = run(U, route, i)
    assert torch.equal(a["grad"], b["grad"])
    two = run(U, route, i, plain=True)
    ran = {k: two["calls"][k] for k in OTHER_BWD if k in two["calls"]}
    assert ran == {"ucd_unce_unkd_bwd": 1, "ucd_upsample_bilinear_bwd": 1}, ran
    assert _rell2(a["grad"], two["grad"]) <= 1e-5


@pytest.mark.parametrize("route,i", LR_CASES, ids=[LP.case_id(*c) for c in LR_CASES])
def test_row_ranges_and_channel_groups(U, monkeypatch, route, i):
    """Ranges of three low-res rows (a short last range, rows shared by two ranges) and three channel groups of 5-6
    channels in blocks of 8 (a partial group), forced through the debug library's knobs: the same bar, same bits on
    a rerun."""
    from ucd_b200 import _lib
    dbg = _lib.debug_lib()
    monkeypatch.setenv("UCD_LRB_VARIANT", "0")
    monkeypatch.setenv("UCD_LRB_ROWS", "3")
    monkeypatch.setenv("UCD_LRB_GROUPS", "3")
    err, r = measure(U, route, i, handle=dbg)
    ran = {k: r["calls"][k] for k in OTHER_BWD if k in r["calls"]}
    assert ran == {"ucd_unce_unkd_bwd_lowres": 1}, ran
    assert err <= 1.0, "gradient off by %.3g x the bar (REL %g, FLOOR %g)" % (err, LP.REL, LP.FLOOR)
    again = run(U, route, i, handle=dbg)
    assert torch.equal(again["grad"], r["grad"])
