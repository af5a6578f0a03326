"""CPU checks of the closed-form oracle of the shared CE + KD logit backward (oracle/logit_pair.py) that
tests/test_gpu_logit_pair.py holds the kernels to: it equals autograd of the reference losses on every configuration
of the grid, the grid covers every pair of factor values, and every slip a kernel could plausibly make misses the GPU
bar by at least 10x wherever it changes the gradient (and changes nothing elsewhere)."""
import functools
import itertools

import pytest
import torch

from oracle import logit_pair as LP
from oracle import ucd_oracle as O


@functools.lru_cache(maxsize=None)
def operands(route, i):
    """fp64 full-res operands (x, t) of a case: for the low-res route the fp64 upsample of the low-res logits."""
    B, C, C_old, h, w, H, W = LP.SHAPES[route]
    d = LP.make_inputs(route, i)
    if route == "lr":
        return O.upsample_bilinear(d["logits"].double(), H, W), O.upsample_bilinear(d["old"].double(), H, W)
    return d["logits"].double(), d["old"].double()


def on_route(route, a):
    """A full-res quantity where the GPU test compares it: itself, or its adjoint for the low-res route."""
    B, C, C_old, h, w, H, W = LP.SHAPES[route]
    return LP.adjoint(a, h, w) if route == "lr" else a


@functools.lru_cache(maxsize=None)
def reference(route, i):
    x, t = operands(route, i)
    dx, mag = LP.oracle(route, i, x, t)
    return on_route(route, dx), on_route(route, mag)


def test_grid_covers_every_pair():
    for route, rows in LP.GRID.items():
        seen = {(f, getattr(r, f), g, getattr(r, g))
                for r in rows for f, g in itertools.combinations(LP.Cfg._fields, 2)}
        for f, g in itertools.combinations(LP.Cfg._fields, 2):
            for a in LP.FACTORS[f]:
                for b in LP.FACTORS[g]:
                    assert (f, a, g, b) in seen, (route, f, a, g, b)
        assert len(rows) <= 16
    assert len(LP.CASES) == sum(len(r) for r in LP.GRID.values())


@pytest.mark.parametrize("route,i", LP.CASES, ids=[LP.case_id(*c) for c in LP.CASES])
def test_closed_form_equals_autograd(route, i):
    """dx of the closed form == autograd of ucd_oracle.unbiased_ce / unbiased_kd / mask_kd (through
    ucd_oracle.upsample_bilinear for the low-res route), to 1e-12 of the largest magnitude."""
    B, C, C_old, h, w, H, W = LP.SHAPES[route]
    cfg = LP.GRID[route][i]
    d = LP.make_inputs(route, i)
    leaf = d["logits"].double().requires_grad_(True)
    if route == "lr":
        x, t = O.upsample_bilinear(leaf, H, W), O.upsample_bilinear(d["old"].double(), H, W)
    else:
        x, t = leaf, d["old"].double()
    ce, kd, _, _ = LP.module_losses(cfg, x, d["y"], t, d["mask"], d["w_ce"], d["w_kd"], C_old)
    a, b = LP.loss_weights(cfg)
    (a * ce + b * kd).backward()
    want, mag = reference(route, i)
    err = float((leaf.grad - want).abs().max())
    assert err <= 1e-12 * float(mag.max()), (err, float(mag.max()))
    assert float(want.abs().max()) > 0


# when a slip changes the gradient at all
APPLIES = {
    "alpha_qc": lambda c: c.alpha != 1.0,
    "ce_mean_bhw": lambda c: c.ce == "mean" and c.old_cl != "C",   # old_cl == C: every CE gradient is 0
    "mask_ignored": lambda c: c.mask is not None,
    "mask_zero_inverted": lambda c: c.kd == "mask" and c.mask is not None,
    "kd_old_from_old_cl": lambda c: c.old_cl != "C_old",
    "ignore_on_kd": lambda c: True,
    "g_px_image_off": lambda c: c.kd_red == "none_w" or (c.ce == "none_w" and c.old_cl != "C"),
}


def test_every_slip_is_listed():
    assert set(APPLIES) == set(LP.SLIPS)


@pytest.mark.parametrize("slip", LP.SLIPS)
def test_slip_misses_the_gpu_bar_by_10x(slip):
    """Each slip, applied to the oracle, differs from it by >= 10x the GPU bar (REL, FLOOR of oracle/logit_pair.py)
    in every grid case it applies to, on every route, and by < 1e-3 of the bar (rounding) where it does not apply."""
    hit = {route: 0 for route in LP.SHAPES}
    for route, i in LP.CASES:
        cfg = LP.GRID[route][i]
        want, mag = reference(route, i)
        x, t = operands(route, i)
        got, _ = LP.oracle(route, i, x, t, slip=slip)
        r = LP.excess(on_route(route, got) - want, mag)
        if APPLIES[slip](cfg):
            assert r >= 10, (slip, LP.case_id(route, i), r)
            hit[route] += 1
        else:
            assert r < 1e-3, (slip, LP.case_id(route, i), r)
    assert all(n > 0 for n in hit.values()), hit
