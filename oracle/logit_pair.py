"""Closed-form fp64 oracle of the shared UNCE + UNKD logit backward (csrc/ce_kd.cu: ``pair_args`` / ``pair_coef`` /
``pair_dx``, run by ``unce_unkd_bwd_kernel`` and, with the bilinear adjoint folded in, ``unce_unkd_bwd_lowres_kernel``).

Per element, with p = softmax(x), q = softmax(alpha t) over the C_old old channels, S_b = {0} u {C_old..C-1}:

    dx_c  = u_ce (p_c - sub_ce) + u_kd (p_c - sub_kd)
    sub_ce = [y' == 0] [c < old_cl] p_c e^(lse - lse_old) + [y' != 0] [c == y']       (y' = y remapped, 0 if y < old_cl)
    sub_kd = [c in S_b] p_c q_0 e^(lse - lse_b) + [1 <= c < C_old] q_c
    mag_c = |u_ce| (p_c + sub_ce) + |u_kd| (p_c + sub_kd)

u_ce / u_kd are the per-pixel upstream gradients after the reduction (``upstreams``): u_ce is 0 on dead pixels (label
== ignore_index, < 0 or >= C), u_kd carries 1 / C_old and the KD pixel weight (mask, or [mask == 0] for the masked
variant).  ``mag`` is the size of the terms whose difference is the gradient: an fp32 kernel that evaluates them with
relative error e is off by about e * mag, whatever the cancellation.  The GPU bar is |g - dx| <= REL mag + FLOOR
median(mag), per full-res element or, through ``adjoint`` (non-negative weights), per low-res cell.

``GRID`` is the set of configurations the tests run: per route (two full-res shapes, one for each vector width of
``unce_unkd_bwd_kernel``, and a 16x upsample that takes the low-res kernel), a covering array in which every pair of
values of the nine loss factors occurs at least once.  ``SLIPS`` are the plausible kernel mistakes the bar must reject:
``pair_dx`` / ``upstreams`` apply one when asked, so that a CPU test can show the bar sits well below each of them.
"""
from collections import namedtuple

import numpy as np
import torch

from . import ucd_oracle as O

REL = 3e-5      # per element: |g - dx| <= REL * mag + FLOOR * median(mag)
FLOOR = 1e-7

# (B, C, C_old, h, w, H, W); h, w = H, W: the logits are full-res (outputs = x * 1.0)
SHAPES = {
    "fr33x35": (2, 20, 14, 33, 35, 33, 35),      # HW odd: unce_unkd_bwd_kernel<1, ...>
    "fr64x96": (2, 20, 14, 64, 96, 64, 96),      # unce_unkd_bwd_kernel<4, ...>
    "lr": (2, 17, 16, 8, 16, 128, 256),          # outputs = interpolate_bilinear(lr): unce_unkd_bwd_lowres_kernel
}

Cfg = namedtuple("Cfg", "ce kd kd_red alpha mask ign old_cl order weights")
# ce: UnbiasedCrossEntropy reduction and how the value is used ('none' then .mean() / (w * ce).sum(), 'mean', 'sum');
# kd: UnbiasedKnowledgeDistillationLoss / MaskKnowledgeDistillationLoss, its reduction ('none' then (w * kd).sum());
# mask: KD pixel weight (None, bool, float in [0, 1] with exact zeros); ign: ignore_index (100 >= C: some pixels carry
# it); old_cl: CE's old_cl relative to KD's C_old; order: which loss is called first; weights: ce + 10 kd / 0.3 ce + kd
FACTORS = dict(ce=("none_mean", "none_w", "mean", "sum"), kd=("unbiased", "mask"), kd_red=("mean", "sum", "none_w"),
               alpha=(1.0, 0.5, 2.5), mask=(None, "bool", "float"), ign=(255, 100), old_cl=("C_old", "C_old-3", "C"),
               order=("ce", "kd"), weights=("ce+10kd", "0.3ce+kd"))
_G = {
    "fr33x35": """
        none_w unbiased sum 1.0 bool 100 C_old-3 kd ce+10kd
        sum mask none_w 2.5 None 255 C_old ce ce+10kd
        none_mean mask none_w 0.5 float 100 C kd 0.3ce+kd
        mean unbiased mean 0.5 bool 255 C ce 0.3ce+kd
        none_mean unbiased mean 2.5 None 100 C_old kd 0.3ce+kd
        none_w mask sum 1.0 float 255 C_old-3 ce 0.3ce+kd
        mean unbiased sum 2.5 float 100 C_old kd ce+10kd
        sum unbiased sum 1.0 None 100 C kd ce+10kd
        sum mask mean 0.5 float 100 C_old-3 ce ce+10kd
        mean mask none_w 2.5 bool 255 C_old-3 kd 0.3ce+kd
        none_mean unbiased sum 0.5 bool 255 C_old kd ce+10kd
        none_w unbiased none_w 0.5 None 100 C kd 0.3ce+kd
        none_mean mask mean 1.0 None 100 C_old-3 ce 0.3ce+kd
        mean mask none_w 1.0 None 100 C_old kd ce+10kd
        none_w unbiased mean 2.5 float 255 C_old ce ce+10kd
        sum unbiased mean 2.5 bool 100 C kd 0.3ce+kd""",
    "fr64x96": """
        none_w mask sum 1.0 float 255 C ce ce+10kd
        sum unbiased mean 2.5 bool 100 C_old ce 0.3ce+kd
        none_mean mask none_w 0.5 None 100 C_old-3 kd ce+10kd
        mean unbiased mean 0.5 float 255 C kd 0.3ce+kd
        mean mask none_w 1.0 None 255 C_old ce 0.3ce+kd
        none_w unbiased sum 2.5 bool 255 C_old-3 kd 0.3ce+kd
        none_mean unbiased none_w 2.5 float 100 C ce ce+10kd
        sum mask mean 1.0 bool 255 C_old-3 ce ce+10kd
        none_mean mask sum 0.5 bool 100 C_old kd 0.3ce+kd
        none_w unbiased mean 1.0 None 100 C_old kd ce+10kd
        mean mask sum 2.5 bool 100 C_old-3 kd ce+10kd
        sum mask sum 2.5 None 255 C kd ce+10kd
        none_w mask none_w 0.5 bool 100 C ce ce+10kd
        none_mean unbiased mean 1.0 float 255 C_old-3 ce ce+10kd
        sum mask none_w 0.5 float 100 C_old ce ce+10kd""",
    "lr": """
        none_w mask sum 2.5 float 100 C_old ce ce+10kd
        sum unbiased mean 1.0 None 255 C ce 0.3ce+kd
        none_w mask none_w 0.5 bool 255 C_old-3 kd 0.3ce+kd
        mean unbiased none_w 2.5 None 100 C_old-3 kd ce+10kd
        none_mean unbiased sum 1.0 bool 255 C_old kd 0.3ce+kd
        mean mask mean 0.5 bool 100 C kd ce+10kd
        none_mean unbiased mean 0.5 float 100 C_old-3 ce 0.3ce+kd
        sum unbiased none_w 2.5 float 255 C kd ce+10kd
        mean mask none_w 1.0 None 255 C_old ce ce+10kd
        sum mask sum 0.5 None 100 C_old ce ce+10kd
        none_mean mask mean 2.5 None 255 C_old ce 0.3ce+kd
        none_w unbiased mean 1.0 None 100 C ce 0.3ce+kd
        none_mean unbiased none_w 2.5 bool 100 C ce ce+10kd
        mean unbiased sum 1.0 float 255 C ce 0.3ce+kd
        sum unbiased sum 1.0 bool 100 C_old-3 kd 0.3ce+kd
        mean unbiased mean 0.5 None 255 C_old ce ce+10kd""",   # last: the trainer's modules with --alpha 0.5
}


def _parse(word, values):
    for v in values:
        if str(v) == word:
            return v
    raise ValueError(word)


GRID = {route: [Cfg(*(_parse(wd, FACTORS[f]) for wd, f in zip(line.split(), Cfg._fields)))
                for line in text.strip().splitlines()] for route, text in _G.items()}

CASES = [(route, i) for route in SHAPES for i in range(len(GRID[route]))]


def case_id(route, i):
    c = GRID[route][i]
    return "%s-%02d-%s-%s-%s" % (route, i, c.ce, c.kd, c.kd_red)


def old_cl_of(cfg, C, C_old):
    return {"C_old": C_old, "C_old-3": C_old - 3, "C": C}[cfg.old_cl]


def loss_weights(cfg):
    return (1.0, 10.0) if cfg.weights == "ce+10kd" else (0.3, 1.0)


def make_inputs(route, i):
    """Seeded fp32 inputs of case i of `route`: logits (low-res for 'lr'), old-model logits at the same resolution,
    int64 labels [B,H,W] (some pixels carry ignore_index), the KD mask (or None) and the per-pixel loss weights used
    by the 'none' reductions."""
    B, C, C_old, h, w, H, W = SHAPES[route]
    cfg = GRID[route][i]
    g = torch.Generator().manual_seed(1000 * list(SHAPES).index(route) + i)
    logits = (torch.randn(B, C, h, w, generator=g) * 3).clamp_(-10, 10)
    old = (torch.randn(B, C_old, h, w, generator=g) * 3).clamp_(-10, 10)
    y = torch.randint(0, C, (B, H, W), generator=g)
    y[torch.rand(B, H, W, generator=g) < 0.08] = cfg.ign
    mask = None
    if cfg.mask == "bool":
        mask = torch.rand(B, H, W, generator=g) > 0.3
    elif cfg.mask == "float":
        mask = torch.rand(B, H, W, generator=g)
        mask[torch.rand(B, H, W, generator=g) < 0.25] = 0.0
    w_ce = torch.rand(B, H, W, generator=g) * 2 - 0.5
    w_kd = torch.rand(B, H, W, generator=g) * 2 - 0.5
    return dict(logits=logits, old=old, y=y, mask=mask, w_ce=w_ce, w_kd=w_kd)


def remap_labels(y, old_cl):
    """What UnbiasedCrossEntropy leaves in its targets (in place, utils/loss.py:104-105)."""
    y = y.clone()
    y[y < old_cl] = 0
    return y


def dead_pixels(y, old_cl, ignore_index, C):
    yy = remap_labels(y, old_cl)
    return (yy == ignore_index) | (yy < 0) | (yy >= C)


def upstreams(cfg, y, C, C_old, w_ce, w_kd, slip=None):
    """(u_ce, u_kd) [B,H,W] fp64: the gradient that reaches each pixel's CE and KD term through the reduction, the use
    of the value (``module_losses``) and the loss weight.  Slips: 'ce_mean_bhw', 'g_px_image_off'."""
    B = y.shape[0]
    n = float(y[0].numel() * B)
    a, b = loss_weights(cfg)
    old_cl = old_cl_of(cfg, C, C_old)
    n_valid = float((~dead_pixels(y, old_cl, cfg.ign, C)).sum())
    one = torch.ones(y.shape, dtype=torch.float64)
    u_ce = {"none_mean": one * (a / n), "none_w": (a / n) * w_ce.double(),
            "mean": one * (a / (n if slip == "ce_mean_bhw" else n_valid)), "sum": one * (a / n)}[cfg.ce]
    u_kd = {"mean": one * (b / n), "sum": one * (b / n), "none_w": (b / n) * w_kd.double()}[cfg.kd_red]
    if slip == "g_px_image_off":
        u_ce, u_kd = u_ce.roll(1, 0), u_kd.roll(1, 0)
    return u_ce, u_kd


def pair_dx(x, y, t, *, old_cl, ignore_index, alpha, mask, variant, ce_up, kd_up, slip=None):
    """(dx, mag) [B,C,H,W] fp64 of the CE + KD pair (module docstring).  x [B,C,H,W] logits, y [B,H,W] int64 labels
    before the remap, t [B,C_old,H,W] old-model logits, variant 0 (unbiased KD, weight = mask) or 2 (masked KD,
    weight = [mask == 0]), ce_up / kd_up from ``upstreams``.  `slip` (one of SLIPS) computes a deliberately wrong
    variant instead."""
    x, t = x.double(), t.double()
    B, C = x.shape[:2]
    C_old = t.shape[1]
    lse = torch.logsumexp(x, 1, keepdim=True)
    p = torch.exp(x - lse)
    ch = torch.arange(C).view(1, C, 1, 1)
    # cross-entropy
    yy = remap_labels(y, old_cl)
    dead = dead_pixels(y, old_cl, ignore_index, C)
    u_ce = torch.where(dead, torch.zeros_like(ce_up), ce_up.double())
    bkg = ((yy == 0) & ~dead).unsqueeze(1) if old_cl > 0 else torch.zeros_like(dead).unsqueeze(1)
    lse_old = torch.logsumexp(x[:, :old_cl], 1, keepdim=True)
    sub_ce = torch.where(bkg, torch.where(ch < old_cl, torch.exp(x - lse_old), 0.0),
                         (ch == yy.unsqueeze(1)).double())
    # distillation
    q = torch.softmax(alpha * t, 1)
    bidx = [0] + list(range(C_old, C))
    lse_b = torch.logsumexp(x[:, bidx], 1, keepdim=True)
    qc = q
    if slip == "alpha_qc":   # q_c = e^(t_c - lse(alpha t)): alpha dropped from q_c, kept in q_0
        qc = torch.exp(t - torch.logsumexp(alpha * t, 1, keepdim=True))
    hi = old_cl if slip == "kd_old_from_old_cl" else C_old
    qpad = torch.zeros_like(x)
    n_t = min(hi, C_old)
    qpad[:, 1:n_t] = qc[:, 1:n_t]
    fg = (ch >= 1) & (ch < hi)
    sub_kd = torch.where(fg, qpad, p * q[:, :1] * torch.exp(lse - lse_b))
    u_kd = kd_up.double() / C_old
    if mask is not None and slip != "mask_ignored":
        m = mask.double()
        if variant == 2:
            m = ((m != 0) if slip == "mask_zero_inverted" else (m == 0)).double()
        u_kd = u_kd * m
    if slip == "ignore_on_kd":
        u_kd = torch.where(dead, torch.zeros_like(u_kd), u_kd)
    u_ce, u_kd = u_ce.unsqueeze(1), u_kd.unsqueeze(1)
    dx = u_ce * (p - sub_ce) + u_kd * (p - sub_kd)
    mag = u_ce.abs() * (p + sub_ce) + u_kd.abs() * (p + sub_kd)
    return dx, mag


SLIPS = ("alpha_qc", "ce_mean_bhw", "mask_ignored", "mask_zero_inverted", "kd_old_from_old_cl", "ignore_on_kd",
         "g_px_image_off")


def _tap_matrix(n_in, n_out):
    i0, i1, w0, w1 = O.bilinear_taps(n_in, n_out, np.float64)
    A = torch.zeros(n_out, n_in, dtype=torch.float64)
    r = torch.arange(n_out)
    A.index_put_((r, torch.from_numpy(i0)), torch.from_numpy(w0), accumulate=True)
    A.index_put_((r, torch.from_numpy(i1)), torch.from_numpy(w1), accumulate=True)
    return A


def adjoint(dx, h, w):
    """The bilinear upsample's adjoint in fp64: d lr [B,C,h,w] of a gradient dx [B,C,H,W] of the upsampled logits
    (F.interpolate(bilinear, align_corners=False) taps, ucd_oracle.bilinear_taps)."""
    H, W = dx.shape[-2:]
    return torch.einsum("bcyx,yi,xj->bcij", dx.double(), _tap_matrix(h, H), _tap_matrix(w, W))


def bar(mag):
    """Per-element tolerance of the GPU gradient."""
    return REL * mag + FLOOR * float(mag.median())


def excess(diff, mag):
    """max |diff| / bar(mag): <= 1 passes the GPU bar."""
    return float((diff.abs() / bar(mag)).max())


def module_losses(cfg, x, y, t, mask, w_ce, w_kd, C_old):
    """(ce value, kd value, ce scale, kd scale) of the configuration in fp64 through the reference losses of
    ucd_oracle (differentiable in x).  A 'sum' value and a weighted sum (w * loss).sum() are used divided by B * HW,
    as a training loop that weights pixels keeps them at the size of a mean: the two terms then reach the gradient at
    comparable size.  Otherwise one is ~B * HW smaller than the other everywhere, and no per-element (or per-cell) bar
    on the sum could see a mistake in it.  The scales are the sums of the magnitudes of the summed per-pixel terms: the
    size a relative tolerance on a value that may cancel is taken against."""
    C = x.shape[1]
    old_cl = old_cl_of(cfg, C, C_old)
    ce_px = O.unbiased_ce(x, y.clone(), old_cl, cfg.ign, "none")
    n_valid = (~dead_pixels(y, old_cl, cfg.ign, C)).sum()
    n = float(ce_px.numel())
    ce = {"none_mean": ce_px.mean(), "none_w": (w_ce.double() * ce_px).sum() / n, "mean": ce_px.sum() / n_valid,
          "sum": ce_px.sum() / n}[cfg.ce]
    ce_scale = {"none_mean": ce_px.abs().mean(), "none_w": (w_ce.double() * ce_px).abs().sum() / n,
                "mean": ce_px.abs().sum() / n_valid, "sum": ce_px.abs().sum() / n}[cfg.ce]
    kd_fn = O.unbiased_kd if cfg.kd == "unbiased" else O.mask_kd
    kd_px = kd_fn(x, t.double(), alpha=cfg.alpha, reduction="none", mask=mask)
    kd = {"mean": kd_px.mean(), "sum": kd_px.sum() / n, "none_w": (w_kd.double() * kd_px).sum() / n}[cfg.kd_red]
    kd_scale = {"mean": kd_px.abs().mean(), "sum": kd_px.abs().sum() / n,
                "none_w": (w_kd.double() * kd_px).abs().sum() / n}[cfg.kd_red]
    return ce, kd, float(ce_scale.detach()), float(kd_scale.detach())


def oracle(route, i, x, t, slip=None):
    """(dx, mag) of case i of `route` for full-res operands x [B,C,H,W] and t [B,C_old,H,W] (for 'lr': the upsampled
    logits the kernel reads)."""
    B, C, C_old, h, w, H, W = SHAPES[route]
    cfg = GRID[route][i]
    d = make_inputs(route, i)
    ce_up, kd_up = upstreams(cfg, d["y"], C, C_old, d["w_ce"], d["w_kd"], slip=slip)
    return pair_dx(x, d["y"], t, old_cl=old_cl_of(cfg, C, C_old), ignore_index=cfg.ign, alpha=cfg.alpha,
                   mask=d["mask"], variant=0 if cfg.kd == "unbiased" else 2, ce_up=ce_up, kd_up=kd_up, slip=slip)
