"""CPU oracle for the UCD distillation-loss hot path.  TEST INFRASTRUCTURE ONLY.

This module is the checker, never the product: only ``tests/``,
``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline / ``--impl reference``
legs may import it.  Nothing under ``ucd_b200/`` imports it, and the product path
raises if the CUDA library is missing instead of falling back to this code.

It restates, in closed form (numpy for the integer/label work, torch-CPU for the
floating point so that autograd yields reference gradients), what the reference
computes on this path:

* ``downsample_labels`` / ``prep_labels``  <- utils/loss.py:259-270, 354-361
* ``pre_contrastive_pixel``               <- utils/loss.py:273-276, 363-395 (``pixel_to_pixel``: :278-289)
* ``pixel_con_loss`` (+ closed-form grad, + row-blocked streaming form for large sizes) <- utils/loss.py:412-466
* ``unbiased_ce``                         <- utils/loss.py:96-109
* ``unbiased_kd``                         <- utils/loss.py:148-184
* ``upsample_bilinear``                   <- segmentation_module.py:133

The arithmetic of ``F.interpolate(mode='bilinear', align_corners=False)`` lives in
a third-party dependency (PyTorch ATen; requirements.txt pins torch==1.2.0, this
image runs 2.11.0).  Its CPU kernel is restated in ``bilinear_taps`` /
``_bilinear_eval_f32`` with the exact fp32 operation order that the x86 build
uses (found by exhaustive search over association orders and verified bit-exact
in tests/test_oracle.py against ``F.interpolate``): this matters because the
reference truncates the interpolated *label map* to int8, so the last ulp decides
labels (SURVEY.md §7 hard part 1).

Pinning: the reference ships no tests or golden vectors for this path.  The oracle
is pinned against outputs of the reference itself, run in the build container by
``oracle/gen_golden.py`` and committed under ``tests/golden/`` (see
tests/test_oracle.py).
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

F32 = np.float32


# ----------------------------------------------------------------------------
# bilinear taps (ATen area_pixel_compute_source_index, align_corners=False)
# ----------------------------------------------------------------------------
def _fma(a, b, c, ft):
    """fused multiply-add in float type ft (fp32 emulated through fp64: the product of two fp32 is
    exact in fp64 and the single rounding back to fp32 then equals a hardware fma up to rare double
    rounding; fp64 has no such emulation here and uses a*b+c)."""
    if ft is F32:
        return (np.asarray(a, F32).astype(np.float64) * np.asarray(b, F32).astype(np.float64)
                + np.asarray(c, F32).astype(np.float64)).astype(F32)
    return np.asarray(a, ft) * np.asarray(b, ft) + np.asarray(c, ft)


def bilinear_taps(in_size: int, out_size: int, ft=F32):
    """Source indices and weights of ATen's bilinear kernel along one axis, computed in the
    tensor's own float type ``ft`` (fp32 for the label map and fp32 logits).

    scale = ft(in)/out ; src = max(0, fma(scale, dst+0.5, -0.5)) ; i0 = floor(src)
    i1 = i0 + (i0 < in-1) ; w1 = src - i0 ; w0 = 1 - w1
    (the x86 build contracts scale*(dst+0.5)-0.5 into one fma; verified against F.interpolate)
    """
    if in_size == out_size:
        idx = np.arange(out_size, dtype=np.int64)
        return idx, idx.copy(), np.ones(out_size, ft), np.zeros(out_size, ft)
    scale = ft(in_size) / ft(out_size)
    dst = np.arange(out_size, dtype=ft)
    src = _fma(np.full_like(dst, scale), dst + ft(0.5), np.full_like(dst, ft(-0.5)), ft)
    src = np.maximum(src, ft(0)).astype(ft)
    i0 = np.minimum(np.floor(src).astype(np.int64), in_size - 1)
    i1 = i0 + (i0 < in_size - 1)
    w1 = np.clip((src - i0.astype(ft)).astype(ft), ft(0), ft(1)).astype(ft)
    w0 = (ft(1) - w1).astype(ft)
    return i0, i1, w0, w1


def _fma32(a, b, c):
    return _fma(a, b, c, F32)


def _bilinear_eval_f32(x: np.ndarray, out_h: int, out_w: int) -> np.ndarray:
    """Bit-exact restatement of ATen's CPU bilinear kernels on contiguous fp32 [..., H, W].

    ATen picks one of two kernels (UpSampleKernel.cpp, _use_vectorized_kernel_cond_2d):
      out_h + out_w <= 128 ("vectorized" kernel, the case of every UCD label map 32x32 .. 32x64):
          out = fma(h1*w1, x11, fma(h1*w0, x10, fma(h0*w0, x00, (h0*w1)*x01)))   weight products rounded first
      otherwise (generic N-d kernel, the case of the 512x512 logit upsample):
          t0 = fma(x00, w0, x01*w1) ; t1 = fma(x10, w0, x11*w1) ; out = fma(t0, h0, t1*h1)
    Both orders were found by exhaustive search and are verified bit-exact in tests/test_oracle.py.
    """
    x = np.asarray(x, F32)
    H, W = x.shape[-2:]
    y0, y1, hy0, hy1 = bilinear_taps(H, out_h)
    x0, x1, wx0, wx1 = bilinear_taps(W, out_w)
    v00 = x[..., y0[:, None], x0[None, :]]
    v01 = x[..., y0[:, None], x1[None, :]]
    v10 = x[..., y1[:, None], x0[None, :]]
    v11 = x[..., y1[:, None], x1[None, :]]
    bc = lambda v: np.broadcast_to(v, v00.shape)  # noqa: E731
    if out_h + out_w <= 128:
        k00 = (hy0[:, None] * wx0[None, :]).astype(F32)
        k01 = (hy0[:, None] * wx1[None, :]).astype(F32)
        k10 = (hy1[:, None] * wx0[None, :]).astype(F32)
        k11 = (hy1[:, None] * wx1[None, :]).astype(F32)
        acc = (k01 * v01).astype(F32)
        acc = _fma32(bc(k00), v00, acc)
        acc = _fma32(bc(k10), v10, acc)
        return _fma32(bc(k11), v11, acc)
    w0, w1, h0, h1 = bc(wx0[None, :]), bc(wx1[None, :]), bc(hy0[:, None]), bc(hy1[:, None])
    t0 = _fma32(v00, w0, (v01 * w1).astype(F32))
    t1 = _fma32(v10, w0, (v11 * w1).astype(F32))
    return _fma32(t0, h0, (t1 * h1).astype(F32))


# ----------------------------------------------------------------------------
# label part of pre_contrastive_pixel (integer results, must be bit exact)
# ----------------------------------------------------------------------------
def downsample_labels(labels, out_h: int, out_w: int, max_label: int = 20) -> np.ndarray:
    """utils/loss.py:261-270: bilinear-resize the label map in fp32, truncate toward
    zero, and zero everything outside [0, max_label].  int64 [B, h, w]."""
    lab = np.asarray(labels).astype(F32)
    g = np.trunc(_bilinear_eval_f32(lab, out_h, out_w)).astype(np.int64)
    # .type(int8) wraps values >= 128 to negatives on CPU; together with the two
    # masked fills (<0 -> 0, >max -> 0) this is "keep iff 0 <= g <= max_label".
    g[(g < 0) | (g > max_label)] = 0
    return g


@dataclass
class LabelPrep:
    label_n: np.ndarray     # int64 [B,h,w]  clamped low-res GT labels
    pseudo: np.ndarray      # int64 [B,h,w]  argmax_c l_po (first max)
    mix: np.ndarray         # int64 [B,h,w]  GT-new label if >0 else pseudo label
    anchor: np.ndarray      # bool  [B*h*w]  mix > 0
    pseudo_mask: np.ndarray  # bool [B*h*w]  anchor & ~is_new
    is_new: np.ndarray      # bool  [B*h*w]
    min_new: int            # min over GT-new labels


NO_NEW = 0x7f7f7f7f   # min_new of a batch without any new-class pixel (only with require_new=False)


def prep_labels(labels, l_po, max_label: int = 20, require_new: bool = True) -> LabelPrep:
    """utils/loss.py:354-361 (v2 branch).  ``require_new=False`` (rank-sharded oracle: the threshold is the minimum
    over all ranks) returns min_new = NO_NEW instead of raising when this batch has no new-class pixel."""
    l_po = np.asarray(l_po, F32)
    B, _, h, w = l_po.shape
    g = downsample_labels(labels, h, w, max_label)
    is_new = g.reshape(-1) > 0
    if not is_new.any() and require_new:
        raise ValueError("no new-class pixel in the batch (reference raises at utils/loss.py:355)")
    min_new = int(g.reshape(-1)[is_new].min()) if is_new.any() else NO_NEW
    pseudo = np.argmax(l_po, axis=1).astype(np.int64)   # first maximal index, like torch.max
    mix = np.where(g > 0, g, pseudo)
    anchor = mix.reshape(-1) > 0
    return LabelPrep(g, pseudo, mix, anchor, anchor & ~is_new, is_new, min_new)


# ----------------------------------------------------------------------------
# feature part + joint probability matrix
# ----------------------------------------------------------------------------
def _rows(x: torch.Tensor) -> torch.Tensor:
    """[B,C,h,w] -> [B*h*w, C] in (b,y,x) order."""
    B, C, h, w = x.shape
    return x.permute(0, 2, 3, 1).reshape(B * h * w, C)


def _unit(x: torch.Tensor, eps: float = 1e-12) -> torch.Tensor:
    return x / x.norm(dim=1, keepdim=True).clamp_min(eps)


def pre_contrastive_pixel(f_n: torch.Tensor, labels: torch.Tensor, l_po: torch.Tensor,
                          f_o: torch.Tensor, max_label: int = 20):
    """Restatement of the v2 branch, utils/loss.py:354-395.

    Returns (A, Cst, la, lc, P, prep): A keeps the autograd link to ``f_n``; Cst and P
    are detached, la/lc are int64 tensors, prep is the LabelPrep of the batch.
    """
    prep = prep_labels(labels.detach().cpu().numpy(), l_po.detach().cpu().numpy(), max_label)
    anchor = torch.from_numpy(prep.anchor)
    pseudo = torch.from_numpy(prep.pseudo_mask)
    mix = torch.from_numpy(prep.mix.reshape(-1))
    A = _unit(_rows(f_n)[anchor])
    Cst = torch.cat([A, _unit(_rows(f_o.detach())[pseudo])], dim=0).detach()
    la = mix[anchor]
    lc = torch.cat([la, mix[pseudo]])
    p = torch.softmax(_rows(l_po.detach()), dim=1)
    P = p[anchor] @ torch.cat([p[anchor], p[pseudo]]).T
    gt_a = la >= prep.min_new
    gt_c = lc >= prep.min_new
    P = torch.where(gt_a[:, None] & gt_c[None, :], torch.ones((), dtype=P.dtype), P)
    return A, Cst, la, lc, P.detach(), prep


def pixel_to_pixel(f_n: torch.Tensor, labels: torch.Tensor, f_o: Optional[torch.Tensor] = None, max_label: int = 20):
    """The branches of utils/loss.py:278-289 (no old-model logits): every pixel is a unit-norm row, labels are the
    clamped low-res label map; with ``f_o`` the detached old-model rows (and the labels again) are appended.
    Returns (Output [n, 1, 256], Lable [n] int64) like loss.py:399."""
    h, w = f_n.shape[-2:]
    lab = torch.from_numpy(downsample_labels(labels.cpu().numpy(), h, w, max_label).reshape(-1))
    out = _unit(_rows(f_n))
    if f_o is not None:
        out = torch.cat([out, _unit(_rows(f_o.detach()))])
        lab = torch.cat([lab, lab])
    return out.unsqueeze(1), lab


SELFCON_CASES = {"a": (300, 5, 1), "b": (777, 9, 1), "c": (260, 4, 2)}   # name: (rows, classes, views)


def selfcon_case(name: str):
    """Seeded inputs of the self-contrast fixtures (tests/golden/selfcon_losses.npz): unit-norm rows [n, views, 256]
    around class prototypes, labels with a dominant class and (case a) a class with a single member."""
    n, n_cls, views = SELFCON_CASES[name]
    g = torch.Generator().manual_seed(4321 + ord(name))
    proto = torch.randn(n_cls, 256, generator=g, dtype=torch.float64)
    lab = torch.randint(0, n_cls, (n,), generator=g)
    lab[:n // 3] = 0
    if name == "a":
        lab[lab == n_cls - 1] = 0
        lab[n - 1] = n_cls - 1
    x = 0.5 * torch.randn(n, views, 256, generator=g, dtype=torch.float64) + proto[lab][:, None, :]
    return torch.nn.functional.normalize(x, dim=2), lab


def pixel_con_loss_v1(features: torch.Tensor, labels: torch.Tensor, temperature: float = 1.0) -> torch.Tensor:
    """``PixelConLoss`` (v1) of utils/loss_new.py:354-400 restated: self-contrast of ``features`` [n, 1, D] (what the
    pixel-to-pixel branches of pre_contrastive_pixel return) with labels [n].

        s = F F^T / tau ;  R_ij = [l_i == l_j] ;  mp = R - I ;  neg_j = sum_k (1 - R_jk) exp(s_jk)
        loss = mean_{i: num_i != 0} ( -(1/num_i) sum_j mp_ij [ s_ij - log(exp(s_ij) + neg_j) ] )

    (loss_new.py:395 adds the COLUMN's negative sum - ``neg_contrast.repeat(batch_size, 1)`` - to exp(s_ij); s, R and
    mp are symmetric and num depends on the label only, so the value equals the row form, but the gradient reaches the
    features through both operands, through exp(s_ij) and through neg_j.)  Unshifted exponentials, like the reference."""
    f = features.reshape(features.shape[0], -1) if features.dim() == 2 else torch.cat(torch.unbind(features, dim=1), dim=0)
    lab = labels.reshape(-1, 1)
    n = f.shape[0]
    R = (lab.T == lab).to(f.dtype)
    mask_p = R - torch.eye(n, dtype=f.dtype)
    mask_n = 1 - R
    s = (f @ f.T) / temperature
    neg = (torch.exp(s) * mask_n).sum(dim=1)
    pos = s * mask_p - torch.log(torch.exp(s) + neg.repeat(n, 1)) * mask_p
    num = mask_p.sum(dim=1)
    keep = num != 0
    return (-(pos.sum(dim=1)[keep] / num[keep])).mean()


def sup_con_loss(features: torch.Tensor, labels: Optional[torch.Tensor] = None, temperature: float = 0.07,
                 contrast_mode: str = "all", base_temperature: float = 0.07) -> torch.Tensor:
    """``SupConLoss`` of utils/loss_new.py:263-352 restated (labels given, or None = SimCLR; the explicit ``mask``
    argument is not part of the path).  features [bsz, n_views, D]."""
    bsz, n_views = features.shape[0], features.shape[1]
    feats = features.reshape(bsz, n_views, -1)
    lab = (torch.arange(bsz) if labels is None else labels.reshape(-1)).reshape(-1, 1)
    mask = (lab == lab.T).float()   # fp32 whatever the feature dtype, like loss_new.py:303 (so `+ 1e-8` acts in fp32)
    contrast = torch.cat(torch.unbind(feats, dim=1), dim=0)
    if contrast_mode == "one":
        anchor, anchor_count = feats[:, 0], 1
    elif contrast_mode == "all":
        anchor, anchor_count = contrast, n_views
    else:
        raise ValueError("Unknown mode: {}".format(contrast_mode))
    adc = (anchor @ contrast.T) / temperature
    logits = adc - adc.max(dim=1, keepdim=True)[0].detach()
    mask = mask.repeat(anchor_count, n_views)
    logits_mask = torch.ones_like(mask)
    idx = torch.arange(bsz * anchor_count)
    logits_mask[idx, idx] = 0
    mask = mask * logits_mask
    exp_logits = torch.exp(logits) * logits_mask
    log_prob = logits - torch.log(exp_logits.sum(1, keepdim=True) + 1e-6)
    mean_log_prob_pos = (mask * log_prob).sum(1) / (mask.sum(1) + 1e-8)
    loss = -(temperature / base_temperature) * mean_log_prob_pos
    return loss.view(anchor_count, bsz).mean()


def contrast_operands(f_n: torch.Tensor, labels: torch.Tensor, l_po: torch.Tensor, f_o: torch.Tensor,
                      max_label: int = 20):
    """``pre_contrastive_pixel`` without the dense joint-probability matrix: returns
    (A, Cst, la, lc, pa, pc, prep) with pa / pc the old-model softmax rows of the anchors / contrast columns,
    so that ``pixel_con_loss_streaming`` can form P = pa pc^T (+ GT-new override, utils/loss.py:369-393) block
    by block.  Same row order as the reference (utils/loss.py:360-366)."""
    prep = prep_labels(labels.detach().cpu().numpy(), l_po.detach().cpu().numpy(), max_label)
    anchor = torch.from_numpy(prep.anchor)
    pseudo = torch.from_numpy(prep.pseudo_mask)
    mix = torch.from_numpy(prep.mix.reshape(-1))
    A = _unit(_rows(f_n)[anchor])
    Cst = torch.cat([A, _unit(_rows(f_o.detach())[pseudo])], dim=0).detach()
    la = mix[anchor]
    lc = torch.cat([la, mix[pseudo]])
    p = torch.softmax(_rows(l_po.detach()), dim=1)
    return A, Cst, la, lc, p[anchor], torch.cat([p[anchor], p[pseudo]]), prep


# ----------------------------------------------------------------------------
# PixelConLossV2 (closed form of SURVEY.md Appendix A.2)
# ----------------------------------------------------------------------------
def pixel_con_loss(A: torch.Tensor, Cst: torch.Tensor, la: torch.Tensor, lc: torch.Tensor,
                   P: Optional[torch.Tensor] = None, temperature: float = 0.07,
                   self_col: Optional[torch.Tensor] = None) -> torch.Tensor:
    """utils/loss.py:435-466.  ``self_col[i]`` is the contrast column holding anchor i
    itself (default i, the reference's ``eye`` on the first N_a columns)."""
    n_a = A.shape[0]
    same = (la.view(-1, 1) == lc.view(1, -1)).to(A.dtype)
    pos = same.clone()
    if self_col is None:
        self_col = torch.arange(n_a)
    ok = self_col >= 0
    pos[torch.arange(n_a)[ok], self_col[ok]] -= 1.0
    s = (A @ Cst.T) / temperature
    neg = (torch.exp(s) * (1.0 - same)).sum(dim=1, keepdim=True)        # unshifted
    sh = s - s.max(dim=1, keepdim=True).values.detach()
    w = pos if P is None else pos * P
    per_row = (w * (torch.log(torch.exp(sh)) - torch.log(torch.exp(sh) + neg))).sum(dim=1)
    num = pos.sum(dim=1)
    keep = num != 0
    return (-(per_row[keep] / num[keep])).mean()


def pixel_con_loss_closed_form(A, Cst, la, lc, P=None, temperature=0.07, self_col=None):
    """Loss and dL/dA without autograd (Appendix A.2) - used to cross-check autograd and
    as the specification of what the fused CUDA sweeps accumulate (V, U, T)."""
    A = A.detach()
    n_a = A.shape[0]
    same = (la.view(-1, 1) == lc.view(1, -1)).to(A.dtype)
    pos = same.clone()
    if self_col is None:
        self_col = torch.arange(n_a)
    ok = self_col >= 0
    pos[torch.arange(n_a)[ok], self_col[ok]] -= 1.0
    s = (A @ Cst.T) / temperature
    e = torch.exp(s)
    neg = (e * (1 - same)).sum(1, keepdim=True)
    m = s.max(1, keepdim=True).values
    sh = s - m
    den = torch.exp(sh) + neg
    w = pos if P is None else pos * P
    num = pos.sum(1)
    keep = num != 0
    M = int(keep.sum())
    row = (w * (sh - torch.log(den))).sum(1)
    loss = (-(row[keep] / num[keep])).sum() / M
    kappa = torch.where(keep, 1.0 / (M * torch.where(keep, num, torch.ones_like(num))),
                        torch.zeros_like(num))
    T = (w / den).sum(1)
    V = (e * (1 - same)) @ Cst                      # sum_k exp(s_ik) c_k over negatives
    U = (w * neg / den) @ Cst                       # sum_j w_ij neg_i/den_ij c_j
    dA = (kappa / temperature)[:, None] * (T[:, None] * V - U)
    return loss, dA


def pixel_con_loss_streaming(A, Cst, la, lc, pa=None, pc=None, min_new=None, temperature=0.07, self_col=None,
                             block=256, want_grad=True):
    """Row-blocked fp64 evaluation of utils/loss.py:412-466 (closed form of SURVEY.md Appendix A.2) with the
    joint-probability weights of utils/loss.py:369-393 formed block by block, so that memory is O(block x N_c)
    instead of O(N_a x N_c): the oracle for sizes where the dense restatement does not fit (the bench workload:
    23 419 x 41 102 pairs).  ``pa`` / ``pc`` are the softmax rows of the anchors / contrast columns (None: P == 1),
    ``min_new`` the GT-new threshold of the override ``P[i,j] = 1 where la_i >= min_new and lc_j >= min_new``.

    Returns (loss, dA or None, n_valid_rows); dA is dL/dA for the unit-norm anchor rows (fp64).  Checked against
    ``pixel_con_loss`` / ``pixel_con_loss_closed_form`` and the reference fixtures in tests/test_oracle.py.
    """
    A = A.detach().double()
    Cst = Cst.detach().double()
    n_a = A.shape[0]
    la, lc = la.reshape(-1).long(), lc.reshape(-1).long()
    if self_col is None:
        self_col = torch.arange(n_a)
    if pa is not None:
        pa, pc = pa.detach().double(), pc.detach().double()
        gt_c = lc >= int(min_new)
    row_sum = torch.zeros(n_a, dtype=torch.float64)
    num_all = torch.zeros(n_a, dtype=torch.float64)
    G = torch.zeros(n_a, A.shape[1], dtype=torch.float64) if want_grad else None
    for r0 in range(0, n_a, block):
        r1 = min(n_a, r0 + block)
        a = A[r0:r1]
        same = (la[r0:r1, None] == lc[None, :])
        pos = same.double()
        sc = self_col[r0:r1]
        ok = sc >= 0
        pos[torch.arange(r1 - r0)[ok], sc[ok]] -= 1.0
        s = (a @ Cst.T) / temperature
        e = torch.exp(s)
        e[same] = 0.0                                    # masked exp: negatives only
        neg = e.sum(1, keepdim=True)
        m = s.max(1, keepdim=True).values
        sh = s - m
        den = torch.exp(sh) + neg
        if pa is not None:
            w = pa[r0:r1] @ pc.T
            gt_a = la[r0:r1] >= int(min_new)
            w[gt_a[:, None] & gt_c[None, :]] = 1.0
            w *= pos
        else:
            w = pos
        num = pos.sum(1)
        row_sum[r0:r1] = (w * (sh - torch.log(den))).sum(1)
        num_all[r0:r1] = num
        if want_grad:
            T = (w / den).sum(1, keepdim=True)
            V = e @ Cst
            U = (w * (neg / den)) @ Cst
            k = torch.where(num != 0, 1.0 / (temperature * torch.where(num != 0, num, torch.ones_like(num))),
                            torch.zeros_like(num))
            G[r0:r1] = k[:, None] * (T * V - U)
    keep = num_all != 0
    M = int(keep.sum())
    loss = (-(row_sum[keep] / num_all[keep])).sum() / M
    return loss, (G / M if want_grad else None), M


# ----------------------------------------------------------------------------
# MiB unbiased cross-entropy / knowledge distillation
# ----------------------------------------------------------------------------
def unbiased_ce(x: torch.Tensor, y: torch.Tensor, old_cl: int, ignore_index: int = 255,
                reduction: str = "mean", mutate_labels: bool = True) -> torch.Tensor:
    """utils/loss.py:96-109.  ``y`` is remapped in place (y < old_cl -> 0) like the reference."""
    lse_all = torch.logsumexp(x, dim=1)
    lse_old = torch.logsumexp(x[:, :old_cl], dim=1)
    yy = y if mutate_labels else y.clone()
    yy[yy < old_cl] = 0
    ign = yy == ignore_index
    gather_idx = torch.where(ign, torch.zeros_like(yy), yy).unsqueeze(1)
    picked = x.gather(1, gather_idx).squeeze(1)
    per_px = torch.where(yy == 0, lse_all - lse_old, lse_all - picked)
    per_px = torch.where(ign, torch.zeros_like(per_px), per_px)
    if reduction == "none":
        return per_px
    if reduction == "sum":
        return per_px.sum()
    return per_px.sum() / (~ign).sum()          # nll_loss 'mean' divides by #non-ignored


def unbiased_kd(x: torch.Tensor, t: torch.Tensor, alpha: float = 1.0, reduction: str = "mean",
                mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """utils/loss.py:148-184 (the dead gamma/enc_out code at :155-156 has no effect)."""
    c_old = t.shape[1]
    lse_all = torch.logsumexp(x, dim=1)
    bkg_idx = [0] + list(range(c_old, x.shape[1]))
    lse_bkg = torch.logsumexp(x[:, bkg_idx], dim=1)
    q = torch.softmax(t * alpha, dim=1)
    per_px = (q[:, 0] * (lse_bkg - lse_all)
              + (q[:, 1:] * (x[:, 1:c_old] - lse_all.unsqueeze(1))).sum(dim=1)) / c_old
    if mask is not None:
        per_px = per_px * mask.to(per_px.dtype)
    if reduction == "mean":
        return -per_px.mean()
    if reduction == "sum":
        return -per_px.sum()
    return -per_px


# ----------------------------------------------------------------------------
# feature hand-off (SURVEY section 8(f), row N2)
# ----------------------------------------------------------------------------
def att_map(x: torch.Tensor) -> torch.Tensor:
    """segmentation_module.py:86-94: per-pixel energy sum_c x^2, divided per image by its Frobenius norm, applied as a
    detached positive per-pixel scale.  pre_contrastive_pixel L2-normalises every pixel's feature vector
    (utils/loss.py:363-365), so this scale cancels there: feeding the raw head output gives the same anchors and
    the same gradient with respect to the head output."""
    a = (x ** 2).sum(dim=1)
    a = a / a.flatten(1).norm(dim=1).view(-1, 1, 1)
    return a.unsqueeze(1).detach() * x


# ----------------------------------------------------------------------------
# sibling losses on the same kernels (SURVEY section 8(f), row N3)
# ----------------------------------------------------------------------------
def _reduce_neg(per_px: torch.Tensor, reduction: str) -> torch.Tensor:
    if reduction == "mean":
        return -per_px.mean()
    if reduction == "sum":
        return -per_px.sum()
    return -per_px


def plain_kd(x: torch.Tensor, t: torch.Tensor, alpha: float = 1.0, reduction: str = "mean",
             mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """utils/loss.py:112-136 (KnowledgeDistillationLoss): only the first C_old channels of x take part."""
    c_old = t.shape[1]
    xo = x[:, :c_old]
    q = torch.softmax(t * alpha, dim=1)
    per_px = (q * (xo - torch.logsumexp(xo, dim=1, keepdim=True))).sum(dim=1) / c_old
    if mask is not None:
        per_px = per_px * mask.to(per_px.dtype)
    return _reduce_neg(per_px, reduction)


def mask_kd(x: torch.Tensor, t: torch.Tensor, alpha: float = 1.0, reduction: str = "mean",
            mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """utils/loss.py:218-256 (MaskKnowledgeDistillationLoss): the unbiased KD of :148-184 on pixels with mask == 0."""
    sel = None if mask is None else (mask == 0)
    return unbiased_kd(x, t, alpha=alpha, reduction=reduction, mask=sel)


def mask_ce(x: torch.Tensor, y: torch.Tensor, old_cl: int, t_old: Optional[torch.Tensor] = None,
            ignore_index: int = 255, reduction: str = "mean") -> torch.Tensor:
    """utils/loss.py:186-216 (MaskCrossEntropy).  Labels are not remapped: a label in [1, old_cl) selects a
    zero-filled channel (contributes 0); pixel weight 1 where argmax(t_old) == 0 or label > old_cl.
    'mean'/'sum' come back negated, as the reference does (:213-215; SURVEY Appendix C6)."""
    lse_all = torch.logsumexp(x, dim=1)
    lse_old = torch.logsumexp(x[:, :old_cl], dim=1)
    y_safe = y.clamp(0, x.shape[1] - 1)
    picked = torch.gather(x, 1, y_safe.unsqueeze(1)).squeeze(1)
    per_px = torch.where(y == 0, lse_all - lse_old, lse_all - picked)
    dead = (y == ignore_index) | ((y >= 1) & (y < old_cl))
    per_px = torch.where(dead, torch.zeros_like(per_px), per_px)
    if t_old is not None:
        w = (torch.argmax(t_old, dim=1) == 0) | (y > old_cl)
        per_px = per_px * w.to(per_px.dtype)
    if reduction == "mean":
        return -per_px.mean()
    if reduction == "sum":
        return -per_px.sum()
    return per_px


# ----------------------------------------------------------------------------
# bilinear logit upsample (differentiable restatement)
# ----------------------------------------------------------------------------
def upsample_bilinear(x: torch.Tensor, out_h: int, out_w: int) -> torch.Tensor:
    """segmentation_module.py:133 - F.interpolate(bilinear, align_corners=False), written as
    explicit 4-tap gathers so autograd gives the adjoint the CUDA backward must match."""
    H, W = x.shape[-2:]
    ft = np.float64 if x.dtype == torch.float64 else F32
    y0, y1, hy0, hy1 = bilinear_taps(H, out_h, ft)
    x0, x1, wx0, wx1 = bilinear_taps(W, out_w, ft)
    ty0, ty1, tx0, tx1 = (torch.from_numpy(a) for a in (y0, y1, x0, x1))
    h0 = torch.from_numpy(hy0).to(x.dtype)[:, None]
    h1 = torch.from_numpy(hy1).to(x.dtype)[:, None]
    w0 = torch.from_numpy(wx0).to(x.dtype)[None, :]
    w1 = torch.from_numpy(wx1).to(x.dtype)[None, :]
    top, bot = x[..., ty0, :], x[..., ty1, :]
    return ((h0 * w1) * top[..., tx1] + (h0 * w0) * top[..., tx0]
            + (h1 * w0) * bot[..., tx0] + (h1 * w1) * bot[..., tx1])


# ----------------------------------------------------------------------------
# whole hot path, as train.py:115-116,133 combines it (5-tuple convention, SURVEY C1)
# ----------------------------------------------------------------------------
@dataclass
class HotPathResult:
    con: torch.Tensor
    ce: torch.Tensor
    kd: torch.Tensor
    total: torch.Tensor
    n_anchor: int
    n_contrast: int


def hot_path(f_n, f_o, l_po, logits_lr, labels, old_cl: int, temperature: float = 0.07,
             alpha: float = 1.0, kd_weight: float = 10.0, max_label: int = 20) -> HotPathResult:
    """loss = UNCE(outputs, labels).mean() + con/100 + kd_weight*UNKD(outputs, outputs_old)."""
    H, W = labels.shape[-2:]
    outputs = upsample_bilinear(logits_lr, H, W)
    outputs_old = upsample_bilinear(l_po.detach(), H, W).detach()
    A, Cst, la, lc, P, _ = pre_contrastive_pixel(f_n, labels, l_po, f_o, max_label)
    con = pixel_con_loss(A, Cst, la, lc, P, temperature)
    ce = unbiased_ce(outputs, labels.clone(), old_cl, 255, "none").mean()
    kd = unbiased_kd(outputs, outputs_old, alpha)
    return HotPathResult(con, ce, kd, ce + con / 100 + kd_weight * kd, A.shape[0], Cst.shape[0])


# ----------------------------------------------------------------------------
# multi-rank oracle: global-batch negatives (SURVEY.md §8e)
# ----------------------------------------------------------------------------
def pre_contrastive_pixel_global(f_n_list: Sequence[torch.Tensor], labels_list, l_po_list, f_o_list,
                                 max_label: int = 20):
    """Rank-sharded extension: rows stay per rank, columns are the concatenation over ranks of
    every rank's [anchors ; pseudo] block, min_new is the global minimum.  Returns per-rank
    (A_r, la_r, P_r, self_col_r) plus the shared (Cst, lc)."""
    preps = [prep_labels(l.cpu().numpy(), lp.detach().cpu().numpy(), max_label, require_new=False)
             for l, lp in zip(labels_list, l_po_list)]
    min_new = min(p.min_new for p in preps)
    if min_new == NO_NEW:
        raise ValueError("no new-class pixel in the global batch (reference raises at utils/loss.py:355)")
    A_l, C_l, la_l, lc_l, pa_l, pc_l, off = [], [], [], [], [], [], []
    col = 0
    for prep, f_n, f_o, l_po in zip(preps, f_n_list, f_o_list, l_po_list):
        anchor = torch.from_numpy(prep.anchor)
        pseudo = torch.from_numpy(prep.pseudo_mask)
        mix = torch.from_numpy(prep.mix.reshape(-1))
        A = _unit(_rows(f_n)[anchor])
        A_l.append(A)
        C_l.append(torch.cat([A.detach(), _unit(_rows(f_o.detach())[pseudo])]))
        la_l.append(mix[anchor])
        lc_l.append(torch.cat([mix[anchor], mix[pseudo]]))
        p = torch.softmax(_rows(l_po.detach()), dim=1)
        pa_l.append(p[anchor])
        pc_l.append(torch.cat([p[anchor], p[pseudo]]))
        off.append(col)
        col += C_l[-1].shape[0]
    Cst, lc, pc = torch.cat(C_l), torch.cat(lc_l), torch.cat(pc_l)
    out = []
    for A, la, pa, o in zip(A_l, la_l, pa_l, off):
        P = pa @ pc.T
        P = torch.where((la >= min_new)[:, None] & (lc >= min_new)[None, :], torch.ones((), dtype=P.dtype), P)
        out.append((A, la, P, o + torch.arange(A.shape[0])))
    return out, Cst, lc, min_new


def pixel_con_loss_global(per_rank, Cst, lc, temperature: float = 0.07) -> torch.Tensor:
    """Mean over all ranks' valid rows == the reference loss on the rank-concatenated batch
    (up to the column order, which the loss does not depend on)."""
    tot, cnt = 0.0, 0
    for A, la, P, self_col in per_rank:
        same = (la.view(-1, 1) == lc.view(1, -1)).to(A.dtype)
        pos = same.clone()
        pos[torch.arange(A.shape[0]), self_col] -= 1.0
        s = (A @ Cst.T) / temperature
        neg = (torch.exp(s) * (1 - same)).sum(1, keepdim=True)
        sh = s - s.max(1, keepdim=True).values.detach()
        row = (pos * P * (sh - torch.log(torch.exp(sh) + neg))).sum(1)
        num = pos.sum(1)
        keep = num != 0
        tot = tot + (-(row[keep] / num[keep])).sum()
        cnt += int(keep.sum())
    return tot / cnt


# ----------------------------------------------------------------------------
# synthetic inputs (SURVEY.md §8d / Appendix B generators)
# ----------------------------------------------------------------------------
def gen(seed: int, *shape, scale: float = 1.0) -> torch.Tensor:
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def blob_labels(B: int, H: int, W: int, c_old: int, c_tot: int) -> torch.Tensor:
    lab = torch.zeros(B, H, W, dtype=torch.int64)
    lab[:, H // 5:3 * H // 5, W // 5:3 * W // 5] = c_old
    lab[:, 3 * H // 5:4 * H // 5, W // 10:2 * W // 5] = c_tot - 1
    lab[:, :H // 25, :] = 255
    return lab


def synthetic_case(B: int, h: int, w: int, H: int, W: int, c_tot: int, c_old: int, rank: int = 0,
                   correlated: bool = False):
    """Seeds 1..4 (+1000*rank) for f_n, f_o, l_po, low-res new logits; blob labels."""
    o = 1000 * rank
    f_n, f_o = gen(1 + o, B, 256, h, w), gen(2 + o, B, 256, h, w)
    l_po = gen(3 + o, B, c_old, h, w, scale=3.0)
    lr = gen(4 + o, B, c_tot, h, w, scale=3.0)
    if correlated:
        proto = gen(9, c_tot, 256)
        cls = l_po.argmax(1)
        add = proto[cls].permute(0, 3, 1, 2)
        f_n, f_o = 0.3 * f_n + 0.7 * add, 0.3 * f_o + 0.7 * add
    return dict(f_n=f_n, f_o=f_o, l_po=l_po, logits_lr=lr, labels=blob_labels(B, H, W, c_old, c_tot))


LABEL_DOWNSAMPLE_SIZES = [(513, 513, 33, 33), (512, 512, 32, 32), (321, 321, 21, 21), (500, 375, 32, 24),
                          (512, 1024, 32, 64), (129, 257, 9, 17)]   # (H, W, h, w)


def label_downsample_maps():
    """Seeded label maps of the label-downsample fixture (tests/golden/label_downsample.npz), in generation order:
    {"rand<i>" / "block<i>": uint8 [2, H, W]} for the i-th entry of LABEL_DOWNSAMPLE_SIZES.  "rand" draws every pixel
    from 0..20; "block" holds constant 37 x 29 blocks (the rounding hazard of the resize) under an ignore band."""
    rng = torch.Generator().manual_seed(77)
    maps = {}
    for i, (H, W, _, _) in enumerate(LABEL_DOWNSAMPLE_SIZES):
        lab = torch.randint(0, 21, (2, H, W), generator=rng)
        blk = torch.randint(0, 21, (2, H // 37 + 1, W // 29 + 1), generator=rng)
        lab_b = blk.repeat_interleave(37, 1).repeat_interleave(29, 2)[:, :H, :W].clone()
        lab_b[:, : H // 20] = 255
        maps["rand%d" % i] = lab.numpy().astype(np.uint8)
        maps["block%d" % i] = lab_b.numpy().astype(np.uint8)
    return maps


def label_map_digest(lab: np.ndarray) -> str:
    """sha256 of a uint8 label map's bytes (C order): the fixture stores it so that generator drift is caught."""
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(lab, dtype=np.uint8).tobytes()).hexdigest()
