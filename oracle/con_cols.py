"""PixelConLossV2 with respect to the contrast features (SURVEY.md Appendix A.2, column side): the fp64 closed form of
dL/dC, and its operand-exact per-column form for the transposed sweep of ucd_con_contrast_grad
(ucd_b200/csrc/contrast.cu: sweep3c_cols).  Test infrastructure only.

    G_ij = dL/ds_ij = kappa_i (-w_ij neg_i / den_ij + negm_ij T_i exp(s_ij)),   kappa_i = [num_i != 0] / (M num_i)
    dL/da_i = (1/tau) sum_j G_ij c_j ;  dL/dc_j = (1/tau) sum_i G_ij a_i

P (w = pos * P) and the row max m_i are constants, as in the reference (P detached, max detached)."""
import torch

from oracle.con_rows import SERIES_NEG, _bf16, _flip_step  # noqa: F401  (SERIES_NEG: re-exported for the tests)


def _terms(A, Cst, la, lc, P, temperature, self_col, kernel_self):
    n_a = A.shape[0]
    same = (la.view(-1, 1) == lc.view(1, -1)).to(A.dtype)
    pos = same.clone()
    if self_col is None:
        self_col = torch.arange(n_a)
    ok = self_col >= 0
    rows, cols = torch.arange(n_a)[ok], self_col[ok]
    pos[rows, cols] -= 1.0       # the reference's R - eye: -1 where the self pair's labels differ
    wpos = pos.clone()
    if kernel_self:              # the sweeps: the self pair never carries a positive weight (it is counted in num_i)
        wpos[rows, cols] = 0.0
    s = (A @ Cst.T) / temperature
    e = torch.exp(s)
    negm = 1.0 - same
    neg = (e * negm).sum(1, keepdim=True)
    m = s.max(1, keepdim=True).values
    den = torch.exp(s - m) + neg
    w = wpos if P is None else wpos * P
    num = pos.sum(1)
    keep = num != 0
    return dict(s=s, e=e, negm=negm, neg=neg, m=m, den=den, w=w, num=num, keep=keep)


def pixel_con_loss_grads(A, Cst, la, lc, P=None, temperature=0.07, self_col=None):
    """(loss, dL/dA, dL/dCst) of utils/loss.py:435-466 in closed form, fp64 on fp64 inputs, P constant.  Same
    conventions as ucd_oracle.pixel_con_loss (``self_col[i]``: the contrast column holding anchor i, default i)."""
    A, Cst = A.detach(), Cst.detach()
    t = _terms(A, Cst, la, lc, None if P is None else P.detach(), temperature, self_col, kernel_self=False)
    keep, num, w, den, neg = t["keep"], t["num"], t["w"], t["den"], t["neg"]
    M = int(keep.sum())
    sh = t["s"] - t["m"]
    row = (w * (sh - torch.log(den))).sum(1)
    loss = (-(row[keep] / num[keep])).sum() / M
    kappa = torch.where(keep, 1.0 / (M * torch.where(keep, num, torch.ones_like(num))), torch.zeros_like(num))
    T = (w / den).sum(1, keepdim=True)
    G = kappa[:, None] * (-w * neg / den + t["negm"] * T * t["e"])
    return loss, (G @ Cst) / temperature, (G.T @ A) / temperature


# bar of the GPU tests on the kernel's own operands: |g_j - g_ref_j| <= REL |g_ref_j| + FLOOR scale_j + flip_j
REL = 5e-4
FLOOR = 3e-5

# plausible kernel slips (contrast_cols(slip=...)); tests/test_con_contrast_grad_cpu.py shows each misses the bar by 10x
SLIPS = ("self_kept", "p_untransposed", "t_missing", "m_all_rows", "max_not_detached")


def contrast_cols(R, rl, C, lc, inv_tau, P=None, self_tile0=0, emulate=True, slip=None):
    """Per contrast column, on the decoded operands of the kernel (fp64): dL/dc_j (g = 1) as ucd_con_contrast_grad +
    ucd_con_bwd form it, inv_tau sum_i H_ji a_i / M with H_ji = M G_ij, and the size of its terms.

    R [rows_pad, 256] decoded anchor tiles, rl [rows_pad] their labels with -2 past n_rows (con_rows.row_labels), C
    [n_c, 256] the decoded contrast columns, lc [n_c]; P None or dense [n_a, n_c]; self_tile0 0: anchor i and column i
    are the self pair (i < min(n_a, n_c)), -1: none.  The self pair follows the sweeps: no positive weight, counted -1 in
    num_i when its labels differ (sweep 1), a negative when they differ.  ``emulate``: round H to bf16 like the kernel.
    ``slip``: one of SLIPS, a deliberately wrong variant.

    Returns dict(grad [n_c, 256], scale [n_c] = inv_tau sum_i |H_ji| |a_i| / M (what fp32 accumulation error is
    relative to), flip [n_c] = inv_tau sum_i dH_ji |a_i| / M with dH the bf16 step of the operands within FLIP_REL of a
    rounding boundary (0 without emulation), M, and num / T / neg of the anchors)."""
    R, C = R.double(), C.double()
    valid = rl != -2
    A = R[valid]
    la = rl[valid].long()
    n_a, n_c = A.shape[0], C.shape[0]
    inv_tau = float(inv_tau)
    ar = torch.arange(n_a)
    if self_tile0 == 0:
        self_col = torch.where(ar < n_c, ar, -torch.ones(n_a, dtype=torch.long))
    else:
        self_col = -torch.ones(n_a, dtype=torch.long)
    Pd = None if P is None else P.double()
    if slip == "p_untransposed" and Pd is not None:   # P[j * ldp + i] read for pair (i, j)
        flat = Pd.reshape(-1)
        idx = torch.arange(n_c)[None, :] * n_c + ar[:, None]
        Pd = torch.where(idx < flat.numel(), flat[idx.clamp_max(flat.numel() - 1)], torch.zeros((), dtype=Pd.dtype))
    t = _terms(A, C, la, lc.long(), Pd, 1.0 / inv_tau, self_col, kernel_self=True)
    keep, num, w, den, neg = t["keep"], t["num"], t["w"], t["den"], t["neg"]
    if slip == "self_kept":     # the self pair weighted like any equal-label pair
        ok = self_col >= 0
        same_d = (la[ar[ok]] == lc.long()[self_col[ok]]).double()
        w = w.clone()
        w[ar[ok], self_col[ok]] = same_d * (1.0 if Pd is None else Pd[ar[ok], self_col[ok]])
    M = int(keep.sum())
    k = torch.where(keep, 1.0 / torch.where(keep, num, torch.ones_like(num)), torch.zeros_like(num))
    T = (w / den).sum(1, keepdim=True)
    if slip == "self_kept":
        T = (t["w"] / den).sum(1, keepdim=True)       # the forward's T is unchanged
    TT = torch.ones_like(T) if slip == "t_missing" else T
    H = k[:, None] * (-w * neg / den + t["negm"] * TT * t["e"])       # [n_a, n_c] = H^T
    if slip == "max_not_detached":   # d loss_i / d m_i = sum_j w_ij neg_i / den_ij / num_i flows to the argmax column
        H = H.clone()
        H[ar, t["s"].argmax(1)] += k * (w * neg / den).sum(1)
    an = A.norm(dim=1)
    Mn = n_a if slip == "m_all_rows" else M
    flip = torch.zeros(n_c, dtype=torch.float64)
    if emulate:
        flip = inv_tau * (_flip_step(H).T @ an) / Mn
        H = _bf16(H)
    grad = inv_tau * (H.T @ A) / Mn
    scale = inv_tau * (H.abs().T @ an) / Mn
    return dict(grad=grad, scale=scale, flip=flip, M=M, num=num, T=T.squeeze(1), neg=neg.squeeze(1))


def excess(g, ref):
    """max over columns of |g_j - g_ref_j| / (REL |g_ref_j| + FLOOR scale_j + flip_j): <= 1 passes the GPU bar."""
    bar = REL * ref["grad"].norm(dim=1) + FLOOR * ref["scale"] + ref["flip"]
    return float(((g - ref["grad"]).norm(dim=1) / bar.clamp_min(1e-300)).max())
