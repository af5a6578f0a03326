"""Operand-exact, per-row fp64 oracle of the contrastive sweeps (ucd_b200/csrc/contrast.cu) and a model of the
kernel's per-tile dispatch.  Test infrastructure only.

The aggregate oracles of ucd_oracle.py take the unrounded fp32 features, so a test that compares against them has to
absorb the bf16 quantisation of the operands.  Here the oracle reads the tiles the kernel multiplies (decoded to fp64),
so what is left between kernel and oracle is fp32 accumulation, the approximate ex2 / lg2 / rcp, the series truncation
and - unless emulated - the kernel's bf16 rounding of the E and Ucoef operands of the V and U products.  That makes a
per-row bar on the loss terms and on the gradient of every single row possible.

Tile layout (include/ucd_b200.h): element (r, k) of a 128-row tile sits at ((k/8)*128 + r)*8 + k%8, i.e. a tile is
[K/8][128][8] and ``tiles.permute(0, 2, 1, 3)`` gives [128][K/8][8] = rows.
"""
from collections import Counter

import torch

TILE = 128
WARP = 32
SERIES_NEG = 4096.0    # contrast.cu:740: a row takes the series form when neg_i >= 4096
NUM_SMS = 148          # kNumSMs (common.cuh)
MAX_TILES_PER_CTA = 4096
FINALIZE_BLOCKS = NUM_SMS * 4
INT_MAX = 0x7fffffff


# ----------------------------------------------------------------------------------------------------------------
# tiles <-> rows
# ----------------------------------------------------------------------------------------------------------------
def decode_tiles(tiles):
    """[T, K/8, 128, 8] tiles (bf16 features or probabilities) -> fp64 rows [T*128, K]."""
    T, kc, r, e = tiles.shape
    assert r == TILE and e == 8
    return tiles.detach().cpu().double().permute(0, 2, 1, 3).reshape(T * TILE, kc * 8)


def encode_tiles(rows, n_tiles):
    """fp32 rows [n, K] -> bf16 tiles [n_tiles, K/8, 128, 8], zero padded (the inverse of decode_tiles)."""
    n, K = rows.shape
    out = torch.zeros(n_tiles * TILE, K, dtype=torch.bfloat16, device=rows.device)
    out[:n] = rows.to(torch.bfloat16)
    return out.view(n_tiles, TILE, K // 8, 8).permute(0, 2, 1, 3).contiguous()


def _bf16(x):
    """Round to bf16 the way the kernel does: fp32 value, round-to-nearest-even (__floats2bfloat162_rn)."""
    return x.float().bfloat16().double()


# The kernel forms E and Ucoef in fp32 (fp32 accumulation of S, ex2.approx, rcp.approx): relative to the fp64 value they
# are off by about 1e-6.  An operand that close to a bf16 rounding boundary may round the other way, one bf16 step
# (2^-8 of the value): across 10^4 columns several per row do, and where one term dominates V or U that moves the row's
# gradient by up to ~0.5 % of its norm.  Either rounding is accepted for operands within FLIP_REL of a boundary.
FLIP_REL = 1e-5


def _flip_step(x):
    """|bf16 step| an operand may take by rounding the other way (0 where it is not within FLIP_REL of a boundary)."""
    return (_bf16(x * (1 + FLIP_REL)) - _bf16(x * (1 - FLIP_REL))).abs()


# ----------------------------------------------------------------------------------------------------------------
# PixelConLossV2 per row
# ----------------------------------------------------------------------------------------------------------------
def row_labels(lab_tiles_flat, n_rows):
    """The label a sweep thread carries for each row slot: the tile label, -2 for slots past n_rows (contrast.cu:728)."""
    rl = lab_tiles_flat.detach().cpu().long().clone()
    rl[n_rows:] = -2
    return rl


def con_rows(R, rl, C, lc, warps, *, inv_tau, pmode=0, pa=None, pc=None, min_new=None, P=None, self_tile0=0,
             emulate=True, want_grad=True, warps_per_block=8):
    """fp64 terms of every row of the given 32-row warps (contrast.cu:5-11), on the decoded operands.

    R [rows_pad, 256] decoded row tiles, rl [rows_pad] row labels with -2 past n_rows (``row_labels``), C [n_c, 256]
    the valid decoded columns, lc [n_c] their labels; ``self_tile0`` 0: row i excludes column i (when i < n_c), -1: no
    self column.  pmode 0: P == 1; 1: P = pa pc^T with the GT-new override (lc_j >= min_new for a row with
    la_i >= min_new); 2: dense P [n_rows, n_c].  inv_tau: the fp32 value the kernel gets.

    ``emulate``: round E_ij = exp(s_ij) and Ucoef_ij to bf16 like the kernel before the V / U products, with Ucoef from
    the formula of the path the row's warp takes: w (1 - x), x = exp(s - m) / neg_i, in the series form (every row of
    the warp has neg_i >= 4096), w neg_i / den_ij otherwise.  Rows past n_rows are evaluated too (as all-negative rows):
    they decide the warp's form together with the valid ones.

    Returns a dict of per-row tensors over rows = the warps' rows in order: row, m (max s), neg, num, L, T, loss
    (-L/num, 0 where num == 0), series (the warp's form), grad [.., 256] = d(sum_i loss_i)/d a_i and, with it, scale =
    (inv_tau/num_i)(|T_i| ||V_i|| + ||U_i||): the size of the two terms whose difference is the gradient, which fp32
    rounding of the V / U accumulation is relative to, and flip = (inv_tau/num_i)(|T_i| sum_j dE_ij |c_j| +
    sum_j dU_ij |c_j|) with dE / dU the bf16 step of the operands that may round either way (_flip_step): the most
    the emulation can be off by (emulate and want_grad)."""
    R, C = R.double(), C.double()
    lc = lc.long()
    n_c = C.shape[0]
    inv_tau = float(inv_tau)
    if pmode == 1:
        pa, pc = pa.double(), pc.double()
        gt_c = lc >= int(min_new)
    res = {k: [] for k in ("row", "m", "neg", "num", "L", "T", "loss", "series", "grad", "scale", "flip")}
    warps = sorted(set(int(w) for w in warps))
    for b0 in range(0, len(warps), warps_per_block):
        rows = torch.cat([torch.arange(w * WARP, (w + 1) * WARP) for w in warps[b0:b0 + warps_per_block]])
        la = rl[rows]
        s = (R[rows] @ C.T) * inv_tau
        same = la[:, None] == lc[None, :]
        pos = same.double()
        if self_tile0 == 0:
            hit = rows < n_c
            pos[hit.nonzero().squeeze(1), rows[hit]] -= 1.0
        e = torch.exp(s)
        e_neg = torch.where(same, torch.zeros_like(e), e)
        neg = e_neg.sum(1)
        m = s.max(1).values
        num = pos.sum(1)
        if pmode == 0:
            w = pos
        elif pmode == 1:
            pp = pa[rows] @ pc.T
            gt_a = la >= int(min_new)
            pp[gt_a[:, None] & gt_c[None, :]] = 1.0
            w = pos * pp
        else:
            valid = (rows < P.shape[0]).nonzero().squeeze(1)
            pp = torch.zeros_like(s)
            pp[valid] = P[rows[valid]].double()
            w = pos * pp
        eh = torch.exp(s - m[:, None])
        den = eh + neg[:, None]
        L = (w * (s - m[:, None] - torch.log(den))).sum(1)
        T = (w / den).sum(1)
        ser = (neg >= SERIES_NEG).view(-1, WARP).all(1).repeat_interleave(WARP)
        ok = num != 0
        loss = torch.where(ok, -L / torch.where(ok, num, torch.ones_like(num)), torch.zeros_like(L))
        res["row"].append(rows), res["m"].append(m), res["neg"].append(neg), res["num"].append(num)
        res["L"].append(L), res["T"].append(T), res["loss"].append(loss), res["series"].append(ser)
        if want_grad:
            ucoef = torch.where(ser[:, None], w * (1.0 - eh / neg[:, None]), w * neg[:, None] / den)
            k = torch.where(ok, inv_tau / torch.where(ok, num, torch.ones_like(num)), torch.zeros_like(num))
            if emulate:
                cn = C.norm(dim=1)
                res["flip"].append(k * (T.abs() * (_flip_step(e_neg) @ cn) + _flip_step(ucoef) @ cn))
                e_neg, ucoef = _bf16(e_neg), _bf16(ucoef)
            V = e_neg @ C
            U = ucoef @ C
            res["grad"].append(k[:, None] * (T[:, None] * V - U))
            res["scale"].append(k * (T.abs() * V.norm(dim=1) + U.norm(dim=1)))
    return {k: torch.cat(v) for k, v in res.items() if v}


def con_row_losses(R, rl, n_rows, C, lc, **kw):
    """(sum of the row losses over rows with num != 0, number of such rows): out[0], out[1] of ucd_con_fwd."""
    warps = range((n_rows + WARP - 1) // WARP)
    r = con_rows(R, rl, C, lc, warps, want_grad=False, **kw)
    keep = (r["row"] < n_rows) & (r["num"] != 0)
    return float(r["loss"][keep].sum()), int(keep.sum())


# ----------------------------------------------------------------------------------------------------------------
# self-contrast losses (PixelConLoss v1, SupConLoss) per row
# ----------------------------------------------------------------------------------------------------------------
def selfcon_rows(F, lab, mode, n_anchor, inv_tau, kappa=1.0):
    """fp64 per-row restatement of the self-contrast losses of ucd_selfcon_fwd on decoded rows F [n, 256]:
    returns (sum of the row losses, rows in the mean, d(sum)/dF [n, 256]).  mode 0 = PixelConLoss v1
    (ucd_oracle.pixel_con_loss_v1), 1 = SupConLoss with anchors = the first n_anchor rows (ucd_oracle.sup_con_loss)."""
    F = F.detach().double().clone().requires_grad_(True)
    n = F.shape[0]
    lab = lab.long().view(-1, 1)
    R = (lab == lab.T).double()
    eye = torch.eye(n, dtype=torch.float64)
    mp = R - eye
    s = (F @ F.T) * float(inv_tau)
    num = mp.sum(1)
    if mode == 0:
        neg = (torch.exp(s) * (1 - R)).sum(1)
        row = -(mp * (s - torch.log(torch.exp(s) + neg[None, :]))).sum(1)
        keep = num != 0
        per = row[keep] / num[keep]
    else:
        m = s.max(1, keepdim=True).values.detach()
        D = (torch.exp(s - m) * (1 - eye)).sum(1) + 1e-6
        mean_pos = (mp * (s - m - torch.log(D)[:, None])).sum(1) / (num.float() + 1e-8).double()   # fp32 like the reference's mask (and the kernel)
        per = -float(kappa) * mean_pos[:n_anchor]
        keep = torch.arange(n) < n_anchor
    total = per.sum()
    total.backward()
    return float(total.detach()), int(keep.sum()), F.grad.detach()


# ----------------------------------------------------------------------------------------------------------------
# plan and dispatch model
# ----------------------------------------------------------------------------------------------------------------
def choose_splits(row_tiles, col_tiles):
    """contrast.cu:1120-1135."""
    best, best_eff = 1, 0.0
    for s in range(1, 17):
        if s > 1 and col_tiles // s < 4:
            break
        ctas = row_tiles * s
        waves = (ctas + NUM_SMS - 1) // NUM_SMS
        eff = ctas / (waves * NUM_SMS)
        if eff > best_eff + 0.03:
            best_eff, best = eff, s
    while (col_tiles + best - 1) // best > MAX_TILES_PER_CTA:
        best += 1
    return best


def make_plan(max_row_tiles, max_col_tiles, plan_row_tiles=0, local_col_tiles=0):
    """contrast.cu:1141-1177 (product build: no tuning knobs).  Returns dict(splits, splits_local, splits2, rows_pad,
    total) with total = ucd_con_workspace_bytes."""
    if plan_row_tiles <= 0 or plan_row_tiles > max_row_tiles:
        plan_row_tiles = max_row_tiles
    if 0 < local_col_tiles < max_col_tiles:
        splits_local = choose_splits(plan_row_tiles, local_col_tiles)
        splits = choose_splits(plan_row_tiles, max_col_tiles - local_col_tiles)
    else:
        splits_local, splits = 0, choose_splits(plan_row_tiles, max_col_tiles)
    best = choose_splits(plan_row_tiles, max_col_tiles)
    splits2 = (best + 1) // 2 if best > 1 else 1
    while (max_col_tiles + splits - 1) // splits > MAX_TILES_PER_CTA:
        splits += 1
    while (max_col_tiles + splits2 - 1) // splits2 > MAX_TILES_PER_CTA:
        splits2 += 1
    rows_pad = max_row_tiles * TILE
    s1 = splits + splits_local
    total = 0
    for nbytes in (s1 * 3 * rows_pad * 4, 3 * rows_pad * 4, splits2 * 2 * rows_pad * 4, s1 * rows_pad * 256 * 4,
                   splits2 * rows_pad * 256 * 4, 2 * FINALIZE_BLOCKS * 4):
        total += (nbytes + 255) & ~255
    return dict(splits=splits, splits_local=splits_local, splits2=splits2, rows_pad=rows_pad, total=total)


def _ranges(labels, n, n_tiles):
    """min / max valid label of every 128-entry tile over entries [0, n) (ucd_con_tile_ranges)."""
    out = []
    for t in range(n_tiles):
        seg = labels[t * TILE:min(n, (t + 1) * TILE)]
        seg = seg[seg >= 0]
        out.append((int(seg.min()), int(seg.max())) if seg.numel() else (INT_MAX, -INT_MAX))
    return out


def dispatch(rl, n_rows, lc, *, pmode, min_new=None, neg=None, self_tile0=0, splits=1, splits2=1, old_uniform=False):
    """Counts of the kernel's epilogue branches over (row block, warp, column tile) for one single-chunk ucd_con_fwd.

    rl: row labels [rows_pad] with -2 past n_rows (row_labels); lc: the valid column labels [n_c]; neg: fp64 neg_i of
    every row slot (con_rows over all warps) or None to skip the series / exact split.  Keys:
      s1_all_neg / s1_full / s1_partial_self  (per row block and tile, contrast.cu:770, 793-798)
      s2_skip (tile outside the row block's label range, contrast.cu:480-496, 498-506), s2_cta_idle (a sweep-2 CTA with
      columns but no active tile), and per warp of an active tile
      s2_uniform_ones / s2_uniform_p / s2_general_full / s2_general_partial_self, each with a _series / _exact suffix
      when neg is given (contrast.cu:817-861; series: every row slot of the warp has neg_i >= 4096, contrast.cu:740-751)
      warp_series / warp_exact / warp_mixed (warps with a valid row), false_uniform (warps the uniform test without the
      row-label condition accepted although their rows carry two labels; with old_uniform=True they are dispatched to
      the uniform path like the kernel before the fix did).
    Returns (Counter, list of (row block, warp, tile) with false_uniform)."""
    rl = rl.long()
    lc = lc.long()
    n_c = lc.numel()
    col_tiles = (n_c + TILE - 1) // TILE
    row_tiles = (n_rows + TILE - 1) // TILE
    lc_pad = torch.full((col_tiles * TILE,), -1, dtype=torch.long)
    lc_pad[:n_c] = lc
    crange = _ranges(lc_pad, n_c, col_tiles)
    rrange = _ranges(rl.clamp_min(-1), n_rows, row_tiles)
    cnt, false_uni = Counter(), []
    for rb in range(row_tiles):
        rlo, rhi = rrange[rb]
        self_tile = rb if self_tile0 == 0 else -1
        active = [t == self_tile or not (crange[t][1] < rlo or crange[t][0] > rhi) for t in range(col_tiles)]
        for t in range(col_tiles):
            full = min(TILE, n_c - t * TILE) == TILE
            is_self = t == self_tile
            cnt["s1_all_neg" if full and not active[t] else
                "s1_full" if full and not is_self else "s1_partial_self"] += 1
        per = (col_tiles + splits2 - 1) // splits2
        for sp in range(splits2):
            k0, k1 = sp * per, min(col_tiles, sp * per + per)
            if k1 > k0 and not any(active[k0:k1]):
                cnt["s2_cta_idle"] += 1
        for wq in range(TILE // WARP):
            r0 = rb * TILE + wq * WARP
            la = rl[r0:r0 + WARP]
            if not bool((la != -2).any()):
                continue
            sfx = ""
            if neg is not None:
                nw = neg[r0:r0 + WARP]
                valid = la != -2
                ser = bool((nw >= SERIES_NEG).all())
                sfx = "_series" if ser else "_exact"
                nv = nw[valid]
                cnt["warp_series" if ser else
                    "warp_mixed" if bool((nv >= SERIES_NEG).any()) else "warp_exact"] += 1
            for t in range(col_tiles):
                if not active[t]:
                    if wq == 0:
                        cnt["s2_skip"] += 1
                    continue
                full = min(TILE, n_c - t * TILE) == TILE
                is_self = t == self_tile
                uni = uni_old = False
                if pmode in (0, 1) and full and not is_self:
                    cols = lc_pad[t * TILE:(t + 1) * TILE].view(WARP, 4)
                    uni_old = bool((cols == la[:, None]).all())
                    uni = uni_old and bool((la == la[0]).all())
                if uni_old and not uni:
                    cnt["false_uniform"] += 1
                    false_uni.append((rb, wq, t))
                if uni or (uni_old and old_uniform):
                    ones = pmode == 0 or int(la[0]) >= int(min_new)
                    cnt[("s2_uniform_ones" if ones else "s2_uniform_p") + sfx] += 1
                else:
                    cnt[("s2_general_full" if full and not is_self else "s2_general_partial_self") + sfx] += 1
    return cnt, false_uni


def class_sorted_labels(labels, l_po, max_label):
    """Class-sorted anchor and contrast labels of a batch as the prep kernels tile them (stable sort by label of the
    anchors, then of the pseudo columns: include/ucd_b200.h:172-175), from the oracle's label prep."""
    from oracle import ucd_oracle as O
    prep = O.prep_labels(labels.numpy() if hasattr(labels, "numpy") else labels,
                         l_po.numpy() if hasattr(l_po, "numpy") else l_po, max_label, require_new=False)
    mix = torch.from_numpy(prep.mix.reshape(-1)).long()
    la = torch.sort(mix[torch.from_numpy(prep.anchor)], stable=True).values
    lo = torch.sort(mix[torch.from_numpy(prep.pseudo_mask)], stable=True).values
    return la, torch.cat([la, lo]), prep.min_new
