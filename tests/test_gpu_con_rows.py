"""Row-by-row checks of the fused contrastive sweeps (ucd_b200/csrc/contrast.cu) through the C ABI, against the
operand-exact fp64 oracle of oracle/con_rows.py evaluated on the very bf16 tiles the kernel multiplies.

The aggregate bars of test_gpu_parity.py (loss within 1e-3, gradient cosine >= 0.999 against the unrounded fp32
features) must absorb the bf16 quantisation of the operands; they cannot see an error confined to a few rows or a
per-row magnitude error.  Here every checked row must satisfy

    || g_i - g_ref_i || <= GRAD_TOL || g_ref_i || + CANCEL_TOL scale_i + flip_i,
    scale_i = (|T_i| ||V_i|| + ||U_i||) / (tau num_i)

with the oracle emulating the kernel's one deliberate rounding (E and Ucoef to bf16).  The gradient is the difference
of the two terms T_i V_i and U_i; fp32 accumulation error is relative to their size, and for a row that is already
well fitted they cancel to a gradient a thousand times smaller, so the second term of the bar is set per row from that
size (not from the largest row).  flip_i bounds what the operands within 1e-5 of a bf16 rounding boundary can do when
the kernel's fp32 value rounds them the other way (oracle/con_rows.py: FLIP_REL): without it a few rows of the
full-size cases, those where one negative dominates V_i, miss the oracle by up to 7e-3 of their norm.  The sum of the row losses must agree to LOSS_TOL and the number of rows in the mean
exactly.  The bars sit well below the smallest effect they must catch: the spurious positives of the old sweep-2
uniform test changed the gradient of the affected rows by a median of 0.9 % (VOC rank 3) to 5.7 % (Cityscapes rank 0).

Each case runs twice, with plan_row_tiles = 1 and with a 48-row-tile plan (other column splits, sweep-2 CTAs without an
active tile); both must meet the bars and agree to fp32 summation order.  need_grad = 0 must give bit-identical
`out`.  The dispatch model of oracle/con_rows.py shows that the hand-built cases reach every epilogue branch.

Observed on an NVIDIA B200 (1000 W power limit), recorded here when the bars were set: see the constants below."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import con_rows as R
from oracle import ucd_oracle as O

pytestmark = pytest.mark.gpu

# bars (about 10x the largest value observed on the B200, see the module docstring)
GRAD_TOL = 5e-4       # per-row gradient error relative to |g_i|, PixelConLossV2 with rounding emulation
CANCEL_TOL = 3e-5     # ... plus this much of scale_i = (|T_i| |V_i| + |U_i|) / (tau num_i) (fp32 rounding of the terms)
LOSS_TOL = 5e-6       # relative error of the sum of row losses
PLAN_TOL = 5e-5       # per-row difference of two plans relative to |g_i| (plus CANCEL_TOL scale_i)
SELF_GRAD_TOL = 5e-2  # self-contrast losses: per-row relative gradient error; H is rounded to bf16 and not emulated
FLOOR_REL = 1e-6      # self-contrast floor relative to the median row norm
TAU = 0.07
BIG_PLAN = 48


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ucd_b200
    from ucd_b200 import _lib
    assert _lib.lib().ucd_device_ok() == 1, "ucd_b200 needs a compute-capability 10.x device"
    torch.set_num_threads(max(1, torch.get_num_threads()))
    return ucd_b200


def _L():
    from ucd_b200 import _lib
    return _lib.lib()


def _p(t):
    from ucd_b200._lib import ptr
    return ptr(t)


def _check(rc, what):
    from ucd_b200._lib import check
    check(rc, what)


# ------------------------------------------------------------------------------------------------------------------
# operands: hand-built (ucd_con_pack_rows, like the compat path) or the main path's pack
# ------------------------------------------------------------------------------------------------------------------
class Operands:
    """Device buffers of one single-chunk ucd_con_fwd call plus the decoded fp64 operands of the oracle."""

    def decode(self):
        self.R = R.decode_tiles(self.rfeat_t)
        self.rl = R.row_labels(self.rlab_t.reshape(-1), self.n_a)
        self.C = R.decode_tiles(self.feat_t)[:self.n_c]
        self.lc = self.lab_t.reshape(-1)[:self.n_c].cpu().long()
        if self.pmode == 1:
            self.pa = R.decode_tiles(self.rprob_t)
            self.pc = R.decode_tiles(self.prob_t)[:self.n_c]
        return self

    def oracle_kw(self):
        kw = dict(inv_tau=np.float32(1 / TAU), pmode=self.pmode, self_tile0=0)
        if self.pmode == 1:
            kw.update(pa=self.pa, pc=self.pc, min_new=self.min_new)
        if self.pmode == 2:
            kw.update(P=self.P.double().cpu())
        return kw


def hand_operands(A, C, la, lc, pmode=0, pa=None, pc=None, min_new=None, P=None):
    L, st = _L(), None
    dev = "cuda"
    n_a, n_c = A.shape[0], C.shape[0]
    rt, ct = -(-n_a // 128), -(-n_c // 128)
    o = Operands()
    o.n_a, o.n_c, o.rt, o.ct, o.pmode = n_a, n_c, rt, ct, pmode
    o.rfeat_t = torch.empty(rt, 32, 128, 8, device=dev, dtype=torch.bfloat16)
    o.feat_t = torch.empty(ct, 32, 128, 8, device=dev, dtype=torch.bfloat16)
    o.rlab_t = torch.empty(rt, 128, device=dev, dtype=torch.int32)
    o.lab_t = torch.empty(ct, 128, device=dev, dtype=torch.int32)
    a32, c32 = A.float().cuda().contiguous(), C.float().cuda().contiguous()
    la32, lc32 = la.int().cuda().contiguous(), lc.int().cuda().contiguous()
    _check(L.ucd_con_pack_rows(_p(a32), _p(la32), n_a, _p(o.rfeat_t), _p(o.rlab_t), rt, st), "pack_rows")
    _check(L.ucd_con_pack_rows(_p(c32), _p(lc32), n_c, _p(o.feat_t), _p(o.lab_t), ct, st), "pack_rows")
    o.rrange = torch.empty(rt, 2, device=dev, dtype=torch.int32)
    o.crange = torch.empty(ct, 2, device=dev, dtype=torch.int32)
    _check(L.ucd_con_tile_ranges(_p(o.rlab_t), rt, None, _p(o.rrange), st), "tile_ranges")
    _check(L.ucd_con_tile_ranges(_p(o.lab_t), ct, None, _p(o.crange), st), "tile_ranges")
    o.counts = torch.tensor([[n_c, 0]], device=dev, dtype=torch.int32)
    o.n_rows = torch.tensor([n_a], device=dev, dtype=torch.int32)
    o.kpad, o.rprob_t, o.prob_t, o.min_new_t, o.P, o.min_new = 16, None, None, None, None, None
    o.row_ref = None
    if pmode == 1:
        o.kpad = L.ucd_con_prob_kpad(pa.shape[1])
        pad = lambda p: F.pad(p.float(), (0, o.kpad - p.shape[1])).cuda()  # noqa: E731
        o.rprob_t = R.encode_tiles(pad(pa), rt)
        o.prob_t = R.encode_tiles(pad(pc), ct)
        o.min_new = int(min_new)
        o.min_new_t = torch.tensor([o.min_new], device=dev, dtype=torch.int32)
    if pmode == 2:
        o.P = P.float().cuda().contiguous()
    return o.decode()


def main_operands(U, case, max_label=20):
    f_n = case["f_n"].cuda()
    tup = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda(),
                                  max_label=max_label)
    pk = tup[4].pack
    o = Operands()
    o.pack = pk
    o.n_a, o.n_c, o.pmode, o.kpad, o.min_new = pk.n_a, pk.n_c, 1, pk.kpad, pk.min_new
    o.rt, o.ct = max(1, -(-pk.n_a // 128)), pk.max_tiles
    o.feat_t, o.prob_t, o.lab_t = pk.feat_tiles, pk.prob_tiles, pk.lab_tiles
    o.rfeat_t, o.rprob_t, o.rlab_t = pk.feat_tiles[:o.rt], pk.prob_tiles[:o.rt], pk.lab_tiles[:o.rt]
    o.rrange, o.crange, o.counts = pk.row_range, pk.tile_range, pk.counts
    o.n_rows, o.min_new_t, o.row_ref, o.P = pk.counts, pk.counts[2:3], pk.row_ref, None
    return o.decode()


def run_fwd(o, need_grad=1, max_row_tiles=None, plan=0):
    L = _L()
    mrt = max_row_tiles or o.rt
    ws_bytes = L.ucd_con_workspace_bytes(mrt, o.ct, plan, 0)
    ws = torch.empty(ws_bytes, device="cuda", dtype=torch.uint8)
    out = torch.full((3,), float("nan"), device="cuda")
    grad = torch.full((mrt * 128, 256), float("nan"), device="cuda") if need_grad else None
    _check(L.ucd_con_fwd(_p(o.feat_t), _p(o.prob_t), _p(o.lab_t), _p(o.counts), 1, o.ct, 0, -1, 0, _p(o.rfeat_t),
                         _p(o.rprob_t), _p(o.rlab_t), _p(o.n_rows), _p(o.crange), _p(o.rrange), 0, _p(o.min_new_t),
                         o.pmode, o.kpad, _p(o.P), 0 if o.P is None else o.P.shape[1], float(np.float32(1 / TAU)),
                         need_grad, _p(out), _p(grad), _p(ws), ws_bytes, mrt, plan, None), "con_fwd")
    torch.cuda.synchronize()
    return out.cpu(), (grad.cpu()[:o.n_a].double() if need_grad else None), grad


def row_errors(g, ref):
    """per-row error, row norm and the floor of the self-contrast bar (from the row-norm distribution: the median, not
    the max)."""
    nr = ref.norm(dim=1)
    err = (g - ref).norm(dim=1)
    floor = FLOOR_REL * float(nr.median())
    return err, nr, floor


STATS = {}


def check_con(name, o, warps=None):
    """The per-row checks of one PixelConLossV2 case; returns the oracle terms."""
    kw = o.oracle_kw()
    all_warps = range(-(-o.n_a // 32))
    ref = R.con_rows(o.R, o.rl, o.C, o.lc, all_warps if warps is None else warps, **kw)
    out1, g1, g1_dev = run_fwd(o, 1, o.rt, 1)
    out2, g2, _ = run_fwd(o, 1, max(BIG_PLAN, o.rt), BIG_PLAN)
    out0, _, _ = run_fwd(o, 0, o.rt, 1)
    assert torch.equal(out0, out1), (name, out0, out1)     # sweep 2's L_i does not read V
    if warps is None:
        keep = (ref["row"] < o.n_a) & (ref["num"] != 0)
        total, M = float(ref["loss"][keep].sum()), int(keep.sum())
    else:
        total, M = R.con_row_losses(o.R, o.rl, o.n_a, o.C, o.lc, **kw)
    assert int(out1[1]) == M, (name, float(out1[1]), M)
    loss_err = abs(float(out1[0]) - total) / abs(total)
    sel = ref["row"] < o.n_a
    rows = ref["row"][sel]
    gref = ref["grad"][sel]
    scale, flip = ref["scale"][sel], ref["flip"][sel]
    nr = gref.norm(dim=1)
    errs, cerrs = {}, {}
    for tag, g in (("plan1", g1), ("plan%d" % BIG_PLAN, g2)):
        err = (g[rows] - gref).norm(dim=1)
        bad = err > GRAD_TOL * nr + CANCEL_TOL * scale + flip
        errs[tag] = float((err / nr.clamp_min(1e-300)).max())
        cerrs[tag] = float((err / scale.clamp_min(1e-300)).max())
        assert not bool(bad.any()), (name, tag, "rows", rows[bad][:8].tolist(),
                                     (err / nr.clamp_min(1e-300))[bad][:8].tolist())
    dp = (g1[rows] - g2[rows]).norm(dim=1)
    dplan = float((dp / nr.clamp_min(1e-300)).max())
    STATS[name] = dict(loss_err=loss_err, grad_err=max(errs.values()), plan_diff=dplan, rows=int(rows.numel()))
    print("\n[%s] rows %d  loss rel err %.2e  row grad err max %.2e of |g_i| (median %.2e), %.2e of scale_i; "
          "plans differ by %.2e of |g_i|, %.2e of scale_i" %
          (name, rows.numel(), loss_err, max(errs.values()), float(((g1[rows] - gref).norm(dim=1) / nr).median()),
           max(cerrs.values()), dplan, float((dp / scale.clamp_min(1e-300)).max())))
    assert loss_err <= LOSS_TOL, (name, loss_err)
    assert abs(float(out1[0]) - float(out2[0])) <= LOSS_TOL * abs(float(out1[0]))
    assert int(out2[1]) == M
    assert not bool((dp > PLAN_TOL * nr + CANCEL_TOL * scale).any()), (name, dplan)
    return ref, out1, g1_dev


# ------------------------------------------------------------------------------------------------------------------
# hand-built cases
# ------------------------------------------------------------------------------------------------------------------
def _unit(x):
    return F.normalize(x, dim=1)


def reproducer(k):
    """N_a = 128, N_c = 256: warp 0 holds labels 1 | 2 split at lane k, column tile 1 holds 1 | 2 split at 4k."""
    g = torch.Generator().manual_seed(100 + k)
    A = _unit(torch.randn(128, 256, generator=g, dtype=torch.float64))
    C = torch.cat([A, _unit(torch.randn(128, 256, generator=g, dtype=torch.float64))])
    la = torch.full((128,), 3, dtype=torch.long)
    la[:k], la[k:32] = 1, 2
    lc = torch.cat([la, torch.full((128,), 2, dtype=torch.long)])
    lc[128:128 + 4 * k] = 1
    return A, C, la, lc


def class_sorted(n, n_lab, g, weights=None):
    w = torch.ones(n_lab) if weights is None else torch.tensor(weights, dtype=torch.float64)
    return torch.sort(torch.multinomial(w.double(), n, replacement=True, generator=g) + 1).values


# name: (n_a, n_c, pmode, c_old, align)  align: "series" (a shared direction: neg_i >> 4096), "exact" (neg_i < 4096),
# "mixed" (the shared direction only in every other row: warps straddle the threshold)
HAND = {
    "a1_c1025_p0_series": (1, 1025, 0, 0, "series"),
    "a31_c1663_p1_k16_exact": (31, 1663, 1, 16, "exact"),
    "a32_c1536_p2_mixed": (32, 1536, 2, 0, "mixed"),
    "a33_c1537_p1_k101_series": (33, 1537, 1, 101, "series"),
    "a127_c1663_p1_k141_exact": (127, 1663, 1, 141, "exact"),
    "a128_c2048_p0_mixed": (128, 2048, 0, 0, "mixed"),
    "a129_c1409_p1_k16_series": (129, 1409, 1, 16, "series"),
    "a300_c2560_p1_k121_mixed": (300, 2560, 1, 121, "mixed"),
    "a700_c3327_p1_k16_series": (700, 3327, 1, 16, "series"),
    "a520_c1793_p2_exact": (520, 1793, 2, 0, "exact"),
    "a400_c2177_p0_exact": (400, 2177, 0, 0, "exact"),
}


def hand_case(name):
    n_a, n_c, pmode, c_old, align = HAND[name]
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    n_lab = 6
    # class-sorted like the prep's tiles: anchors, then the other columns; the top label is "GT-new" (>= min_new)
    la = class_sorted(n_a, n_lab, g, [3, 1, 4, 1, 2, 3])
    lo = class_sorted(n_c - n_a, n_lab, g, [2, 5, 1, 3, 1, 2])
    lc = torch.cat([la, lo])
    proto = torch.randn(n_lab + 1, 256, generator=g, dtype=torch.float64)
    common = _unit(torch.randn(1, 256, generator=g, dtype=torch.float64))

    def feats(lab, n):
        x = 0.6 * _unit(proto[lab]) + 0.8 * _unit(torch.randn(n, 256, generator=g, dtype=torch.float64))
        if align == "series":
            x = 0.45 * _unit(x) + 0.55 * common
        elif align == "mixed":
            x = _unit(x) + (torch.arange(n) % 2 == 0).double()[:, None] * 1.2 * common
        return _unit(x)
    A = feats(la, n_a)
    C = torch.cat([A, feats(lo, n_c - n_a)])
    kw = {}
    if pmode == 1:
        pa = torch.softmax(3 * torch.randn(n_a, c_old, generator=g), 1)
        pc = torch.cat([pa, torch.softmax(3 * torch.randn(n_c - n_a, c_old, generator=g), 1)])
        kw = dict(pa=pa, pc=pc, min_new=n_lab)
    if pmode == 2:
        kw = dict(P=torch.rand(n_a, n_c, generator=g))
    return A, C, la, lc, pmode, kw


@pytest.mark.parametrize("k", [1, 5, 17, 31])
def test_reproducer_compat_p_none(U, k):
    """PixelConLossV2 compat path, P = None (PMODE 0): warp 0 of row block 0 holds two labels split at lane k and
    column tile 1 the same labels split at column 4k.  The uniform test without the row-label condition took that
    pair for an all-positive tile and added 4k or 128 - 4k spurious positives to every row of the warp."""
    A, C, la, lc = reproducer(k)
    o = hand_operands(A, C, la, lc)
    check_con("repro_p0_k%d" % k, o)


def test_reproducer_main_path_city_rank0(U):
    """The single-GPU Cityscapes bench input (bench.make_inputs('city') rank 0, 5777 x 10159): rows 3392-3423 (row
    block 26, warp 2) against column tile 71, labels 10 | 11.  Every row is checked."""
    case = O.synthetic_case(3, 32, 64, 512, 1024, 20, 14, rank=0, correlated=True)
    o = main_operands(U, case)
    assert (o.n_a, o.n_c) == (5777, 10159)
    ref, out, _ = check_con("city_rank0", o)
    assert set(range(3392, 3424)) <= set(ref["row"].tolist())


def test_reproducer_main_path_small_seed(U):
    """A seeded two-image VOC-like batch (rank 40 of the bench generator) with a false-uniform warp: row block 4,
    warp 0 against column tile 19 (tests/test_con_rows_cpu.py keeps the seed honest)."""
    case = O.synthetic_case(2, 32, 32, 512, 512, 17, 16, rank=40, correlated=True)
    o = main_operands(U, case)
    check_con("small_rank40", o)


def test_reproducer_pixelconloss_v1(U):
    """PixelConLoss v1 (ucd_selfcon_fwd mode 0) launches the same sweep 2 with P == 1: n = 256, row block 0 warp 0
    split at lane 17, column tile 1 split at column 68."""
    A, C, la, lc = reproducer(17)
    rows = C.clone()
    lab = lc.clone()
    check_selfcon("repro_v1_k17", rows, lab, 0, 256, 1.0)


@pytest.mark.parametrize("name", sorted(HAND))
def test_hand_built_case(U, name):
    A, C, la, lc, pmode, kw = hand_case(name)
    o = hand_operands(A, C, la, lc, pmode, **kw)
    check_con(name, o)


@pytest.mark.parametrize("c_tot,c_old,max_label", [(151, 101, 150), (151, 141, 150)])
def test_main_path_wide_joint_probability(U, c_tot, c_old, max_label):
    """The prep's pack with ADE-like class counts: kpad 112 (chunked pC) and 144 (both probability operands
    streamed)."""
    case = O.synthetic_case(2, 32, 32, 512, 512, c_tot, c_old, correlated=True)
    o = main_operands(U, case, max_label)
    check_con("main_k%d" % c_old, o)


def test_con_bwd_scatter(U):
    """ucd_con_bwd: d_anchor[row_ref[i]] = g g_mul / out[1] grad_unit[i] to fp32 rounding; rows it does not own stay
    untouched."""
    case = O.synthetic_case(2, 32, 32, 512, 512, 17, 16, rank=40, correlated=True)
    o = main_operands(U, case)
    out, _, grad_dev = run_fwd(o, 1)
    out_dev = out.cuda()
    g = torch.tensor([0.37], device="cuda")
    extra = 40
    d = torch.full((o.n_a + extra, 256), 7.0, device="cuda")
    _check(_L().ucd_con_bwd(_p(grad_dev), _p(out_dev), _p(g), 2.0, _p(o.n_rows), _p(o.row_ref), _p(d), o.n_a + extra,
                            None), "con_bwd")
    torch.cuda.synchronize()
    d = d.cpu()
    ref = torch.zeros(o.n_a, 256, dtype=torch.float64)
    ref[o.row_ref.cpu().long()[:o.n_a]] = grad_dev.cpu()[:o.n_a].double() * (0.37 * 2.0 / float(out[1]))
    torch.testing.assert_close(d[:o.n_a].double(), ref, rtol=4e-7, atol=1e-30)
    assert bool((d[o.n_a:] == 7.0).all())
    # identity scatter (row_ref NULL) on a hand-built case
    A, C, la, lc = reproducer(5)
    h = hand_operands(A, C, la, lc)
    out, _, grad_dev = run_fwd(h, 1)
    d = torch.zeros(128, 256, device="cuda")
    _check(_L().ucd_con_bwd(_p(grad_dev), _p(out.cuda()), _p(g), 1.0, _p(h.n_rows), None, _p(d), 128, None), "con_bwd")
    torch.cuda.synchronize()
    torch.testing.assert_close(d.cpu().double(), grad_dev.cpu()[:128].double() * (0.37 / float(out[1])),
                               rtol=4e-7, atol=1e-30)


# ------------------------------------------------------------------------------------------------------------------
# self-contrast losses
# ------------------------------------------------------------------------------------------------------------------
def check_selfcon(name, rows, lab, mode, n_anchor, tau, kappa=1.0):
    L = _L()
    n = rows.shape[0]
    tiles = -(-n // 128)
    x = F.pad(rows.float(), (0, 256 - rows.shape[1])).cuda().contiguous()
    lab32 = lab.int().cuda().contiguous()
    feat = torch.empty(tiles, 32, 128, 8, device="cuda", dtype=torch.bfloat16)
    ltile = torch.empty(tiles, 128, device="cuda", dtype=torch.int32)
    rng = torch.empty(tiles, 2, device="cuda", dtype=torch.int32)
    _check(L.ucd_con_pack_rows(_p(x), _p(lab32), n, _p(feat), _p(ltile), tiles, None), "pack_rows")
    _check(L.ucd_con_tile_ranges(_p(ltile), tiles, None, _p(rng), None), "tile_ranges")
    meta = torch.tensor([n, 0, n], device="cuda", dtype=torch.int32)
    ws_bytes = L.ucd_selfcon_workspace_bytes(tiles)
    ws = torch.empty(ws_bytes, device="cuda", dtype=torch.uint8)
    res = []
    for need_grad in (1, 0):
        out = torch.empty(3, device="cuda")
        grad = torch.empty(n, 256, device="cuda") if need_grad else None
        _check(L.ucd_selfcon_fwd(_p(feat), _p(ltile), _p(rng), _p(meta), meta.data_ptr() + 8, n, n_anchor, mode,
                                 float(np.float32(1 / tau)), kappa, need_grad, _p(out), _p(grad), _p(ws), ws_bytes,
                                 None), "selfcon_fwd")
        torch.cuda.synchronize()
        res.append((out.cpu(), None if grad is None else grad.cpu().double()))
    (out, g), (out0, _) = res
    assert torch.equal(out, out0), (name, out, out0)
    Fd = R.decode_tiles(feat)[:n]
    total, M, gref = R.selfcon_rows(Fd, lab, mode, n_anchor, float(np.float32(1 / tau)), kappa)
    assert int(out[1]) == M
    loss_err = abs(float(out[0]) - total) / abs(total)
    err, nr, floor = row_errors(g, gref)
    rel = err / nr.clamp_min(1e-300)
    STATS[name] = dict(loss_err=loss_err, grad_err=float(rel.max()), rows=n)
    print("\n[%s] rows %d  loss rel err %.2e  max row grad rel err %.2e (median %.2e)" %
          (name, n, loss_err, float(rel.max()), float(rel.median())))
    assert loss_err <= LOSS_TOL, (name, loss_err)
    bad = err > SELF_GRAD_TOL * nr + floor
    assert not bool(bad.any()), (name, torch.nonzero(bad).view(-1)[:8].tolist(), rel[bad][:8].tolist())


@pytest.mark.parametrize("mode,anchors,case", [(0, "all", "b"), (0, "all", "sorted"), (1, "all", "c"),
                                               (1, "one", "c"), (1, "all", "sorted")])
def test_selfcon_rows(U, mode, anchors, case):
    """PixelConLoss v1 and SupConLoss ('all' / 'one'), every row against the operand-exact oracle; the gradient flows
    through both operands via sweep 3.  'sorted': a class-sorted set with tiles of one label (uniform sweep-2 tiles)."""
    if case == "sorted":
        g = torch.Generator().manual_seed(5)
        lab = class_sorted(700, 4, g, [5, 1, 3, 2]) - 1
        proto = torch.randn(4, 256, generator=g, dtype=torch.float64)
        x = _unit(proto[lab] + 1.5 * torch.randn(700, 256, generator=g, dtype=torch.float64))[:, None]
    else:
        x, lab = O.selfcon_case(case)
    views = x.shape[1]
    rows = torch.cat(torch.unbind(x, dim=1), dim=0)
    labs = lab.repeat(views)
    tau = 1.0 if mode == 0 else 0.1
    n_anchor = x.shape[0] if anchors == "one" else rows.shape[0]
    check_selfcon("selfcon_m%d_%s_%s" % (mode, anchors, case), rows, labs, mode, n_anchor, tau,
                  tau / 0.07 if mode else 1.0)


# ------------------------------------------------------------------------------------------------------------------
# branch coverage of the hand-built cases (dispatch model)
# ------------------------------------------------------------------------------------------------------------------
BRANCHES = ["s1_all_neg", "s1_full", "s1_partial_self", "s2_skip", "s2_cta_idle",
            "s2_uniform_ones_series", "s2_uniform_ones_exact", "s2_uniform_p_series", "s2_uniform_p_exact",
            "s2_general_full_series", "s2_general_full_exact", "s2_general_partial_self_series",
            "s2_general_partial_self_exact", "warp_series", "warp_exact", "warp_mixed", "false_uniform"]


def test_hand_built_cases_reach_every_branch():
    """The dispatch model replayed on the hand-built cases (the bf16-rounded operands, fp64 neg_i) reaches every
    epilogue branch of both sweeps, every PMODE and probability width, partial last tiles of N_c mod 128 in
    {0, 1, 127}, N_a in {1, 31, 32, 33, 127, 128, 129} and row labels on both sides of min_new."""
    total = {}
    kinds = set()
    for name in sorted(HAND):
        A, C, la, lc, pmode, kw = hand_case(name)
        n_a, n_c = A.shape[0], C.shape[0]
        Rw = torch.zeros(-(-n_a // 128) * 128, 256, dtype=torch.float64)
        Rw[:n_a] = A.float().bfloat16().double()
        rl = torch.full((Rw.shape[0],), -2, dtype=torch.long)
        rl[:n_a] = la
        Cb = C.float().bfloat16().double()
        ref = R.con_rows(Rw, rl, Cb, lc, range(Rw.shape[0] // 32), inv_tau=1 / TAU, want_grad=False)
        neg = torch.zeros(Rw.shape[0], dtype=torch.float64)
        neg[ref["row"]] = ref["neg"]
        for plan in (1, BIG_PLAN):
            p = R.make_plan(max(plan, -(-n_a // 128)), -(-n_c // 128), plan)
            cnt, _ = R.dispatch(rl, n_a, lc, pmode=pmode, min_new=kw.get("min_new"), neg=neg,
                                splits=p["splits"], splits2=p["splits2"])
            for k, v in cnt.items():
                total[k] = total.get(k, 0) + v
        kinds.add(("pmode", pmode))
        if pmode == 1:
            kp = -(-kw["pa"].shape[1] // 16) * 16
            kinds.add(("kpad", kp if kp <= 112 else "stream"))
            if bool((la >= kw["min_new"]).any()) and bool((la < kw["min_new"]).any()):
                kinds.add("both_sides_of_min_new")
        kinds.add(("n_c_mod_128", n_c % 128))
        kinds.add(("n_a", n_a))
    for k in range(1, 32):   # the reproducers
        A, C, la, lc = reproducer(k)
        cnt, _ = R.dispatch(la, 128, lc, pmode=0)
        total["false_uniform"] = total.get("false_uniform", 0) + cnt["false_uniform"]
    print("\nbranch counts:", {b: total.get(b, 0) for b in BRANCHES})
    missing = [b for b in BRANCHES if total.get(b, 0) == 0]
    assert not missing, missing
    want = {("pmode", 0), ("pmode", 1), ("pmode", 2), ("kpad", 16), ("kpad", 112), ("kpad", "stream"),
            "both_sides_of_min_new", ("n_c_mod_128", 0), ("n_c_mod_128", 1), ("n_c_mod_128", 127)}
    want |= {("n_a", n) for n in (1, 31, 32, 33, 127, 128, 129)}
    assert want <= kinds, want - kinds
