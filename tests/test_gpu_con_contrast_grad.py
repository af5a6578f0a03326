"""GPU tests of the contrast-side gradient of PixelConLossV2 (``contrast_grad=True``; ucd_con_contrast_grad, the
transposed third sweep of ucd_b200/csrc/contrast.cu), through the C ABI and through the module.

Per contrast column, against the operand-exact fp64 oracle of oracle/con_cols.py on the bf16 operands the kernel
multiplies, with the kernel's bf16 rounding of the pair gradient H emulated:

    || g_j - g_ref_j || <= REL || g_ref_j || + FLOOR scale_j + flip_j,   scale_j = (1/tau) sum_i |H_ji| |a_i| / M

scale_j is the size of the terms whose sum is the gradient (positive and negative pairs cancel), flip_j what operands
within 1e-5 of a bf16 rounding boundary can do when rounded the other way.  In aggregate, against fp32 torch autograd of
the reference formula: loss within 1e-3, gradient cosine >= 0.999 for both operands.

Observed on an NVIDIA B200 (1000 W power limit), as a fraction of the per-column bar: at most 0.30 (series_none); hand
cases 0.08 / 0.03, tau = 0.5 cases 0.09-0.18, median column error 3e-7 to 6e-7 of |g_j|."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import con_cols as CC
from oracle import con_rows as R
from oracle import ucd_oracle as O

pytestmark = pytest.mark.gpu

REL = 1e-3      # aggregate loss tolerance (as test_gpu_parity.py)
COS = 0.999     # aggregate gradient cosine
STATS = {}


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ucd_b200
    from ucd_b200 import _lib
    assert _lib.lib().ucd_device_ok() == 1, "ucd_b200 needs a compute-capability 10.x device"
    return ucd_b200


def _p(t):
    from ucd_b200._lib import ptr
    return ptr(t)


def _check(rc, what):
    from ucd_b200._lib import check
    check(rc, what)


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


def _unit(x):
    return F.normalize(x, dim=1)


# ------------------------------------------------------------------------------------------------------------------
# C ABI
# ------------------------------------------------------------------------------------------------------------------
def cabi_run(A, C, la, lc, P, tau, need_grad=1, plan=0):
    """ucd_con_fwd + ucd_con_contrast_grad + ucd_con_bwd (g = 1) on freshly packed tiles; returns (out, dC, tiles)."""
    from ucd_b200 import _lib
    L = _lib.lib()
    dev = "cuda"
    n_a, n_c = A.shape[0], C.shape[0]
    rt, ct = -(-n_a // 128), -(-n_c // 128)
    rfeat = torch.empty(rt, 32, 128, 8, device=dev, dtype=torch.bfloat16)
    cfeat = torch.empty(ct, 32, 128, 8, device=dev, dtype=torch.bfloat16)
    rlab = torch.empty(rt, 128, device=dev, dtype=torch.int32)
    clab = torch.empty(ct, 128, device=dev, dtype=torch.int32)
    a32, c32 = A.float().cuda().contiguous(), C.float().cuda().contiguous()
    la32, lc32 = la.int().cuda().contiguous(), lc.int().cuda().contiguous()
    _check(L.ucd_con_pack_rows(_p(a32), _p(la32), n_a, _p(rfeat), _p(rlab), rt, None), "pack_rows")
    _check(L.ucd_con_pack_rows(_p(c32), _p(lc32), n_c, _p(cfeat), _p(clab), ct, None), "pack_rows")
    rr = torch.empty(rt, 2, device=dev, dtype=torch.int32)
    cr = torch.empty(ct, 2, device=dev, dtype=torch.int32)
    _check(L.ucd_con_tile_ranges(_p(rlab), rt, None, _p(rr), None), "tile_ranges")
    _check(L.ucd_con_tile_ranges(_p(clab), ct, None, _p(cr), None), "tile_ranges")
    counts = torch.tensor([[n_c, 0]], device=dev, dtype=torch.int32)
    n_rows = torch.tensor([n_a], device=dev, dtype=torch.int32)
    Pd = None if P is None else P.float().cuda().contiguous()
    p_mode, ldp = (0, 0) if Pd is None else (2, n_c)
    inv_tau = float(np.float32(1 / tau))
    ws_bytes = L.ucd_con_contrast_grad_workspace_bytes(rt, ct, plan)
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    out = torch.full((3,), float("nan"), device=dev)
    gu = torch.empty(rt * 128, 256, device=dev) if need_grad else None
    _check(L.ucd_con_fwd(_p(cfeat), None, _p(clab), _p(counts), 1, ct, 0, -1, 0, _p(rfeat), None, _p(rlab),
                         _p(n_rows), _p(cr), _p(rr), 0, None, p_mode, 16, _p(Pd), ldp, inv_tau, need_grad, _p(out),
                         _p(gu), _p(ws), ws_bytes, rt, plan, None), "con_fwd")
    cu = torch.full((ct * 128, 256), float("nan"), device=dev)
    _check(L.ucd_con_contrast_grad(_p(cfeat), _p(clab), _p(counts), 1, ct, 0, _p(rfeat), _p(rlab), _p(n_rows), _p(cr),
                                   _p(rr), 0, p_mode, _p(Pd), ldp, inv_tau, _p(cu), _p(ws), ws_bytes, rt, plan, None),
           "con_contrast_grad")
    one = torch.ones(1, device=dev)
    dC = torch.empty(n_c, 256, device=dev)
    _check(L.ucd_con_bwd(_p(cu), _p(out), _p(one), 1.0, _p(counts), None, _p(dC), n_c, None), "con_bwd")
    torch.cuda.synchronize()
    assert bool(torch.isfinite(cu).all()) and float(cu[n_c:].abs().max() if ct * 128 > n_c else 0) == 0
    return out.cpu(), dC.cpu().double(), (rfeat, rlab, cfeat, clab)


def cabi_anchor(A, C, la, lc, P, tau):
    """The forward alone with the anchor gradient: (out, d(sum of row losses)/dA on the tiles' rows, None)."""
    from ucd_b200 import _lib
    L = _lib.lib()
    n_a, n_c = A.shape[0], C.shape[0]
    rt, ct = -(-n_a // 128), -(-n_c // 128)
    dev = "cuda"
    rfeat = torch.empty(rt, 32, 128, 8, device=dev, dtype=torch.bfloat16)
    cfeat = torch.empty(ct, 32, 128, 8, device=dev, dtype=torch.bfloat16)
    rlab = torch.empty(rt, 128, device=dev, dtype=torch.int32)
    clab = torch.empty(ct, 128, device=dev, dtype=torch.int32)
    a32, c32 = A.float().cuda().contiguous(), C.float().cuda().contiguous()
    la32, lc32 = la.int().cuda().contiguous(), lc.int().cuda().contiguous()
    _check(L.ucd_con_pack_rows(_p(a32), _p(la32), n_a, _p(rfeat), _p(rlab), rt, None), "pack_rows")
    _check(L.ucd_con_pack_rows(_p(c32), _p(lc32), n_c, _p(cfeat), _p(clab), ct, None), "pack_rows")
    rr = torch.empty(rt, 2, device=dev, dtype=torch.int32)
    cr = torch.empty(ct, 2, device=dev, dtype=torch.int32)
    _check(L.ucd_con_tile_ranges(_p(rlab), rt, None, _p(rr), None), "tile_ranges")
    _check(L.ucd_con_tile_ranges(_p(clab), ct, None, _p(cr), None), "tile_ranges")
    counts = torch.tensor([[n_c, 0]], device=dev, dtype=torch.int32)
    n_rows = torch.tensor([n_a], device=dev, dtype=torch.int32)
    Pd = None if P is None else P.float().cuda().contiguous()
    p_mode, ldp = (0, 0) if Pd is None else (2, n_c)
    ws_bytes = L.ucd_con_workspace_bytes(rt, ct, 0, 0)
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    out = torch.empty(3, device=dev)
    gu = torch.empty(rt * 128, 256, device=dev)
    _check(L.ucd_con_fwd(_p(cfeat), None, _p(clab), _p(counts), 1, ct, 0, -1, 0, _p(rfeat), None, _p(rlab),
                         _p(n_rows), _p(cr), _p(rr), 0, None, p_mode, 16, _p(Pd), ldp, float(np.float32(1 / tau)), 1,
                         _p(out), _p(gu), _p(ws), ws_bytes, rt, 0, None), "con_fwd")
    torch.cuda.synchronize()
    return out.cpu(), gu.cpu().double(), None


def check_anchor_rows(name, A, C, la, lc, P, tau, Rd, rl, Cd, lcd):
    """The anchor side of the same forward, row by row against oracle/con_rows.py with the bars of
    tests/test_gpu_con_rows.py (GRAD_TOL 5e-4 of |g_i|, CANCEL_TOL 3e-5 of scale_i, plus flip_i), and the sum of the
    row losses to 5e-6."""
    n_a = A.shape[0]
    out, ga, _ = cabi_anchor(A, C, la, lc, P, tau)
    ar = R.con_rows(Rd, rl, Cd, lcd, range(-(-n_a // 32)), inv_tau=np.float32(1 / tau),
                    pmode=0 if P is None else 2, P=None if P is None else P.float().double())
    sel = ar["row"] < n_a
    rows = ar["row"][sel]
    keep = sel & (ar["num"] != 0)
    total, M = float(ar["loss"][keep].sum()), int(keep.sum())
    assert int(out[1]) == M, (name, float(out[1]), M)
    assert abs(float(out[0]) - total) <= 5e-6 * abs(total), (name, float(out[0]), total)
    gref = ar["grad"][sel]
    err = (ga[rows] - gref).norm(dim=1)
    bad = err > 5e-4 * gref.norm(dim=1) + 3e-5 * ar["scale"][sel] + ar["flip"][sel]
    assert not bool(bad.any()), (name, "anchor rows", rows[bad][:8].tolist())


def check_cols(name, A, C, la, lc, P, tau):
    out, dC, (rfeat, rlab, cfeat, clab) = cabi_run(A, C, la, lc, P, tau)
    n_a, n_c = A.shape[0], C.shape[0]
    Rd = R.decode_tiles(rfeat)
    rl = R.row_labels(rlab.reshape(-1), n_a)
    Cd = R.decode_tiles(cfeat)[:n_c]
    lcd = clab.reshape(-1)[:n_c].cpu().long()
    ref = CC.contrast_cols(Rd, rl, Cd, lcd, float(np.float32(1 / tau)), None if P is None else P.float().double())
    assert int(out[1]) == ref["M"], (name, float(out[1]), ref["M"])
    ex = CC.excess(dC, ref)
    rel = float(((dC - ref["grad"]).norm(dim=1) / ref["grad"].norm(dim=1).clamp_min(1e-300)).median())
    STATS[name] = ex
    print("\n[%s] columns %d  max error %.3f of the bar, median %.2e of |g_j|" % (name, n_c, ex, rel))
    assert ex <= 1.0, (name, ex)
    if n_a > n_c:   # anchors past the last column: sweep 1 must not count a self column for them (num_i)
        check_anchor_rows(name, A, C, la, lc, P, tau, Rd, rl, Cd, lcd)
    # reruns are bit-identical; the forward without the anchor gradient gives the same contrast gradient
    out2, dC2, _ = cabi_run(A, C, la, lc, P, tau)
    out3, dC3, _ = cabi_run(A, C, la, lc, P, tau, need_grad=0)
    assert torch.equal(dC, dC2) and torch.equal(out, out2)
    assert torch.equal(dC, dC3) and torch.equal(out[:2], out3[:2])
    return ref


def hand_case(with_p):
    """N_a = 200, N_c = 300: every branch of the pair function - negatives, positives, self pairs with equal labels
    (excluded) and with different labels (negatives), padding anchors (tile 1 holds 72) and padding columns (tile 2
    holds 44), P = 0 on some positive pairs, an anchor row without positives."""
    g = torch.Generator().manual_seed(7 + with_p)
    n_a, n_c = 200, 300
    A = _unit(torch.randn(n_a, 256, generator=g, dtype=torch.float64))
    C = _unit(torch.randn(n_c, 256, generator=g, dtype=torch.float64))
    C[:n_a] = A
    la = torch.randint(1, 5, (n_a,), generator=g)
    lc = torch.randint(1, 5, (n_c,), generator=g)
    lc[:n_a] = la
    lc[:n_a:7] = la[:n_a:7] % 4 + 1          # self pairs with different labels
    la[5] = 9                                 # no positive at all (num = -1 + 0: the self pair differs) ...
    la[6] = 9
    lc[6] = 9                                 # ... and num = 0 (its only equal label is itself)
    P = None
    if with_p:
        P = torch.rand(n_a, n_c, generator=g, dtype=torch.float64)
        P[torch.rand(n_a, n_c, generator=g) < 0.25] = 0.0
    return A, C, la, lc, P


@pytest.mark.parametrize("with_p", [False, True])
def test_hand_built_columns(U, with_p):
    A, C, la, lc, P = hand_case(with_p)
    check_cols("hand_p%d" % with_p, A, C, la, lc, P, 0.07)


RANDOM = {  # name: (N_a, N_c, labels, dense P, tau)
    "series_none": (2000, 6001, 4, False, 0.07),     # neg_i >= 4096: sweep 2's series regime; 4 anchor-tile splits
    "series_dense": (1500, 5003, 4, True, 0.07),
    "tau05_none": (777, 1301, 6, False, 0.5),
    "tau05_dense": (1301, 777, 3, True, 0.5),        # N_a > N_c: anchors 777..895 have no self column
    "tau05_none_wide": (1301, 777, 3, False, 0.5),
    "tau05_dense_tall": (777, 1301, 3, True, 0.5),
}


def random_case(name):
    n_a, n_c, n_lab, with_p, tau = RANDOM[name]
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    A = _unit(torch.randn(n_a, 256, generator=g, dtype=torch.float64))
    C = _unit(torch.randn(n_c, 256, generator=g, dtype=torch.float64))
    k = min(n_a, n_c)
    C[:k] = A[:k]
    la = torch.randint(1, n_lab + 1, (n_a,), generator=g)
    lc = torch.randint(1, n_lab + 1, (n_c,), generator=g)
    lc[:k] = la[:k]
    P = torch.rand(n_a, n_c, generator=g, dtype=torch.float64) if with_p else None
    return A, C, la, lc, P, tau


@pytest.mark.parametrize("name", list(RANDOM))
def test_random_columns(U, name):
    A, C, la, lc, P, tau = random_case(name)
    ref = check_cols(name, A, C, la, lc, P, tau)
    if name.startswith("series"):
        assert float((ref["neg"] >= R.SERIES_NEG).double().mean()) > 0.9   # the rows take the series form


# ------------------------------------------------------------------------------------------------------------------
# the module
# ------------------------------------------------------------------------------------------------------------------
def cos(a, b):
    a, b = a.double().reshape(-1).cpu(), b.double().reshape(-1).cpu()
    return float(a @ b / (a.norm() * b.norm()).clamp_min(1e-300))


def module_run(U, A, C, la, lc, P, tau, anchor_grad=True, contrast_grad=True, flag=True):
    a = A.float().cuda().requires_grad_(anchor_grad)
    c = C.float().cuda().requires_grad_(contrast_grad)
    out = U.PixelConLossV2(temperature=tau, contrast_grad=flag)(a, c, la.cuda(), lc.cuda(),
                                                                 None if P is None else P.float().cuda())
    out.backward()
    return out.detach(), a.grad, c.grad


@pytest.mark.parametrize("name", ["tau05_none", "series_dense"])
def test_module_columns_and_aggregate(U, name):
    """The module's contrast.grad per column on its bf16 operands, and loss / both gradients against fp32 torch
    autograd of the reference formula (ucd_oracle.pixel_con_loss) on the GPU."""
    A, C, la, lc, P, tau = random_case(name)
    out, ga, gc = module_run(U, A, C, la, lc, P, tau)
    n_a = A.shape[0]
    rows_pad = -(-n_a // 128) * 128
    Rd = torch.zeros(rows_pad, 256, dtype=torch.float64)
    Rd[:n_a] = A.float().bfloat16().double()
    rl = torch.full((rows_pad,), -2, dtype=torch.long)
    rl[:n_a] = la
    ref = CC.contrast_cols(Rd, rl, C.float().bfloat16().double(), lc, float(np.float32(1 / tau)),
                           None if P is None else P.float().double())
    ex = CC.excess(gc.cpu().double(), ref)
    STATS["module_" + name] = ex
    assert ex <= 1.0, ex
    a = A.float().cuda().requires_grad_(True)
    c = C.float().cuda().requires_grad_(True)
    assert n_a <= C.shape[0]   # the default self_col: anchor i <-> column i
    r = O.pixel_con_loss(a, c, la.cuda(), lc.cuda(), None if P is None else P.float().cuda(), tau)
    r.backward()
    assert float(out) == pytest.approx(float(r), rel=REL)
    assert cos(ga, a.grad) >= COS and cos(gc, c.grad) >= COS


def test_aliased_contrast(U):
    """contrast = cat(anchor, other) with the anchor requiring grad: anchor.grad sums both paths, as autograd of the
    reference does."""
    g = torch.Generator().manual_seed(11)
    n_a, n_o = 900, 1500
    A = _unit(torch.randn(n_a, 256, generator=g))
    Oth = _unit(torch.randn(n_o, 256, generator=g))
    la = torch.randint(1, 5, (n_a,), generator=g)
    lc = torch.cat([la, torch.randint(1, 5, (n_o,), generator=g)])
    P = torch.rand(n_a, n_a + n_o, generator=g)
    got = []
    for fused in (True, False):
        a = A.cuda().requires_grad_(True)
        o = Oth.cuda().requires_grad_(True)
        if fused:
            out = U.PixelConLossV2(temperature=0.07, contrast_grad=True)(a, torch.cat([a, o]), la.cuda(), lc.cuda(),
                                                                         P.cuda())
        else:
            out = O.pixel_con_loss(a, torch.cat([a, o]), la.cuda(), lc.cuda(), P.cuda(), 0.07)
        out.backward()
        got.append((float(out), a.grad, o.grad))
    assert got[0][0] == pytest.approx(got[1][0], rel=REL)
    assert cos(got[0][1], got[1][1]) >= COS and cos(got[0][2], got[1][2]) >= COS


def test_flag_changes_nothing_else(U):
    """With the flag: the loss and the anchor gradient are bit-identical to the call with a detached contrast, reruns
    are bit-identical, and without a contrast gradient to form (no_grad, detached contrast) the C-ABI calls are those
    of the default module."""
    from ucd_b200 import _lib
    A, C, la, lc, P, tau = random_case("tau05_dense")
    out1, ga1, gc1 = module_run(U, A, C, la, lc, P, tau)
    out2, ga2, gc2 = module_run(U, A, C, la, lc, P, tau)
    out0, ga0, gc0 = module_run(U, A, C, la, lc, P, tau, contrast_grad=False)
    assert gc0 is None
    assert torch.equal(out1, out0) and torch.equal(ga1, ga0)
    assert torch.equal(out1, out2) and torch.equal(ga1, ga2) and torch.equal(gc1, gc2)
    # the contrast alone: the anchors' V / U accumulation is skipped, the contrast gradient is the same
    out3, ga3, gc3 = module_run(U, A, C, la, lc, P, tau, anchor_grad=False)
    assert ga3 is None and torch.equal(out3, out1) and torch.equal(gc3, gc1)

    prod = _lib.lib()
    calls = {}
    try:
        for flag in (False, True):
            for mode in ("no_grad", "detached"):
                cnt = _Counter(prod)
                _lib._lib = cnt
                if mode == "no_grad":
                    with torch.no_grad():
                        module_run_nograd(U, A, C, la, lc, P, tau, flag)
                else:
                    module_run(U, A, C, la, lc, P, tau, contrast_grad=False, flag=flag)
                calls[(flag, mode)] = dict(cnt.counts)
    finally:
        _lib._lib = prod
    for mode in ("no_grad", "detached"):
        assert calls[(True, mode)] == calls[(False, mode)], calls
        assert "ucd_con_contrast_grad" not in calls[(True, mode)]


def module_run_nograd(U, A, C, la, lc, P, tau, flag):
    a = A.float().cuda().requires_grad_(True)
    c = C.float().cuda().requires_grad_(True)
    return U.PixelConLossV2(temperature=tau, contrast_grad=flag)(a, c, la.cuda(), lc.cuda(),
                                                                  None if P is None else P.float().cuda())


def test_joint_prob_with_contrast_grad_raises(U):
    case = O.synthetic_case(2, 8, 8, 128, 128, 6, 4)
    f_n = case["f_n"].cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
    con = U.PixelConLossV2(temperature=0.07, contrast_grad=True)
    with pytest.raises(ValueError, match="compat path"):
        con(tup[0], tup[1].clone().requires_grad_(True), tup[2], tup[3], tup[4])
    ref = U.PixelConLossV2(temperature=0.07)(*tup)
    assert torch.equal(con(*tup), ref)       # a contrast without grad: the fast path as before


def test_zz_report():
    """Largest observed error per case as a fraction of the bar (printed with -s)."""
    print("\nmax error / bar:", {k: round(v, 4) for k, v in STATS.items()})
