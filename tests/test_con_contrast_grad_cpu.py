"""CPU checks of the contrast-side gradient of PixelConLossV2 (oracle/con_cols.py, ucd_con_contrast_grad): the
closed form equals fp64 autograd of the reference restatement, plausible kernel slips miss the GPU bar by at least 10x
wherever they change the gradient, and the new C-ABI entry points are exported, bound and refuse what they do not
support."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from oracle import con_cols as CC
from oracle import ucd_oracle as O


def _unit(x):
    return F.normalize(x, dim=1)


def make_case(name):
    """fp64 (A, Cst, la, lc, P, aliased) of a named case; aliased: Cst = cat(A, other) with the anchors' own rows."""
    g = torch.Generator().manual_seed(sum(map(ord, name)))
    n_a, n_c, n_lab, with_p, alias = dict(
        none=(40, 70, 4, False, True), dense=(40, 70, 4, True, True), diag_differs=(30, 50, 3, True, False),
        no_positive_rows=(40, 60, 12, False, True), no_negatives=(20, 30, 1, True, True),
        na_gt_nc=(70, 40, 4, True, False), na_lt_nc=(25, 90, 3, False, False))[name]
    A = _unit(torch.randn(n_a, 256, generator=g, dtype=torch.float64))
    Cst = _unit(torch.randn(n_c, 256, generator=g, dtype=torch.float64))
    la = torch.randint(1, n_lab + 1, (n_a,), generator=g)
    lc = torch.randint(1, n_lab + 1, (n_c,), generator=g)
    k = min(n_a, n_c)
    if alias:
        Cst[:k] = A[:k]
        lc[:k] = la[:k]
    if name == "diag_differs":
        lc[:k] = la[:k]
        lc[:k:3] = la[:k:3] % n_lab + 1          # every third self pair carries two different labels
    P = None
    if with_p:
        P = torch.rand(n_a, n_c, generator=g, dtype=torch.float64)
        P[torch.rand(n_a, n_c, generator=g) < 0.2] = 0.0     # exact zeros
    return A, Cst, la, lc, P, alias


CASES = ["none", "dense", "diag_differs", "no_positive_rows", "no_negatives", "na_gt_nc", "na_lt_nc"]


def _self_col(n_a, n_c):
    ar = torch.arange(n_a)
    return torch.where(ar < n_c, ar, -torch.ones(n_a, dtype=torch.long))


@pytest.mark.parametrize("name", CASES)
def test_closed_form_equals_autograd(name):
    """dC (and dA, the loss) of the closed form == fp64 autograd of ucd_oracle.pixel_con_loss w.r.t. Cst (and A)."""
    A, Cst, la, lc, P, _ = make_case(name)
    n_a, n_c = A.shape[0], Cst.shape[0]
    a, c = A.clone().requires_grad_(True), Cst.clone().requires_grad_(True)
    ref = O.pixel_con_loss(a, c, la, lc, P, 0.07, self_col=_self_col(n_a, n_c))
    ref.backward()
    loss, dA, dC = CC.pixel_con_loss_grads(A, Cst, la, lc, P, 0.07, self_col=_self_col(n_a, n_c))
    assert abs(float(loss) - float(ref.detach())) <= 1e-12 * abs(float(ref.detach()))
    assert float((dA - a.grad).abs().max()) <= 1e-12 * float(a.grad.abs().max())
    assert float((dC - c.grad).abs().max()) <= 1e-12 * float(c.grad.abs().max())
    if name == "no_negatives":   # neg_i = 0: every pair gradient is 0 (not NaN)
        assert bool((la.view(-1, 1) == lc.view(1, -1)).all()) and float(dC.abs().max()) == 0
    else:
        assert float(dC.abs().max()) > 0
    if name == "no_positive_rows":
        t = CC._terms(A, Cst, la, lc, None, 0.07, _self_col(n_a, n_c), False)
        assert 0 < int(t["keep"].sum()) < n_a


def test_aliased_contrast_sums_both_paths():
    """Cst = cat(A, other) with A requiring grad: autograd sums the anchor and the contrast path into A.grad; so does
    dA + dC[:N_a] of the closed form."""
    A, Cst, la, lc, _, _ = make_case("none")
    n_a, n_c = A.shape[0], Cst.shape[0]
    other = Cst[n_a:]
    a = A.clone().requires_grad_(True)
    o = other.clone().requires_grad_(True)
    ref = O.pixel_con_loss(a, torch.cat([a, o]), la, lc, None, 0.07)
    ref.backward()
    _, dA, dC = CC.pixel_con_loss_grads(A, torch.cat([A, other]), la, lc, None, 0.07)
    want = dA + dC[:n_a]
    assert float((want - a.grad).abs().max()) <= 1e-12 * float(a.grad.abs().max())
    assert float((dC[n_a:] - o.grad).abs().max()) <= 1e-12 * float(o.grad.abs().max())


def _kernel_operands(name):
    """The case as the kernel sees it: bf16-rounded operands, anchors padded to whole tiles with label -2."""
    A, Cst, la, lc, P, _ = make_case(name)
    n_a = A.shape[0]
    rows_pad = -(-n_a // 128) * 128
    R = torch.zeros(rows_pad, 256, dtype=torch.float64)
    R[:n_a] = A.float().bfloat16().double()
    rl = torch.full((rows_pad,), -2, dtype=torch.long)
    rl[:n_a] = la
    return R, rl, Cst.float().bfloat16().double(), lc, None if P is None else P.float().double()


def test_kernel_convention_matches_reference_where_the_self_labels_agree():
    """contrast_cols (the sweeps' self convention) == the closed form of the reference wherever every self pair has
    equal labels (the UCD prep, the aliased case); only a self pair with different labels tells them apart."""
    for name in CASES:
        R, rl, C, lc, P = _kernel_operands(name)
        n_a = int((rl != -2).sum())
        got = CC.contrast_cols(R, rl, C, lc, 1 / 0.07, P, emulate=False)
        _, _, dC = CC.pixel_con_loss_grads(R[:n_a], C, rl[:n_a], lc, P, 0.07, self_col=_self_col(n_a, C.shape[0]))
        err = float((got["grad"] - dC).abs().max()) / max(float(dC.abs().max()), 1e-300)
        k = min(n_a, C.shape[0])
        if bool((rl[:k] == lc[:k]).all()):
            assert err <= 1e-12, (name, err)
        else:
            assert err > 1e-6, (name, err)


# when a slip changes the gradient at all
APPLIES = {
    "self_kept": lambda rl, lc, P, k: bool((rl[:k] == lc[:k]).any()),
    "p_untransposed": lambda rl, lc, P, k: P is not None,
    "t_missing": lambda rl, lc, P, k: True,
    "m_all_rows": lambda rl, lc, P, k: None,   # decided from M below
    "max_not_detached": lambda rl, lc, P, k: True,
}


def test_every_slip_is_listed():
    assert set(APPLIES) == set(CC.SLIPS)


@pytest.mark.parametrize("slip", CC.SLIPS)
def test_slip_misses_the_gpu_bar_by_10x(slip):
    """Each slip, applied to the operand-exact oracle, differs from it by >= 10x the GPU bar (REL, FLOOR of
    oracle/con_cols.py) in every case it applies to, and by < 1e-3 of the bar where it does not apply."""
    hit = 0
    for name in CASES:
        R, rl, C, lc, P = _kernel_operands(name)
        n_a = int((rl != -2).sum())
        ref = CC.contrast_cols(R, rl, C, lc, 1 / 0.07, P)
        got = CC.contrast_cols(R, rl, C, lc, 1 / 0.07, P, slip=slip)["grad"]
        applies = APPLIES[slip](rl, lc, P, min(n_a, C.shape[0]))
        if slip == "m_all_rows":
            applies = ref["M"] != n_a
        if name == "no_negatives":
            applies = False       # neg_i = 0: the gradient is 0, whatever the slip
        r = CC.excess(got, ref)
        if applies:
            assert r >= 10, (slip, name, r)
            hit += 1
        else:
            assert r < 1e-3, (slip, name, r)
    assert hit > 0


# ------------------------------------------------------------------------------------------------------------------
# C ABI
# ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def L():
    import ucd_b200  # noqa: F401  (the package must import without a GPU)
    from ucd_b200 import _lib
    return _lib


def test_new_symbols_exported_and_bound(L):
    h = ctypes.CDLL(L.LIB_PATH)
    for n in ("ucd_con_contrast_grad", "ucd_con_contrast_grad_workspace_bytes"):
        assert hasattr(h, n) and n in L.EXPORTED, n
    lib = L.lib()
    fwd = lib.ucd_con_workspace_bytes(24, 49, 0, 0)
    assert lib.ucd_con_contrast_grad_workspace_bytes(24, 49, 0) > fwd + 49 * 128 * 256 * 4
    assert lib.ucd_con_contrast_grad_workspace_bytes(0, 49, 0) == 0
    import ucd_b200
    import inspect
    assert inspect.signature(ucd_b200.PixelConLossV2).parameters["contrast_grad"].default is False


def _call(L, **over):
    """ucd_con_contrast_grad with plausible (never dereferenced) host addresses; argument checks run first."""
    buf = (ctypes.c_char * 4096)()
    a = ctypes.addressof(buf)
    a16 = (a + 15) & ~15
    lib = L.lib()
    ws = lib.ucd_con_contrast_grad_workspace_bytes(1, 1, 0)
    args = dict(feat=a16, lab=a16, counts=a16, n_chunks=1, chunk_tiles=1, stride=0, rfeat=a16, rlab=a16, n_rows=a16,
                trange=a16, rrange=a16, self_tile0=0, p_mode=0, dense_p=None, ldp=0, inv_tau=1 / 0.07, grad=a16,
                ws=a16, ws_bytes=ws, max_row_tiles=1, plan=0)
    args.update(over)
    rc = lib.ucd_con_contrast_grad(*args.values(), None)
    return rc, lib.ucd_last_error().decode()


def test_argument_checks_refuse_with_a_message(L):
    EINVAL = L.UCD_EINVAL if hasattr(L, "UCD_EINVAL") else None
    for over, pat in ((dict(feat=None), "null pointer"), (dict(grad=None), "null pointer"),
                      (dict(ws=None), "null pointer"), (dict(p_mode=1), "p_mode"),
                      (dict(p_mode=2), "dense P"), (dict(n_chunks=2), "single-chunk"),
                      (dict(stride=4096), "single-chunk"), (dict(self_tile0=3), "self_tile0"),
                      (dict(ws_bytes=16), "workspace too small")):
        rc, msg = _call(L, **over)
        assert rc != 0 and pat in msg, (over, rc, msg)
        if EINVAL is not None:
            assert rc == EINVAL
