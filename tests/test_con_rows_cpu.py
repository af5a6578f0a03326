"""CPU checks of the per-row contrastive oracle and the dispatch model that tests/test_gpu_con_rows.py relies on:
the oracle equals the aggregate oracles of ucd_oracle.py row by row, the plan model equals the library's workspace
sizing, and the dispatch model still finds the false-uniform warps in the seeded inputs the GPU tests pin."""
import pytest
import torch
import torch.nn.functional as F

from oracle import con_rows as R
from oracle import ucd_oracle as O

# (case, (row block, warp, column tile)) the uniform test of sweep 2 accepted before it checked the row labels:
# bench.make_inputs == O.synthetic_case(..., correlated=True)
FALSE_UNIFORM = {
    "city_rank0": ((3, 32, 64, 512, 1024, 20, 14, 0), [(26, 2, 71)]),
    "voc_rank3": ((24, 32, 32, 512, 512, 17, 16, 3), [(28, 0, 210)]),
    "small_rank40": ((2, 32, 32, 512, 512, 17, 16, 40), [(4, 0, 19)]),
    "voc_rank0": ((24, 32, 32, 512, 512, 17, 16, 0), []),
    "ade_rank0": ((3, 32, 32, 512, 512, 151, 101, 0), []),
}


def padded(A, la):
    """rows padded to whole warps, row labels -2 past the valid rows (what the sweep threads carry)."""
    n = A.shape[0]
    pad = -(-n // 32) * 32
    Rw = torch.zeros(pad, A.shape[1], dtype=torch.float64)
    Rw[:n] = A
    rl = torch.full((pad,), -2, dtype=torch.long)
    rl[:n] = la
    return Rw, rl


def small_case(seed, n_a, n_c, c_old):
    g = torch.Generator().manual_seed(seed)
    A = F.normalize(torch.randn(n_a, 256, generator=g, dtype=torch.float64), dim=1)
    C = F.normalize(torch.randn(n_c, 256, generator=g, dtype=torch.float64), dim=1)
    C[:n_a] = A
    la = torch.randint(1, 7, (n_a,), generator=g)
    lc = torch.randint(1, 7, (n_c,), generator=g)
    lc[:n_a] = la
    pa = torch.softmax(3 * torch.randn(n_a, c_old, generator=g, dtype=torch.float64), 1)
    pc = torch.softmax(3 * torch.randn(n_c, c_old, generator=g, dtype=torch.float64), 1)
    pc[:n_a] = pa
    return A, C, la, lc, pa, pc


@pytest.mark.parametrize("pmode", [0, 1, 2])
@pytest.mark.parametrize("n_a,n_c", [(70, 300), (33, 129)])
def test_row_oracle_equals_streaming_oracle(pmode, n_a, n_c):
    """Without the rounding emulation the per-row oracle is the closed form of ucd_oracle: the same loss and, row by
    row, the same gradient as pixel_con_loss_streaming (P None / joint probability with the GT-new override) and
    pixel_con_loss_closed_form (dense P)."""
    A, C, la, lc, pa, pc = small_case(n_a * 7 + n_c + pmode, n_a, n_c, 5)
    min_new = 5
    Rw, rl = padded(A, la)
    tau = 0.07
    kw = dict(inv_tau=1 / tau, emulate=False)
    if pmode == 0:
        loss, G, M = O.pixel_con_loss_streaming(A, C, la, lc, temperature=tau, block=64)
    elif pmode == 1:
        loss, G, M = O.pixel_con_loss_streaming(A, C, la, lc, pa, pc, min_new, temperature=tau, block=64)
        Pw, _ = padded(pa, la)
        kw.update(pmode=1, pa=Pw, pc=pc, min_new=min_new)
    else:
        P = torch.rand(n_a, n_c, generator=torch.Generator().manual_seed(3), dtype=torch.float64)
        loss, G = O.pixel_con_loss_closed_form(A, C, la, lc, P, temperature=tau)
        M = int((((la[:, None] == lc[None, :]).double().sum(1) - 1) != 0).sum())
        kw.update(pmode=2, P=P)
    r = R.con_rows(Rw, rl, C, lc, range(Rw.shape[0] // 32), **kw)
    keep = r["row"] < n_a
    total, m = R.con_row_losses(Rw, rl, n_a, C, lc, **{k: v for k, v in kw.items() if k != "emulate"})
    assert m == M
    assert total / M == pytest.approx(float(loss), rel=1e-12)
    # per row (T V - U cancels: element-wise relative errors of fp64 sums in another order are meaningless)
    err = (r["grad"][keep] / M - G).norm(dim=1)
    assert float((err / G.norm(dim=1).clamp_min(1e-300)).max()) < 1e-9
    # rows past n_a are all-negative rows: nothing in their weights, no positive
    assert float(r["num"][~keep].abs().max() if (~keep).any() else 0.0) <= 1.0


def test_row_oracle_rounding_emulation_is_bf16_of_the_operands():
    """With the emulation on, only the V / U operands change: L, T, num are the same and the gradient moves by about
    the bf16 step of E and Ucoef (relative 2^-9), not more."""
    A, C, la, lc, pa, pc = small_case(11, 96, 400, 5)
    Rw, rl = padded(A, la)
    a = R.con_rows(Rw, rl, C, lc, range(3), inv_tau=1 / 0.07, emulate=False)
    b = R.con_rows(Rw, rl, C, lc, range(3), inv_tau=1 / 0.07, emulate=True)
    for k in ("L", "T", "num", "neg"):
        assert torch.equal(a[k], b[k]), k
    d = (a["grad"] - b["grad"]).norm(dim=1) / a["grad"].norm(dim=1)
    assert 0 < float(d.max()) < 2 ** -8


@pytest.mark.parametrize("mode,views,anchors", [(0, 1, "all"), (1, 2, "all"), (1, 2, "one"), (1, 1, "all")])
def test_selfcon_row_oracle_equals_reference_oracles(mode, views, anchors):
    """selfcon_rows on the view-major rows equals ucd_oracle.pixel_con_loss_v1 / sup_con_loss (times the number of
    rows in the mean), gradient included."""
    x, lab = O.selfcon_case("c")
    x = x[:, :views]
    bsz = x.shape[0]
    tau = 1.0 if mode == 0 else 0.1
    xr = x.clone().requires_grad_(True)
    if mode == 0:
        ref = O.pixel_con_loss_v1(xr, lab, tau)
    else:
        ref = O.sup_con_loss(xr, lab, tau, anchors, 0.07)
    ref.backward()
    rows = torch.cat(torch.unbind(x, dim=1), dim=0)
    labs = lab.repeat(views)
    n_anchor = bsz if anchors == "one" else rows.shape[0]
    total, M, g = R.selfcon_rows(rows, labs, mode, n_anchor, 1 / tau, tau / 0.07)
    assert total / M == pytest.approx(float(ref), rel=1e-12)
    g_ref = torch.cat(torch.unbind(xr.grad, dim=1), dim=0) * M
    torch.testing.assert_close(g, g_ref, rtol=1e-9, atol=1e-12)


def test_plan_model_equals_workspace_bytes():
    """choose_splits / make_plan of the model reproduce ucd_con_workspace_bytes (a host-only call) over a grid of
    (max_row_tiles, col_tiles, plan_row_tiles, local_col_tiles): the splits the GPU tests reason about are the
    library's.  The workspace size is a function of (splits + splits_local, splits2), so the grid covers the values
    where they change."""
    from ucd_b200 import _lib
    L = _lib.lib()
    n = 0
    for mrt in (1, 2, 3, 5, 37, 48, 75, 148, 183, 400):
        for ct in (1, 3, 4, 7, 8, 9, 16, 17, 33, 64, 81, 160, 321, 642, 4097, 9000):
            for prt in sorted({0, 1, 2, mrt // 2, mrt, mrt + 5}):
                for loc in (0, max(1, ct // 8)):
                    want = L.ucd_con_workspace_bytes(mrt, ct, prt, loc)
                    got = R.make_plan(mrt, ct, prt, loc)["total"]
                    assert got == want, (mrt, ct, prt, loc, got, want)
                    n += 1
    assert n > 1000
    # the plans the GPU tests use differ in their splits
    assert R.make_plan(48, 12, 1)["splits"] != R.make_plan(48, 12, 48)["splits"]


@pytest.mark.parametrize("name", sorted(FALSE_UNIFORM))
def test_dispatch_model_finds_false_uniform_warps(name):
    """The seeded inputs the GPU reproducers use still hold a warp whose rows carry two labels a | b split at lane K
    against a full column tile split a | b at column 4K: generator drift cannot silently drop a reproducer."""
    (B, h, w, H, W, C, c_old, rank), want = FALSE_UNIFORM[name]
    case = O.synthetic_case(B, h, w, H, W, C, c_old, rank=rank, correlated=True)
    la, lc, min_new = R.class_sorted_labels(case["labels"], case["l_po"], max(20, C - 1))
    rt = -(-la.numel() // 128)
    rl = torch.full((rt * 128,), -2, dtype=torch.long)
    rl[:la.numel()] = la
    cnt, found = R.dispatch(rl, la.numel(), lc, pmode=1, min_new=min_new)
    assert found == want, found
    for rb, wq, t in found:
        rows = la[rb * 128 + wq * 32:rb * 128 + wq * 32 + 32]
        cols = lc[t * 128:(t + 1) * 128]
        k = int((rows == rows[0]).sum())
        assert 0 < k < 32 and bool((cols[:4 * k] == rows[0]).all()) and bool((cols[4 * k:] == rows[-1]).all())


@pytest.mark.parametrize("k", [1, 5, 17, 31])
def test_dispatch_model_on_the_constructed_reproducer(k):
    """The hand-built reproducer of the GPU tests (N_a = 128, N_c = 256, split at K / 4K): the model sends warp 0
    down the general path with the fix and down the uniform path without it."""
    la = torch.full((128,), 3, dtype=torch.long)
    la[:k], la[k:32] = 1, 2
    lc = torch.cat([la, torch.full((128,), 2, dtype=torch.long)])
    lc[128:128 + 4 * k] = 1
    cnt, found = R.dispatch(la, 128, lc, pmode=0)
    assert found == [(0, 0, 1)] and cnt["s2_uniform_ones"] == 0
    cnt_old, _ = R.dispatch(la, 128, lc, pmode=0, old_uniform=True)
    assert cnt_old["s2_uniform_ones"] == 1
