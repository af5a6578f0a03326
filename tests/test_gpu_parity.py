"""GPU parity tests (run on the B200 box: ``pytest -m gpu``): the CUDA path, called through the
reference-shaped modules / the C ABI, against the CPU oracle and the golden fixtures.

Bars (BASELINE.json): bit-exact for label maps, pseudo labels, masks, counts, ignore handling and the
in-place label remap; loss within 1e-3 relative; gradient cosine >= 0.999.
"""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import ucd_oracle as O

pytestmark = pytest.mark.gpu

REL = 1e-3      # loss tolerance stated by north_star
COS = 0.999     # gradient cosine stated by north_star


@pytest.fixture(scope="module")
def U():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import ucd_b200
    from ucd_b200 import _lib
    assert _lib.lib().ucd_device_ok() == 1, "ucd_b200 needs a compute-capability 10.x device"
    return ucd_b200


def cos(a, b):
    a, b = a.double().reshape(-1).cpu(), b.double().reshape(-1).cpu()
    return float(a @ b / (a.norm() * b.norm()).clamp_min(1e-300))


def load_case(golden_dir, name):
    fx = np.load(os.path.join(golden_dir, name + ".npz"))
    B, h, w, H, W, C, C_old, corr = (int(v) for v in fx["shape"])
    return fx, O.synthetic_case(B, h, w, H, W, C, C_old, correlated=bool(corr)), (B, h, w, H, W, C, C_old)


# ------------------------------------------------------------------------------------------------
def test_umma_selftest(U):
    from ucd_b200 import _lib
    for variant in (0, 1, 2):
        err = ctypes.c_float(-1.0)
        _lib.check(_lib.debug_lib().ucd_selftest_umma(variant, ctypes.byref(err)), "selftest")
        assert 0 <= err.value < 2e-3, (variant, err.value)


@pytest.mark.parametrize("shape,size", [((2, 5, 9, 13), (144, 208)), ((2, 21, 33, 33), (513, 513)),
                                        ((1, 17, 32, 32), (512, 512)), ((1, 3, 32, 64), (512, 1024)),
                                        ((1, 2, 7, 5), (7, 5)), ((1, 1, 16, 16), (40, 24)),
                                        # interval / sweep kernels: scales 8, 32, mixed, rows that do not fill a segment
                                        ((2, 3, 64, 64), (512, 512)), ((1, 2, 16, 16), (512, 512)),
                                        ((1, 4, 24, 24), (384, 384)), ((2, 2, 32, 32), (256, 512)),
                                        ((1, 2, 40, 16), (320, 256)), ((1, 2, 33, 32), (66, 512)),
                                        # largest scale of the interval kernel (40x) and beyond it (generic kernel)
                                        ((1, 2, 4, 8), (160, 320)), ((1, 1, 3, 8), (144, 384)), ((1, 1, 5, 7), (171, 93)),
                                        # sweep backward with a shortened segment (37x along y) over several segments
                                        ((1, 2, 8, 8), (296, 256)), ((1, 1, 24, 8), (888, 256)),
                                        # sweep backward: row ranges that cross plane boundaries (100 planes of 5 rows on
                                        # 148 blocks), a single low-res row per plane
                                        ((4, 25, 5, 32), (80, 512)), ((2, 40, 1, 32), (16, 512))])
def test_upsample_fwd_bwd(U, shape, size):
    g = torch.Generator().manual_seed(11)
    x = torch.randn(*shape, generator=g)
    go = torch.randn(*shape[:2], *size, generator=g)
    xr = x.clone().requires_grad_(True)
    ref = F.interpolate(xr, size=size, mode="bilinear", align_corners=False)
    ref.backward(go)
    xc = x.cuda().requires_grad_(True)
    out = U.interpolate_bilinear(xc, size)
    out.backward(go.cuda())
    # forward: same taps and the same fp32 operation order as ATen's CPU kernels -> bit exact
    assert torch.equal(out.cpu(), ref.detach()), float((out.cpu() - ref.detach()).abs().max())
    assert np.array_equal(out.detach().cpu().numpy(), O._bilinear_eval_f32(x.numpy(), *size))
    # adjoint: fixed but different summation order -> fp32 tolerance
    torch.testing.assert_close(xc.grad.cpu(), xr.grad, rtol=1e-4, atol=3e-6 * float(xr.grad.abs().max()))
    torch.testing.assert_close(out.cpu(), O.upsample_bilinear(x, *size), rtol=1e-5, atol=1e-5)
    # the adjoint hands a range's trailing partial row to its neighbour with atomicAdd (two operands: commutative):
    # repeated runs must be bit-identical
    for _ in range(3):
        xc2 = x.cuda().requires_grad_(True)
        U.interpolate_bilinear(xc2, size).backward(go.cuda())
        assert torch.equal(xc2.grad, xc.grad)


@pytest.mark.parametrize("shape", [(2, 7, 9, 11), (2, 21, 64, 64), (1, 17, 33, 33), (3, 151, 16, 20)])
@pytest.mark.parametrize("reduction", ["none", "mean", "sum"])
def test_unce(U, shape, reduction):
    B, C, H, W = shape
    old_cl = max(1, (C * 3) // 4)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, C, H, W, generator=g) * 3
    y = torch.randint(0, C, (B, H, W), generator=g)
    y[0, :2] = 255
    y[-1, -1, -3:] = 255
    xr = x.double().requires_grad_(True)
    y_ref = y.clone()
    ref = O.unbiased_ce(xr, y_ref, old_cl, 255, reduction)
    w8 = torch.randn(B, H, W, generator=g).double()
    (ref * w8).sum().backward() if reduction == "none" else ref.backward()
    xc, yc = x.cuda().requires_grad_(True), y.cuda()
    out = U.UnbiasedCrossEntropy(old_cl=old_cl, reduction=reduction, ignore_index=255)(xc, yc)
    (out * w8.cuda().float()).sum().backward() if reduction == "none" else out.backward()
    assert torch.equal(yc.cpu(), y_ref), "in-place label remap must be bit exact"
    torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=2e-5, atol=2e-5)
    if reduction == "none":
        assert (out.cpu()[y_ref == 255] == 0).all()
    assert cos(xc.grad, xr.grad) > 1 - 1e-6
    torch.testing.assert_close(xc.grad.cpu().double(), xr.grad, rtol=1e-3, atol=5e-6 * float(xr.grad.abs().max()) + 1e-9)


def test_unce_broadcast_grad_and_noncontiguous_targets(U):
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 6, 8, 12, generator=g)
    y = torch.randint(0, 6, (2, 8, 24), generator=g)[:, :, ::2]          # non-contiguous view
    y_ref = y.clone()
    xr = x.double().requires_grad_(True)
    O.unbiased_ce(xr, y_ref, 4, 255, "none").mean().backward()
    xc = x.cuda().requires_grad_(True)
    yc = torch.zeros(2, 8, 24, dtype=torch.int64, device="cuda")[:, :, ::2]
    yc.copy_(y.cuda())
    assert not yc.is_contiguous()
    U.UnbiasedCrossEntropy(old_cl=4, reduction="none")(xc, yc).mean().backward()   # train.py:116 usage
    assert torch.equal(yc.cpu(), y_ref)
    assert cos(xc.grad, xr.grad) > 1 - 1e-6


@pytest.mark.parametrize("shape,c_old", [((2, 7, 9, 11), 4), ((2, 21, 64, 64), 16), ((1, 17, 33, 33), 16),
                                         ((2, 151, 16, 20), 101), ((1, 5, 8, 8), 5)])
@pytest.mark.parametrize("reduction,alpha,use_mask", [("mean", 1.0, False), ("sum", 0.5, True), ("none", 2.0, True)])
def test_unkd(U, shape, c_old, reduction, alpha, use_mask):
    B, C, H, W = shape
    g = torch.Generator().manual_seed(4)
    x = torch.randn(B, C, H, W, generator=g) * 3
    t = torch.randn(B, c_old, H, W, generator=g) * 3
    mask = (torch.rand(B, H, W, generator=g) > 0.3) if use_mask else None
    xr = x.double().requires_grad_(True)
    ref = O.unbiased_kd(xr, t.double(), alpha, reduction, mask)
    w8 = torch.randn(B, H, W, generator=g).double()
    (ref * w8).sum().backward() if reduction == "none" else ref.backward()
    xc = x.cuda().requires_grad_(True)
    mod = U.UnbiasedKnowledgeDistillationLoss(reduction=reduction, alpha=alpha)
    out = mod(xc, t.cuda(), None if mask is None else mask.cuda())
    (out * w8.cuda().float()).sum().backward() if reduction == "none" else out.backward()
    torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=5e-5, atol=5e-5)
    assert cos(xc.grad, xr.grad) > 1 - 1e-6
    torch.testing.assert_close(xc.grad.cpu().double(), xr.grad, rtol=1e-3, atol=5e-6 * float(xr.grad.abs().max()) + 1e-9)


# ------------------------------------------------------------------------------------------------
def test_label_downsample_bit_exact(U, golden_dir):
    """label_n of the prep kernel == the reference's resize+int8+clamp on every golden label map."""
    from ucd_b200.losses import _build_pack
    fx = np.load(os.path.join(golden_dir, "label_downsample.npz"))
    maps = O.label_downsample_maps()
    names = sorted(k[:-len("_in_sha256")] for k in fx.files if k.endswith("_in_sha256"))
    assert len(names) == 12 and sorted(maps) == names
    for n in names:
        assert O.label_map_digest(maps[n]) == str(fx[n + "_in_sha256"]), "label map generator drifted: " + n
        lab = torch.from_numpy(maps[n].astype(np.int64)).cuda()
        want = fx[n + "_out"].astype(np.int64)
        B, h, w = want.shape
        l_po = torch.zeros(B, 2, h, w, device="cuda")
        l_po[:, 1] = 1.0                                           # pseudo label 1 everywhere -> every pixel anchors
        f = torch.randn(B, 256, h, w, device="cuda")
        pk = _build_pack(f, f, l_po, lab, 20)
        assert np.array_equal(pk.label_n.view(B, h, w).cpu().numpy().astype(np.int64), want), n
        assert np.array_equal(pk.label_n.cpu().numpy(), O.downsample_labels(maps[n].astype(np.int64), h, w).reshape(-1)), n


@pytest.mark.parametrize("name", ["tiny_b2", "voc15-5_b2_513", "voc15-5s_b3_512", "city13-6_b3", "voc15-5s_b2_corr"])
def test_contrastive_prep_integer_artefacts_and_rows(U, golden_dir, name):
    fx, case, (B, h, w, H, W, C, C_old) = load_case(golden_dir, name)
    tup = U.pre_contrastive_pixel(case["f_n"].cuda(), case["labels"].cuda(), l_po=case["l_po"].cuda(),
                                  f_o=case["f_o"].cuda())
    A, Cst, la, lc, JP = tup
    pk = JP.pack
    prep = O.prep_labels(case["labels"].numpy(), case["l_po"].numpy())
    # bit-exact integer artefacts: vs the reference's fixture and vs the oracle
    assert np.array_equal(la.cpu().numpy(), fx["la"]) and np.array_equal(lc.cpu().numpy(), fx["lc"])
    assert np.array_equal(pk.label_n.cpu().numpy().reshape(B, h, w), fx["label_n"].astype(np.int32))
    assert pk.min_new == prep.min_new and pk.n_a == int(prep.anchor.sum()) and pk.n_o == int(prep.pseudo_mask.sum())
    flags = pk.flags.cpu().numpy()
    assert np.array_equal((flags & 1) > 0, prep.anchor) and np.array_equal((flags & 2) > 0, prep.pseudo_mask)
    assert np.array_equal(pk.mix.cpu().numpy(), prep.mix.reshape(-1))
    # normalised rows and the dense joint-probability matrix
    Ao, Co, lao, lco, Po, _ = O.pre_contrastive_pixel(case["f_n"], case["labels"], case["l_po"], case["f_o"])
    torch.testing.assert_close(A.cpu(), Ao, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(Cst.cpu(), Co, rtol=1e-5, atol=1e-6)
    Pd = JP.dense().cpu()
    assert int((Pd == 1).sum()) == int(fx["p_ones"][0])
    torch.testing.assert_close(Pd, Po, rtol=1e-4, atol=1e-6)
    # packed bf16 tiles hold the same rows (bf16 rounding only) in CLASS-SORTED order: stable sort by label of the
    # anchors, then of the pseudo columns; row_ref maps sorted anchor rows back; padding labels are -1
    perm_a = torch.argsort(lao, stable=True)
    perm_o = torch.argsort(lco[pk.n_a:], stable=True) + pk.n_a
    perm = torch.cat([perm_a, perm_o])
    assert torch.equal(pk.row_ref[:pk.n_a].cpu().long(), perm_a)
    ft = pk.feat_tiles.float().cpu()                     # [T, 32, 128, 8]
    rows = ft.permute(0, 2, 1, 3).reshape(-1, 256)[:pk.n_c]
    assert float((rows - Co[perm]).abs().max()) < 2 ** -8
    lt = pk.lab_tiles.cpu().reshape(-1)
    # padding of the last tile the sweeps read: label -1, zero features / probabilities (tiles beyond it are never read)
    pad_end = ((pk.n_c + 127) // 128) * 128
    assert torch.equal(lt[:pk.n_c].long(), lco[perm]) and bool((lt[pk.n_c:pad_end] == -1).all())
    assert float(ft.permute(0, 2, 1, 3).reshape(-1, 256)[pk.n_c:pad_end].abs().sum()) == 0.0
    tr = pk.tile_range.cpu()
    for t in range((pk.n_c + 127) // 128):
        seg = lt[t * 128:min(pk.n_c, (t + 1) * 128)]
        assert int(tr[t, 0]) == int(seg.min()) and int(tr[t, 1]) == int(seg.max())
    # bf16 softmax tiles follow the same order
    p_ref = torch.softmax(case["l_po"].permute(0, 2, 3, 1).reshape(-1, C_old), 1)
    pc = torch.cat([p_ref[torch.from_numpy(prep.anchor)], p_ref[torch.from_numpy(prep.pseudo_mask)]])[perm]
    pt_all = pk.prob_tiles.float().cpu().permute(0, 2, 1, 3).reshape(-1, pk.kpad)
    assert float(pt_all[pk.n_c:pad_end].abs().sum()) == 0.0
    pt = pt_all[:pk.n_c]
    assert float((pt[:, :C_old] - pc).abs().max()) < 2 ** -8
    assert pk.kpad == C_old or float(pt[:, C_old:].abs().max()) == 0.0


@pytest.mark.parametrize("name", ["tiny_b2", "voc15-5_b2_513", "voc15-5s_b3_512", "city13-6_b3", "voc15-5s_b2_corr"])
def test_contrastive_loss_and_grad_vs_reference_fixture(U, golden_dir, name):
    fx, case, (B, h, w, H, W, C, C_old) = load_case(golden_dir, name)
    f_n = case["f_n"].cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
    loss = U.PixelConLossV2(temperature=0.07)(*tup)
    loss.backward()
    assert loss.item() == pytest.approx(fx["con"][1], rel=REL)
    s = int(fx["stride"][0])
    got = f_n.grad.reshape(-1)[::s].cpu()
    assert cos(got, torch.from_numpy(fx["g_fn_sample"])) >= COS
    assert float(f_n.grad.norm()) == pytest.approx(fx["g_fn_norm"][1], rel=2e-2)
    if "full_g_fn" in fx.files:
        assert cos(f_n.grad, torch.from_numpy(fx["full_g_fn"])) >= COS


@pytest.mark.parametrize("n_a,n_c,with_p", [(200, 333, "none"), (200, 333, "dense"), (129, 128, "dense"),
                                            (64, 700, "none"), (300, 300, "dense")])
def test_pixelconloss_compat_dense_inputs(U, n_a, n_c, with_p):
    """PixelConLossV2.forward with plain dense tensors, arbitrary labels, P None / dense (loss.py:412-466)."""
    g = torch.Generator().manual_seed(n_a * 1000 + n_c)
    A = F.normalize(torch.randn(n_a, 256, generator=g), dim=1)
    Cst = F.normalize(torch.randn(n_c, 256, generator=g), dim=1)
    k = min(n_a, n_c)
    Cst[:k] = A[:k]
    la = torch.randint(1, 6, (n_a,), generator=g)
    lc = torch.randint(1, 6, (n_c,), generator=g)
    lc[:k] = la[:k]
    P = torch.rand(n_a, n_c, generator=g) if with_p == "dense" else None
    Ar = A.double().requires_grad_(True)
    ref = O.pixel_con_loss(Ar, Cst.double(), la, lc, None if P is None else P.double(), 0.07,
                           self_col=torch.where(torch.arange(n_a) < n_c, torch.arange(n_a), -torch.ones(n_a, dtype=torch.long)))
    ref.backward()
    Ac = A.cuda().requires_grad_(True)
    out = U.PixelConLossV2(temperature=0.07)(Ac, Cst.cuda(), la.to(torch.int8).cuda(), lc.to(torch.int8).cuda(),
                                             None if P is None else P.cuda())
    out.backward()
    assert out.item() == pytest.approx(ref.item(), rel=REL)
    assert cos(Ac.grad, Ar.grad) >= COS


@pytest.mark.parametrize("c_tot,c_old,max_label", [(151, 101, 150), (40, 30, 39), (70, 60, 69),
                                                    # beyond 112 old classes both probability operands are streamed
                                                    # (ADE 100-10 from its second step on: 111, 121, ... 141 old classes)
                                                    (151, 121, 150), (151, 141, 150), (230, 200, 229)])
def test_contrastive_wide_joint_probability(U, c_tot, c_old, max_label):
    """ADE-like class counts (BASELINE config 3): joint-probability width > 16 (K-chunked P GEMM) and labels > 20.
    The reference itself cannot run this (hard-coded VOC clamp + int8 cast, SURVEY A.1), so the bar is the oracle
    with ``max_label`` (the "patched oracle")."""
    case = O.synthetic_case(2, 16, 16, 256, 256, c_tot, c_old, correlated=True)
    f_ref = case["f_n"].double().requires_grad_(True)
    A, Cst, la, lc, P, prep = O.pre_contrastive_pixel(f_ref, case["labels"], case["l_po"].double(), case["f_o"].double(),
                                                       max_label=max_label)
    ref = O.pixel_con_loss(A, Cst, la, lc, P)
    ref.backward()
    f_n = case["f_n"].cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda(),
                                  max_label=max_label)
    assert np.array_equal(tup[2].cpu().numpy(), la.numpy()) and np.array_equal(tup[3].cpu().numpy(), lc.numpy())
    assert tup[4].pack.min_new == prep.min_new
    loss = U.PixelConLossV2(temperature=0.07)(*tup)
    loss.backward()
    assert loss.item() == pytest.approx(ref.item(), rel=REL)
    assert cos(f_n.grad, f_ref.grad) >= COS


@pytest.mark.parametrize("name", ["voc15-5_b2_513", "voc15-5s_b3_512"])
def test_whole_hot_path_matches_reference(U, golden_dir, name):
    """train.py:115-116,133: UNCE(outputs,labels).mean() + con/100 + 10*UNKD(outputs, outputs_old)."""
    fx, case, (B, h, w, H, W, C, C_old) = load_case(golden_dir, name)
    f_n = case["f_n"].cuda().requires_grad_(True)
    lr = case["logits_lr"].cuda().requires_grad_(True)
    labels = case["labels"].cuda()
    l_po, f_o = case["l_po"].cuda(), case["f_o"].cuda()
    outputs = U.interpolate_bilinear(lr, (H, W))
    with torch.no_grad():
        outputs_old = U.interpolate_bilinear(l_po, (H, W))
    con = U.PixelConLossV2(temperature=0.07)(*U.pre_contrastive_pixel(f_n, labels, l_po=l_po, f_o=f_o))
    ce = U.UnbiasedCrossEntropy(old_cl=C_old, ignore_index=255, reduction="none")(outputs, labels).mean()
    kd = U.UnbiasedKnowledgeDistillationLoss(alpha=1.0)(outputs, outputs_old)
    (ce + con / 100 + 10 * kd).backward()
    assert con.item() == pytest.approx(fx["con"][1], rel=REL)
    assert ce.item() == pytest.approx(fx["ce"][1], rel=REL)
    assert kd.item() == pytest.approx(fx["kd"][1], rel=REL)
    s = int(fx["stride"][0])
    assert cos(lr.grad.reshape(-1)[::s], torch.from_numpy(fx["g_lr_sample"])) >= COS
    assert float(lr.grad.norm()) == pytest.approx(fx["g_lr_norm"][1], rel=1e-3)
    assert int((labels.cpu() != case["labels"]).sum()) == int(fx["lab_ce_changed"][0])


# ------------------------------------------------------------------------------------------------
# size-independent properties at BASELINE config-2 size (batch 24 @ 512x512)
# ------------------------------------------------------------------------------------------------
def _run_con(U, case, order=None):
    f_n = case["f_n"].cuda()
    labels, l_po, f_o = case["labels"].cuda(), case["l_po"].cuda(), case["f_o"].cuda()
    if order is not None:
        f_n, labels, l_po, f_o = f_n[order], labels[order], l_po[order], f_o[order]
    f_n = f_n.clone().requires_grad_(True)
    loss = U.PixelConLossV2(temperature=0.07)(*U.pre_contrastive_pixel(f_n, labels, l_po=l_po, f_o=f_o))
    loss.backward()
    return loss.detach(), f_n.grad


def test_full_size_properties(U):
    case = O.synthetic_case(24, 32, 32, 512, 512, 17, 16, correlated=True)
    l1, g1 = _run_con(U, case)
    l2, g2 = _run_con(U, case)
    assert torch.isfinite(l1) and torch.isfinite(g1).all()
    assert torch.equal(l1, l2) and torch.equal(g1, g2), "fixed-order reductions: runs must be bit-identical"
    # the loss is invariant to the order of images (rows and columns are both permuted)
    perm = torch.randperm(24, generator=torch.Generator().manual_seed(1)).cuda()
    l3, g3 = _run_con(U, case, perm)
    assert l3.item() == pytest.approx(l1.item(), rel=1e-4)
    assert cos(g3, g1[perm]) > 0.9999
    # normalisation adjoint: the gradient of every pixel is orthogonal to its feature vector
    dots = (g1 * case["f_n"].cuda()).sum(1)
    assert float(dots.abs().max()) < 1e-3 * float(g1.abs().max()) * float(case["f_n"].norm(dim=1).max())
    # non-anchor pixels get exactly zero gradient
    prep = O.prep_labels(case["labels"].numpy(), case["l_po"].numpy())
    gz = g1.permute(0, 2, 3, 1).reshape(-1, 256)[torch.from_numpy(~prep.anchor).cuda()]
    assert gz.numel() == 0 or float(gz.abs().max()) == 0.0


def _streaming_reference(case, max_label=20, block=256):
    """fp64 reference loss and d loss / d f_n at sizes where the dense N_a x N_c restatement does not fit: the
    row-blocked oracle (pinned against the reference fixtures in tests/test_oracle.py) + autograd through the
    anchor gather / normalisation."""
    f_ref = case["f_n"].double().requires_grad_(True)
    A, Cst, la, lc, pa, pc, prep = O.contrast_operands(f_ref, case["labels"], case["l_po"].double(),
                                                       case["f_o"].double(), max_label=max_label)
    loss, dA, _ = O.pixel_con_loss_streaming(A, Cst, la, lc, pa, pc, prep.min_new, block=block)
    A.backward(dA)
    return loss, f_ref.grad, prep, (la, lc)


def test_bench_workload_against_streaming_oracle(U):
    """The benchmarked size itself (BASELINE configs[1] per GPU: B=24 @512x512, 23 419 anchors x 41 102 contrast
    columns, 4 column splits): loss within 1e-3 and gradient cosine >= 0.999 against the fp64 oracle, for the whole
    gradient, and per anchor row on a seeded sample of 512 rows plus the rows either side of every 128-row tile
    boundary next to a column-split boundary (the rows whose column ranges start / end a CTA)."""
    case = O.synthetic_case(24, 32, 32, 512, 512, 17, 16, correlated=True)
    ref_loss, ref_grad, prep, (la, lc) = _streaming_reference(case)
    f_n = case["f_n"].cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
    assert tup[0].shape[0] == la.numel() == 23419 and tup[1].shape[0] == lc.numel() == 41102
    assert np.array_equal(tup[2].cpu().numpy(), la.numpy()) and np.array_equal(tup[3].cpu().numpy(), lc.numpy())
    loss = U.PixelConLossV2(temperature=0.07)(*tup)
    loss.backward()
    assert loss.item() == pytest.approx(ref_loss.item(), rel=REL)
    assert cos(f_n.grad, ref_grad) >= COS
    # per-row check (pixel = one anchor row of the gradient)
    g = f_n.grad.permute(0, 2, 3, 1).reshape(-1, 256).double().cpu()
    r = ref_grad.permute(0, 2, 3, 1).reshape(-1, 256)
    anchor_px = np.nonzero(prep.anchor)[0]
    n_a = anchor_px.size
    rs = np.random.RandomState(7)
    rows = set(rs.choice(n_a, 512, replace=False).tolist())
    for b in range(128, n_a, 128):
        rows.update((b - 1, b))
    rows.update((0, n_a - 1))
    rows = np.array(sorted(rows))
    px = torch.from_numpy(anchor_px[rows])
    gs, rs_ = g[px], r[px]
    norms = rs_.norm(dim=1)
    row_cos = (gs * rs_).sum(1) / (gs.norm(dim=1) * norms).clamp_min(1e-300)
    big = norms > 1e-3 * norms.max()          # rows whose gradient is not pure cancellation noise
    assert int(big.sum()) >= 256
    assert float(row_cos[big].min()) >= COS, float(row_cos[big].min())
    # pixels that are not anchors get exactly zero
    assert float(g[torch.from_numpy(~prep.anchor)].abs().max()) == 0.0


def test_ade_real_size_unbiased_losses(U):
    """BASELINE configs[2] at its real size: ADE 100-50 step 1, 3 x 151 / 101 classes at 512x512 (475 MB of logits):
    upsample + UNCE(.mean) + UNKD through the drop-in modules and through the fused N1 module, against the fp64
    oracle chain evaluated image by image (losses 1e-3 - in fact 1e-5 - and logit-gradient cosine >= 0.999)."""
    B, h, w, H, W, C, C_old = 3, 32, 32, 512, 512, 151, 101
    case = O.synthetic_case(B, h, w, H, W, C, C_old)
    n_px = float(B * H * W)
    ce_ref = kd_ref = 0.0
    g_ref = torch.zeros(B, C, h, w, dtype=torch.float64)
    for b in range(B):                         # per image: bounds the fp64 temporaries (317 MB per logit tensor)
        lr = case["logits_lr"][b:b + 1].double().requires_grad_(True)
        x = O.upsample_bilinear(lr, H, W)
        t = O.upsample_bilinear(case["l_po"][b:b + 1].double(), H, W)
        ce = O.unbiased_ce(x, case["labels"][b:b + 1].clone(), C_old, 255, "none").sum() / n_px
        kd = O.unbiased_kd(x, t, 1.0, "sum") / n_px      # 'mean' = sum over pixels / (B H W), sign included
        (ce + 10 * kd).backward()
        ce_ref, kd_ref = ce_ref + ce.item(), kd_ref + kd.item()
        g_ref[b] = lr.grad[0]
    lr = case["logits_lr"].cuda().requires_grad_(True)
    labels = case["labels"].cuda()
    out = U.interpolate_bilinear(lr, (H, W))
    with torch.no_grad():
        old = U.interpolate_bilinear(case["l_po"].cuda(), (H, W))
    ce = U.UnbiasedCrossEntropy(old_cl=C_old, ignore_index=255, reduction="none")(out, labels).mean()
    kd = U.UnbiasedKnowledgeDistillationLoss(alpha=1.0)(out, old)
    (ce + 10 * kd).backward()
    assert ce.item() == pytest.approx(ce_ref, rel=1e-5) and kd.item() == pytest.approx(kd_ref, rel=1e-5)
    assert cos(lr.grad, g_ref) >= COS
    torch.testing.assert_close(lr.grad.cpu().double(), g_ref, rtol=2e-3, atol=1e-5 * float(g_ref.abs().max()))
    del out, old
    lr2 = case["logits_lr"].cuda().requires_grad_(True)
    ce2, kd2 = U.FusedUnbiasedLosses(old_cl=C_old, ignore_index=255, alpha=1.0)(lr2, case["l_po"].cuda(),
                                                                              case["labels"].cuda())
    (ce2 + 10 * kd2).backward()
    assert ce2.item() == pytest.approx(ce_ref, rel=1e-5) and kd2.item() == pytest.approx(kd_ref, rel=1e-5)
    assert cos(lr2.grad, g_ref) >= COS


def test_ade_real_size_wide_joint_probability(U):
    """ADE 100-50 step 1 contrastive term at its real per-GPU size (3 x 32 x 32 pixels, 101 old classes -> K = 112
    joint-probability width streamed in K chunks, labels up to 150): the reference itself crashes here (SURVEY A.1);
    the oracle is the patched reference (max_label = C - 1)."""
    case = O.synthetic_case(3, 32, 32, 512, 512, 151, 101, correlated=True)
    _compare_contrastive(U, case, max_label=150)


@pytest.mark.parametrize("tag", ["single", "double"])
def test_pixel_to_pixel_branches(U, golden_dir, tag):
    """pre_contrastive_pixel without old-model logits (utils/loss.py:278-289) against the reference's own outputs:
    labels bit-exact, rows and gradient to fp32 accuracy."""
    fx = np.load(os.path.join(golden_dir, "pixel_to_pixel.npz"))
    B, h, w, H, W, C, C_old = (int(v) for v in fx["shape"])
    case = O.synthetic_case(B, h, w, H, W, C, C_old)
    f_n = case["f_n"].cuda().requires_grad_(True)
    out, lab = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), f_o=case["f_o"].cuda() if tag == "double" else None)
    assert out.shape == fx[tag + "_out"].shape and lab.dtype == torch.int8
    assert np.array_equal(lab.cpu().numpy(), fx[tag + "_lab"])
    torch.testing.assert_close(out.cpu().double(), torch.from_numpy(fx[tag + "_out"]), rtol=1e-5, atol=1e-6)
    (out * torch.from_numpy(fx["w"])[:out.shape[0]].float().cuda()).sum().backward()
    torch.testing.assert_close(f_n.grad.cpu().double(), torch.from_numpy(fx[tag + "_grad"]), rtol=1e-4, atol=1e-5)
    with pytest.raises(UnboundLocalError):   # l_po without f_o: `Output` is unassigned in the reference (loss.py:399)
        U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda())


def test_foreign_anchor_tensor_is_loud(U):
    """A cast / clone of the anchors cannot use the packed operands: the dense fallback warns, and refuses above
    max_dense_bytes; contrast features that require grad are refused (only d/d anchor is formed)."""
    case = O.synthetic_case(2, 8, 8, 128, 128, 6, 4)
    f_n = case["f_n"].cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
    con = U.PixelConLossV2(temperature=0.07)
    ref = con(*tup)
    with pytest.warns(RuntimeWarning, match="dense"):
        out = con(tup[0].clone(), *tup[1:])
    assert out.item() == pytest.approx(ref.item(), rel=REL)   # fp32 dense P vs the bf16 probability tiles
    con.max_dense_bytes = 16
    with pytest.raises(RuntimeError, match="max_dense_bytes"):
        con(tup[0].clone(), *tup[1:])
    with pytest.raises(RuntimeError, match="requires grad"):
        U.PixelConLossV2(temperature=0.07)(tup[0].detach(), tup[1].clone().requires_grad_(True), tup[2], tup[3], None)


def test_shared_logit_gradient_chain(U):
    """UNCE and UNKD on the same `outputs` tensor (train.py:116,133) write ONE gradient buffer (the second backward
    accumulates in its kernel): same gradients as the oracle's autograd in every usage pattern - both losses, either
    one alone, reversed call order, a third consumer of `outputs`, two backward passes with retain_graph - and no
    full-size elementwise add kernel on the way."""
    from torch.profiler import ProfilerActivity, profile
    B, C, C_old, H, W = 2, 9, 6, 64, 96
    g = torch.Generator().manual_seed(21)
    x0 = torch.randn(B, C, H, W, generator=g) * 2
    t0 = torch.randn(B, C_old, H, W, generator=g) * 2
    y0 = torch.randint(0, C, (B, H, W), generator=g)
    y0[0, :3] = 255

    def ref(use_ce, use_kd, extra):
        x = x0.double().requires_grad_(True)
        out = x * 1.0
        loss = 0
        if use_ce:
            loss = loss + O.unbiased_ce(out, y0.clone(), C_old, 255, "none").mean()
        if use_kd:
            loss = loss + 10 * O.unbiased_kd(out, t0.double(), 1.0)
        if extra:
            loss = loss + (out * 0.01).sum()
        loss.backward()
        return x.grad

    def ours(use_ce, use_kd, extra, order="ce_first", passes=1):
        x = x0.cuda().requires_grad_(True)
        out = x * 1.0                       # a non-leaf `outputs`, like the upsampled logits
        ce_m = U.UnbiasedCrossEntropy(old_cl=C_old, ignore_index=255, reduction="none")
        kd_m = U.UnbiasedKnowledgeDistillationLoss(alpha=1.0)
        calls = [("ce", lambda: ce_m(out, y0.cuda()).mean()), ("kd", lambda: 10 * kd_m(out, t0.cuda()))]
        if order != "ce_first":
            calls.reverse()
        vals = {k: f() for k, f in calls}       # both forwards always run; only the selected ones enter the loss
        loss = (out * 0.01).sum() if extra else 0
        if use_ce:
            loss = loss + vals["ce"]
        if use_kd:
            loss = loss + vals["kd"]
        for i in range(passes):
            loss.backward(retain_graph=i + 1 < passes)
        return x.grad / passes

    for use_ce, use_kd, extra, order, passes in [(True, True, False, "ce_first", 1), (True, True, False, "kd_first", 1),
                                                 (True, False, False, "ce_first", 1), (False, True, False, "ce_first", 1),
                                                 (False, True, True, "kd_first", 1), (True, True, True, "ce_first", 2)]:
        want = ref(use_ce, use_kd, extra)
        got = ours(use_ce, use_kd, extra, order, passes)
        assert cos(got, want) > 1 - 1e-6, (use_ce, use_kd, extra, order, passes)
        torch.testing.assert_close(got.cpu().double(), want, rtol=1e-3, atol=1e-5 * float(want.abs().max()))
    # a persistent input tensor used step after step (forward + backward each time, and forward-only evaluations in
    # between) must not link one step's graph to the previous one's
    xp = x0.cuda().requires_grad_(True)
    ce_m = U.UnbiasedCrossEntropy(old_cl=C_old, ignore_index=255, reduction="none")
    kd_m = U.UnbiasedKnowledgeDistillationLoss(alpha=1.0)
    want = ref(True, True, False)
    for it in range(3):
        for _ in range(it * 3):                       # evaluations whose graph is dropped
            ce_m(xp, y0.cuda()).mean()
        xp.grad = None
        (ce_m(xp, y0.cuda()).mean() + 10 * kd_m(xp, t0.cuda())).backward()
        assert cos(xp.grad, want) > 1 - 1e-6, it
    (gx,) = torch.autograd.grad(kd_m(xp, t0.cuda()), xp)
    assert cos(gx, ref(False, True, False) / 10) > 1 - 1e-6
    # no elementwise add over the full-size gradients
    x = x0.cuda().requires_grad_(True)
    out = U.interpolate_bilinear(x, (2 * H, 2 * W))
    yy = torch.zeros(B, 2 * H, 2 * W, dtype=torch.int64, device="cuda")
    tt = U.interpolate_bilinear(t0.cuda(), (2 * H, 2 * W))
    loss = (U.UnbiasedCrossEntropy(old_cl=C_old, reduction="none")(out, yy).mean()
            + 10 * U.UnbiasedKnowledgeDistillationLoss()(out, tt))
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss.backward()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages()]
    assert any("unce_unkd_bwd_kernel" in n for n in names), names   # one pass over the logits for both losses
    big_adds = [e for e in prof.key_averages() if "CUDAFunctor_add" in e.key and e.device_time_total / max(e.count, 1) > 20]
    assert not big_adds, [e.key for e in big_adds]


# ------------------------------------------------------------------------------------------------
# edge cases and randomised shapes
# ------------------------------------------------------------------------------------------------
def _compare_contrastive(U, case, max_label=20, rel=REL):
    f_ref = case["f_n"].double().requires_grad_(True)
    A, Cst, la, lc, P, prep = O.pre_contrastive_pixel(f_ref, case["labels"], case["l_po"].double(), case["f_o"].double(),
                                                       max_label=max_label)
    ref = O.pixel_con_loss(A, Cst, la, lc, P)
    ref.backward()
    f_n = case["f_n"].cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(f_n, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda(),
                                  max_label=max_label)
    pk = tup[4].pack
    assert np.array_equal(pk.label_n.cpu().numpy(), prep.label_n.reshape(-1))
    assert np.array_equal(tup[2].cpu().numpy(), la.numpy()) and np.array_equal(tup[3].cpu().numpy(), lc.numpy())
    loss = U.PixelConLossV2(temperature=0.07)(*tup)
    loss.backward()
    if torch.isnan(ref):                      # no row with a positive: the reference's mean of an empty set
        assert torch.isnan(loss)
        return
    assert loss.item() == pytest.approx(ref.item(), rel=rel)
    if float(f_ref.grad.norm()) > 0:
        assert cos(f_n.grad, f_ref.grad) >= COS


@pytest.mark.parametrize("seed", range(12))
def test_contrastive_random_shapes(U, seed):
    g = torch.Generator().manual_seed(100 + seed)
    ri = lambda lo, hi: int(torch.randint(lo, hi + 1, (1,), generator=g))  # noqa: E731
    B, h, w = ri(1, 3), ri(3, 20), ri(3, 20)
    scale = (8, 16)[ri(0, 1)]
    H, W = h * scale + ri(0, 1), w * scale + ri(0, 1)
    c_old, n_new = ri(2, 20), ri(1, 5)
    c_tot = min(c_old + n_new, 21)
    c_old = c_tot - n_new
    case = dict(f_n=torch.randn(B, 256, h, w, generator=g), f_o=torch.randn(B, 256, h, w, generator=g),
                l_po=torch.randn(B, c_old, h, w, generator=g) * 3)
    lab = torch.zeros(B, H, W, dtype=torch.int64)
    for _ in range(ri(1, 4)):                  # random rectangles of new-class labels, plus an ignore band
        y0, x0 = ri(0, H - 2), ri(0, W - 2)
        lab[ri(0, B - 1), y0:y0 + ri(1, H), x0:x0 + ri(1, W)] = ri(c_old, c_tot - 1)
    lab[:, :ri(0, H // 8)] = 255
    lab[0, H // 2:H // 2 + max(2 * scale, 2), W // 2:W // 2 + max(2 * scale, 2)] = c_old   # guarantee a new-class pixel
    case["labels"] = lab
    _compare_contrastive(U, case)


def test_contrastive_no_pseudo_pixels(U):
    """Old model predicts background everywhere: N_o = 0, the contrast set is the anchors themselves."""
    case = O.synthetic_case(2, 12, 12, 192, 192, 8, 6)
    case["l_po"][:, 0] = 100.0
    _compare_contrastive(U, case)


def test_contrastive_single_image_and_tiny_sets(U):
    """B = 1 (the reference's squeeze() breaks there; the oracle and the kernels do not), N_a below one tile."""
    case = O.synthetic_case(1, 6, 7, 96, 112, 8, 6)
    _compare_contrastive(U, case)


def test_contrastive_raises_without_new_class_pixel(U):
    case = O.synthetic_case(2, 8, 8, 128, 128, 6, 4)
    lab = torch.zeros_like(case["labels"])
    with pytest.raises(RuntimeError, match="no new-class pixel"):
        U.pre_contrastive_pixel(case["f_n"].cuda(), lab.cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
    with pytest.raises(ValueError):
        O.prep_labels(lab.numpy(), case["l_po"].numpy())


def test_contrastive_bit_identical_reruns(U):
    """Fixed-order reductions and race-free role pipelines: 20 reruns of a multi-row-block case are bit-identical
    (this caught a shared-memory scratch that aliased an in-flight bulk copy)."""
    case = O.synthetic_case(3, 32, 64, 512, 1024, 20, 14)
    inp = {k: v.cuda() for k, v in case.items()}
    con = U.PixelConLossV2(temperature=0.07)

    def run():
        f_n = inp["f_n"].clone().requires_grad_(True)
        loss = con(*U.pre_contrastive_pixel(f_n, inp["labels"], l_po=inp["l_po"], f_o=inp["f_o"]))
        loss.backward()
        return loss.detach().clone(), f_n.grad.clone()

    l0, g0 = run()
    for _ in range(20):
        l, g = run()
        assert torch.equal(l, l0) and torch.equal(g, g0)


def test_contrastive_no_grad_mode(U, golden_dir):
    """validation-style call under no_grad: sweeps run without the V/U accumulation, same loss."""
    fx, case, _ = load_case(golden_dir, "voc15-5s_b3_512")
    with torch.no_grad():
        tup = U.pre_contrastive_pixel(case["f_n"].cuda(), case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
        loss = U.PixelConLossV2(temperature=0.07)(*tup)
    assert not loss.requires_grad
    assert loss.item() == pytest.approx(fx["con"][1], rel=REL)


def test_unce_all_ignored_and_old_only_labels(U):
    x = torch.randn(1, 5, 8, 8, device="cuda", requires_grad=True)
    y = torch.full((1, 8, 8), 255, dtype=torch.int64, device="cuda")
    out = U.UnbiasedCrossEntropy(old_cl=3, reduction="none")(x, y)
    out.sum().backward()
    assert float(out.detach().abs().max()) == 0.0 and float(x.grad.abs().max()) == 0.0
    y2 = torch.randint(0, 3, (1, 8, 8), device="cuda")            # only old labels: all remapped to 0
    out2 = U.UnbiasedCrossEntropy(old_cl=3, reduction="mean")(x, y2)
    assert int(y2.abs().max()) == 0
    ref = O.unbiased_ce(x.detach().cpu().double(), torch.zeros(1, 8, 8, dtype=torch.int64), 3, 255, "mean")
    assert out2.item() == pytest.approx(ref.item(), rel=1e-5)


# ------------------------------------------------------------------------------------------------
# N1: fused upsample + UNCE + UNKD from the low-res logits
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B,C,c_old,h,w,scale", [(2, 21, 16, 9, 11, 16), (2, 17, 16, 32, 32, 16), (1, 8, 6, 5, 7, 8),
                                                 (2, 151, 101, 6, 5, 16), (1, 6, 6, 4, 4, 16), (2, 20, 14, 8, 16, 16)])
def test_fused_unbiased_losses(U, B, C, c_old, h, w, scale):
    H, W = h * scale + (1 if (h + w) % 2 else 0), w * scale + (1 if (h + w) % 2 else 0)   # also 513-style sizes
    g = torch.Generator().manual_seed(B * 1000 + C)
    lr = torch.randn(B, C, h, w, generator=g) * 3
    lo = torch.randn(B, c_old, h, w, generator=g) * 3
    lab = torch.randint(0, C, (B, H, W), generator=g)
    lab[:, : max(1, H // 20)] = 255
    # reference: the three separate reference ops (oracle restatements), fp64
    lr_ref = lr.double().requires_grad_(True)
    out = O.upsample_bilinear(lr_ref, H, W)
    old = O.upsample_bilinear(lo.double(), H, W)
    lab_ref = lab.clone()
    ce_ref = O.unbiased_ce(out, lab_ref, c_old, 255, "none").mean()
    kd_ref = O.unbiased_kd(out, old, 1.0)
    (ce_ref + 10 * kd_ref).backward()
    lr_c, lab_c = lr.cuda().requires_grad_(True), lab.cuda()
    ce, kd = U.FusedUnbiasedLosses(old_cl=c_old, alpha=1.0)(lr_c, lo.cuda(), lab_c)
    (ce + 10 * kd).backward()
    assert torch.equal(lab_c.cpu(), lab_ref), "in-place label remap"
    assert ce.item() == pytest.approx(ce_ref.item(), rel=REL)
    assert kd.item() == pytest.approx(kd_ref.item(), rel=REL)
    assert cos(lr_c.grad, lr_ref.grad) >= COS
    torch.testing.assert_close(lr_c.grad.cpu().double(), lr_ref.grad, rtol=2e-3, atol=2e-5 * float(lr_ref.grad.abs().max()))
    # and equal to the unfused drop-in modules
    lr_d = lr.cuda().requires_grad_(True)
    o = U.interpolate_bilinear(lr_d, (H, W))
    ce_d = U.UnbiasedCrossEntropy(old_cl=c_old, reduction="none")(o, lab.cuda()).mean()
    kd_d = U.UnbiasedKnowledgeDistillationLoss()(o, U.interpolate_bilinear(lo.cuda(), (H, W)))
    assert ce.item() == pytest.approx(ce_d.item(), rel=1e-4) and kd.item() == pytest.approx(kd_d.item(), rel=1e-4)
    # fixed-order cross-block sums: reruns are bit-identical
    for _ in range(5):
        lr_r = lr.cuda().requires_grad_(True)
        ce_r, kd_r = U.FusedUnbiasedLosses(old_cl=c_old, alpha=1.0)(lr_r, lo.cuda(), lab.cuda())
        (ce_r + 10 * kd_r).backward()
        assert torch.equal(ce_r, ce) and torch.equal(kd_r, kd) and torch.equal(lr_r.grad, lr_c.grad)


# ------------------------------------------------------------------------------------------------
# SURVEY section 8(f) row N3: sibling losses on the same kernels
@pytest.mark.parametrize("red", ["mean", "sum", "none"])
def test_sibling_losses_vs_reference_fixture(U, golden_dir, red):
    fx = np.load(os.path.join(golden_dir, "sibling_losses.npz"))
    x0, t = torch.from_numpy(fx["x"]), torch.from_numpy(fx["t"]).cuda()
    y, mask = torch.from_numpy(fx["y"]).cuda(), torch.from_numpy(fx["mask"]).cuda()
    old_cl, alpha = int(fx["old_cl"][0]), float(fx["alpha"][0])
    runs = {
        "kd": lambda x: U.KnowledgeDistillationLoss(reduction=red, alpha=alpha)(x, t),
        "kd_mask": lambda x: U.KnowledgeDistillationLoss(reduction=red, alpha=alpha)(x, t, mask > 0),
        "mkd": lambda x: U.MaskKnowledgeDistillationLoss(reduction=red, alpha=alpha)(x, t),
        "mkd_mask": lambda x: U.MaskKnowledgeDistillationLoss(reduction=red, alpha=alpha)(x, t, mask),
        "mce": lambda x: U.MaskCrossEntropy(old_cl=old_cl, reduction=red)(x, y),
        "mce_old": lambda x: U.MaskCrossEntropy(old_cl=old_cl, reduction=red)(x, y, t),
    }
    y_before = y.clone()
    for tag, fn in runs.items():
        x = x0.cuda().requires_grad_(True)
        out = fn(x)
        want = torch.from_numpy(np.asarray(fx[f"{tag}_{red}_out"]))
        torch.testing.assert_close(out.detach().cpu().double(), want, rtol=1e-4, atol=1e-5, msg=lambda m: f"{tag}: {m}")
        w = torch.linspace(0.5, 1.5, out.numel(), dtype=torch.float64).reshape(out.shape) if out.dim() else None
        (out if w is None else (out * w.float().cuda()).sum()).backward()
        gw = torch.from_numpy(fx[f"{tag}_{red}_grad"])
        assert cos(x.grad, gw) > 1 - 1e-6, tag
        torch.testing.assert_close(x.grad.cpu().double(), gw, rtol=1e-3, atol=5e-6 * float(gw.abs().max()) + 1e-9,
                                   msg=lambda m: f"{tag} grad: {m}")
    assert torch.equal(y, y_before)  # MaskCrossEntropy leaves the caller's labels alone (unlike UNCE)


@pytest.mark.parametrize("shape,c_old", [((2, 21, 33, 35), 16), ((1, 17, 64, 64), 16), ((2, 151, 16, 20), 101)])
def test_sibling_losses_vs_oracle(U, shape, c_old):
    """Odd plane sizes (scalar path), many channels, NaN-free ties in the old model's argmax."""
    B, C, H, W = shape
    g = torch.Generator().manual_seed(9)
    x = torch.randn(B, C, H, W, generator=g) * 3
    t = torch.randn(B, c_old, H, W, generator=g) * 3
    t[:, :, 0] = 0.0                                    # ties: argmax must pick index 0
    y = torch.randint(0, C, (B, H, W), generator=g)
    y[:, -1] = 255
    mask = torch.randint(0, 2, (B, H, W), generator=g)
    for tag, ofn, mfn in [
        ("kd", lambda v: O.plain_kd(v, t.double(), 1.3, "mean", mask), lambda v: U.KnowledgeDistillationLoss(alpha=1.3)(v, t.cuda(), mask.cuda())),
        ("mkd", lambda v: O.mask_kd(v, t.double(), 1.3, "mean", mask), lambda v: U.MaskKnowledgeDistillationLoss(alpha=1.3)(v, t.cuda(), mask.cuda())),
        ("mce", lambda v: O.mask_ce(v, y, c_old, t.double(), 255, "mean"), lambda v: U.MaskCrossEntropy(old_cl=c_old)(v, y.cuda(), t.cuda())),
    ]:
        xr = x.double().requires_grad_(True)
        ref = ofn(xr)
        ref.backward()
        xc = x.cuda().requires_grad_(True)
        out = mfn(xc)
        out.backward()
        torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=5e-5, atol=5e-6, msg=lambda m: f"{tag}: {m}")
        assert cos(xc.grad, xr.grad) > 1 - 1e-6, tag


def test_raw_head_features_equal_att_map_features(U, golden_dir):
    """Row N2: the attention map of segmentation_module.py:86-94 cancels under the anchor normalisation, so the prep
    kernel may read the RAW head output.  Checker = the CPU oracle evaluated the reference's way (att_map applied to
    both models' features, fp64, autograd through att_map down to the raw head output); the CUDA path gets the raw
    features only: same loss (1e-3), same gradient with respect to the head output (cosine >= 0.999)."""
    fx, case, (B, h, w, H, W, C, C_old) = load_case(golden_dir, "voc15-5s_b2_corr")
    x_ref = case["f_n"].double().requires_grad_(True)
    A, Cst, la, lc, P, _ = O.pre_contrastive_pixel(O.att_map(x_ref), case["labels"], case["l_po"].double(),
                                                   O.att_map(case["f_o"].double()))
    ref = O.pixel_con_loss(A, Cst, la, lc, P)
    ref.backward()
    x = case["f_n"].cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(x, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
    loss = U.PixelConLossV2(temperature=0.07)(*tup)
    loss.backward()
    assert loss.item() == pytest.approx(ref.item(), rel=REL)
    assert cos(x.grad, x_ref.grad) >= COS
    # and the CUDA path fed with attended features agrees with itself on raw ones (the round-1 check)
    x2 = case["f_n"].cuda().requires_grad_(True)
    tup2 = U.pre_contrastive_pixel(O.att_map(x2), case["labels"].cuda(), l_po=case["l_po"].cuda(),
                                   f_o=O.att_map(case["f_o"].cuda()))
    loss2 = U.PixelConLossV2(temperature=0.07)(*tup2)
    loss2.backward()
    assert loss2.item() == pytest.approx(loss.item(), rel=1e-4) and cos(x2.grad, x.grad) > 1 - 1e-5


# ------------------------------------------------------------------------------------------------
# SURVEY section 8(f) row N3, second half: the self-contrast losses of utils/loss_new.py on the sweep kernels
@pytest.mark.parametrize("name", ["a", "b", "c"])
def test_selfcon_losses_vs_reference_fixture(U, golden_dir, name):
    """PixelConLoss (v1) and SupConLoss against the values and gradients of the UNMODIFIED reference classes
    (tests/golden/selfcon_losses.npz, fp64): loss 1e-3, gradient cosine 0.999 on the stored samples, gradient norm 1 %."""
    fx = np.load(os.path.join(golden_dir, "selfcon_losses.npz"))
    st = int(fx["stride"][0])
    n, n_cls, views = O.SELFCON_CASES[name]
    x, lab = O.selfcon_case(name)
    runs = []
    if views == 1:
        runs += [("%s_v1_t%g" % (name, tau), U.PixelConLoss(temperature=tau), True) for tau in (1.0, 0.5)]
    for mode in ("all", "one"):
        for use_lab in (True, False):
            runs.append(("%s_sup_%s_%s" % (name, mode, "lab" if use_lab else "simclr"),
                         U.SupConLoss(temperature=0.07, contrast_mode=mode), use_lab))
    for key, module, use_lab in runs:
        xr = x.float().cuda().requires_grad_(True)
        loss = module(xr, lab.cuda()) if use_lab else module(xr)
        loss.backward()
        want = float(fx[key + "_loss"][0])
        assert loss.item() == pytest.approx(want, rel=REL, abs=2e-6), key
        gs = xr.grad.double().cpu().reshape(-1)[::st]
        ref = torch.from_numpy(fx[key + "_gsample"])
        if float(ref.norm()) > 1e-12:
            assert cos(gs, ref) >= COS, key
            assert xr.grad.double().norm().item() == pytest.approx(float(fx[key + "_gnorm"][0]), rel=1e-2), key
        else:   # SimCLR with one view: no positives, zero loss and zero gradient
            assert float(xr.grad.abs().max()) == 0.0, key


def test_selfcon_losses_vs_oracle_on_pixel_to_pixel_rows(U):
    """The use the reference made of v1: PixelConLoss on the rows of the pixel-to-pixel prep (every pixel a unit-norm row,
    labels from the downsampled label map), ragged size (not a multiple of 128), narrow features, SupCon with 3 views."""
    case = O.synthetic_case(2, 17, 19, 272, 304, 21, 16)
    f_ref = case["f_n"].double().requires_grad_(True)
    out_ref, lab_ref = O.pixel_to_pixel(f_ref, case["labels"])
    ref = O.pixel_con_loss_v1(out_ref, lab_ref, 0.5)
    ref.backward()
    f = case["f_n"].cuda().requires_grad_(True)
    out, lab = U.pre_contrastive_pixel(f, case["labels"].cuda())
    loss = U.PixelConLoss(temperature=0.5)(out, lab)
    loss.backward()
    assert loss.item() == pytest.approx(ref.item(), rel=REL) and cos(f.grad, f_ref.grad) >= COS
    g = torch.Generator().manual_seed(5)
    x = torch.nn.functional.normalize(torch.randn(150, 3, 64, generator=g, dtype=torch.float64), dim=2)
    lab = torch.randint(0, 7, (150,), generator=g)
    for mode in ("all", "one"):
        xr = x.clone().requires_grad_(True)
        want = O.sup_con_loss(xr, lab, 0.1, mode, 0.07)
        want.backward()
        xc = x.float().cuda().requires_grad_(True)
        got = U.SupConLoss(temperature=0.1, contrast_mode=mode, base_temperature=0.07)(xc, lab.cuda())
        got.backward()
        assert got.item() == pytest.approx(want.item(), rel=REL) and cos(xc.grad, xr.grad) >= COS
    with pytest.raises(NotImplementedError):
        U.SupConLoss()(x.float().cuda(), mask=torch.eye(150).cuda())


@pytest.mark.parametrize("name", ["voc15-5s_b2_corr", "city13-6_b3"])
def test_bf16_feature_handoff(U, golden_dir, name):
    """Row N2, second half: a head that runs in bf16 hands its features over as bf16 NCHW; the prep kernel reads them
    as they are and the adjoint writes the bf16 gradient.  Checker = the CPU oracle (fp64) on the bf16-rounded
    features; the integer artefacts must not depend on the feature dtype at all; and the fp32 entry point fed with
    the same rounded values must produce the same operand tiles bit for bit."""
    fx, case, (B, h, w, H, W, C, C_old) = load_case(golden_dir, name)
    fn16, fo16 = case["f_n"].to(torch.bfloat16), case["f_o"].to(torch.bfloat16)
    x_ref = fn16.double().requires_grad_(True)
    A, Cst, la, lc, P, _ = O.pre_contrastive_pixel(x_ref, case["labels"], case["l_po"].double(), fo16.double())
    ref = O.pixel_con_loss(A, Cst, la, lc, P)
    ref.backward()
    x = fn16.cuda().requires_grad_(True)
    tup = U.pre_contrastive_pixel(x, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=fo16.cuda())
    assert tup[4].pack.bf16_feats
    loss = U.PixelConLossV2(temperature=0.07)(*tup)
    loss.backward()
    assert x.grad.dtype == torch.bfloat16 and x.grad.shape == x.shape
    assert loss.item() == pytest.approx(ref.item(), rel=REL)
    assert cos(x.grad.float(), x_ref.grad) >= COS
    assert torch.equal(tup[2].cpu().long(), la.long()) and torch.equal(tup[3].cpu().long(), lc.long())
    # same values through the fp32 entry point: identical rows and tiles, gradient equal up to the final bf16 rounding
    x32 = fn16.float().cuda().requires_grad_(True)
    tup32 = U.pre_contrastive_pixel(x32, case["labels"].cuda(), l_po=case["l_po"].cuda(), f_o=fo16.float().cuda())
    assert not tup32[4].pack.bf16_feats
    assert torch.equal(tup32[0], tup[0]) and torch.equal(tup32[1], tup[1])
    used = (tup[4].pack.n_c + 127) // 128
    assert torch.equal(tup32[4].pack.feat_tiles[:used], tup[4].pack.feat_tiles[:used])
    loss32 = U.PixelConLossV2(temperature=0.07)(*tup32)
    loss32.backward()
    assert loss32.item() == loss.item()
    assert torch.equal(x32.grad.to(torch.bfloat16), x.grad)
    # the sync-free module takes the same route
    x3 = fn16.cuda().requires_grad_(True)
    out = U.PixelContrastiveDistillation(temperature=0.07)(x3, case["labels"].cuda(), case["l_po"].cuda(), fo16.cuda())
    out.backward()
    assert x3.grad.dtype == torch.bfloat16
    assert out.item() == pytest.approx(loss.item(), rel=2e-6) and cos(x3.grad.float(), x.grad.float()) > 1 - 1e-5


# ------------------------------------------------------------------------------------------------
# SURVEY section 8(f) row N4: sync-free contrastive module, CUDA-graph capture of forward + backward
@pytest.mark.parametrize("name", ["tiny_b2", "voc15-5s_b3_512", "city13-6_b3", "voc15-5s_b2_corr"])
def test_sync_free_contrastive_matches_tuple_path(U, golden_dir, name):
    fx, case, (B, h, w, H, W, C, C_old) = load_case(golden_dir, name)
    dev = {k: v.cuda() for k, v in case.items()}
    f1 = dev["f_n"].clone().requires_grad_(True)
    ref = U.PixelConLossV2(temperature=0.07)(*U.pre_contrastive_pixel(f1, dev["labels"], l_po=dev["l_po"], f_o=dev["f_o"]))
    ref.backward()
    f2 = dev["f_n"].clone().requires_grad_(True)
    out = U.PixelContrastiveDistillation(temperature=0.07)(f2, dev["labels"], dev["l_po"], dev["f_o"])
    out.backward()
    assert out.item() == pytest.approx(ref.item(), rel=2e-6)          # same kernels, other split -> summation order
    assert out.item() == pytest.approx(float(fx["con"][1]), rel=REL)  # and the reference fixture
    assert cos(f2.grad, f1.grad) > 1 - 1e-6
    torch.testing.assert_close(f2.grad, f1.grad, rtol=1e-3, atol=1e-5 * float(f1.grad.abs().max()))


def test_sync_free_step_in_cuda_graph(U, golden_dir):
    """Capture contrastive + fused CE/KD forward and backward once, replay on new data: equal to the eager modules."""
    _, case_a, (B, h, w, H, W, C, C_old) = load_case(golden_dir, "voc15-5s_b3_512")
    case_b = O.synthetic_case(B, h, w, H, W, C, C_old, rank=1)
    con = U.PixelContrastiveDistillation(temperature=0.07)
    fused = U.FusedUnbiasedLosses(old_cl=C_old, alpha=1.0)
    st = {k: v.cuda().clone() for k, v in case_a.items()}
    st["f_n"].requires_grad_(True), st["logits_lr"].requires_grad_(True)

    def step():
        ce, kd = fused(st["logits_lr"], st["l_po"], st["labels"])
        loss = ce + con(st["f_n"], st["labels"], st["l_po"], st["f_o"]) / 100 + 10 * kd
        loss.backward()
        return loss

    if hasattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch"):
        torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)   # warm-up and capture streams differ
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            st["f_n"].grad = st["logits_lr"].grad = None
            step()
    torch.cuda.current_stream().wait_stream(side)
    st["f_n"].grad = st["logits_lr"].grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss_s = step()
    for case in (case_b, case_a):
        with torch.no_grad():
            for k in ("f_n", "f_o", "l_po", "logits_lr", "labels"):
                st[k].copy_(case[k].cuda())
        graph.replay()
        torch.cuda.synchronize()
        # eager reference through the drop-in modules on the same data
        f = case["f_n"].cuda().requires_grad_(True)
        lr = case["logits_lr"].cuda().requires_grad_(True)
        lab = case["labels"].cuda()
        ce, kd = U.FusedUnbiasedLosses(old_cl=C_old, alpha=1.0)(lr, case["l_po"].cuda(), lab.clone())
        tup = U.pre_contrastive_pixel(f, lab, l_po=case["l_po"].cuda(), f_o=case["f_o"].cuda())
        ref = ce + U.PixelConLossV2(temperature=0.07)(*tup) / 100 + 10 * kd
        ref.backward()
        assert loss_s.item() == pytest.approx(ref.item(), rel=1e-5)
        assert cos(st["f_n"].grad, f.grad) > 1 - 1e-6 and cos(st["logits_lr"].grad, lr.grad) > 1 - 1e-6

