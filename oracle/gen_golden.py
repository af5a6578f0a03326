"""Generate tests/golden/*.npz by running the UNMODIFIED reference (utils/loss.py imported from
/root/reference) on seeded synthetic inputs.  TEST INFRASTRUCTURE ONLY.

Run in the build container (the reference tree does not exist on the GPU box):

    python oracle/gen_golden.py            # rewrites tests/golden/

The fixtures pin the oracle (tests/test_oracle.py) and, through it and directly, the CUDA path
(tests/test_gpu_parity.py).  Inputs are regenerated from seeds by ``oracle.ucd_oracle.synthetic_case``;
each fixture stores input checksums so generator drift is detected instead of silently accepted.
"""
import os
import sys
import warnings

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("UCD_REFERENCE", "/root/reference")
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
warnings.filterwarnings("ignore")

from oracle.ucd_oracle import (LABEL_DOWNSAMPLE_SIZES, label_downsample_maps, label_map_digest,  # noqa: E402
                               synthetic_case)
from utils.loss import (PixelConLossV2, UnbiasedCrossEntropy,  # noqa: E402  (the reference)
                        UnbiasedKnowledgeDistillationLoss, pre_contrastive_pixel)

OUT = os.path.join(ROOT, "tests", "golden")
STRIDE = 997  # gradient sampling stride (prime)

CASES = {
    # name: (B, h, w, H, W, C, C_old, correlated)
    "voc15-5_b2_513": (2, 33, 33, 513, 513, 21, 16, False),     # BASELINE config 1 / Appendix B row 1
    "voc15-5s_b3_512": (3, 32, 32, 512, 512, 17, 16, False),    # per-GPU slice of config 2
    "city13-6_b3": (3, 32, 64, 512, 1024, 20, 14, False),       # per-GPU slice of config 4
    "voc15-5s_b2_corr": (2, 32, 32, 512, 512, 17, 16, True),    # class-correlated features
    "tiny_b2": (2, 8, 8, 128, 128, 6, 4, False),                # full tensors stored
}


def run_reference(case, dtype):
    d = {k: (v.to(dtype) if v.is_floating_point() else v.clone()) for k, v in case.items()}
    f_n = d["f_n"].requires_grad_(True)
    lr = d["logits_lr"].requires_grad_(True)
    labels = d["labels"]
    H, W = labels.shape[-2:]
    c_old = d["l_po"].shape[1]
    outputs = F.interpolate(lr, size=(H, W), mode="bilinear", align_corners=False)
    outputs_old = F.interpolate(d["l_po"], size=(H, W), mode="bilinear", align_corners=False)
    tup = pre_contrastive_pixel(f_n, labels, l_po=d["l_po"], f_o=d["f_o"])
    A, Cst, la, lc, P = tup
    con = PixelConLossV2(temperature=0.07)(A, Cst, la, lc, P)
    lab_ce = labels.clone()
    ce_px = UnbiasedCrossEntropy(old_cl=c_old, reduction="none", ignore_index=255)(outputs, lab_ce)
    ce = ce_px.mean()
    kd = UnbiasedKnowledgeDistillationLoss(alpha=1.0)(outputs, outputs_old)
    (g_fn,) = torch.autograd.grad(con, f_n, retain_graph=True)
    (g_lr,) = torch.autograd.grad(ce + 10 * kd, lr)
    # the v2 branch leaves the mixed labels in label_n; the plain branch returns the clamped map
    _, lab_flat = pre_contrastive_pixel(d["f_n"], labels)
    return dict(A=A.detach(), Cst=Cst, la=la, lc=lc, P=P, con=con.detach(), ce=ce.detach(), kd=kd.detach(),
                ce_px=ce_px.detach(), g_fn=g_fn, g_lr=g_lr, lab_ce=lab_ce, label_n=lab_flat,
                outputs=outputs.detach())


def gen_sibling():
    """KnowledgeDistillationLoss, MaskKnowledgeDistillationLoss, MaskCrossEntropy (utils/loss.py) on stored inputs."""
    from utils.loss import KnowledgeDistillationLoss, MaskCrossEntropy, MaskKnowledgeDistillationLoss
    g = torch.Generator().manual_seed(4242)
    B, C, C_old, H, W = 2, 7, 4, 20, 24
    x = (torch.randn(B, C, H, W, generator=g) * 2.0).float()
    t = (torch.randn(B, C_old, H, W, generator=g) * 2.0).float()
    y = torch.randint(0, C, (B, H, W), generator=g)
    y[:, :2] = 255
    mask = torch.randint(0, 3, (B, H, W), generator=g)
    fx = dict(x=x.numpy(), t=t.numpy(), y=y.numpy().astype(np.int64), mask=mask.numpy().astype(np.int64),
              old_cl=np.array([C_old]), alpha=np.array([0.7]))

    def run(tag, fn):
        xd = x.double().requires_grad_(True)
        out = fn(xd)
        w = torch.linspace(0.5, 1.5, out.numel(), dtype=torch.float64).reshape(out.shape) if out.dim() else None
        (out if w is None else (out * w).sum()).backward()
        fx[tag + "_out"] = out.detach().numpy()
        fx[tag + "_grad"] = xd.grad.numpy()

    for red in ("mean", "sum", "none"):
        run("kd_" + red, lambda xd: KnowledgeDistillationLoss(reduction=red, alpha=0.7)(xd, t.double()))
        run("kd_mask_" + red, lambda xd: KnowledgeDistillationLoss(reduction=red, alpha=0.7)(xd, t.double(), (mask > 0)))
        run("mkd_" + red, lambda xd: MaskKnowledgeDistillationLoss(reduction=red, alpha=0.7)(xd, t.double()))
        run("mkd_mask_" + red, lambda xd: MaskKnowledgeDistillationLoss(reduction=red, alpha=0.7)(xd, t.double(), mask))
        run("mce_" + red, lambda xd: MaskCrossEntropy(old_cl=C_old, reduction=red)(xd, y.clone()))
        run("mce_old_" + red, lambda xd: MaskCrossEntropy(old_cl=C_old, reduction=red)(xd, y.clone(), t.double()))
    np.savez_compressed(os.path.join(OUT, "sibling_losses.npz"), **fx)
    print("sibling_losses:", {k: float(v) for k, v in fx.items() if k.endswith("_out") and v.ndim == 0})


def gen_att_map():
    """segmentation_module.py:86-94 `att_map` (the module itself needs inplace_abn, which is not installed: the method is
    lifted out of the reference source with ast and executed unmodified)."""
    import ast
    src = open(os.path.join(REF, "segmentation_module.py")).read()
    fn = next(n for n in ast.walk(ast.parse(src)) if isinstance(n, ast.FunctionDef) and n.name == "att_map")
    ns = {"torch": torch}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), "segmentation_module.py", "exec"), ns)
    g = torch.Generator().manual_seed(99)
    x = torch.randn(3, 16, 6, 5, generator=g, dtype=torch.float64)
    y = ns["att_map"](None, x.clone())
    np.savez_compressed(os.path.join(OUT, "att_map.npz"), x=x.numpy(), y=y.numpy())
    print("att_map:", float(y.abs().sum()))


def gen_p2p():
    """The pixel-to-pixel branches of pre_contrastive_pixel (utils/loss.py:278-289: no old-model logits) on a small
    seeded case: outputs, labels and the gradient of a fixed linear functional, single (f_o None) and double."""
    case = synthetic_case(2, 5, 7, 80, 112, 21, 16)
    fx = dict(shape=np.array([2, 5, 7, 80, 112, 21, 16]))
    w = torch.randn(2 * 2 * 5 * 7, 1, 256, generator=torch.Generator().manual_seed(77), dtype=torch.float64)
    fx["w"] = w.numpy()
    for tag, f_o in (("single", None), ("double", case["f_o"].double())):
        f_n = case["f_n"].double().requires_grad_(True)
        out, lab = pre_contrastive_pixel(f_n, case["labels"], l_po=None, f_o=f_o)
        (out * w[:out.shape[0]]).sum().backward()
        fx[tag + "_out"], fx[tag + "_lab"], fx[tag + "_grad"] = out.detach().numpy(), lab.numpy(), f_n.grad.numpy()
    np.savez_compressed(os.path.join(OUT, "pixel_to_pixel.npz"), **fx)
    print("pixel_to_pixel", fx["single_out"].shape, fx["double_out"].shape, np.unique(fx["single_lab"]))


def gen_selfcon():
    """PixelConLoss (v1) and SupConLoss of utils/loss_new.py on the seeded cases of oracle.ucd_oracle.selfcon_case: loss
    values, gradient norms and strided gradient samples of the UNMODIFIED reference classes, fp64."""
    from utils.loss_new import PixelConLoss, SupConLoss
    from oracle.ucd_oracle import SELFCON_CASES, selfcon_case
    fx = {"stride": np.array([13])}

    def put(key, loss, grad):
        fx[key + "_loss"] = np.array([loss.item()])
        fx[key + "_gnorm"] = np.array([grad.norm().item()])
        fx[key + "_gsample"] = grad.reshape(-1)[::13].numpy()

    for name, (n, n_cls, views) in SELFCON_CASES.items():
        x, lab = selfcon_case(name)
        fx[name + "_in_sums"] = np.array([x.sum().item(), float(lab.sum())])
        if views == 1:
            for tau in (1.0, 0.5):
                xr = x.clone().requires_grad_(True)
                loss = PixelConLoss(temperature=tau)(xr, lab)
                loss.backward()
                put("%s_v1_t%g" % (name, tau), loss, xr.grad)
        for mode in ("all", "one"):
            for use_lab in (True, False):
                xr = x.clone().requires_grad_(True)
                loss = SupConLoss(temperature=0.07, contrast_mode=mode)(xr, lab if use_lab else None)
                loss.backward()
                put("%s_sup_%s_%s" % (name, mode, "lab" if use_lab else "simclr"), loss, xr.grad)
    np.savez_compressed(os.path.join(OUT, "selfcon_losses.npz"), **fx)
    print("selfcon_losses:", {k: float(v[0]) for k, v in fx.items() if k.endswith("_loss")})


def main():
    os.makedirs(OUT, exist_ok=True)
    if len(sys.argv) > 1 and sys.argv[1] == "selfcon":
        return gen_selfcon()
    gen_selfcon()
    if len(sys.argv) > 1 and sys.argv[1] == "p2p":
        return gen_p2p()
    gen_p2p()
    if len(sys.argv) > 1 and sys.argv[1] == "att_map":
        return gen_att_map()
    gen_att_map()
    if len(sys.argv) > 1 and sys.argv[1] == "sibling":
        return gen_sibling()
    gen_sibling()
    for name, (B, h, w, H, W, C, C_old, corr) in CASES.items():
        case = synthetic_case(B, h, w, H, W, C, C_old, correlated=corr)
        r32 = run_reference(case, torch.float32)
        r64 = run_reference(case, torch.float64)
        fx = dict(
            shape=np.array([B, h, w, H, W, C, C_old, int(corr)]),
            in_sums=np.array([case[k].double().sum().item() for k in ("f_n", "f_o", "l_po", "logits_lr", "labels")]),
            la=r32["la"].numpy().astype(np.int8), lc=r32["lc"].numpy().astype(np.int8),
            label_n=r32["label_n"].numpy().astype(np.int8).reshape(B, h, w),
            lab_ce_changed=np.array([(r32["lab_ce"] != case["labels"]).sum().item()]),
            p_ones=np.array([(r32["P"] == 1).sum().item()]),
            p_sum=np.array([r64["P"].sum().item()]),
            con=np.array([r32["con"].item(), r64["con"].item()]),
            ce=np.array([r32["ce"].item(), r64["ce"].item()]),
            kd=np.array([r32["kd"].item(), r64["kd"].item()]),
            g_fn_norm=np.array([r32["g_fn"].norm().item(), r64["g_fn"].norm().item()]),
            g_lr_norm=np.array([r32["g_lr"].norm().item(), r64["g_lr"].norm().item()]),
            g_fn_sample=r64["g_fn"].reshape(-1)[::STRIDE].numpy(),
            g_lr_sample=r64["g_lr"].reshape(-1)[::STRIDE].numpy(),
            ce_px_sample=r64["ce_px"].reshape(-1)[::STRIDE].numpy(),
            out_sample=r32["outputs"].reshape(-1)[::STRIDE].numpy(),
            stride=np.array([STRIDE]),
        )
        if name.startswith("tiny"):
            fx.update(full_A=r64["A"].numpy(), full_Cst=r64["Cst"].numpy(), full_P=r64["P"].numpy(),
                      full_g_fn=r64["g_fn"].numpy(), full_g_lr=r64["g_lr"].numpy())
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **fx)
        print(f"{name}: N_a={len(fx['la'])} N_c={len(fx['lc'])} sum_la={fx['la'].astype(int).sum()} "
              f"sum_lc={fx['lc'].astype(int).sum()} P1={fx['p_ones'][0]} con={fx['con']} ce={fx['ce']} kd={fx['kd']} "
              f"|g_fn|={fx['g_fn_norm'][0]:.6g} |g_lr|={fx['g_lr_norm'][0]:.6g}")

    # label-downsample vectors: the reference's own resize+cast+clamp on assorted label maps.  The maps themselves are
    # regenerated from their seed by the tests (stored, they would take 1.7 MB); the fixture keeps their digests.
    maps, lab_fx = label_downsample_maps(), {}
    for i, (H, W, h, w) in enumerate(LABEL_DOWNSAMPLE_SIZES):
        for n in ("rand%d" % i, "block%d" % i):
            _, flat = pre_contrastive_pixel(torch.zeros(2, 4, h, w), torch.from_numpy(maps[n].astype(np.int64)))
            lab_fx[n + "_in_sha256"] = np.array(label_map_digest(maps[n]))
            lab_fx[n + "_out"] = flat.numpy().astype(np.int8).reshape(2, h, w)
    np.savez_compressed(os.path.join(OUT, "label_downsample.npz"), **lab_fx)
    print("label_downsample: ", len(lab_fx) // 2, "maps")


if __name__ == "__main__":
    main()
