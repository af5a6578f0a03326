"""Device time of the two passes that the low-res output mode takes off the full-resolution logits:

  step-0 loss, forward + backward to the low-res logits, three forms:
    (a) interpolate_bilinear + F.cross_entropy(reduction='none').mean()       what a trainer runs today
    (b) interpolate_bilinear + UnbiasedCrossEntropy(old_cl=0, 'none').mean()  the drop-in module
    (c) FusedUnbiasedLosses(0)(lr, None, labels)                              the CE-only fused form
  prediction:
    (a) interpolate_bilinear(lr, size).argmax(1)
    (b) predict_bilinear(lr, size)

The forms alternate in one process after a warm-up of each.  Before every timed call a 256 MB buffer is overwritten,
so no call finds its inputs in the 126 MB L2; CUDA events bracket the call alone.  Reported per form: the median
over the repeats of the per-repeat median call time, and the spread (min - max) of those medians.  The outputs of the
forms are compared on the timed inputs (loss rel. error, gradient rel. L2, prediction equality).

    python scripts/bench_lowres_only.py [--repeats 7] [--iters 20] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import ucd_b200 as U  # noqa: E402

# step 0 of each protocol: only the base classes (+ background) exist
LOSS_SHAPES = {
    "voc15-5_step0": dict(B=24, C=16, h=32, w=32, H=512, W=512),
    "ade100-50_step0": dict(B=3, C=101, h=32, w=32, H=512, W=512),
    "city13-6_step0": dict(B=3, C=14, h=32, w=64, H=512, W=1024),
}
# validation / test: every class of the protocol
PRED_SHAPES = {
    "voc_c21": dict(B=24, C=21, h=32, w=32, H=512, W=512),
    "ade_c151": dict(B=3, C=151, h=32, w=32, H=512, W=512),
    "city_c20": dict(B=3, C=20, h=32, w=64, H=512, W=1024),
}


def inputs(s, seed):
    g = torch.Generator().manual_seed(seed)
    lr = torch.randn(s["B"], s["C"], s["h"], s["w"], generator=g) * 3
    cls = torch.randint(0, s["C"], (s["B"], 1, s["h"] // 4, s["w"] // 4), generator=g).float()
    y = F.interpolate(cls, size=(s["H"], s["W"]), mode="nearest")[:, 0].long()
    y[:, :s["H"] // 25] = 255
    return lr.cuda(), y.cuda()


def loss_forms(s):
    size = (s["H"], s["W"])
    unce = U.UnbiasedCrossEntropy(old_cl=0, ignore_index=255, reduction="none")
    fused = U.FusedUnbiasedLosses(0, ignore_index=255)
    return {
        "interp+F.cross_entropy": lambda x, y: F.cross_entropy(U.interpolate_bilinear(x, size), y, ignore_index=255,
                                                               reduction="none").mean(),
        "interp+UnbiasedCE(0)": lambda x, y: unce(U.interpolate_bilinear(x, size), y).mean(),
        "fused_ce_only": lambda x, y: fused(x, None, y)[0],
    }


def pred_forms(s):
    size = (s["H"], s["W"])
    return {
        "interp.argmax": lambda x: U.interpolate_bilinear(x, size).argmax(1),
        "predict_bilinear": lambda x: U.predict_bilinear(x, size),
    }


def run_loss(fn, lr, y):
    x = lr.detach().requires_grad_(True)
    loss = fn(x, y)
    loss.backward()
    return loss.detach(), x.grad


def time_forms(calls, repeats, iters, flush):
    """calls: {name: zero-argument callable}.  Returns {name: [per-repeat median ms]}."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(iters)]
    for fn in calls.values():   # warm-up
        fn()
        fn()
    out = {k: [] for k in calls}
    for _ in range(repeats):
        for name, fn in calls.items():
            for a, b in ev:
                flush.zero_()
                a.record()
                fn()
                b.record()
            torch.cuda.synchronize()
            out[name].append(statistics.median(a.elapsed_time(b) for a, b in ev))
    return out


def summary(ms):
    return dict(median=round(statistics.median(ms), 4), min=round(min(ms), 4), max=round(max(ms), 4))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_lowres_only.py: needs a CUDA device")
    torch.cuda.set_device(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device="cuda")
    res = dict(gpu=gpu, cache="256 MB overwritten before every timed call", loss={}, prediction={})
    for name, s in LOSS_SHAPES.items():
        lr, y = inputs(s, 1)
        forms = loss_forms(s)
        outs = {k: run_loss(fn, lr, y.clone()) for k, fn in forms.items()}
        ref_l, ref_g = outs["interp+F.cross_entropy"]
        check = {k: dict(loss_rel=abs(float(l) - float(ref_l)) / abs(float(ref_l)),
                         grad_rel_l2=float((g - ref_g).double().norm() / ref_g.double().norm()))
                 for k, (l, g) in outs.items() if k != "interp+F.cross_entropy"}
        t = time_forms({k: (lambda fn=fn: run_loss(fn, lr, y)) for k, fn in forms.items()}, args.repeats, args.iters,
                       flush)
        res["loss"][name] = dict(shape=s, ms={k: summary(v) for k, v in t.items()}, vs_cross_entropy=check)
        print(name, {k: res["loss"][name]["ms"][k]["median"] for k in t}, flush=True)
        del lr, y, outs, ref_g
        torch.cuda.empty_cache()
    for name, s in PRED_SHAPES.items():
        lr, _ = inputs(s, 2)
        forms = pred_forms(s)
        same = bool(torch.equal(forms["interp.argmax"](lr), forms["predict_bilinear"](lr)))
        t = time_forms({k: (lambda fn=fn: fn(lr)) for k, fn in forms.items()}, args.repeats, args.iters, flush)
        res["prediction"][name] = dict(shape=s, ms={k: summary(v) for k, v in t.items()}, equal=same,
                                       full_res_logit_bytes=4 * s["B"] * s["C"] * s["H"] * s["W"])
        print(name, {k: res["prediction"][name]["ms"][k]["median"] for k in t}, "equal", same, flush=True)
        del lr
        torch.cuda.empty_cache()
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
