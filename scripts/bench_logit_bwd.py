"""Device time of the logit backward of the drop-in step, two ways, at the bench.py workload shapes:

  (a) two-step   ucd_unce_unkd_bwd (dx [B,C,H,W] written) + ucd_upsample_bilinear_bwd (dx read back)
  (b) fused      ucd_unce_unkd_bwd_lowres (the adjoint folded in: dx never written)

Both run on the same saved statistics (from ucd_unce_fwd / ucd_kd_fwd), alternately in one process, over input sets
that rotate so that the working set exceeds the 126 MB L2.  Reported: the median of the repeats and their spread (min
- max), and the rate on the algorithmic bytes of (b): 4C + 4C_old + 24 bytes per full-res pixel (x, t, labels int64,
lse_all, the per-pixel loss plane, lse_bkg and lse_t), against a device-to-device copy measured in the same process.

    python scripts/bench_logit_bwd.py [--workloads voc,ade,city] [--repeats 7] [--iters 20] [--out FILE]
    python scripts/bench_logit_bwd.py --tune       # debug library: sweep the knobs UCD_LRB_VARIANT / UCD_LRB_ROWS
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

from bench import WORKLOADS, gen  # noqa: E402
from ucd_b200 import _lib  # noqa: E402
from ucd_b200._lib import check, ptr  # noqa: E402


def make_set(wl, seed, L, dev):
    B, C, C_old, h, w, H, W = (wl[k] for k in ("B", "C", "C_old", "h", "w", "H", "W"))
    HW = H * W
    st = torch.cuda.current_stream().cuda_stream
    lr = gen(4 + seed, B, C, h, w, scale=3.0).to(dev)
    lpo = gen(3 + seed, B, C_old, h, w, scale=3.0).to(dev)
    x = torch.empty(B, C, H, W, device=dev)
    t = torch.empty(B, C_old, H, W, device=dev)
    check(L.ucd_upsample_bilinear_fwd(ptr(lr), ptr(x), B * C, h, w, H, W, st))
    check(L.ucd_upsample_bilinear_fwd(ptr(lpo), ptr(t), B * C_old, h, w, H, W, st))
    y = torch.zeros(B, H, W, dtype=torch.int64)
    y[:, H // 5:3 * H // 5, W // 5:3 * W // 5] = C_old
    y[:, 3 * H // 5:4 * H // 5, W // 10:2 * W // 5] = C - 1
    y[:, :H // 25, :] = 255
    y = y.to(dev)
    f32 = dict(device=dev, dtype=torch.float32)
    s = dict(x=x, t=t, y=y, loss_px=torch.empty(B, H, W, **f32), lse=torch.empty(B, H, W, **f32),
             stats=torch.empty(2, **f32), kstats=torch.empty(1, **f32), lse3=torch.empty(3, B, H, W, **f32),
             scratch=torch.empty(L.ucd_reduce_scratch_floats(), **f32), g=torch.ones(1, **f32),
             dx=torch.empty(B, C, H, W, **f32), d_a=torch.empty(B, C, h, w, **f32), d_b=torch.empty(B, C, h, w, **f32))
    check(L.ucd_unce_fwd(ptr(x), ptr(y), ptr(s["loss_px"]), ptr(s["lse"]), None, ptr(s["stats"]), ptr(s["scratch"]),
                         B, C, C_old, HW, 255, st))
    check(L.ucd_kd_fwd(ptr(x), ptr(t), None, 1.0, None, ptr(s["kstats"]), ptr(s["lse3"]), ptr(s["scratch"]), B, C,
                       C_old, HW, 0, -1.0 / (B * HW), st))
    return s


def call_two_step(L, s, wl):
    B, C, C_old, h, w, H, W = (wl[k] for k in ("B", "C", "C_old", "h", "w", "H", "W"))
    st = torch.cuda.current_stream().cuda_stream
    check(L.ucd_unce_unkd_bwd(ptr(s["x"]), ptr(s["y"]), ptr(s["lse"]), ptr(s["loss_px"]), None, ptr(s["g"]), 1.0 / (B * H * W),
                              ptr(s["stats"]), 0, C_old, 255, ptr(s["t"]), None, 1.0, ptr(s["lse3"]), None, ptr(s["g"]),
                              10.0 / (B * H * W), 0, ptr(s["dx"]), 0, B, C, C_old, H * W, st), "unce_unkd_bwd")
    check(L.ucd_upsample_bilinear_bwd(ptr(s["dx"]), ptr(s["d_a"]), B * C, h, w, H, W, st), "upsample_bilinear_bwd")


def call_fused(L, s, wl):
    B, C, C_old, h, w, H, W = (wl[k] for k in ("B", "C", "C_old", "h", "w", "H", "W"))
    st = torch.cuda.current_stream().cuda_stream
    check(L.ucd_unce_unkd_bwd_lowres(ptr(s["x"]), ptr(s["y"]), ptr(s["lse"]), ptr(s["loss_px"]), None, ptr(s["g"]),
                                     1.0 / (B * H * W), ptr(s["stats"]), 0, C_old, 255, ptr(s["t"]), None, 1.0,
                                     ptr(s["lse3"]), None, ptr(s["g"]), 10.0 / (B * H * W), 0, ptr(s["d_b"]), B, C,
                                     C_old, h, w, H, W, st), "unce_unkd_bwd_lowres")


def timed(fn, sets, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        fn(sets[i % len(sets)])
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


def copy_gbs(dev, iters=20):
    src = torch.empty(512 * 2 ** 20, device=dev, dtype=torch.uint8)
    dst = torch.empty_like(src)
    dst.copy_(src)
    ms = timed(lambda _: dst.copy_(src), [None], iters)
    return 2 * src.numel() / (ms * 1e-3) / 1e9


def bench(L, names, repeats, iters, dev):
    res = {}
    copy = copy_gbs(dev)
    for name in names:
        wl = WORKLOADS[name]
        npx = wl["B"] * wl["H"] * wl["W"]
        per_set = npx * (4 * wl["C"] * 2 + 4 * wl["C_old"] + 24)
        sets = [make_set(wl, 10 * k, L, dev) for k in range(max(2, -(-2 * 126 * 2 ** 20 // per_set)))]
        for s in sets:          # warm-up of both variants on every set
            call_two_step(L, s, wl)
            call_fused(L, s, wl)
        torch.cuda.synchronize()
        diff = (sets[0]["d_a"] - sets[0]["d_b"]).double().norm() / sets[0]["d_a"].double().norm()
        ta, tb = [], []
        for _ in range(repeats):
            ta.append(timed(lambda s: call_two_step(L, s, wl), sets, iters))
            tb.append(timed(lambda s: call_fused(L, s, wl), sets, iters))
        alg = npx * (4 * wl["C"] + 4 * wl["C_old"] + 24)
        mb = statistics.median(tb)
        res[name] = dict(shape=[wl[k] for k in ("B", "C", "C_old", "h", "w", "H", "W")], input_sets=len(sets),
                         two_step_ms=dict(median=round(statistics.median(ta), 4), min=round(min(ta), 4), max=round(max(ta), 4)),
                         fused_ms=dict(median=round(mb, 4), min=round(min(tb), 4), max=round(max(tb), 4)),
                         alg_bytes=alg, fused_gbs=round(alg / (mb * 1e-3) / 1e9, 1),
                         fused_frac_of_copy=round(alg / (mb * 1e-3) / 1e9 / copy, 3), rel_l2_fused_vs_two_step=float(diff))
        del sets
        torch.cuda.empty_cache()
    return dict(copy_gbs=round(copy, 1), workloads=res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="voc,ade,city")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--tune", action="store_true")
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_logit_bwd.py: needs a CUDA device")
    dev = torch.device("cuda", 0)
    names = args.workloads.split(",")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    out = dict(gpu=gpu)
    if args.tune:
        L = _lib.debug_lib()
        out["tune"] = {}
        for variant in ("0", "1", "2", "3"):
            for rows in ("", "1", "2", "4", "8"):
                os.environ["UCD_LRB_VARIANT"] = variant
                os.environ["UCD_LRB_ROWS"] = rows
                for name in names:
                    r = bench(L, [name], 3, args.iters, dev)["workloads"][name]
                    key = "%s variant=%s rows=%s" % (name, variant, rows or "auto")
                    out["tune"][key] = r["fused_ms"]["median"]
                    print(key, r["fused_ms"], flush=True)
    else:
        out.update(bench(_lib.lib(), names, args.repeats, args.iters, dev))
    print(json.dumps(out, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
