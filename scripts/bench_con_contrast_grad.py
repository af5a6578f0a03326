"""Device time of PixelConLossV2's compat path (plain dense tensors) forward + backward, with and without the contrast
gradient (``contrast_grad=True``: ucd_con_contrast_grad, the transposed third sweep), and of fp32 torch autograd of the
reference formula (ucd_oracle.pixel_con_loss) where its dense N_a x N_c temporaries fit.

Operands: the anchors, contrast columns, labels and joint probability of the bench generator (bench.py's VOC workload,
B = 24, and two smaller batches), taken from pre_contrastive_pixel and passed as plain tensors; P None and the dense P.
The forms alternate in one process after a warm-up of each; before every timed call a 256 MB buffer is overwritten,
so no call finds its inputs in the 126 MB L2; CUDA events bracket the call alone.  Reported per form: the median over
the repeats of the per-repeat median call time and the spread (min - max) of those medians.  The contrast sweep alone
is timed by calling the entry point on the forward's workspace; its algorithmic rate counts 4 D = 1024 flop per pair
(S recomputed and H A) against the burst bf16 peak of BASELINE.md.

    python scripts/bench_con_contrast_grad.py [--repeats 5] [--iters 10] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import ucd_b200 as U  # noqa: E402
from oracle import ucd_oracle as O  # noqa: E402
from ucd_b200._lib import check, lib, ptr  # noqa: E402

BURST_BF16_TFLOPS = 1691.9      # BASELINE.md section 2: measured bf16 dense matmul, burst
SIZES = {"voc_b24": 24, "voc_b8": 8, "voc_b2": 2}     # batch of the VOC workload: ~23.4k x 41.1k, ~8k x 14k, ~2k x 3.6k
TAU = 0.07
REF_MAX_PAIRS = 120e6           # fp32 autograd of the dense reference: ~10 live [N_a, N_c] temporaries


def operands(B):
    s = dict(h=32, w=32, H=512, W=512, C=17, C_old=16)
    case = O.synthetic_case(B, s["h"], s["w"], s["H"], s["W"], s["C"], s["C_old"])
    tup = U.pre_contrastive_pixel(case["f_n"].cuda(), case["labels"].cuda(), l_po=case["l_po"].cuda(),
                                  f_o=case["f_o"].cuda(), max_label=20)
    A = tup[0].detach().clone()
    C = tup[1].detach().clone()
    return A, C, tup[2].long().clone(), tup[3].long().clone(), tup[4].dense()


def run(con, A, C, la, lc, P, c_grad):
    a = A.detach().requires_grad_(True)
    c = C.detach().requires_grad_(c_grad)
    out = con(a, c, la, lc, P)
    out.backward()
    return out.detach(), a.grad, c.grad


def run_ref(A, C, la, lc, P):
    a = A.detach().requires_grad_(True)
    c = C.detach().requires_grad_(True)
    out = O.pixel_con_loss(a, c, la, lc, P, TAU)   # self pair: anchor i <-> column i (N_a <= N_c)
    out.backward()
    return out.detach(), a.grad, c.grad


def sweep_only(A, C, la, lc, P):
    """A zero-argument callable running ucd_con_contrast_grad alone on a finished forward's workspace."""
    L = lib()
    n_a, n_c = A.shape[0], C.shape[0]
    rt, ct = -(-n_a // 128), -(-n_c // 128)
    bf = dict(device="cuda", dtype=torch.bfloat16)
    rfeat, cfeat = torch.empty(rt, 32, 128, 8, **bf), torch.empty(ct, 32, 128, 8, **bf)
    rlab = torch.empty(rt, 128, device="cuda", dtype=torch.int32)
    clab = torch.empty(ct, 128, device="cuda", dtype=torch.int32)
    la32, lc32 = la.int().contiguous(), lc.int().contiguous()
    check(L.ucd_con_pack_rows(ptr(A), ptr(la32), n_a, ptr(rfeat), ptr(rlab), rt, None), "pack")
    check(L.ucd_con_pack_rows(ptr(C), ptr(lc32), n_c, ptr(cfeat), ptr(clab), ct, None), "pack")
    rr = torch.empty(rt, 2, device="cuda", dtype=torch.int32)
    cr = torch.empty(ct, 2, device="cuda", dtype=torch.int32)
    check(L.ucd_con_tile_ranges(ptr(rlab), rt, None, ptr(rr), None), "ranges")
    check(L.ucd_con_tile_ranges(ptr(clab), ct, None, ptr(cr), None), "ranges")
    counts = torch.tensor([[n_c, 0]], device="cuda", dtype=torch.int32)
    n_rows = torch.tensor([n_a], device="cuda", dtype=torch.int32)
    p_mode, ldp = (0, 0) if P is None else (2, n_c)
    inv_tau = float(np.float32(1 / TAU))
    ws_bytes = L.ucd_con_contrast_grad_workspace_bytes(rt, ct, 0)
    ws = torch.empty(ws_bytes, device="cuda", dtype=torch.uint8)
    out = torch.empty(3, device="cuda")
    cu = torch.empty(ct * 128, 256, device="cuda")
    check(L.ucd_con_fwd(ptr(cfeat), None, ptr(clab), ptr(counts), 1, ct, 0, -1, 0, ptr(rfeat), None, ptr(rlab),
                        ptr(n_rows), ptr(cr), ptr(rr), 0, None, p_mode, 16, ptr(P), ldp, inv_tau, 0, ptr(out), None,
                        ptr(ws), ws_bytes, rt, 0, None), "con_fwd")

    def call():
        check(L.ucd_con_contrast_grad(ptr(cfeat), ptr(clab), ptr(counts), 1, ct, 0, ptr(rfeat), ptr(rlab), ptr(n_rows),
                                      ptr(cr), ptr(rr), 0, p_mode, ptr(P), ldp, inv_tau, ptr(cu), ptr(ws), ws_bytes,
                                      rt, 0, None), "con_contrast_grad")
    return call


def time_forms(calls, repeats, iters, flush):
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


def cos(a, b):
    a, b = a.double().reshape(-1), b.double().reshape(-1)
    return float(a @ b / (a.norm() * b.norm()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_con_contrast_grad.py: needs a CUDA device")
    torch.cuda.set_device(0)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device="cuda")
    res = dict(gpu=gpu, cache="256 MB overwritten before every timed call", tau=TAU,
               flop_per_pair=4 * 256, burst_bf16_tflops=BURST_BF16_TFLOPS, sizes={})
    base = U.PixelConLossV2(temperature=TAU)
    flag = U.PixelConLossV2(temperature=TAU, contrast_grad=True)
    for name, B in SIZES.items():
        A, C, la, lc, Pd = operands(B)
        n_a, n_c = A.shape[0], C.shape[0]
        entry = dict(batch=B, n_a=n_a, n_c=n_c, pairs=n_a * n_c)
        for pname, P in (("P_none", None), ("P_dense", Pd)):
            forms = {"anchor_grad_only": lambda P=P: run(base, A, C, la, lc, P, False),
                     "contrast_grad": lambda P=P: run(flag, A, C, la, lc, P, True),
                     "contrast_sweep_alone": sweep_only(A, C, la, lc, P)}
            fit = n_a * n_c <= REF_MAX_PAIRS
            if fit:
                forms["torch_autograd_fp32_reference"] = lambda P=P: run_ref(A, C, la, lc, P)
            got0, got1 = run(base, A, C, la, lc, P, False), run(flag, A, C, la, lc, P, True)
            chk = dict(loss_bit_identical=bool(torch.equal(got0[0], got1[0])),
                       anchor_grad_bit_identical=bool(torch.equal(got0[1], got1[1])))
            if fit:
                r = run_ref(A, C, la, lc, P)
                chk.update(loss_rel_vs_reference=abs(float(got1[0]) - float(r[0])) / abs(float(r[0])),
                           cos_anchor_grad=cos(got1[1], r[1]), cos_contrast_grad=cos(got1[2], r[2]))
                del r
            t = time_forms(forms, args.repeats, args.iters, flush)
            ms = {k: summary(v) for k, v in t.items()}
            sweep_ms = ms["contrast_sweep_alone"]["median"]
            tflops = 1024.0 * n_a * n_c / (sweep_ms * 1e-3) / 1e12
            entry[pname] = dict(ms=ms, check=chk,
                                extra_ms=round(ms["contrast_grad"]["median"] - ms["anchor_grad_only"]["median"], 4),
                                contrast_sweep_tflops=round(tflops, 1),
                                contrast_sweep_frac_of_burst_bf16=round(tflops / BURST_BF16_TFLOPS, 3))
            print(name, pname, {k: v["median"] for k, v in ms.items()}, "sweep %.0f TFLOP/s" % tflops, chk,
                  flush=True)
            torch.cuda.empty_cache()
        res["sizes"][name] = entry
        del A, C, la, lc, Pd
        torch.cuda.empty_cache()
    print(json.dumps(res, indent=1))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
