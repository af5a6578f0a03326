#!/usr/bin/env python
"""Benchmark of the UCD distillation-loss hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--workload voc|ade|city|sweep:<pixels>] [--batch B] [--dump-outputs DIR]

One "step" = one pass of the hot path over one synthetic batch, forward + backward:
  bilinear logit upsample (old model under no_grad first, then the new one: train.py:100-108) -> pre_contrastive_pixel -> PixelConLossV2
  -> UnbiasedCrossEntropy(...).mean() + con/100 + 10 * UnbiasedKnowledgeDistillationLoss -> backward
through the reference-shaped modules of ucd_b200 (train.py:115-116,133 wiring).

Workloads (BASELINE.json configs; default = configs[1] held on one GPU, which is what the metric is quoted on):
  voc    VOC 15-5s step 1, 17/16 classes, batch 24 @512x512 per GPU (32x32 embeddings); --batch 3 = the real per-GPU
         batch of configs[1] on 8 GPUs
  ade    ADE 100-50 step 1, 151/101 classes, batch 3 @512x512 (wide log-softmax, K = 112 joint probability)
  city   Cityscapes 13-6 step 1, 20/14 classes, batch 3 @512x1024 (32x64 embeddings)
  sweep:<px>  contrastive term only (prep + loss, fwd + bwd), VOC-like 21/16 classes, <px> pixels per GPU as images of
         32x32 (configs[4]: 8k .. 256k pixels per GPU)
Weak scaling: each rank holds its own images; with N>1 the contrast columns of all ranks are exchanged (one
all-gather over NCCL, overlapped with the sweep over the local columns) so negatives span the global batch.
metric = pixel pairs (N_a local x N_c global, summed over ranks) per second, in Mpairs/s.

--dump-outputs DIR writes what the last timed step handed back to its caller (rank 0): the losses and the gradients
with respect to f_n and the low-res logits, one float32 DIR/<name>.npy each.  Inputs are seeded, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ucd_loss_fwd_bwd_pixel_pairs_per_s"
UNIT = "Mpixel-pairs/s"
WORKLOADS = {
    "voc": dict(name="VOC 15-5s step 1, batch 24 @512x512 per GPU", B=24, h=32, w=32, H=512, W=512, C=17, C_old=16,
                max_label=20, cpu_sample_B=3),
    "ade": dict(name="ADE20K 100-50 step 1, batch 3 @512x512 per GPU", B=3, h=32, w=32, H=512, W=512, C=151, C_old=101,
                max_label=150, cpu_sample_B=1),
    "city": dict(name="Cityscapes 13-6 step 1, batch 3 @512x1024 per GPU", B=3, h=32, w=64, H=512, W=1024, C=20,
                 C_old=14, max_label=20, cpu_sample_B=1),
}
WORKLOAD = WORKLOADS["voc"]   # default; scripts/ import it


def get_workload(spec, batch):
    if spec.startswith("sweep:"):
        px = int(spec.split(":", 1)[1])
        if px % 1024:
            raise SystemExit("--workload sweep:<pixels>: pixels must be a multiple of 1024 (images of 32x32)")
        wl = dict(name="contrastive sweep, %d pixels per GPU (VOC-like 21/16 classes, 32x32 embeddings)" % px,
                  B=px // 1024, h=32, w=32, H=512, W=512, C=21, C_old=16, max_label=20, cpu_sample_B=3, con_only=True)
    else:
        if spec not in WORKLOADS:
            raise SystemExit("--workload must be one of %s or sweep:<pixels>" % ", ".join(WORKLOADS))
        wl = dict(WORKLOADS[spec], con_only=False)
    if batch:
        wl["name"] = wl["name"].replace("batch %d " % wl["B"], "batch %d " % batch)
        wl["B"] = batch
    wl["cpu_sample_B"] = min(wl["cpu_sample_B"], wl["B"])
    return wl


# kernels launched by each C-ABI entry point (for gpu_launches; memsets are not kernels).  ucd_con_fwd: sweep 1,
# combine, sweep 2, finalize, reduce = 5 (a part-1 call launches sweep 1 only: counted from its `part` argument).
KERNELS_PER_CALL = {"ucd_upsample_bilinear_fwd": 1, "ucd_upsample_bilinear_bwd": 1, "ucd_unce_fwd": 1,
                    "ucd_unce_bwd": 1, "ucd_kd_fwd": 2, "ucd_kd_bwd": 1, "ucd_con_prep_labels": 2,
                    "ucd_con_prep_pack": 4, "ucd_con_prep_bwd": 1, "ucd_con_fwd": 5, "ucd_con_bwd": 1,
                    "ucd_con_pack_rows": 1, "ucd_seg_fused_fwd": 2, "ucd_rows_normalize_fwd": 1,
                    "ucd_rows_normalize_bwd": 1, "ucd_con_tile_ranges": 1, "ucd_unce_unkd_bwd": 1}
HOST_ONLY_CALLS = ("ucd_last_error", "ucd_version", "ucd_device_ok", "ucd_con_max_tiles", "ucd_con_prob_kpad",
                   "ucd_con_num_bins", "ucd_con_px_meta_ints", "ucd_con_blk_meta_ints", "ucd_con_workspace_bytes",
                   "ucd_reduce_scratch_floats", "ucd_seg_fused_workspace_floats")


DUMP_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, outputs):
    """One float32 <name>.npy per output.  When the outputs exceed DUMP_BYTES together, every non-scalar one is cut to
    the same fraction of its elements: a seeded (seed 0), sorted sample of its flattened indices, so that the sample is
    the same from run to run and from build to build."""
    os.makedirs(out_dir, exist_ok=True)
    limit = (DUMP_BYTES - 4096) // 4            # elements; 4 KB left for the .npy headers
    total = sum(t.numel() for t in outputs.values())
    for name, t in outputs.items():
        a = t.detach().float().cpu()
        if total > limit and a.numel() > 1:
            keep = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:a.numel() * limit // total]
            a = a.reshape(-1)[keep.sort().values]
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())


def gen(seed, *shape, scale=1.0):
    return torch.randn(*shape, generator=torch.Generator().manual_seed(seed)) * scale


def make_inputs(rank, B, wl):
    """Synthetic inputs of SURVEY.md 8d: seeds 1-4 (+1000*rank), class-correlated features, blob labels."""
    h, w, H, W, C, C_old = wl["h"], wl["w"], wl["H"], wl["W"], wl["C"], wl["C_old"]
    o = 1000 * rank
    f_n, f_o = gen(1 + o, B, 256, h, w), gen(2 + o, B, 256, h, w)
    l_po = gen(3 + o, B, C_old, h, w, scale=3.0)
    lr = gen(4 + o, B, C, h, w, scale=3.0)
    proto = gen(9, C, 256)
    add = proto[l_po.argmax(1)].permute(0, 3, 1, 2)
    f_n, f_o = 0.3 * f_n + 0.7 * add, 0.3 * f_o + 0.7 * add
    lab = torch.zeros(B, H, W, dtype=torch.int64)
    lab[:, H // 5:3 * H // 5, W // 5:3 * W // 5] = C_old
    lab[:, 3 * H // 5:4 * H // 5, W // 10:2 * W // 5] = C - 1
    lab[:, :H // 25, :] = 255
    return dict(f_n=f_n.contiguous(), f_o=f_o.contiguous(), l_po=l_po, logits_lr=lr, labels=lab)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (NVML every 5 ms in a thread; the
    nvidia-smi query of the profiling recipe is the fallback)."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, gpu_index):
        self.idx, self.rows, self.stop_flag, self.thr, self.max_mhz = gpu_index, [], False, None, None
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[gpu_index]) if visible and visible.split(",")[gpu_index].isdigit() else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _loop(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    rs = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    rs = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((mhz, rs))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nvml is not None:
            self.thr = threading.Thread(target=self._loop, daemon=True)
            self.thr.start()

    def stop(self):
        if self.nvml is None:
            return self._smi_once()
        self.stop_flag = True
        self.thr.join(timeout=1)
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for _, rs in self.rows:
            bits |= rs
        return dict(sm_mhz=(sm[len(sm) // 2] if sm else None), sm_max_mhz=self.max_mhz,
                    reasons=[n for n, b in self.REASONS if bits & b], samples=len(sm), source="nvml, 5 ms period")

    def _smi_once(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            out = subprocess.run(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                 capture_output=True, text=True, timeout=10).stdout.strip().split(",")
            names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
            return dict(sm_mhz=float(out[0]), sm_max_mhz=float(out[1]),
                        reasons=[n for n, v in zip(names, out[2:6]) if v.strip().lower().startswith("active")],
                        samples=1, source="nvidia-smi after the timed region (NVML unavailable)")
        except Exception:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["clock query unavailable"], samples=0)


class CallTimer:
    """Proxy around the ctypes library: records a CUDA-event pair on the current stream around every C-ABI call that
    launches kernels, so per-kernel-group device times come from the same timed region as the headline number."""

    def __init__(self, handle):
        self._h, self.events, self.counts, self.launches, self.enabled = handle, {}, {}, 0, False

    def __getattr__(self, name):
        fn = getattr(self._h, name)
        if not name.startswith("ucd_") or name in HOST_ONLY_CALLS:
            return fn

        def wrapped(*args):
            if not self.enabled:
                return fn(*args)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*args)
            e1.record()
            key = name
            k = KERNELS_PER_CALL.get(name, 1)
            if name == "ucd_con_fwd":      # args[8] = part: 1 = sweep 1 over the local columns only
                part = int(args[8])
                key, k = name + (":local" if part == 1 else (":rest" if part == 2 else "")), (1 if part == 1 else 5)
            self.events.setdefault(key, []).append((e0, e1))
            self.counts[key] = self.counts.get(key, 0) + 1
            self.launches += k
            return rc
        return wrapped

    def totals_ms(self):
        return {k: sum(a.elapsed_time(b) for a, b in v) for k, v in self.events.items()}


def cpu_reference_sample(steps, warmup, wl):
    """The reference's CPU implementation of the path (oracle port, torch CPU, all host threads) on a bounded
    sample of the workload: cpu_sample_B images of the same shapes (the N^2 fp32 temporaries of the reference
    formulation bound what the host can hold and finish in seconds)."""
    from oracle import ucd_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    nb = wl["cpu_sample_B"]
    case = make_inputs(0, nb, wl)
    times, pairs = [], 0
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        f_n = case["f_n"].clone().requires_grad_(True)
        if wl["con_only"]:
            A, Cst, la, lc, P, _ = O.pre_contrastive_pixel(f_n, case["labels"], case["l_po"], case["f_o"],
                                                           max_label=wl["max_label"])
            O.pixel_con_loss(A, Cst, la, lc, P).backward()
            n_a, n_c = A.shape[0], Cst.shape[0]
        else:
            lr = case["logits_lr"].clone().requires_grad_(True)
            res = O.hot_path(f_n, case["f_o"], case["l_po"], lr, case["labels"].clone(), old_cl=wl["C_old"],
                             max_label=wl["max_label"])
            res.total.backward()
            n_a, n_c = res.n_anchor, res.n_contrast
        dt = time.perf_counter() - t0
        pairs = n_a * n_c
        if i >= warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    what = "contrastive term" if wl["con_only"] else "whole path"
    return dict(value=pairs / (ms * 1e-3) / 1e6, unit=UNIT, cores=torch.get_num_threads(), kind="port",
                sample="%d of the %d images of one step (N_a x N_c = %d pairs), fwd+bwd of the %s, mean of %d steps"
                       % (nb, wl["B"], pairs, what, len(times)), ms_per_step=ms, pairs=pairs), ms


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)   # as asked; each step is a bounded sample (seconds)
    cb, ms = cpu_reference_sample(steps, warmup, wl)
    line = dict(metric=METRIC, value=cb["value"], unit=UNIT, n_gpus=args.gpus, steps=steps, warmup=warmup,
                ms_per_step=ms, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", impl="reference",
                config=dict(workload=wl["name"], sample=cb["sample"], classes=[wl["C"], wl["C_old"]]),
                cpu_baseline=cb,
                e2e=dict(value=cb["value"], unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                gpu_launches=0)
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ucd_b200")
    ap.add_argument("--workload", default="voc", help="voc | ade | city | sweep:<pixels per GPU>")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the informational legs (N1 / N4 variants, GPU arm at the CPU sample size)")
    ap.add_argument("--no-parity", action="store_true", help="N>1: skip the concatenated-batch parity check on rank 0")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the losses and gradients of the last timed step as DIR/<name>.npy (float32, at most "
                         "64 MB in all: larger outputs are cut to a seeded sample of their elements)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the ucd_b200 arm; the reference arm runs a smaller sample")
    wl = get_workload(args.workload, args.batch)
    if args.impl == "reference":
        return run_reference(args, wl)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the ucd_b200 path has no CPU fallback "
                         "(use --impl reference for the CPU reference arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import ucd_b200 as U
    from ucd_b200 import _lib
    timer = CallTimer(_lib.lib())
    _lib._lib = timer

    B, H, W, C, C_old, max_label, con_only = wl["B"], wl["H"], wl["W"], wl["C"], wl["C_old"], wl["max_label"], wl["con_only"]
    host = make_inputs(rank, B, wl)
    if con_only:
        host.pop("logits_lr")
    # the dataloader hands labels over as uint8 and the trainer casts them on the device (train.py:97-98,
    # dataset/transform.py:350): the end-to-end leg copies uint8 labels and casts after the copy, like the reference
    pinned = {k: (v.to(torch.uint8) if k == "labels" else v).pin_memory() for k, v in host.items()}
    devin = {k: v.to(dev) for k, v in host.items()}
    conloss = U.PixelConLossV2(temperature=0.07, gather_negatives=world > 1)
    unce = U.UnbiasedCrossEntropy(old_cl=C_old, ignore_index=255, reduction="none")
    unkd = U.UnbiasedKnowledgeDistillationLoss(alpha=1.0)
    state = {}

    def step(inp):
        f_n = inp["f_n"].detach().requires_grad_(True)
        if con_only:
            tup = U.pre_contrastive_pixel(f_n, inp["labels"], l_po=inp["l_po"], f_o=inp["f_o"], max_label=max_label)
            con = conloss(*tup)
            (con / 100).backward()
            state.update(n_a=tup[0].shape[0], n_c=tup[1].shape[0], con=con.detach(), g_fn=f_n.grad)
            return con
        lr = inp["logits_lr"].detach().requires_grad_(True)
        with torch.no_grad():   # the old model runs first (train.py:100-102), then the new one (:105-108)
            outputs_old = U.interpolate_bilinear(inp["l_po"], (H, W))
        outputs = U.interpolate_bilinear(lr, (H, W))
        # evaluation order of train.py:115-116,133: prep, criterion, contrastive loss, distillation
        tup = U.pre_contrastive_pixel(f_n, inp["labels"], l_po=inp["l_po"], f_o=inp["f_o"], max_label=max_label)
        ce = unce(outputs, inp["labels"]).mean()
        con = conloss(*tup)
        kd = unkd(outputs, outputs_old)
        loss = ce + con / 100 + 10 * kd
        loss.backward()
        state.update(n_a=tup[0].shape[0], n_c=tup[1].shape[0], con=con.detach(), ce=ce.detach(), kd=kd.detach(),
                     loss=loss.detach(), g_fn=f_n.grad, g_lr=lr.grad)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(n):
            fn()
        a1.record()
        barrier()
        return a0.elapsed_time(a1) / n

    # ---- device-resident timing (value): the plain step loop, nothing but the step inside the timed region ----
    for _ in range(args.warmup):
        step(devin)
    barrier()
    # A full collection of the interpreter's heap (about a million objects once torch is imported) takes 15-150 ms:
    # one of them inside a 20-40 ms timed region doubled a B=3 bench line (round 2: ADE 2.7 instead of 1.3 ms, one
    # e2e leg 16.9 instead of 1.3 ms).  Freeze what exists so that collections during the loops only see the
    # objects the steps create (the collector itself stays on).
    gc.collect()
    gc.freeze()
    sampler = ClockSampler(local)
    if rank == 0 and not os.environ.get("UCD_BENCH_NO_SAMPLER"):
        sampler.start()
    t_wall0 = time.perf_counter()
    ms_dev = timed(lambda: step(devin), args.steps)
    timed_region_s = time.perf_counter() - t_wall0
    clocks = sampler.stop() if (rank == 0 and sampler.thr is not None) else None
    if args.dump_outputs and rank == 0:
        names = (("loss", "loss"), ("con", "con"), ("ce", "ce"), ("kd", "kd"), ("grad_f_n", "g_fn"),
                 ("grad_logits_lr", "g_lr"))
        dump_outputs(args.dump_outputs, {name: state[key] for name, key in names if key in state})
    # ---- the same loop once more with a CUDA-event pair around every C-ABI call: per-kernel-group device times for
    #      the rooflines and the launch count.  (The ~35 extra event records per step cost host time and stream slots:
    #      this pass runs up to 15 % slower than the plain loop, which is why it is not the headline.) ----
    timer.enabled = True
    ms_dev_instrumented = timed(lambda: step(devin), args.steps)
    timer.enabled = False
    call_ms = {k: v / args.steps for k, v in timer.totals_ms().items()}
    launches = timer.launches
    g_rank0 = state["g_fn"].clone()
    con_multi = float(state["con"])

    # ---- the GPU arm at the CPU arm's sample size: a like-for-like ratio for the reference arm ----
    ms_sample, pairs_sample = None, None
    if world == 1 and wl["cpu_sample_B"] != B and not args.no_extras:
        small = {k: v[:wl["cpu_sample_B"]].contiguous() for k, v in devin.items()}
        for _ in range(3):
            step(small)
        barrier()
        ms_sample = timed(lambda: step(small), args.steps)
        pairs_sample = state["n_a"] * state["n_c"]
        step(devin)   # restore `state` for the legs below
        barrier()

    ms_fused = ms_static = ms_graph = None
    if not con_only and not args.no_extras:
        # ---- the same step with the opt-in N1 fusion (FusedUnbiasedLosses: no full-res logits), for information ----
        fused = U.FusedUnbiasedLosses(old_cl=C_old, ignore_index=255, alpha=1.0)

        def step_fused():
            f_n = devin["f_n"].detach().requires_grad_(True)
            lr = devin["logits_lr"].detach().requires_grad_(True)
            tup = U.pre_contrastive_pixel(f_n, devin["labels"], l_po=devin["l_po"], f_o=devin["f_o"], max_label=max_label)
            con = conloss(*tup)
            ce, kd = fused(lr, devin["l_po"], devin["labels"])
            (ce + con / 100 + 10 * kd).backward()

        for _ in range(3):
            step_fused()
        barrier()
        ms_fused = timed(step_fused, args.steps)

        # ---- opt-in sync-free step (N1 fused CE/KD + N4 contrastive without the 5-tuple), for information: eager,
        #      and (single GPU) forward + backward replayed from one CUDA graph ----
        con_static = U.PixelContrastiveDistillation(temperature=0.07, max_label=max_label, gather_negatives=world > 1)
        gs = {k: devin[k].clone() for k in ("f_n", "f_o", "l_po", "logits_lr", "labels")}
        gs["f_n"].requires_grad_(True), gs["logits_lr"].requires_grad_(True)

        def step_static():
            gs["f_n"].grad = gs["logits_lr"].grad = None
            ce, kd = fused(gs["logits_lr"], gs["l_po"], gs["labels"])
            (ce + con_static(gs["f_n"], gs["labels"], gs["l_po"], gs["f_o"]) / 100 + 10 * kd).backward()

        for _ in range(3):
            step_static()
        barrier()
        ms_static = timed(step_static, args.steps)
        if world == 1:
            try:
                if hasattr(torch.autograd.graph, "set_warn_on_accumulate_grad_stream_mismatch"):
                    torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    step_static()
                torch.cuda.current_stream().wait_stream(side)
                gs["f_n"].grad = gs["logits_lr"].grad = None
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    ce, kd = fused(gs["logits_lr"], gs["l_po"], gs["labels"])
                    (ce + con_static(gs["f_n"], gs["labels"], gs["l_po"], gs["f_o"]) / 100 + 10 * kd).backward()
                for _ in range(3):
                    graph.replay()
                barrier()
                ms_graph = timed(graph.replay, args.steps)
            except Exception as exc:  # informational leg only
                ms_graph = "capture failed: %s" % (str(exc).splitlines()[0][:120],)

    # ---- end-to-end through the public API with host buffers (e2e) ----
    # Every step copies its inputs from pinned host memory and copies losses + gradients back.  Like a DataLoader
    # with pin_memory / non_blocking prefetch, the copies of step i+1 / i-1 run on side streams (one per direction:
    # two copy engines) while step i computes; all of them are inside the timed region.
    out_host = dict(losses=torch.empty(3).pin_memory(), g_fn=torch.empty_like(host["f_n"]).pin_memory())
    if not con_only:
        out_host["g_lr"] = torch.empty_like(host["logits_lr"]).pin_memory()
    h2d_stream, d2h_stream = torch.cuda.Stream(), torch.cuda.Stream()
    main_s = torch.cuda.current_stream()
    # two preallocated device slots for the inputs (no allocator traffic inside the loop), filled alternately
    slots = [dict(buf={k: torch.empty_like(v, device=dev) for k, v in pinned.items()}, free=None) for _ in range(2)]
    copy_ev = {"h2d": [], "d2h": []}   # (start, end) event pairs on the copy streams: time the copies themselves take

    def prefetch(slot):
        with torch.cuda.stream(h2d_stream):
            if slot["free"] is not None:
                h2d_stream.wait_event(slot["free"])          # the step that last read this slot has finished
            a = torch.cuda.Event(enable_timing=True)
            a.record(h2d_stream)
            for k, v in pinned.items():
                slot["buf"][k].copy_(v, non_blocking=True)
            slot["ready"] = torch.cuda.Event(enable_timing=True)
            slot["ready"].record(h2d_stream)
            copy_ev["h2d"].append((a, slot["ready"]))

    def e2e_run(n_steps):
        prefetch(slots[0])
        for i in range(n_steps):
            cur = slots[i % 2]
            main_s.wait_event(cur["ready"])
            if i + 1 < n_steps:
                prefetch(slots[(i + 1) % 2])
            inp = dict(cur["buf"])
            inp["labels"] = inp["labels"].to(torch.long)          # train.py:98
            step(inp)
            losses = (torch.stack([state["con"], state["ce"], state["kd"]]) if not con_only
                      else torch.stack([state["con"]] * 3))
            done = torch.cuda.Event()
            done.record(main_s)
            cur["free"] = done
            with torch.cuda.stream(d2h_stream):
                d2h_stream.wait_event(done)
                a = torch.cuda.Event(enable_timing=True)
                a.record(d2h_stream)
                out_host["losses"].copy_(losses, non_blocking=True)
                out_host["g_fn"].copy_(state["g_fn"], non_blocking=True)
                outs = [losses, state["g_fn"]]
                if not con_only:
                    out_host["g_lr"].copy_(state["g_lr"], non_blocking=True)
                    outs.append(state["g_lr"])
                for t_ in outs:
                    t_.record_stream(d2h_stream)
                b = torch.cuda.Event(enable_timing=True)
                b.record(d2h_stream)
                copy_ev["d2h"].append((a, b))
        main_s.wait_stream(d2h_stream)

    e2e_run(max(3, args.warmup // 2))
    barrier()
    copy_ev["h2d"].clear(), copy_ev["d2h"].clear()
    t0 = time.perf_counter()
    e2a, e2b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2a.record()
    e2e_run(args.steps)
    e2b.record()
    barrier()
    wall_ms = 1e3 * (time.perf_counter() - t0) / args.steps
    ev_ms = e2a.elapsed_time(e2b) / args.steps
    ms_e2e = max(ev_ms, wall_ms)
    copy_ms = {k: sum(a.elapsed_time(b) for a, b in v) / max(len(v), 1) for k, v in copy_ev.items()}
    h2d = sum(v.numel() * v.element_size() for v in pinned.values())
    d2h = sum(v.numel() * v.element_size() for v in out_host.values())

    # ---- N>1: parity of the data-parallel path, evaluated on rank 0 (the oracle of SURVEY 8e: the single-chunk path
    #      on the rank-concatenated batch; the CPU oracle itself checks that path at this size in tests/) ----
    parity = None
    if world > 1 and not args.no_parity:
        keys = ("f_n", "f_o", "l_po", "labels")
        cat = {}
        for k in keys:
            parts = [torch.empty_like(devin[k]) for _ in range(world)] if rank == 0 else None
            dist.gather(devin[k], parts, dst=0)
            if rank == 0:
                cat[k] = torch.cat(parts)
        if rank == 0:
            f_all = cat["f_n"].detach().requires_grad_(True)
            single = U.PixelConLossV2(temperature=0.07)
            tup = U.pre_contrastive_pixel(f_all, cat["labels"], l_po=cat["l_po"], f_o=cat["f_o"], max_label=max_label,
                                          require_new_class=True)
            con_single = single(*tup)
            con_single.backward()
            g_single = f_all.grad[:B].double()          # rank 0's images come first
            g_multi = g_rank0.double() * (100.0 / world)  # step() back-propagates con/100; ddp_grad_scale = world
            g_single = g_single / 1.0
            cosv = float((g_single * g_multi).sum() / (g_single.norm() * g_multi.norm()).clamp_min(1e-300))
            rel = abs(con_multi - float(con_single)) / abs(float(con_single))
            ratio = float(g_multi.norm() / g_single.norm().clamp_min(1e-300))
            parity = dict(parity_checked=True, loss_data_parallel=con_multi, loss_concatenated_batch=float(con_single),
                          loss_rel_err=rel, grad_cosine_rank0=cosv, grad_norm_ratio_rank0=ratio,
                          ok=bool(rel <= 1e-3 and cosv >= 0.999 and abs(ratio - 1) < 2e-2),
                          n_anchor_global=int(tup[0].shape[0]), n_contrast_global=int(tup[1].shape[0]),
                          note="rank 0: PixelConLossV2 on the rank-concatenated batch (one chunk) vs the exchanged path; "
                               "bars: loss 1e-3 rel, gradient cosine 0.999 (BASELINE.json)")
            del cat, f_all, tup
        barrier()

    # ---- aggregate over ranks: max time, sum of pairs ----
    n_a = state["n_a"]
    stats = torch.tensor([ms_dev, ms_e2e, float(n_a), float(state["n_c"]), ms_fused or 0.0, ev_ms, wall_ms], device=dev,
                         dtype=torch.float64)
    if world > 1:
        allst = [torch.zeros_like(stats) for _ in range(world)]
        dist.all_gather(allst, stats)
    else:
        allst = [stats]
    allst = torch.stack(allst).cpu()
    ms_dev_max, ms_e2e_max, ms_fused_max = float(allst[:, 0].max()), float(allst[:, 1].max()), float(allst[:, 4].max())
    n_c_global = float(allst[:, 3].sum())
    pairs_total = float((allst[:, 2] * n_c_global).sum())
    pairs_local = float(n_a) * n_c_global

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # a timed region of well under a second runs at full clocks (see `clocks`): the burst figure applies; a long
        # region under the power cap is compared with the sustained one
        burst = timed_region_s < 1.0
        bf16_peak = peaks.get("bf16_tflops" if burst else "bf16_tflops_sustained", 1590.0 if burst else 1400.0)
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        peak_src = ("measured (MEASURED_PEAKS.json: %s bf16, copy bandwidth); timed region %.2f s"
                    % ("burst" if burst else "sustained", timed_region_s)) if peaks else "fallback (B200_PROFILING.md)"
        f_pair = 4 * 256 + 2 * C_old                                 # algorithmic flop per pixel pair (BASELINE.md 3)
        con_ms = sum(v for k, v in call_ms.items() if k.startswith("ucd_con_fwd"))
        con_tflops = pairs_local * f_pair / (con_ms * 1e-3) / 1e12
        npx = B * H * W
        hbm = {}
        if not con_only:
            # SURVEY 8(d) algorithmic bytes per full-res pixel (fp32 logits, int64 labels); the per-pixel statistics a
            # kernel saves for its backward are extra traffic, listed as saved_stat_bytes, NOT counted as achieved
            for name, nbytes, extra in (
                    ("ucd_unce_fwd", npx * (4 * C + 8 + 4), npx * 4), ("ucd_unce_bwd", npx * (8 * C + 8 + 4 + 4), npx * 4),
                    ("ucd_kd_fwd", npx * (4 * C + 4 * C_old), npx * 12), ("ucd_kd_bwd", npx * (8 * C + 4 * C_old), npx * 12),
                    # the two backward passes run as ONE kernel when both losses consume the same logits: judged
                    # against the fused lower bound of SURVEY 8(d) (read x, t and the labels once, write dx once)
                    ("ucd_unce_unkd_bwd", npx * (8 * C + 4 * C_old + 8), npx * 16),
                    ("ucd_upsample_bilinear_fwd", npx * 4 * (C + C_old), 0), ("ucd_upsample_bilinear_bwd", npx * 4 * C, 0)):
                if name in call_ms:
                    gbs = nbytes / (call_ms[name] * 1e-3) / 1e9
                    hbm[name] = dict(ms=round(call_ms[name], 4), algorithmic_bytes=nbytes, saved_stat_bytes=extra,
                                     achieved_gbs=round(gbs, 1), frac=round(gbs / hbm_peak, 4))
            stream_ms = sum(v["ms"] for v in hbm.values())
            # whole streaming chain: the separate-module bytes of SURVEY 8(d), minus what the fused backward no longer
            # has to move (one read of x, the labels and one lse plane: 4C + 12), so that fusion does not inflate it
            chain_bpp = 32 * C + 12 * C_old + 28 - ((4 * C + 12) if "ucd_unce_unkd_bwd" in call_ms else 0)
            hbm["chain"] = dict(bytes_per_px=chain_bpp, ms=round(stream_ms, 4),
                                achieved_gbs=round(npx * chain_bpp / (stream_ms * 1e-3) / 1e9, 1),
                                frac=round(npx * chain_bpp / (stream_ms * 1e-3) / 1e9 / hbm_peak, 4))
        cpu_baseline = None
        if world == 1 and not args.no_cpu_baseline:
            cpu_baseline, _ = cpu_reference_sample(3, 1, wl)
        traffic = None
        traffic_note = "not captured for this workload (ncu --set full is run on the default workload only)"
        if world == 1 and args.workload == "voc" and B == WORKLOADS["voc"]["B"]:
            traffic = 9.30e7
            traffic_note = ("RECORDED, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum of the two "
                            "sweep kernels per step from ncu --set full, profiles/r02c_ncu_full.md (21.5 + 45.1 MB sweep 1, "
                            "22.9 + 3.5 MB sweep 2; algorithmic operands + gradient: 46 MB - the rest are the V / U partials "
                            "of the column splits)")
        line = dict(
            metric=METRIC, value=pairs_total / (ms_dev_max * 1e-3) / 1e6, unit=UNIT, n_gpus=world, steps=args.steps,
            warmup=args.warmup, ms_per_step=ms_dev_max, higher_is_better=True, scaling="weak", vs_baseline=None,
            dtype="bf16 operands / f32 accumulate (contrastive); f32 (CE, KD, upsample)", data="synthetic",
            config=dict(workload=wl["name"], step="contrastive term only" if con_only else "whole hot path",
                        classes=[C, C_old], pixels_per_gpu=B * wl["h"] * wl["w"], n_anchor_rank0=n_a,
                        n_contrast_global=int(n_c_global), pairs_per_step=int(pairs_total), temperature=0.07,
                        l2=("no flush: the inputs of a step exceed the 126 MB L2 (full-res logits %.0f MB; bf16 column "
                            "tiles %.0f MB are meant to be L2-resident)" % (npx * C * 4 / 1e6, n_c_global * 512 / 1e6))
                        if not con_only else "no flush: column tiles (%.0f MB) are meant to be L2-resident; V partials "
                        "stream through" % (n_c_global * 512 / 1e6),
                        parallelism="dp%d, contrast columns exchanged in one all-gather overlapped with the local sweep" % world),
            roofline=dict(bound="tensor", kernel="ucd_con_fwd (sweep 1 + combine + sweep 2 + finalize)",
                          achieved=con_tflops, peak=bf16_peak, unit="TFLOP/s", frac=con_tflops / bf16_peak,
                          traffic=traffic, traffic_note=traffic_note, flop_per_pair=f_pair, ms=con_ms,
                          peak_source=peak_src,
                          frac_of_sustained=con_tflops / peaks.get("bf16_tflops_sustained", 1400.0)),
            roofline_hbm=hbm,
            call_ms={k: round(v, 4) for k, v in sorted(call_ms.items())},
            call_ms_note="CUDA events around every C-ABI call in a second, instrumented pass of the same loop "
                         "(%.3f ms per step there)" % ms_dev_instrumented,
            cpu_baseline=cpu_baseline,
            value_at_cpu_sample=(dict(value=pairs_sample / (ms_sample * 1e-3) / 1e6, unit=UNIT, ms_per_step=ms_sample,
                                      pairs=pairs_sample, note="this GPU arm on the CPU arm's bounded sample (%d images): "
                                      "the like-for-like figure for the reference arm" % wl["cpu_sample_B"])
                                 if ms_sample else None),
            e2e=dict(value=pairs_total / (ms_e2e_max * 1e-3) / 1e6, unit=UNIT, ms_per_step=ms_e2e_max,
                     h2d_bytes_per_step=h2d, d2h_bytes_per_step=d2h,
                     rank0_device_event_ms=ev_ms, rank0_wall_ms=wall_ms,
                     rank0_h2d_copy_ms_per_step=round(copy_ms["h2d"], 4), rank0_d2h_copy_ms_per_step=round(copy_ms["d2h"], 4),
                     copy_note="copy times = CUDA events on the two copy streams around the step's transfers (they "
                               "overlap the compute of the neighbouring steps; at N ranks they share the host's PCIe / "
                               "memory bandwidth, which is what the e2e figure runs into at N=8)",
                     per_rank_ms=[round(float(v), 4) for v in allst[:, 1]]),
            n1_fused=(dict(note="same step with the opt-in FusedUnbiasedLosses (upsample+CE+KD from low-res logits)",
                           ms_per_step=ms_fused_max, value=pairs_total / (ms_fused_max * 1e-3) / 1e6, unit=UNIT)
                      if ms_fused else None),
            n4_sync_free=(dict(note="rank 0: N1 fused CE/KD + PixelContrastiveDistillation (no 5-tuple, no host sync); "
                                    "graph = forward+backward replayed from one CUDA graph (single GPU only)",
                               ms_per_step_eager=ms_static, ms_per_step_graph=ms_graph) if ms_static else None),
            parity=parity,
            gpu_launches=int(launches), clocks=clocks,
            losses={k: float(state[k]) for k in ("con", "ce", "kd") if k in state},
        )
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
