"""Host-side mirror of the reference loss interface for the UCD hot path.

Same class names, constructor and ``forward`` signatures as the reference so that ``train.py`` and
``segmentation_module.py`` can use this module as a drop-in:

* ``UnbiasedCrossEntropy(old_cl=None, reduction='mean', ignore_index=255)``      utils/loss.py:89-109
* ``UnbiasedKnowledgeDistillationLoss(reduction='mean', alpha=1.)``              utils/loss.py:139-184
* ``PixelConLossV2(sample_method='none', temperature=0.07)``                     utils/loss.py:403-466
* ``pre_contrastive_pixel(f_n, l_n, l_po=None, f_o=None)`` (alias ``pre_contractive_pixel``)
                                                            utils/loss.py:258-399 / utils/utils.py:256-397
* ``interpolate_bilinear(x, size)`` for ``F.interpolate(..., mode='bilinear')``   segmentation_module.py:133
* siblings on the same kernels (SURVEY 8f N3): ``KnowledgeDistillationLoss`` (loss.py:112-136),
  ``MaskKnowledgeDistillationLoss`` (:218-256), ``MaskCrossEntropy`` (:186-216)

Opt-in, beyond the drop-in surface: ``FusedUnbiasedLosses`` (N1: upsample + UNCE + UNKD from the low-res logits; CE
only at the base step), ``predict_bilinear`` (the argmax prediction of the upsampled logits, without the upsample),
``PixelContrastiveDistillation`` (N4: prep + contrastive loss without the 5-tuple, no host sync, CUDA-graph capturable).

Everything runs in hand-written sm_100a CUDA kernels behind the C ABI of include/ucd_b200.h
(ucd_b200/_lib.py).  PyTorch is used for device memory, streams, autograd glue and NCCL only.
There is no CPU path: CPU tensors or a missing library raise.
"""
from __future__ import annotations

import weakref

import torch
import torch.nn as nn

from . import _lib
from ._lib import check, cur_stream, ptr

FEAT_DIM = 256
TILE = 128


def _need_cuda(*tensors):
    cur = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("ucd_b200: expected CUDA tensors (there is no CPU fallback for this path)")
        if cur is None:
            cur = torch.cuda.current_device()
        if t.device.index != cur:
            # kernels are launched on the current device / its current stream: a tensor living elsewhere would be
            # dereferenced in the wrong context
            raise RuntimeError("ucd_b200: tensor on cuda:%d but the current device is cuda:%d - wrap the call in "
                               "`with torch.cuda.device(tensor.device):`" % (t.device.index, cur))


def _f32c(t):
    """fp32 contiguous view/copy of a floating tensor (the reference runs this path in fp32, amp O0)."""
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _scalar_grad(g):
    """A broadcast upstream gradient (e.g. from ``.mean()``) as a 1-element tensor, else None."""
    if g.dim() == 0:
        return g.reshape(1)
    if all(s == 0 for s in g.stride()):
        return g.as_strided((1,), (1,))
    return None


# ----------------------------------------------------------------------------------------------
# bilinear logit upsample
# ----------------------------------------------------------------------------------------------
class _UpsampleFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, out_h, out_w):
        _need_cuda(x)
        ctx.set_materialize_grads(False)   # no gradient reaches `out` when a loss chain hands d x straight to x (_Route)
        x = _f32c(x)
        lead, (h, w) = x.shape[:-2], x.shape[-2:]
        planes = 1
        for d in lead:
            planes *= d
        out = torch.empty(*lead, out_h, out_w, device=x.device, dtype=torch.float32)
        if planes > 0:
            check(_lib.lib().ucd_upsample_bilinear_fwd(ptr(x), ptr(out), planes, h, w, out_h, out_w, cur_stream()),
                  "upsample_bilinear_fwd")
        ctx.shape = (lead, h, w, out_h, out_w, planes)
        return out

    @staticmethod
    def backward(ctx, g):
        if g is None:
            return None, None, None
        lead, h, w, out_h, out_w, planes = ctx.shape
        g = _f32c(g)
        gin = torch.empty(*lead, h, w, device=g.device, dtype=torch.float32)
        if planes > 0:
            check(_lib.lib().ucd_upsample_bilinear_bwd(ptr(g), ptr(gin), planes, h, w, out_h, out_w, cur_stream()),
                  "upsample_bilinear_bwd")
        return gin, None, None


def interpolate_bilinear(x, size):
    """``F.interpolate(x, size=size, mode='bilinear', align_corners=False)`` (segmentation_module.py:133)."""
    out = _UpsampleFn.apply(x, int(size[0]), int(size[1]))
    if out.requires_grad:   # where `out` came from, for a loss chain that folds the adjoint into its backward (_Route)
        out._ucd_upsample = (x, x._version, out._version)
    return out


@torch.no_grad()
def predict_bilinear(logits_lr, size):
    """``interpolate_bilinear(logits_lr, size).max(dim=1)[1]`` - the int64 [B,H,W] prediction of validation and test -
    without the [B,C,H,W] upsample: one kernel interpolates every channel on the fly and keeps a running argmax per
    pixel.  Bit-identical to the argmax of ``interpolate_bilinear`` (ties to the first channel, NaN maximal, as
    ``torch.argmax``).  Upsampling only; no autograd."""
    _need_cuda(logits_lr)
    if logits_lr.dim() != 4:
        raise ValueError("predict_bilinear: logits must be [B,C,h,w]")
    x = _f32c(logits_lr)
    B, C, h, w = x.shape
    H, W = int(size[0]), int(size[1])
    pred = torch.empty(B, H, W, device=x.device, dtype=torch.int64)
    if pred.numel() > 0:
        check(_lib.lib().ucd_upsample_argmax(ptr(x), ptr(pred), B, C, h, w, H, W, cur_stream()), "upsample_argmax")
    return pred


class _Route:
    """Lets the head of a gradient chain on `outputs` = interpolate_bilinear(lr) hand the gradient of the LOW-RES logits
    straight to `lr` (``ucd_unce_unkd_bwd_lowres``: the full-size dx is never written, nor read back by the adjoint),
    instead of dx to `outputs`.  The head's Function then takes `lr` as an extra autograd input; `outputs`' own node
    receives no gradient from the chain (other consumers of `outputs` still flow through it and add up at `lr`).

    That is only equivalent while nobody observes the gradient of `outputs` itself.  `route_now()` decides in the
    head's backward, and anything it cannot classify takes the old path (dx for `outputs`):
      * `outputs.retains_grad` or tensor hooks on `outputs`: old path;
      * the pass must be a plain ``backward()``: ``autograd.grad`` / ``backward(inputs=...)`` may capture the gradient of
        `outputs`, and the engine cannot say whether it does (a captured node reads as "will execute").  A private leaf
        (`probe`) that no caller can name is an extra input of the head: its node executes in a plain pass only.
    Not covered: hooks registered on the NODE of `outputs` (``outputs.grad_fn.register_prehook`` / ``register_hook``)
    receive no gradient from the chain when it reroutes - torch offers no way to see them.  A tensor hook
    (``outputs.register_hook``) observes the same gradient and keeps the old path."""

    __slots__ = ("lr_shape", "out_ref", "out_hw", "probe_node")
    _probes = {}

    def __init__(self, src, out, probe_node):
        self.lr_shape, self.out_hw, self.probe_node = tuple(src.shape), tuple(out.shape[2:]), probe_node
        self.out_ref = weakref.ref(out)

    @staticmethod
    def of(outputs):
        """(route, lr, probe) when `outputs` is still what interpolate_bilinear(lr) returned, else None."""
        rec = getattr(outputs, "_ucd_upsample", None)
        if rec is None:
            return None
        src, src_version, out_version = rec
        if (src._version != src_version or outputs._version != out_version or not src.requires_grad
                or src.dim() != 4 or outputs.dim() != 4):
            return None
        probe = _Route._probes.get(outputs.device)
        if probe is None:
            probe = _Route._probes[outputs.device] = torch.empty((), device=outputs.device, requires_grad=True)
        return _Route(src, outputs, torch.autograd.graph.get_gradient_edge(probe).node), src, probe

    def route_now(self):
        out = self.out_ref()
        if out is None or out.retains_grad or out._backward_hooks:
            return False
        try:
            return bool(torch._C._will_engine_execute_node(self.probe_node))
        except Exception:   # noqa: BLE001 - e.g. a torch that no longer offers it: the old path is always right
            return False


# ----------------------------------------------------------------------------------------------
# one logit gradient for the losses that consume the same logits
# ----------------------------------------------------------------------------------------------
class _GradChain:
    """`outputs` feeds both the cross-entropy (train.py:116) and the distillation loss (train.py:133).  Autograd would
    run the two backward kernels and then sum their full-size logit gradients with a kernel of its own: x read twice,
    dx written twice and read twice more (2.5 GB + 1.3 GB at the BASELINE workload, a fifth of the drop-in step).
    Instead the loss modules of this file that are called on the SAME tensor object form a chain: every call after the
    first takes the previous call's `token` (a 0-d auxiliary output) as an extra autograd input, which makes the engine
    run their backward passes in reverse call order.  A backward that is not the head of the chain only records its
    term; the head - the first call - then launches ONE kernel for a cross-entropy + distillation pair
    (``ucd_unce_unkd_bwd``: x and softmax read once, dx written once) and, for any other combination, the individual
    kernels with ``accumulate`` into one shared buffer.  Only the head returns a gradient for `outputs`, so the engine
    sees exactly one, complete gradient from this family of losses; other consumers of `outputs` are accumulated with
    it the usual way."""

    __slots__ = ("token", "calls", "pending", "closed")
    MAX_MEMBERS = 4   # bounds what a chain keeps alive when losses are evaluated over and over without a backward

    def __init__(self):
        self.token, self.calls, self.pending, self.closed = None, 0, [], False

    @staticmethod
    def of(t):
        """The chain of tensor `t` (created on first use); None when no gradient is needed or the kernels would run
        on a private copy of `t` (not fp32 / not contiguous)."""
        if not (torch.is_grad_enabled() and t.requires_grad and t.dtype == torch.float32 and t.is_contiguous()):
            return None
        chain = getattr(t, "_ucd_grad_chain", None)
        # a chain only links calls of ONE forward pass: once a backward pass has touched it (or it is full) the next
        # call on the same tensor object - a persistent input used step after step - starts a new chain.  Two chains
        # on one tensor simply hand autograd two gradients.
        if chain is None or chain.closed or chain.calls >= _GradChain.MAX_MEMBERS:
            chain = t._ucd_grad_chain = _GradChain()
        return chain

    def submit(self, term, seq, is_head, route=None):
        """Called from a member's backward: returns (gradient for `inputs`, gradient for the link token, gradient for
        the head's low-res source, see _Route)."""
        self.closed = True
        if seq == self.calls:      # the last call runs first in a backward pass: drop what a pass that died left behind
            self.pending = []
        if not is_head:
            if term is not None:
                self.pending.append(term)
            return None, None, None   # the token's gradient stays undefined: the edge alone orders the backward passes
        terms, self.pending = self.pending + ([term] if term is not None else []), []
        self.token = None   # chain -> token -> grad_fn -> ctx -> chain would leave the pass's objects to the cycle collector
        if not terms:
            return None, None, None
        d_lr = _launch_lowres(terms, route) if route is not None else None
        if d_lr is not None:
            return None, None, d_lr
        return _launch_terms(terms), None, None


def _pair(terms):
    """(ce term, kd term) that one kernel can run together, or None."""
    ce = [t for t in terms if t["kind"] == "ce"]
    kd = [t for t in terms if t["kind"] == "kd" and t["variant"] in (0, 2)]
    if ce and kd and ce[0]["C"] == kd[0]["C"] and ce[0]["HW"] == kd[0]["HW"]:
        return ce[0], kd[0]
    return None


def _launch_lowres(terms, route):
    """d lr for a chain of exactly a cross-entropy + distillation pair, with the upsample adjoint folded in; None when
    the pass may observe the gradient of `outputs` or the shape is not one the kernel takes (the caller then runs the
    old path)."""
    pair = _pair(terms)
    if pair is None or len(terms) != 2 or not route.route_now():
        return None
    c, k = pair
    B, C, h, w = route.lr_shape
    H, W = route.out_hw
    d_lr = torch.empty(B, C, h, w, device=c["x"].device, dtype=torch.float32)
    rc = _lib.lib().ucd_unce_unkd_bwd_lowres(
        ptr(c["x"]), ptr(c["targets"]), ptr(c["lse"][0]), ptr(c["lse"][1]), ptr(c["g_px"]), ptr(c["g_sc"]), 1.0,
        ptr(c["stats"]), c["mean_over_valid"], c["old_cl"], c["ignore_index"], ptr(k["t"]), ptr(k["m"]), k["alpha"],
        ptr(k["lse3"]), ptr(k["g_px"]), ptr(k["g_sc"]), k["g_mul"], k["variant"], ptr(d_lr), B, C, k["C_old"], h, w,
        H, W, cur_stream())
    if rc == _lib.UCD_ENOSUP:
        return None
    check(rc, "unce_unkd_bwd_lowres")
    return d_lr


def _launch_terms(terms):
    """dx = sum of the terms' logit gradients, written by as few passes over the logits as possible."""
    dx = torch.empty_like(terms[0]["x"])
    pair = _pair(terms)
    acc = False
    if pair is not None:
        c, k = pair
        check(_lib.lib().ucd_unce_unkd_bwd(
            ptr(c["x"]), ptr(c["targets"]), ptr(c["lse"][0]), ptr(c["lse"][1]), ptr(c["g_px"]), ptr(c["g_sc"]), 1.0,
            ptr(c["stats"]), c["mean_over_valid"], c["old_cl"], c["ignore_index"], ptr(k["t"]), ptr(k["m"]), k["alpha"],
            ptr(k["lse3"]), ptr(k["g_px"]), ptr(k["g_sc"]), k["g_mul"], k["variant"], ptr(dx), 0, c["B"], c["C"],
            k["C_old"], c["HW"], cur_stream()), "unce_unkd_bwd")
        terms = [t for t in terms if t is not c and t is not k]
        acc = True
    for t in terms:
        _launch_term(t, dx, acc)
        acc = True
    return dx


def _launch_term(t, dx, acc):
    if t["kind"] == "ce":
        check(_lib.lib().ucd_unce_bwd(ptr(t["x"]), ptr(t["targets"]), ptr(t["lse"][0]), ptr(t["lse"][1]), ptr(t["g_px"]),
                                      ptr(t["g_sc"]), 1.0, ptr(t["stats"]), t["mean_over_valid"], ptr(dx),
                                      1 if acc else 0, t["B"], t["C"], t["old_cl"], t["HW"], t["ignore_index"],
                                      cur_stream()), "unce_bwd")
    else:
        check(_lib.lib().ucd_kd_bwd(ptr(t["x"]), ptr(t["t"]), ptr(t["m"]), t["alpha"], ptr(t["lse3"]), ptr(t["g_px"]),
                                    ptr(t["g_sc"]), t["g_mul"], ptr(dx), 1 if acc else 0, t["B"], t["C"], t["C_old"],
                                    t["HW"], t["variant"], cur_stream()), "kd_bwd")


# ----------------------------------------------------------------------------------------------
# MiB unbiased cross-entropy
# ----------------------------------------------------------------------------------------------
class _UnceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inputs, targets, old_cl, ignore_index, reduction, chain=None, link=None, route=None, src=None,
                probe=None):
        ctx.chain, ctx.is_head, ctx.seq = chain, link is None, (chain.calls if chain is not None else 0)
        ctx.route = route
        ctx.set_materialize_grads(False)   # the link token's gradient stays undefined: no zero tensors, no fill kernels
        B, C = inputs.shape[0], inputs.shape[1]
        HW = inputs.numel() // max(B * C, 1)
        x = _f32c(inputs)
        dev = x.device
        loss_px = torch.empty(targets.shape, device=dev, dtype=torch.float32)
        # ONE saved statistic plane: lse over all channels.  The backward's other need, lse_all - lse_old at label-0
        # pixels, is loss_px itself there (saved below: autograd guards it against in-place changes by the caller)
        lse = torch.empty(targets.shape, device=dev, dtype=torch.float32)
        want_stats = reduction != "none"
        stats = torch.empty(2, device=dev, dtype=torch.float32) if want_stats else None
        scratch = (torch.empty(_lib.lib().ucd_reduce_scratch_floats(), device=dev, dtype=torch.float32)
                   if want_stats else None)
        check(_lib.lib().ucd_unce_fwd(ptr(x), ptr(targets), ptr(loss_px), ptr(lse), None, ptr(stats),
                                      ptr(scratch), B, C, old_cl, HW, ignore_index, cur_stream()), "unce_fwd")
        ctx.save_for_backward(x, targets, lse, stats, loss_px)
        ctx.cfg = (B, C, HW, old_cl, ignore_index, reduction)
        out = loss_px if reduction == "none" else (stats[0].clone() if reduction == "sum" else stats[0] / stats[1])
        if chain is None:
            return out
        # token: orders the chain's backward passes; its value is never read (no fill kernel)
        return out, torch.empty((), device=dev, dtype=torch.float32)

    @staticmethod
    def backward(ctx, g, g_token=None):
        x, targets, lse, stats, loss_px = ctx.saved_tensors
        B, C, HW, old_cl, ignore_index, reduction = ctx.cfg
        if g is None:   # this loss value was not used: only the chain bookkeeping remains
            if ctx.chain is None:
                return (None,) * 10
            d_in, d_link, d_src = ctx.chain.submit(None, ctx.seq, ctx.is_head, ctx.route)
            return d_in, None, None, None, None, None, d_link, None, d_src, None
        g_px, g_sc = None, None
        if reduction == "none":
            g_sc = _scalar_grad(g)
            if g_sc is None:
                g_px = _f32c(g)
        else:
            g_sc = g.reshape(1)
        if g_sc is not None:
            g_sc = _f32c(g_sc)
        term = dict(kind="ce", x=x, targets=targets, lse=(lse, loss_px), stats=stats, g_px=g_px, g_sc=g_sc,
                    mean_over_valid=1 if reduction == "mean" else 0, B=B, C=C, HW=HW, old_cl=old_cl,
                    ignore_index=ignore_index)
        if ctx.chain is None:
            dx = torch.empty_like(x)
            _launch_term(term, dx, False)
            return (dx,) + (None,) * 9
        d_in, d_link, d_src = ctx.chain.submit(term, ctx.seq, ctx.is_head, ctx.route)
        return d_in, None, None, None, None, None, d_link, None, d_src, None


def _chained(fn, inputs, args):
    """Apply the autograd Function `fn` to `inputs`, linked into the gradient chain of that tensor (see _GradChain)."""
    chain = _GradChain.of(inputs)
    if chain is None:
        return fn.apply(inputs, *args)
    route = None
    if chain.token is None:   # the head: it may hand the gradient to the low-res logits directly (_Route)
        route = _Route.of(inputs)
    chain.calls += 1
    if route is None:
        out, token = fn.apply(inputs, *args, chain, chain.token)
    else:
        out, token = fn.apply(inputs, *args, chain, chain.token, *route)
    chain.token = token
    return out


class UnbiasedCrossEntropy(nn.Module):
    """MiB unbiased cross-entropy (utils/loss.py:89-109).  Like the reference it remaps ``targets`` in
    place (labels below ``old_cl`` become 0, loss.py:104-105)."""

    def __init__(self, old_cl=None, reduction='mean', ignore_index=255):
        super().__init__()
        self.reduction = reduction
        self.ignore_index = ignore_index
        self.old_cl = old_cl

    def forward(self, inputs, targets):
        _need_cuda(inputs, targets)
        if self.reduction not in ("none", "mean", "sum"):
            raise ValueError("reduction must be 'none', 'mean' or 'sum'")
        if targets.dtype != torch.int64:
            raise TypeError("UnbiasedCrossEntropy: targets must be int64 (train.py:98 casts labels to long)")
        if inputs.dim() < 2 or targets.shape != inputs.shape[:1] + inputs.shape[2:]:
            raise ValueError("UnbiasedCrossEntropy: inputs [B,C,...] and targets [B,...] shapes disagree")
        old_cl = inputs.shape[1] if self.old_cl is None else int(self.old_cl)  # x[:, 0:None] == all channels
        tgt = targets if targets.is_contiguous() else targets.contiguous()
        out = _chained(_UnceFn, inputs, (tgt, old_cl, int(self.ignore_index), self.reduction))
        if tgt is not targets:
            targets.copy_(tgt)  # keep the in-place remap visible to the caller
        return out


# ----------------------------------------------------------------------------------------------
# MiB unbiased knowledge distillation
# ----------------------------------------------------------------------------------------------
class _UnkdFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, inputs, targets, mask, alpha, reduction, variant=0, chain=None, link=None, route=None, src=None,
                probe=None):
        ctx.chain, ctx.is_head, ctx.seq = chain, link is None, (chain.calls if chain is not None else 0)
        ctx.route = route
        ctx.set_materialize_grads(False)   # see _UnceFn
        B, C, C_old = inputs.shape[0], inputs.shape[1], targets.shape[1]
        HW = inputs.numel() // max(B * C, 1)
        x, t = _f32c(inputs), _f32c(targets)
        m = None if mask is None else _f32c(mask)
        dev = x.device
        px_shape = (B,) + tuple(inputs.shape[2:])
        out_px = torch.empty(px_shape, device=dev, dtype=torch.float32) if reduction == "none" else None
        stats = torch.empty(1, device=dev, dtype=torch.float32)
        lse3 = torch.empty((3,) + px_shape, device=dev, dtype=torch.float32)
        scratch = torch.empty(_lib.lib().ucd_reduce_scratch_floats(), device=dev, dtype=torch.float32)
        # the reduce kernel applies the sign and the 1/(B*HW) of the reduction: no scalar torch kernels afterwards
        scale = -1.0 / float(B * HW) if reduction == "mean" else -1.0
        check(_lib.lib().ucd_kd_fwd(ptr(x), ptr(t), ptr(m), float(alpha), ptr(out_px), ptr(stats), ptr(lse3),
                                    ptr(scratch), B, C, C_old, HW, variant, scale, cur_stream()), "kd_fwd")
        ctx.save_for_backward(x, t, m, lse3)
        ctx.cfg = (B, C, C_old, HW, float(alpha), reduction, variant)
        out = out_px if reduction == "none" else stats[0]
        if chain is None:
            return out
        return out, torch.empty((), device=dev, dtype=torch.float32)   # token: orders the chain's backward passes

    @staticmethod
    def backward(ctx, g, g_token=None):
        x, t, m, lse3 = ctx.saved_tensors
        B, C, C_old, HW, alpha, reduction, variant = ctx.cfg
        if g is None:   # this loss value was not used: only the chain bookkeeping remains
            if ctx.chain is None:
                return (None,) * 11
            d_in, d_link, d_src = ctx.chain.submit(None, ctx.seq, ctx.is_head, ctx.route)
            return d_in, None, None, None, None, None, None, d_link, None, d_src, None
        g_px, g_sc, g_mul = None, None, 1.0
        if reduction == "none":
            g_sc = _scalar_grad(g)
            if g_sc is None:
                g_px = _f32c(g)
        else:
            g_sc = g.reshape(1)
            if reduction == "mean":
                g_mul = 1.0 / float(B * HW)
        if g_sc is not None:
            g_sc = _f32c(g_sc)
        term = dict(kind="kd", x=x, t=t, m=m, lse3=lse3, g_px=g_px, g_sc=g_sc, g_mul=g_mul, alpha=alpha, B=B, C=C,
                    C_old=C_old, HW=HW, variant=variant)
        if ctx.chain is None:
            dx = torch.empty_like(x)
            _launch_term(term, dx, False)
            return (dx,) + (None,) * 10
        d_in, d_link, d_src = ctx.chain.submit(term, ctx.seq, ctx.is_head, ctx.route)
        return d_in, None, None, None, None, None, None, d_link, None, d_src, None


class UnbiasedKnowledgeDistillationLoss(nn.Module):
    """MiB unbiased KD (utils/loss.py:139-184).  ``targets`` (old-model logits) get no gradient, as in
    the reference where they are produced under ``no_grad`` (train.py:100-102)."""

    def __init__(self, reduction='mean', alpha=1.):
        super().__init__()
        self.reduction = reduction
        self.alpha = alpha

    def forward(self, inputs, targets, mask=None):
        _need_cuda(inputs, targets, mask)
        if inputs.shape[1] < targets.shape[1] or inputs.shape[2:] != targets.shape[2:]:
            raise ValueError("UnbiasedKnowledgeDistillationLoss: inputs [B,C,...] / targets [B,C_old,...] disagree")
        if mask is not None and tuple(mask.shape) != (inputs.shape[0],) + tuple(inputs.shape[2:]):
            raise ValueError("UnbiasedKnowledgeDistillationLoss: mask must be [B,...]")
        red = self.reduction if self.reduction in ("mean", "sum") else "none"
        return _chained(_UnkdFn, inputs, (targets.detach(), mask, self.alpha, red, 0))


def _kd_forward(name, variant, self, inputs, targets, mask):
    _need_cuda(inputs, targets, mask)
    if inputs.shape[1] < targets.shape[1] or inputs.shape[2:] != targets.shape[2:]:
        raise ValueError("%s: inputs [B,C,...] / targets [B,C_old,...] disagree" % name)
    if mask is not None and tuple(mask.shape) != (inputs.shape[0],) + tuple(inputs.shape[2:]):
        raise ValueError("%s: mask must be [B,...]" % name)
    red = self.reduction if self.reduction in ("mean", "sum") else "none"
    return _chained(_UnkdFn, inputs, (targets.detach(), mask, self.alpha, red, variant))


class KnowledgeDistillationLoss(nn.Module):
    """Plain KD of the LwF-style baselines (utils/loss.py:112-136): log-softmax over the first C_old channels of
    ``inputs`` against softmax(alpha * targets), averaged over those channels.  Same kernels as the unbiased loss
    (SURVEY section 8(f) N3); the narrowed view is read in place, never copied."""

    def __init__(self, reduction='mean', alpha=1.):
        super().__init__()
        self.reduction = reduction
        self.alpha = alpha

    def forward(self, inputs, targets, mask=None):
        return _kd_forward("KnowledgeDistillationLoss", 1, self, inputs, targets, mask)


class MaskKnowledgeDistillationLoss(nn.Module):
    """Unbiased KD restricted to the pixels where ``mask == 0`` (utils/loss.py:218-256)."""

    def __init__(self, reduction='mean', alpha=1.):
        super().__init__()
        self.reduction = reduction
        self.alpha = alpha

    def forward(self, inputs, targets, mask=None):
        return _kd_forward("MaskKnowledgeDistillationLoss", 2, self, inputs, targets, mask)


class MaskCrossEntropy(nn.Module):
    """utils/loss.py:186-216: unbiased log-probabilities (background = all old classes), labels NOT remapped -
    a label in [1, old_cl) picks the zero-filled channel, i.e. contributes 0 - and, when ``outputs_old`` is given,
    only pixels the old model calls background or whose label is > old_cl count.  Keeps the reference's sign:
    'mean' / 'sum' return the NEGATED reduction (loss.py:213-215; SURVEY Appendix C6), 'none' the positive map."""

    def __init__(self, old_cl=None, reduction='mean', ignore_index=255):
        super().__init__()
        self.reduction = reduction
        self.ignore_index = ignore_index
        self.old_cl = old_cl

    def forward(self, inputs, targets, outputs_old=None):
        _need_cuda(inputs, targets, outputs_old)
        if targets.dtype != torch.int64:
            raise TypeError("MaskCrossEntropy: targets must be int64")
        if inputs.dim() < 2 or targets.shape != inputs.shape[:1] + inputs.shape[2:]:
            raise ValueError("MaskCrossEntropy: inputs [B,C,...] and targets [B,...] shapes disagree")
        if outputs_old is not None and self.old_cl is None:
            raise TypeError("MaskCrossEntropy: old_cl=None cannot be compared with the labels (loss.py:210)")
        old_cl = 0 if self.old_cl is None else int(self.old_cl)  # None: every channel is a plain log-softmax
        ign = int(self.ignore_index)
        # the reference leaves `targets` untouched here; a label in [1, old_cl) must give zero loss and zero gradient
        # (the zero-filled channel): map it to ignore_index in a private copy (torch.where: no host sync)
        if old_cl > 1:
            tgt = torch.where((targets >= 1) & (targets < old_cl), torch.full_like(targets, ign), targets).contiguous()
        else:
            tgt = targets.clone()
        loss = _UnceFn.apply(inputs, tgt, old_cl, ign, "none")
        if outputs_old is not None:
            t = _f32c(outputs_old.detach())
            B, C_old = t.shape[0], t.shape[1]
            mask = torch.empty(targets.shape, device=t.device, dtype=torch.float32)
            lab = targets if targets.is_contiguous() else targets.contiguous()
            check(_lib.lib().ucd_bkg_mask(ptr(t), ptr(lab), ptr(mask), B, C_old, t[0, 0].numel(), old_cl,
                                          cur_stream()), "bkg_mask")
            loss = loss * mask
        if self.reduction == 'mean':
            return -torch.mean(loss)
        if self.reduction == 'sum':
            return -torch.sum(loss)
        return loss


# ----------------------------------------------------------------------------------------------
# contrastive prep
# ----------------------------------------------------------------------------------------------
def payload_layout(max_tiles, kpad):
    """Byte layout of one rank's exchange payload: the ONE contiguous buffer that holds everything another rank needs
    of this rank's contrast columns (SURVEY.md 8e), so that the exchange step is a single all-gather.  Sections are
    256-byte aligned: header int32[4] = {N_a, N_o, min_new, n_px} | tile ranges int32[T,2] | label tiles int32[T,128] |
    probability tiles bf16[T,kpad/8,128,8] | feature tiles bf16[T,32,128,8]."""
    al = lambda n: (n + 255) & ~255  # noqa: E731
    off = {"counts": 0}
    o = 256
    for name, nbytes in (("range", max_tiles * 8), ("lab", max_tiles * TILE * 4), ("prob", max_tiles * kpad * TILE * 2),
                         ("feat", max_tiles * FEAT_DIM * TILE * 2)):
        off[name] = o
        o += al(nbytes)
    off["nbytes"] = o
    return off


def payload_views(buf, max_tiles, kpad):
    """Typed views into a payload buffer ``buf`` uint8 [..., nbytes] (one rank's, or the gathered [W, nbytes])."""
    lay = payload_layout(max_tiles, kpad)
    assert buf.dtype == torch.uint8 and buf.shape[-1] == lay["nbytes"]

    def sec(name, nbytes, dtype, shape):
        v = buf[..., lay[name]:lay[name] + nbytes].view(dtype)
        return v.unflatten(-1, shape)
    T = max_tiles
    return dict(counts=sec("counts", 16, torch.int32, (4,)), range=sec("range", T * 8, torch.int32, (T, 2)),
                lab=sec("lab", T * TILE * 4, torch.int32, (T, TILE)),
                prob=sec("prob", T * kpad * TILE * 2, torch.bfloat16, (T, kpad // 8, TILE, 8)),
                feat=sec("feat", T * FEAT_DIM * TILE * 2, torch.bfloat16, (T, FEAT_DIM // 8, TILE, 8)))


class ContrastPack:
    """Device-side product of the prep kernels for one batch: bf16 operand tiles for the tensor-core
    sweeps plus the metadata the backward needs.  Shared by the 5 tuple slots."""

    def __init__(self):
        self.n_px = 0
        self.shape = None          # (B, h, w)
        self.c_old = 0
        self.kpad = 0
        self.max_tiles = 0
        self.payload = None        # uint8 [payload_layout(...)["nbytes"]]: counts + range + lab + prob + feat tiles
        self.addr = None           # device address of every payload section (what the C calls take)
        self._views = None         # typed tensor views of the sections, built on first use (15 tensor ops: kept off
                                   # the host's critical path between the prep kernels and the next loss module)
        self.n_a = self.n_o = self.min_new = None   # host copies (one sync)
        self.px_meta = self.blk_meta = None         # see include/ucd_b200.h (ucd_con_prep_labels)
        self.label_n = self.mix = self.flags = None  # views of px_meta planes 0..2
        self.anchor_f32 = self.contrast_f32 = None   # reference row order (b,y,x)
        self.la = self.lc = None
        # feat_tiles / prob_tiles / lab_tiles (class-sorted bf16 / int32 tiles), tile_range ([T,2] min/max label per
        # column tile) and counts (int32[4] device: N_a, N_o, min_new, n_px) are properties: views into the payload
        self.row_range = None                        # [ceil(n_px/128),2] same over the anchor rows only
        self.row_ref = self.inv_norm = None          # sorted anchor row -> reference row
        self.max_label = 20
        self.l_po = None
        self.bf16_feats = False    # the head features arrived (and their gradient leaves) in bf16

    @property
    def n_c(self):
        return self.n_a + self.n_o

    def _view(self, name):
        if self._views is None:
            self._views = payload_views(self.payload, self.max_tiles, self.kpad)
        return self._views[name]

    counts = property(lambda self: self._view("counts"))
    tile_range = property(lambda self: self._view("range"))
    lab_tiles = property(lambda self: self._view("lab"))
    prob_tiles = property(lambda self: self._view("prob"))
    feat_tiles = property(lambda self: self._view("feat"))


_PINNED = {}


def _pinned_counts(dev):
    """Per-device pinned int32[4] staging buffer for the {N_a, N_o, min_new, n_px} read-back."""
    key = (dev.type, dev.index)
    buf = _PINNED.get(key)
    if buf is None:
        buf = _PINNED[key] = torch.empty(4, dtype=torch.int32).pin_memory()
    return buf


def _multi_rank():
    import torch.distributed as dist
    return dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1


def _build_pack(f_n, f_o, l_po, labels, max_label, sync=True, require_new_class=True):
    _need_cuda(f_n, f_o, l_po, labels)
    if f_n.dim() != 4 or f_n.shape[1] != FEAT_DIM or f_o.shape != f_n.shape:
        raise ValueError("pre_contrastive_pixel: f_n / f_o must be [B,%d,h,w]" % FEAT_DIM)
    B, _, h, w = f_n.shape
    if l_po.dim() != 4 or l_po.shape[0] != B or tuple(l_po.shape[2:]) != (h, w):
        raise ValueError("pre_contrastive_pixel: l_po must be [B,C_old,h,w]")
    if labels.dim() != 3 or labels.shape[0] != B:
        raise ValueError("pre_contrastive_pixel: l_n must be [B,H,W]")
    L = _lib.lib()
    dev = f_n.device
    labels = labels.to(torch.int64).contiguous()
    # N2 (feature hand-off): a head that runs in bf16 hands its features over as they are - the pack kernel reads bf16
    # NCHW directly (no fp32 copy of the two feature maps) and the adjoint writes the bf16 gradient
    bf16_feats = f_n.dtype == torch.bfloat16 and f_o.dtype == torch.bfloat16
    if bf16_feats:
        f_n, f_o = f_n.contiguous(), f_o.contiguous()
    else:
        f_n, f_o = _f32c(f_n), _f32c(f_o)
    l_po = _f32c(l_po)
    H, W = labels.shape[-2:]
    pk = ContrastPack()
    pk.bf16_feats = bf16_feats
    pk.shape, pk.n_px, pk.c_old = (B, h, w), B * h * w, l_po.shape[1]
    pk.kpad = L.ucd_con_prob_kpad(pk.c_old)
    pk.max_tiles = L.ucd_con_max_tiles(pk.n_px)
    n_px = pk.n_px
    i32 = dict(device=dev, dtype=torch.int32)
    pk.max_label = int(max_label)
    nb = L.ucd_con_num_bins(pk.max_label, pk.c_old)
    pk.px_meta = torch.empty(7, n_px, **i32)
    pk.label_n, pk.mix, pk.flags = pk.px_meta[0], pk.px_meta[1], pk.px_meta[2]
    pk.blk_meta = torch.empty(L.ucd_con_blk_meta_ints(n_px, nb), **i32)
    # everything another rank needs of this rank's columns lives in ONE buffer (the exchange payload); the kernels
    # write their outputs straight into its sections
    lay = payload_layout(pk.max_tiles, pk.kpad)
    pk.payload = torch.empty(lay["nbytes"], device=dev, dtype=torch.uint8)
    base = pk.payload.data_ptr()
    ad = pk.addr = {k: base + lay[k] for k in ("counts", "range", "lab", "prob", "feat")}
    st = cur_stream()
    # The tuple API needs N_a / N_o on the host (tensor shapes).  The scan kernel stores them straight into mapped
    # pinned host memory (no D2H copy that could queue behind other transfers on the copy engine); the host waits
    # for the event only after the pack kernels are queued, so the GPU has work while the host catches up.
    counts_host = _pinned_counts(dev)
    check(L.ucd_con_prep_labels(ptr(labels), ptr(l_po), B, pk.c_old, h, w, H, W, pk.max_label, ptr(pk.px_meta),
                                ptr(pk.blk_meta), ad["counts"], counts_host.data_ptr(), st), "con_prep_labels")
    copied = None
    if sync:
        copied = torch.cuda.Event()
        copied.record()
    pk.anchor_f32 = torch.empty(n_px, FEAT_DIM, device=dev, dtype=torch.float32)
    pk.contrast_f32 = torch.empty(2 * n_px, FEAT_DIM, device=dev, dtype=torch.float32)
    # the tuple's label vectors come out of the pack kernel in their final type; they hold GT labels (<= max_label)
    # and pseudo labels (old-model argmax, <= C_old - 1)
    ldt = _label_dtype(max(pk.max_label, pk.c_old - 1))
    pk.la = torch.empty(n_px, device=dev, dtype=ldt)
    pk.lc = torch.empty(2 * n_px, device=dev, dtype=ldt)
    pk.row_range = torch.empty((n_px + TILE - 1) // TILE, 2, **i32)
    pk.row_ref = torch.empty(n_px, **i32)
    pk.inv_norm = torch.empty(n_px, device=dev, dtype=torch.float32)
    pack_fn = L.ucd_con_prep_pack_bf16 if bf16_feats else L.ucd_con_prep_pack
    check(pack_fn(ptr(f_n), ptr(f_o), ptr(l_po), ptr(pk.px_meta), ptr(pk.blk_meta), ad["counts"], B,
                  pk.c_old, h, w, pk.max_label, ptr(pk.anchor_f32), ptr(pk.contrast_f32), ptr(pk.la),
                  ptr(pk.lc), pk.la.element_size(), ad["feat"], ad["prob"], ad["lab"],
                  ad["range"], ptr(pk.row_range), ptr(pk.row_ref), ptr(pk.inv_norm),
                  pk.max_tiles, st),
          "con_prep_pack")
    pk.l_po = l_po
    if not sync:  # sync-free path: N_a / N_o stay on the device, buffers keep their worst-case sizes
        return pk
    # the one host sync of the tuple API: the 5-tuple's tensor shapes depend on N_a / N_o
    copied.synchronize()
    pk.n_a, pk.n_o, pk.min_new, _ = (int(v) for v in counts_host.tolist())
    if require_new_class and pk.n_a > 0 and pk.min_new > max(int(max_label), 0):
        # no GT new-class pixel in the batch: the reference raises at utils/loss.py:355 (min() of empty)
        raise RuntimeError("pre_contrastive_pixel: no new-class pixel in the batch "
                           "(the reference raises here too, utils/loss.py:355)")
    return pk


class _AnchorFn(torch.autograd.Function):
    """Autograd link f_n -> Output_anchor (gather of anchor pixels + F.normalize, loss.py:363-365)."""

    @staticmethod
    def forward(ctx, f_n, pack):
        ctx.pack = pack
        ctx.in_dtype = f_n.dtype
        return pack.anchor_f32[:pack.n_a]

    @staticmethod
    def backward(ctx, g):
        pk = ctx.pack
        B, h, w = pk.shape
        g = _f32c(g)
        if pk.n_a == 0:   # no anchor in this batch: nothing flows back
            return torch.zeros(B, FEAT_DIM, h, w, device=g.device, dtype=ctx.in_dtype), None
        direct_bf16 = pk.bf16_feats and ctx.in_dtype == torch.bfloat16
        df = torch.empty(B, FEAT_DIM, h, w, device=g.device, dtype=torch.bfloat16 if direct_bf16 else torch.float32)
        bwd_fn = _lib.lib().ucd_con_prep_bwd_bf16 if direct_bf16 else _lib.lib().ucd_con_prep_bwd
        check(bwd_fn(ptr(g), ptr(pk.anchor_f32), ptr(pk.inv_norm), ptr(pk.px_meta),
                     ptr(pk.blk_meta), ptr(df), B, h, w, cur_stream()), "con_prep_bwd")
        return df.to(ctx.in_dtype), None


class JointProb:
    """Lazy stand-in for the reference's dense ``JM_p`` [N_a, N_c] (utils/loss.py:369-395): it carries
    the bf16 softmax tiles and the GT-new threshold so that ``PixelConLossV2`` evaluates
    P_ij = p_i.p_j (or 1 for GT-new x GT-new pairs) tile by tile on the tensor cores.  ``dense()``
    materialises the fp32 matrix for inspection / compatibility."""

    def __init__(self, pack):
        self.pack = pack

    @property
    def shape(self):
        return (self.pack.n_a, self.pack.n_c)

    def dense(self):
        pk = self.pack
        B, h, w = pk.shape
        p = torch.softmax(pk.l_po.permute(0, 2, 3, 1).reshape(pk.n_px, pk.c_old), dim=1)
        anchor = (pk.flags & 1).bool()
        pseudo = (pk.flags & 2).bool()
        pa = p[anchor]
        pc = torch.cat([pa, p[pseudo]])
        P = pa @ pc.T
        la, lc = pk.la[:pk.n_a].to(torch.int32), pk.lc[:pk.n_c].to(torch.int32)
        P[(la >= pk.min_new)[:, None] & (lc >= pk.min_new)[None, :]] = 1.0
        return P

    def detach(self):
        return self


def _label_dtype(max_label):
    return torch.int8 if max_label <= 127 else torch.int32


class _RowsFn(torch.autograd.Function):
    """Every pixel of f [B,256,h,w] as a unit-norm row [B*h*w, 256] (utils/loss.py:273-276 + F.normalize)."""

    @staticmethod
    def forward(ctx, f):
        x = _f32c(f)
        B, D, h, w = x.shape
        rows = torch.empty(B * h * w, D, device=x.device, dtype=torch.float32)
        inv = torch.empty(B * h * w, device=x.device, dtype=torch.float32)
        check(_lib.lib().ucd_rows_normalize_fwd(ptr(x), ptr(rows), ptr(inv), B, h, w, cur_stream()), "rows_normalize_fwd")
        ctx.save_for_backward(rows, inv)
        ctx.shape, ctx.in_dtype = (B, D, h, w), f.dtype
        return rows

    @staticmethod
    def backward(ctx, g):
        rows, inv = ctx.saved_tensors
        B, D, h, w = ctx.shape
        df = torch.empty(B, D, h, w, device=g.device, dtype=torch.float32)
        check(_lib.lib().ucd_rows_normalize_bwd(ptr(_f32c(g)), ptr(rows), ptr(inv), ptr(df), B, h, w, cur_stream()),
              "rows_normalize_bwd")
        return df.to(ctx.in_dtype)


def _pixel_to_pixel(f_n, l_n, f_o, max_label):
    """The branches of utils/loss.py:278-289 (no old-model logits): all pixels, labels = the clamped low-res label map."""
    _need_cuda(f_n, l_n, f_o)
    if f_n.dim() != 4 or f_n.shape[1] != FEAT_DIM or (f_o is not None and f_o.shape != f_n.shape):
        raise ValueError("pre_contrastive_pixel: f_n / f_o must be [B,%d,h,w]" % FEAT_DIM)
    B, _, h, w = f_n.shape
    if l_n.dim() != 3 or l_n.shape[0] != B:
        raise ValueError("pre_contrastive_pixel: l_n must be [B,H,W]")
    L = _lib.lib()
    dev = f_n.device
    labels = l_n.to(torch.int64).contiguous()
    H, W = labels.shape[-2:]
    n_px = B * h * w
    i32 = dict(device=dev, dtype=torch.int32)
    # the label kernel of the v2 path with a one-channel dummy old-model map (its argmax is 0 everywhere): plane 0 of
    # px_meta is the reference's label_n (bilinear downsample, truncation, clamp to [0, max_label]; loss.py:261-270)
    px_meta = torch.empty(7, n_px, **i32)
    blk_meta = torch.empty(L.ucd_con_blk_meta_ints(n_px, L.ucd_con_num_bins(int(max_label), 1)), **i32)
    counts = torch.empty(4, **i32)
    dummy = torch.zeros(B, 1, h, w, device=dev, dtype=torch.float32)
    check(L.ucd_con_prep_labels(ptr(labels), ptr(dummy), B, 1, h, w, H, W, int(max_label), ptr(px_meta), ptr(blk_meta),
                                ptr(counts), None, cur_stream()), "con_prep_labels")
    lab = px_meta[0].to(_label_dtype(int(max_label)))
    out = _RowsFn.apply(f_n)
    if f_o is not None:   # "pixel to pixel double": new-model rows, then the (detached) old-model rows
        out = torch.cat((out, _RowsFn.apply(f_o.detach())), dim=0)
        lab = torch.cat((lab, lab))
    return out.unsqueeze(1), lab


def pre_contrastive_pixel(f_n, l_n, l_po=None, f_o=None, max_label=20, require_new_class=None):
    """Drop-in for utils/loss.py:258 ``pre_contrastive_pixel``.

    With ``l_po`` and ``f_o`` (the v2 branch ``train.py`` reaches) it returns the 5-tuple ``(Output_anchor,
    Output_contrast, Lable_anchor, Lable_contrast, JM_p)`` in the reference's row order; ``JM_p`` is a
    :class:`JointProb` handle (call ``.dense()`` for the matrix).  Without ``l_po`` it returns ``(Output.unsqueeze(1),
    Lable)`` of the pixel-to-pixel branches (loss.py:278-289: all pixels; with ``f_o`` the old-model rows are appended).
    ``l_po`` without ``f_o`` raises like the reference does (its ``Output`` is undefined there, loss.py:399).
    ``max_label`` generalises the reference's hard-coded VOC clamp ``label_n > 20 -> 0`` (loss.py:270).

    ``require_new_class``: the reference raises when the batch holds no new-class pixel (``min()`` of an empty tensor,
    loss.py:355).  True keeps that; False never raises (the GT-new override of P then simply never fires).  The default
    None means True in a single process and False when a multi-rank process group is initialised: there one rank
    raising alone would leave the other ranks blocked in the exchange collectives of ``PixelConLossV2(gather_negatives
    =True)``, and the threshold that matters is the global minimum anyway.
    """
    if l_po is None:
        return _pixel_to_pixel(f_n, l_n, f_o, max_label)
    if f_o is None:
        raise UnboundLocalError("pre_contrastive_pixel: l_po without f_o is undefined in the reference too "
                                "(utils/loss.py:399 returns an unassigned `Output`)")
    if require_new_class is None:
        require_new_class = not _multi_rank()
    pack = _build_pack(f_n.detach(), f_o.detach(), l_po.detach(), l_n, max_label, require_new_class=require_new_class)
    anchor = _AnchorFn.apply(f_n, pack)
    anchor._ucd_pack = pack   # lets PixelConLossV2 recognise the tensor it may run the packed operands for
    out = (anchor, pack.contrast_f32[:pack.n_c], pack.la[:pack.n_a], pack.lc[:pack.n_c], JointProb(pack))
    return out


pre_contractive_pixel = pre_contrastive_pixel  # spelling used by utils/utils.py:256 and train.py:9


# ----------------------------------------------------------------------------------------------
# PixelConLossV2
# ----------------------------------------------------------------------------------------------
def _local_cols(pack):
    """Column-side arguments of the sweeps for this rank's own pack (single chunk)."""
    ad = pack.addr   # raw section addresses: no tensor views on the hot path (ptr() takes ints)
    return dict(feat=ad["feat"], prob=ad["prob"], lab=ad["lab"], range=ad["range"],
                counts=ad["counts"], n_chunks=1, chunk_tiles=pack.max_tiles, kpad=pack.kpad, min_new=ad["counts"] + 8,
                payload=pack.payload)


def gather_contrast_columns(payload, max_tiles, kpad, group, async_op=False):
    """The one exchange step of the data-parallel path (SURVEY.md 8e): a SINGLE all-gather of every rank's payload
    (:func:`payload_layout`); rank r's columns become chunk r of the gathered buffer.  ``max_tiles`` / ``kpad`` must be
    equal on all ranks (same per-rank pixel count and old-class count).

    Returns dict(buf [W, nbytes] uint8, feat / prob / lab / range / counts = typed views [W, ...], n_chunks,
    chunk_tiles, chunk_stride (bytes), self_tile0, work).  The global GT-new threshold is the minimum of
    ``counts[:, 2]`` - the sweeps take it from the headers, no MIN all-reduce.  With ``async_op=True`` the collective is
    only enqueued (NCCL stream) and ``work.wait()`` must be called before the gathered buffer is consumed: sweep 1 over
    the LOCAL columns runs in between.  No gradient flows through the gathered columns (they are detached in the
    reference, loss.py:366,395), so backward needs no collective."""
    import torch.distributed as dist
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    payload = payload.contiguous()
    buf = torch.empty(world, payload.numel(), device=payload.device, dtype=torch.uint8)
    work = dist.all_gather_into_tensor(buf.view(-1), payload, group=group, async_op=async_op)
    out = payload_views(buf, max_tiles, kpad)
    out.update(buf=buf, n_chunks=world, chunk_tiles=max_tiles, chunk_stride=payload.numel(),
               self_tile0=rank * max_tiles, rank=rank, work=work if async_op else None)
    return out


class _ConFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, anchor, cols, rows, inv_tau, p_mode, dense_p, group, ddp_scale):
        """cols / rows: dicts of device buffers (see PixelConLossV2.forward).  With a process group, ``cols`` holds the
        LOCAL payload; the all-gather of all ranks' payloads is enqueued first and sweep 1 over the local columns runs
        while it is in flight."""
        L = _lib.lib()
        dev = anchor.device
        max_row_tiles = rows["max_tiles"]
        plan_tiles = rows.get("plan_tiles", 0)
        out = torch.empty(3, device=dev, dtype=torch.float32)
        need_grad = bool(ctx.needs_input_grad[0])
        grad_unit = (torch.empty(max_row_tiles * TILE, FEAT_DIM, device=dev, dtype=torch.float32)
                     if need_grad else None)

        def run(c, part, n_chunks, stride, local_chunk, self_tile0, ws, ws_bytes):
            check(L.ucd_con_fwd(ptr(c["feat"]), ptr(c["prob"]), ptr(c["lab"]), ptr(c["counts"]), n_chunks,
                                c["chunk_tiles"], stride, local_chunk, part, ptr(rows["feat"]), ptr(rows["prob"]),
                                ptr(rows["lab"]), ptr(rows["n_rows"]), ptr(c["range"]), ptr(rows["range"]),
                                self_tile0, ptr(c["min_new"]), p_mode, c["kpad"], ptr(dense_p),
                                0 if dense_p is None else dense_p.shape[1], inv_tau, 1 if need_grad else 0, ptr(out),
                                ptr(grad_unit), ptr(ws), ws_bytes, max_row_tiles, plan_tiles, cur_stream()),
                  "con_fwd")

        if group is None:
            ws_bytes = L.ucd_con_workspace_bytes(max_row_tiles, cols["n_chunks"] * cols["chunk_tiles"], plan_tiles, 0)
            ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
            run(cols, 0, cols["n_chunks"], 0, -1, rows["self_tile0"], ws, ws_bytes)
        else:
            # one all-gather of the payloads, overlapped with sweep 1 over the local columns
            g = gather_contrast_columns(cols["payload"], cols["chunk_tiles"], cols["kpad"], group, async_op=True)
            world, rank, T = g["n_chunks"], g["rank"], cols["chunk_tiles"]
            ws_bytes = L.ucd_con_workspace_bytes(max_row_tiles, world * T, plan_tiles, T)
            ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
            run(cols, 1, world, g["chunk_stride"], rank, g["self_tile0"], ws, ws_bytes)
            g["work"].wait()   # the current stream waits for the gathered buffer; the host does not
            gc = dict(feat=g["feat"][0], prob=g["prob"][0], lab=g["lab"][0], range=g["range"][0],
                      counts=g["counts"][0], min_new=g["counts"][0, 2:3], chunk_tiles=T, kpad=cols["kpad"])
            run(gc, 2, world, g["chunk_stride"], rank, g["self_tile0"], ws, ws_bytes)
            ctx.gathered = g["buf"]   # keep the buffer alive until the kernels that read it have run
        world = 1
        if group is not None:
            import torch.distributed as dist
            dist.all_reduce(out[:2], group=group)  # {sum of row losses, #valid rows} over all ranks
            world = dist.get_world_size(group)
        n_rows = rows["n_rows"]
        if isinstance(n_rows, int):   # a device address inside the pack's payload: keep that buffer alive instead
            ctx.n_rows_addr, ctx.keep = n_rows, rows.get("keep")
            ctx.save_for_backward(grad_unit, out, None, rows.get("row_ref"))
        else:
            ctx.n_rows_addr = None
            ctx.save_for_backward(grad_unit, out, n_rows, rows.get("row_ref"))
        ctx.static_pack = rows.get("static_pack")   # sync-free path: `anchor` is f_n itself
        ctx.n_a = anchor.shape[0] if ctx.static_pack is None else ctx.static_pack.n_px
        ctx.in_dtype = anchor.dtype
        ctx.world = world if ddp_scale else 1
        if group is not None:
            return out[0] / out[1]
        return out[2]  # the ratio comes from the reduce kernel: no extra launch

    @staticmethod
    def backward(ctx, g):
        grad_unit, out, n_rows, row_ref = ctx.saved_tensors
        if ctx.n_rows_addr is not None:
            n_rows = ctx.n_rows_addr
        d_anchor = torch.empty(ctx.n_a, FEAT_DIM, device=g.device, dtype=torch.float32)
        if ctx.n_a == 0:   # a rank without anchors (it only took part in the collectives)
            return d_anchor.to(ctx.in_dtype), None, None, None, None, None, None, None
        # With DDP averaging parameter gradients over ranks, the exact gradient of the global-batch loss needs
        # each rank's local contribution scaled by world (columns carry no gradient, loss.py:366,395).
        check(_lib.lib().ucd_con_bwd(ptr(grad_unit), ptr(out), ptr(_f32c(g.reshape(1))), float(ctx.world),
                                     ptr(n_rows), ptr(row_ref), ptr(d_anchor), ctx.n_a, cur_stream()), "con_bwd")
        pk = ctx.static_pack
        if pk is not None:  # continue through the anchor gather + normalise adjoint to f_n (rows >= N_a are never read)
            B, h, w = pk.shape
            direct_bf16 = pk.bf16_feats and ctx.in_dtype == torch.bfloat16
            df = torch.empty(B, FEAT_DIM, h, w, device=g.device,
                             dtype=torch.bfloat16 if direct_bf16 else torch.float32)
            bwd_fn = _lib.lib().ucd_con_prep_bwd_bf16 if direct_bf16 else _lib.lib().ucd_con_prep_bwd
            check(bwd_fn(ptr(d_anchor), ptr(pk.anchor_f32), ptr(pk.inv_norm), ptr(pk.px_meta),
                         ptr(pk.blk_meta), ptr(df), B, h, w, cur_stream()), "con_prep_bwd")
            d_anchor = df.to(ctx.in_dtype)
        return d_anchor, None, None, None, None, None, None, None


class PixelConLossV2(nn.Module):
    """Supervised pixel contrastive loss with uncertainty (joint-probability) weights
    (utils/loss.py:403-466), evaluated by the fused sm_100a sweeps without materialising any
    N_a x N_c matrix.

    ``forward(anchor_features, contrast_feature, anchor_labels, contrast_labels, P=None)`` accepts the
    tuple returned by :func:`pre_contrastive_pixel` (fast path: operands are already packed) or plain
    dense tensors / ``P=None`` / a dense ``P`` matrix (compat path: packed on the fly).

    Extension (SURVEY.md 8e): with ``gather_negatives=True`` and an initialised process group the
    contrast columns of all ranks are all-gathered over NCCL so negatives span the global batch.
    """

    def __init__(self, sample_method='none', temperature=0.07, *, gather_negatives=False, process_group=None,
                 ddp_grad_scale=True):
        super(PixelConLossV2, self).__init__()
        self.temperature = temperature
        self.sample_method = sample_method
        self.gather_negatives = gather_negatives
        self.process_group = process_group
        # under DDP's gradient averaging the exact global-batch gradient needs the local part scaled by world
        self.ddp_grad_scale = ddp_grad_scale
        self.max_dense_bytes = 2 << 30   # largest dense P the compat fallback may materialise (see forward)
        print(temperature)  # the reference prints it on construction (utils/loss.py:410)

    # -- helpers ---------------------------------------------------------------------------------
    def _group(self):
        if not self.gather_negatives:
            return None
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return None
        g = self.process_group if self.process_group is not None else dist.group.WORLD
        return g if dist.get_world_size(g) > 1 else None

    def forward(self, anchor_features, contrast_feature, anchor_labels, contrast_labels, P=None):
        _need_cuda(anchor_features, contrast_feature)
        inv_tau = 1.0 / float(self.temperature)
        L = _lib.lib()
        dev = anchor_features.device
        pack = P.pack if isinstance(P, JointProb) else None
        # the tuple's first slot carries its pack; a view of the packed rows is accepted too (an empty tensor has no
        # data pointer, so N_a == 0 is decided by the tag or the shape alone)
        own = pack is not None and (getattr(anchor_features, "_ucd_pack", None) is pack or (
            anchor_features.dtype == torch.float32 and tuple(anchor_features.shape) == (pack.n_a, FEAT_DIM)
            and (pack.n_a == 0 or anchor_features.data_ptr() == pack.anchor_f32.data_ptr())))
        if pack is not None and not own:
            # the handle came with other features than the ones it was packed from (a cast, clone or slice of the
            # anchors): the sweeps must run on the caller's values, so the operands are re-packed (compat path) and P
            # is materialised - N_a x N_c fp32.  Never silently: this is ~1000x the memory of the fused path.
            import warnings
            n_bytes = 4.0 * pack.n_a * pack.n_c
            msg = ("PixelConLossV2: anchor_features is not the tensor pre_contrastive_pixel returned (cast / clone / "
                   "slice?): falling back to a dense %d x %d joint-probability matrix (%.2f GB).  Pass the tuple "
                   "through unchanged, or use PixelContrastiveDistillation." % (pack.n_a, pack.n_c, n_bytes / 1e9))
            if n_bytes > self.max_dense_bytes:
                raise RuntimeError(msg + "  Refusing: above max_dense_bytes=%d." % self.max_dense_bytes)
            warnings.warn(msg, RuntimeWarning, stacklevel=2)
            P, pack = P.dense(), None
        if pack is not None:
            # ---- fast path: operands packed by pre_contrastive_pixel ----
            group = self._group()
            ad = pack.addr
            rows = dict(feat=ad["feat"], prob=ad["prob"], lab=ad["lab"], n_rows=ad["counts"], keep=pack.payload,
                        range=pack.row_range, row_ref=pack.row_ref, max_tiles=max(1, (pack.n_a + TILE - 1) // TILE),
                        self_tile0=0)
            cols = _local_cols(pack)
            if pack.n_a == 0 and group is None:
                return anchor_features.sum() * 0.0
            # with a process group every rank must take part in the collectives, anchors or not: the kernels exit for
            # row blocks beyond N_a and this rank then contributes {0, 0} to the global sums
            return _ConFn.apply(anchor_features, cols, rows, inv_tau, 1, None, group, self.ddp_grad_scale)

        # ---- compat path: dense caller-supplied tensors ----
        if anchor_features.dim() != 2 or anchor_features.shape[1] != FEAT_DIM or contrast_feature.shape[1] != FEAT_DIM:
            raise ValueError("PixelConLossV2: features must be [N,%d]" % FEAT_DIM)
        n_a, n_c = anchor_features.shape[0], contrast_feature.shape[0]
        if n_a == 0 or n_c == 0:
            return anchor_features.sum() * 0.0
        if contrast_feature.requires_grad and torch.is_grad_enabled():
            # the reference back-propagates through contrast_feature when it carries a graph (utils/loss.py:445-466);
            # the sweeps only form d loss / d anchor_features (the v2 prep detaches the contrast side, loss.py:366)
            raise RuntimeError("PixelConLossV2: contrast_feature requires grad, but this implementation only "
                               "differentiates w.r.t. anchor_features (the UCD prep detaches the contrast side, "
                               "utils/loss.py:366); pass contrast_feature.detach() if that is what you mean")
        a32, c32 = _f32c(anchor_features.detach()), _f32c(contrast_feature.detach())
        la = anchor_labels.reshape(-1).to(device=dev, dtype=torch.int32).contiguous()
        lc = contrast_labels.reshape(-1).to(device=dev, dtype=torch.int32).contiguous()
        if la.numel() != n_a or lc.numel() != n_c:
            raise ValueError("PixelConLossV2: label / feature counts disagree")
        rt, ct = (n_a + TILE - 1) // TILE, (n_c + TILE - 1) // TILE
        bf = dict(device=dev, dtype=torch.bfloat16)
        rfeat = torch.empty(rt, FEAT_DIM // 8, TILE, 8, **bf)
        cfeat = torch.empty(ct, FEAT_DIM // 8, TILE, 8, **bf)
        rlab = torch.empty(rt, TILE, device=dev, dtype=torch.int32)
        clab = torch.empty(ct, TILE, device=dev, dtype=torch.int32)
        st = cur_stream()
        check(L.ucd_con_pack_rows(ptr(a32), ptr(la), n_a, ptr(rfeat), ptr(rlab), rt, st), "con_pack_rows")
        check(L.ucd_con_pack_rows(ptr(c32), ptr(lc), n_c, ptr(cfeat), ptr(clab), ct, st), "con_pack_rows")
        rrange = torch.empty(rt, 2, device=dev, dtype=torch.int32)
        crange = torch.empty(ct, 2, device=dev, dtype=torch.int32)
        check(L.ucd_con_tile_ranges(ptr(rlab), rt, None, ptr(rrange), st), "con_tile_ranges")
        check(L.ucd_con_tile_ranges(ptr(clab), ct, None, ptr(crange), st), "con_tile_ranges")
        counts = torch.tensor([[n_c, 0]], device=dev, dtype=torch.int32)
        n_rows = torch.tensor([n_a], device=dev, dtype=torch.int32)
        dense_p, p_mode = None, 0
        if P is not None:
            if tuple(P.shape) != (n_a, n_c):
                raise ValueError("PixelConLossV2: P must be [N_a, N_c]")
            dense_p, p_mode = _f32c(P.detach()), 2
        cols = dict(feat=cfeat, prob=None, lab=clab, range=crange, counts=counts, n_chunks=1, chunk_tiles=ct, kpad=16,
                    min_new=None)
        rows = dict(feat=rfeat, prob=None, lab=rlab, range=rrange, n_rows=n_rows, max_tiles=rt, self_tile0=0)
        return _ConFn.apply(anchor_features, cols, rows, inv_tau, p_mode, dense_p, None, False)


# ----------------------------------------------------------------------------------------------
# N3: the self-contrast siblings of utils/loss_new.py (PixelConLoss v1, SupConLoss) on the same sweeps
# ----------------------------------------------------------------------------------------------
class _SelfConFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, rows, labels, mode, n_anchor, inv_tau, kappa):
        """rows [n, D <= 256] (any float dtype), labels [n] integer (>= 0); mode 0 = PixelConLoss v1, 1 = SupConLoss."""
        L = _lib.lib()
        dev = rows.device
        n, D = rows.shape
        x = _f32c(rows.detach())
        if D < FEAT_DIM:   # zero columns change no dot product
            x = torch.nn.functional.pad(x, (0, FEAT_DIM - D))
        lab = labels.to(device=dev, dtype=torch.int32).contiguous()
        tiles = (n + TILE - 1) // TILE
        feat = torch.empty(tiles, FEAT_DIM // 8, TILE, 8, device=dev, dtype=torch.bfloat16)
        ltile = torch.empty(tiles, TILE, device=dev, dtype=torch.int32)
        rng = torch.empty(tiles, 2, device=dev, dtype=torch.int32)
        st = cur_stream()
        check(L.ucd_con_pack_rows(ptr(x), ptr(lab), n, ptr(feat), ptr(ltile), tiles, st), "con_pack_rows")
        check(L.ucd_con_tile_ranges(ptr(ltile), tiles, None, ptr(rng), st), "con_tile_ranges")
        meta = torch.tensor([n, 0, n], device=dev, dtype=torch.int32)   # {columns, 0} | rows
        need_grad = bool(ctx.needs_input_grad[0])
        out = torch.empty(3, device=dev, dtype=torch.float32)
        grad_unit = torch.empty(n, FEAT_DIM, device=dev, dtype=torch.float32) if need_grad else None
        ws_bytes = L.ucd_selfcon_workspace_bytes(tiles)
        ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
        check(L.ucd_selfcon_fwd(ptr(feat), ptr(ltile), ptr(rng), ptr(meta), meta.data_ptr() + 8, n, n_anchor, mode,
                                inv_tau, kappa, 1 if need_grad else 0, ptr(out), ptr(grad_unit), ptr(ws), ws_bytes, st),
              "selfcon_fwd")
        ctx.save_for_backward(grad_unit, out, meta)
        ctx.shape, ctx.in_dtype = (n, D), rows.dtype
        return out[2]

    @staticmethod
    def backward(ctx, g):
        grad_unit, out, meta = ctx.saved_tensors
        n, D = ctx.shape
        d = torch.empty(n, FEAT_DIM, device=g.device, dtype=torch.float32)
        check(_lib.lib().ucd_con_bwd(ptr(grad_unit), ptr(out), ptr(_f32c(g.reshape(1))), 1.0, meta.data_ptr() + 8, None,
                                     ptr(d), n, cur_stream()), "con_bwd")
        return d[:, :D].to(ctx.in_dtype), None, None, None, None, None


def _selfcon_rows(features, what):
    if features.dim() < 3:
        raise ValueError('`features` needs to be [bsz, n_views, ...],'
                         'at least 3 dimensions are required')
    _need_cuda(features)
    feats = features.reshape(features.shape[0], features.shape[1], -1)
    if feats.shape[2] > FEAT_DIM:
        raise NotImplementedError("%s: feature width %d > %d is not supported by the sweep kernels"
                                  % (what, feats.shape[2], FEAT_DIM))
    # torch.cat(torch.unbind(features, dim=1), dim=0): view-major rows (loss_new.py:309,383)
    return feats, feats.transpose(0, 1).reshape(-1, feats.shape[2])


class PixelConLoss(nn.Module):
    """``PixelConLoss`` (v1) of utils/loss_new.py:354-400: supervised contrastive loss of a pixel set with itself (the
    output of the pixel-to-pixel branches of ``pre_contrastive_pixel``), unshifted exponentials, gradients through both
    operands.  Same constructor and ``forward(features [n, 1, D], labels [n])``; D <= 256."""

    def __init__(self, sample_method='none', temperature=1):
        super().__init__()
        self.temperature = temperature
        self.sample_method = sample_method

    def forward(self, features, labels=None):
        feats, rows = _selfcon_rows(features, "PixelConLoss")
        if labels is None:
            raise AttributeError("PixelConLoss: labels are required (the reference calls labels.view, loss_new.py:376)")
        lab = labels.reshape(-1)
        if lab.numel() != feats.shape[0] or feats.shape[1] != 1:
            # the reference compares [bsz, bsz] masks with the [n_views*bsz]^2 logits: only n_views == 1 is well formed
            raise ValueError("PixelConLoss: expected features [n, 1, D] and n labels")
        lab = lab.to(rows.device)
        lab = lab - lab.min()   # the kernels reserve negative labels for padding; equality is all that matters
        return _SelfConFn.apply(rows, lab, 0, rows.shape[0], 1.0 / float(self.temperature), 1.0)


class SupConLoss(nn.Module):
    """``SupConLoss`` of utils/loss_new.py:263-352 (supervised contrastive learning / SimCLR when ``labels`` is None).
    Same constructor and ``forward(features [bsz, n_views, ...], labels=None, mask=None)``.  An explicit ``mask`` (an
    arbitrary, possibly asymmetric positive relation) is not a label structure the sweeps can skip tiles on: it raises
    NotImplementedError.  Feature width <= 256."""

    def __init__(self, temperature=0.07, contrast_mode='all', base_temperature=0.07):
        super().__init__()
        self.temperature = temperature
        self.contrast_mode = contrast_mode
        self.base_temperature = base_temperature

    def forward(self, features, labels=None, mask=None):
        feats, rows = _selfcon_rows(features, "SupConLoss")
        bsz, n_views = feats.shape[0], feats.shape[1]
        if labels is not None and mask is not None:
            raise ValueError('Cannot define both `labels` and `mask`')
        if mask is not None:
            raise NotImplementedError("SupConLoss: an explicit `mask` is not supported; pass labels (or nothing: SimCLR)")
        if labels is None:
            lab = torch.arange(bsz, device=rows.device)
        else:
            lab = labels.contiguous().view(-1).to(rows.device)
            if lab.shape[0] != bsz:
                raise ValueError('Num of labels does not match num of features')
            lab = lab - lab.min()
        if self.contrast_mode == 'one':
            n_anchor = bsz
        elif self.contrast_mode == 'all':
            n_anchor = bsz * n_views
        else:
            raise ValueError('Unknown mode: {}'.format(self.contrast_mode))
        return _SelfConFn.apply(rows, lab.repeat(n_views), 1, n_anchor, 1.0 / float(self.temperature),
                                float(self.temperature) / float(self.base_temperature))


class PixelContrastiveDistillation(nn.Module):
    """Opt-in, sync-free form of ``PixelConLossV2()(*pre_contrastive_pixel(f_n, l_n, l_po=..., f_o=...))``
    (train.py:115-116; SURVEY section 8(f) row N4): the same kernels, but the 5-tuple is never materialised, so N_a / N_o
    stay on the device, nothing waits for the host, and forward + backward can be captured in a CUDA graph
    (buffers have their worst-case sizes; row blocks beyond N_a exit at once).

    Differences a caller must know: a batch without any new-class pixel does not raise (the reference does,
    utils/loss.py:355) - the GT-new override of P simply never fires; a batch without anchors gives NaN (0/0).
    ``expected_anchor_fraction`` only steers how the column range is split over CTAs."""

    def __init__(self, temperature=0.07, max_label=20, *, gather_negatives=False, process_group=None,
                 ddp_grad_scale=True, expected_anchor_fraction=1.0):
        super().__init__()
        self.temperature = temperature
        self.max_label = int(max_label)
        self.gather_negatives = gather_negatives
        self.process_group = process_group
        self.ddp_grad_scale = ddp_grad_scale
        self.expected_anchor_fraction = float(expected_anchor_fraction)

    def _group(self):
        if not self.gather_negatives:
            return None
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return None
        group = self.process_group if self.process_group is not None else dist.group.WORLD
        return group if dist.get_world_size(group) > 1 else None

    def forward(self, f_n, l_n, l_po, f_o):
        pack = _build_pack(f_n.detach(), f_o.detach(), l_po.detach(), l_n, self.max_label, sync=False)
        cap_tiles = (pack.n_px + TILE - 1) // TILE
        plan_tiles = max(1, min(cap_tiles, int(cap_tiles * self.expected_anchor_fraction + 0.999)))
        ad = pack.addr
        rows = dict(feat=ad["feat"], prob=ad["prob"], lab=ad["lab"], n_rows=ad["counts"], keep=pack.payload,
                    range=pack.row_range, row_ref=pack.row_ref, max_tiles=cap_tiles, self_tile0=0,
                    plan_tiles=plan_tiles, static_pack=pack)
        group = self._group()
        cols = _local_cols(pack)
        return _ConFn.apply(f_n, cols, rows, 1.0 / float(self.temperature), 1, None, group, self.ddp_grad_scale)


# ----------------------------------------------------------------------------------------------
# N1 (opt-in): upsample + unbiased CE + unbiased KD fused, from the low-res logits
# ----------------------------------------------------------------------------------------------
class _SegFusedFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, lr, lr_old, labels, old_cl, ignore_index, alpha, grad_enabled):
        _need_cuda(lr, lr_old, labels)
        x = _f32c(lr)
        t = None if lr_old is None else _f32c(lr_old)   # None: the CE-only form (C_old = 0, the kd sum is 0)
        B, C, h, w = x.shape
        C_old = 0 if t is None else t.shape[1]
        H, W = labels.shape[-2:]
        dev = x.device
        # needs_input_grad only sees requires_grad: under no_grad no gradient buffer is allocated or written
        need_grad = bool(ctx.needs_input_grad[0]) and grad_enabled
        sums = torch.empty(3, device=dev, dtype=torch.float32)
        g = torch.empty(2 if t is not None else 1, B, C, h, w, device=dev, dtype=torch.float32) if need_grad else None
        n_ws = int(_lib.lib().ucd_seg_fused_workspace_floats(B, C, C_old, h, w, H, W))
        if n_ws == 0:
            raise ValueError("FusedUnbiasedLosses: shapes not supported (%s)" % ((B, C, C_old, h, w, H, W),))
        ws = torch.empty(n_ws, device=dev, dtype=torch.float32)
        check(_lib.lib().ucd_seg_fused_fwd(ptr(x), ptr(t), ptr(labels), ptr(g[0]) if need_grad else None,
                                           ptr(g[1]) if need_grad and t is not None else None, ptr(sums), ptr(ws), n_ws, B, C, C_old,
                                           h, w, H, W, old_cl, ignore_index, float(alpha), 1 if need_grad else 0,
                                           cur_stream()), "seg_fused_fwd")
        ctx.save_for_backward(g)
        ctx.n_px = float(B * H * W)
        ctx.in_dtype = lr.dtype
        return sums[0] / ctx.n_px, sums[2] / ctx.n_px, sums[1]

    @staticmethod
    def backward(ctx, g_ce, g_kd, _g_cnt):
        (g,) = ctx.saved_tensors
        d = g[0] * (g_ce / ctx.n_px)
        if g.shape[0] == 2:
            d = d + g[1] * (g_kd / ctx.n_px)   # two [B,C,h,w] tensors: negligible
        return d.to(ctx.in_dtype), None, None, None, None, None, None


class FusedUnbiasedLosses(nn.Module):
    """Opt-in fusion of ``interpolate`` (segmentation_module.py:133), ``UnbiasedCrossEntropy(reduction='none')
    (...).mean()`` (train.py:116) and ``UnbiasedKnowledgeDistillationLoss`` (train.py:133), computed straight from
    the LOW-RES logits of the new and the old model: the full-resolution logits are never materialised
    (SURVEY.md 8f, row N1).

        ce, kd = FusedUnbiasedLosses(old_cl, alpha=opts.alpha)(out_lowres, out_old_lowres, labels)
        loss = ce + con / 100 + opts.loss_kd * kd

    ``ce`` averages over ALL pixels of the batch (the trainer's ``.mean()`` of the 'none'-reduced loss);
    ``ce_reduction='valid'`` divides by the number of non-ignored pixels instead (nll_loss 'mean').
    Labels are remapped in place like ``UnbiasedCrossEntropy`` does.

    The base step has no old model: ``FusedUnbiasedLosses(0)(out_lowres, None, labels)`` returns ``(ce, None)``,
    computed by the CE-only form of the kernel.  With ``old_cl=0`` the unbiased CE is plain cross-entropy: for labels
    in [0, C) and ``ignore_index >= 0`` it equals ``F.cross_entropy(interpolate(lr), labels, ignore_index=ii,
    reduction='none').mean()`` ('valid': nll 'mean').  This relies on the kernels' reading of ``old_cl=0``, which
    ``UnbiasedCrossEntropy(old_cl=0)`` shares: the background branch needs ``old_cl > 0``.  (The reference's
    log-sum-exp over zero old channels would make label-0 pixels +inf.)  As in ``UnbiasedCrossEntropy``, labels below
    ``old_cl`` - negative ones included - are remapped to 0 in place, so a negative ``ignore_index`` is not ignored.
    """

    def __init__(self, old_cl, ignore_index=255, alpha=1., ce_reduction='mean'):
        super().__init__()
        self.old_cl, self.ignore_index, self.alpha, self.ce_reduction = int(old_cl), int(ignore_index), alpha, ce_reduction

    def forward(self, logits_lr, logits_old_lr, labels):
        if labels.dtype != torch.int64 or labels.dim() != 3:
            raise TypeError("FusedUnbiasedLosses: labels must be int64 [B,H,W]")
        if logits_old_lr is None:   # base step: the CE-only form
            if logits_lr.dim() != 4 or logits_lr.shape[0] != labels.shape[0]:
                raise ValueError("FusedUnbiasedLosses: logits [B,C,h,w] / labels [B,H,W] disagree")
        elif logits_lr.dim() != 4 or logits_old_lr.dim() != 4 or logits_lr.shape[0] != labels.shape[0] \
                or logits_lr.shape[2:] != logits_old_lr.shape[2:] or logits_old_lr.shape[1] > logits_lr.shape[1]:
            raise ValueError("FusedUnbiasedLosses: logits [B,C,h,w] / old logits [B,C_old,h,w] / labels [B,H,W] disagree")
        old = None if logits_old_lr is None else logits_old_lr.detach()
        tgt = labels if labels.is_contiguous() else labels.contiguous()
        ce, kd, cnt = _SegFusedFn.apply(logits_lr, old, tgt, self.old_cl, self.ignore_index, self.alpha,
                                        torch.is_grad_enabled())
        if tgt is not labels:
            labels.copy_(tgt)
        if self.ce_reduction == 'valid':
            ce = ce * (float(labels.numel()) / cnt)
        return ce, (None if old is None else kd)
