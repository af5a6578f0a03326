"""CPU tests of the guard that lets a loss chain hand the gradient of the low-res logits straight to them
(ucd_b200/losses.py::_Route): it may only do so in a plain ``backward()`` where nobody observes the gradient of the
upsampled `outputs`.  A toy autograd Function stands in for the chain head; the decision rests on
``torch._C._will_engine_execute_node``, whose behaviour is pinned here so that a torch upgrade that changes it fails
loudly instead of silently rerouting gradients."""
import pytest
import torch

from ucd_b200.losses import _Route


class _Head(torch.autograd.Function):
    """out.sum() with the route's extra inputs, like the head of a chain; records what the guard decided."""
    seen = []

    @staticmethod
    def forward(ctx, out, route, src, probe):
        ctx.route = route
        return out.sum()

    @staticmethod
    def backward(ctx, g):
        _Head.seen.append(ctx.route.route_now())
        return torch.ones(ctx.route.out_ref().shape), None, None, None


def _graph(leaf):
    lr0 = torch.randn(2, 3, 4, 4, requires_grad=True)
    lr = lr0 if leaf else lr0 * 1.0
    out = lr.repeat_interleave(2, dim=2).repeat_interleave(2, dim=3)   # stands in for interpolate_bilinear(lr)
    out._ucd_upsample = (lr, lr._version, out._version)
    return lr, out


def _decide(leaf, observe, run):
    lr, out = _graph(leaf)
    observe(out)
    r = _Route.of(out)
    assert r is not None
    route, src, probe = r
    assert src is lr and probe.is_leaf and probe.requires_grad
    loss = _Head.apply(out, route, src, probe)
    _Head.seen.clear()
    run(loss, out, lr)
    assert len(_Head.seen) == 1
    return _Head.seen[0]


def _nothing(out):
    pass


PASSES = {
    "backward": (lambda loss, out, lr: loss.backward(), True),
    "grad_out": (lambda loss, out, lr: torch.autograd.grad(loss, out), False),
    "grad_out_lr": (lambda loss, out, lr: torch.autograd.grad(loss, [out, lr], allow_unused=True), False),
    "grad_lr": (lambda loss, out, lr: torch.autograd.grad(loss, lr, allow_unused=True), False),
    "backward_inputs_out": (lambda loss, out, lr: loss.backward(inputs=[out]), False),
    "backward_inputs_out_lr": (lambda loss, out, lr: loss.backward(inputs=[out, lr]), False),
}


@pytest.mark.parametrize("leaf", [True, False])
@pytest.mark.parametrize("how", sorted(PASSES))
def test_route_only_in_a_plain_backward(leaf, how):
    run, want = PASSES[how]
    assert _decide(leaf, _nothing, run) is want


@pytest.mark.parametrize("leaf", [True, False])
def test_observers_of_outputs_keep_the_old_path(leaf):
    assert _decide(leaf, lambda out: out.retain_grad(), PASSES["backward"][0]) is False
    assert _decide(leaf, lambda out: out.register_hook(lambda g: g), PASSES["backward"][0]) is False
    # a hook that was removed again observes nothing
    assert _decide(leaf, lambda out: out.register_hook(lambda g: g).remove(), PASSES["backward"][0]) is True


def test_record_invalidated_by_in_place_changes():
    lr, out = _graph(False)
    out.mul_(2)
    assert _Route.of(out) is None
    lr, out = _graph(False)
    lr.add_(1)
    assert _Route.of(out) is None
    lr, out = _graph(True)
    with torch.no_grad():
        lr.add_(1)
    assert _Route.of(out) is None
    assert _Route.of(torch.randn(2, 3, 8, 8, requires_grad=True)) is None   # not an upsample output


def test_will_engine_execute_node_semantics():
    """What the guard relies on (torch 2.x): a private leaf's node reads True only in a plain backward(); a captured
    node reads True as well (so the source's own node cannot tell a capture of `outputs` apart); a captured leaf
    raises inside autograd.grad."""
    will = torch._C._will_engine_execute_node
    probe = torch.empty((), requires_grad=True)
    probe_node = torch.autograd.graph.get_gradient_edge(probe).node
    got = {}

    class F(torch.autograd.Function):
        @staticmethod
        def forward(ctx, a, p):
            return a.sum()

        @staticmethod
        def backward(ctx, g):
            res = {}
            for name, node in (("probe", probe_node), ("a_node", ctx.a_node), ("leaf", ctx.leaf_node)):
                try:
                    res[name] = will(node)
                except RuntimeError:
                    res[name] = "raises"
            got.update(res)
            return torch.ones(3), None

    leaf = torch.randn(3, requires_grad=True)
    a = leaf * 2.0
    y = F.apply(a, probe)
    y.grad_fn.a_node, y.grad_fn.leaf_node = a.grad_fn, a.grad_fn.next_functions[0][0]
    y.backward(retain_graph=True)
    assert got == {"probe": True, "a_node": True, "leaf": True}
    torch.autograd.grad(y, a, retain_graph=True)
    assert got["probe"] is False and got["a_node"] is True   # captured, not executed: still reads True
    torch.autograd.grad(y, [a, leaf], retain_graph=True)
    assert got["probe"] is False and got["leaf"] == "raises"
