"""torch.autograd Functions over the fused kernels: the opt-in (opt.autograd / DM_Router(autograd=True)) that lets the
reference's own training loop -- forward, loss, loss.backward(), clip_grad_norm_, optimizer.step() -- run on
MRNNet, Model and DM_Router.  Every backward is a kernel of the library; the Functions only map the kernels' flat
arenas back to the nn.Parameters, so gradients land in .grad with autograd's usual accumulation.  They are
once_differentiable: a double backward raises.

  * RoutedSoft: MRNNet's soft route (experts -> DM-Router -> gate -> combine).  Gradients reach route.*,
    channel_route.* and dm_router.0.* through mrnb_gate_combine_backward and mrnb_router_backward (domain = NULL).
    The experts are frozen, as in MRN stage 1 (il_modules/mrn.py:154-157,285-287).
  * ExpertTrain: one expert end to end through its training pack (activation-keeping forward, full backward).
  * DmRouter: DM_Router on its own through mrnb_dm_router_backward (input and parameter gradients).
"""
import torch
from torch.autograd.function import once_differentiable

from . import ops


def _arena_grads(grads, params, names, n_experts, T, D):
    """Views of the gradient arena `grads` shaped like `params` (router slot names `names`, C-ABI order)."""
    _, off = ops.router_param_offsets(n_experts, T, D)
    slot = {n: k for k, n in enumerate(ops.ROUTER_PARAM_NAMES)}
    return tuple(grads[off[slot[n]]:off[slot[n]] + p.numel()].view(p.shape) for n, p in zip(names, params))


class RoutedSoft(torch.autograd.Function):
    """(net, image, *net.router_parameters()) -> (combined logits [B,T,C], gate [B,I])."""

    @staticmethod
    def forward(ctx, net, image, *params):
        rws = ops.RouterWorkspace()          # the backward reads the activations this forward leaves in it
        r = net.route_and_combine(image, is_train=True, want_logits=True, with_backward=True, rws=rws)
        ctx.net, ctx.rws = net, rws
        ctx.expert_logits = r["expert_logits"]
        ctx.save_for_backward(net.router_arena(), r["features"], r["gate"])
        return r["logits"], r["gate"]

    @staticmethod
    @once_differentiable
    def backward(ctx, d_logits, d_gate):
        from .modules.model import _precision
        arena, feats, gate = ctx.saved_tensors
        net = ctx.net
        B, I, T, D = feats.shape
        dgate = torch.zeros_like(gate)
        if d_logits is not None:
            dgate = ops.gate_combine_backward(ctx.expert_logits, d_logits.float())
        if d_gate is not None:
            dgate = dgate + d_gate.float()
        grads = torch.empty_like(arena)
        ops.router_backward(arena, feats, gate, dgate.contiguous(), None, grads, ctx.rws, prec=_precision(net.opt))
        params = net.router_parameters()
        return (None, None) + _arena_grads(grads, params, ops.ROUTER_PARAM_NAMES, I, T, D)


class ExpertTrain(torch.autograd.Function):
    """(run, keys, image, *params) -> logits [B,T,C].  `run(image)` runs the expert's training-pack forward and returns
    (backward, logits), backward(dlogits) -> {state_dict key: gradient in the reference layout}; `params` are the
    expert's parameters named by `keys`."""

    @staticmethod
    def forward(ctx, run, keys, image, *params):
        backward, logits = run(image)
        ctx.run_backward, ctx.keys = backward, keys
        return logits

    @staticmethod
    @once_differentiable
    def backward(ctx, d_logits):
        grads = ctx.run_backward(d_logits.float().contiguous())
        # copies: the pack's gradient arena is overwritten by another backward through the same graph
        return (None, None, None) + tuple(None if grads.get(k) is None else grads[k].clone(memory_format=torch.contiguous_format)
                                          for k in ctx.keys)


class DmRouter(torch.autograd.Function):
    """(module, x [B,I,T,D], *module parameters) -> DM_Router(x)."""

    @staticmethod
    def forward(ctx, module, x, *params):
        arena = module._standalone_arena(x.device)
        ws = ops.RouterWorkspace()
        out, _, _, _ = ops.router_forward(arena, x, ws, with_backward=True)
        ctx.module, ctx.ws = module, ws
        ctx.save_for_backward(arena, x)
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, d_out):
        arena, x = ctx.saved_tensors
        B, I, T, D = x.shape
        grads = torch.empty_like(arena)
        dx = ops.dm_router_backward(arena, x, d_out.float().contiguous(), grads, ctx.ws, want_dx=ctx.needs_input_grad[1])
        names = ["dm_router.0." + n for n, _ in ctx.module.named_parameters()]
        params = [p for _, p in ctx.module.named_parameters()]
        return (None, dx) + _arena_grads(grads, params, names, I, T, D)
