"""torch.autograd Functions over the fused kernels: the opt-in (opt.autograd / DM_Router(autograd=True)) that lets the
reference's own training loop -- forward, loss, loss.backward(), clip_grad_norm_, optimizer.step() -- run on
MRNNet, Model and DM_Router.  Every backward is a kernel of the library; the Functions only map the kernels' flat
arenas back to the nn.Parameters, so gradients land in .grad with autograd's usual accumulation.  They are
once_differentiable: a double backward raises.

  * RoutedSoft: MRNNet's soft route (experts -> DM-Router -> gate -> combine).  Gradients reach route.*,
    channel_route.* and dm_router.0.* through mrnb_gate_combine_backward and mrnb_router_backward (domain = NULL).
    The experts are frozen, as in MRN stage 1 (il_modules/mrn.py:154-157,285-287) -- unless opt.autograd_experts names
    trainable experts: those run their training packs, and the backward is mrnb_gate_combine_backward_experts (dgate
    and each trainable expert's logit gradient dz_i = g_i dY in one pass), mrnb_router_backward_dx (the router's input
    gradient dx) and one training-pack backward per trainable expert with dz_i and dx[:, i] as the feature gradient.
    An image that requires grad makes every expert run its training pack: the frozen ones take the input-only backward
    (no parameter gradient), and the image gradient is the sum of the experts' image gradients in expert order.
  * ExpertTrain: one expert end to end through its training pack (activation-keeping forward, full backward, or the
    input-only backward when no expert parameter requires grad); logits, and the feature when asked for.
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


def _expert_grads(grads, keys):
    """{state_dict key: gradient} of a training-pack backward -> one tensor (or None: a tensor the forward never reads)
    per key, copied: the pack's gradient arena is overwritten by another backward through the same graph."""
    return tuple(None if grads.get(k) is None else grads[k].clone(memory_format=torch.contiguous_format) for k in keys)


class RoutedSoft(torch.autograd.Function):
    """(net, image, trainable, *net.router_parameters(), *parameters of the trainable experts in order) ->
    (combined logits [B,T,C], gate [B,I]).  trainable: indices of the experts that train with the router (empty: the
    experts are frozen and run the grouped forward alone)."""

    @staticmethod
    def forward(ctx, net, image, trainable, *params):
        rws = ops.RouterWorkspace()          # the backward reads the activations this forward leaves in it
        experts_out, ctx.expert_backward = None, {}
        if trainable or ctx.needs_input_grad[1]:
            feats, logits, ctx.expert_backward = net.joint_experts_forward(image, trainable,
                                                                           input_grad=ctx.needs_input_grad[1])
            experts_out = (feats, logits)
        r = net.route_and_combine(image, is_train=True, want_logits=True, with_backward=True, rws=rws,
                                  experts_out=experts_out)
        ctx.net, ctx.rws, ctx.trainable = net, rws, trainable
        ctx.expert_logits = r["expert_logits"]
        ctx.save_for_backward(net.router_arena(), r["features"], r["gate"])
        return r["logits"], r["gate"]

    @staticmethod
    @once_differentiable
    def backward(ctx, d_logits, d_gate):
        from .modules.model import _precision
        arena, feats, gate = ctx.saved_tensors
        net, trainable = ctx.net, ctx.trainable
        packs = sorted(ctx.expert_backward)  # the experts that ran a training pack: trainable ones, or all for the image
        B, I, T, D = feats.shape
        dz = [None] * I
        for e in packs:                      # rows padded to 4 floats, as the kernel writes them
            z = ctx.expert_logits[e]
            dz[e] = torch.zeros(B, T, ops.round_up(z.shape[2], 4), device=z.device)[:, :, :z.shape[2]]
        dgate = torch.zeros_like(gate)
        if d_logits is not None:
            if packs:
                dgate = ops.gate_combine_backward_experts(ctx.expert_logits, d_logits.float(), gate, dz)
            else:
                dgate = ops.gate_combine_backward(ctx.expert_logits, d_logits.float())
        if d_gate is not None:
            dgate = dgate + d_gate.float()
        grads = torch.empty_like(arena)
        dx = torch.empty_like(feats) if packs else None
        ops.router_backward(arena, feats, gate, dgate.contiguous(), None, grads, ctx.rws, prec=_precision(net.opt), dx=dx)
        out = _arena_grads(grads, net.router_parameters(), ops.ROUTER_PARAM_NAMES, I, T, D)
        dimage = None
        for e in packs:
            g, di = ctx.expert_backward[e](dz[e], dx[:, e].contiguous(), dimage=ctx.needs_input_grad[1])
            if e in trainable:
                out += _expert_grads(g, [k for k, _ in net.model[e].named_parameters()])
            if di is not None:               # summed in expert order
                dimage = di if dimage is None else dimage.add_(di)
        return (None, dimage, None) + out


class ExpertTrain(torch.autograd.Function):
    """(run, keys, want_features, image, *params) -> logits [B,T,C], or (logits, features [B,T,256]) with
    want_features.  `run(image, want_features=, param_grads=)` is modules.model._train_pack_run for one expert:
    (logits, features, backward), backward(dlogits, dfeatures, dimage=) -> ({state_dict key: gradient in the reference
    layout} or None, image gradient or None); `params` are the expert's parameters named by `keys`.  The pack is built
    without a gradient arena (input-only backward) when none of `params` requires grad."""

    @staticmethod
    def forward(ctx, run, keys, want_features, image, *params):
        param_grads = any(ctx.needs_input_grad[4:])
        logits, feats, backward = run(image, want_features=want_features, param_grads=param_grads)
        ctx.run_backward, ctx.keys, ctx.param_grads = backward, keys, param_grads
        ctx.set_materialize_grads(False)
        ctx.logits_shape = logits.shape
        return (logits, feats) if want_features else logits

    @staticmethod
    @once_differentiable
    def backward(ctx, d_logits, d_features=None):
        if d_logits is None:                 # only the feature reached the loss
            d_logits = torch.zeros(ctx.logits_shape, device=d_features.device)
        dfeat = None if d_features is None else d_features.float().contiguous()
        grads, dimage = ctx.run_backward(d_logits.float().contiguous(), dfeat, dimage=ctx.needs_input_grad[3])
        pgrads = _expert_grads(grads, ctx.keys) if ctx.param_grads else (None,) * len(ctx.keys)
        return (None, None, None, dimage) + pgrads


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
