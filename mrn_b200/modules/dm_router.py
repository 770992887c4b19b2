"""DM_Router with the reference's constructor, sub-module names and state_dict keys (modules/dm_router.py:35-67).
forward() runs the fused CUDA router (mrn_b200.ops.router_forward); parameters are views into the flat router
arena owned by MRNNet when the module is part of one."""
import torch
import torch.nn as nn

from .. import ops


class SpatialDomainGating(nn.Module):
    def __init__(self, d_ffn, seq_len):
        super().__init__()
        self.norm = nn.LayerNorm(d_ffn // 2)
        self.proj = nn.Linear(seq_len, seq_len)


class ChannelDomainGating(nn.Module):
    def __init__(self, d_ffn, seq_len):
        super().__init__()
        self.norm = nn.LayerNorm(d_ffn)
        self.proj = nn.Linear(seq_len, seq_len)


class DM_Router(nn.Module):
    def __init__(self, channel, d_ffn, patch, domain, autograd=False):
        super().__init__()
        self.autograd = autograd        # forward() builds an autograd graph (input and parameter gradients)
        self.patch = patch
        self.channel = channel
        self.domain = domain
        self.norm = nn.LayerNorm(channel)
        self.proj_1 = nn.Linear(channel, d_ffn)
        self.activation = nn.GELU()
        self.spatial_gating = SpatialDomainGating(d_ffn, patch * domain)
        self.channel_gating = ChannelDomainGating(patch, domain * channel)
        self.proj_2 = nn.Linear(d_ffn // 2, channel)
        self.proj_3 = nn.Linear(channel, channel)
        self._ws = ops.RouterWorkspace()

    def _standalone_arena(self, device):
        """Flat arena in the C-ABI order with zero route / channel_route slots (module used on its own)."""
        n, off = ops.router_param_offsets(self.domain, self.patch, self.channel)
        arena = torch.zeros(n, device=device, dtype=torch.float32)
        sd = {"dm_router.0." + k: v for k, v in self.state_dict().items()}
        for k, name in enumerate(ops.ROUTER_PARAM_NAMES):
            if name in sd:
                arena[off[k]:off[k] + sd[name].numel()] = sd[name].reshape(-1).to(device)
        return arena

    def forward(self, x):
        """x [B, D(omain), P(atch), C] -> same shape (modules/dm_router.py:50-67).  With autograd=True and grad mode on,
        the output is differentiable with respect to x and every parameter (mrnb_dm_router_backward)."""
        if not x.is_cuda:
            raise RuntimeError("DM_Router.forward needs a CUDA tensor: mrn_b200 has no CPU fallback")
        if self.autograd and torch.is_grad_enabled():
            from ..autograd import DmRouter
            return DmRouter.apply(self, x.contiguous().float(), *self.parameters())
        out, _, _, _ = ops.router_forward(self._standalone_arena(x.device), x.contiguous().float(), self._ws)
        return out
