"""Thin Python wrappers over the C ABI (include/mrn_b200.h): torch tensors in, torch tensors out.

torch is used for device memory, streams and (elsewhere) torch.distributed only; every FLOP on the path runs in
libmrn_b200.so.  All wrappers require CUDA tensors and raise otherwise -- there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, List, Optional, Sequence

import torch

from . import _lib as L

T_FRAMES = 64      # MRNNet.patch for SVTR (modules/model.py:324)
T_FRAMES_CRNN = 63  # MRNNet.patch for CRNN (modules/model.py:322-323)
D_FEAT = 256       # opt.hidden_size


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t: Optional[torch.Tensor]):
    if t is None:
        return C.c_void_p(0)
    if not t.is_cuda:
        raise RuntimeError("mrn_b200 ops need CUDA tensors (no CPU fallback)")
    return C.c_void_p(t.data_ptr())


def _chk_f32(*ts):
    for t in ts:
        if t is not None and (t.dtype != torch.float32 or not t.is_contiguous()):
            raise RuntimeError("expected a contiguous float32 tensor, got %s contiguous=%s" % (t.dtype, t.is_contiguous()))


def launch_count() -> int:
    return int(L.load().mrnb_launch_count())


def reset_launch_count() -> None:
    L.load().mrnb_reset_launch_count()


PROFILE_FAMILIES = ("tc_gemm_kernel", "sgemm_kernel", "attn_tc_kernel", "layernorm_kernel", "patch_embed", "combine_row_kernel",
                    "ctc_lattice_kernel", "router_elementwise", "optimizer", "misc", "mlp_tc_kernel", "tc_gemm2_kernel",
                    "mixer_tc_kernel")


def profile_enable(on: bool):
    L.load().mrnb_profile_enable(int(on))


def profile_reset():
    L.load().mrnb_profile_reset()


def profile_read():
    """{family: dict(ms, calls, flops, bytes)} summed over the recorded launches (synchronises)."""
    out = {}
    for k, name in enumerate(PROFILE_FAMILIES):
        ms, calls, fl, by = C.c_double(), C.c_long(), C.c_double(), C.c_double()
        L.check(L.load().mrnb_profile_read(k, C.byref(ms), C.byref(calls), C.byref(fl), C.byref(by)), "profile_read")
        out[name] = dict(ms=ms.value, calls=calls.value, flops=fl.value, bytes=by.value)
    return out


# ------------------------------------------------------------------------------------------------ building blocks
def linear_f32(a, w, bias=None, residual=None, gelu=False):
    _chk_f32(a, w, bias, residual)
    M, K = a.shape
    N = w.shape[0]
    out = torch.empty(M, N, device=a.device, dtype=torch.float32)
    L.check(L.load().mrnb_linear_f32(_p(a), _p(w), _p(bias), _p(residual), _p(out), M, N, K, int(gelu), _stream()), "linear_f32")
    return out


def cast_bf16(x: torch.Tensor) -> torch.Tensor:
    _chk_f32(x)
    y = torch.empty(x.shape, device=x.device, dtype=torch.bfloat16)
    L.check(L.load().mrnb_cast_f32_to_bf16(_p(x), _p(y), x.numel(), _stream()), "cast")
    return y


def cast_f16(x: torch.Tensor) -> torch.Tensor:
    _chk_f32(x)
    y = torch.empty(x.shape, device=x.device, dtype=torch.float16)
    L.check(L.load().mrnb_cast_f32_to_f16(_p(x), _p(y), x.numel(), _stream()), "cast")
    return y


def _out(out, shape, device, dtype):
    """A caller-supplied output (e.g. NaN pre-filled by a test, so that an element the kernel never writes shows) or a
    fresh one."""
    if out is None:
        return torch.empty(shape, device=device, dtype=dtype)
    if tuple(out.shape) != tuple(shape) or out.dtype != dtype or not out.is_contiguous() or out.device != device:
        raise RuntimeError("out: expected a contiguous %s tensor of shape %s on %s, got %s %s on %s"
                           % (dtype, tuple(shape), device, out.dtype, tuple(out.shape), out.device))
    return out


def linear_bf16(a, w, bias=None, residual=None, gelu=False, out_f32=True, out=None):
    assert a.dtype == torch.bfloat16 and w.dtype == torch.bfloat16 and a.is_contiguous() and w.is_contiguous()
    _chk_f32(bias, residual)
    M, K = a.shape
    N = w.shape[0]
    out = _out(out, (M, N), a.device, torch.float32 if out_f32 else torch.bfloat16)
    L.check(L.load().mrnb_linear_bf16(_p(a), _p(w), _p(bias), _p(residual), _p(out), int(out_f32), M, N, K, int(gelu),
                                      _stream()), "linear_bf16")
    return out


def tc_gemm_general(a, a_mn, b, b_mn, M, N, K, splitk=1):
    """Test entry of the general tcgen05 GEMM: a is [M,K] or (a_mn) [K,M]; b is [N,K] or (b_mn) [K,N]; bf16."""
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.is_contiguous() and b.is_contiguous()
    out = torch.zeros(M, N, device=a.device, dtype=torch.float32)
    L.check(L.load().mrnb_tc_gemm_general(_p(a), int(a_mn), _p(b), int(b_mn), _p(out), M, N, K, int(splitk), _stream()),
            "tc_gemm_general")
    return out


def mlp_bf16(a16, w1_16, b1, w2_16, b2, x, rowscale=None, rows_per_scale=1, ln_gamma=None, ln_beta=None, ln_eps=1e-6):
    """Fused MLP branch; x [M,D] fp32 is updated IN PLACE.  Returns the fused LayerNorm output (bf16) or None."""
    assert a16.dtype == torch.bfloat16 and w1_16.dtype == torch.bfloat16 and w2_16.dtype == torch.float16
    _chk_f32(b1, b2, x, rowscale, ln_gamma, ln_beta)
    M, D = x.shape
    ln_out = torch.empty(M, D, device=x.device, dtype=torch.bfloat16) if ln_gamma is not None else None
    L.check(L.load().mrnb_mlp_bf16(_p(a16), _p(w1_16), _p(b1), _p(w2_16), _p(b2), _p(x), _p(rowscale), int(rows_per_scale),
                                   _p(ln_out), _p(ln_gamma), _p(ln_beta), float(ln_eps), M, D, _stream()), "mlp_bf16")
    return ln_out


def mixer_bf16(a16, wqkv16, bqkv, wproj16, bproj, x, local, rowscale=None, ln_gamma=None, ln_beta=None, ln_eps=1e-6):
    """Fused mixer branch (qkv GEMM -> attention -> proj + DropPath + residual [+ LayerNorm]); x [units,N,D] fp32 is
    updated IN PLACE.  a16 = LN1(x) bf16 [units,N,D].  Returns the fused LayerNorm output (bf16) or None."""
    assert a16.dtype == torch.bfloat16 and wqkv16.dtype == torch.bfloat16 and wproj16.dtype == torch.bfloat16
    _chk_f32(bqkv, bproj, x, rowscale, ln_gamma, ln_beta)
    units, N, D = x.shape
    assert N * D == 32768 and a16.shape == x.shape and a16.is_contiguous()
    ln_out = torch.empty(units, N, D, device=x.device, dtype=torch.bfloat16) if ln_gamma is not None else None
    L.check(L.load().mrnb_mixer_bf16(_p(a16), _p(wqkv16), _p(bqkv), _p(wproj16), _p(bproj), _p(x), _p(rowscale), _p(ln_out),
                                     _p(ln_gamma), _p(ln_beta), float(ln_eps), units, D, int(local), _stream()), "mixer_bf16")
    return ln_out


def layernorm(x, gamma, beta, eps):
    _chk_f32(x, gamma, beta)
    y = torch.empty_like(x)
    rows = x.numel() // x.shape[-1]
    L.check(L.load().mrnb_layernorm_f32(_p(x), _p(y), _p(gamma), _p(beta), rows, x.shape[-1], float(eps), _stream()), "layernorm")
    return y


def svtr_attention(qkv, heads, H, W, local):
    _chk_f32(qkv)
    G, N, d3 = qkv.shape
    out = torch.empty(G, N, d3 // 3, device=qkv.device, dtype=torch.float32)
    L.check(L.load().mrnb_svtr_attention_f32(_p(qkv), _p(out), G, N, d3 // 3, heads, H, W, int(local), _stream()), "attention")
    return out


def svtr_attention_bf16(qkv, heads, H, W, local, out=None):
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous()
    G, N, d3 = qkv.shape
    out = _out(out, (G, N, d3 // 3), qkv.device, torch.bfloat16)
    L.check(L.load().mrnb_svtr_attention_bf16(_p(qkv), _p(out), G, N, d3 // 3, heads, H, W, int(local), _stream()),
            "attention_bf16")
    return out


def attn_tc_train_forward(qkv, heads, W, local, P=None, O=None):
    """Training attention forward of one stage (bf16 mode): qkv [B, N, 3d] bf16 -> (P [B*heads, N, N] bf16 = the
    probabilities kept for the backward, O [B, N, d] bf16)."""
    assert qkv.dtype == torch.bfloat16 and qkv.is_contiguous()
    B, N, d3 = qkv.shape
    d = d3 // 3
    P = _out(P, (B * heads, N, N), qkv.device, torch.bfloat16)
    O = _out(O, (B, N, d), qkv.device, torch.bfloat16)
    L.check(L.load().mrnb_attn_tc_train_forward(_p(qkv), _p(P), _p(O), B, N, d, heads, W, int(local), _stream()),
            "attn_tc_train_forward")
    return P, O


def attn_tc_train_backward(qkv, O, P, dO, dO16, heads, dS=None, dqkv=None):
    """Training attention backward of one stage (bf16 mode): dO [B, N, d] fp32 and its bf16 copy dO16, with the
    forward's qkv, O and P -> (dS [B*heads, N, N] bf16, dqkv [B, N, 3d] bf16 = dQ | dK | dV)."""
    assert qkv.dtype == O.dtype == P.dtype == dO16.dtype == torch.bfloat16
    assert qkv.is_contiguous() and O.is_contiguous() and P.is_contiguous() and dO16.is_contiguous()
    _chk_f32(dO)
    B, N, d3 = qkv.shape
    d = d3 // 3
    assert O.shape == dO.shape == dO16.shape == (B, N, d) and P.shape == (B * heads, N, N)
    dS = _out(dS, (B * heads, N, N), qkv.device, torch.bfloat16)
    dqkv = _out(dqkv, (B, N, d3), qkv.device, torch.bfloat16)
    L.check(L.load().mrnb_attn_tc_train_backward(_p(qkv), _p(O), _p(dO), _p(dO16), _p(P), _p(dS), _p(dqkv), B, N, d, heads,
                                                 _stream()), "attn_tc_train_backward")
    return dS, dqkv


# ------------------------------------------------------------------------------------------------ SVTR experts
_BLOCK_KEYS = ("norm1.weight", "norm1.bias", "mixer.qkv.weight", "mixer.qkv.bias", "mixer.proj.weight",
               "mixer.proj.bias", "norm2.weight", "norm2.bias", "mlp.fc1.weight", "mlp.fc1.bias", "mlp.fc2.weight",
               "mlp.fc2.bias")
_BLOCK_NAMES = [f"blocks1.{j}" for j in range(3)] + [f"blocks2.{j}" for j in range(6)] + [f"blocks3.{j}" for j in range(3)]
_GEMM_W_SLOTS = {L.PB_QKV_W, L.PB_PROJ_W, L.PB_FC1_W, L.PB_FC2_W}


def _mask(flag):
    """bool -> every expert / none; int -> per-expert bit mask as is (include/mrn_b200.h: MRNB_ALL_EXPERTS)."""
    if isinstance(flag, bool):
        return -1 if flag else 0
    return int(flag)


def round_up(v, a):
    return (v + a - 1) // a * a


def _grow_workspace(pack, need):
    """pack._ws, reallocated only when it holds fewer than `need` bytes: later calls (and CUDA-graph replays) keep
    using the same buffer."""
    if pack._ws is None or pack._ws.numel() < need:
        pack._ws = torch.empty(need, dtype=torch.uint8, device=pack.device)
    return pack._ws


class SvtrPack:
    """Device-resident, expert-stacked copy of the SVTR expert parameters in the layout the kernels consume
    (include/mrn_b200.h: MRNB_P_* slots).  Built from a reference-format state_dict; rebuilt when experts change
    (experts are frozen during router training, il_modules/mrn.py:154-157)."""

    arch = "svtr"
    n_frames = 64

    def __init__(self, state_dict: Dict[str, torch.Tensor], n_experts: int, device, prec: int, prefix: str = ""):
        self.n_experts = n_experts
        self.prec = prec
        self.device = torch.device(device)
        self.tensors: List[torch.Tensor] = []      # keep-alive
        self.struct = L.MrnbSvtrPack()
        self.struct.n_experts = n_experts
        self.n_class: List[int] = []
        self.slot_tensors: Dict[int, torch.Tensor] = {}
        sd = state_dict

        def conv(i):
            return f"{prefix}model.{i}.model.FeatureExtraction.ConvNet."

        def stack(suffix, permute=None):
            ts = []
            for i in range(n_experts):
                t = sd[conv(i) + suffix].detach().to(self.device, torch.float32)
                if permute is not None:
                    t = t.permute(*permute)
                ts.append(t.contiguous())
            return torch.stack(ts, 0).contiguous()

        def put(slot, t, gemm_weight=False):
            self.tensors.append(t)
            self.slot_tensors[slot] = t
            self.struct.p[slot] = t.data_ptr()
            if gemm_weight and prec == L.PREC_BF16:
                # mlp.fc2 feeds the fused MLP's second GEMM, whose A operand (GELU output) is f16
                is_fc2 = slot >= L.P_BLOCK0 and slot < L.P_SUB0 and (slot - L.P_BLOCK0) % L.PB_COUNT == L.PB_FC2_W
                h = cast_f16(t) if is_fc2 else cast_bf16(t)
                self.tensors.append(h)
                self.struct.h[slot] = h.data_ptr()

        put(L.P_POS_EMBED, stack("pos_embed").reshape(n_experts, 512, 64).contiguous())
        put(L.P_CONV0_W, stack("patch_embed.proj.0.weight"))
        put(L.P_CONV0_B, stack("patch_embed.proj.0.bias"))
        for base, idx in ((L.P_BN0_W, 1), (L.P_BN1_W, 4)):
            for k, nm in enumerate(("weight", "bias", "running_mean", "running_var")):
                put(base + k, stack(f"patch_embed.proj.{idx}.{nm}"))
        put(L.P_CONV1_W, stack("patch_embed.proj.3.weight", permute=(0, 2, 3, 1)))
        if prec == L.PREC_BF16:
            # implicit-GEMM layout of conv1: k = kh*128 + kw*32 + c with a zero fourth tap ({kw0,kw1}, {kw2,0} slots)
            w = self.slot_tensors[L.P_CONV1_W]                                   # [I,64,3,3,32]
            wg = torch.zeros(n_experts, 64, 3, 4, 32, device=self.device, dtype=torch.float32)
            wg[:, :, :, :3, :] = w
            h = cast_bf16(wg.reshape(n_experts, 64, 384).contiguous())
            self.tensors.append(h)
            self.struct.h[L.P_CONV1_W] = h.data_ptr()
        put(L.P_CONV1_B, stack("patch_embed.proj.3.bias"))
        for b, name in enumerate(_BLOCK_NAMES):
            for k, key in enumerate(_BLOCK_KEYS):
                put(L.P_BLOCK0 + b * L.PB_COUNT + k, stack(f"{name}.{key}"), gemm_weight=k in _GEMM_W_SLOTS)
        for s in range(3):
            base = L.P_SUB0 + s * L.PS_COUNT
            put(base + L.PS_CONV_W, stack(f"sub_sample{s + 1}.conv.weight", permute=(0, 2, 3, 1)), gemm_weight=True)
            put(base + L.PS_CONV_B, stack(f"sub_sample{s + 1}.conv.bias"))
            put(base + L.PS_NORM_W, stack(f"sub_sample{s + 1}.norm.weight"))
            put(base + L.PS_NORM_B, stack(f"sub_sample{s + 1}.norm.bias"))
        seq_w = torch.stack([sd[f"{prefix}model.{i}.model.SequenceModeling.0.weight"].detach().to(self.device, torch.float32)
                             for i in range(n_experts)], 0).contiguous()
        seq_b = torch.stack([sd[f"{prefix}model.{i}.model.SequenceModeling.0.bias"].detach().to(self.device, torch.float32)
                             for i in range(n_experts)], 0).contiguous()
        put(L.P_SEQ_W, seq_w, gemm_weight=True)
        put(L.P_SEQ_B, seq_b)
        fc_ws = [sd[f"{prefix}model.{i}.fc.weight"].detach().to(self.device, torch.float32).contiguous() for i in range(n_experts)]
        # bf16 heads stacked in ONE allocation in expert order: mrnb_svtr_heads / the forward run every ragged head
        # (C_i differs per expert) as a single grouped tcgen05 launch over one TMA map
        stacked16 = None
        if prec == L.PREC_BF16:
            stacked16 = torch.zeros(sum(int(w.shape[0]) for w in fc_ws) + 128, fc_ws[0].shape[1], device=self.device, dtype=torch.bfloat16)
            self.tensors.append(stacked16)
        row = 0
        for i in range(n_experts):
            w = fc_ws[i]
            b = sd[f"{prefix}model.{i}.fc.bias"].detach().to(self.device, torch.float32).contiguous()
            self.tensors += [w, b]
            self.struct.fc_w[i] = w.data_ptr()
            self.struct.fc_b[i] = b.data_ptr()
            self.struct.n_class[i] = w.shape[0]
            self.n_class.append(int(w.shape[0]))
            if stacked16 is not None:
                h = stacked16[row:row + w.shape[0]]
                L.check(L.load().mrnb_cast_f32_to_bf16(_p(w), C.c_void_p(h.data_ptr()), w.numel(), _stream()), "cast")
                self.struct.fc_w16[i] = h.data_ptr()
                row += int(w.shape[0])
        self._ws: Optional[torch.Tensor] = None
        self._ws_key = None

    def bn_running_stats(self):
        """(mean0, var0, mean1, var1), each [I, C]: updated in place by train-mode forwards."""
        return tuple(self.slot_tensors[s] for s in (L.P_BN0_MEAN, L.P_BN0_VAR, L.P_BN1_MEAN, L.P_BN1_VAR))

    def workspace(self, B, chunk):
        return _grow_workspace(self, int(L.load().mrnb_svtr_workspace_bytes(self.n_experts, B, chunk, self.prec)))


def _logit_buffers(pack, B, device, want):
    """Per-expert logit buffers [B, pack.n_frames, C_i rounded up to 4] for the grouped heads.  Returns (ptrs, lds,
    [logits_i [B,T,C_i] views]); with want=False the pointers are NULL (no logits written) and the views None."""
    I = pack.n_experts
    ptrs = (C.c_void_p * I)()
    lds = (C.c_long * I)()
    logits = []
    for i in range(I):
        ld = round_up(pack.n_class[i], 4)
        lds[i] = ld
        if want:
            buf = torch.empty(B, pack.n_frames, ld, device=device, dtype=torch.float32)
            ptrs[i] = buf.data_ptr()
            logits.append(buf[:, :, :pack.n_class[i]])
        else:
            ptrs[i] = None
            logits.append(None)
    return ptrs, lds, logits


def svtr_heads(pack: SvtrPack, B: int, route_index: Optional[torch.Tensor] = None):
    """Classifier heads on the features the last svtr_experts_forward(pack, image[B], chunk=0) left in the pack's
    workspace.  route_index int32 [B]: hard route -- only the routed expert's head is evaluated per sample; the other
    (expert, sample) rows of the returned buffers are uninitialised and must not be read (gate_combine with the matching
    one-hot gate never does).  Returns [logits_i [B,64,C_i] views]."""
    if pack._ws is None or pack._ws_key != (B, 0):
        raise RuntimeError("svtr_heads: no features of a B=%d, chunk=0 forward in the pack's workspace" % B)
    if route_index is not None and (route_index.dtype != torch.int32 or not route_index.is_cuda or route_index.numel() != B):
        raise RuntimeError("svtr_heads: route_index must be a CUDA int32 tensor [B]")
    ptrs, lds, logits = _logit_buffers(pack, B, pack._ws.device, True)
    L.check(L.load().mrnb_svtr_heads(C.byref(pack.struct), B, pack.prec, _p(route_index), ptrs, lds, _p(pack._ws),
                                     pack._ws.numel(), _stream()), "svtr_heads")
    return logits


def svtr_experts_forward(pack: SvtrPack, image: torch.Tensor, bn_batch_stats: bool = False, update_running: bool = False,
                         drop_scales: Optional[torch.Tensor] = None, chunk: int = 0, want_logits: bool = True):
    """Runs every expert on `image` [B,4,32,256].  Returns (features [B,I,64,256], [logits_i [B,64,C_i] views])."""
    _chk_f32(image, drop_scales)
    B = image.shape[0]
    feats = torch.empty(B, pack.n_experts, T_FRAMES, D_FEAT, device=image.device, dtype=torch.float32)
    ptrs, lds, logits = _logit_buffers(pack, B, image.device, want_logits)
    ws = pack.workspace(B, chunk)
    pack._ws_key = (B, int(chunk) if 0 < int(chunk) < B else 0)
    rc = L.load().mrnb_svtr_experts_forward(C.byref(pack.struct), _p(image), B, int(chunk), pack.prec, _mask(bn_batch_stats),
                                            _mask(update_running), _p(drop_scales), _p(feats), ptrs, lds, _p(ws),
                                            ws.numel(), _stream())
    L.check(rc, "svtr_experts_forward")
    return feats, logits


# ------------------------------------------------------------------------------------------------ stage-0 expert training
def _train_slots():
    """The SVTR arena's slot table: every trainable MrnbSvtrPack slot, then the classifier head ("fc_w", "fc_b")."""
    cn = "model.FeatureExtraction.ConvNet."
    out = [(L.P_POS_EMBED, cn + "pos_embed", None), (L.P_CONV0_W, cn + "patch_embed.proj.0.weight", None),
           (L.P_CONV0_B, cn + "patch_embed.proj.0.bias", None), (L.P_BN0_W, cn + "patch_embed.proj.1.weight", None),
           (L.P_BN0_B, cn + "patch_embed.proj.1.bias", None),
           (L.P_CONV1_W, cn + "patch_embed.proj.3.weight", (0, 2, 3, 1)), (L.P_CONV1_B, cn + "patch_embed.proj.3.bias", None),
           (L.P_BN1_W, cn + "patch_embed.proj.4.weight", None), (L.P_BN1_B, cn + "patch_embed.proj.4.bias", None)]
    for b, name in enumerate(_BLOCK_NAMES):
        for k, key in enumerate(_BLOCK_KEYS):
            out.append((L.P_BLOCK0 + b * L.PB_COUNT + k, f"{cn}{name}.{key}", None))
    for s_ in range(3):
        base = L.P_SUB0 + s_ * L.PS_COUNT
        out += [(base + L.PS_CONV_W, f"{cn}sub_sample{s_ + 1}.conv.weight", (0, 2, 3, 1)),
                (base + L.PS_CONV_B, f"{cn}sub_sample{s_ + 1}.conv.bias", None),
                (base + L.PS_NORM_W, f"{cn}sub_sample{s_ + 1}.norm.weight", None),
                (base + L.PS_NORM_B, f"{cn}sub_sample{s_ + 1}.norm.bias", None)]
    out += [(L.P_SEQ_W, "model.SequenceModeling.0.weight", None), (L.P_SEQ_B, "model.SequenceModeling.0.bias", None),
            ("fc_w", "fc.weight", None), ("fc_b", "fc.bias", None)]
    return [(slot, [(key, perm)]) for slot, key, perm in out]


_BN_STAT_SLOTS = ((L.P_BN0_MEAN, "patch_embed.proj.1.running_mean"), (L.P_BN0_VAR, "patch_embed.proj.1.running_var"),
                  (L.P_BN1_MEAN, "patch_embed.proj.4.running_mean"), (L.P_BN1_VAR, "patch_embed.proj.4.running_var"))


class _TrainPack:
    """ONE expert's trainable parameters in a single flat fp32 arena, a gradient arena with the same layout, in bf16
    mode a bf16 shadow of the arena at the same element offsets (refreshed before every forward), and the expert's
    BatchNorm running statistics.  The arena is what mrnb_clip_adam updates and what the data-parallel all-reduce
    averages (stage 0, il_modules/mrn.py:225-279).  `entries` maps each arena slice back to its state_dict key.

    A subclass passes its slot table [(slot, [(key, permute), ...])] in arena order (the parts of a slot adjacent, each
    slot padded to 8 floats), names its C struct (_Struct) and puts a slot's pointers into it (_point).
    param_grads=False: no gradient arena (grads is None) -- the pack of a frozen expert that only carries the image
    gradient, run by the input-only backward."""

    def __init__(self, expert_sd: Dict[str, torch.Tensor], device, prec, slots, param_grads=True):
        self.device = torch.device(device)
        self.prec = prec
        self.entries = []                         # (slot, key, permute, offset, kernel-layout shape)
        self.slot_offset = {}
        off = 0
        for slot, parts in slots:
            self.slot_offset[slot] = off
            for key, perm in parts:
                shp = tuple(expert_sd[key].shape)
                if perm is not None:
                    shp = tuple(shp[a] for a in perm)
                self.entries.append((slot, key, perm, off, shp))
                n = math.prod(shp)
                assert n % 8 == 0 or len(parts) == 1, key
                off += n
            off = round_up(off, 8)
        self.numel = off
        self.params = torch.zeros(off, device=self.device, dtype=torch.float32)
        self.grads = torch.zeros(off, device=self.device, dtype=torch.float32) if param_grads else None
        self.shadow16 = torch.zeros(off, device=self.device, dtype=torch.bfloat16) if prec == L.PREC_BF16 else None
        self.n_class = int(expert_sd["fc.weight"].shape[0])
        self.struct = self._Struct()
        self.gstruct = self._Struct()
        for slot, o in self.slot_offset.items():
            self._point(self.struct, slot, self.params.data_ptr() + 4 * o,
                        None if self.shadow16 is None else self.shadow16.data_ptr() + 2 * o)
            if self.grads is not None:
                self._point(self.gstruct, slot, self.grads.data_ptr() + 4 * o, None)
        self.load_state(expert_sd)
        self._ws: Optional[torch.Tensor] = None

    def _bn_stat(self, expert_sd, key):
        return expert_sd["model.FeatureExtraction.ConvNet." + key].detach().to(self.device, torch.float32).clone().contiguous()

    def view(self, arena, entry):
        slot, key, perm, o, shp = entry
        return arena[o:o + math.prod(shp)].view(shp)

    def load_state(self, expert_sd):
        with torch.no_grad():
            for e in self.entries:
                t = expert_sd[e[1]].detach().to(self.device, torch.float32)
                if e[2] is not None:
                    t = t.permute(*e[2])
                self.view(self.params, e).copy_(t)

    def state(self, arena=None) -> Dict[str, torch.Tensor]:
        """{state_dict key: tensor in the reference's layout} read back from the arena (params by default)."""
        arena = self.params if arena is None else arena
        out = {}
        for e in self.entries:
            t = self.view(arena, e)
            if e[2] is not None:
                inv = [0] * len(e[2])
                for a, b in enumerate(e[2]):
                    inv[b] = a
                t = t.permute(*inv)
            out[e[1]] = t
        return out

    def refresh_shadow(self):
        if self.shadow16 is not None:
            L.check(L.load().mrnb_cast_f32_to_bf16(_p(self.params), _p(self.shadow16), self.numel, _stream()), "cast")


class SvtrTrainPack(_TrainPack):
    """An SVTR expert's training arena laid out in MrnbSvtrPack slots (n_experts = 1; conv weights as [Cout,kh,kw,Cin]);
    the BatchNorm running statistics sit in their MrnbSvtrPack slots, keyed by slot in `bn_stats`."""

    arch = "svtr"
    _Struct = L.MrnbSvtrPack

    def __init__(self, expert_sd: Dict[str, torch.Tensor], device, prec: int = L.PREC_FP32, param_grads: bool = True):
        super().__init__(expert_sd, device, prec, _train_slots(), param_grads)
        for st_ in (self.struct, self.gstruct):
            st_.n_experts = 1
            st_.n_class[0] = self.n_class
        self.bn_stats = {slot: self._bn_stat(expert_sd, key) for slot, key in _BN_STAT_SLOTS}
        for slot, t in self.bn_stats.items():
            self.struct.p[slot] = t.data_ptr()

    def bn_running_stats(self):
        """(mean0, var0, mean1, var1): updated in place by train-mode forwards."""
        return tuple(self.bn_stats[s] for s in (L.P_BN0_MEAN, L.P_BN0_VAR, L.P_BN1_MEAN, L.P_BN1_VAR))

    @staticmethod
    def _point(st, slot, ptr, ptr16):
        if slot == "fc_w":
            st.fc_w[0], st.fc_w16[0] = ptr, ptr16
        elif slot == "fc_b":
            st.fc_b[0] = ptr                      # the bias has no bf16 copy
        else:
            st.p[slot], st.h[slot] = ptr, ptr16

    def workspace(self, B):
        return _grow_workspace(self, int(L.load().mrnb_svtr_train_workspace_bytes(B, self.n_class, self.prec)))


def _features_out(B, T, device):
    """The training packs' feature output [B,T,256] fp32 (dense)."""
    return torch.empty(B, T, D_FEAT, device=device, dtype=torch.float32)


def _chk_dfeatures(dfeatures, B, T):
    if dfeatures is not None:
        _chk_f32(dfeatures)
        assert tuple(dfeatures.shape) == (B, T, D_FEAT) and dfeatures.is_contiguous(), "dfeatures must be dense [B,T,256]"


def svtr_train_forward(tp: SvtrTrainPack, image, bn_batch_stats=True, update_running=True, drop_scales=None,
                       want_features=False):
    """Activation-keeping forward of the expert being trained.  Returns logits [B,64,C] (a view of a padded buffer), or
    (logits, features [B,64,256]) with want_features."""
    _chk_f32(image, drop_scales)
    B = image.shape[0]
    ld = round_up(tp.n_class, 4)
    buf = torch.empty(B, T_FRAMES, ld, device=image.device, dtype=torch.float32)
    feats = _features_out(B, T_FRAMES, image.device) if want_features else None
    ws = tp.workspace(B)
    tp.refresh_shadow()
    L.check(L.load().mrnb_svtr_train_forward_features(C.byref(tp.struct), _p(image), B, tp.prec, int(bn_batch_stats),
                                                      int(update_running), _p(drop_scales), _p(buf), ld, _p(feats), _p(ws),
                                                      ws.numel(), _stream()), "svtr_train_forward")
    return (buf[:, :, :tp.n_class], feats) if want_features else buf[:, :, :tp.n_class]


def _grad_args(tp, param_grads, dimage, B):
    """(grads struct, arena, arena length) of a training-pack backward: NULLs for the input-only backward."""
    if dimage is not None:
        _chk_f32(dimage)
        assert tuple(dimage.shape) == (B, 4, 32, 256), "dimage must be dense [B,4,32,256]"
    if not param_grads:
        assert dimage is not None, "the input-only backward (param_grads=False) needs dimage"
        return None, None, 0
    assert tp.grads is not None, "this training pack has no gradient arena (built with param_grads=False)"
    return C.byref(tp.gstruct), tp.grads, tp.numel


def svtr_train_backward(tp: SvtrTrainPack, image, dlogits, bn_batch_stats=True, drop_scales=None, dfeatures=None,
                        dimage=None, param_grads=True):
    """Fills tp.grads (overwritten) from d loss / d logits [B,64,C] (+ d loss / d features [B,64,256] reaching the
    feature from outside the expert); must follow svtr_train_forward on the same batch.  dimage: None or an output
    tensor [B,4,32,256] fp32 that receives d loss / d image.  param_grads=False: the input-only backward (no parameter
    gradient; dimage required).  Returns tp.grads, or None without parameter gradients."""
    _chk_f32(image, drop_scales)
    assert dlogits.dtype == torch.float32 and dlogits.stride(2) == 1 and dlogits.stride(0) == dlogits.shape[1] * dlogits.stride(1)
    B = image.shape[0]
    _chk_dfeatures(dfeatures, B, T_FRAMES)
    gstruct, grads, n = _grad_args(tp, param_grads, dimage, B)
    ws = tp.workspace(B)
    L.check(L.load().mrnb_svtr_train_backward_input(C.byref(tp.struct), gstruct, _p(image), _p(dlogits), dlogits.stride(1),
                                                    _p(dfeatures), B, tp.prec, int(bn_batch_stats), _p(drop_scales), _p(grads),
                                                    n, _p(dimage), _p(ws), ws.numel(), _stream()), "svtr_train_backward")
    return grads


class CrnnTrainPack(_TrainPack):
    """A CRNN expert's training arena in MrnbCrnnTrainPack slots: conv weights as [Cout,kh,kw,Cin]; each LSTM tensor =
    forward direction then reverse direction in one slot.  `bn_stats` holds the two BatchNorms' running statistics,
    keyed (0 / 1, "mean" / "var")."""

    arch = "crnn"
    n_frames = 63
    _Struct = L.MrnbCrnnTrainPack

    def __init__(self, expert_sd: Dict[str, torch.Tensor], device, prec: int = L.PREC_FP32, param_grads: bool = True):
        cn = "model.FeatureExtraction.ConvNet."
        hwc = (0, 2, 3, 1)
        slots = [(L.T_CONV0_W, [(cn + "0.weight", hwc)]), (L.T_CONV0_B, [(cn + "0.bias", None)]),
                 (L.T_CONV1_W, [(cn + "3.weight", hwc)]), (L.T_CONV1_B, [(cn + "3.bias", None)]),
                 (L.T_CONV2_W, [(cn + "6.weight", hwc)]), (L.T_CONV2_B, [(cn + "6.bias", None)]),
                 (L.T_CONV3_W, [(cn + "8.weight", hwc)]), (L.T_CONV3_B, [(cn + "8.bias", None)]),
                 (L.T_CONV4_W, [(cn + "11.weight", hwc)]), (L.T_BN4_W, [(cn + "12.weight", None)]), (L.T_BN4_B, [(cn + "12.bias", None)]),
                 (L.T_CONV5_W, [(cn + "14.weight", hwc)]), (L.T_BN5_W, [(cn + "15.weight", None)]), (L.T_BN5_B, [(cn + "15.bias", None)]),
                 (L.T_CONV6_W, [(cn + "18.weight", hwc)]), (L.T_CONV6_B, [(cn + "18.bias", None)])]
        for k in range(2):
            q = f"model.SequenceModeling.{k}."
            base = L.T_LSTM0 + k * L.TL_COUNT
            for sl, nm in ((L.TL_WIH, "weight_ih_l0"), (L.TL_WHH, "weight_hh_l0"), (L.TL_BIH, "bias_ih_l0"), (L.TL_BHH, "bias_hh_l0")):
                slots.append((base + sl, [(q + "rnn." + nm, None), (q + "rnn." + nm + "_reverse", None)]))
            slots += [(base + L.TL_LIN_W, [(q + "linear.weight", None)]), (base + L.TL_LIN_B, [(q + "linear.bias", None)])]
        slots += [(L.T_FC_W, [("fc.weight", None)]), (L.T_FC_B, [("fc.bias", None)])]
        super().__init__(expert_sd, device, prec, slots, param_grads)
        self.bn_stats = {}
        for q, idx in enumerate((12, 15)):
            self.bn_stats[(q, "mean")] = self._bn_stat(expert_sd, f"{idx}.running_mean")
            self.bn_stats[(q, "var")] = self._bn_stat(expert_sd, f"{idx}.running_var")
        for st_ in (self.struct, self.gstruct):
            st_.n_class = self.n_class
            for q in range(2):
                st_.bn_mean[q] = self.bn_stats[(q, "mean")].data_ptr()
                st_.bn_var[q] = self.bn_stats[(q, "var")].data_ptr()

    def bn_running_stats(self):
        """(mean4, var4, mean5, var5): updated in place by train-mode forwards."""
        return tuple(self.bn_stats[(q, s)] for q in range(2) for s in ("mean", "var"))

    @staticmethod
    def _point(st, slot, ptr, ptr16):
        st.p[slot], st.h[slot] = ptr, ptr16

    def workspace(self, B):
        return _grow_workspace(self, int(L.load().mrnb_crnn_train_workspace_bytes(B, self.n_class, self.prec)))


def crnn_train_forward(tp: CrnnTrainPack, image, bn_batch_stats=True, update_running=True, want_features=False):
    """Activation-keeping forward of the CRNN expert being trained.  Returns logits [B,63,C], or (logits, features
    [B,63,256]) with want_features."""
    _chk_f32(image)
    B = image.shape[0]
    ld = round_up(tp.n_class, 4)
    buf = torch.empty(B, T_FRAMES_CRNN, ld, device=image.device, dtype=torch.float32)
    feats = _features_out(B, T_FRAMES_CRNN, image.device) if want_features else None
    ws = tp.workspace(B)
    tp.refresh_shadow()
    L.check(L.load().mrnb_crnn_train_forward_features(C.byref(tp.struct), _p(image), B, tp.prec, int(bn_batch_stats),
                                                      int(update_running), _p(buf), ld, _p(feats), _p(ws), ws.numel(),
                                                      _stream()), "crnn_train_forward")
    return (buf[:, :, :tp.n_class], feats) if want_features else buf[:, :, :tp.n_class]


def crnn_train_backward(tp: CrnnTrainPack, dlogits, B, bn_batch_stats=True, dfeatures=None, dimage=None, param_grads=True):
    """As svtr_train_backward, for the CRNN expert (dimage in the caller's NCHW layout)."""
    assert dlogits.dtype == torch.float32 and dlogits.stride(2) == 1 and dlogits.stride(0) == dlogits.shape[1] * dlogits.stride(1)
    _chk_dfeatures(dfeatures, B, T_FRAMES_CRNN)
    gstruct, grads, n = _grad_args(tp, param_grads, dimage, B)
    ws = tp.workspace(B)
    L.check(L.load().mrnb_crnn_train_backward_input(C.byref(tp.struct), gstruct, _p(dlogits), dlogits.stride(1), _p(dfeatures),
                                                    B, tp.prec, int(bn_batch_stats), _p(grads), n, _p(dimage), _p(ws),
                                                    ws.numel(), _stream()), "crnn_train_backward")
    return grads


def conv0_dimage(arch, d, w, out=None):
    """The conv0 input-gradient kernel of an expert's training-pack backward on its own: d = the gradient at conv0's
    output (NHWC [B,16,128,32] svtr / [B,32,256,64] crnn, fp32), w = the pack's conv0 weight ([32,4,3,3] / [64,3,3,4]).
    Returns dimage [B,4,32,256] (NCHW; `out` when given, overwritten)."""
    _chk_f32(d, w, out)
    B = d.shape[0]
    shape, wshape = ((B, 16, 128, 32), (32, 4, 3, 3)) if arch == "svtr" else ((B, 32, 256, 64), (64, 3, 3, 4))
    assert tuple(d.shape) == shape and tuple(w.shape) == wshape, (tuple(d.shape), tuple(w.shape))
    if out is None:
        out = torch.empty(B, 4, 32, 256, device=d.device, dtype=torch.float32)
    assert tuple(out.shape) == (B, 4, 32, 256)
    fn = L.load().mrnb_svtr_conv0_dimage if arch == "svtr" else L.load().mrnb_crnn_conv0_dimage
    L.check(fn(_p(d), _p(w), _p(out), B, _stream()), "conv0_dimage")
    return out


# ------------------------------------------------------------------------------------------------ CRNN experts

_VGG_GEMM_CONVS = ((L.C_CONV1_W, L.C_CONV1_B, 3), (L.C_CONV2_W, L.C_CONV2_B, 6), (L.C_CONV3_W, L.C_CONV3_B, 8),
                   (L.C_CONV4_W, None, 11), (L.C_CONV5_W, None, 14), (L.C_CONV6_W, L.C_CONV6_B, 18))


class CrnnPack:
    """Device-resident, expert-stacked copy of the CRNN expert parameters (include/mrn_b200.h: MRNB_C_* slots):
    VGG convolutions re-laid as [Cout, kh, kw, Cin], LSTM input weights of both directions concatenated, the two
    LSTM biases pre-summed.  Built from a reference-format state_dict."""

    arch = "crnn"
    n_frames = T_FRAMES_CRNN

    def __init__(self, state_dict: Dict[str, torch.Tensor], n_experts: int, device, prec: int, prefix: str = ""):
        self.n_experts = n_experts
        self.prec = prec
        self.device = torch.device(device)
        self.tensors: List[torch.Tensor] = []
        self.struct = L.MrnbCrnnPack()
        self.struct.n_experts = n_experts
        self.n_class: List[int] = []
        self.slot_tensors: Dict[int, torch.Tensor] = {}
        sd = state_dict

        def get(i, key):
            return sd[f"{prefix}model.{i}.{key}"].detach().to(self.device, torch.float32)

        def stack(fn):
            return torch.stack([fn(i).contiguous() for i in range(n_experts)], 0).contiguous()

        def put(slot, t, gemm_weight=False):
            self.tensors.append(t)
            self.slot_tensors[slot] = t
            self.struct.p[slot] = t.data_ptr()
            if gemm_weight and prec == L.PREC_BF16:
                h = cast_bf16(t)
                self.tensors.append(h)
                self.struct.h[slot] = h.data_ptr()

        cn = "model.FeatureExtraction.ConvNet."
        put(L.C_CONV0_W, stack(lambda i: get(i, cn + "0.weight")))
        if prec == L.PREC_BF16:
            # tensor-core conv0: [64, (c,kh,kw) = 36 taps zero-padded to 64] bf16 (im2col GEMM, crnn.cu)
            w0 = torch.zeros(n_experts, 64, 64, device=self.device, dtype=torch.float32)
            w0[:, :, :36] = self.slot_tensors[L.C_CONV0_W].reshape(n_experts, 64, 36)
            h0 = cast_bf16(w0.contiguous())
            self.tensors.append(h0)
            self.struct.h[L.C_CONV0_W] = h0.data_ptr()
        put(L.C_CONV0_B, stack(lambda i: get(i, cn + "0.bias")))
        for wslot, bslot, idx in _VGG_GEMM_CONVS:
            put(wslot, stack(lambda i: get(i, cn + f"{idx}.weight").permute(0, 2, 3, 1)), gemm_weight=True)
            if bslot is not None:
                put(bslot, stack(lambda i: get(i, cn + f"{idx}.bias")))
        for base, idx in ((L.C_BN4_W, 12), (L.C_BN5_W, 15)):
            for k, nm in enumerate(("weight", "bias", "running_mean", "running_var")):
                put(base + k, stack(lambda i: get(i, cn + f"{idx}.{nm}")))
        # gate axis interleaved per hidden unit: packed row 4*j + k <- nn.LSTM row k*256 + j (k = i,f,g,o)
        perm = (torch.arange(4).view(1, 4) * 256 + torch.arange(256).view(256, 1)).reshape(-1).to(self.device)

        def il(t):
            return t.index_select(0, perm)

        for layer in range(2):
            q = f"model.SequenceModeling.{layer}."
            base = L.C_LSTM0 + layer * L.CL_COUNT
            put(base + L.CL_WIH, stack(lambda i: torch.cat([il(get(i, q + "rnn.weight_ih_l0")),
                                                            il(get(i, q + "rnn.weight_ih_l0_reverse"))], 0)), gemm_weight=True)
            put(base + L.CL_WHH, stack(lambda i: torch.stack([il(get(i, q + "rnn.weight_hh_l0")),
                                                              il(get(i, q + "rnn.weight_hh_l0_reverse"))], 0)), gemm_weight=True)
            put(base + L.CL_BIAS, stack(lambda i: torch.cat([
                il(get(i, q + "rnn.bias_ih_l0") + get(i, q + "rnn.bias_hh_l0")),
                il(get(i, q + "rnn.bias_ih_l0_reverse") + get(i, q + "rnn.bias_hh_l0_reverse"))], 0)))
            put(base + L.CL_LIN_W, stack(lambda i: get(i, q + "linear.weight")), gemm_weight=True)
            put(base + L.CL_LIN_B, stack(lambda i: get(i, q + "linear.bias")))
        for i in range(n_experts):
            w = get(i, "fc.weight").contiguous()
            b = get(i, "fc.bias").contiguous()
            self.tensors += [w, b]
            self.struct.fc_w[i] = w.data_ptr()
            self.struct.fc_b[i] = b.data_ptr()
            self.struct.n_class[i] = w.shape[0]
            self.n_class.append(int(w.shape[0]))
            if prec == L.PREC_BF16:
                h = cast_bf16(w)
                self.tensors.append(h)
                self.struct.fc_w16[i] = h.data_ptr()
        self._ws: Optional[torch.Tensor] = None

    def bn_running_stats(self):
        """(mean4, var4, mean5, var5), each [I, 512]: updated in place by train-mode forwards."""
        return tuple(self.slot_tensors[s] for s in (L.C_BN4_MEAN, L.C_BN4_VAR, L.C_BN5_MEAN, L.C_BN5_VAR))

    def workspace(self, B, chunk=0):
        return _grow_workspace(self, int(L.load().mrnb_crnn_workspace_bytes(self.n_experts, B, self.prec)))


def crnn_experts_forward(pack: CrnnPack, image: torch.Tensor, bn_batch_stats: bool = False, update_running: bool = False,
                         want_logits: bool = True):
    """Runs every CRNN expert on `image` [B,4,32,256].  Returns (features [B,I,63,256], [logits_i [B,63,C_i] views])."""
    _chk_f32(image)
    B = image.shape[0]
    feats = torch.empty(B, pack.n_experts, T_FRAMES_CRNN, D_FEAT, device=image.device, dtype=torch.float32)
    ptrs, lds, logits = _logit_buffers(pack, B, image.device, want_logits)
    ws = pack.workspace(B)
    rc = L.load().mrnb_crnn_experts_forward(C.byref(pack.struct), _p(image), B, pack.prec, _mask(bn_batch_stats),
                                            _mask(update_running), _p(feats), ptrs, lds, _p(ws), ws.numel(), _stream())
    L.check(rc, "crnn_experts_forward")
    return feats, logits


# ------------------------------------------------------------------------------------------------ router
ROUTER_PARAM_NAMES = ("route.weight", "route.bias", "channel_route.weight", "channel_route.bias",
                      "dm_router.0.norm.weight", "dm_router.0.norm.bias",
                      "dm_router.0.proj_1.weight", "dm_router.0.proj_1.bias",
                      "dm_router.0.spatial_gating.norm.weight", "dm_router.0.spatial_gating.norm.bias",
                      "dm_router.0.spatial_gating.proj.weight", "dm_router.0.spatial_gating.proj.bias",
                      "dm_router.0.channel_gating.norm.weight", "dm_router.0.channel_gating.norm.bias",
                      "dm_router.0.channel_gating.proj.weight", "dm_router.0.channel_gating.proj.bias",
                      "dm_router.0.proj_2.weight", "dm_router.0.proj_2.bias",
                      "dm_router.0.proj_3.weight", "dm_router.0.proj_3.bias")


def router_param_offsets(n_experts: int, T: int = T_FRAMES, D: int = D_FEAT):
    off = (C.c_long * (L.ROUTER_NPARAMS + 1))()
    n = L.load().mrnb_router_param_offsets(n_experts, T, D, off)
    return int(n), [int(v) for v in off]


class RouterWorkspace:
    def __init__(self):
        self.buf: Optional[torch.Tensor] = None

    def get(self, B, I, T, D, bwd, device):
        need = int(L.load().mrnb_router_workspace_bytes(B, I, T, D, int(bwd)))
        if self.buf is None or self.buf.numel() < need or self.buf.device != device:
            self.buf = torch.empty(need, dtype=torch.uint8, device=device)
        return self.buf


def router_forward(params: torch.Tensor, x: torch.Tensor, ws: RouterWorkspace, with_backward=False, prec=L.PREC_FP32,
                   want_out=True):
    """params: flat fp32 arena; x [B,I,T,D].  Returns (out or None, scores [B,I], gate [B,I], index [B] int32)."""
    _chk_f32(params, x)
    B, I, T, D = x.shape
    out = torch.empty_like(x) if want_out else None
    scores = torch.empty(B, I, device=x.device, dtype=torch.float32)
    gate = torch.empty(B, I, device=x.device, dtype=torch.float32)
    index = torch.empty(B, device=x.device, dtype=torch.int32)
    w = ws.get(B, I, T, D, with_backward, x.device)
    L.check(L.load().mrnb_router_forward(_p(params), _p(x), B, I, T, D, prec, _p(out), _p(scores), _p(gate), _p(index),
                                         _p(w), w.numel(), _stream()), "router_forward")
    return out, scores, gate, index


def router_backward(params, x, gate, dgate_ctc, domain, grads, ws: RouterWorkspace, prec=L.PREC_FP32, dx=None):
    """domain [B] int64: loss = pi*CTC + CE(gate, domain), returns the CE term.  domain None: dgate_ctc is the whole
    dL/dgate of an arbitrary loss (no CE term), returns None.  dx (optional, like x): also the input gradient dL/dx
    (mrnb_router_backward_dx)."""
    _chk_f32(params, x, gate, dgate_ctc, grads)
    assert domain is None or domain.dtype == torch.int64
    B, I, T, D = x.shape
    taski = torch.empty(1, device=x.device, dtype=torch.float32) if domain is not None else None
    w = ws.get(B, I, T, D, True, x.device)
    if dx is None:
        L.check(L.load().mrnb_router_backward(_p(params), _p(x), _p(gate), _p(dgate_ctc), _p(domain), B, I, T, D, prec,
                                              _p(grads), _p(taski), _p(w), w.numel(), _stream()), "router_backward")
    else:
        _chk_f32(dx)
        assert dx.shape == x.shape and dx.is_contiguous()
        L.check(L.load().mrnb_router_backward_dx(_p(params), _p(x), _p(gate), _p(dgate_ctc), _p(domain), B, I, T, D, prec,
                                                 _p(grads), _p(dx), _p(taski), _p(w), w.numel(), _stream()), "router_backward_dx")
    return taski


def dm_router_backward(params, x, d_out, grads, ws: RouterWorkspace, want_dx=True, prec=L.PREC_FP32):
    _chk_f32(params, x, d_out, grads)
    B, I, T, D = x.shape
    dx = torch.empty_like(x) if want_dx else None
    w = ws.get(B, I, T, D, True, x.device)
    L.check(L.load().mrnb_dm_router_backward(_p(params), _p(x), _p(d_out), B, I, T, D, prec, _p(grads), _p(dx), _p(w),
                                             w.numel(), _stream()), "dm_router_backward")
    return dx


# ------------------------------------------------------------------------------------------------ combine / CTC / decode
def _expert_tables(logits: Sequence[torch.Tensor]):
    I = len(logits)
    ptrs = (C.c_void_p * I)()
    lds = (C.c_long * I)()
    cs = (C.c_int * I)()
    for i, z in enumerate(logits):
        if z.dtype != torch.float32 or z.stride(-1) != 1 or z.stride(0) != z.shape[1] * z.stride(1):
            raise RuntimeError("expert logits must be fp32 [B,T,C_i] with a dense row layout")
        ptrs[i] = z.data_ptr()
        lds[i] = z.stride(1)
        cs[i] = z.shape[2]
    return ptrs, lds, cs


def gate_combine(logits: Sequence[torch.Tensor], gate: torch.Tensor, targets: Optional[torch.Tensor] = None,
                 lengths: Optional[torch.Tensor] = None, want_logits=False, want_E=False, want_decode=False):
    """Fused pad-with-ones + gated sum + row log-sum-exp (+ label gathers, + argmax).  Returns a dict."""
    _chk_f32(gate)
    B, T, _ = logits[0].shape
    I = len(logits)
    Cmax = logits[-1].shape[2]
    dev = gate.device
    ptrs, lds, cs = _expert_tables(logits)
    r = dict(lse=torch.empty(B, T, device=dev, dtype=torch.float32))
    ldo = round_up(Cmax, 4)
    if want_logits:
        buf = torch.empty(B, T, ldo, device=dev, dtype=torch.float32)
        r["logits_buf"] = buf
        r["logits"] = buf[:, :, :Cmax]
    if want_E:
        r["E"] = torch.empty(B, T, I, device=dev, dtype=torch.float32)
    if want_decode:
        r["amax"] = torch.empty(B, T, device=dev, dtype=torch.int32)
        r["maxprob"] = torch.empty(B, T, device=dev, dtype=torch.float32)
    Lmax = 0
    if targets is not None:
        assert targets.dtype == torch.int64 and lengths.dtype == torch.int32 and targets.is_contiguous()
        Lmax = targets.shape[1]
        r["lpe"] = torch.empty(B, T, Lmax + 1, device=dev, dtype=torch.float32)
        r["zlab"] = torch.empty(B, T, Lmax + 1, I, device=dev, dtype=torch.float32)
    L.check(L.load().mrnb_gate_combine(ptrs, lds, cs, I, _p(gate), B, T, _p(r.get("logits_buf")), ldo, _p(r["lse"]),
                                       _p(r.get("E")), _p(r.get("amax")), _p(r.get("maxprob")), _p(targets), _p(lengths),
                                       Lmax, _p(r.get("lpe")), _p(r.get("zlab")), _stream()), "gate_combine")
    return r


def _aligned_dY(logits: Sequence[torch.Tensor], dY: torch.Tensor):
    """dY [B,T,C] checked and, when its rows are not 16-byte aligned, copied into a padded buffer."""
    B, T, _ = logits[0].shape
    I, C = len(logits), logits[-1].shape[2]
    ptrs, lds, cs = _expert_tables(logits)
    if dY.dtype != torch.float32 or tuple(dY.shape) != (B, T, C) or not dY.is_cuda:
        raise RuntimeError("gate_combine_backward: dY must be a CUDA float32 tensor [B,T,C] = %s" % ((B, T, C),))
    if not (dY.stride(2) == 1 and dY.stride(1) % 4 == 0 and dY.stride(0) == T * dY.stride(1) and dY.data_ptr() % 16 == 0):
        buf = torch.zeros(B, T, round_up(C, 4), device=dY.device, dtype=torch.float32)
        buf[:, :, :C].copy_(dY)
        dY = buf[:, :, :C]
    ws = torch.empty(int(L.load().mrnb_gate_combine_backward_workspace_bytes(B, T, I)), dtype=torch.uint8, device=dY.device)
    return dY, ptrs, lds, cs, ws


def gate_combine_backward(logits: Sequence[torch.Tensor], dY: torch.Tensor, out: Optional[torch.Tensor] = None):
    """dgate [B,I] = d<dY, combined logits>/dgate for a dense upstream gradient dY [B,T,C] over the union charset (same
    expert table as gate_combine; the pad value 1.0 counts).  dY rows that are not 16-byte aligned are first copied
    into a padded buffer.  `out` may supply dgate."""
    dY, ptrs, lds, cs, ws = _aligned_dY(logits, dY)
    B, T, I = dY.shape[0], dY.shape[1], len(logits)
    dgate = _out(out, (B, I), dY.device, torch.float32)
    L.check(L.load().mrnb_gate_combine_backward(ptrs, lds, cs, I, B, T, _p(dY), dY.stride(1), _p(dgate), _p(ws), ws.numel(),
                                                _stream()), "gate_combine_backward")
    return dgate


def gate_combine_backward_experts(logits: Sequence[torch.Tensor], dY: torch.Tensor, gate: torch.Tensor,
                                  dz: Sequence[Optional[torch.Tensor]], out: Optional[torch.Tensor] = None):
    """gate_combine_backward plus, in the same pass, dz[i] = gate[:, i] * dY[:, :, :C_i] for every dz[i] given (fp32
    [B,T,C_i] views with a dense row layout, 16-byte aligned rows); a None entry (a frozen expert) is skipped.
    Returns dgate."""
    dY, ptrs, lds, cs, ws = _aligned_dY(logits, dY)
    B, T, I = dY.shape[0], dY.shape[1], len(logits)
    _chk_f32(gate)
    assert tuple(gate.shape) == (B, I) and len(dz) == I
    dzp = (C.c_void_p * I)()
    ldz = (C.c_long * I)()
    for i, t in enumerate(dz):
        if t is not None:
            if t.dtype != torch.float32 or tuple(t.shape) != (B, T, cs[i]) or t.stride(2) != 1 or t.stride(0) != T * t.stride(1):
                raise RuntimeError("gate_combine_backward_experts: dz[%d] must be fp32 [B,T,C_i] with a dense row layout" % i)
            dzp[i], ldz[i] = t.data_ptr(), t.stride(1)
    dgate = _out(out, (B, I), dY.device, torch.float32)
    L.check(L.load().mrnb_gate_combine_backward_experts(ptrs, lds, cs, I, B, T, _p(dY), dY.stride(1), _p(gate), dzp, ldz,
                                                        _p(dgate), _p(ws), ws.numel(), _stream()),
            "gate_combine_backward_experts")
    return dgate


def ctc_lattice(lpe, targets, lengths, zlab=None, E=None, grad_scale=0.0, want_dgate=False, want_occ=False):
    B, T, S1 = lpe.shape
    I = zlab.shape[-1] if zlab is not None else 0
    dev = lpe.device
    nll = torch.empty(B, device=dev, dtype=torch.float32)
    loss = torch.empty(1, device=dev, dtype=torch.float32)
    dgate = torch.empty(B, I, device=dev, dtype=torch.float32) if want_dgate else None
    occ = torch.empty(B, T, S1, device=dev, dtype=torch.float32) if want_occ else None
    L.check(L.load().mrnb_ctc_lattice(_p(lpe), _p(zlab), _p(E), _p(targets), _p(lengths), S1 - 1, B, T, I, float(grad_scale),
                                      _p(nll), _p(loss), _p(dgate), _p(occ), _stream()), "ctc_lattice")
    return dict(nll=nll, loss=loss, dgate=dgate, occ=occ)


def ctc_dense_grad(logits_view, lse, occ, nll, targets, lengths, grad_scale):
    B, T, Cc = logits_view.shape
    ld = round_up(Cc, 4)                     # 16-byte aligned rows for the consumers' vector loads
    buf = torch.empty(B, T, ld, device=lse.device, dtype=torch.float32)
    L.check(L.load().mrnb_ctc_dense_grad(_p(logits_view), logits_view.stride(1), _p(lse), _p(occ), _p(nll), _p(targets),
                                         _p(lengths), targets.shape[1], B, T, Cc, float(grad_scale), _p(buf), ld, _stream()),
            "ctc_dense_grad")
    return buf[:, :, :Cc]


def greedy_decode(amax, maxprob):
    B, T = amax.shape
    ids = torch.empty(B, T, device=amax.device, dtype=torch.int32)
    lens = torch.empty(B, device=amax.device, dtype=torch.int32)
    conf = torch.empty(B, device=amax.device, dtype=torch.float32)
    L.check(L.load().mrnb_greedy_decode(_p(amax), _p(maxprob), B, T, _p(ids), _p(lens), _p(conf), _stream()), "greedy_decode")
    return ids, lens, conf


def ctc_topk(logits: Sequence[torch.Tensor], gate: torch.Tensor, lse: torch.Tensor, K: int, out=None):
    """Per-frame CTC candidates for the beam search: the K best non-blank classes of the combined logits (same expert
    table and gate as gate_combine, lse from it).  Returns (top_ids [B,T,K] int32, top_lp [B,T,K], blank_lp [B,T]);
    `out` may supply those three tensors."""
    _chk_f32(gate, lse)
    B, T, _ = logits[0].shape
    dev = gate.device
    ptrs, lds, cs = _expert_tables(logits)
    if tuple(gate.shape) != (B, len(logits)) or tuple(lse.shape) != (B, T):
        raise RuntimeError("ctc_topk: gate must be [B,I] and lse [B,T]")
    o = out or (None, None, None)
    top_ids = _out(o[0], (B, T, K), dev, torch.int32)
    top_lp = _out(o[1], (B, T, K), dev, torch.float32)
    blank_lp = _out(o[2], (B, T), dev, torch.float32)
    L.check(L.load().mrnb_ctc_topk(ptrs, lds, cs, len(logits), _p(gate), _p(lse), B, T, K, _p(top_ids), _p(top_lp),
                                   _p(blank_lp), _stream()), "ctc_topk")
    return top_ids, top_lp, blank_lp


def ctc_beam_search(top_ids: torch.Tensor, top_lp: torch.Tensor, blank_lp: torch.Tensor, W: int, n_best: int = 1,
                    out=None):
    """CTC prefix beam search of width W over the ctc_topk candidates.  Returns (ids [B,n_best,T] int32 compact and
    -1 padded, lens [B,n_best] int32, scores [B,n_best] = log p of each labeling), best first; `out` may supply them."""
    _chk_f32(top_lp, blank_lp)
    if top_ids.dtype != torch.int32 or not top_ids.is_contiguous():
        raise RuntimeError("ctc_beam_search: top_ids must be a contiguous int32 tensor")
    B, T, K = top_ids.shape
    if tuple(top_lp.shape) != (B, T, K) or tuple(blank_lp.shape) != (B, T):
        raise RuntimeError("ctc_beam_search: top_lp must be [B,T,K] and blank_lp [B,T]")
    dev = top_ids.device
    o = out or (None, None, None)
    ids = _out(o[0], (B, n_best, T), dev, torch.int32)
    lens = _out(o[1], (B, n_best), dev, torch.int32)
    scores = _out(o[2], (B, n_best), dev, torch.float32)
    L.check(L.load().mrnb_ctc_beam_search(_p(top_ids), _p(top_lp), _p(blank_lp), B, T, K, int(W), int(n_best), _p(ids),
                                          _p(lens), _p(scores), _stream()), "ctc_beam_search")
    return ids, lens, scores


# ------------------------------------------------------------------------------------------------ optimiser
def clip_adam(params, grads, exp_avg, exp_avg_sq, lr, step, max_norm=5.0, betas=(0.9, 0.999), eps=1e-8, scratch=None,
              norm_out=None):
    _chk_f32(params, grads, exp_avg, exp_avg_sq)
    if scratch is None:
        scratch = torch.empty(4096, dtype=torch.uint8, device=params.device)
    if norm_out is None:
        norm_out = torch.empty(1, dtype=torch.float32, device=params.device)
    L.check(L.load().mrnb_clip_adam(_p(params), _p(grads), _p(exp_avg), _p(exp_avg_sq), params.numel(), float(lr),
                                    float(betas[0]), float(betas[1]), float(eps), float(max_norm), int(step), _p(norm_out),
                                    _p(scratch), _stream()), "clip_adam")
    return norm_out
