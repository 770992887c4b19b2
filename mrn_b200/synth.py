"""Deterministic synthetic weights and inputs shared by bench.py, the tests and the golden generator, and the one
set-up the tests and tools build the mirror's MRNNet / MRN learner with (make_opt, build_net, build_learner).

Data generation only (no reference code, no oracle arithmetic): numpy PCG64 streams keyed by
(seed, crc32(name)) so the same tensors can be rebuilt on the GPU box without shipping weights.
Key names and shapes are the reference's state_dict contract (SURVEY.md §8b; verified strict=True against
the reference modules by oracle/make_golden.py).
"""
from __future__ import annotations

import argparse
import zlib
from collections import OrderedDict
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch

MLT17_CLASS_COUNTS = (1899, 2224, 3844, 4968, 5041, 5153)   # README.md:100 cumulative + 4 specials


def _rng(seed: int, name: str):
    return np.random.default_rng([seed, zlib.crc32(name.encode())])


def randn(seed: int, name: str, shape, scale=1.0) -> torch.Tensor:
    a = _rng(seed, name).standard_normal(tuple(shape), dtype=np.float32) * np.float32(scale)
    return torch.from_numpy(a)


def svtr_expert_shapes(prefix: str, n_class: int) -> "OrderedDict[str, Tuple[int, ...]]":
    """state_dict keys of one Model(opt) with SVTR / None / CTC (modules/model.py:105-199, modules/svtr.py:315-479)."""
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    c = prefix + "model.FeatureExtraction.ConvNet."
    s[c + "pos_embed"] = (1, 512, 64)
    for idx, (ci, co) in ((0, (4, 32)), (3, (32, 64))):
        s[c + f"patch_embed.proj.{idx}.weight"] = (co, ci, 3, 3)
        s[c + f"patch_embed.proj.{idx}.bias"] = (co,)
        for nm in ("weight", "bias", "running_mean", "running_var"):
            s[c + f"patch_embed.proj.{idx + 1}.{nm}"] = (co,)
        s[c + f"patch_embed.proj.{idx + 1}.num_batches_tracked"] = ()
    dims, depth = (64, 128, 256), (3, 6, 3)
    outs = (128, 256, 512)
    for st in range(3):
        d = dims[st]
        for j in range(depth[st]):
            b = c + f"blocks{st + 1}.{j}."
            s[b + "norm1.weight"] = (d,); s[b + "norm1.bias"] = (d,)
            s[b + "mixer.qkv.weight"] = (3 * d, d); s[b + "mixer.qkv.bias"] = (3 * d,)
            s[b + "mixer.proj.weight"] = (d, d); s[b + "mixer.proj.bias"] = (d,)
            s[b + "norm2.weight"] = (d,); s[b + "norm2.bias"] = (d,)
            s[b + "mlp.fc1.weight"] = (4 * d, d); s[b + "mlp.fc1.bias"] = (4 * d,)
            s[b + "mlp.fc2.weight"] = (d, 4 * d); s[b + "mlp.fc2.bias"] = (d,)
        ss = c + f"sub_sample{st + 1}."
        s[ss + "conv.weight"] = (outs[st], d, 3, 3); s[ss + "conv.bias"] = (outs[st],)
        s[ss + "norm.weight"] = (outs[st],); s[ss + "norm.bias"] = (outs[st],)
    # constructed but never used in forward (modules/svtr.py:464-479)
    s[c + "linear.weight"] = (512, 384); s[c + "linear.bias"] = (512,)
    s[c + "last_conv.weight"] = (512, 256, 1, 1)
    s[c + "norm.weight"] = (256,); s[c + "norm.bias"] = (256,)
    s[prefix + "model.SequenceModeling.0.weight"] = (256, 512)
    s[prefix + "model.SequenceModeling.0.bias"] = (256,)
    s[prefix + "fc.weight"] = (n_class, 256); s[prefix + "fc.bias"] = (n_class,)
    s[prefix + "Prediction.weight"] = (n_class, 256); s[prefix + "Prediction.bias"] = (n_class,)
    return s


VGG_CONVS = ((0, 4, 64, 3, True), (3, 64, 128, 3, True), (6, 128, 256, 3, True), (8, 256, 256, 3, True),
             (11, 256, 512, 3, False), (14, 512, 512, 3, False), (18, 512, 512, 2, True))   # (index, Cin, Cout, k, bias)
VGG_BNS = (12, 15)


def crnn_expert_shapes(prefix: str, n_class: int) -> "OrderedDict[str, Tuple[int, ...]]":
    """state_dict keys of one Model(opt) with VGG / BiLSTM / CTC (modules/feature_extraction.py:19-47,
    modules/sequence_modeling.py:4-22, modules/model.py:46-78,176-181)."""
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    c = prefix + "model.FeatureExtraction.ConvNet."
    for idx, ci, co, k, bias in VGG_CONVS:
        s[c + f"{idx}.weight"] = (co, ci, k, k)
        if bias:
            s[c + f"{idx}.bias"] = (co,)
        if idx + 1 in VGG_BNS:
            for nm in ("weight", "bias", "running_mean", "running_var"):
                s[c + f"{idx + 1}.{nm}"] = (co,)
            s[c + f"{idx + 1}.num_batches_tracked"] = ()
    for layer, kin in ((0, 512), (1, 256)):
        q = prefix + f"model.SequenceModeling.{layer}."
        for suf in ("", "_reverse"):
            s[q + "rnn.weight_ih_l0" + suf] = (1024, kin)
            s[q + "rnn.weight_hh_l0" + suf] = (1024, 256)
            s[q + "rnn.bias_ih_l0" + suf] = (1024,)
            s[q + "rnn.bias_hh_l0" + suf] = (1024,)
        s[q + "linear.weight"] = (256, 512); s[q + "linear.bias"] = (256,)
    s[prefix + "fc.weight"] = (n_class, 256); s[prefix + "fc.bias"] = (n_class,)
    s[prefix + "Prediction.weight"] = (n_class, 256); s[prefix + "Prediction.bias"] = (n_class,)
    return s


def crnn_mrn_shapes(class_counts: Sequence[int]) -> "OrderedDict[str, Tuple[int, ...]]":
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    for i, c in enumerate(class_counts):
        s.update(crnn_expert_shapes(f"model.{i}.", c))
    s.update(router_shapes(len(class_counts), T=63))          # modules/model.py:322-323: patch = 63 for VGG
    return s


def router_shapes(n_experts: int, T: int = 64, D: int = 256) -> "OrderedDict[str, Tuple[int, ...]]":
    """route / channel_route / dm_router.0.* (modules/model.py:437-452, modules/dm_router.py:35-47)."""
    I = n_experts
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    s["route.weight"] = (1, T); s["route.bias"] = (1,)
    s["channel_route.weight"] = (I, I * D); s["channel_route.bias"] = (I,)
    r = "dm_router.0."
    s[r + "norm.weight"] = (D,); s[r + "norm.bias"] = (D,)
    s[r + "proj_1.weight"] = (2 * D, D); s[r + "proj_1.bias"] = (2 * D,)
    s[r + "spatial_gating.norm.weight"] = (D,); s[r + "spatial_gating.norm.bias"] = (D,)
    s[r + "spatial_gating.proj.weight"] = (I * T, I * T); s[r + "spatial_gating.proj.bias"] = (I * T,)
    s[r + "channel_gating.norm.weight"] = (T,); s[r + "channel_gating.norm.bias"] = (T,)
    s[r + "channel_gating.proj.weight"] = (I * D, I * D); s[r + "channel_gating.proj.bias"] = (I * D,)
    s[r + "proj_2.weight"] = (D, D); s[r + "proj_2.bias"] = (D,)
    s[r + "proj_3.weight"] = (D, D); s[r + "proj_3.bias"] = (D,)
    return s


def svtr_mrn_shapes(class_counts: Sequence[int]) -> "OrderedDict[str, Tuple[int, ...]]":
    s: "OrderedDict[str, Tuple[int, ...]]" = OrderedDict()
    for i, c in enumerate(class_counts):
        s.update(svtr_expert_shapes(f"model.{i}.", c))
    s.update(router_shapes(len(class_counts)))
    return s


def synth_tensor(seed: int, key: str, shape) -> torch.Tensor:
    """Value rule per parameter kind; scales keep activations O(1) through 12 blocks so that logits,
    gates and CTC are numerically non-trivial (random-init gates are otherwise all ~1/I)."""
    leaf = key.rsplit(".", 1)[-1]
    if leaf == "num_batches_tracked":
        return torch.tensor(0, dtype=torch.long)
    if leaf == "running_var":
        return 0.5 + randn(seed, key, shape).abs()
    if leaf == "running_mean":
        return randn(seed, key, shape, 0.1)
    if key.endswith("pos_embed"):
        return randn(seed, key, shape, 0.2)
    is_norm = (".norm" in key) or ("patch_embed.proj.1." in key) or ("patch_embed.proj.4." in key) \
        or ("ConvNet.12." in key) or ("ConvNet.15." in key)
    if is_norm and len(shape) == 1:
        return (1.0 + randn(seed, key, shape, 0.1)) if leaf == "weight" else randn(seed, key, shape, 0.1)
    if leaf == "bias":
        return randn(seed, key, shape, 0.05)
    fan_in = int(np.prod(shape[1:])) if len(shape) > 1 else int(shape[0])
    gain = 1.0
    if "ConvNet." in key and key.split("ConvNet.")[1].split(".")[0].isdigit():
        gain = 1.4         # VGG: ReLU halves the second moment, keep activations O(1) through 7 convolutions
    if "rnn.weight_hh" in key:
        fan_in = 256
    if key.startswith("route.") or key.startswith("channel_route."):
        gain = 1.5         # spread the gate away from uniform
    if ".fc." in key or ".Prediction." in key:
        gain = 4.0         # logits with a few-unit spread so argmax / CTC are informative
    return randn(seed, key, shape, gain / np.sqrt(fan_in))


def synth_state_dict(class_counts: Sequence[int], seed: int = 111, arch: str = "svtr") -> "OrderedDict[str, torch.Tensor]":
    sd: "OrderedDict[str, torch.Tensor]" = OrderedDict()
    shapes = svtr_mrn_shapes(class_counts) if arch == "svtr" else crnn_mrn_shapes(class_counts)
    for k, shp in shapes.items():
        kk = k.replace(".Prediction.", ".fc.")      # Prediction is the same nn.Linear object as fc (model.py:181)
        sd[k] = synth_tensor(seed, kk, shp)
    return sd


def synth_batch(B: int, class_counts: Sequence[int], seed: int = 111, max_len: int = 25):
    """Synthetic batch per SURVEY.md §8d: images randn.clamp(-1,1) [B,4,32,256]; target lengths 1..25;
    label ids in [2, C); padded with 1; domain ids in [0, I)."""
    C = class_counts[-1]
    img = randn(seed, "image", (B, 4, 32, 256)).clamp_(-1, 1)
    g = _rng(seed, "labels")
    lens = g.integers(1, max_len + 1, size=B)
    tgt = np.ones((B, max_len), dtype=np.int64)
    for b in range(B):
        tgt[b, :lens[b]] = g.integers(2, C, size=lens[b])
    dom = g.integers(0, len(class_counts), size=B)
    return img, torch.from_numpy(tgt), torch.from_numpy(lens.astype(np.int32)), torch.from_numpy(dom.astype(np.int64))


def synth_drop_scales(n_experts: int, B: int, rates: Sequence[float], seed: int = 111) -> torch.Tensor:
    """DropPath multipliers [I, 12, 2, B]: 0 with prob p, else 1/(1-p) (modules/svtr.py:7-22)."""
    g = _rng(seed, "droppath")
    out = np.ones((n_experts, len(rates), 2, B), dtype=np.float32)
    for j, p in enumerate(rates):
        if p <= 0:
            continue
        keep = g.random(size=(n_experts, 2, B)) >= p
        out[:, j] = keep.astype(np.float32) / np.float32(1.0 - p)
    return torch.from_numpy(out)


def ctor_state_dict(class_counts: Sequence[int], seed: int = 111, arch: str = "svtr") -> "OrderedDict[str, torch.Tensor]":
    """Random-init weights drawn by the mirror modules' own constructors, which restate the reference's initialisers
    (modules/svtr.py:488-498 trunc_normal / LayerNorm bias 1.0 / kaiming convs; nn.Linear, nn.Conv2d and nn.LSTM defaults
    elsewhere; router rebuilt by update_fc, modules/model.py:437-452) -- the "random-init weights" BASELINE.json's
    tolerances and metric are quoted on.  Gates come out soft (~1/I), unlike the gate-spreading synth_state_dict.
    Deterministic on the CPU generator for a given (seed, class_counts, arch)."""
    gen_state = torch.get_rng_state()
    torch.manual_seed(seed)
    try:
        net = build_net(class_counts, arch=arch, device=None)
        sd = OrderedDict((k, v.detach().clone()) for k, v in net.state_dict().items())
        for k in sd:                        # non-trivial BatchNorm running statistics (eval-mode experts use them)
            if k.endswith("running_var"):
                sd[k] = 0.5 + torch.rand_like(sd[k])
            elif k.endswith("running_mean"):
                sd[k] = 0.1 * torch.randn_like(sd[k])
    finally:
        torch.set_rng_state(gen_state)
    return sd


# ------------------------------------------------------------------------------------------------ set-up outside a run
def make_opt(arch: str = "svtr", precision: str = "fp32", **overrides) -> argparse.Namespace:
    """The reference's option namespace (config/svtr_mrn.py, config/crnn_mrn.py) for building MRNNet / MRN without the
    data pipeline: the model fields of `arch`, the training fields the learner reads, `overrides` on top."""
    opt = argparse.Namespace(Transformation="None", FeatureExtraction="SVTR" if arch == "svtr" else "VGG",
                             SequenceModeling="None" if arch == "svtr" else "BiLSTM", Prediction="CTC", num_fiducial=20,
                             input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256, batch_max_length=25,
                             lr=5e-4, num_iter=10000, grad_clip=5, exp_name="test", precision=precision, drop_path=False,
                             autograd=False, expert_chunk=0, lan_list=list("abcdef"), val_interval=5000, start_task=0,
                             optimizer="adam", schedule="super")
    vars(opt).update(overrides)
    return opt


def build_net(class_counts: Sequence[int], state_dict=None, opt=None, *, device="cuda", **opt_kw):
    """MRNNet grown one expert per class count as the reference grows it per task (update_fc + build_prediction),
    `state_dict` loaded strict=True when given, moved to `device` (None: left on the CPU).  Without `opt` the options
    are make_opt(**opt_kw)."""
    from .modules.model import MRNNet
    assert opt is None or not opt_kw, "options come from opt or from make_opt keywords, not both"
    if opt is None:
        opt = make_opt(**opt_kw)
    net = MRNNet(opt)
    for c in class_counts:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    if state_dict is not None:
        res = net.load_state_dict(state_dict, strict=True)      # the state_dict contract (SURVEY.md §8b)
        assert not res.missing_keys and not res.unexpected_keys
    return net if device is None else net.to(device)


def build_learner(net, *, train: bool = True, total_steps=None, schedule: str = "const"):
    """MRN learner over `net` with net.opt, its model in train or eval mode; with `total_steps` also the fused router
    optimiser (lr and grad_clip from net.opt)."""
    from .il_modules.mrn import MRN, RankLocal, FusedAdam
    learner = MRN(net.opt)
    learner.model = RankLocal(net)
    learner.model.train(train)
    if total_steps is not None:
        learner.optimizer = FusedAdam(net, net.opt.lr, total_steps, grad_clip=net.opt.grad_clip, schedule=schedule)
    return learner
