"""Joint expert and router training through autograd (opt.autograd + opt.autograd_experts): MRNNet's soft route
differentiated with respect to the router AND the trainable experts, as the reference differentiates it -- nothing is
detached between the experts and the DM-Router (modules/model.py:397-423), so a trainable expert gets gradient through
its logits (gated combine) and through its feature (DM-Router + gate head).

The three kernels the backward adds are checked on their own first (combine backward with per-expert logit gradients,
router backward with the input gradient, training packs with a feature output and a feature-gradient input), then the
reference's stage-1 loop end to end against fp64 autograd of the oracle with the expert parameters requiring grad."""
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import mrn_oracle as O
from mrn_b200 import synth
from conftest import rel_err
from persistent_walk import assert_walk, combine_walk

ROUTER_PREFIXES = ("route.", "channel_route.", "dm_router.0.")


def _ctc(logits, tgt, lens):
    B, T = logits.shape[:2]
    return F.ctc_loss(logits.log_softmax(2).permute(1, 0, 2), tgt, torch.full((B,), T, dtype=torch.long, device=tgt.device),
                      lens.long(), blank=0, reduction="mean", zero_infinity=True)


def _stage1_loop(net, x, tgt, lens, dom):
    """The reference's stage-1 loss (il_modules/mrn.py:338-362): 15 * CTC + CrossEntropy on the softmaxed gate."""
    out = net(x, True, None, True)
    loss = 15 * _ctc(out["logits"], tgt, lens) + F.cross_entropy(out["index"], dom)
    loss.backward()
    return loss


def _set_trainable(net, trainable):
    for e, m in enumerate(net.model):
        for p in m.parameters():
            p.requires_grad = e in trainable


def _joint_oracle(sd, I, img, tgt, lens, dom, trainable, bn_mode="eval", drop=None, stats=None):
    """fp64 autograd of O.mrn_forward's soft route under the stage-1 loss, with the router keys and the expert keys of
    `trainable` requiring grad.  The frozen experts run under no_grad (host memory).  stats: a dict that receives each
    batch-statistics BatchNorm input's (mean, unbiased var) by parameter prefix."""
    sd64 = {k: (v.detach().double() if v.is_floating_point() else v) for k, v in sd.items()}
    keys = list(O.ROUTER_KEYS) + [k for e in trainable for k in O.expert_param_keys(sd, e)]
    for k in keys:
        sd64[k].requires_grad_(True)
    bn = O._bn

    def recording_bn(x, sd_, p, mode, eps=1e-5):
        if mode != "eval" and stats is not None:
            xd = x.detach()
            stats[p] = (xd.mean(dim=(0, 2, 3)), xd.var(dim=(0, 2, 3), unbiased=True))
        return bn(x, sd_, p, mode, eps)

    feats, preds = [], []
    with pytest.MonkeyPatch.context() as m:
        m.setattr(O, "_bn", recording_bn)
        for i in range(I):
            ds = None if drop is None else drop[i].double()
            with torch.set_grad_enabled(i in trainable):
                f, z = O.expert_forward(sd64, i, img.double(), bn_mode, ds)
            feats.append(f)
            preds.append(z)
    gate = torch.softmax(O.gate_scores(sd64, O.dm_router(sd64, torch.stack(feats, 1))), -1)
    logits = O.combine_soft(preds, gate)
    loss = 15 * _ctc(logits, tgt, lens) + F.cross_entropy(gate, dom)
    grads = torch.autograd.grad(loss, [sd64[k] for k in keys], allow_unused=True)
    return dict(loss=float(loss.detach()), logits=logits.detach(), gate=gate.detach(),
                grads={k: (g if g is not None else torch.zeros_like(sd64[k])) for k, g in zip(keys, grads)})


# ------------------------------------------------------------------------------------------------ 1. combine kernel
@pytest.mark.gpu
@pytest.mark.parametrize("gate_kind", ["soft", "onehot", "zero"])
def test_combine_backward_experts_matches_fp64(gate_kind):
    """mrnb_gate_combine_backward_experts at B = 64 with the MLT17 class counts, dz asked for experts 0, 3 and 5: every
    dz element within 1e-6 relative of gate * dY in fp64 (one fp32 product), NaN-prefilled outputs overwritten, the
    frozen experts' buffers and every ld padding column still NaN, dgate bitwise mrnb_gate_combine_backward's, two runs
    bitwise equal, >= 4 rows per persistent CTA."""
    from mrn_b200 import ops
    cc, B, T = synth.MLT17_CLASS_COUNTS, 64, 64
    I, C = len(cc), cc[-1]
    rows, grid = combine_walk(B, T)
    assert_walk(rows, grid, "combine_bwd_tma_kernel")
    gen = torch.Generator(device="cuda").manual_seed(9)

    def padded(c, fill=None):
        buf = torch.full((B, T, ops.round_up(c, 4)), float("nan"), device="cuda")
        if fill is None:
            buf[:, :, :c] = torch.randn(B, T, c, device="cuda", generator=gen)
        return buf, buf[:, :, :c]
    z = [padded(c)[1] for c in cc]
    dY = padded(C)[1]
    gate = torch.softmax(torch.randn(B, I, device="cuda", generator=gen), -1)
    if gate_kind == "onehot":
        gate = F.one_hot(torch.randint(0, I, (B,), device="cuda", generator=gen), I).float()
    elif gate_kind == "zero":
        gate[:, 3] = 0.0
    want = (0, 3, 5)
    bufs = [padded(c, fill=False) for c in cc]
    dz = [bufs[i][1] if i in want else None for i in range(I)]
    dgate = ops.gate_combine_backward_experts(z, dY, gate, dz)
    ref_dgate = ops.gate_combine_backward(z, dY)
    assert torch.equal(dgate, ref_dgate)
    again = [padded(c, fill=False) for c in cc]
    dgate2 = ops.gate_combine_backward_experts(z, dY, gate, [again[i][1] if i in want else None for i in range(I)])
    assert torch.equal(dgate, dgate2)
    for i, c in enumerate(cc):
        full = bufs[i][0]
        if i not in want:
            assert torch.isnan(full).all(), i
            continue
        assert torch.isnan(full[:, :, c:]).all(), i                        # ld padding untouched
        got = full[:, :, :c]
        assert not torch.isnan(got).any(), i
        assert torch.equal(got, again[i][0][:, :, :c]), i
        ref = gate[:, i, None, None].double() * dY[:, :, :c].double()
        assert bool(((got.double() - ref).abs() <= 1e-6 * ref.abs()).all()), i


# ------------------------------------------------------------------------------------------------ 2. router dx
@pytest.mark.gpu
@pytest.mark.parametrize("prec_name", ["fp32", "bf16"])
@pytest.mark.parametrize("T", [64, 63])
@pytest.mark.parametrize("B", [2, 256])
def test_router_backward_dx_matches_fp64_autograd(prec_name, T, B):
    """mrnb_router_backward_dx for L = <dgate, gate> against fp64 autograd of O.dm_router -> O.gate_scores -> softmax
    (the fp64 autograd runs on the device).  dx: fp32 within 2e-4 of its maximum (the input-gradient budget of
    test_dm_router_module_backward_matches_fp64_autograd), bf16 within 3e-2 (test_dm_router_tensor_core_engine's).
    Parameter gradients: the budgets of test_router_training_backward_matches_fp64_autograd (5e-4 / 5e-2) and, in fp32,
    within 1e-4 of mrnb_router_backward's on the same scale: the kernels are the same, but the bias column sums add
    their split partials with atomics, so two runs of either entry differ in the last bits (measured on a B200: up to
    1.2e-5 of the tensor's maximum for proj_3.bias).  T = 63 in bf16 runs the padded 64-frame engine."""
    from mrn_b200 import ops
    from mrn_b200 import _lib as L
    I, seed = 3, 90 + T + B
    prec = L.PREC_BF16 if prec_name == "bf16" else L.PREC_FP32
    sd = {k: synth.synth_tensor(seed, k, s) for k, s in synth.router_shapes(I, T=T).items()}
    x = synth.randn(seed, "router_x", (B, I, T, 256))
    dg = synth.randn(seed, "dgate", (B, I)) * 0.3
    sdd = {k: v.cuda().double().requires_grad_(True) for k, v in sd.items()}
    x64 = x.cuda().double().requires_grad_(True)
    gate_ref = torch.softmax(O.gate_scores(sdd, O.dm_router(sdd, x64)), -1)
    (gate_ref * dg.cuda().double()).sum().backward()
    n, off = ops.router_param_offsets(I, T)
    arena = torch.zeros(n, dtype=torch.float32)
    for k, name in enumerate(ops.ROUTER_PARAM_NAMES):
        arena[off[k]:off[k] + sd[name].numel()] = sd[name].reshape(-1)
    arena = arena.cuda()
    ws = ops.RouterWorkspace()
    _, _, gate, _ = ops.router_forward(arena, x.cuda(), ws, with_backward=True, prec=prec)
    grads = torch.full_like(arena, float("nan"))
    dx = torch.full((B, I, T, 256), float("nan"), device="cuda")
    ops.router_backward(arena, x.cuda(), gate, dg.cuda(), None, grads, ws, prec=prec, dx=dx)
    plain = torch.full_like(arena, float("nan"))
    ops.router_backward(arena, x.cuda(), gate, dg.cuda(), None, plain, ws, prec=prec)
    assert torch.isfinite(dx).all() and torch.isfinite(grads).all()
    fp32 = prec_name == "fp32"
    assert rel_err(dx.cpu().numpy(), x64.grad.cpu().numpy()) < (2e-4 if fp32 else 3e-2)
    gmax = max(float(v.grad.abs().max()) for v in sdd.values())
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        got = grads[off[k]:off[k] + sd[pname].numel()]
        ref = sdd[pname].grad.reshape(-1)
        scale = max(float(ref.abs().max()), 1e-3 * gmax)
        assert float((got.double() - ref).abs().max()) / scale < (5e-4 if fp32 else 5e-2), pname
        if fp32:
            base = plain[off[k]:off[k] + sd[pname].numel()]
            assert float((got - base).abs().max()) / scale < 1e-4, pname


# ------------------------------------------------------------------------------------------------ 3. training packs
def _pack(arch, esd, prec):
    from mrn_b200 import ops
    return (ops.CrnnTrainPack if arch == "crnn" else ops.SvtrTrainPack)(esd, "cuda", prec)


def _fwd(arch, tp, x, train, features=True):
    from mrn_b200 import ops
    if arch == "crnn":
        return ops.crnn_train_forward(tp, x, bn_batch_stats=train, update_running=False, want_features=features)
    return ops.svtr_train_forward(tp, x, bn_batch_stats=train, update_running=False, want_features=features)


def _bwd(arch, tp, x, dl, train, dfeat):
    """The backward consumes some of the activations it reads (CRNN: the gate pre-activations become their gradients in
    place), so each backward follows its own forward."""
    from mrn_b200 import ops
    _fwd(arch, tp, x, train, features=False)
    if arch == "crnn":
        ops.crnn_train_backward(tp, dl, x.shape[0], bn_batch_stats=train, dfeatures=dfeat)
    else:
        ops.svtr_train_backward(tp, x, dl, bn_batch_stats=train, dfeatures=dfeat)
    return {k: v.detach().clone() for k, v in tp.state(tp.grads).items()}


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_train_pack_features_match_grouped_forward_and_oracle(arch):
    """Eval mode, fp32: the training pack's feature output equals the grouped forward's features and the oracle's
    within 1e-5, and its logits are unchanged by asking for it."""
    from mrn_b200 import ops
    from mrn_b200 import _lib as L
    cc, B, seed = (37,), 3, 21
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    x = synth.synth_batch(B, cc, seed)[0].cuda()
    esd = {k[len("model.0."):]: v for k, v in sd.items() if k.startswith("model.0.")}
    tp = _pack(arch, esd, L.PREC_FP32)
    logits, feats = _fwd(arch, tp, x, False)
    plain = _fwd(arch, tp, x, False, features=False)
    assert torch.equal(logits, plain)
    net = synth.build_net(cc, sd, arch=arch)
    net.eval()
    grouped = net.extract_vector(x).view(B, -1, 1, 256)[:, :, 0]
    assert rel_err(feats.cpu().numpy(), grouped.cpu().numpy()) < 1e-5
    with torch.no_grad():
        ref, _ = O.expert_forward({k: v.double() for k, v in sd.items()}, 0, x.cpu().double(), "eval")
    assert rel_err(feats.cpu().numpy(), ref.numpy()) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("prec_name", ["fp32", "bf16"])
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
@pytest.mark.parametrize("B", [5, 41])
def test_train_pack_feature_gradient_matches_fp64(arch, prec_name, B):
    """Batch-statistics BatchNorm.  Random dlogits and dfeatures give every gradient of <dlogits, z> + <dfeatures, f>
    within the budgets of test_stage0_step_matches_fp64_oracle_at_scale (fp32: max |d| against max(max |ref|, 1e-4 |g|),
    1e-3 except the CRNN's VGG tensors; bf16: relative Frobenius with the floor 2e-3 |g|, the VGG tensors with a cosine
    above 0.97).  The CRNN's VGG tensors take the 5e-2 fp32 budget at both batch sizes: their largest elements hinge on
    ReLU / max-pool decisions (see _fp32_max_budget), and with these random upstream gradients B = 41 measured 1.2e-2
    on a B200.  dfeatures = 0 gives the gradients of dfeatures = NULL within the same budgets: the two runs differ only
    in the order of the backward's atomic accumulations (and, through the forward's BatchNorm statistics, in the same
    ReLU / max-pool ties)."""
    from mrn_b200 import _lib as L
    from test_gpu_stage0_scale import Case, _fp32_max_budget
    from test_gpu_stage0 import _abs_scale_only
    cc, seed = (53,), 300 + B
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    x = synth.synth_batch(B, cc, seed)[0].cuda()
    esd = {k[len("model.0."):]: v for k, v in sd.items() if k.startswith("model.0.")}
    tp = _pack(arch, esd, L.PREC_FP32 if prec_name == "fp32" else L.PREC_BF16)
    T = _fwd(arch, tp, x, True)[0].shape[1]
    dl = synth.randn(seed, "dlogits", (B, T, cc[0]), 1e-2)
    df = synth.randn(seed, "dfeatures", (B, T, 256), 1e-2)
    case = Case(arch, max(B, 5), cc[0], True, False, "synth")

    def compare(got, ref, what):
        tn = math.sqrt(sum(float((g ** 2).sum()) for g in ref.values()))
        bad = []
        for k, rg in ref.items():
            gg = got[k].double().cpu()
            if not bool(torch.isfinite(gg).all()):
                bad.append(f"{what} {k}: not finite")
                continue
            vgg = arch == "crnn" and "ConvNet" in k
            if prec_name == "fp32":
                scale = tn if _abs_scale_only(k, True) else max(float(rg.abs().max()), 1e-4 * tn)
                e, budget = float((gg - rg).abs().max()) / scale, (5e-2 if vgg else _fp32_max_budget(case, k))
            else:
                e = float((gg - rg).norm()) / max(float(rg.norm()), 2e-3 * tn)
                budget = 0.25 if vgg else (3e-2 if arch == "crnn" else 5e-2)
                if vgg:
                    cos = float((gg * rg).sum() / (gg.norm() * rg.norm() + 1e-30))
                    if not cos > 0.97:
                        bad.append(f"{what} {k}: cosine {cos:.4f}")
            if not e < budget:
                bad.append(f"{what} {k}: {e:.3e} (budget {budget:g})")
        return bad

    g_none = _bwd(arch, tp, x, dl.cuda(), True, None)
    g_zero = _bwd(arch, tp, x, dl.cuda(), True, torch.zeros(B, T, 256, device="cuda"))
    bad = compare(g_zero, {k: v.double().cpu() for k, v in g_none.items()}, "dfeatures=0 vs NULL:")
    got = _bwd(arch, tp, x, dl.cuda(), True, df.cuda().contiguous())
    keys = O.expert_param_keys(sd, 0)
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in sd.items()}
    for k in keys:
        sd64[k].requires_grad_(True)
    f, z = O.expert_forward(sd64, 0, x.cpu().double(), "batch")
    gr = torch.autograd.grad((z * dl.double()).sum() + (f * df.double()).sum(), [sd64[k] for k in keys], allow_unused=True)
    ref = {k[len("model.0."):]: (g if g is not None else torch.zeros_like(sd64[k])) for k, g in zip(keys, gr)}
    assert set(got) == set(ref)
    bad += compare(got, ref, "vs fp64:")
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------------------------------------ 4. reference loop
@pytest.mark.gpu
@pytest.mark.parametrize("which", ["all", "newest"])
@pytest.mark.parametrize("mode", ["eval", "train"])
@pytest.mark.parametrize("I", [2, 3])
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_joint_stage1_loop_matches_fp64_oracle(arch, I, mode, which, monkeypatch):
    """15 * CTC + CE on the gate, loss.backward(), fp32, B = 4: every router .grad within 1e-3 of its scale, every
    trainable expert .grad within the stage-0 fp32 budgets of its scale (max(max |ref|, 1e-4 |g|)), the frozen experts'
    .grad None.  train: BatchNorm batch statistics (and, SVTR, injected DropPath for every expert): each trainable
    expert's running statistics are 0.9 old + 0.1 the batch statistic, updated once (num_batches_tracked == 1)."""
    import mrn_b200.modules.model as M
    from mrn_b200.modules.model import _expert_bns
    from test_gpu_stage0_scale import Case, _fp32_max_budget
    from test_gpu_stage0 import _abs_scale_only
    cc = (37, 61, 96)[:I]
    B, seed = 4, 40 + I
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    train = mode == "train"
    drop = synth.synth_drop_scales(I, B, O.svtr_drop_path_rates(), seed) if (train and arch == "svtr") else None
    trainable = tuple(range(I)) if which == "all" else (I - 1,)
    net = synth.build_net(cc, sd, arch=arch, drop_path=True, autograd=True, autograd_experts=True)
    net.train(train)
    _set_trainable(net, trainable)
    if drop is not None:
        monkeypatch.setattr(M, "sample_drop_scales", lambda n_, b_, rates, dev, generator=None: drop.to(dev).clone())
    old_bn = {e: [(bn.running_mean.clone().cpu(), bn.running_var.clone().cpu()) for bn in _expert_bns(net.model[e], arch)]
              for e in trainable}
    loss = _stage1_loop(net, img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda())
    stats = {}
    ref = _joint_oracle(sd, I, img, tgt, lens, dom, trainable, "batch" if train else "eval", drop, stats)
    assert abs(float(loss) - ref["loss"]) / abs(ref["loss"]) < 1e-4
    named = dict(net.named_parameters())
    tn = math.sqrt(sum(float((g ** 2).sum()) for g in ref["grads"].values()))
    bad = []
    for k, rg in ref["grads"].items():
        p = named[k]
        if p.grad is None:
            bad.append(f"{k}: no grad")
            continue
        gg = p.grad.detach().double().cpu()
        if k.startswith(ROUTER_PREFIXES):
            e, budget = float((gg - rg).abs().max()) / max(float(rg.abs().max()), 1e-4 * tn), 1e-3
        else:
            sub = k.split(".", 2)[2]
            scale = tn if _abs_scale_only(sub, train) else max(float(rg.abs().max()), 1e-4 * tn)
            e, budget = float((gg - rg).abs().max()) / scale, _fp32_max_budget(Case(arch, B, 0, train, False, "synth"), sub)
        if not e < budget:
            bad.append(f"{k}: {e:.3e} (budget {budget:g})")
    assert not bad, "\n".join(bad)
    for e in range(I):
        if e not in trainable:
            assert all(p.grad is None for p in net.model[e].parameters()), e
    if train:
        conv = {e: "model.%d.model.FeatureExtraction.ConvNet." % e for e in trainable}
        for e in trainable:
            prefixes = ("12.", "15.") if arch == "crnn" else ("patch_embed.proj.1.", "patch_embed.proj.4.")
            for bn, (m0, v0), pre in zip(_expert_bns(net.model[e], arch), old_bn[e], prefixes):
                mean, var = stats[conv[e] + pre]
                assert int(bn.num_batches_tracked) == 1
                assert rel_err(bn.running_mean.cpu().numpy(), (0.9 * m0.double() + 0.1 * mean).numpy()) < 1e-4
                assert rel_err(bn.running_var.cpu().numpy(), (0.9 * v0.double() + 0.1 * var).numpy()) < 1e-4


# ------------------------------------------------------------------------------------------------ 5. full size
@pytest.mark.gpu
def test_joint_full_size_newest_expert_matches_fp64_oracle():
    """I = 6, B = 256, the MLT17 class counts, bf16, batch statistics: the newest expert trainable.  Its gradients and
    the router's against the fp64 oracle (frozen experts under no_grad): relative Frobenius within 5e-2 with the floor
    2e-3 |g| (the bf16 SVTR budget of test_stage0_step_matches_fp64_oracle_at_scale), the loss within 2e-2."""
    import gc
    cc, B, seed = synth.MLT17_CLASS_COUNTS, 256, 5
    I = len(cc)
    sd = synth.ctor_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    net = synth.build_net(cc, sd, precision="bf16", autograd=True, autograd_experts=True)
    net.train()
    _set_trainable(net, (I - 1,))
    loss = _stage1_loop(net, img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda())
    torch.cuda.synchronize()
    got = {k: p.grad.detach().double().cpu() for k, p in net.named_parameters() if p.grad is not None}
    del net
    gc.collect()
    ref = _joint_oracle(sd, I, img, tgt, lens, dom, (I - 1,), "batch")
    assert abs(float(loss) - ref["loss"]) / abs(ref["loss"]) < 2e-2
    assert set(got) == set(ref["grads"])
    tn = math.sqrt(sum(float((g ** 2).sum()) for g in ref["grads"].values()))
    bad = []
    for k, rg in ref["grads"].items():
        e = float((got[k] - rg).norm()) / max(float(rg.norm()), 2e-3 * tn)
        if not e < 5e-2:
            bad.append(f"{k}: {e:.3e}")
    assert not bad, "\n".join(bad)


@pytest.mark.gpu
def test_joint_full_size_all_experts_train():
    """I = 6, B = 256, MLT17, bf16, every expert trainable: finite gradients on every parameter the forward reads, and
    the loss falls over three torch.optim.Adam steps on a fixed batch."""
    cc, B, seed = synth.MLT17_CLASS_COUNTS, 256, 6
    sd = synth.ctor_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    x, t, l, d = img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda()
    net = synth.build_net(cc, sd, precision="bf16", autograd=True, autograd_experts=True)
    net.train()
    opt = torch.optim.Adam(net.parameters(), lr=1e-4)
    losses = []
    for step in range(4):
        opt.zero_grad()
        losses.append(float(_stage1_loop(net, x, t, l, d)))
        if step == 0:
            n_grad = 0
            for n, p in net.named_parameters():
                if p.grad is not None:
                    assert torch.isfinite(p.grad).all(), n
                    n_grad += 1
            assert n_grad > 6 * 100
        if step < 3:
            opt.step()
    assert losses[3] < losses[0], losses


# ------------------------------------------------------------------------------------------------ 6. inertness, errors
@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_switch_with_every_expert_frozen_is_bitwise_today(arch):
    """opt.autograd_experts with every expert frozen runs today's routed autograd: outputs bitwise equal to the switch
    off, router .grad equal up to the run-to-run spread of the router backward (its bias column sums and split-K weight
    gradients accumulate with atomics, so two runs with the switch off differ in the last bits too): 1e-4 of each
    tensor's scale max(max |g|, 1e-3 max_all |g|)."""
    cc, B, seed = (37, 61, 96), 3, 12
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    res = []
    for on in (False, True):
        net = synth.build_net(cc, sd, arch=arch, autograd=True, autograd_experts=on)
        net.eval()
        _set_trainable(net, ())
        out = net(img.cuda(), True, None, True)
        loss = 15 * _ctc(out["logits"], tgt.cuda(), lens.cuda()) + F.cross_entropy(out["index"], dom.cuda())
        loss.backward()
        res.append((out["logits"].detach(), out["index"].detach(),
                    {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None}))
    (l0, g0, d0), (l1, g1, d1) = res
    assert torch.equal(l0, l1) and torch.equal(g0, g1)
    assert set(d0) == set(d1) and all(k.startswith(ROUTER_PREFIXES) for k in d0)
    gmax = max(float(v.abs().max()) for v in d0.values())
    for k in d0:
        scale = max(float(d0[k].abs().max()), 1e-3 * gmax)
        assert float((d0[k] - d1[k]).abs().max()) / scale < 1e-4, k


@pytest.mark.gpu
def test_switch_without_autograd_builds_no_graph():
    cc = (37, 61)
    sd = synth.synth_state_dict(cc, 3)
    net = synth.build_net(cc, sd, autograd=False, autograd_experts=True)
    net.eval()
    out = net(synth.synth_batch(2, cc, 3)[0].cuda(), True, None, True)
    assert out["logits"].grad_fn is None and out["index"].grad_fn is None


def test_trainable_experts_without_the_switch_are_refused_with_a_hint():
    """No device needed: the check runs before any kernel.  The refusal still says "frozen" and names the switch."""
    net = synth.build_net((5, 9), device=None, autograd=True)
    with pytest.raises(NotImplementedError, match="frozen") as e:
        net(torch.zeros(1, 4, 32, 256), True, None, True)
    assert "autograd_experts" in str(e.value)


def test_switch_without_autograd_takes_no_autograd_path():
    """No device needed: without opt.autograd the switch is not consulted; the routed forward goes to the kernels, which
    need CUDA tensors."""
    net = synth.build_net((5, 9), device=None, autograd=False, autograd_experts=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 4, 32, 256), True, None, True)


@pytest.mark.gpu
def test_joint_double_backward_raises():
    cc = (37, 61)
    sd = synth.synth_state_dict(cc, 4)
    net = synth.build_net(cc, sd, autograd=True, autograd_experts=True)
    net.eval()
    _set_trainable(net, (1,))
    out = net(synth.synth_batch(2, cc, 4)[0].cuda(), True, None, True)
    p = net.model[1].fc.weight
    (gp,) = torch.autograd.grad(out["logits"].square().sum(), p, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable|differentiate twice"):
        gp.sum().backward()
