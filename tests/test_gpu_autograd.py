"""Autograd through MRNNet, Model and DM_Router (opt.autograd / DM_Router(autograd=True)): the reference's own training
loop -- forward, log_softmax + F.ctc_loss, CE on the gate, loss.backward(), clip_grad_norm_, torch.optim.Adam
(il_modules/mrn.py:338-367 and :236-267) -- on the fused kernels, against the reference goldens, the fused learner
step and fp64; the combine backward kernel against fp64; the switch left off changes nothing."""
import argparse

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import mrn_oracle as O
from oracle import synth
from conftest import load_golden, gview, rel_err
from persistent_walk import assert_walk, combine_walk

ROUTER_PREFIXES = ("route.", "channel_route.", "dm_router.0.")


def _opt(arch, precision="fp32", autograd=True):
    feat, seq = ("SVTR", "None") if arch == "svtr" else ("VGG", "BiLSTM")
    return argparse.Namespace(Transformation="None", FeatureExtraction=feat, SequenceModeling=seq, Prediction="CTC",
                              num_fiducial=20, input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256,
                              batch_max_length=25, lr=5e-4, num_iter=10000, grad_clip=5, exp_name="test", precision=precision,
                              drop_path=True, lan_list=list("abcdef"), val_interval=5000, start_task=0, optimizer="adam",
                              schedule="super", autograd=autograd)


def _net(arch, cc, sd, precision="fp32", autograd=True):
    from mrn_b200.modules.model import MRNNet
    opt = _opt(arch, precision, autograd)
    net = MRNNet(opt)
    for c in cc:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    res = net.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    return net.cuda()


def _freeze_experts(net):
    for p in net.model.parameters():
        p.requires_grad = False


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


def _router_grads(net):
    return {n: p.grad for n, p in net.named_parameters() if n.startswith(ROUTER_PREFIXES)}


# ------------------------------------------------------------------------------------------------ 1. stage 1 vs goldens
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["svtr_mrn_i3_b3", "svtr_mrn_i2_b4", "crnn_mrn_i2_b4", "crnn_mrn_i3_b2"])
def test_stage1_torch_loop_matches_reference_golden(name):
    """Router .grad within 1e-3 of each parameter's scale (the rule of test_stage1_step_matches_reference_golden), the
    total norm of clip_grad_norm_ within 5e-4 and one torch.optim.Adam step against adam1.*."""
    from mrn_b200 import ops
    g = load_golden(name)
    arch = "crnn" if name.startswith("crnn") else "svtr"
    T = 63 if arch == "crnn" else 64
    cc, B, seed = tuple(int(c) for c in g["class_counts"]), int(g["B"]), int(g["seed"])
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    net = _net(arch, cc, sd)
    net.eval()                                          # the goldens were made with eval-mode, frozen experts
    _freeze_experts(net)
    _stage1_loop(net, img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda())
    grads = _router_grads(net)
    assert set(grads) == set(ops.ROUTER_PARAM_NAMES) and all(v is not None for v in grads.values())
    tn = float(g["grad_total_norm"])
    for pname in ops.ROUTER_PARAM_NAMES:
        ref = g["grad." + pname].reshape(-1)
        scale = max(float(np.abs(ref).max()), 1e-4 * tn)
        assert np.abs(gview(grads[pname].reshape(-1), g) - ref).max() / scale < 1e-3, pname
    params = net.router_parameters()
    norm = float(torch.nn.utils.clip_grad_norm_(params, 5))
    assert abs(norm - tn) / tn < 5e-4
    torch.optim.Adam(params, lr=5e-4).step()
    shapes = synth.router_shapes(len(cc), T=T)
    for pname, p in zip(ops.ROUTER_PARAM_NAMES, params):
        assert tuple(p.shape) == tuple(shapes[pname])
        if pname == "route.bias":
            continue
        d = np.abs(gview(p.detach().reshape(-1), g) - g["adam1." + pname].reshape(-1))
        assert d.max() <= 5e-4 * 1.01 and (d > 2e-5).mean() < 1e-2, pname


# ------------------------------------------------------------------------------------------------ 2. == fused step
@pytest.mark.gpu
@pytest.mark.parametrize("arch,precision,mode", [("svtr", "fp32", "eval"), ("svtr", "bf16", "eval"),
                                                 ("svtr", "fp32", "train"), ("crnn", "fp32", "eval")])
def test_autograd_gradients_match_fused_stage1_step(arch, precision, mode, monkeypatch):
    """Same batch, same weights: the .grad of the torch loop against MRN.train_step_stage1's gradient arena.

    fp32: 1e-4 of each parameter's scale.  The two paths differ only in how d loss / d gate is formed (F.ctc_loss +
    dense combine backward vs the fused lattice contraction), both in fp32, so they agree to fp32 round-off.
    bf16: the experts and the router run the same bf16 kernels in both paths; the router backward rounds its
    gate-derived operands to bf16, where an fp32-level difference in dL/dgate moves a value across a rounding boundary
    at most by one bf16 ulp (2^-8 relative).  Such flips are rare and of both signs, so the budget is one ulp of the
    parameter's scale, 2^-8 ~ 4e-3, taken as 1e-2.
    train: experts in .train() (BatchNorm batch statistics) with the same injected DropPath scales on both paths."""
    import mrn_b200.modules.model as M
    from mrn_b200 import ops
    from mrn_b200.il_modules.mrn import MRN, RankLocal, FusedAdam
    cc, B, seed = (37, 61, 96), 4, 7
    sd = synth.ctor_state_dict(cc, seed) if precision == "bf16" else synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    drop = synth.synth_drop_scales(len(cc), B, O.svtr_drop_path_rates(), seed).cuda() if mode == "train" else None
    x, t, l, d = img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda()

    fused = _net(arch, cc, sd, precision, autograd=False)
    fused.train(mode == "train")
    learner = MRN(fused.opt)
    learner.model = RankLocal(fused)
    learner.optimizer = FusedAdam(fused, 5e-4, 20000, grad_clip=5, schedule="const")
    learner.train_step_stage1(x, t, l, d, drop_scales=drop)
    n, off = ops.router_param_offsets(len(cc), 63 if arch == "crnn" else 64)
    arena = fused.router_grad_arena()

    net = _net(arch, cc, sd, precision)
    net.train(mode == "train")
    _freeze_experts(net)
    if drop is not None:
        monkeypatch.setattr(M, "sample_drop_scales", lambda n_, b_, rates, dev, generator=None: drop)
    _stage1_loop(net, x, t, l, d)
    grads = _router_grads(net)
    tn = float(arena.norm())
    tol = 1e-4 if precision == "fp32" else 1e-2
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        got = grads[pname].reshape(-1)
        ref = arena[off[k]:off[k] + got.numel()]
        scale = max(float(ref.abs().max()), 1e-4 * tn)
        err = float((got - ref).abs().max()) / scale
        assert err < tol, (pname, err)


# ------------------------------------------------------------------------------------------------ 3. stage 0 vs goldens
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["svtr_stage0_i1_b2_eval", "crnn_stage0_i1_b2_eval", "svtr_stage0_i2_b3",
                                  "crnn_stage0_i2_b3"])
def test_stage0_torch_loop_matches_reference_golden(name, monkeypatch):
    """net(image, cross=False) -> mean CTC (zero_infinity) -> backward: every gradient of the newest expert within 1e-3
    of its own maximum (conv biases in front of a batch-statistics BatchNorm are analytically zero: compared on the
    scale of the whole gradient), BatchNorm running statistics as the reference's."""
    import mrn_b200.modules.model as M
    from test_oracle_pinning import pview, stage0_case
    g, cc, B, sd, img, tgt, lens, bn_train, drop = stage0_case(name)
    arch = str(g["arch"]) if "arch" in g else "svtr"
    net = _net(arch, cc, sd)
    net.train(bn_train)
    if drop is not None:
        monkeypatch.setattr(M, "sample_drop_scales", lambda n_, b_, rates, dev, generator=None: drop.unsqueeze(0).to(dev))
    out = net(img.cuda(), cross=False)
    loss = _ctc(out["logits"], tgt.cuda(), lens.cuda())
    assert abs(float(loss) - float(g["loss"])) / abs(float(g["loss"])) < 1e-4
    loss.backward()
    i = len(cc) - 1
    expert = net.model[i]
    tn = float(g["grad_total_norm"])
    checked = set()
    for key, p in expert.named_parameters():
        gk = "grad.model.%d.%s" % (i, key)
        if gk not in g:
            continue
        ref = g[gk]
        scale = max(float(np.abs(ref).max()), 1e-4 * tn)
        if bn_train and key.endswith(("patch_embed.proj.0.bias", "patch_embed.proj.3.bias")):
            scale = tn
        assert p.grad is not None, key
        assert np.abs(pview(p.grad.contiguous(), g) - ref).max() / scale < 1e-3, key
        checked.add(gk)
    assert checked == {k for k in g if k.startswith("grad.model.%d." % i)}
    # frozen / older experts and the router get nothing from cross=False
    assert all(p.grad is None for n, p in net.named_parameters() if not n.startswith("model.%d." % i))
    if bn_train:
        from mrn_b200.modules.model import _expert_bns
        bns = _expert_bns(expert, arch)
        for bn, q in zip(bns, ("bn0", "bn1")):
            assert rel_err(bn.running_mean.cpu().numpy(), g[q + "_running_mean"]) < 1e-4
            assert rel_err(bn.running_var.cpu().numpy(), g[q + "_running_var"]) < 1e-4
            assert int(bn.num_batches_tracked) == 1


# ------------------------------------------------------------------------------------------------ 4. DM_Router alone
@pytest.mark.gpu
@pytest.mark.parametrize("T", [64, 63])
def test_dm_router_module_backward_matches_fp64_autograd(T):
    """DM_Router(autograd=True) vs torch autograd of the fp64 oracle: x.grad within 2e-4 and every parameter's grad
    within 5e-4 of its maximum (the fp32 budgets of test_dm_router_forward_backward; T = 63 runs the padded frames)."""
    from mrn_b200.modules.dm_router import DM_Router
    I, B, seed = 3, 4, 11
    shapes = synth.router_shapes(I, T=T)
    sd = {k: synth.synth_tensor(seed, k, s) for k, s in shapes.items() if k.startswith("dm_router.0.")}
    m = DM_Router(256, 512, T, I, autograd=True)
    m.load_state_dict({k[len("dm_router.0."):]: v for k, v in sd.items()}, strict=True)
    m = m.cuda()
    x = synth.randn(seed, "router_x", (B, I, T, 256))
    dy = synth.randn(seed, "router_dy", (B, I, T, 256))
    xc = x.cuda().requires_grad_(True)
    m(xc).backward(dy.cuda())
    sdd = {k: v.double().requires_grad_(True) for k, v in sd.items()}
    x64 = x.double().requires_grad_(True)
    O.dm_router(sdd, x64).backward(dy.double())
    assert rel_err(xc.grad.cpu().numpy(), x64.grad.numpy()) < 2e-4
    for n, p in m.named_parameters():
        assert rel_err(p.grad.cpu().numpy(), sdd["dm_router.0." + n].grad.numpy()) < 5e-4, n


# ------------------------------------------------------------------------------------------------ 5. combine backward kernel
@pytest.mark.gpu
@pytest.mark.parametrize("gate_kind", ["soft", "onehot", "zero"])
def test_gate_combine_backward_kernel_matches_fp64(gate_kind):
    """mrnb_gate_combine_backward at B = 64 with the MLT17 class counts against torch autograd of the fp64 combine
    (pad with ones) with respect to the gate: the derivative does not depend on the gate, so a one-hot gate and a gate
    with an exact zero give every expert its full gradient.  The ld padding of every row holds NaN (must not be read as
    data), the output is NaN-prefilled, each persistent CTA walks >= 4 rows, two runs are bitwise equal.
    Budget: 1e-5 of sum |dY * pad| per (b, i) (fp32 accumulation over T * C = 330 k terms)."""
    from mrn_b200 import ops
    cc, B, T = synth.MLT17_CLASS_COUNTS, 64, 64
    I, C = len(cc), cc[-1]
    rows, grid = combine_walk(B, T)
    assert_walk(rows, grid, "combine_bwd_tma_kernel")
    gen = torch.Generator(device="cuda").manual_seed(5)

    def padded(c):
        buf = torch.full((B, T, ops.round_up(c, 4)), float("nan"), device="cuda")
        buf[:, :, :c] = torch.randn(B, T, c, device="cuda", generator=gen)
        return buf[:, :, :c]
    z = [padded(c) for c in cc]
    dY = padded(C)
    if gate_kind == "soft":
        gate = torch.softmax(torch.randn(B, I, device="cuda", generator=gen), -1)
    elif gate_kind == "onehot":
        gate = F.one_hot(torch.randint(0, I, (B,), device="cuda", generator=gen), I).float()
    else:
        gate = torch.softmax(torch.randn(B, I, device="cuda", generator=gen), -1)
        gate[:, 2] = 0.0
    out = torch.full((B, I), float("nan"), device="cuda")
    got = ops.gate_combine_backward(z, dY, out=out).clone()
    again = ops.gate_combine_backward(z, dY)
    assert torch.equal(got, again)
    g64 = gate.double().requires_grad_(True)
    pads = [F.pad(zi.double(), (0, C - zi.shape[2]), value=1.0) for zi in z]
    comb = sum(g64[:, i, None, None] * pads[i] for i in range(I))
    (comb * dY.double()).sum().backward()
    ref = g64.grad
    bound = torch.stack([(dY.double() * p).abs().sum((1, 2)) for p in pads], 1)
    assert not torch.isnan(got).any()
    assert float(((got.double() - ref).abs() / bound).max()) < 1e-5


# ------------------------------------------------------------------------------------------------ 6. the switch off is inert
@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_autograd_switch_off_is_inert_and_on_keeps_forward_values(arch):
    """Without opt.autograd no output requires grad (even with parameters that do and grad mode on).  With it, the soft
    and hard routes return bitwise the values of the default forward (same kernels), and cross=False -- which then runs
    the training pack's forward -- returns the default forward's logits within fp32 round-off (1e-5 relative)."""
    cc, B, seed = (37, 61, 96), 3, 111
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    x = synth.synth_batch(B, cc, seed)[0].cuda()
    off = _net(arch, cc, sd, autograd=False)
    on = _net(arch, cc, sd)
    for n in (off, on):
        n.eval()
    _freeze_experts(on)
    res = {}
    for key, kw in (("soft", dict(cross=True, is_train=True)), ("hard", dict(cross=True, is_train=False)),
                    ("last", dict(cross=False, is_train=False))):
        if key == "last":                       # the newest expert is what cross=False differentiates
            for p in on.model[-1].parameters():
                p.requires_grad = True
        a = off(x, **kw)
        assert not a["logits"].requires_grad and (a["index"] is None or not a["index"].requires_grad), key
        b = on(x, **kw)
        res[key] = (a, b)
    for key in ("soft", "hard"):
        a, b = res[key]
        assert torch.equal(a["logits"], b["logits"].detach()) and torch.equal(a["index"], b["index"].detach()), key
    a, b = res["last"]
    assert b["logits"].requires_grad
    assert rel_err(b["logits"].detach().cpu().numpy(), a["logits"].cpu().numpy()) < 1e-5
    assert res["soft"][1]["logits"].requires_grad and res["soft"][1]["index"].requires_grad
    assert not res["hard"][1]["logits"].requires_grad
    with torch.no_grad():
        assert not on(x, True, None, True)["logits"].requires_grad


# ------------------------------------------------------------------------------------------------ 7. errors
def test_routed_autograd_refuses_experts_that_require_grad():
    """No device needed: the check runs before any kernel."""
    from mrn_b200.modules.model import MRNNet
    opt = _opt("svtr")
    net = MRNNet(opt)
    for c in (5, 9):
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    assert net.dm_router[0].autograd is True
    with pytest.raises(NotImplementedError, match="frozen"):
        net(torch.zeros(1, 4, 32, 256), True, None, True)


def test_router_backward_without_domain_needs_dgate():
    """A NULL domain makes dgate_ctc the whole dL/dgate: a NULL dgate_ctc is rejected by the argument checks (before any
    device work)."""
    import ctypes as C
    import os
    from mrn_b200 import _lib as L
    if not os.path.exists(L.LIB_PATH):
        from mrn_b200.build import build
        build()
    lib = L.load()
    fake = C.c_void_p(256)                      # never dereferenced: the checks fail first
    rc = lib.mrnb_router_backward(fake, fake, fake, None, None, 2, 3, 64, 256, 0, fake, None, fake, 1 << 30, None)
    assert rc == -1 and b"dgate_ctc" in lib.mrnb_last_error()


@pytest.mark.gpu
def test_double_backward_raises():
    from mrn_b200.modules.dm_router import DM_Router
    m = DM_Router(256, 512, 64, 2, autograd=True).cuda()
    x = torch.randn(1, 2, 64, 256, device="cuda", requires_grad=True)
    (gx,) = torch.autograd.grad(m(x).square().sum(), x, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable|differentiate twice"):
        gx.sum().backward()
