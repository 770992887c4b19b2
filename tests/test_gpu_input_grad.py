"""Gradients with respect to the input image through the experts (opt.autograd with image.requires_grad_()): what a
differentiable module in front of the recogniser -- a rectification front end, learned augmentation, inversion of the
frozen experts, a saliency map -- needs from Model and MRNNet.

The conv0 input-gradient kernels are checked on their own first, then one expert through Model.forward, MRNNet's soft
route with frozen and trainable experts, the full-size stage-1 configuration, the input-only backward of frozen experts
against the full backward, and that nothing changes while the image does not require grad.  The oracle is fp64 autograd
of oracle.mrn_oracle with the image requiring grad.  The SVTR oracle runs in fp64 on the device (its Local-mixer mask,
built on the host, is moved there); the CRNN oracle keeps its LSTM state on the host and runs there."""
import contextlib
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import mrn_oracle as O
from mrn_b200 import synth
from conftest import rel_err

ROUTER_PREFIXES = ("route.", "channel_route.", "dm_router.0.")


def _ctc(logits, tgt, lens):
    B, T = logits.shape[:2]
    return F.ctc_loss(logits.log_softmax(2).permute(1, 0, 2), tgt, torch.full((B,), T, dtype=torch.long, device=tgt.device),
                      lens.long(), blank=0, reduction="mean", zero_infinity=True)


def _set_trainable(net, trainable):
    for e, m in enumerate(net.model):
        for p in m.parameters():
            p.requires_grad = e in trainable


def _rel_fro(got, ref):
    return float((got.double() - ref.double()).norm() / max(float(ref.double().norm()), 1e-30))


def _cos(got, ref):
    g, r = got.double().flatten(), ref.double().flatten()
    return float((g * r).sum() / (g.norm() * r.norm() + 1e-30))


# ------------------------------------------------------------------------------------------------ the fp64 oracle
@contextlib.contextmanager
def _oracle_env(dev, stats=None):
    """O.local_mask moved to `dev`; with `stats`, each batch-statistics BatchNorm input's (mean, unbiased var) recorded
    by parameter prefix (the values nn.BatchNorm2d folds into its running statistics)."""
    mask, bn = O.local_mask, O._bn

    def recording_bn(x, sd_, p, mode, eps=1e-5):
        if mode != "eval" and stats is not None:
            xd = x.detach().cpu()
            stats[p] = (xd.mean(dim=(0, 2, 3)), xd.var(dim=(0, 2, 3), unbiased=True))
        return bn(x, sd_, p, mode, eps)

    with pytest.MonkeyPatch.context() as m:
        m.setattr(O, "local_mask", lambda *a, **k: mask(*a, **k).to(dev))
        m.setattr(O, "_bn", recording_bn)
        yield


def _expert_sd64(sd, e, dev):
    return {k: v.detach().to(dev, torch.float64) for k, v in sd.items() if k.startswith(f"model.{e}.") and v.is_floating_point()}


def _oracle_dev(sd, e):
    return "cuda" if O.expert_arch(sd, e) == "svtr" else "cpu"


def _expert_oracle(sd, e, img, bn_mode, drop, loss_fn, keys=()):
    """fp64 autograd of loss_fn(feature, predict) (host tensors) through expert e: (loss, d loss / d image, {key: grad},
    feature, predict), all on the host."""
    dev = _oracle_dev(sd, e)
    sd64 = _expert_sd64(sd, e, dev)
    for k in keys:
        sd64[k].requires_grad_(True)
    x = img.detach().to(dev, torch.float64).requires_grad_(True)
    with _oracle_env(dev):
        f, z = O.expert_forward(sd64, e, x, bn_mode, None if drop is None else drop.to(dev, torch.float64))
    fc, zc = f.cpu(), z.cpu()
    loss = loss_fn(fc, zc)
    gr = torch.autograd.grad(loss, [x] + [sd64[k] for k in keys], allow_unused=True)
    grads = {k: (g.cpu() if g is not None else torch.zeros_like(sd64[k]).cpu()) for k, g in zip(keys, gr[1:])}
    return float(loss.detach()), gr[0].cpu(), grads, fc.detach(), zc.detach()


def _routed_oracle(sd, I, img, tgt, lens, dom, trainable, bn_mode="eval", drop=None, stats=None):
    """fp64 autograd of the reference's stage-1 loss (15 * CTC + CE on the gate) over O's soft route, with respect to
    the image, the router and the experts in `trainable`.  One expert's graph at a time: the experts' outputs first
    (no grad), then the loss and its gradients at the features and logits, then each expert's vector-Jacobian product.
    The image gradient is summed in expert order."""
    feats, preds = [], []
    with torch.no_grad():
        for i in range(I):
            dev = _oracle_dev(sd, i)
            with _oracle_env(dev, stats):
                f, z = O.expert_forward(_expert_sd64(sd, i, dev), i, img.to(dev, torch.float64), bn_mode,
                                        None if drop is None else drop[i].to(dev, torch.float64))
            feats.append(f.cpu())
            preds.append(z.cpu())
    sdr = {k: sd[k].detach().double().requires_grad_(True) for k in O.ROUTER_KEYS}
    fx = torch.stack(feats, 1).requires_grad_(True)
    px = [z.requires_grad_(True) for z in preds]
    gate = torch.softmax(O.gate_scores(sdr, O.dm_router(sdr, fx)), -1)
    loss = 15 * _ctc(O.combine_soft(px, gate), tgt, lens) + F.cross_entropy(gate, dom)
    g = torch.autograd.grad(loss, [sdr[k] for k in O.ROUTER_KEYS] + [fx] + px)
    grads = dict(zip(O.ROUTER_KEYS, g[:len(O.ROUTER_KEYS)]))
    gf, gz = g[len(O.ROUTER_KEYS)], g[len(O.ROUTER_KEYS) + 1:]
    dimage = None
    for i in range(I):
        keys = O.expert_param_keys(sd, i) if i in trainable else ()
        _, gx, ge, _, _ = _expert_oracle(sd, i, img, bn_mode, None if drop is None else drop[i],
                                         lambda f, z: (f * gf[:, i]).sum() + (z * gz[i]).sum(), keys)
        grads.update(ge)
        dimage = gx if dimage is None else dimage + gx
    return dict(loss=float(loss), image=dimage, grads=grads)


def _check_image_grad(got, ref, arch, prec, B, what=""):
    """fp32: 1e-3 relative max and relative Frobenius error.  The CRNN is widened, as _fp32_max_budget widens its VGG
    tensors, to 0.1 relative max and 2e-2 relative Frobenius: measured on a B200, up to 4.95e-2 max (B = 256, train) and
    8.1e-3 Frobenius (B = 4, train).  The image gradient inherits this from the VGG backward upstream of conv0: in the
    same B = 4 runs the conv0 weight gradient of that backward is off by 1.6e-3 (eval) / 8.0e-3 (train) relative
    Frobenius, ConvNet.3 and .6 by ~4e-4 / ~5e-3, everything from ConvNet.8 on by ~1e-5, while the input-gradient kernel
    alone matches fp64 to 1e-5 (test_conv0_dimage_kernel_matches_fp64).  bf16: the VGG / SVTR budgets of
    test_stage0_step_matches_fp64_oracle_at_scale (SVTR 5e-2 relative Frobenius; CRNN 0.25 and a cosine above 0.97)."""
    assert bool(torch.isfinite(got).all()), what + " image grad not finite"
    got, ref = got.double().cpu(), ref.double().cpu()
    if prec == "fp32":
        emax, efro = rel_err(got.numpy(), ref.numpy()), _rel_fro(got, ref)
        bmax, bfro = (0.1, 2e-2) if arch == "crnn" else (1e-3, 1e-3)
        assert emax < bmax and efro < bfro, f"{what} image grad: max {emax:.3e} (budget {bmax:g}), fro {efro:.3e}"
    elif arch == "svtr":
        efro = _rel_fro(got, ref)
        assert efro < 5e-2, f"{what} image grad: fro {efro:.3e}"
    else:
        efro, cos = _rel_fro(got, ref), _cos(got, ref)
        assert efro < 0.25 and cos > 0.97, f"{what} image grad: fro {efro:.3e}, cosine {cos:.4f}"


# ------------------------------------------------------------------------------------------------ 1. kernels
@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 5, 41, 256])
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_conv0_dimage_kernel_matches_fp64(arch, B):
    """mrnb_{svtr,crnn}_conv0_dimage against torch.nn.grad.conv2d_input in fp64: relative max error within 1e-5, a
    NaN-filled output fully overwritten, two runs bitwise equal."""
    from mrn_b200 import ops
    seed = 70 + B
    if arch == "svtr":
        d = synth.randn(seed, "d", (B, 16, 128, 32)).cuda()
        w = synth.randn(seed, "w", (32, 4, 3, 3), 0.2).cuda()
        w_oihw, stride = w, 2
    else:
        d = synth.randn(seed, "d", (B, 32, 256, 64)).cuda()
        w = synth.randn(seed, "w", (64, 3, 3, 4), 0.2).cuda()
        w_oihw, stride = w.permute(0, 3, 1, 2), 1
    out = torch.full((B, 4, 32, 256), float("nan"), device="cuda")
    ops.conv0_dimage(arch, d, w, out=out)
    again = torch.full_like(out, float("nan"))
    ops.conv0_dimage(arch, d, w, out=again)
    assert not torch.isnan(out).any()
    assert torch.equal(out, again)
    ref = torch.nn.grad.conv2d_input((B, 4, 32, 256), w_oihw.double(), d.permute(0, 3, 1, 2).double(), stride=stride,
                                     padding=1)
    assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < 1e-5


# ------------------------------------------------------------------------------------------------ 2. one expert
EXPERT_CASES = [(arch, B, mode) for arch in ("svtr", "crnn") for B in (5, 41) for mode in ("eval", "train")]
EXPERT_CASES += [("svtr", 256, "train"), ("crnn", 256, "train")]
_EXPERT_ORACLE = {}


def _expert_inputs(arch, B, mode):
    cc = (5153,) if B == 256 else (53,)
    seed = 500 + B + (arch == "crnn")
    sd = (synth.ctor_state_dict if B == 256 else synth.synth_state_dict)(cc, seed, arch=arch)
    img, tgt, lens, _ = synth.synth_batch(B, cc, seed)
    drop = synth.synth_drop_scales(1, B, O.svtr_drop_path_rates(), seed) if (mode == "train" and arch == "svtr") else None
    T = 64 if arch == "svtr" else 63
    R = synth.randn(seed, "feature_functional", (B, T, 256), 1e-2 / B)
    return cc, sd, img, tgt, lens, drop, R


@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("arch,B,mode", EXPERT_CASES, ids=[f"{a}-B{b}-{m}" for a, b, m in EXPERT_CASES])
def test_model_forward_image_grad_matches_fp64(arch, B, mode, prec, monkeypatch):
    """Model.forward under opt.autograd with image.requires_grad, loss = CTC(predict) + <R, feature> for a fixed random
    R: image.grad against the oracle (_check_image_grad); "feature" against the oracle (fp32 eval: 1e-5 and the grouped
    forward's within 1e-5, as test_train_pack_features_match_grouped_forward_and_oracle; otherwise 1e-3 fp32 / 5e-2 bf16
    relative max); every parameter .grad against the same call without image grad, within the budgets the
    dfeatures = 0 / NULL comparison of test_train_pack_feature_gradient_matches_fp64 uses for the backward's
    run-to-run spread (1e-3 of max(|ref|, 1e-3 |g|), the CRNN's VGG tensors 5e-2; bf16 1e-2 and 0.25).
    train: BatchNorm batch statistics and, SVTR, injected DropPath."""
    import mrn_b200.modules.model as M
    cc, sd, img, tgt, lens, drop, R = _expert_inputs(arch, B, mode)
    train = mode == "train"
    if drop is not None:
        monkeypatch.setattr(M, "sample_drop_scales", lambda n_, b_, rates, dev, generator=None: drop.to(dev).clone())
    net = synth.build_net(cc, sd, arch=arch, precision=prec, drop_path=True, autograd=True)
    model = net.model[0]
    model.train(train)
    x, t, l, Rc = img.cuda(), tgt.cuda(), lens.cuda(), R.cuda()

    def run(image_grad):
        model.zero_grad(set_to_none=True)
        xi = x.clone().requires_grad_(image_grad)
        out = model(xi)
        loss = _ctc(out["predict"], t, l) + (out["feature"] * Rc).sum()
        loss.backward()
        torch.cuda.synchronize()
        return (xi.grad, out["feature"].detach(), out["predict"].detach(), float(loss.detach()),
                {n: p.grad.detach().clone() for n, p in model.named_parameters() if p.grad is not None})

    gx, feat, pred, loss, grads = run(True)
    _, _, pred0, _, grads0 = run(False)
    assert torch.equal(pred, pred0)
    key = (arch, B, mode)
    if key not in _EXPERT_ORACLE:
        _EXPERT_ORACLE.clear()
        bn = "batch" if train else "eval"
        _EXPERT_ORACLE[key] = _expert_oracle(sd, 0, img, bn, None if drop is None else drop[0],
                                             lambda f, z: _ctc(z, tgt, lens) + (f * R.double()).sum())
    ref_loss, ref_img, _, ref_f, _ = _EXPERT_ORACLE[key]
    fp32 = prec == "fp32"
    assert abs(loss - ref_loss) / abs(ref_loss) < (1e-4 if fp32 else 2e-2)
    _check_image_grad(gx, ref_img, arch, prec, B)
    if fp32 and not train:
        assert rel_err(feat.cpu().numpy(), ref_f.numpy()) < 1e-5
        net.eval()
        grouped = net.extract_vector(x).view(B, -1, 1, 256)[:, :, 0]
        assert rel_err(feat.cpu().numpy(), grouped.cpu().numpy()) < 1e-5
    else:
        assert rel_err(feat.cpu().numpy(), ref_f.numpy()) < (1e-3 if fp32 else 5e-2)
    assert set(grads) == set(grads0)
    tn = math.sqrt(sum(float((g.double() ** 2).sum()) for g in grads0.values()))
    bad = []
    for k, g0 in grads0.items():
        vgg = arch == "crnn" and "ConvNet" in k
        e = float((grads[k].double() - g0.double()).norm()) / max(float(g0.double().norm()), 1e-3 * tn)
        budget = (5e-2 if vgg else 1e-3) if fp32 else (0.25 if vgg else 1e-2)
        if not e < budget:
            bad.append(f"{k}: {e:.3e} (budget {budget:g})")
    assert not bad, "\n".join(bad)


# ------------------------------------------------------------------------------------------------ 3. soft route
def _record_packs(monkeypatch):
    """Wraps modules.model._train_pack_run: [(expert index in its MRNNet, param_grads)] of every pack built."""
    import mrn_b200.modules.model as M
    calls, orig = [], M._train_pack_run

    def wrapped(expert, x, opt, net=None, **kw):
        idx = next((e for e, m in enumerate(net.model) if m is expert), None) if net is not None else None
        calls.append((idx, kw.get("param_grads", True)))
        return orig(expert, x, opt, net=net, **kw)
    monkeypatch.setattr(M, "_train_pack_run", wrapped)
    return calls


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["frozen", "newest"])
@pytest.mark.parametrize("mode", ["eval", "train"])
@pytest.mark.parametrize("I", [2, 3])
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_routed_image_grad_matches_fp64_oracle(arch, I, mode, which, monkeypatch):
    """15 * CTC + CE on the gate with image.requires_grad, fp32, B = 4: image.grad against the oracle
    (_check_image_grad); router .grad within 1e-3 of its scale (the CRNN's route.bias 5e-3, see below) and the trainable
    expert's within the stage-0 fp32 budgets, as test_joint_stage1_loop_matches_fp64_oracle; the frozen experts' .grad
    None and their packs built without
    a gradient arena.  train: BatchNorm batch statistics (SVTR: injected DropPath); every expert's running statistics
    0.9 old + 0.1 the batch statistic, updated once."""
    import mrn_b200.modules.model as M
    from mrn_b200.modules.model import _expert_bns
    from test_gpu_stage0_scale import Case, _fp32_max_budget
    from test_gpu_stage0 import _abs_scale_only
    cc = (37, 61, 96)[:I]
    B, seed = 4, 40 + I                     # the cases of test_joint_stage1_loop_matches_fp64_oracle
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    train = mode == "train"
    drop = synth.synth_drop_scales(I, B, O.svtr_drop_path_rates(), seed) if (train and arch == "svtr") else None
    trainable = () if which == "frozen" else (I - 1,)
    net = synth.build_net(cc, sd, arch=arch, drop_path=True, autograd=True, autograd_experts=True)
    net.train(train)
    _set_trainable(net, trainable)
    if drop is not None:
        monkeypatch.setattr(M, "sample_drop_scales", lambda n_, b_, rates, dev, generator=None: drop.to(dev).clone())
    calls = _record_packs(monkeypatch)
    old_bn = [[(bn.running_mean.clone().cpu(), bn.running_var.clone().cpu()) for bn in _expert_bns(m, arch)]
              for m in net.model]
    x = img.cuda().requires_grad_(True)
    out = net(x, True, None, True)
    loss = 15 * _ctc(out["logits"], tgt.cuda(), lens.cuda()) + F.cross_entropy(out["index"], dom.cuda())
    loss.backward()
    assert sorted(calls) == [(e, e in trainable) for e in range(I)]
    stats = {}
    ref = _routed_oracle(sd, I, img, tgt, lens, dom, trainable, "batch" if train else "eval", drop, stats)
    assert abs(float(loss) - ref["loss"]) / abs(ref["loss"]) < 1e-4
    _check_image_grad(x.grad, ref["image"], arch, "fp32", B)
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
            # route.bias is one scalar summed over the batch and the frames with heavy cancellation; with every CRNN
            # expert on its training pack it measured 2.4e-3 (I = 2, eval) and 1.7e-3 (I = 3, train) on a B200
            budget = 5e-3 if (k == "route.bias" and arch == "crnn") else 1e-3
            e = float((gg - rg).abs().max()) / max(float(rg.abs().max()), 1e-4 * tn)
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
        prefixes = ("12.", "15.") if arch == "crnn" else ("patch_embed.proj.1.", "patch_embed.proj.4.")
        for e, m in enumerate(net.model):
            for bn, (m0, v0), pre in zip(_expert_bns(m, arch), old_bn[e], prefixes):
                mean, var = stats["model.%d.model.FeatureExtraction.ConvNet.%s" % (e, pre)]
                assert int(bn.num_batches_tracked) == 1, e
                assert rel_err(bn.running_mean.cpu().numpy(), (0.9 * m0.double() + 0.1 * mean).numpy()) < 1e-4
                assert rel_err(bn.running_var.cpu().numpy(), (0.9 * v0.double() + 0.1 * var).numpy()) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_module_in_front_of_the_net_trains(arch):
    """The use the image gradient exists for: a 1 x 1 Conv2d(4, 4) in front of MRNNet (frozen experts, I = 2, fp32,
    eval) gets the weight and bias gradients of the fp64 oracle: the oracle's image gradient pulled back through the
    convolution in fp64, within 1e-3 (SVTR) / 5e-3 (CRNN) relative max error."""
    cc, B, seed = (37, 61), 4, 81
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    torch.manual_seed(seed)
    front = torch.nn.Conv2d(4, 4, 1)
    with torch.no_grad():
        front.weight.copy_(torch.eye(4).view(4, 4, 1, 1) + 0.1 * front.weight)
    front = front.cuda()
    net = synth.build_net(cc, sd, arch=arch, autograd=True)
    net.eval()
    _set_trainable(net, ())
    y = front(img.cuda())
    out = net(y, True, None, True)
    loss = 15 * _ctc(out["logits"], tgt.cuda(), lens.cuda()) + F.cross_entropy(out["index"], dom.cuda())
    loss.backward()
    assert front.weight.grad is not None and front.bias.grad is not None
    ref = _routed_oracle(sd, 2, y.detach().cpu(), tgt, lens, dom, ())
    w64 = front.weight.detach().double().cpu().requires_grad_(True)
    b64 = front.bias.detach().double().cpu().requires_grad_(True)
    y64 = F.conv2d(img.double(), w64, b64)
    gw, gb = torch.autograd.grad(y64, [w64, b64], grad_outputs=ref["image"].double())
    budget = 1e-3 if arch == "svtr" else 5e-3
    assert rel_err(front.weight.grad.cpu().numpy(), gw.numpy()) < budget
    assert rel_err(front.bias.grad.cpu().numpy(), gb.numpy()) < budget


# ------------------------------------------------------------------------------------------------ 4. full size
@pytest.mark.gpu
def test_full_size_frozen_experts_image_grad_matches_fp64_oracle():
    """I = 6, B = 256, the MLT17 class counts, bf16, batch statistics, every expert frozen: image.grad within 5e-2
    relative Frobenius error of the fp64 oracle (the bf16 SVTR budget), the loss within 2e-2."""
    import gc
    cc, B, seed = synth.MLT17_CLASS_COUNTS, 256, 15
    I = len(cc)
    sd = synth.ctor_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    net = synth.build_net(cc, sd, precision="bf16", autograd=True)
    net.train()
    _set_trainable(net, ())
    x = img.cuda().requires_grad_(True)
    out = net(x, True, None, True)
    loss = 15 * _ctc(out["logits"], tgt.cuda(), lens.cuda()) + F.cross_entropy(out["index"], dom.cuda())
    loss.backward()
    got = x.grad.detach().cpu()
    assert all(p.grad is None for m in net.model for p in m.parameters())
    del net, out, x
    gc.collect()
    torch.cuda.empty_cache()
    ref = _routed_oracle(sd, I, img, tgt, lens, dom, (), "batch")
    assert abs(float(loss) - ref["loss"]) / abs(ref["loss"]) < 2e-2
    _check_image_grad(got, ref["image"], "svtr", "bf16", B)


# ------------------------------------------------------------------------------------------------ 5. input-only backward
@pytest.mark.gpu
@pytest.mark.parametrize("prec", ["fp32", "bf16"])
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_input_only_backward_equals_full_backward(arch, prec):
    """One pack, one input, batch statistics: dimage of the input-only backward (a pack built without a gradient arena,
    and the full pack asked for no parameter gradient) equals the full backward's within the run-to-run spread of the
    backward's atomics on the input-gradient path (BatchNorm reductions, the CRNN's split-K recurrent GEMMs): 1e-4
    relative max error in fp32, 1e-2 in bf16."""
    from mrn_b200 import ops
    from mrn_b200 import _lib as L
    cc, B, seed = (53,), 7, 91
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    x = synth.synth_batch(B, cc, seed)[0].cuda()
    esd = {k[len("model.0."):]: v for k, v in sd.items() if k.startswith("model.0.")}
    pk = L.PREC_FP32 if prec == "fp32" else L.PREC_BF16
    Pack = ops.CrnnTrainPack if arch == "crnn" else ops.SvtrTrainPack
    full, bare = Pack(esd, "cuda", pk), Pack(esd, "cuda", pk, param_grads=False)
    assert bare.grads is None
    T = 63 if arch == "crnn" else 64
    dl = synth.randn(seed, "dlogits", (B, T, cc[0]), 1e-2).cuda()

    def run(tp, param_grads):
        di = torch.full((B, 4, 32, 256), float("nan"), device="cuda")
        if arch == "crnn":
            ops.crnn_train_forward(tp, x, bn_batch_stats=True, update_running=False)
            g = ops.crnn_train_backward(tp, dl, B, bn_batch_stats=True, dimage=di, param_grads=param_grads)
        else:
            ops.svtr_train_forward(tp, x, bn_batch_stats=True, update_running=False)
            g = ops.svtr_train_backward(tp, x, dl, bn_batch_stats=True, dimage=di, param_grads=param_grads)
        assert (g is None) == (not param_grads)
        return di
    ref = run(full, True)
    budget = 1e-4 if prec == "fp32" else 1e-2
    for tp in (full, bare):
        got = run(tp, False)
        assert not torch.isnan(got).any()
        assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) < budget


def test_backward_without_gradients_or_image_is_refused():
    """No device needed: the argument check runs before any launch.  Neither a gradient arena nor dimage, or a
    gradient struct without its arena, is MRNB_ERR_ARG with a message naming the entry."""
    import ctypes as C
    from mrn_b200 import _lib as L
    from mrn_b200.build import build
    if not __import__("os").path.exists(L.LIB_PATH):
        build()
    lib = L.load()
    dummy = C.c_void_p(256)
    sp, cp = L.MrnbSvtrPack(), L.MrnbCrnnTrainPack()
    sp.n_experts = 1
    rc = lib.mrnb_svtr_train_backward_input(C.byref(sp), None, dummy, dummy, 64, None, 2, 0, 0, None, None, 0, None,
                                            dummy, 1 << 20, None)
    assert rc != 0 and b"svtr_train_backward" in lib.mrnb_last_error()
    rc = lib.mrnb_svtr_train_backward_input(C.byref(sp), C.byref(sp), dummy, dummy, 64, None, 2, 0, 0, None, None, 0,
                                            dummy, dummy, 1 << 20, None)
    assert rc != 0 and b"grad_arena" in lib.mrnb_last_error()
    rc = lib.mrnb_crnn_train_backward_input(C.byref(cp), None, dummy, 64, None, 2, 0, 0, None, 0, None, dummy, 1 << 20,
                                            None)
    assert rc != 0 and b"crnn_train_backward" in lib.mrnb_last_error()


# ------------------------------------------------------------------------------------------------ 6. inert when off
@pytest.mark.gpu
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_image_without_grad_is_inert(arch, monkeypatch):
    """Without image grad: the frozen soft route builds no training pack and returns bitwise the default forward's
    outputs; the joint soft route builds a pack for the trainable expert only (with its gradient arena) and its
    gradients repeat within the backward's run-to-run spread (1e-4 of max(max |g|, 1e-3 max_all |g|), as
    test_switch_with_every_expert_frozen_is_bitwise_today allows); Model.forward's "predict" is bitwise the cross=False
    logits; no image gradient appears anywhere."""
    cc, B, seed = (37, 61, 96), 3, 33
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    x, t, l, d = img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda()
    off = synth.build_net(cc, sd, arch=arch)
    on = synth.build_net(cc, sd, arch=arch, autograd=True, autograd_experts=True)
    for n in (off, on):
        n.eval()
    _set_trainable(on, ())
    calls = _record_packs(monkeypatch)
    a, b = off(x, True, None, True), on(x, True, None, True)
    assert torch.equal(a["logits"], b["logits"].detach()) and torch.equal(a["index"], b["index"].detach())
    assert calls == []
    _set_trainable(on, (2,))
    res = []
    for _ in range(2):
        on.zero_grad(set_to_none=True)
        xi = x.clone()
        out = on(xi, True, None, True)
        (15 * _ctc(out["logits"], t, l) + F.cross_entropy(out["index"], d)).backward()
        assert xi.grad is None
        res.append((out["logits"].detach(), {n: p.grad.clone() for n, p in on.named_parameters() if p.grad is not None}))
    assert calls == [(2, True), (2, True)]
    assert torch.equal(res[0][0], res[1][0])
    g0, g1 = res[0][1], res[1][1]
    assert set(g0) == set(g1)
    gmax = max(float(v.abs().max()) for v in g0.values())
    for k in g0:
        scale = max(float(g0[k].abs().max()), 1e-3 * gmax)
        assert float((g0[k] - g1[k]).abs().max()) / scale < 1e-4, k
    model = on.model[-1]
    last = on(x, cross=False)["logits"]
    pred = model(x)
    assert torch.equal(pred["predict"].detach(), last.detach()) and pred["feature"].requires_grad


@pytest.mark.gpu
def test_image_double_backward_raises():
    cc = (37,)
    sd = synth.synth_state_dict(cc, 4)
    net = synth.build_net(cc, sd, autograd=True)
    net.eval()
    x = synth.synth_batch(2, cc, 4)[0].cuda().requires_grad_(True)
    out = net.model[0](x)
    (gx,) = torch.autograd.grad(out["predict"].square().sum(), x, create_graph=True)
    with pytest.raises(RuntimeError, match="once_differentiable|differentiate twice"):
        gx.sum().backward()
