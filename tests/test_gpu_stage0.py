"""Stage-0 expert training (il_modules/mrn.py:225-279) on the GPU through the C ABI: the activation-keeping forward,
the hand-written backward to every parameter of the newest SVTR expert, clip + Adam on the arena -- against the golden
fixtures produced by the unmodified reference (autograd) and against the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import mrn_oracle as O
from mrn_b200 import synth
from conftest import load_golden, gview, rel_err
from test_oracle_pinning import STAGE0_CASES, STAGE0_CRNN_CASES, pview, stage0_case

pytestmark = pytest.mark.gpu

# analytically zero gradients (a conv bias in front of a batch-statistics BatchNorm; the key third of qkv.bias):
# what is left is round-off, compared on the scale of the whole gradient
def _abs_scale_only(key, bn_train):
    return bn_train and key.endswith(("patch_embed.proj.0.bias", "patch_embed.proj.3.bias"))


def _run_step(name, prec=0):
    from mrn_b200 import ops
    g, cc, B, sd, img, tgt, lens, bn_train, drop = stage0_case(name)
    i = len(cc) - 1
    pre = f"model.{i}."
    esd = {k[len(pre):]: v for k, v in sd.items() if k.startswith(pre)}
    crnn = str(g["arch"]) == "crnn" if "arch" in g else False
    x = img.cuda()
    dsc = drop.cuda().contiguous() if drop is not None else None
    if crnn:
        tp = ops.CrnnTrainPack(esd, "cuda", prec)
        logits = ops.crnn_train_forward(tp, x, bn_batch_stats=bn_train, update_running=bn_train)
    else:
        tp = ops.SvtrTrainPack(esd, "cuda", prec)
        logits = ops.svtr_train_forward(tp, x, bn_batch_stats=bn_train, update_running=bn_train, drop_scales=dsc)
    t, l = tgt.cuda(), lens.cuda()
    r = ops.gate_combine([logits], torch.ones(B, 1, device="cuda"), t, l)
    c = ops.ctc_lattice(r["lpe"], t, l, want_occ=True)
    dlogits = ops.ctc_dense_grad(logits, r["lse"], c["occ"], c["nll"], t, l, 1.0 / B)
    if crnn:
        ops.crnn_train_backward(tp, dlogits, B, bn_batch_stats=bn_train)
    else:
        ops.svtr_train_backward(tp, x, dlogits, bn_batch_stats=bn_train, drop_scales=dsc)
    torch.cuda.synchronize()
    return g, cc, sd, tp, logits, c, bn_train, pre


@pytest.mark.parametrize("name", STAGE0_CASES + STAGE0_CRNN_CASES)
def test_stage0_forward_loss_and_every_gradient_match_reference_golden(name):
    g, cc, sd, tp, logits, c, bn_train, pre = _run_step(name)
    assert rel_err(gview(logits.cpu(), g), g["logits"]) < 1e-4
    assert abs(float(c["loss"]) - float(g["loss"])) / abs(float(g["loss"])) < 1e-4
    tn = float(g["grad_total_norm"])
    grads = tp.state(tp.grads)
    total = 0.0
    bad = []
    for key, gg in grads.items():
        gk = "grad." + pre + key
        ref = g[gk]
        total += float((gg.double() ** 2).sum())
        scale = max(float(np.abs(ref).max()), 1e-4 * tn)
        if _abs_scale_only(key, bn_train):
            scale = tn
        err = np.abs(pview(gg.contiguous().cpu(), g) - ref).max() / scale
        nerr = abs(float(gg.double().norm()) - float(g["gradnorm." + pre + key])) / max(float(g["gradnorm." + pre + key]), 1e-4 * tn)
        if err > 1e-3 or (nerr > 1e-3 and not _abs_scale_only(key, bn_train)):
            bad.append((key, float(err), float(nerr)))
    assert not bad, bad
    assert abs(total ** 0.5 - tn) / tn < 5e-4
    if bn_train:                                   # running statistics, momentum 0.1 (nn.BatchNorm2d in .train())
        from mrn_b200 import _lib as L
        if getattr(tp, "arch", "svtr") == "crnn":
            keys = (((0, "mean"), "bn0_running_mean"), ((0, "var"), "bn0_running_var"), ((1, "mean"), "bn1_running_mean"),
                    ((1, "var"), "bn1_running_var"))
        else:
            keys = ((L.P_BN0_MEAN, "bn0_running_mean"), (L.P_BN0_VAR, "bn0_running_var"),
                    (L.P_BN1_MEAN, "bn1_running_mean"), (L.P_BN1_VAR, "bn1_running_var"))
        for slot, gk in keys:
            assert rel_err(tp.bn_stats[slot].cpu().numpy().reshape(-1), g[gk]) < 1e-4, gk


@pytest.mark.parametrize("name", STAGE0_CASES)
def test_stage0_clip_and_adam_step_matches_reference_golden(name):
    from mrn_b200 import ops
    g, cc, sd, tp, logits, c, bn_train, pre = _run_step(name)
    m, v = torch.zeros_like(tp.params), torch.zeros_like(tp.params)
    norm = ops.clip_adam(tp.params, tp.grads, m, v, 5e-4, 1, max_norm=5.0)
    assert abs(float(norm) - float(g["grad_total_norm"])) / float(g["grad_total_norm"]) < 5e-4
    for key, p in tp.state().items():
        d = np.abs(pview(p.contiguous().cpu(), g) - g["adam1." + pre + key])
        if _abs_scale_only(key, bn_train):
            continue
        if key.endswith("qkv.bias"):
            n = d.size // 3
            d = np.concatenate([d[:n], d[2 * n:]])
        # Adam's first step is lr * g / (|g| + eps): elements whose clipped gradient is ~eps are round-off sensitive
        assert d.max() <= 5e-4 * 2.01 and (d > 2e-5).sum() <= max(2, 0.02 * d.size), key


@pytest.mark.parametrize("name", STAGE0_CRNN_CASES)
def test_crnn_stage0_bf16_mode_runs_at_ragged_batch_sizes(name):
    """CRNN bf16 mode at B = 2 / 3 (B * 63 rows is not a multiple of the 64-wide contraction block: TMA zero-fill pads
    it): loss within 2e-2 of the reference, head / LSTM gradients within 8e-2 (two or three samples: little averaging
    of the bf16 rounding, and every layer below -- conv0 included -- runs on bf16 operands), total norm within 5e-2."""
    g, cc, sd, tp, logits, c, bn_train, pre = _run_step(name, prec=1)
    assert abs(float(c["loss"]) - float(g["loss"])) / abs(float(g["loss"])) < 2e-2
    tn = float(g["grad_total_norm"])
    total = 0.0
    for key, gg in tp.state(tp.grads).items():
        total += float((gg.double() ** 2).sum())
        if "ConvNet" in key:
            continue
        ref = g["grad." + pre + key]
        diff = np.linalg.norm(pview(gg.contiguous().cpu(), g) - ref)
        scale = max(np.linalg.norm(ref), 2e-3 * tn * (ref.size / max(gg.numel(), 1)) ** 0.5)
        assert diff / scale < 8e-2, (key, diff / scale)
    assert abs(total ** 0.5 - tn) / tn < 5e-2


@pytest.mark.parametrize("name", STAGE0_CASES)
def test_stage0_bf16_tensor_core_mode_within_budget(name):
    """MRNB_PREC_BF16: every GEMM of the expert forward and backward on tcgen05 (bf16 operands, fp32 accumulation).
    Budget (BASELINE.json north_star: 2e-2 in bf16): loss and logits within 2e-2; each parameter's gradient within
    5e-2 of the reference in relative Frobenius norm over the stored subsample (noise-only tensors on the scale of
    the whole gradient); total gradient norm within 2e-2."""
    g, cc, sd, tp, logits, c, bn_train, pre = _run_step(name, prec=1)
    assert rel_err(gview(logits.cpu(), g), g["logits"]) < 2e-2
    assert abs(float(c["loss"]) - float(g["loss"])) / abs(float(g["loss"])) < 2e-2
    tn = float(g["grad_total_norm"])
    total = 0.0
    bad = []
    for key, gg in tp.state(tp.grads).items():
        ref = g["grad." + pre + key]
        total += float((gg.double() ** 2).sum())
        diff = np.linalg.norm(pview(gg.contiguous().cpu(), g) - ref)
        scale = max(np.linalg.norm(ref), 2e-3 * tn * (ref.size / max(gg.numel(), 1)) ** 0.5)
        if diff / scale > 5e-2:
            bad.append((key, float(diff / scale)))
    assert not bad, bad
    assert abs(total ** 0.5 - tn) / tn < 2e-2


def test_stage0_matches_oracle_on_a_fresh_batch_with_edge_case_targets():
    """Oracle (autograd over the CPU restatement, fp64) vs the CUDA path on inputs that are not in the fixtures:
    repeated labels, an empty target and an infeasible (too long for T with repeats) target."""
    from mrn_b200 import ops
    cc, B, seed = (41, 77), 4, 5
    sd = synth.synth_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    tgt[0, :6] = torch.tensor([5, 5, 5, 9, 9, 5]); lens[0] = 6
    lens[1] = 0; tgt[1] = 1
    drop = synth.synth_drop_scales(2, B, O.svtr_drop_path_rates(), seed)[1]
    r = O.stage0_loss_and_grads(sd, 1, img, tgt, lens, "batch", drop)
    esd = {k[len("model.1."):]: v for k, v in sd.items() if k.startswith("model.1.")}
    tp = ops.SvtrTrainPack(esd, "cuda")
    x, t, l, dsc = img.cuda(), tgt.cuda(), lens.cuda(), drop.cuda().contiguous()
    logits = ops.svtr_train_forward(tp, x, True, True, dsc)
    rr = ops.gate_combine([logits], torch.ones(B, 1, device="cuda"), t, l)
    c = ops.ctc_lattice(rr["lpe"], t, l, want_occ=True)
    dlogits = ops.ctc_dense_grad(logits, rr["lse"], c["occ"], c["nll"], t, l, 1.0 / B)
    ops.svtr_train_backward(tp, x, dlogits, True, dsc)
    assert rel_err(logits.cpu().double().numpy(), r["logits"].numpy()) < 1e-4
    assert abs(float(c["loss"]) - float(r["loss"])) / abs(float(r["loss"])) < 1e-4
    tn = sum(float((v.double() ** 2).sum()) for v in r["grads"].values()) ** 0.5
    for key, gg in tp.state(tp.grads).items():
        ref = r["grads"]["model.1." + key].numpy()
        scale = max(float(np.abs(ref).max()), 1e-4 * tn)
        if _abs_scale_only(key, True):
            scale = tn
        assert np.abs(gg.cpu().double().numpy() - ref).max() / scale < 1e-3, key


class _Loader:
    """Stands in for data/data_manage.py's loader: get_batch() -> (images [B,4,32,256], label strings)."""

    def __init__(self, images, labels):
        self.images, self.labels, self.k = images, labels, 0

    def get_batch(self):
        self.k += 1
        return self.images, self.labels

    def __iter__(self):
        yield self.images, self.labels


@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_learner_init_train_follows_the_oracle_for_three_iterations(tmp_path, monkeypatch, arch):
    """MRN._init_train (reference API) on a fixed batch: per-iteration losses follow the CPU oracle's
    stage0_step_cpu (same DropPath masks, OneCycle learning rates), the trained weights land back in the nn.Module
    tree (state_dict keys unchanged) and the FF validation path sees them."""
    from mrn_b200.il_modules.mrn import MRN, RankLocal, one_cycle_lr
    from mrn_b200 import ops
    monkeypatch.chdir(tmp_path)
    cc, B, seed = (30,), 3, 3
    chars = [chr(0x4E00 + i) for i in range(cc[0] - 4)]
    sd = synth.synth_state_dict(cc, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    tgt[tgt == 2] = 4; tgt[tgt == 3] = 5      # [UNK] / ' ' are multi-character or stripped entries: keep plain characters
    opt = synth.make_opt(arch, num_iter=3, val_interval=100, lan_list=["x"], drop_path=True)
    opt.cuda_graph = False                    # eager steps: the injected DropPath masks must be consumed one per iteration
    learner = MRN(opt)
    learner.character = chars
    learner.converter = learner.build_converter()
    idx2ch = learner.converter.character
    labels = ["".join(idx2ch[int(c)] for c in tgt[b, :int(lens[b])]) for b in range(B)]
    learner.build_model()
    learner.net.load_state_dict(sd, strict=True)
    learner.model = RankLocal(learner.net).cuda()
    learner.model.train()
    # fixed DropPath masks for both sides
    drops = [synth.synth_drop_scales(1, B, O.svtr_drop_path_rates(), 100 + k)[0] for k in range(3)]
    import mrn_b200.il_modules.mrn as M
    it = iter(drops)
    monkeypatch.setattr(M, "sample_drop_scales", lambda n, b, rates, dev: next(it).unsqueeze(0).to(dev))
    losses = []
    orig = MRN.train_step_stage0

    def spy(self, *a, **k):
        out = orig(self, *a, **k)
        losses.append(float(out))
        return out
    monkeypatch.setattr(MRN, "train_step_stage0", spy)
    learner._init_train(0, 0, _Loader(img, labels), _Loader(img, labels))
    # oracle
    sdo = {k: v.clone() for k, v in sd.items()}
    state = dict(step=0, m={}, v={})
    ref_losses = []
    for k in range(3):
        ref_losses.append(O.stage0_step_cpu(sdo, 0, state, img, tgt, lens, lr=one_cycle_lr(k, 3, opt.lr), bn_mode="batch",
                                            drop_scales=drops[k] if arch == "svtr" else None))
    assert np.allclose(losses, ref_losses, rtol=2e-3), (losses, ref_losses)
    new_sd = learner.model.state_dict()
    assert set(new_sd) == {"module." + k for k in sd}
    w = ("model.0.model.FeatureExtraction.ConvNet.blocks2.3.mlp.fc1.weight" if arch == "svtr"
         else "model.0.model.SequenceModeling.1.linear.weight")
    assert float((new_sd["module." + w].cpu() - sd[w]).abs().max()) > 1e-5            # it trained
    assert rel_err(new_sd["module." + w].cpu().numpy(), sdo[w].numpy()) < 2e-2
    out = learner.net(img.cuda(), cross=False, is_train=False)
    assert torch.isfinite(out["logits"]).all()


def test_crnn_stage0_bf16_tensor_core_mode_tracks_fp32_mode_at_batch_64():
    """CRNN expert training in MRNB_PREC_BF16 (every conv / Linear / LSTM input-projection GEMM and its gradients on
    tcgen05) against the fp32 parity mode on the same batch: loss within 2e-2; the
    gradients of the CTC head and both BidirectionalLSTMs within 3e-2 in relative Frobenius norm.  Through the seven
    ReLU convolution layers below them the bf16 operand rounding compounds on these random-init weights (measured
    2 % at ConvNet.18 growing to 19 % at ConvNet.0, while the bf16 forward moves the logits by 1.3 %): those tensors
    are held to 0.25 and to a cosine similarity above 0.97 with the fp32 gradient."""
    from mrn_b200 import ops
    cc, B, seed = (53,), 64, 9
    sd = synth.synth_state_dict(cc, seed, arch="crnn")
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    esd = {k[len("model.0."):]: v for k, v in sd.items() if k.startswith("model.0.")}
    x, t, l = img.cuda(), tgt.cuda(), lens.cuda()
    res = []
    for prec in (0, 1):
        tp = ops.CrnnTrainPack(esd, "cuda", prec)
        logits = ops.crnn_train_forward(tp, x, True, True)
        rr = ops.gate_combine([logits], torch.ones(B, 1, device="cuda"), t, l)
        c = ops.ctc_lattice(rr["lpe"], t, l, want_occ=True)
        dlogits = ops.ctc_dense_grad(logits, rr["lse"], c["occ"], c["nll"], t, l, 1.0 / B)
        ops.crnn_train_backward(tp, dlogits, B, True)
        torch.cuda.synchronize()
        res.append((float(c["loss"]), {k: v.clone() for k, v in tp.state(tp.grads).items()}))
    (l32, g32), (l16, g16) = res
    assert abs(l16 - l32) / abs(l32) < 2e-2
    tn = sum(float((v.double() ** 2).sum()) for v in g32.values()) ** 0.5
    bad = []
    for k in g32:
        a, b = g32[k].double().reshape(-1), g16[k].double().reshape(-1)
        scale = max(float(a.norm()), 2e-3 * tn)
        e = float((b - a).norm()) / scale
        cos = float((a * b).sum() / (a.norm() * b.norm() + 1e-30))
        budget = 0.25 if "ConvNet" in k else 3e-2
        if e > budget or cos < 0.97:
            bad.append((k, e, cos))
    assert not bad, bad


@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_stage0_cuda_graph_replay_matches_eager(arch):
    """train_step_stage0_graphed (forward + CTC + backward replayed from a CUDA graph) == the eager step, over three
    iterations on rotating batches (DropPath off: the graph draws its masks from torch's graph-safe generator)."""
    from mrn_b200.il_modules.mrn import MRN, RankLocal
    cc, B = (40,), 4
    sd = synth.synth_state_dict(cc, 13, arch=arch)
    batches = [synth.synth_batch(B, cc, 50 + k) for k in range(2)]
    outs = []
    for graphed in (False, True):
        opt = synth.make_opt(arch, num_iter=100, schedule="const")
        learner = MRN(opt)
        learner.model.update_fc(opt.hidden_size, cc[0]); learner.model.build_prediction(opt, cc[0])
        learner.model.load_state_dict(sd, strict=True)
        learner.model = RankLocal(learner.net).cuda()
        learner.model.train()
        learner.begin_expert_training()
        losses = []
        for k in range(4):
            img, tgt, lens, _ = batches[k % 2]
            step = learner.train_step_stage0_graphed if graphed else learner.train_step_stage0
            losses.append(float(step(img.cuda(), tgt.cuda(), lens.cuda())))
        torch.cuda.synchronize()
        outs.append((losses, learner._tp.params.clone()))
    (l0, p0), (l1, p1) = outs
    # split-K atomics reorder the fp32 sums; Adam's first steps (lr * sign-like) amplify that round-off in later losses
    assert np.allclose(l0[:2], l1[:2], rtol=1e-5) and np.allclose(l0, l1, rtol=1e-3), (l0, l1)
    d = (p0 - p1).abs()
    assert float(d.max()) <= 5e-4 * 4.01 and float((d > 5e-5).float().mean()) < 2e-2


@pytest.mark.parametrize("arch,precision", [("svtr", "fp32"), ("svtr", "bf16"), ("crnn", "fp32")])
def test_stage0_training_reduces_the_loss_on_a_fixed_batch(arch, precision):
    """Sixty expert-training iterations on one batch (constant learning rate): the CTC loss must fall well below its
    starting value -- gradients, clip + Adam and the arena write-back work together."""
    from mrn_b200.il_modules.mrn import MRN, RankLocal
    cc, B = (40,), 8
    sd = synth.synth_state_dict(cc, 21, arch=arch)
    img, tgt, lens, _ = synth.synth_batch(B, cc, 77)
    lens = lens.clamp(max=8); tgt[:, 8:] = 1
    opt = synth.make_opt(arch, precision, num_iter=1000, schedule="const")
    learner = MRN(opt)
    learner.model.update_fc(opt.hidden_size, cc[0]); learner.model.build_prediction(opt, cc[0])
    learner.model.load_state_dict(sd, strict=True)
    learner.model = RankLocal(learner.net).cuda()
    learner.model.train()
    learner.begin_expert_training()
    x, t, l = img.cuda(), tgt.cuda(), lens.cuda()
    losses = [float(learner.train_step_stage0(x, t, l)) for _ in range(60)]
    print(arch, precision, [round(v, 2) for v in losses[::5]])
    assert all(np.isfinite(losses)), losses
    assert np.mean(losses[-10:]) < 0.8 * losses[0], (losses[0], losses[-10:])
    learner.end_expert_training()
    out = learner.net(x, cross=False, is_train=False)          # the inference path sees the trained weights
    assert torch.isfinite(out["logits"]).all()


@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_stage0_full_size_properties(arch):
    """BASELINE.json's full size (B = 256, union charset C = 5153, bf16 tensor-core mode): size-independent properties
    of the step, which hold without a reference (test_gpu_stage0_scale.py compares this size with the fp64 oracle).
    (1) softmax - occupancy sums to zero over the classes of every frame, so the fc.bias gradient sums to zero; (2) the gradient of the mean loss is linear in the per-sample weights: the step
    on the batch equals the average of the steps on its two halves for every parameter that does not see batch
    statistics (eval-mode BatchNorm); (3) two runs agree up to the order of the split-K reductions."""
    from mrn_b200 import ops
    cc, B = (5153,), 256
    sd = synth.synth_state_dict(cc, 111, arch=arch)
    img, tgt, lens, _ = synth.synth_batch(B, cc, 2024)
    esd = {k[len("model.0."):]: v for k, v in sd.items() if k.startswith("model.0.")}
    x, t, l = img.cuda(), tgt.cuda(), lens.cuda()
    tp = (ops.SvtrTrainPack if arch == "svtr" else ops.CrnnTrainPack)(esd, "cuda", 1)

    def run(lo, hi):
        xs, ts, ls = x[lo:hi].contiguous(), t[lo:hi].contiguous(), l[lo:hi].contiguous()
        n = hi - lo
        if arch == "svtr":
            logits = ops.svtr_train_forward(tp, xs, False, False, None)
        else:
            logits = ops.crnn_train_forward(tp, xs, False, False)
        rr = ops.gate_combine([logits], torch.ones(n, 1, device="cuda"), ts, ls)
        c = ops.ctc_lattice(rr["lpe"], ts, ls, want_occ=True)
        dlogits = ops.ctc_dense_grad(logits, rr["lse"], c["occ"], c["nll"], ts, ls, 1.0 / n)
        if arch == "svtr":
            ops.svtr_train_backward(tp, xs, dlogits, False, None)
        else:
            ops.crnn_train_backward(tp, dlogits, n, False)
        torch.cuda.synchronize()
        return float(c["loss"]), tp.grads.clone()

    loss, g = run(0, B)
    loss2, g2 = run(0, B)
    la, ga = run(0, B // 2)
    lb, gb = run(B // 2, B)
    assert np.isfinite(loss) and torch.isfinite(g).all()
    gn = float(g.double().norm())
    fcb = tp.state(g)["fc.bias"].double()
    assert abs(float(fcb.sum())) < 1e-3 * float(fcb.abs().sum())                   # (1)
    assert abs(0.5 * (la + lb) - loss) / abs(loss) < 2e-3                          # (2) mean of the half-batch means
    assert float((0.5 * (ga + gb) - g).double().norm()) / gn < 2e-2
    assert abs(loss2 - loss) / abs(loss) < 1e-5 and float((g2 - g).double().norm()) / gn < 1e-3      # (3)
