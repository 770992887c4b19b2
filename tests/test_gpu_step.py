"""End-to-end GPU parity through the reference-facing API (mrn_b200.modules.model.MRNNet, mrn_b200.il_modules.mrn.MRN)
against the golden fixtures produced by the unmodified reference and against the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import mrn_oracle as O
from mrn_b200 import synth
from conftest import gview, rel_err
from golden_cases import golden_case

pytestmark = pytest.mark.gpu


def ref_numel(g, pname):
    """Element count of a router parameter (arena slots are padded to 8 floats)."""
    cc = [int(c) for c in g["class_counts"]]
    shapes = synth.router_shapes(len(cc))
    return int(np.prod(shapes[pname]))


@pytest.mark.parametrize("name", ["svtr_mrn_i3_b3", "svtr_mrn_i2_b4"])
def test_mrnnet_forward_matches_reference_golden(name):
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case(name)
    net = synth.build_net(cc, sd)
    net.eval()
    x = img.cuda()
    out = net(x, True, None, True)                      # soft route (modules/model.py:397-423)
    assert np.abs(out["index"].cpu().numpy() - g["gate"]).max() < 1e-4               # gate weights within 1e-4
    assert rel_err(gview(out["logits"].cpu(), g), g["logits_soft"]) < 1e-4           # logits within 1e-4 relative
    ev = net(x, True, None, False)                      # hard route (modules/model.py:366-395)
    assert (ev["index"].cpu().numpy() == g["index_hard"]).all()
    assert rel_err(gview(ev["logits"].cpu(), g), g["logits_hard"]) < 1e-4
    ff = net(x, False, None, False)                     # cross=False: last expert only (modules/model.py:346-348)
    assert rel_err(gview(ff["logits"].cpu(), g), g["logits_last_expert"]) < 1e-4


@pytest.mark.parametrize("name", ["svtr_mrn_i3_b3", "svtr_mrn_i2_b4"])
def test_learner_eval_decode_matches_reference_golden(name):
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case(name)
    learner = synth.build_learner(synth.build_net(cc, sd), train=False)
    r = learner.infer_batch(img.cuda(), "TF", tgt.cuda(), lens.cuda())
    ties = 0
    for b in range(B):
        n = int(r["lens"][b])
        same = n == int(g["decode_len"][b]) and r["ids"][b, :n].cpu().tolist() == [int(v) for v in g["decode_ids"][b][:n]]
        ties += 0 if same else 1
    assert ties == 0, "decoded label indices differ from the reference on %d samples" % ties
    assert abs(float(r["loss"]) - float(g["valid_loss"])) / abs(float(g["valid_loss"])) < 1e-4
    assert rel_err(r["conf"].cpu().double().numpy(), g["confidence"]) < 1e-3


@pytest.mark.parametrize("name", ["svtr_mrn_i3_b3", "svtr_mrn_i2_b4"])
def test_stage1_step_matches_reference_golden(name):
    """loss = 15*CTC + CE(gate, domain), router gradients, clip_grad_norm_(5) and one Adam step (il_modules/mrn.py:338-367)."""
    from mrn_b200 import ops
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case(name)
    net = synth.build_net(cc, sd)
    learner = synth.build_learner(net, train=False, total_steps=20000)   # the golden step used eval-mode (frozen) experts
    loss_clf, taski = learner.train_step_stage1(img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda())
    assert abs(float(loss_clf) - float(g["loss_clf"])) / abs(float(g["loss_clf"])) < 1e-4
    assert abs(float(taski) - float(g["taski_loss"])) < 1e-4
    n, off = ops.router_param_offsets(len(cc))
    grads = net.router_grad_arena().cpu()
    tn = float(g["grad_total_norm"])
    assert abs(float(learner.optimizer.norm) - tn) / tn < 5e-4
    params = net.router_arena().cpu()
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        got = grads[off[k]:off[k] + ref_numel(g, pname)]
        ref = g["grad." + pname]
        scale = max(float(np.abs(ref).max()), 1e-4 * tn)
        assert np.abs(gview(got, g) - ref.reshape(-1)).max() / scale < 1e-3, pname
        if pname == "route.bias":
            continue
        d = np.abs(gview(params[off[k]:off[k] + ref_numel(g, pname)], g) - g["adam1." + pname].reshape(-1))
        assert d.max() <= 5e-4 * 1.01 and (d > 2e-5).mean() < 1e-2, pname


def test_train_mode_experts_match_oracle():
    """BN batch statistics + injected DropPath masks (reference quirk 4) through the module API."""
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case("svtr_mrn_i3_b3")
    net = synth.build_net(cc, sd)
    net.train()
    drop = synth.synth_drop_scales(len(cc), B, O.svtr_drop_path_rates(), seed)
    r = net.route_and_combine(img.cuda(), is_train=True, want_logits=True, drop_scales=drop.cuda())
    assert np.abs(r["gate"].cpu().numpy() - g["train_gate"]).max() < 1e-4
    assert rel_err(gview(r["logits"].cpu(), g), g["train_logits_soft"]) < 1e-4
    sd2 = net.state_dict()      # running statistics written back under the reference's keys
    k = "model.0.model.FeatureExtraction.ConvNet.patch_embed.proj.1.running_mean"
    assert np.abs(sd2[k].cpu().numpy() - g["train_bn1_running_mean_e0"]).max() < 1e-5
    assert int(sd2["model.0.model.FeatureExtraction.ConvNet.patch_embed.proj.1.num_batches_tracked"]) == 1


def test_bf16_mode_within_north_star_budget():
    """bf16 operands / fp32 accumulate for the expert GEMMs: logits within 2e-2 relative of the fp32 oracle on
    random-init weights (BASELINE.json north_star); gate deviation and expert flips are reported."""
    cc, B = (37, 61, 96), 4
    sd = synth.ctor_state_dict(cc, 5)
    img, tgt, lens, dom = synth.synth_batch(B, cc, 5)
    with torch.no_grad():
        o = O.mrn_forward(sd, len(cc), img, True, True)
        e = O.mrn_forward(sd, len(cc), img, True, False)
    net = synth.build_net(cc, sd, precision="bf16")
    net.eval()
    out = net(img.cuda(), True, None, True)
    assert rel_err(out["logits"].cpu().numpy(), o["logits"].numpy()) < 2e-2           # logits within 2e-2 in bf16
    gate_dev = float((out["index"].cpu() - o["index"]).abs().max())
    ev = net(img.cuda(), True, None, False)
    flips = int((ev["index"].cpu() != e["index"]).sum())
    print("bf16: gate max abs deviation %.2e, expert flips %d of %d" % (gate_dev, flips, B))
    assert gate_dev < 2e-2
    # fp32 mode on the same weights meets the fp32 tolerances
    net32 = synth.build_net(cc, sd, precision="fp32")
    net32.eval()
    out32 = net32(img.cuda(), True, None, True)
    assert rel_err(out32["logits"].cpu().numpy(), o["logits"].numpy()) < 1e-4
    assert float((out32["index"].cpu() - o["index"]).abs().max()) < 1e-4


def test_full_size_properties_6_experts():
    """BASELINE size (I=6, union charset 5153, B=32 here): size-independent properties -- gates are a distribution,
    hard route == soft route with a one-hot gate, logsumexp consistency, decode idempotence."""
    from mrn_b200 import ops
    cc = synth.MLT17_CLASS_COUNTS
    sd = synth.synth_state_dict(cc, 3)
    img, tgt, lens, dom = synth.synth_batch(32, cc, 3)
    net = synth.build_net(cc, sd, precision="bf16")
    net.eval()
    x = img.cuda()
    r = net.route_and_combine(x, is_train=True, want_logits=True, targets=tgt.cuda(), lengths=lens.cuda(), want_E=True,
                              want_decode=True)
    gate = r["gate"]
    assert torch.allclose(gate.sum(-1), torch.ones(32, device="cuda"), atol=1e-5) and (gate >= 0).all()
    assert torch.allclose(torch.logsumexp(r["logits"], -1), r["lse"], atol=1e-4)
    assert (r["logits"].max(-1)[1] == r["amax"].long()).all()
    # E_i rows are convex combinations of pad_i values -> bounded by them
    E = r["E"]
    for i, z in enumerate(r["expert_logits"]):
        hi = torch.maximum(z.max(-1)[0], torch.ones_like(z[..., 0])) if z.shape[-1] < cc[-1] else z.max(-1)[0]
        assert (E[..., i] <= hi + 1e-3).all()
    ev = net.route_and_combine(x, is_train=False, want_logits=True)
    onehot = torch.nn.functional.one_hot(ev["index"], 6).float()
    again = ops.gate_combine(r["expert_logits"], onehot, want_logits=True)
    assert torch.equal(again["logits"], ev["logits"])
    ids, n, conf = ops.greedy_decode(r["amax"], r["maxprob"])
    assert (n <= 64).all() and (conf >= 0).all() and (conf <= 1).all()      # 64-frame products of ~1e-2 underflow in fp32, as in the reference
    for b in range(4):      # a decoded sequence never contains blank or adjacent repeats of the raw path... it is collapsed
        seq = ids[b, :int(n[b])].tolist()
        assert 0 not in seq and -1 not in seq


def test_infer_batch_cuda_graph_replay_matches_eager():
    """The per-batch-size CUDA graph of the hard-routed inference call returns exactly what the eager call returns, for
    fresh inputs on every replay."""
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case("svtr_mrn_i3_b3")
    learner = synth.build_learner(synth.build_net(cc, sd), train=False)
    for k in range(3):
        x = synth.synth_batch(B, cc, 50 + k)[0].cuda()
        eager = learner.infer_batch(x, "TF")
        ref = {n: eager[n].clone() for n in ("ids", "lens", "conf", "index")}
        rep = learner.infer_batch_graphed(x, "TF")
        torch.cuda.synchronize()
        for n in ref:
            assert torch.equal(rep[n], ref[n]), n
    assert len(learner._infer_graphs) == 1


def test_train_step_cuda_graph_replay_matches_eager():
    """Stage-1 steps replayed from the CUDA graph update the router exactly like eager steps on the same batches
    (eval-mode experts: no DropPath randomness)."""
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case("svtr_mrn_i2_b4")
    arenas, losses = [], []
    for graphed in (False, True):
        net = synth.build_net(cc, sd)
        learner = synth.build_learner(net, train=False, total_steps=100, schedule="super")
        step = learner.train_step_stage1_graphed if graphed else learner.train_step_stage1
        ls = []
        for k in range(4):
            x, t, l, d = synth.synth_batch(B, cc, 70 + k)
            a, b = step(x.cuda(), t.cuda(), l.cuda(), d.cuda())
            ls.append((float(a), float(b)))
        arenas.append(net.router_arena().clone())
        losses.append(ls)
        if graphed:
            assert isinstance(learner._train_graphs[(B, "cuda:0", (False,) * len(cc))], tuple)
    # split-K fp32 atomics make the weight gradients run-to-run non-deterministic at the 1e-6 level: compare with tolerance
    assert torch.allclose(arenas[0], arenas[1], rtol=1e-4, atol=2e-5)
    for (a0, b0), (a1, b1) in zip(*losses):
        assert abs(a0 - a1) < 1e-4 * abs(a0) + 1e-6 and abs(b0 - b1) < 1e-4


# ------------------------------------------------------------------------------------------------ bf16 twins
def _oracle_stage1(sd, cc, img, tgt, lens, dom, bn_mode, drop):
    with torch.no_grad():
        feats, preds = [], []
        for i in range(len(cc)):
            f, z = O.expert_forward(sd, i, img, bn_mode, None if drop is None else drop[i])
            feats.append(f)
            preds.append(z)
    return O.stage1_router_grads(sd, torch.stack(feats, 1), preds, tgt, lens, dom, dtype=torch.float32), preds


@pytest.mark.parametrize("weights", ["ctor", "golden_fixture"])
def test_bf16_train_mode_experts_match_oracle(weights):
    """bf16 tensor-core twin of test_train_mode_experts_match_oracle: BN batch statistics + injected DropPath masks
    through svtr_experts_forward in the mode bench.py times.  Random-init weights: north_star's 2e-2 budget on logits and
    gates.  Gate-spreading golden fixture: per-expert logits within 2e-2; the soft-routed sum is as gate-sensitive as the
    reference under autocast (SURVEY.md §7), so it is bounded loosely."""
    cc, B, seed = (37, 61, 96), 3, 111
    sd = synth.ctor_state_dict(cc, seed) if weights == "ctor" else synth.synth_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    drop = synth.synth_drop_scales(len(cc), B, O.svtr_drop_path_rates(), seed)
    ref, preds = _oracle_stage1(sd, cc, img, tgt, lens, dom, "batch", drop)
    net = synth.build_net(cc, sd, precision="bf16")
    net.train()
    r = net.route_and_combine(img.cuda(), is_train=True, want_logits=True, drop_scales=drop.cuda())
    for i, z in enumerate(r["expert_logits"]):
        assert rel_err(z.cpu().numpy(), preds[i].numpy()) < 2e-2, i
    gate_dev = float((r["gate"].cpu() - ref["gate"]).abs().max())
    lerr = rel_err(r["logits"].cpu().numpy(), ref["logits"].numpy())
    print("bf16 train-mode (%s): gate dev %.2e, soft logits rel err %.2e" % (weights, gate_dev, lerr))
    if weights == "ctor":
        assert gate_dev < 2e-2 and lerr < 2e-2
    else:
        assert gate_dev < 0.25 and lerr < 0.25


def test_bf16_stage1_step_matches_oracle():
    """bf16 twin of test_stage1_step_matches_reference_golden on random-init weights: losses within 2e-2, router
    gradients (bf16 router GEMMs, fp32 accumulation) within 5e-2 of the fp32 oracle's, grad norm within 2e-2."""
    from mrn_b200 import ops
    cc, B, seed = (37, 61, 96), 4, 7
    sd = synth.ctor_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    ref, _ = _oracle_stage1(sd, cc, img, tgt, lens, dom, "eval", None)
    net = synth.build_net(cc, sd, precision="bf16")
    learner = synth.build_learner(net, train=False, total_steps=20000)
    loss_clf, taski = learner.train_step_stage1(img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda())
    assert abs(float(loss_clf) - float(ref["loss_clf"])) / abs(float(ref["loss_clf"])) < 2e-2
    assert abs(float(taski) - float(ref["taski_loss"])) < 2e-2
    tn = float(torch.sqrt(sum((g.double() ** 2).sum() for g in ref["grads"].values())))
    assert abs(float(learner.optimizer.norm) - tn) / tn < 2e-2
    n, off = ops.router_param_offsets(len(cc))
    grads = net.router_grad_arena().cpu()
    worst = 0.0
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        g_ref = ref["grads"][pname].reshape(-1)
        got = grads[off[k]:off[k] + g_ref.numel()]
        scale = max(float(g_ref.abs().max()), 1e-3 * tn)
        worst = max(worst, float((got - g_ref).abs().max()) / scale)
    print("bf16 stage-1 step: worst router-gradient deviation %.2e of its parameter's max" % worst)
    assert worst < 5e-2


def test_mixed_expert_modes_follow_each_modules_flag():
    """The reference can hold experts in different modes (newest expert .eval() after update_step1 while the frozen older
    ones are still .train(), il_modules/mrn.py:284-287 vs :107): each expert's BatchNorm follows its own module flag."""
    cc, B, seed = (37, 61, 96), 3, 111
    sd = synth.synth_state_dict(cc, seed)
    img = synth.synth_batch(B, cc, seed)[0]
    net = synth.build_net(cc, sd)
    net.train()
    net.model[-1].eval()
    assert net._experts_train_mode() == (True, True, False)
    r = net.route_and_combine(img.cuda(), is_train=True, want_logits=True)
    with torch.no_grad():
        want = [O.expert_forward(sd, i, img, "batch" if i < 2 else "eval", None)[1] for i in range(3)]
    for i in range(3):
        assert rel_err(r["expert_logits"][i].cpu().numpy(), want[i].numpy()) < 1e-4, i
    sd2 = net.state_dict()
    k = "model.%d.model.FeatureExtraction.ConvNet.patch_embed.proj.1.num_batches_tracked"
    assert int(sd2[k % 0]) == 1 and int(sd2[k % 2]) == 0          # only the train-mode experts updated their statistics
