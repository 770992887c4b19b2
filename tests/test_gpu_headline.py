"""Parity on the MEASURED configuration (BASELINE.json configs[3], what bench.py times): SVTR-MRN, I = 6 experts with
the MLT17 union charset (C = 5153), B = 256, bf16 tensor-core mode, experts in train mode (BatchNorm batch statistics
+ DropPath, reference quirk 4), random-init weights from the constructors -- against the fp32 CPU oracle of the same
step (oracle.mrn_oracle, restating il_modules/mrn.py:338-371 and modules/model.py:397-423)."""
import math

import pytest
import torch

from oracle import mrn_oracle as O
from oracle import synth
from mrn_b200 import synth as psynth

pytestmark = pytest.mark.gpu

CC = synth.MLT17_CLASS_COUNTS
B = 256
TOL = 2e-2          # BASELINE.json north_star: logits / CTC loss within 2e-2 relative in bf16


def _learner(sd, drop_path=True, precision="bf16"):
    """The bench's options (bench.make_opt) with DropPath on or off."""
    from bench import make_opt
    opt = make_opt(precision, 0, "svtr")
    opt.drop_path = drop_path
    net = psynth.build_net(CC, sd, opt)
    return psynth.build_learner(net, total_steps=20000), net


def _oracle_step(sd, state, batch, drop):
    """One fp32 CPU step; returns (loss_clf, taski, gate, logits) BEFORE the update and applies clip + Adam to sd."""
    img, tgt, lens, dom = batch
    with torch.no_grad():
        feats, preds = [], []
        for i in range(len(CC)):
            f, z = O.expert_forward(sd, i, img, "batch", None if drop is None else drop[i])
            feats.append(f)
            preds.append(z)
        x = torch.stack(feats, 1)
    r = O.stage1_router_grads(sd, x, preds, tgt, lens, dom, 15.0, dtype=torch.float32)
    O.clip_and_adam({k: sd[k] for k in O.ROUTER_KEYS}, r["grads"], state, 5e-4)
    return float(r["loss_clf"]), float(r["taski_loss"]), r["gate"], r["logits"]


def test_headline_step_b256_bf16_train_mode_matches_oracle():
    sd = psynth.ctor_state_dict(CC, 111)
    learner, net = _learner(sd)
    sd_o = {k: v.clone() for k, v in sd.items()}
    state = dict(step=0, m={}, v={})
    rates = O.svtr_drop_path_rates()
    got, ref = [], []
    for k in range(10):
        batch = synth.synth_batch(B, CC, 1000 + k)
        drop = synth.synth_drop_scales(len(CC), B, rates, 7 + k)
        img, tgt, lens, dom = (t.cuda() for t in batch)
        if k == 0:          # forward-only probe of the same batch: gate and combined logits against the oracle
            r = net.route_and_combine(img, is_train=True, want_logits=True, drop_scales=drop.cuda())
            gate0, logits0 = r["gate"].cpu(), r["logits"].cpu()
            # the probe's train-mode forward updated the BN running statistics once more than the reference would; they
            # do not enter a train-mode forward, so the step below is unaffected
        l1, l2 = learner.train_step_stage1(img, tgt, lens, dom, drop_scales=drop.cuda())
        got.append((float(l1), float(l2)))
        if k < 2:           # the oracle costs ~15 s per step on the host: pin the first two steps (2nd = after one update)
            ref.append(_oracle_step(sd_o, state, batch, drop))
    assert all(math.isfinite(a) and math.isfinite(b) for a, b in got), got
    assert float(learner.optimizer.norm) == float(learner.optimizer.norm)        # grad norm of the last step is not NaN
    assert torch.isfinite(net.router_arena()).all()
    gate_ref, logits_ref = ref[0][2], ref[0][3]
    assert float((gate0 - gate_ref).abs().max()) < TOL
    assert float((logits0 - logits_ref).abs().max() / logits_ref.abs().max()) < TOL
    for k in range(2):
        assert abs(got[k][0] - ref[k][0]) / abs(ref[k][0]) < TOL, (k, got[k], ref[k][:2])
        assert abs(got[k][1] - ref[k][1]) < TOL, (k, got[k], ref[k][:2])
    print("headline parity: GPU (loss_clf, taski) %s vs oracle %s; gate max dev %.2e" %
          (got[:2], [r[:2] for r in ref], float((gate0 - gate_ref).abs().max())))


def test_headline_step_graphed_equals_eager_and_stays_finite():
    """CUDA-graph replay of the B=256 step: with DropPath off both paths are deterministic and must agree; with DropPath
    on (masks drawn inside the graph) the losses must stay finite and close to the eager first-step loss."""
    sd = psynth.ctor_state_dict(CC, 111)
    runs = {}
    for graphed in (False, True):
        learner, net = _learner(sd, drop_path=False)
        step = learner.train_step_stage1_graphed if graphed else learner.train_step_stage1
        ls = []
        for k in range(10):
            img, tgt, lens, dom = (t.cuda() for t in synth.synth_batch(B, CC, 1000 + k % 4))
            a, b = step(img, tgt, lens, dom)
            ls.append((float(a), float(b)))
        runs[graphed] = ls
        assert torch.isfinite(net.router_arena()).all()
    for (a0, b0), (a1, b1) in zip(runs[False], runs[True]):
        assert math.isfinite(a1) and math.isfinite(b1)
        assert abs(a0 - a1) < 2e-3 * abs(a0) and abs(b0 - b1) < 2e-3, (runs[False], runs[True])
    learner, net = _learner(sd, drop_path=True)
    ls = []
    for k in range(10):
        img, tgt, lens, dom = (t.cuda() for t in synth.synth_batch(B, CC, 1000 + k % 4))
        a, b = learner.train_step_stage1_graphed(img, tgt, lens, dom)
        ls.append((float(a), float(b)))
    assert all(math.isfinite(a) and math.isfinite(b) for a, b in ls), ls
    assert abs(ls[0][0] - runs[False][0][0]) < 0.1 * abs(runs[False][0][0])


def test_expert_forward_is_deterministic_b256():
    """Reruns of the grouped 6-expert forward on identical inputs (train mode, fixed DropPath masks) are bitwise equal."""
    from mrn_b200 import _lib as L, ops
    sd = psynth.ctor_state_dict(CC, 111)
    learner, net = _learner(sd)
    img = synth.synth_batch(B, CC, 1000)[0].cuda()
    drop = synth.synth_drop_scales(len(CC), B, O.svtr_drop_path_rates(), 7).cuda()
    pack = net._cache.get(list(net.model), img.device, L.PREC_BF16)
    outs = []
    for _ in range(4):
        f, z = ops.svtr_experts_forward(pack, img, bn_batch_stats=True, update_running=False, drop_scales=drop)
        outs.append((f.clone(), [t.clone() for t in z]))
    for f, z in outs[1:]:
        assert torch.equal(f, outs[0][0])
        for a, b in zip(z, outs[0][1]):
            assert torch.equal(a, b)
    assert torch.isfinite(outs[0][0]).all()
