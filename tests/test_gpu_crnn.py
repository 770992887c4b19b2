"""CRNN-MRN (VGG + BiLSTM + CTC, T = 63; config/crnn_mrn.py, BASELINE.json configs[0-1]) on the GPU through the
reference-facing API, against the golden fixtures produced by the unmodified reference and the CPU oracle."""
import numpy as np
import pytest
import torch

from oracle import mrn_oracle as O
from mrn_b200 import synth
from conftest import gview, rel_err
from golden_cases import golden_case

pytestmark = pytest.mark.gpu
CASES = ["crnn_mrn_i2_b4", "crnn_mrn_i3_b2"]


@pytest.mark.parametrize("name", CASES)
def test_crnn_forward_matches_reference_golden(name):
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case(name)
    net = synth.build_net(cc, sd, arch="crnn")
    net.eval()
    x = img.cuda()
    r = net.route_and_combine(x, is_train=True, want_logits=True)
    assert r["features"].shape == (B, len(cc), 63, 256)
    assert rel_err(gview(r["features"].cpu(), g), g["features"]) < 1e-4
    out = net(x, True, None, True)
    assert out["logits"].shape == (B, 63, cc[-1])
    assert np.abs(out["index"].cpu().numpy() - g["gate"]).max() < 1e-4
    assert rel_err(gview(out["logits"].cpu(), g), g["logits_soft"]) < 1e-4
    ev = net(x, True, None, False)
    assert (ev["index"].cpu().numpy() == g["index_hard"]).all()
    assert rel_err(gview(ev["logits"].cpu(), g), g["logits_hard"]) < 1e-4
    ff = net(x, False, None, False)
    assert rel_err(gview(ff["logits"].cpu(), g), g["logits_last_expert"]) < 1e-4
    one = net.model[0](x)                               # Model.forward of a single expert (modules/model.py:133-148)
    assert one["predict"].shape == (B, 63, cc[0]) and one["feature"].shape == (B, 63, 256)


@pytest.mark.parametrize("name", CASES)
def test_crnn_eval_decode_and_loss_match_reference_golden(name):
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case(name)
    learner = synth.build_learner(synth.build_net(cc, sd, arch="crnn"), train=False)
    r = learner.infer_batch(img.cuda(), "TF", tgt.cuda(), lens.cuda())
    for b in range(B):
        n = int(r["lens"][b])
        assert n == int(g["decode_len"][b])
        assert r["ids"][b, :n].cpu().tolist() == [int(v) for v in g["decode_ids"][b][:n]]
    assert abs(float(r["loss"]) - float(g["valid_loss"])) / abs(float(g["valid_loss"])) < 1e-4
    assert rel_err(r["conf"].cpu().double().numpy(), g["confidence"]) < 1e-3


@pytest.mark.parametrize("name", CASES)
def test_crnn_stage1_step_matches_reference_golden(name):
    """Router-training step with T = 63: loss, router gradients, clip + Adam (il_modules/mrn.py:338-367)."""
    from mrn_b200 import ops
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case(name)
    net = synth.build_net(cc, sd, arch="crnn")
    learner = synth.build_learner(net, train=False, total_steps=20000)
    loss_clf, taski = learner.train_step_stage1(img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda())
    assert abs(float(loss_clf) - float(g["loss_clf"])) / abs(float(g["loss_clf"])) < 1e-4
    assert abs(float(taski) - float(g["taski_loss"])) < 1e-4
    n, off = ops.router_param_offsets(len(cc), 63)
    grads = net.router_grad_arena().cpu()
    tn = float(g["grad_total_norm"])
    assert abs(float(learner.optimizer.norm) - tn) / tn < 5e-4
    shapes = synth.router_shapes(len(cc), T=63)
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        numel = int(np.prod(shapes[pname]))
        got = grads[off[k]:off[k] + numel]
        ref = g["grad." + pname]
        scale = max(float(np.abs(ref).max()), 1e-4 * tn)
        assert np.abs(gview(got, g) - ref.reshape(-1)).max() / scale < 1e-3, pname


def test_crnn_train_mode_batchnorm_matches_reference_golden():
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case("crnn_mrn_i2_b4")
    net = synth.build_net(cc, sd, arch="crnn")
    net.train()
    r = net.route_and_combine(img.cuda(), is_train=True, want_logits=True)
    assert rel_err(gview(r["features"].cpu(), g), g["train_features"]) < 1e-4
    assert np.abs(r["gate"].cpu().numpy() - g["train_gate"]).max() < 1e-4
    assert rel_err(gview(r["logits"].cpu(), g), g["train_logits_soft"]) < 1e-4
    sd2 = net.state_dict()
    k = "model.0.model.FeatureExtraction.ConvNet.12.running_mean"
    assert np.abs(sd2[k].cpu().numpy() - g["train_bn1_running_mean_e0"]).max() < 1e-5
    assert rel_err(sd2[k.replace("mean", "var")].cpu().numpy(), g["train_bn1_running_var_e0"]) < 1e-4
    assert int(sd2["model.0.model.FeatureExtraction.ConvNet.12.num_batches_tracked"]) == 1


def test_crnn_bf16_mode_within_north_star_budget():
    """Tensor-core mode (implicit-GEMM convolutions on tcgen05, bf16 LSTM GEMMs): logits within 2e-2 relative of the
    fp32 oracle on random-init weights; gate deviation and expert flips reported."""
    cc, B = (37, 61, 96), 4
    sd = synth.ctor_state_dict(cc, 9, arch="crnn")
    img, tgt, lens, dom = synth.synth_batch(B, cc, 9)
    with torch.no_grad():
        o = O.mrn_forward(sd, len(cc), img, True, True)
        e = O.mrn_forward(sd, len(cc), img, True, False)
    net = synth.build_net(cc, sd, arch="crnn", precision="bf16")
    net.eval()
    out = net(img.cuda(), True, None, True)
    err = rel_err(out["logits"].cpu().numpy(), o["logits"].numpy())
    gate_dev = float((out["index"].cpu() - o["index"]).abs().max())
    ev = net(img.cuda(), True, None, False)
    flips = int((ev["index"].cpu() != e["index"]).sum())
    print("crnn bf16: logits rel err %.2e, gate max abs deviation %.2e, expert flips %d of %d" % (err, gate_dev, flips, B))
    assert err < 2e-2 and gate_dev < 2e-2
    net.train()                                          # batch-statistics BatchNorm in tensor-core mode
    with torch.no_grad():
        ot = O.mrn_forward(sd, len(cc), img, True, True, bn_mode="batch")
    rt = net.route_and_combine(img.cuda(), is_train=True, want_logits=True)
    assert rel_err(rt["logits"].cpu().numpy(), ot["logits"].numpy()) < 2e-2


def test_crnn_persistent_lstm_kernel_matches_per_step_launches(monkeypatch):
    """The persistent BidirectionalLSTM kernel (one 4-CTA-cluster launch per layer, W_hh resident in shared memory; taken
    when the batch is a multiple of 128) against the per-step grouped GEMM + cell kernel path it replaces
    (MRNB_LSTM_SEQ=0) on the same weights and batch: same MMA shapes, k-block order and cell arithmetic, so features and
    logits must agree to bf16 rounding noise at most (identical on the boxes measured); and both stay within the bf16
    budget of the fp32 oracle on a 4-sample slice.  modules/sequence_modeling.py:12-22."""
    import os
    cc, B = (37, 61), 128
    sd = synth.ctor_state_dict(cc, 11, arch="crnn")
    img, tgt, lens, dom = synth.synth_batch(B, cc, 11)
    net = synth.build_net(cc, sd, arch="crnn", precision="bf16")
    net.eval()
    x = img.cuda()
    res = {}
    for mode in ("1", "0"):
        monkeypatch.setenv("MRNB_LSTM_SEQ", mode)
        assert os.environ["MRNB_LSTM_SEQ"] == mode
        r = net.route_and_combine(x, is_train=True, want_logits=True)
        torch.cuda.synchronize()
        res[mode] = (r["features"].float().cpu(), r["logits"].float().cpu())
    monkeypatch.delenv("MRNB_LSTM_SEQ")
    f1, l1 = res["1"]
    f0, l0 = res["0"]
    assert torch.isfinite(f1).all() and torch.isfinite(l1).all()
    fd, ld = float((f1 - f0).abs().max()), float((l1 - l0).abs().max())
    print("persistent LSTM vs per-step: max |d features| %.3e, max |d logits| %.3e" % (fd, ld))
    assert fd <= 2e-2 * float(f0.abs().max()) and ld <= 2e-2 * float(l0.abs().max())
    with torch.no_grad():
        o = O.mrn_forward(sd, len(cc), img[:4], True, True)
    assert rel_err(l1[:4].numpy(), o["logits"].numpy()) < 2e-2


def test_crnn_baseline_config0_two_tasks_batch64():
    """BASELINE.json configs[0]: CRNN-MRN forward + CTC loss, 2 tasks (Chinese + Latin class counts), batch 64,
    synthetic 32x256 crops -- the CUDA path against the CPU oracle on the same inputs."""
    cc, B = synth.MLT17_CLASS_COUNTS[:2], 64
    sd = synth.synth_state_dict(cc, 17, arch="crnn")
    img, tgt, lens, dom = synth.synth_batch(B, cc, 17)
    torch.set_num_threads(max(1, torch.get_num_threads()))
    with torch.no_grad():
        o = O.mrn_forward(sd, 2, img, True, True)
        loss_ref = float(O.ctc_loss_mean(o["logits"], tgt, lens))
        e = O.mrn_forward(sd, 2, img, True, False)
        raw, seqs, conf = O.greedy_decode(e["logits"])
    net = synth.build_net(cc, sd, arch="crnn")
    net.eval()
    r = net.route_and_combine(img.cuda(), is_train=True, want_logits=True, targets=tgt.cuda(), lengths=lens.cuda())
    assert rel_err(r["logits"].cpu().numpy(), o["logits"].numpy()) < 1e-4
    assert float((r["gate"].cpu() - o["index"]).abs().max()) < 1e-4
    learner = synth.build_learner(net, train=False)
    # CTC loss of the soft-routed logits (forward + loss of configs[0])
    from mrn_b200 import ops
    lat = ops.ctc_lattice(r["lpe"], tgt.cuda(), lens.cuda())
    assert abs(float(lat["loss"]) - loss_ref) / abs(loss_ref) < 1e-4
    ev = learner.infer_batch(img.cuda(), "TF", tgt.cuda(), lens.cuda())
    ties = 0
    for b in range(B):
        n = int(ev["lens"][b])
        if ev["ids"][b, :n].cpu().tolist() != seqs[b]:
            ties += 1
    print("configs[0]: decoded sequences differing from the oracle: %d of %d" % (ties, B))
    assert ties == 0


def test_crnn_stage1_step_bf16_tensor_core_router():
    """bf16 mode runs the T = 63 router on tcgen05 through the 64-frame padded problem; the step must stay within the
    bf16 budget of the reference's loss and router gradients (compared on the caller's un-padded arena)."""
    from mrn_b200 import ops
    g, cc, B, seed, sd, img, tgt, lens, dom = golden_case("crnn_mrn_i3_b2")
    net = synth.build_net(cc, sd, arch="crnn", precision="bf16")
    learner = synth.build_learner(net, train=False, total_steps=20000)
    loss_clf, taski = learner.train_step_stage1(img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda())
    assert abs(float(loss_clf) - float(g["loss_clf"])) / abs(float(g["loss_clf"])) < 2e-2
    assert abs(float(taski) - float(g["taski_loss"])) < 2e-2
    n, off = ops.router_param_offsets(len(cc), 63)
    grads = net.router_grad_arena().cpu()
    tn = float(g["grad_total_norm"])
    assert abs(float(learner.optimizer.norm) - tn) / tn < 5e-2
    shapes = synth.router_shapes(len(cc), T=63)
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        numel = int(np.prod(shapes[pname]))
        got = grads[off[k]:off[k] + numel]
        ref = g["grad." + pname]
        scale = max(float(np.abs(ref).max()), 1e-3 * tn)
        assert np.abs(gview(got, g) - ref.reshape(-1)).max() / scale < 8e-2, pname


def test_crnn_fused_lstm_cell_path_batch128():
    """B % 128 == 0 in tensor-core mode switches the recurrence to the GEMM with the LSTM cell fused into its epilogue
    (interleaved gate columns); compare the expert outputs with the fp32 oracle and with the unfused fp32 CUDA path."""
    cc, B = (61,), 128
    sd = synth.ctor_state_dict(cc, 13, arch="crnn")
    img, tgt, lens, dom = synth.synth_batch(B, cc, 13)
    with torch.no_grad():
        feat, pred = O.expert_forward(sd, 0, img)
    net16 = synth.build_net(cc, sd, arch="crnn", precision="bf16")
    net16.eval()
    one16 = net16.model[0](img.cuda())
    assert rel_err(one16["feature"].cpu().numpy(), feat.numpy()) < 2e-2
    assert rel_err(one16["predict"].cpu().numpy(), pred.numpy()) < 2e-2
    net32 = synth.build_net(cc, sd, arch="crnn", precision="fp32")
    net32.eval()
    one32 = net32.model[0](img[:8].cuda())
    assert rel_err(one32["predict"].cpu().numpy(), pred[:8].numpy()) < 1e-4
