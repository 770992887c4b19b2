"""CTC prefix beam search on the device (mrn_b200/csrc/ctc_beam.cu): the per-frame top-K pass against an fp64 torch
statement of the same selection, the beam kernel against the fp64 oracle (oracle/ctc_beam_oracle.py) and against exact
labeling probabilities, and MRN.infer_batch(decode="beam") end to end.  Both kernels give every warp one row / one
sample and are not persistent, so there is no multi-item walk to cover."""
import argparse

import pytest
import torch

from oracle import ctc_beam_oracle as BO
from oracle import mrn_oracle as O
from oracle import synth
from conftest import load_golden

pytestmark = pytest.mark.gpu
MLT17 = (1899, 2224, 3844, 4968, 5041, 5153)


def _ops():
    from mrn_b200 import ops
    return ops


def _table(cc, B, T, gen, scale=3.0, keep=None):
    """Ragged expert logits [B,T,C_i] in 16-byte aligned rows; rows of (expert, sample) pairs outside `keep` are NaN,
    so that a kernel reading an expert whose gate is 0 shows."""
    ops = _ops()
    out = []
    for i, c in enumerate(cc):
        buf = torch.full((B, T, ops.round_up(c, 4)), float("nan"), device="cuda")
        z = torch.randn(B, T, c, device="cuda", generator=gen) * scale
        rows = torch.ones(B, dtype=torch.bool, device="cuda") if keep is None else keep[:, i]
        buf[:, :, :c][rows] = z[rows]
        out.append(buf[:, :, :c])
    return out


def _nan_outs(B, T, K):
    return (torch.full((B, T, K), -2, dtype=torch.int32, device="cuda"), torch.full((B, T, K), float("nan"), device="cuda"),
            torch.full((B, T), float("nan"), device="cuda"))


def _check_topk(zs, gate, ref_logits, K):
    """Kernel top-K vs the fp64 selection on the combine's own fp32 values (`ref_logits`)."""
    ops = _ops()
    B, T, _ = zs[0].shape
    r = ops.gate_combine(zs, gate, want_decode=True)
    ids, lp, blank = ops.ctc_topk(zs, gate, r["lse"], K, out=_nan_outs(B, T, K))
    rid, rlp, rblank = BO.ctc_topk(ref_logits, K)
    assert not bool((ids == -2).any()) and not bool(lp.isnan().any()) and not bool(blank.isnan().any())   # all written
    bad = (ids.long() != rid).any(-1)
    assert not bool(bad.any()), "top_ids differ at (sample, frame) %s" % (bad.nonzero()[:5].tolist(),)
    fin = rlp > float("-inf")
    assert torch.equal(lp.isinf(), ~fin)
    assert float((lp.double()[fin] - rlp[fin]).abs().max()) < 1e-5
    assert float((blank.double() - rblank).abs().max()) < 1e-5
    amax = r["amax"].long()
    nz = amax != 0
    assert torch.equal(ids[..., 0].long()[nz], amax[nz])          # top-1 is the combine's arg-max bit for bit
    return ids, lp, blank


@pytest.mark.parametrize("C,K", [(50, 16), (50, 32), (10, 16)])
def test_topk_single_expert(C, K):
    gen = torch.Generator(device="cuda").manual_seed(C + K)
    B, T = 3, 63
    zs = _table((C,), B, T, gen)
    ids, _, _ = _check_topk(zs, torch.ones(B, 1, device="cuda"), zs[0].double(), K)
    if K > C - 1:
        assert bool((ids[..., C - 1:] == -1).all())


def test_topk_hard_route_mlt17_with_ones_plateau():
    """B = 256 on the MLT17 class counts, one-hot gate; the other experts' rows are NaN (never read).  Every 5th sample
    has all real logits < 1, so its top-K is the first K columns of the ones plateau: C_i, C_i + 1, ..."""
    gen = torch.Generator(device="cuda").manual_seed(17)
    B, T, K, I = 256, 64, 16, len(MLT17)
    index = torch.randint(0, I, (B,), device="cuda", generator=gen)
    gate = torch.nn.functional.one_hot(index, I).float()
    zs = _table(MLT17, B, T, gen, keep=gate.bool())
    plateau = torch.arange(B, device="cuda") % 5 == 0
    for z in zs:
        z[plateau] = -z[plateau].abs() - 0.01
    ref = torch.stack([torch.nn.functional.pad(zs[int(index[b])][b], (0, MLT17[-1] - MLT17[int(index[b])]), value=1.0)
                       for b in range(B)])
    ids, _, _ = _check_topk(zs, gate, ref.double(), K)
    for b in plateau.nonzero().flatten().tolist():
        Ci = MLT17[int(index[b])]
        if Ci + K <= MLT17[-1]:
            want = torch.arange(Ci, Ci + K, device="cuda", dtype=torch.int32).expand(T, K)
            assert torch.equal(ids[b], want), b


@pytest.mark.parametrize("cc,B", [((37, 61, 96), 5), (MLT17, 4)])
def test_topk_soft_gate(cc, B):
    ops = _ops()
    gen = torch.Generator(device="cuda").manual_seed(len(cc))
    T, K = 64, 16
    zs = _table(cc, B, T, gen)
    gate = torch.softmax(torch.randn(B, len(cc), device="cuda", generator=gen) * 2, -1)
    r = ops.gate_combine(zs, gate, want_logits=True)
    ref64 = O.combine_soft([z.double().cpu() for z in zs], gate.double().cpu())
    assert float((r["logits"].double().cpu() - ref64).abs().max()) < 1e-6 * float(ref64.abs().max())
    _check_topk(zs, gate, r["logits"].double(), K)


def test_beam_tiny_case_is_exact():
    """T = 4, C = 3, K = C - 1 and W = 32 >= the 31 labelings: nothing is pruned, so every listed score is the exact
    log p(labeling | x)."""
    ops = _ops()
    gen = torch.Generator(device="cuda").manual_seed(4)
    B, T, C, W = 16, 4, 3, 32
    zs = _table((C,), B, T, gen, scale=1.5)
    gate = torch.ones(B, 1, device="cuda")
    r = ops.gate_combine(zs, gate)
    top = ops.ctc_topk(zs, gate, r["lse"], C - 1)
    ids, lens, scores = ops.ctc_beam_search(*top, W, W)
    for b in range(B):
        exact = {k: v for k, v in BO.ctc_labeling_distribution(zs[0][b].double().cpu()).items() if v > float("-inf")}
        got = []
        for n in range(W):
            if int(lens[b, n]) == 0 and float(scores[b, n]) == float("-inf"):
                continue
            got.append((tuple(ids[b, n, :int(lens[b, n])].tolist()), float(scores[b, n])))
        assert len(got) == len(exact) and len({g[0] for g in got}) == len(got)
        for lab, s in got:
            assert abs(s - exact[lab]) < 1e-5, (b, lab)
        assert got[0][0] == max(exact, key=exact.get)
        assert all(bool((ids[b, n, int(lens[b, n]):] == -1).all()) for n in range(W))


@pytest.mark.parametrize("T", [64, 63])
def test_beam_full_size_matches_oracle(T):
    """B = 256, W = 16, K = 16 on peaked CTC-like frames (C = 200); the fp64 oracle runs on the same fp32 candidates
    for 16 samples spread over the batch.  A sample counts as a near-tie for the beam sets when, at ANY frame, the W-th
    kept and the best dropped candidate are within 1e-4 (fp32 rounding may flip that choice); wide logits (scale 6)
    keep the candidate scores at the cut sparse enough for that to be rare."""
    ops = _ops()
    gen = torch.Generator(device="cuda").manual_seed(T)
    B, C, K, W = 256, 200, 16, 16
    z = torch.randn(B, T, C, device="cuda", generator=gen) * 6.0
    path = torch.randint(0, C, (B, T), device="cuda", generator=gen)
    path[torch.rand(B, T, device="cuda", generator=gen) < 0.4] = 0
    z.scatter_add_(2, path[..., None], torch.full((B, T, 1), 10.0, device="cuda"))
    zs = [z.contiguous()]
    gate = torch.ones(B, 1, device="cuda")
    top = ops.ctc_topk(zs, gate, ops.gate_combine(zs, gate)["lse"], K)
    outs = (torch.full((B, W, T), -2, dtype=torch.int32, device="cuda"), torch.full((B, W), -2, dtype=torch.int32, device="cuda"),
            torch.full((B, W), float("nan"), device="cuda"))
    ids, lens, scores = ops.ctc_beam_search(*top, W, W, out=outs)
    assert not bool((ids == -2).any()) and not bool((lens == -2).any()) and not bool(scores.isnan().any())
    tid, tlp, tbl = (t.cpu() for t in top)
    ids, lens, scores = ids.cpu(), lens.cpu(), scores.cpu()
    samples = list(range(0, B, B // 16))
    tie_best = tie_set = 0
    for b in samples:
        st = {}
        ref = BO.ctc_prefix_beam_search(tid[b].tolist(), tlp[b].double().tolist(), tbl[b].double().tolist(), W, W, st)
        got = [(tuple(ids[b, n, :int(lens[b, n])].tolist()), float(scores[b, n])) for n in range(W)]
        assert all(bool((ids[b, n, int(lens[b, n]):] == -1).all()) for n in range(W))
        if ref[0][1] - ref[1][1] > 1e-4:
            assert got[0][0] == ref[0][0], b
        else:
            tie_best += 1
        if st["prune_margin"] > 1e-4:
            assert {g[0] for g in got} == {r[0] for r in ref}, b
            want = dict(ref)
            for lab, s in got:
                assert abs(s - want[lab]) < 1e-4, (b, lab, s, want[lab])
        else:
            tie_set += 1
    print("near-ties excluded: %d of %d samples from the best-beam check, %d from the beam-set check"
          % (tie_best, len(samples), tie_set))
    assert tie_best <= len(samples) // 4 and tie_set <= len(samples) // 4


def test_argument_errors_raise_with_the_kernel_message():
    ops = _ops()
    B, T = 2, 8
    zs = [torch.zeros(B, T, 12, device="cuda")]
    gate = torch.ones(B, 1, device="cuda")
    lse = torch.zeros(B, T, device="cuda")
    with pytest.raises(RuntimeError, match="K = 0 out of range"):
        ops.ctc_topk(zs, gate, lse, 0)
    top = ops.ctc_topk(zs, gate, lse, 4)
    with pytest.raises(RuntimeError, match="beam width 33 out of range"):
        ops.ctc_beam_search(*top, 33, 1)
    with pytest.raises(RuntimeError, match="n_best = 9 out of range"):
        ops.ctc_beam_search(*top, 8, 9)


def _learner(arch, name):
    from mrn_b200.il_modules.mrn import MRN, RankLocal
    from mrn_b200.modules.model import MRNNet
    g = load_golden(name)
    cc = tuple(int(c) for c in g["class_counts"])
    B, seed = int(g["B"]), int(g["seed"])
    opt = argparse.Namespace(Transformation="None", FeatureExtraction="SVTR" if arch == "svtr" else "VGG",
                             SequenceModeling="None" if arch == "svtr" else "BiLSTM", Prediction="CTC", num_fiducial=20,
                             input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256, batch_max_length=25,
                             lr=5e-4, num_iter=10000, grad_clip=5, exp_name="test", precision="fp32", drop_path=False,
                             lan_list=["a", "b", "c", "d", "e", "f"], val_interval=5000, start_task=0, optimizer="adam",
                             schedule="super")
    net = MRNNet(opt)
    for c in cc:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    net.load_state_dict(synth.synth_state_dict(cc, seed, arch=arch), strict=True)
    learner = MRN(opt)
    learner.model = RankLocal(net.cuda())
    learner.model.eval()
    return learner, cc, B


@pytest.mark.parametrize("arch,name", [("svtr", "svtr_mrn_i3_b3"), ("crnn", "crnn_mrn_i2_b4")])
@pytest.mark.parametrize("route", ["TF", "FF"])
def test_infer_batch_beam_decode(arch, name, route):
    learner, cc, B = _learner(arch, name)
    W = 8
    for k in range(2):
        x = synth.synth_batch(B, cc, 70 + k)[0].cuda()
        plain = {n: v.clone() for n, v in learner.infer_batch(x, route).items() if torch.is_tensor(v)}
        greedy = learner.infer_batch(x, route, decode="greedy")
        for n in plain:
            assert torch.equal(greedy[n], plain[n]), n
        eager = {n: v.clone() for n, v in learner.infer_batch(x, route, decode="beam", beam_width=W, n_best=W).items()
                 if torch.is_tensor(v)}
        rep = learner.infer_batch_graphed(x, route, decode="beam", beam_width=W, n_best=W)
        torch.cuda.synchronize()
        for n in eager:
            assert torch.equal(rep[n], eager[n]), n
        sc = eager["nbest_scores"]
        assert bool((sc[:, :1] >= sc).all())
        assert torch.equal(eager["ids"], eager["nbest_ids"][:, 0]) and torch.equal(eager["lens"], eager["nbest_lens"][:, 0])
        assert torch.equal(eager["conf"], sc[:, 0].exp())
        one = learner.infer_batch(x, route, decode="beam", beam_width=W)
        assert "nbest_ids" not in one and torch.equal(one["ids"], eager["ids"])
    assert len(learner._infer_graphs) == 1
