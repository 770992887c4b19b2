#!/usr/bin/env python
"""Localise non-finite values / nondeterminism in the bf16 train-mode stage-1 step (bench.py's workload).

    python tools/nan_hunt.py [--batch 256] [--reps 6]

Prints, per stage of the step (experts -> router -> combine -> CTC -> router backward), whether every output is finite,
how far the bf16 tensor-core path is from the fp32 CUDA-core path on the same inputs, and whether repeated launches
on identical inputs give identical results (a mismatch = a race).
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import CLASS_COUNTS, make_opt  # noqa: E402
from mrn_b200 import _lib as L  # noqa: E402
from mrn_b200 import ops, synth  # noqa: E402
from mrn_b200.modules.model import sample_drop_scales  # noqa: E402


def fin(t):
    return bool(torch.isfinite(t).all())


def rel(a, b):
    return float((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-30))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--reps", type=int, default=6)
    ap.add_argument("--init", default="synth", choices=["synth", "ctor"])
    ap.add_argument("--no-fp32", action="store_true")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    B = a.batch
    nets = {}
    for prec in ("bf16", "fp32"):
        if a.init == "synth":
            sd = synth.synth_state_dict(CLASS_COUNTS, 111, arch="svtr")
        else:                                   # ctor: the bf16 net's constructor draws, shared by the fp32 net
            sd = nets["bf16"].state_dict() if prec == "fp32" else None
        torch.manual_seed(111)
        nets[prec] = synth.build_net(CLASS_COUNTS, sd, make_opt(prec, 0, "svtr"), device=dev)
    rates = nets["bf16"].model[0].model.FeatureExtraction.ConvNet.drop_path_rates()
    for mode in ("eval", "train_nodrop", "train_drop"):
        for k in range(2):
            img, tgt, lens, dom = (t.to(dev) for t in synth.synth_batch(B, CLASS_COUNTS, 1000 + k))
            g = torch.Generator(device=dev)
            g.manual_seed(5 + k)
            drop = sample_drop_scales(6, B, rates, dev, generator=g) if mode == "train_drop" else None
            train = mode != "eval"
            outs = []
            for rep in range(a.reps):
                net = nets["bf16"]
                pack = net._cache.get(list(net.model), dev, L.PREC_BF16)
                feats, logits = ops.svtr_experts_forward(pack, img, bn_batch_stats=train, update_running=False,
                                                         drop_scales=drop)
                torch.cuda.synchronize()
                outs.append((feats.clone(), [z.clone() for z in logits]))
            f0, z0 = outs[0]
            line = "[%s batch %d] feats finite=%s |max|=%.3g" % (mode, k, fin(f0), float(f0.abs().max()))
            line += " logits finite=%s" % ([fin(z) for z in z0],)
            nd = [float((o[0] - f0).abs().max()) for o in outs[1:]]
            ndz = [max(float((zz - zz0).abs().max()) for zz, zz0 in zip(o[1], z0)) for o in outs[1:]]
            line += " | rerun max|d feats|=%s max|d logits|=%s" % (["%.2g" % v for v in nd], ["%.2g" % v for v in ndz])
            print(line, flush=True)
            if not a.no_fp32 and k == 0:
                net32 = nets["fp32"]
                pack32 = net32._cache.get(list(net32.model), dev, L.PREC_FP32)
                f32, z32 = ops.svtr_experts_forward(pack32, img, bn_batch_stats=train, update_running=False, drop_scales=drop)
                torch.cuda.synchronize()
                print("    vs fp32 path: feats rel %.3g per-expert %s ; logits rel %s" % (
                    rel(f0, f32), ["%.3g" % rel(f0[:, i], f32[:, i]) for i in range(6)],
                    ["%.3g" % rel(x, y) for x, y in zip(z0, z32)]), flush=True)
                # worst sample
                d = (f0 - f32).abs().amax(dim=(2, 3))
                bi = int(d.max(dim=1).values.argmax())
                print("    worst sample %d per-expert abs err %s (|f32| max %.3g)" % (bi, ["%.3g" % float(v) for v in d[bi]],
                                                                                        float(f32.abs().max())), flush=True)
            # router + combine + ctc on these features
            net = nets["bf16"]
            arena = net.router_arena(dev)
            for rprec, name in ((L.PREC_BF16, "bf16"), (L.PREC_FP32, "fp32")):
                _, scores, gate, index = ops.router_forward(arena, f0, net._rws, with_backward=True, prec=rprec, want_out=False)
                r = ops.gate_combine(z0, gate, tgt, lens, want_logits=False, want_E=True)
                c = ops.ctc_lattice(r["lpe"], tgt, lens, r["zlab"], r["E"], grad_scale=15.0 / B, want_dgate=True)
                grads = torch.zeros_like(arena)
                taski = ops.router_backward(arena, f0, gate, c["dgate"], dom, grads, net._rws, prec=rprec)
                torch.cuda.synchronize()
                print("    router[%s]: scores fin=%s |max|=%.3g gate fin=%s min=%.3g max=%.3g lse fin=%s E fin=%s lpe fin=%s nll fin=%s "
                      "loss=%.5f dgate fin=%s taski=%.5f grads fin=%s |g|=%.4g" % (
                          name, fin(scores), float(scores.abs().max()), fin(gate), float(gate.min()), float(gate.max()), fin(r["lse"]),
                          fin(r["E"]), fin(r["lpe"]), fin(c["nll"]), float(c["loss"]), fin(c["dgate"]), float(taski), fin(grads),
                          float(grads.norm())), flush=True)


    # ---- the learner's step, eager then graphed, losses of every step
    for graphed in (False, True):
        opt = make_opt("bf16", 0, "svtr")
        net = synth.build_net(CLASS_COUNTS, nets["bf16"].state_dict(), opt, device=dev)
        learner = synth.build_learner(net, total_steps=opt.num_iter * 2, schedule="super")
        losses = []
        for k in range(10):
            img, tgt, lens, dom = (t.to(dev) for t in synth.synth_batch(B, CLASS_COUNTS, 1000 + k % 4))
            fn = learner.train_step_stage1_graphed if graphed else learner.train_step_stage1
            l1, l2 = fn(img, tgt, lens, dom)
            losses.append((round(float(l1), 4), round(float(l2), 4), round(float(learner.optimizer.norm), 4)))
        print("learner steps graphed=%s: (loss_clf, taski, grad norm) %s" % (graphed, losses), flush=True)


if __name__ == "__main__":
    main()
