"""Stage-1 router step three ways, alternating in one run, timed with CUDA events: SVTR-MRN, I = 6 experts with the
MLT17 class counts, bf16 tensor-core mode, B = 256, experts frozen in .eval().

  (a) fused   MRN.train_step_stage1: one device step, the CTC gradient contracted in place, fused clip + Adam;
  (b) torch   the reference's loop over the mirror with opt.autograd=True (il_modules/mrn.py:338-367): forward with the
              combined logits, log_softmax, F.ctc_loss, CE on the gate, backward, clip_grad_norm_, torch.optim.Adam;
  (c) combine mrnb_gate_combine_backward alone on the same expert logits: bytes moved (sum C_i + C) * T * 4 per sample,
              over the kernel time, and that rate's share of a device-to-device copy measured in the same run.

(b) materialises the dense logits and runs the library CTC, so it is expected to be slower than (a); the ratio is
reported, no target is set.  Prints one JSON line with the GPU name and power limit read in the same run.

    python tools/autograd_bench.py [--batch 256] [--iters 20] [--warmup 3]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402


def _opt(autograd):
    return argparse.Namespace(Transformation="None", FeatureExtraction="SVTR", SequenceModeling="None", Prediction="CTC",
                              num_fiducial=20, input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256,
                              batch_max_length=25, lr=5e-4, num_iter=10000, grad_clip=5, exp_name="bench", precision="bf16",
                              drop_path=False, lan_list=list("abcdef"), val_interval=5000, start_task=0, autograd=autograd)


def _net(cc, sd, autograd):
    from mrn_b200.modules.model import MRNNet
    opt = _opt(autograd)
    net = MRNNet(opt)
    for c in cc:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    net.load_state_dict(sd, strict=True)
    net = net.cuda().eval()
    for p in net.model.parameters():
        p.requires_grad = False
    return net


def _timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("autograd_bench.py needs a CUDA device")
    from mrn_b200 import ops, synth
    from mrn_b200.il_modules.mrn import MRN, RankLocal, FusedAdam
    cc, B, seed = synth.MLT17_CLASS_COUNTS, args.batch, 3
    sd = synth.ctor_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    x, t, l, d = img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda()

    fused = _net(cc, sd, False)
    learner = MRN(fused.opt)
    learner.model = RankLocal(fused)
    learner.optimizer = FusedAdam(fused, 5e-4, 10 ** 6, grad_clip=5, schedule="const")

    net = _net(cc, sd, True)
    params = net.router_parameters()
    adam = torch.optim.Adam(params, lr=5e-4)
    T = net.patch
    sizes = torch.full((B,), T, dtype=torch.long, device="cuda")

    def torch_step():
        adam.zero_grad(set_to_none=True)
        out = net(x, True, None, True)
        loss = 15 * F.ctc_loss(out["logits"].log_softmax(2).permute(1, 0, 2), t, sizes, l.long(), zero_infinity=True) \
            + F.cross_entropy(out["index"], d)
        loss.backward()
        torch.nn.utils.clip_grad_norm_(params, 5)
        adam.step()

    with torch.no_grad():
        r = net.route_and_combine(x, is_train=True, want_logits=False)
    z = r["expert_logits"]
    C = cc[-1]
    dY = torch.randn(B, T, ops.round_up(C, 4), device="cuda")[:, :, :C]
    dgate = torch.empty(B, len(cc), device="cuda")
    comb_bytes = 4.0 * B * T * (sum(cc) + C)

    copy_src = torch.empty(int(comb_bytes) // 4, device="cuda")
    copy_dst = torch.empty_like(copy_src)

    arms = dict(fused=lambda: learner.train_step_stage1(x, t, l, d), torch=torch_step,
                combine=lambda: ops.gate_combine_backward(z, dY, out=dgate), copy=lambda: copy_dst.copy_(copy_src))
    for _ in range(args.warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    ms = {k: [] for k in arms}
    for _ in range(args.iters):
        for k, fn in arms.items():
            ms[k].append(_timed(fn))
    med = {k: sorted(v)[len(v) // 2] for k, v in ms.items()}
    copy_bps = 2 * comb_bytes / (med["copy"] * 1e-3)
    comb_bps = comb_bytes / (med["combine"] * 1e-3)
    print(json.dumps(dict(
        gpu=torch.cuda.get_device_name(), power_limit=_power_limit(), batch=B, experts=len(cc), precision="bf16",
        iters=args.iters, fused_step_ms=round(med["fused"], 3), torch_loop_ms=round(med["torch"], 3),
        torch_over_fused=round(med["torch"] / med["fused"], 2), combine_backward_ms=round(med["combine"], 4),
        combine_backward_bytes=comb_bytes, combine_backward_TBps=round(comb_bps / 1e12, 3),
        d2d_copy_TBps=round(copy_bps / 1e12, 3), combine_share_of_copy=round(comb_bps / copy_bps, 3),
        combine_share_of_6p54=round(comb_bps / 6.54e12, 3))))


if __name__ == "__main__":
    main()
