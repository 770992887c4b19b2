"""Joint expert + router training through autograd (opt.autograd_experts), timed with CUDA events in one run:
I = 6 experts with the MLT17 class counts, B = 256, bf16 tensor-core mode, experts in .eval(), the reference's
stage-1 loss (15 * CTC + CE on the gate) forward + backward.

  frozen   every expert frozen (today's routed autograd: grouped expert forward, router backward, no dx)
  newest   the newest expert trainable (its training pack + the frozen five through the grouped forward)
  all      all six trainable (six training packs)

for SVTR and CRNN, the three variants alternating per repeat; then mrnb_gate_combine_backward_experts alone (dz for the
newest expert and for all six) with the bytes the algorithm moves -- dY and every z_i read once, each requested dz_i
written once -- over its time.  Each timed window is `--iters` calls after `--warmup` untimed ones; the spread is the
min / median / max over `--repeats` windows.  The per-expert training workspace (mrnb_*_train_workspace_bytes) times
the trainable count is printed, with the GPU's name and power limit read in the same run.  The full result is one JSON,
written to --out when given (profiles/joint_autograd_bench.json is such a file), else printed as the last line.

    python tools/joint_bench.py [--batch 256] [--iters 5] [--warmup 2] [--repeats 3] [--out results.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402


def _power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        return out.stdout.strip() or None
    except (OSError, subprocess.SubprocessError):
        return None


def _window(fn, iters):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / iters


def _spread(v):
    return dict(min=min(v), median=statistics.median(v), max=max(v))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None, help="path of the JSON result (default: print it)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("joint_bench needs a CUDA device: there is nothing to measure without one")
    from mrn_b200 import ops, synth
    from mrn_b200 import _lib as L
    cc, B = synth.MLT17_CLASS_COUNTS, args.batch
    I = len(cc)
    res = dict(gpu=torch.cuda.get_device_name(), power_limit=_power_limit(), B=B, I=I, class_counts=list(cc),
               precision="bf16", iters=args.iters, warmup=args.warmup, repeats=args.repeats, step_ms={}, workspace={})
    lib = L.load()
    for arch in ("svtr", "crnn"):
        sd = synth.ctor_state_dict(cc, 11, arch=arch)
        img, tgt, lens, dom = synth.synth_batch(B, cc, 11)
        x, t, l, d = img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda()
        net = synth.build_net(cc, sd, arch=arch, precision="bf16", autograd=True, autograd_experts=True).eval()
        variants = {"frozen": (), "newest": (I - 1,), "all": tuple(range(I))}

        def step(trainable):
            for e, m in enumerate(net.model):
                for p in m.parameters():
                    p.requires_grad = e in trainable
                    p.grad = None
            for p in net.router_parameters():
                p.grad = None
            out = net(x, True, None, True)
            lp = out["logits"].log_softmax(2).permute(1, 0, 2)
            T = lp.shape[0]
            loss = 15 * F.ctc_loss(lp, t, torch.full((B,), T, dtype=torch.long, device="cuda"), l.long(), blank=0,
                                   reduction="mean", zero_infinity=True) + F.cross_entropy(out["index"], d)
            loss.backward()

        times = {k: [] for k in variants}
        for k, tr in variants.items():
            _window(lambda: step(tr), args.warmup)
        for _ in range(args.repeats):
            for k, tr in variants.items():
                times[k].append(_window(lambda: step(tr), args.iters))
        res["step_ms"][arch] = {k: _spread(v) for k, v in times.items()}
        fn = lib.mrnb_svtr_train_workspace_bytes if arch == "svtr" else lib.mrnb_crnn_train_workspace_bytes
        per = [int(fn(B, c, L.PREC_BF16)) for c in cc]
        res["workspace"][arch] = dict(per_expert_bytes=per, newest_bytes=per[-1], all_bytes=sum(per))
        print(arch, json.dumps(res["step_ms"][arch]), "workspace GB: newest %.2f, all %.2f" % (per[-1] / 1e9, sum(per) / 1e9))
        del net
        torch.cuda.empty_cache()

    # combine backward with per-expert logit gradients, alone
    T, C = 64, cc[-1]
    gen = torch.Generator(device="cuda").manual_seed(3)

    def padded(c):
        return torch.randn(B, T, ops.round_up(c, 4), device="cuda", generator=gen)[:, :, :c]
    z = [padded(c) for c in cc]
    dY = padded(C)
    gate = torch.softmax(torch.randn(B, I, device="cuda", generator=gen), -1)
    comb = {}
    for name, want in (("none", ()), ("newest", (I - 1,)), ("all", tuple(range(I)))):
        dz = [padded(c) if i in want else None for i, c in enumerate(cc)]
        if want:
            fn = lambda: ops.gate_combine_backward_experts(z, dY, gate, dz)   # noqa: E731
        else:
            fn = lambda: ops.gate_combine_backward(z, dY)                       # noqa: E731
        nbytes = 4 * B * T * (C + sum(cc) + sum(cc[i] for i in want))
        _window(fn, 5)
        ms = [_window(fn, 50) for _ in range(args.repeats)]
        comb[name] = dict(ms=_spread(ms), bytes=nbytes, GBps=nbytes / statistics.median(ms) / 1e6,
                          hbm_share=nbytes / statistics.median(ms) / 1e6 / 7700.0)
        print("combine backward, dz", name, json.dumps(comb[name]))
    res["combine_backward"] = comb
    res["power_limit_after"] = _power_limit()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps(dict(gpu=res["gpu"], power_limit=res["power_limit"], out=args.out)))
    else:
        print(json.dumps(res))


if __name__ == "__main__":
    main()
