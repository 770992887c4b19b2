"""Image gradients through the experts (opt.autograd with image.requires_grad_()), timed with CUDA events in one run:
I = 6 experts with the MLT17 class counts, B = 256, bf16 tensor-core mode, experts in .eval(), the reference's stage-1
loss (15 * CTC + CE on the gate) forward + backward through MRNNet's soft route.

  frozen             every expert frozen, image without grad (the grouped expert forward, router backward only)
  frozen_image       every expert frozen, image with grad (six training packs, input-only backwards)
  newest             the newest expert trainable, image without grad (its training pack + the grouped forward)
  newest_image       the newest expert trainable, image with grad (one full backward + five input-only backwards)

for SVTR and CRNN, the four variants alternating per repeat.  frozen_image against newest_image shows what the
input-only backward saves per frozen expert (newest_image - frozen_image = one full backward less one input-only one).
Then the conv0 input-gradient kernels alone (mrnb_{svtr,crnn}_conv0_dimage) with the bytes the algorithm moves -- the
gradient at conv0's output read once, the image gradient written once -- over their time.  Each timed window is `--iters`
calls after `--warmup` untimed ones; the spread is the min / median / max over `--repeats` windows.  The GPU's name and
power limit are read in the same run.  The result is one JSON, written to --out when given
(profiles/input_grad_bench.json is such a file), else printed as the last line.

    python tools/input_grad_bench.py [--batch 256] [--iters 5] [--warmup 2] [--repeats 3] [--out results.json]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from joint_bench import _power_limit, _spread, _window  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None, help="path of the JSON result (default: print it)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("input_grad_bench needs a CUDA device: there is nothing to measure without one")
    from mrn_b200 import ops, synth
    cc, B = synth.MLT17_CLASS_COUNTS, args.batch
    I = len(cc)
    res = dict(gpu=torch.cuda.get_device_name(), power_limit=_power_limit(), B=B, I=I, class_counts=list(cc),
               precision="bf16", iters=args.iters, warmup=args.warmup, repeats=args.repeats, step_ms={}, peak_mem_GB={})
    for arch in ("svtr", "crnn"):
        sd = synth.ctor_state_dict(cc, 11, arch=arch)
        img, tgt, lens, dom = synth.synth_batch(B, cc, 11)
        x, t, l, d = img.cuda(), tgt.cuda(), lens.cuda(), dom.cuda()
        net = synth.build_net(cc, sd, arch=arch, precision="bf16", autograd=True, autograd_experts=True).eval()
        variants = {"frozen": ((), False), "frozen_image": ((), True), "newest": ((I - 1,), False),
                    "newest_image": ((I - 1,), True)}

        def step(trainable, image_grad):
            for e, m in enumerate(net.model):
                for p in m.parameters():
                    p.requires_grad = e in trainable
                    p.grad = None
            for p in net.router_parameters():
                p.grad = None
            xi = x.detach().requires_grad_(image_grad)
            out = net(xi, True, None, True)
            lp = out["logits"].log_softmax(2).permute(1, 0, 2)
            T = lp.shape[0]
            loss = 15 * F.ctc_loss(lp, t, torch.full((B,), T, dtype=torch.long, device="cuda"), l.long(), blank=0,
                                   reduction="mean", zero_infinity=True) + F.cross_entropy(out["index"], d)
            loss.backward()
            assert (xi.grad is not None) == image_grad

        times = {k: [] for k in variants}
        peak = {}
        for k, v in variants.items():
            torch.cuda.reset_peak_memory_stats()
            _window(lambda: step(*v), args.warmup)
            peak[k] = torch.cuda.max_memory_allocated() / 1e9
        for _ in range(args.repeats):
            for k, v in variants.items():
                times[k].append(_window(lambda: step(*v), args.iters))
        res["step_ms"][arch] = {k: _spread(v) for k, v in times.items()}
        res["peak_mem_GB"][arch] = peak
        print(arch, json.dumps(res["step_ms"][arch]), "peak GB", json.dumps(peak))
        del net
        torch.cuda.empty_cache()

    # the conv0 input-gradient kernels alone
    gen = torch.Generator(device="cuda").manual_seed(5)
    kern = {}
    for arch, dshape, wshape in (("svtr", (B, 16, 128, 32), (32, 4, 3, 3)), ("crnn", (B, 32, 256, 64), (64, 3, 3, 4))):
        dd = torch.randn(*dshape, device="cuda", generator=gen)
        w = torch.randn(*wshape, device="cuda", generator=gen) * 0.2
        out = torch.empty(B, 4, 32, 256, device="cuda")
        fn = lambda: ops.conv0_dimage(arch, dd, w, out=out)      # noqa: E731
        nbytes = 4 * (dd.numel() + out.numel() + w.numel())
        fma = B * 4 * 32 * 256 * (9 * wshape[0] if arch == "crnn" else 9 * wshape[0] / 4)   # taps x channels per pixel
        _window(fn, 5)
        ms = [_window(fn, 50) for _ in range(args.repeats)]
        med = statistics.median(ms)
        kern[arch] = dict(ms=_spread(ms), bytes=nbytes, GBps=nbytes / med / 1e6, hbm_share=nbytes / med / 1e6 / 7700.0,
                          fp32_fma=fma, GFMAps=fma / med / 1e6)
        print("conv0_dimage", arch, json.dumps(kern[arch]))
    res["conv0_dimage"] = kern
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
