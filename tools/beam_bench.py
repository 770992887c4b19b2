"""CTC prefix beam search on the device: kernel times and the cost of beam decoding in the inference step.

    python tools/beam_bench.py [--batch 256] [--iters 50]

Prints one JSON line.  Setup: MLT17 class counts (union charset 5153), hard route (one-hot gate over 6 experts),
K = 16 candidates per frame, T = 64 (SVTR) and 63 (CRNN).
  topk      ctc_topk time and its rate on the algorithmic bytes: the routed expert's rows (B*T*C_sel*4, the ones
            plateau past C_sel is not read) + lse + the outputs.  About 250 MB per pass at B = 256, twice the 126 MB L2,
            so the rows come from HBM.  Share of the 6.54 TB/s HBM rate the project measured on its B200.
  beam      ctc_beam_search time for W in {1, 4, 8, 16, 32} on those candidates.
  infer     MRN.infer_batch_graphed samples/s, greedy vs beam (W = 8, K = 16), SVTR bf16, eval-mode experts, the two
            modes alternated in rounds in the same process; median over rounds.
All times are CUDA events over warmed-up launches.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from mrn_b200 import ops, synth                      # noqa: E402

CLASS_COUNTS = synth.MLT17_CLASS_COUNTS
HBM_PEAK = 6.54e12                                   # bytes/s, measured by the project on a B200 (DESIGN.md §4)
K = 16
WIDTHS = (1, 4, 8, 16, 32)


def card():
    name = torch.cuda.get_device_name()
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=power.limit",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(fn, iters, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernels(B, T, iters):
    gen = torch.Generator(device="cuda").manual_seed(T)
    I = len(CLASS_COUNTS)
    index = torch.randint(0, I, (B,), device="cuda", generator=gen)
    gate = torch.nn.functional.one_hot(index, I).float()
    zs = []
    for c in CLASS_COUNTS:
        buf = torch.randn(B, T, ops.round_up(c, 4), device="cuda", generator=gen) * 3.0
        zs.append(buf[:, :, :c])
    lse = ops.gate_combine(zs, gate)["lse"]
    outs = (torch.empty(B, T, K, dtype=torch.int32, device="cuda"), torch.empty(B, T, K, device="cuda"),
            torch.empty(B, T, device="cuda"))
    ms = timed(lambda: ops.ctc_topk(zs, gate, lse, K, out=outs), iters)
    c_sel = torch.tensor(CLASS_COUNTS, device="cuda")[index].double()
    nbytes = float(T * (c_sel * 4).sum()) + B * T * (4 + K * 8 + 4)
    res = {"T": T, "topk_ms": round(ms, 4), "topk_bytes": int(nbytes), "topk_TBps": round(nbytes / ms / 1e9, 3),
           "topk_share_of_hbm_peak": round(nbytes / ms / 1e9 / (HBM_PEAK / 1e12), 3), "beam_ms": {}}
    for W in WIDTHS:
        bo = (torch.empty(B, 1, T, dtype=torch.int32, device="cuda"), torch.empty(B, 1, dtype=torch.int32, device="cuda"),
              torch.empty(B, 1, device="cuda"))
        res["beam_ms"][W] = round(timed(lambda: ops.ctc_beam_search(*outs, W, 1, out=bo), iters), 4)
    return res


def infer(B, rounds, steps):
    from mrn_b200.il_modules.mrn import MRN, RankLocal
    from mrn_b200.modules.model import MRNNet
    opt = argparse.Namespace(Transformation="None", FeatureExtraction="SVTR", SequenceModeling="None", Prediction="CTC",
                             num_fiducial=20, input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256,
                             batch_max_length=25, lr=5e-4, num_iter=10000, grad_clip=5, exp_name="beam_bench",
                             precision="bf16", drop_path=True, expert_chunk=0,
                             lan_list=["Chinese", "Latin", "Japanese", "Korean", "Arabic", "Bangla"], val_interval=5000,
                             start_task=0, optimizer="adam", schedule="super")
    net = MRNNet(opt)
    for c in CLASS_COUNTS:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    net.load_state_dict(synth.synth_state_dict(CLASS_COUNTS, 111), strict=True)
    learner = MRN(opt)
    learner.model = RankLocal(net.cuda())
    learner.model.eval()
    imgs = [synth.synth_batch(B, CLASS_COUNTS, 2000 + k)[0].cuda() for k in range(2)]
    modes = {"greedy": dict(decode="greedy"), "beam_w8": dict(decode="beam", beam_width=8, beam_topk=K)}
    ms = {m: [] for m in modes}
    for r in range(rounds):
        for m, kw in modes.items():
            ms[m].append(timed(lambda: learner.infer_batch_graphed(imgs[0], "TF", **kw), steps, warmup=3 if r == 0 else 1))
    out = {m: {"ms_per_batch": round(statistics.median(v), 3), "samples_per_s": round(B * 1000.0 / statistics.median(v), 1)}
           for m, v in ms.items()}
    out["beam_over_greedy"] = round(out["beam_w8"]["ms_per_batch"] / out["greedy"]["ms_per_batch"], 4)
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("beam_bench needs a CUDA device")
    name, power = card()
    res = {"gpu": name, "power_limit": power, "batch": a.batch, "K": K,
           "kernels": [kernels(a.batch, T, a.iters) for T in (64, 63)],
           "infer": infer(a.batch, a.rounds, 10)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
