#!/usr/bin/env python
"""The bench.py headline step (SVTR-MRN, 6 experts, B = 256, bf16, train-mode experts) between cudaProfilerStart / Stop,
eager launches, for ncu:

    ncu --profile-from-start off --metrics gpu__time_duration.sum,dram__bytes_read.sum,dram__bytes_write.sum \
        --clock-control none --csv --log-file gpurun_out/launches.csv python tools/profile_step.py [--steps 2]
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from bench import CLASS_COUNTS, make_opt  # noqa: E402
from mrn_b200 import synth  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--steps", type=int, default=2)
ap.add_argument("--batch", type=int, default=256)
ap.add_argument("--mode", default="train", choices=["train", "infer"])
a = ap.parse_args()
net = synth.build_net(CLASS_COUNTS, synth.ctor_state_dict(CLASS_COUNTS, 111), make_opt("bf16", 0, "svtr"))
learner = synth.build_learner(net, train=a.mode == "train", total_steps=20000, schedule="super")
batches = [tuple(t.cuda() for t in synth.synth_batch(a.batch, CLASS_COUNTS, 1000 + k)) for k in range(2)]


def step(k):
    img, tgt, lens, dom = batches[k % 2]
    if a.mode == "train":
        return learner.train_step_stage1(img, tgt, lens, dom)
    return learner.infer_batch(img, "TF")


for k in range(3):
    step(k)
torch.cuda.synchronize()
torch.cuda.profiler.start()
for k in range(a.steps):
    out = step(k)
torch.cuda.synchronize()
torch.cuda.profiler.stop()
print("profile_step done")
