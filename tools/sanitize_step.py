#!/usr/bin/env python
"""One small bf16 stage-1 step + one hard-routed inference call (the workload of tools/sanitize.sh).
ARCH=crnn B=128 covers the CRNN experts, including the persistent LSTM kernel (it needs 128-sample tiles)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
from bench import CLASS_COUNTS, make_opt  # noqa: E402
from mrn_b200 import synth  # noqa: E402

ARCH = os.environ.get("ARCH", "svtr")
B = int(os.environ.get("B", 4))
net = synth.build_net(CLASS_COUNTS, synth.ctor_state_dict(CLASS_COUNTS, 111, arch=ARCH), make_opt("bf16", 0, ARCH))
learner = synth.build_learner(net, total_steps=100)
img, tgt, lens, dom = (t.cuda() for t in synth.synth_batch(B, CLASS_COUNTS, 1000))
l1, l2 = learner.train_step_stage1(img, tgt, lens, dom)
learner.model.eval()
r = learner.infer_batch(img, "TF")
torch.cuda.synchronize()
print("sanitize_step ok: loss_clf %.4f taski %.4f decoded lens %s" % (float(l1), float(l2), r["lens"].cpu().tolist()))
