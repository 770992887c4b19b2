"""The reference's whole task loop (tiny_train.py:195-294 -> il_modules/mrn.py:136-167) on the CUDA path with an
in-memory synthetic dataset layer: task 0 expert training (stage 0), task 1 expert training + router training
(stage 0 + stage 1), validation, checkpoint save / strict reload, benchmark test."""
import os

import numpy as np
import pytest
import torch

from mrn_b200 import synth


N_NEW = (12, 10)           # new characters per task


def _chars(k):
    return [chr(0x4E00 + i) for i in range(sum(N_NEW[:k + 1]))]


class _Manager:
    """Dataset_Manager surface: get_dataset(taski, memory), get_batch() -> (images, labels), get_batch2() ->
    (images, labels, domain ids).  Labels of task k only use that task's new characters; images are synthetic."""

    def __init__(self, B):
        self.B, self.taski, self.calls = B, 0, []
        self.rng = np.random.default_rng(5)

    def init_start(self, opt, select_data, log, taski):
        self.get_dataset(taski, memory=None)

    def get_dataset(self, taski, memory=None, index_list=None):
        self.taski = taski
        self.calls.append((taski, memory))

    def _labels(self, task, n):
        lo = sum(N_NEW[:task])
        pool = _chars(len(N_NEW) - 1)[lo:lo + N_NEW[task]]
        return ["".join(self.rng.choice(pool, size=int(self.rng.integers(1, 9)))) for _ in range(n)]

    def get_batch(self):
        img = synth.randn(int(self.rng.integers(1 << 30)), "img", (self.B, 4, 32, 256)).clamp_(-1, 1)
        return img, self._labels(self.taski, self.B)

    def get_batch2(self):
        img = synth.randn(int(self.rng.integers(1 << 30)), "img", (self.B, 4, 32, 256)).clamp_(-1, 1)
        dom = self.rng.integers(0, self.taski + 1, size=self.B)
        labels = [self._labels(int(d), 1)[0] for d in dom]
        return img, labels, [torch.tensor(dom)]


class _Valid:
    def __init__(self, mgr, taski):
        self.mgr, self.taski = mgr, taski

    def create_dataset(self):
        img, lab = self.mgr.get_batch()
        return [(img, lab)]

    def create_list_dataset(self):
        out = []
        for k in range(self.taski + 1):
            self.mgr.taski = k
            out.append(self.mgr.get_batch())
        self.mgr.taski = self.taski
        return out


@pytest.mark.gpu
def test_two_task_incremental_run(tmp_path, monkeypatch):
    from mrn_b200 import tiny_train
    monkeypatch.chdir(tmp_path)
    opt = synth.make_opt(il="mrn", exp_name="inc", lan_list=["A", "B"], num_iter=4, val_interval=10, batch_size=4,
                         memory="random", memory_num=8, drop_path=True)
    tiny_train.seed_everything(111)
    mgr = _Manager(opt.batch_size)
    best, ned = tiny_train.train(opt, mgr, lambda k: _Valid(mgr, k), lambda k: _chars(k),
                                 lambda k: [[b] for b in _Valid(mgr, k).create_list_dataset()])   # one loader per benchmark set
    assert len(best) == 2 and len(ned) == 2 and all(0.0 <= v <= 100.0 for v in best + ned)
    # protocol: task 0 dataset, task 1 stage-0 dataset (memory None), task 1 stage-1 rehearsal dataset
    assert mgr.calls[:3] == [(0, None), (1, None), (1, "random")]
    for f in ("A_0_0_best_score.pth", "B_1_0_best_score.pth", "B_1_1_best_score.pth"):
        assert os.path.exists(os.path.join("saved_models", "inc", f)), f
    sd = torch.load(os.path.join("saved_models", "inc", "B_1_1_best_score.pth"), map_location="cpu")
    assert sd["module.model.0.fc.weight"].shape[0] == N_NEW[0] + 4
    assert sd["module.model.1.fc.weight"].shape[0] == sum(N_NEW) + 4
    assert sd["module.channel_route.weight"].shape == (2, 512)
    assert all(torch.isfinite(v).all() for v in sd.values() if v.is_floating_point())
    log = open(os.path.join("saved_models", "inc", "log_train.txt")).read()
    assert "Train_taski_loss" in log and "Test Average Incremental Accuracy" in log


def test_load_config_reads_a_reference_style_config(tmp_path):
    from mrn_b200 import tiny_train
    p = tmp_path / "cfg.py"
    p.write_text('common=dict(exp_name="X", il="mrn", manual_seed=111, start_task=0, batch_max_length=25, imgH=32, imgW=256)\n'
                 'model=dict(Transformation="None", FeatureExtraction="SVTR", SequenceModeling="None", Prediction="CTC",\n'
                 '           input_channel=4, output_channel=512, hidden_size=256, num_fiducial=20)\n'
                 'optimizer=dict(schedule="super", optimizer="adam", lr=0.0005)\n'
                 'train=dict(lan_list=["Chinese", "Latin"], batch_size=256, num_iter=10000, val_interval=5000, grad_clip=5)\n')
    opt = tiny_train.load_config(str(p))
    assert opt.FeatureExtraction == "SVTR" and opt.lr == 0.0005 and opt.lan_list == ["Chinese", "Latin"] and opt.il == "mrn"
