"""2-GPU data-parallel parity: two ranks, each on its shard, all-reduced (NCCL) gradient arena + identical clip/Adam
== one GPU on the concatenated batch (SURVEY.md §4, §8e).  Skipped on boxes with fewer than 2 GPUs."""
import argparse
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _opt():
    return argparse.Namespace(Transformation="None", FeatureExtraction="SVTR", SequenceModeling="None", Prediction="CTC",
                              num_fiducial=20, input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256,
                              batch_max_length=25, lr=5e-4, num_iter=100, grad_clip=5, exp_name="dp", precision="fp32",
                              drop_path=False, lan_list=["a", "b", "c"], val_interval=50, start_task=0)


def _build(cc, sd, dev):
    from mrn_b200.il_modules.mrn import MRN, RankLocal, FusedAdam
    from mrn_b200.modules.model import MRNNet
    opt = _opt()
    net = MRNNet(opt)
    for c in cc:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval()
    learner = MRN(opt)
    learner.model = RankLocal(net)
    learner.optimizer = FusedAdam(net, 5e-4, 200, schedule="const")
    return net, learner


def _worker(rank, world, port, out):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    from mrn_b200 import dist as mdist, synth
    mdist.init_from_env("nccl")
    dev = torch.device("cuda", rank)
    cc, B, seed = (37, 61, 96), 4, 21
    sd = synth.synth_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    net, learner = _build(cc, sd, dev)
    lo, hi = mdist.shard_bounds(B, rank, world)
    l1, l2 = learner.train_step_stage1(img[lo:hi].to(dev), tgt[lo:hi].to(dev), lens[lo:hi].to(dev), dom[lo:hi].to(dev))
    torch.cuda.synchronize()
    out[rank] = (net.router_arena().cpu(), float(l1), float(l2))
    torch.distributed.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_step_equals_single_gpu_step():
    from mrn_b200 import synth
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    cc, B, seed = (37, 61, 96), 4, 21
    sd = synth.synth_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    dev = torch.device("cuda", 0)
    net, learner = _build(cc, sd, dev)
    l1, l2 = learner.train_step_stage1(img.to(dev), tgt.to(dev), lens.to(dev), dom.to(dev))
    ref = net.router_arena().cpu()
    a0, a1 = out[0][0], out[1][0]
    assert torch.equal(a0, a1), "ranks diverged after the all-reduced step"
    d = (a0 - ref).abs()
    assert float(d.max()) <= 5e-4 * 1.01 and float((d > 2e-5).float().mean()) < 1e-2      # Adam amplifies fp32 round-off
    assert abs(0.5 * (out[0][1] + out[1][1]) - float(l1)) / abs(float(l1)) < 1e-5         # mean of shard means


# ---- stage 0 (expert training): all-reduce of the expert's gradient arena -----------------------------------------
def _worker_stage0(rank, world, port, out):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR="127.0.0.1",
                      MASTER_PORT=str(port))
    from mrn_b200 import dist as mdist, synth
    mdist.init_from_env("nccl")
    dev = torch.device("cuda", rank)
    cc, B, seed = (37, 61), 4, 23
    sd = synth.synth_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    net, learner = _build(cc, sd, dev)
    learner.opt.schedule = "const"
    learner.begin_expert_training(total_steps=100)
    net.model[-1].eval()                      # running-statistics BatchNorm: shards and the full batch see the same network
    lo, hi = mdist.shard_bounds(B, rank, world)
    loss = learner.train_step_stage0(img[lo:hi].to(dev), tgt[lo:hi].to(dev), lens[lo:hi].to(dev))
    torch.cuda.synchronize()
    out[rank] = (learner._tp.params.cpu(), float(loss))
    torch.distributed.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_stage0_step_equals_single_gpu_step():
    from mrn_b200 import synth
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker_stage0, args=(2, port, out), nprocs=2, join=True)
    cc, B, seed = (37, 61), 4, 23
    sd = synth.synth_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    dev = torch.device("cuda", 0)
    net, learner = _build(cc, sd, dev)
    learner.opt.schedule = "const"
    learner.begin_expert_training(total_steps=100)
    net.model[-1].eval()
    loss = learner.train_step_stage0(img.to(dev), tgt.to(dev), lens.to(dev))
    ref = learner._tp.params.cpu()
    a0, a1 = out[0][0], out[1][0]
    assert torch.equal(a0, a1), "ranks diverged after the all-reduced step"
    d = (a0 - ref).abs()
    assert float(d.max()) <= 5e-4 * 2.01 and float((d > 2e-5).float().mean()) < 2e-2      # Adam amplifies fp32 round-off
    assert abs(0.5 * (out[0][1] + out[1][1]) - float(loss)) / abs(float(loss)) < 1e-4
