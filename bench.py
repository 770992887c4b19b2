#!/usr/bin/env python
"""bench.py -- MRN-SVTR 6-expert router-training (stage-1) step on N B200s; prints ONE JSON line on rank 0.

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
    python bench.py --impl reference ...      # the UNMODIFIED reference (baseline/_ref) running its own stage-1 loop on the host cores
    python bench.py --dump-outputs DIR ...    # also writes what the last timed step computed, DIR/<name>.npy

Workload (BASELINE.json configs[3], SURVEY.md §8d cfg 4): SVTR-MRN, I = 6 experts, union charset C_i =
[1899, 2224, 3844, 4968, 5041, 5153], per-GPU batch 256 (weak scaling), synthetic 32x256x4 crops, one
`_update_representation` iteration (il_modules/mrn.py:329-371): 6 frozen expert forwards in train mode (BN batch
statistics + DropPath, reference quirk 4) -> DM-Router -> softmax gate -> gated combine -> CTC -> loss = 15*CTC + CE ->
router backward -> [NCCL all-reduce] -> clip + Adam.

value  = samples/s with the batch resident in HBM (CUDA events, max over ranks).
e2e    = same metric through MRN.train_step_stage1 with pinned-host inputs copied H2D and both losses read back D2H
         every step (what il_modules/mrn.py's loop does); the copy of batch k+1 is issued on the learner's staging
         stream (mrn_b200.utils.DevicePrefetcher) while batch k computes -- every copy is inside the timed region.
roofline / kernel_families = CUDA-event time per kernel family recorded on the launching stream inside the timed region.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

CLASS_COUNTS = (1899, 2224, 3844, 4968, 5041, 5153)
METRIC = "MRN-SVTR 6-expert train samples/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=256, help="per-GPU batch (config/svtr_mrn.py: batch_size=256)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--chunk", type=int, default=0, help="samples per expert-forward chunk (0 = whole batch)")
    ap.add_argument("--cpu-sample", type=int, default=0, help="samples per CPU step (0 = the full per-GPU batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-reference", action="store_true", help="skip the eager-torch reference on the same GPU (N=1 only)")
    ap.add_argument("--no-parity-probe", action="store_true", help="skip the first-step comparison with the CPU oracle (N=1 only)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --batch samples per GPU (the headline); strong: --batch is the GLOBAL batch, split over the ranks "
                         "(what nn.DataParallel does with batch_size=256, il_modules/mrn.py:106,133)")
    ap.add_argument("--init", default="ctor", choices=["ctor", "synth"],
                    help="ctor: random-init weights from the constructors (BASELINE north_star, soft gates); synth: gate-spreading fixtures")
    ap.add_argument("--arch", default="svtr", choices=["svtr", "crnn"],
                    help="expert recogniser: svtr = headline (BASELINE.json configs[3-4]); crnn = VGG+BiLSTM (configs[1])")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the CUDA-graph replay of the step")
    ap.add_argument("--sweep", default="", help="infer mode only: comma-separated per-GPU batch sizes (BASELINE configs[4]: 1..4096); "
                                               "adds a `sweep` array to the JSON line")
    ap.add_argument("--mode", default="train", choices=["train", "infer", "stage0"],
                    help="train: router-training step (the BASELINE metric); infer: hard-routed forward + greedy decode (cfg 5); "
                         "stage0: expert-training step of the newest expert (SURVEY.md §8(f)3, il_modules/mrn.py:225-279)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed as DIR/<name>.npy (float32, at most 64 MB in all), so that "
                         "two builds run with the same arguments can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def make_opt(precision, chunk, arch="svtr"):
    return argparse.Namespace(Transformation="None", FeatureExtraction="SVTR" if arch == "svtr" else "VGG",
                              SequenceModeling="None" if arch == "svtr" else "BiLSTM", Prediction="CTC",
                              num_fiducial=20, input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256,
                              batch_max_length=25, lr=5e-4, num_iter=10000, grad_clip=5, exp_name="bench",
                              precision=precision, drop_path=True, expert_chunk=chunk,
                              lan_list=["Chinese", "Latin", "Japanese", "Korean", "Arabic", "Bangla"], val_interval=5000,
                              start_task=0, optimizer="adam", schedule="super")


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2])
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_stage1(sample, steps, warmup, arch="svtr"):
    """The reference algorithm's CPU path (oracle port, fp32, all host threads) on a bounded sample of the workload."""
    from oracle import mrn_oracle as O
    from mrn_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    sd = synth.synth_state_dict(CLASS_COUNTS, 111, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(sample, CLASS_COUNTS, 111)
    drop = synth.synth_drop_scales(6, sample, O.svtr_drop_path_rates(), 111) if arch == "svtr" else None
    state = dict(step=0, m={}, v={})
    for _ in range(warmup):
        O.stage1_step_cpu(sd, 6, state, img, tgt, lens, dom, drop_scales=drop)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.stage1_step_cpu(sd, 6, state, img, tgt, lens, dom, drop_scales=drop)
    dt = time.perf_counter() - t0
    return sample * steps / dt, dt / steps * 1000.0, torch.get_num_threads()


def cpu_stage0(sample, steps, warmup, arch="svtr"):
    """Stage-0 expert-training step of the oracle port (torch CPU autograd) on a bounded sample."""
    from oracle import mrn_oracle as O
    from mrn_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cc = CLASS_COUNTS[-1:]
    sd = synth.synth_state_dict(cc, 111, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(sample, cc, 111)
    drop = synth.synth_drop_scales(1, sample, O.svtr_drop_path_rates(), 111)[0] if arch == "svtr" else None
    state = dict(step=0, m={}, v={})
    for _ in range(warmup):
        O.stage0_step_cpu(sd, 0, state, img, tgt, lens, drop_scales=drop)
    t0 = time.perf_counter()
    for _ in range(steps):
        O.stage0_step_cpu(sd, 0, state, img, tgt, lens, drop_scales=drop)
    dt = time.perf_counter() - t0
    return sample * steps / dt, dt / steps * 1000.0, torch.get_num_threads()


def workload_config(arch, B, world, chunk, precision):
    return {"workload": "%s-MRN 6-expert stage-1 (router-training) step, B=%d/GPU, union charset 5153, 32x256x4 crops, "
                        "experts frozen in train mode (BN batch stats%s)" % (arch.upper(), B, " + DropPath" if arch == "svtr" else ""),
            "global_batch": B * world, "parallelism": "dp%d" % world, "expert_chunk": chunk,
            "init": "random-init weights from the constructors (soft gates)",
            "l2": "4 rotating input batches; >1 GB of activations streamed per step (>> 126 MB L2), no explicit flush",
            "router_precision": "bf16 operands / fp32 accumulate (tcgen05)" if precision == "bf16" else "fp32",
            "expert_precision": precision}


def ref_arm(device, B, steps, warmup, gpu_index=0, timeout=1500):
    """Runs baseline/ref_arm.py (the unmodified reference's own stage-1 loop from baseline/_ref) in a child process and
    returns its JSON dict; {"unavailable": why} when the reference is not staged."""
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    if device == "cuda":
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        env["CUDA_VISIBLE_DEVICES"] = vis.split(",")[gpu_index] if vis else str(gpu_index)
    cmd = [sys.executable, os.path.join(ROOT, "baseline", "ref_arm.py"), "--device", device, "--batch", str(B),
           "--steps", str(steps), "--warmup", str(warmup)]
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=timeout)
        line = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
        if not line:
            return {"unavailable": "reference arm printed no result (rc %d): %s" % (r.returncode, r.stderr[-300:])}
        return json.loads(line[-1])
    except Exception as ex:                              # noqa: BLE001
        return {"unavailable": "reference arm failed: %s" % (ex,)}


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores.  SVTR: the
    unmodified reference from baseline/_ref driving MRN._update_representation (kind "reference"); if it is not staged,
    or for --arch crnn, the oracle port (kind "port")."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    B = args.batch
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    sample = args.cpu_sample or B
    if not args.cpu_sample and steps + warmup > 30:      # keep the whole run within a few minutes
        sample = max(32, B // 2)
    res = ref_arm("cpu", sample, steps, warmup) if args.arch == "svtr" else {"unavailable": "crnn arm uses the port"}
    if "unavailable" not in res:
        v, ms, cores, kind = res["samples_per_s"], res["ms_per_step"], res["threads"], "reference"
        desc = ("%d-sample iterations of the UNMODIFIED reference loop (baseline/_ref: il_modules/mrn.py::_update_representation, "
                "MRNNet.cross_forward, CTCLoss, Adam, OneCycleLR), fp32, %d threads, torch %s" % (sample, cores, res["torch"]))
    else:
        sys.stderr.write("bench.py: %s; timing the oracle port instead\n" % res["unavailable"])
        sample = min(sample, 32)
        v, ms, cores = cpu_stage1(sample, steps, warmup, args.arch)
        kind, desc = "port", "%d-sample router-training step per iteration, oracle port, fp32, %d threads" % (sample, cores)
    cfg = workload_config(args.arch, B, 1, 0, "fp32")
    cfg.update({"per_step_samples": sample, "parallelism": "cpu", "router_precision": "fp32", "expert_precision": "fp32"})
    out = {
        "impl": "reference", "metric": METRIC.replace("SVTR", args.arch.upper()), "value": round(v, 3), "unit": "samples/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": round(v, 3), "unit": "samples/s", "cores": cores, "kind": kind, "sample": desc},
        "e2e": {"value": round(v, 3), "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if "unavailable" not in res:
        out["loss_first"] = {"loss_clf": res.get("loss_clf_first"), "taski_loss": res.get("taski_loss_first")}
        out["reference_flags"] = res.get("flags")
    print(json.dumps(out))


def ncu_traffic(kernel, arch="svtr"):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed `ncu --set full` capture
    (profiles/ncu_traffic.json, written by tools/ncu_traffic.py; captured on the SVTR workload), or None."""
    if arch != "svtr":
        return None
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        return t.get(kernel, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def infer_sweep(learner, batches, dev):
    """BASELINE configs[4]: hard-routed inference + device greedy decode over a range of batch sizes (resident inputs,
    CUDA events, 3 warm-up + >=5 timed steps per size; two rotating input batches)."""
    from mrn_b200 import synth
    rows = []
    for B in batches:
        imgs = [synth.synth_batch(B, CLASS_COUNTS, 2000 + k)[0].to(dev) for k in range(2)]
        for k in range(3):
            learner.infer_batch(imgs[k % 2], "TF")
        torch.cuda.synchronize()
        steps = 20 if B <= 256 else (8 if B <= 1024 else 5)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(steps):
            r = learner.infer_batch(imgs[k % 2], "TF")
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        row = {"batch": B, "ms_per_batch": round(ms, 3), "samples_per_s": round(B * 1000.0 / ms, 1)}
        if B <= 128:                    # launch-bound sizes: the same call replayed from a CUDA graph
            for k in range(3):
                learner.infer_batch_graphed(imgs[k % 2], "TF")
            torch.cuda.synchronize()
            e0.record()
            for k in range(steps):
                r = learner.infer_batch_graphed(imgs[k % 2], "TF")
            e1.record()
            torch.cuda.synchronize()
            msg = e0.elapsed_time(e1) / steps
            row.update({"graph_ms_per_batch": round(msg, 3), "graph_samples_per_s": round(B * 1000.0 / msg, 1)})
        rows.append(row)
        del imgs, r
        torch.cuda.empty_cache()
    return rows


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(learner, loss, infer, stage0):
    """What a caller holds after the last timed step, as host float32 arrays: the step's return values and, for the
    training modes, the parameters the step updated and the gradients it computed."""
    if infer:
        r = loss[2]
        out = {k: r[k] for k in ("ids", "lens", "conf", "index")}
    elif stage0:
        out = {"loss": loss[0], "params": learner._tp.params, "grads": learner._tp.grads}
    else:
        net = learner.net
        out = {"loss_clf": loss[0], "taski_loss": loss[1], "router_params": net.router_arena(),
               "router_grads": net.router_grad_arena()}
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def dump_outputs(out_dir, arrays):
    """Writes DIR/<name>.npy.  An array larger than an equal share of DUMP_LIMIT_BYTES is cut to every k-th element of
    its flattened form: a fixed sample, the same on every run with the same arguments."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    share = DUMP_LIMIT_BYTES // 4 // len(arrays)
    for name, a in arrays.items():
        if a.size > share:
            a = a.reshape(-1)[:: -(-a.size // share)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------ GPU arm
def run_ours(args):
    from mrn_b200 import dist as mdist
    from mrn_b200 import ops, synth
    from mrn_b200.il_modules.mrn import MRN, RankLocal, FusedAdam
    from mrn_b200.modules.model import MRNNet
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: mrn_b200 has no CPU fallback")
    rank, local_rank, world = mdist.init_from_env("nccl")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch
    if args.scaling == "strong":
        if B % world:
            raise SystemExit("--scaling strong needs --batch divisible by the number of GPUs")
        B = B // world
    opt = make_opt(args.precision, args.chunk, args.arch)
    # the train-mode steps draw their DropPath masks from torch's device generator: a fixed seed gives every run with
    # the same arguments the same masks, whichever --init is chosen
    torch.manual_seed(111)
    sd = (synth.ctor_state_dict if args.init == "ctor" else synth.synth_state_dict)(CLASS_COUNTS, 111, arch=args.arch)
    T = 64 if args.arch == "svtr" else 63
    net = MRNNet(opt)
    for c in CLASS_COUNTS:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    net.load_state_dict(sd, strict=True)
    net = net.to(dev)
    learner = MRN(opt)
    learner.model = RankLocal(net)
    learner.model.train()                               # steady state of the reference loop (quirk 4)
    for p in net.model.parameters():
        p.requires_grad = False
    learner.optimizer = FusedAdam(net, opt.lr, opt.num_iter * 2, grad_clip=opt.grad_clip, schedule="super")
    mdist.broadcast_(net.router_arena())

    # distinct synthetic batches per rank (seeded); pinned host copies for the e2e leg
    n_batches = 4
    host = []
    for k in range(n_batches):
        img, tgt, lens, dom = synth.synth_batch(B, CLASS_COUNTS, 1000 + 17 * rank + k)
        host.append(tuple(t.pin_memory() for t in (img, tgt, lens, dom)))
    resident = [tuple(t.to(dev) for t in hb) for hb in host]
    h2d = sum(t.numel() * t.element_size() for t in host[0])

    infer = args.mode == "infer"
    stage0 = args.mode == "stage0"
    if stage0:
        opt.num_iter = 1000000
        learner.begin_expert_training()                 # newest expert (C = 5153) -> flat training arena + fused Adam
        mdist.broadcast_(learner._tp.params)
    if infer:
        learner.model.eval()                            # validation(): model.eval(), hard route, greedy decode (test.py:139-221)

    use_graph = not args.no_graph
    train_step = learner.train_step_stage1_graphed if use_graph else learner.train_step_stage1
    infer_step = learner.infer_batch_graphed if use_graph else learner.infer_batch

    def step_resident(k, eager=False):
        img, tgt, lens, dom = resident[k % n_batches]
        if infer:
            r = (learner.infer_batch if eager else infer_step)(img, "TF")
            return r["conf"], r["lens"], r                  # the whole result rides along for --dump-outputs
        if stage0:
            l0 = (learner.train_step_stage0 if (eager or not use_graph) else learner.train_step_stage0_graphed)(img, tgt, lens)
            return l0, l0
        return (learner.train_step_stage1 if eager else train_step)(img, tgt, lens, dom)

    from mrn_b200.utils import DevicePrefetcher
    pf = DevicePrefetcher(dev)              # the learner's own staging: batch k+1 is copied while batch k computes

    def step_e2e(k):
        if pf.pending is None:
            pf.submit(host[k % n_batches])
        img, tgt, lens, dom = pf.take()
        pf.submit(host[(k + 1) % n_batches])
        if infer:
            r = infer_step(img, "TF")
            ids = r["ids"].cpu()                        # the single D2H copy of the decoded ids (+ lengths, confidences)
            return float(r["conf"].sum()), float(r["lens"].sum()) + float(ids[0, 0])
        if stage0:
            l0 = float((learner.train_step_stage0_graphed if use_graph else learner.train_step_stage0)(img, tgt, lens))
            return l0, l0
        l1, l2 = train_step(img, tgt, lens, dom)
        return float(l1), float(l2)                     # D2H read of both losses (the reference logs them)

    # ---- parity probe (N = 1, stage-1 train): the FIRST step runs eagerly with injected DropPath masks and is compared
    # with the fp32 CPU oracle of the same step on the same batch / masks / weights (2e-2 bf16 budget of north_star)
    probe = None
    if world == 1 and not infer and not stage0 and not args.no_parity_probe:
        from oracle import mrn_oracle as O
        drop = synth.synth_drop_scales(6, B, O.svtr_drop_path_rates(), 111) if args.arch == "svtr" else None
        sd_o = {k: v.clone() for k, v in sd.items()}
        img, tgt, lens, dom = resident[0]
        l1, l2 = learner.train_step_stage1(img, tgt, lens, dom, drop_scales=None if drop is None else drop.to(dev))
        got = (float(l1), float(l2))
        torch.set_num_threads(os.cpu_count() or 1)
        t0 = time.perf_counter()
        ref = O.stage1_step_cpu(sd_o, 6, dict(step=0, m={}, v={}), *host[0], drop_scales=drop)
        probe = {"loss_first": {"loss_clf": got[0], "taski_loss": got[1]},
                 "oracle_loss_first": {"loss_clf": ref[0], "taski_loss": ref[1]},
                 "rel_err_loss_clf": abs(got[0] - ref[0]) / max(abs(ref[0]), 1e-30), "abs_err_taski": abs(got[1] - ref[1]),
                 "tolerance": 2e-2 if args.precision == "bf16" else 1e-4, "oracle_cpu_s": round(time.perf_counter() - t0, 2)}
        probe["ok"] = bool(probe["rel_err_loss_clf"] < probe["tolerance"] and probe["abs_err_taski"] < probe["tolerance"])
        del sd_o

    hist = torch.zeros(3, max(args.steps, 1), 2, device=dev)      # losses of every timed step (checked after each region)

    def record(phase, k, loss):
        hist[phase, k, 0].copy_(loss[0].float().sum(), non_blocking=True)
        hist[phase, k, 1].copy_(loss[1].float().sum(), non_blocking=True)

    try:
        for k in range(max(3, args.warmup)):
            step_resident(k)
        torch.cuda.synchronize()
    except Exception as ex:                             # graph capture unavailable: time the eager launches instead
        if not use_graph:
            raise
        sys.stderr.write("bench.py: CUDA-graph capture failed (%s); falling back to eager launches\n" % (ex,))
        learner.reset_graphs()
        use_graph = False
        train_step, infer_step = learner.train_step_stage1, learner.infer_batch
        for k in range(max(3, args.warmup)):
            step_resident(k)
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # ---- per-kernel-family pass: eager launches with CUDA events around every family (cannot live inside a graph)
    mdist.barrier(); torch.cuda.synchronize()
    ops.reset_launch_count(); ops.profile_reset(); ops.profile_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        loss = step_resident(k, eager=True)
        record(0, k, loss)
    e1.record()
    mdist.barrier(); torch.cuda.synchronize()
    ops.profile_enable(False)
    ms_eager = mdist.max_over_ranks(e0.elapsed_time(e1), dev)
    launches = ops.launch_count()
    fam = ops.profile_read()
    ms_total = ms_eager
    if use_graph:
        # ---- timed region 1: batch resident in HBM, the step replayed from its CUDA graph (the product path)
        for k in range(3):
            step_resident(k)
        mdist.barrier(); torch.cuda.synchronize()
        e0.record()
        for k in range(args.steps):
            loss = step_resident(k)
            record(1, k, loss)
        e1.record()
        mdist.barrier(); torch.cuda.synchronize()
        ms_total = mdist.max_over_ranks(e0.elapsed_time(e1), dev)
    if args.dump_outputs and rank == 0:
        # `loss` and the learner's state are those of the last step of the region `value` is timed on; the e2e steps
        # below change the parameters again
        dump_outputs(args.dump_outputs, step_outputs(learner, loss, infer, stage0))
    # ---- timed region 2: end to end from pinned host memory
    for k in range(2):
        step_e2e(k)
    mdist.barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_losses = []
    for k in range(args.steps):
        last = step_e2e(k)
        e2e_losses.append(last)
    torch.cuda.synchronize()
    e2e_ms = mdist.max_over_ranks((time.perf_counter() - t0) * 1000.0, dev)
    clocks = sampler.stop() if rank == 0 else None
    # ---- a step that computes on NaNs is not a measurement: every loss of every timed step must be finite
    hist_h = hist[: 2 if use_graph else 1, :args.steps].cpu()
    bad = (not bool(torch.isfinite(hist_h).all())) or any(not (v[0] == v[0] and abs(v[0]) != float("inf") and v[1] == v[1]
                                                                 and abs(v[1]) != float("inf")) for v in e2e_losses)
    if bad:
        sys.stderr.write("bench.py: NON-FINITE LOSS inside the timed region (rank %d): eager %s graph %s e2e %s -- no value is reported\n"
                         % (rank, hist_h[0].tolist(), hist_h[1].tolist() if use_graph else None, e2e_losses))
        sys.stderr.flush()
        os._exit(3)
    if rank != 0:
        return

    ms_step = ms_total / args.steps
    value = B * world * 1000.0 / ms_step
    e2e_value = B * world * args.steps * 1000.0 / e2e_ms
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    tf_peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    fams = {}
    for name, f in fam.items():
        if f["calls"] == 0:
            continue
        per_step = f["ms"] / args.steps
        d = {"ms_per_step": round(per_step, 3), "share": round(f["ms"] / ms_eager, 4), "launches_per_step": f["calls"] // args.steps}
        if f["flops"] > 0 and f["ms"] > 0:
            d["tflops"] = round(f["flops"] / f["ms"] / 1e9, 2)
        if f["bytes"] > 0 and f["ms"] > 0:
            d["gbs"] = round(f["bytes"] / f["ms"] / 1e6, 1)
        fams[name] = d
    # SURVEY.md §8(d): the expert / router contractions are bounded by the tensor cores, everything else on the path
    # (gated combine, log-softmax / CTC, LayerNorm, router element-wise stages, optimiser) by HBM bandwidth.
    TENSOR_BOUND = {"tc_gemm_kernel", "tc_gemm2_kernel", "attn_tc_kernel", "mlp_tc_kernel", "sgemm_kernel", "mixer_tc_kernel",
                    "patch_embed"}
    dom_name = max(fams, key=lambda k: fams[k]["ms_per_step"]) if fams else None
    roofline = None
    traffic_db = {}
    try:
        traffic_db = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
    except Exception:
        pass
    if dom_name:
        d, f = fams[dom_name], fam[dom_name]
        n_launch = max(1, f["calls"])
        frac_t = d.get("tflops", 0.0) / tf_peak
        frac_h = d.get("gbs", 0.0) / hbm_peak
        if dom_name in TENSOR_BOUND:
            roofline = {"kernel": dom_name, "bound": "tensor", "achieved": d.get("tflops"), "peak": tf_peak, "unit": "TFLOP/s",
                        "frac": round(frac_t, 4), "traffic": ncu_traffic(dom_name, args.arch),
                        "algorithmic_flops_per_launch": f["flops"] / n_launch, "peak_source": peak_src + ", sustained"}
        else:
            roofline = {"kernel": dom_name, "bound": "hbm", "achieved": d.get("gbs"), "peak": hbm_peak, "unit": "GB/s",
                        "frac": round(frac_h, 4), "traffic": ncu_traffic(dom_name, args.arch),
                        "algorithmic_bytes_per_launch": f["bytes"] / n_launch, "peak_source": peak_src}
        roofline.update({"bound_source": "SURVEY.md 8(d)", "launches_per_step": f["calls"] // args.steps,
                         "avg_launch_us": round(f["ms"] / n_launch * 1e3, 1),
                         "frac_tensor": round(frac_t, 4), "frac_hbm": round(frac_h, 4)})
        if not infer and not stage0 and args.arch == "svtr":
            # whole step against the tensor roof: SURVEY.md 8(d) counts 15.20 GFLOP per sample (dense-equivalent attention)
            step_tf = 15.20e9 * B / (ms_step * 1e-3) / 1e12
            roofline["step"] = {"gflop_per_sample": 15.20, "tflops": round(step_tf, 1),
                                "frac_tensor_sustained": round(step_tf / tf_peak, 4),
                                "dram_bytes_per_step_ncu": traffic_db.get("_step", {}).get("dram_bytes_per_step"),
                                "dram_bytes_per_step_algorithmic": int(B * (4 * 32 * 256 * 4 + 5.92e6) + 43.4e6 * 2)}
    ctc_router_ms = sum(fams.get(k, {}).get("ms_per_step", 0.0) for k in ("sgemm_kernel", "tc_gemm2_kernel", "router_elementwise",
                                                                          "combine_row_kernel", "ctc_lattice_kernel"))
    cfg = workload_config(args.arch, B, world, args.chunk, args.precision)
    if args.init != "ctor":
        cfg["init"] = "synthetic gate-spreading fixtures (mrn_b200/synth.py)"
    out = {
        "metric": (METRIC if not infer else "MRN-SVTR 6-expert inference + greedy decode samples/s").replace("SVTR", args.arch.upper()),
        "value": round(value, 2),
        "unit": "samples/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": args.scaling,
        "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": cfg,
        "e2e": {"value": round(e2e_value, 2), "unit": "samples/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": 8 if not infer else B * T * 4 + B * 8,
                "ms_per_step": round(e2e_ms / args.steps, 3)},
        "cuda_graph": bool(use_graph), "ms_per_step_eager": round(ms_eager / args.steps, 3),
        "gpu_launches": int(launches),
        "gpu_launches_per_step": int(launches // args.steps),
        "clocks": clocks,
        "roofline": roofline,
        "kernel_families": fams,
        "ctc_router_ms_per_batch": round(ctc_router_ms, 3),
        "loss_clf": float(last[0]), "taski_loss": float(last[1]),
        "losses_finite": True,
        "loss_last": {"loss_clf": float(last[0]), "taski_loss": float(last[1])},
    }
    if probe:
        out.update({"loss_first": probe["loss_first"], "oracle_loss_first": probe["oracle_loss_first"], "parity_probe": probe})
    if stage0:
        out["metric"] = "MRN-%s stage-0 expert-training samples/s" % args.arch.upper()
        out["dtype"] = "f32" if learner._tp.prec == 0 else "bf16"
        out["config"]["workload"] = ("%s-MRN stage-0 step: newest expert (C=5153) forward + CTC + full backward + clip/Adam, "
                                     "B=%d/GPU, train mode (BN batch stats%s)" % (args.arch.upper(), B, " + DropPath" if args.arch == "svtr" else ""))
        out["config"]["expert_precision"] = out["dtype"]
        out.pop("taski_loss", None)
    if infer:
        out["config"]["workload"] = ("%s-MRN 6-expert hard-routed inference + device greedy decode, B=%d/GPU, union charset 5153"
                                     % (args.arch.upper(), B))
        if args.sweep:
            out["sweep"] = infer_sweep(learner, [int(x) for x in args.sweep.split(",") if x], dev)
        if world == 1 and not args.no_parity_probe and args.arch == "svtr":
            # decode parity on a bounded sample: routed expert, greedy-decoded ids and confidence of the first 16 crops
            # against the fp32 CPU oracle (north_star: identical decoded indices except exact-tie arg-max cases, counted)
            from oracle import mrn_oracle as O
            ns = min(16, B)
            torch.set_num_threads(os.cpu_count() or 1)
            t0 = time.perf_counter()
            with torch.no_grad():
                ref = O.mrn_forward({k: v.clone() for k, v in sd.items()}, 6, host[0][0][:ns].float(), is_train=False, bn_mode="eval")
                k_ref, seq_ref, conf_ref = O.greedy_decode(ref["logits"])
            r = learner.infer_batch(resident[0][0][:ns].contiguous(), "TF")
            ids, lens, conf = r["ids"].cpu(), r["lens"].cpu(), r["conf"].cpu()
            same, tie_like = 0, 0
            top2 = ref["logits"].topk(2, dim=2)[0]
            margin = (top2[..., 0] - top2[..., 1])                       # [ns, T] arg-max margin of the oracle logits
            for b_ in range(ns):
                got = [int(v) for v in ids[b_, :int(lens[b_])]]
                if got == seq_ref[b_]:
                    same += 1
                elif float(margin[b_].min()) < 2e-2 * float(ref["logits"][b_].abs().max()):
                    tie_like += 1                                          # a frame whose top-2 logits sit within the bf16 budget
            out["decode_parity"] = {
                "samples": ns, "route_identical": int((r["index"].cpu() == ref["index"]).sum()), "decoded_identical": same,
                "mismatches_at_near_ties": tie_like, "mismatches_other": ns - same - tie_like,
                "max_conf_abs_err": float((conf - conf_ref).abs().max()), "max_conf_ref": float(conf_ref.max()),
                "oracle_cpu_s": round(time.perf_counter() - t0, 2),
                "note": "fp32 CPU oracle vs the %s device path, eval-mode experts, hard route" % args.precision}
    if world == 1 and not args.no_cpu_baseline and stage0:
        cs = args.cpu_sample or 32
        v, ms, cores = cpu_stage0(cs, 2, 1, args.arch)
        out["cpu_baseline"] = {"value": round(v, 3), "unit": "samples/s", "cores": cores, "kind": "port",
                               "sample": "2 timed expert-training steps of %d samples, oracle port (torch CPU autograd), fp32, "
                                         "%d threads" % (cs, cores)}
    elif world == 1 and not args.no_cpu_baseline and not infer:
        cs = args.cpu_sample or B
        res = ref_arm("cpu", cs, 2, 1) if args.arch == "svtr" else {"unavailable": "crnn uses the port"}
        if "unavailable" not in res:
            out["cpu_baseline"] = {"value": round(res["samples_per_s"], 3), "unit": "samples/s", "cores": res["threads"], "kind": "reference",
                                   "sample": "1 warm-up + 2 timed %d-sample iterations of the unmodified reference loop (baseline/_ref: "
                                             "MRN._update_representation), fp32, %d threads" % (cs, res["threads"]),
                                   "ms_per_step": round(res["ms_per_step"], 1)}
        else:
            cs = min(cs, 32)
            v, ms, cores = cpu_stage1(cs, 2, 1, args.arch)
            out["cpu_baseline"] = {"value": round(v, 3), "unit": "samples/s", "cores": cores, "kind": "port",
                                   "sample": "2 timed router-training steps of %d samples (batch reduced from %d), oracle port of the "
                                             "reference algorithm, fp32, %d threads; %s" % (cs, B, cores, res["unavailable"])}
    if world == 1 and not args.no_gpu_reference and not infer and not stage0 and args.arch == "svtr":
        # the GPU bar (SURVEY.md 8d): the same unmodified reference loop, eager torch library kernels, on this B200
        del learner, resident
        torch.cuda.empty_cache()
        res = ref_arm("cuda", B, 10, 3, gpu_index=local_rank)
        if "unavailable" in res:
            out["gpu_eager_reference"] = res
        else:
            out["gpu_eager_reference"] = {"value": round(res["samples_per_s"], 2), "unit": "samples/s", "ms_per_step": round(res["ms_per_step"], 3),
                                          "batch": B, "steps": res["steps"], "warmup": res["warmup"], "flags": res["flags"],
                                          "torch": res["torch"], "peak_mem_gb": res.get("peak_mem_gb"), "code": res["code"],
                                          "timing": "wall clock between loader calls with cuda.synchronize (H2D of the batch and loss D2H inside, as in e2e)",
                                          "speedup_e2e": round(e2e_value / res["samples_per_s"], 2),
                                          "speedup_resident": round(value / res["samples_per_s"], 2)}
    print(json.dumps(out))


def _shutdown():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        try:
            run_ours(a)
        finally:
            _shutdown()
