"""MRN learner: the reference's il_modules/mrn.py API (MRN(opt).incremental_train / _update_representation / val /
test / after_task / change_model / build_model) driving the CUDA path.

What runs where
  * stage 1 (router training, il_modules/mrn.py:298-384) -- the north-star hot path -- is one fused device step:
    grouped frozen experts -> DM-Router -> gate -> fused combine + CTC -> analytic gate gradient -> router backward
    -> [NCCL all-reduce of the gradient arena] -> clip + Adam.  No autograd graph, no host sync inside the step.
  * validation (test.py:139-279) uses the hard route + device-side greedy decode (one D2H copy per batch), or with
    opt.decode = "beam" the device CTC prefix beam search (an addition beyond the reference).
  * stage 0 (training the newest expert end to end, il_modules/mrn.py:225-279; SURVEY.md §8(f)3) for SVTR experts:
    activation-keeping forward -> fused log-softmax + CTC -> dense CTC gradient -> hand-written backward to every
    parameter of the expert (mrnb_svtr_train_forward / _backward) -> [NCCL all-reduce of the expert's gradient arena]
    -> clip + Adam on the arena.  CRNN experts run the same step (VGG + BiLSTM BPTT, mrnb_crnn_train_forward /
    _backward).
Host-side schedule / logging logic follows il_modules/base.py.
"""
import math
import os
import time

import numpy as np
import torch

from .. import dist as mdist
from .. import ops
from ..modules.model import MRNNet, _arch, _precision, _train_forward_ran, _writeback_train_pack_bn, sample_drop_scales
from ..utils import Averager, CTCLabelConverter, DevicePrefetcher


def one_cycle_lr(step, total_steps, max_lr, div_factor=20.0, final_div_factor=1000.0, pct_start=0.3):
    """torch.optim.lr_scheduler.OneCycleLR (cosine, two phases) as configured at il_modules/mrn.py:77-84; `step` is the
    number of scheduler.step() calls made so far."""
    initial = max_lr / div_factor
    min_lr = initial / final_div_factor
    end1 = float(pct_start * total_steps) - 1
    end2 = total_steps - 1

    def cos(a, b, pct):
        return b + (a - b) / 2.0 * (math.cos(math.pi * pct) + 1)
    if step <= end1:
        return cos(initial, max_lr, step / end1)
    return cos(max_lr, min_lr, (step - end1) / (end2 - end1))


def L_PREC_TRAIN(opt):
    """Arithmetic mode of the stage-0 step: opt.precision ('fp32' parity mode / 'bf16' tensor-core GEMMs)."""
    return _precision(opt)


def _domain_ids(indexs):
    """get_batch2() returns one index tensor per underlying loader (data/data_manage.py:174-196); the reference
    flattens them with torch.LongTensor(indexs).squeeze() (il_modules/mrn.py:333)."""
    if isinstance(indexs, (list, tuple)) and indexs and isinstance(indexs[0], torch.Tensor):
        return torch.cat([t.reshape(-1) for t in indexs]).to(torch.long).cpu()
    return torch.as_tensor(indexs, dtype=torch.long).reshape(-1).cpu()


def _capture(fn, inputs):
    """CUDA graph of fn(*static), `static` being clones of `inputs`.  Returns the graph-cache entry (graph, static,
    out); `out` is what fn returned, device tensors that every replay overwrites."""
    static = tuple(t.clone() for t in inputs)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fn(*static)
    return graph, static, out


def _replay(entry, inputs):
    """Copies `inputs` into the static inputs of a _capture entry, replays its graph and returns its outputs."""
    graph, static, out = entry
    for dst, src in zip(static, inputs):
        dst.copy_(src, non_blocking=True)
    graph.replay()
    return out


def edit_distance(a, b):
    prev = list(range(len(b) + 1))
    for i, ca in enumerate(a, 1):
        cur = [i]
        for j, cb in enumerate(b, 1):
            cur.append(min(prev[j] + 1, cur[j - 1] + 1, prev[j - 1] + (ca != cb)))
        prev = cur
    return prev[-1]


class RankLocal(torch.nn.Module):
    """Stand-in for nn.DataParallel in the reference (il_modules/mrn.py:106,133): exposes `.module`, forwards calls and
    prefixes state_dict keys with `module.` so reference checkpoints load strict=True.  Parallelism is one process
    per GPU (mrn_b200.dist), not threads in one process."""

    def __init__(self, module):
        super().__init__()
        self.module = module

    def forward(self, *a, **k):
        return self.module(*a, **k)


class FusedAdam:
    """Adam + grad-norm clip over the router arena (fused kernel) with the reference's OneCycleLR bookkeeping
    (built for num_iter * the steps, il_modules/mrn.py:52-88)."""

    def __init__(self, net: MRNNet, lr, total_steps, grad_clip=5.0, schedule="super"):
        self.net = net
        self.max_lr = lr
        self.total_steps = total_steps
        self.grad_clip = grad_clip
        self.schedule = schedule
        arena = net.router_arena()
        self.exp_avg = torch.zeros_like(arena)
        self.exp_avg_sq = torch.zeros_like(arena)
        self.scratch = torch.empty(4096, dtype=torch.uint8, device=arena.device)
        self.norm = torch.zeros(1, dtype=torch.float32, device=arena.device)
        self.steps = 0
        self.param_groups = [{"lr": self.current_lr()}]

    def current_lr(self):
        if "super" in self.schedule:
            return one_cycle_lr(self.steps, self.total_steps, self.max_lr)
        return self.max_lr

    def step(self):
        lr = self.current_lr()
        self.steps += 1
        ops.clip_adam(self.net.router_arena(), self.net.router_grad_arena(), self.exp_avg, self.exp_avg_sq, lr, self.steps,
                      max_norm=self.grad_clip, scratch=self.scratch, norm_out=self.norm)
        self.param_groups[0]["lr"] = self.current_lr()


class ArenaAdam:
    """clip_grad_norm_ + Adam over one flat (params, grads) arena pair with the OneCycleLR bookkeeping of
    il_modules/base.py:84-108 (stage 0: total_steps = num_iter)."""

    def __init__(self, params, grads, lr, total_steps, grad_clip=5.0, schedule="super"):
        self.params, self.grads = params, grads
        self.max_lr, self.total_steps, self.grad_clip, self.schedule = lr, total_steps, grad_clip, schedule
        self.exp_avg = torch.zeros_like(params)
        self.exp_avg_sq = torch.zeros_like(params)
        self.scratch = torch.empty(4096, dtype=torch.uint8, device=params.device)
        self.norm = torch.zeros(1, dtype=torch.float32, device=params.device)
        self.steps = 0
        self.param_groups = [{"lr": self.current_lr()}]

    def current_lr(self):
        if "super" in str(self.schedule):
            return one_cycle_lr(min(self.steps, self.total_steps - 1), self.total_steps, self.max_lr)
        return self.max_lr

    def step(self):
        lr = self.current_lr()
        self.steps += 1
        ops.clip_adam(self.params, self.grads, self.exp_avg, self.exp_avg_sq, lr, self.steps, max_norm=self.grad_clip,
                      scratch=self.scratch, norm_out=self.norm)
        self.param_groups[0]["lr"] = self.current_lr()


class MRN(object):
    def __init__(self, opt):
        self.opt = opt
        self.device = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else None
        if self.device is None:
            raise RuntimeError("mrn_b200.il_modules.mrn.MRN needs a CUDA device (sm_100a); there is no CPU fallback")
        self.model = MRNNet(opt)
        self._known_classes = 0
        self._total_classes = 0
        self._old_network = None
        self.optimizer = None
        self.character = None
        self.converter = None
        self.memory_index = []                 # il_modules/base.py:40: one rehearsal index array per earlier task
        self.pi = 15

    # ---- reference plumbing ------------------------------------------------------------------------
    @property
    def net(self) -> MRNNet:
        return self.model.module if isinstance(self.model, RankLocal) else self.model

    def after_task(self):
        self.model = self.net
        self._known_classes = self._total_classes
        self._old_network = None       # the reference keeps a frozen deepcopy that MRN never reads again (mrn.py:42)

    def build_converter(self):
        converter = CTCLabelConverter(self.character, device=self.device)
        self._total_classes = len(converter.character)
        return converter

    def build_criterion(self, reduction="mean"):
        return "ctc-mean-zero-infinity"      # fused in mrnb_ctc_lattice (il_modules/base.py:131)

    def change_model(self):
        self.model = self.net
        self.model.update_fc(self.opt.hidden_size, self._total_classes)
        self.model.build_prediction(self.opt, self._total_classes)
        self.model = RankLocal(self.model).to(self.device)
        self.model.train()

    def build_model(self):
        self.model.build_fc(self.opt.hidden_size, self._total_classes)
        self.model.build_prediction(self.opt, self._total_classes)
        for name, param in self.model.named_parameters():       # il_modules/mrn.py:117-130
            try:
                if "bias" in name:
                    torch.nn.init.constant_(param, 0.0)
                elif "weight" in name:
                    torch.nn.init.kaiming_normal_(param)
            except Exception:
                if "weight" in name:
                    param.data.fill_(1)
        self.model = RankLocal(self.model).to(self.device)
        self.model.train()

    def count_param(self):
        return [p for p in self.model.parameters() if p.requires_grad]

    def write_log(self, line):
        d = f"./saved_models/{self.opt.exp_name}"
        os.makedirs(d, exist_ok=True)
        with open(os.path.join(d, "log_train.txt"), "a") as f:
            f.write(line)

    def build_custom_optimizer(self, filtered_parameters=None, optimizer="adam", schedule="super", scale=1.0, the=2):
        if optimizer != "adam":
            raise NotImplementedError("the fused optimiser implements Adam (config/svtr_mrn.py optimizer='adam')")
        self.optimizer = FusedAdam(self.net, self.opt.lr * scale, self.opt.num_iter * the,
                                   grad_clip=self.opt.grad_clip, schedule=schedule)
        self.scheduler = self.optimizer
        mdist.broadcast_(self.net.router_arena())     # the freshly built router (modules/model.py:437-452) is rank 0's on every rank

    # ---- training ------------------------------------------------------------------------------------
    def incremental_train(self, taski, character, train_loader, valid_loader):
        self.character = character
        self.converter = self.build_converter()
        if taski > 0:
            self.change_model()
        else:
            self.criterion = self.build_criterion()
            self.build_model()
        if taski > 0:
            for i in range(taski):
                for p in self.net.model[i].parameters():
                    p.requires_grad = False
        self._train(0, taski, train_loader, valid_loader, step=0)
        if taski > 0:
            self._train(0, taski, train_loader, valid_loader, step=1)

    def _train(self, start_iter, taski, train_loader, valid_loader, step=0):
        """il_modules/mrn.py:180-223.  The loader objects follow the reference's protocol when they implement it
        (Dataset_Manager.get_dataset, Val_Dataset.create_dataset / create_list_dataset); plain loaders are used as is."""
        def dataset(memory):
            if hasattr(train_loader, "get_dataset"):
                train_loader.get_dataset(taski, memory=memory)

        def rehearsal():
            if getattr(self.opt, "memory", None) is not None and hasattr(train_loader, "get_dataset") \
                    and hasattr(train_loader, "rehearsal_prev_model"):
                self.build_rehearsal_memory(train_loader, taski)
            else:
                dataset(getattr(self.opt, "memory", None))

        if self.opt.start_task > taski + step * 0.5:
            name = self.opt.lan_list[taski]
            path = f"./saved_models/{self.opt.exp_name}/{name}_{taski}_{step}_best_score.pth"
            mdist.barrier()
            self.model.load_state_dict(torch.load(path, map_location=self.device), strict=True)
            self.net._cache.key = None
            if taski > 0 and step == 0:
                dataset(None)
            elif taski > 0 and step == 1:
                rehearsal()
            return
        single = valid_loader.create_dataset() if hasattr(valid_loader, "create_dataset") else valid_loader
        if taski == 0:
            self._init_train(start_iter, taski, train_loader, single, cross=False)
        elif step == 0:
            dataset(None)
            self.update_step1(start_iter, taski, train_loader, single)
        else:
            rehearsal()
            multi = valid_loader.create_list_dataset() if hasattr(valid_loader, "create_list_dataset") else valid_loader
            self._update_representation(start_iter, taski, train_loader, multi)

    def build_rehearsal_memory(self, train_loader, taski):
        """Random rehearsal memory (il_modules/mrn.py:169-178; il_modules/base.py:292-302): `memory_index` holds one
        index array per earlier task.  Entering stage 1 of task `taski` draws a sample of the task-(taski-1) dataset
        without replacement (numpy global RNG, as the reference) and, when memory_num < 5000, trims every earlier
        task's array so that the total stays at memory_num; the arrays are then handed to the dataset layer."""
        memory_num = int(self.opt.memory_num)
        per_task = memory_num if memory_num >= 5000 else int(memory_num / taski)
        _, n_prev = train_loader.rehearsal_prev_model(taski)
        self.memory_index.append(np.random.choice(range(n_prev), per_task, replace=False))
        if memory_num < 5000 and len(self.memory_index) * len(self.memory_index[0]) > memory_num:
            self.memory_index[:taski] = [ix[:per_task] for ix in self.memory_index[:taski]]
        train_loader.get_dataset(taski, memory=self.opt.memory, index_list=self.memory_index)
        print("Is using rehearsal memory, has {} prev datasets, each has {}\n".format(len(self.memory_index), self.memory_index[0].size))

    # ---- stage 0: the newest expert trained end to end ---------------------------------------------
    def begin_expert_training(self, total_steps=None):
        """Moves the newest expert's parameters into a flat training arena (ops.SvtrTrainPack) and builds the fused
        optimiser over it (Adam + OneCycle over num_iter steps, il_modules/base.py:84-108)."""
        net = self.net
        expert = net.model[-1]
        net._sync_bn()
        sd = {k: v for k, v in expert.state_dict().items()}
        pack_cls = ops.SvtrTrainPack if _arch(net.opt) == "svtr" else ops.CrnnTrainPack
        self._tp = pack_cls(sd, self.device, L_PREC_TRAIN(net.opt))
        self.optimizer = ArenaAdam(self._tp.params, self._tp.grads, self.opt.lr,
                                   int(total_steps or self.opt.num_iter), grad_clip=self.opt.grad_clip,
                                   schedule=getattr(self.opt, "schedule", "super"))
        self.scheduler = self.optimizer
        self._tp_steps = 0
        mdist.broadcast_(self._tp.params)      # replicas start stage 0 from rank 0's weights (per-rank RNG may differ)
        return self._tp

    def end_expert_training(self):
        """Writes the trained arena (and BatchNorm running statistics) back into the expert's nn.Module parameters, so
        that state_dict() / checkpoints / the grouped inference pack see the new weights."""
        tp = self._tp
        expert = self.net.model[-1]
        with torch.no_grad():
            own = dict(expert.named_parameters())
            for key, t in tp.state().items():
                own[key].copy_(t)                       # bumps the version counter -> inference packs are rebuilt
        _writeback_train_pack_bn(expert, tp, self._tp_steps)
        self._tp_steps = 0
        self.net._cache.key = None                      # BN buffers changed without a parameter version bump
        self.reset_graphs()

    def _stage0_device(self, image, labels_index, labels_length, drop_scales=None):
        """Forward of the newest expert (keeping activations), mean CTC loss, full backward into the gradient arena.
        Pure device work on the current stream (capturable in a CUDA graph).  Returns the loss (1-element tensor)."""
        tp = self._tp
        expert = self.net.model[-1]
        train_mode = bool(expert.training)
        B = image.shape[0]
        crnn = tp.arch == "crnn"
        if not crnn and train_mode and drop_scales is None and getattr(self.opt, "drop_path", True):
            rates = expert.model.FeatureExtraction.ConvNet.drop_path_rates()
            drop_scales = sample_drop_scales(1, B, rates, image.device)[0].contiguous()
        image = image.contiguous().float()
        if crnn:
            logits = ops.crnn_train_forward(tp, image, bn_batch_stats=train_mode, update_running=train_mode)
        else:
            logits = ops.svtr_train_forward(tp, image, bn_batch_stats=train_mode, update_running=train_mode,
                                            drop_scales=drop_scales)
        gate = self.__dict__.get("_ones")
        if gate is None or gate.shape[0] != B or gate.device != image.device:
            gate = self._ones = torch.ones(B, 1, device=image.device, dtype=torch.float32)
        r = ops.gate_combine([logits], gate, labels_index, labels_length)        # row log-sum-exp + label gathers
        c = ops.ctc_lattice(r["lpe"], labels_index, labels_length, want_occ=True)
        dlogits = ops.ctc_dense_grad(logits, r["lse"], c["occ"], c["nll"], labels_index, labels_length, 1.0 / B)
        if crnn:
            ops.crnn_train_backward(tp, dlogits, B, bn_batch_stats=train_mode)
        else:
            ops.svtr_train_backward(tp, image, dlogits, bn_batch_stats=train_mode, drop_scales=drop_scales)
        return c["loss"]

    def train_step_stage0(self, image, labels_index, labels_length, drop_scales=None):
        """One expert-training iteration (il_modules/mrn.py:236-267) on the device: forward of the newest expert in its
        current mode (train: BatchNorm batch statistics + DropPath), mean CTC loss, full backward, gradient all-reduce,
        clip + Adam.  Returns the loss as a 1-element device tensor."""
        loss = self._stage0_device(image, labels_index, labels_length, drop_scales)
        mdist.allreduce_mean_(self._tp.grads)            # the ONE exchange step (28 MB; replaces nn.DataParallel)
        self.optimizer.step()                            # clip_grad_norm_(5) + Adam + OneCycle
        if self.net.model[-1].training:
            self._tp_steps += 1
        return loss

    def train_step_stage0_graphed(self, image, labels_index, labels_length):
        """train_step_stage0 with the device work up to the gradients (450 - 740 launches, many of them the tiny
        sequential LSTM steps of a CRNN expert) replayed from a CUDA graph captured per batch size; the gradient
        all-reduce and the optimiser step stay eager.  First call eager (lazy allocations), second captures, later ones
        replay.  DropPath masks are drawn inside the graph by torch's graph-safe generator."""
        B = int(image.shape[0])
        cache = self.__dict__.setdefault("_train_graphs", {})
        key = ("stage0", B, str(image.device), bool(self.net.model[-1].training))
        ent = cache.get(key)
        if ent is None:
            cache[key] = "warm"
            return self.train_step_stage0(image, labels_index, labels_length)
        if ent == "warm":
            ent = cache[key] = _capture(self._stage0_device, (image, labels_index, labels_length))
        loss = _replay(ent, (image, labels_index, labels_length))
        mdist.allreduce_mean_(self._tp.grads)
        self.optimizer.step()
        if key[3]:
            self._tp_steps += 1
        return loss

    def _init_train(self, start_iter, taski, train_loader, valid_loader, cross=False):
        """il_modules/mrn.py:225-279."""
        train_loss_avg = Averager()
        start_time = time.time()
        best_score = -1
        self.begin_expert_training()
        pf = DevicePrefetcher(self.device)

        def stage(batch):
            image_tensors, labels = batch
            li, ll = self.converter.encode(labels, batch_max_length=self.opt.batch_max_length, device="cpu")
            pf.submit((image_tensors, li, ll))
        if start_iter + 1 <= self.opt.num_iter:
            stage(train_loader.get_batch())
        for iteration in range(start_iter + 1, self.opt.num_iter + 1):
            image, labels_index, labels_length = pf.take()
            if iteration < self.opt.num_iter:
                stage(train_loader.get_batch())             # H2D of the next batch overlaps this step's kernels
            step = self.train_step_stage0_graphed if getattr(self.opt, "cuda_graph", True) else self.train_step_stage0
            loss = step(image, labels_index, labels_length)
            train_loss_avg.add(loss)
            if iteration % self.opt.val_interval == 0 or iteration == self.opt.num_iter:
                self.end_expert_training()
                self.val(valid_loader, self.opt, best_score, start_time, iteration, train_loss_avg, None, taski, 0, "FF")
                train_loss_avg.reset()
        self.end_expert_training()

    def update_step1(self, start_iter, taski, train_loader, valid_loader):
        self._init_train(start_iter, taski, train_loader, valid_loader, cross=False)
        for p in self.net.model[-1].parameters():       # il_modules/mrn.py:284-287
            p.requires_grad = False
        self.net.model[-1].eval()

    def model_eval_and_train(self, taski):
        """il_modules/mrn.py:45-50 (only reached from the reference's commented-out call sites; kept for interface
        parity): everything in train mode, then the experts of the earlier tasks in eval mode."""
        self.model.train()
        self.net.model[-1].train()
        for i in range(taski if taski >= 1 else 0):
            self.net.model[i].eval()

    def freeze_step1(self, taski):
        """il_modules/mrn.py:289-295 (dead code in the reference's MRN loop, mirrored for completeness): modes as in
        `model_eval_and_train`, then the newest expert frozen and in eval mode."""
        self.model_eval_and_train(taski)
        self.model.train()
        for p in self.net.model[-1].parameters():
            p.requires_grad = False
        self.net.model[-1].eval()

    def _stage1_device(self, image, labels_index, labels_length, indexs, drop_scales=None):
        """Experts, router forward, fused combine + CTC, analytic gate gradient and router backward into the router's
        gradient arena.  Pure device work on the current stream (capturable in a CUDA graph).  Returns (loss_clf,
        taski_loss) as 1-element tensors."""
        net = self.net
        B = image.shape[0]
        r = net.route_and_combine(image, is_train=True, want_logits=False, targets=labels_index, lengths=labels_length,
                                  want_E=True, with_backward=True, drop_scales=drop_scales)
        c = ops.ctc_lattice(r["lpe"], labels_index, labels_length, r["zlab"], r["E"], grad_scale=float(self.pi) / B,
                            want_dgate=True)
        taski_loss = ops.router_backward(net.router_arena(), r["features"], r["gate"], c["dgate"], indexs,
                                         net.router_grad_arena(), net._rws, prec=_precision(net.opt))
        return c["loss"], taski_loss

    def train_step_stage1(self, image, labels_index, labels_length, indexs, drop_scales=None):
        """One router-training iteration (il_modules/mrn.py:338-371) entirely on the device.
        image [B,4,32,256] fp32, labels_index [B,25] int64 (pad 1), labels_length [B] int32, indexs [B] int64.
        Returns (loss_clf, taski_loss) as 1-element device tensors."""
        loss, taski_loss = self._stage1_device(image, labels_index, labels_length, indexs, drop_scales)
        mdist.allreduce_mean_(self.net.router_grad_arena())     # the ONE exchange step (replaces nn.DataParallel)
        self.optimizer.step()                            # clip_grad_norm_(5) + Adam + OneCycle
        return loss, taski_loss

    def train_step_stage1_graphed(self, image, labels_index, labels_length, indexs):
        """train_step_stage1 with the device work up to the router gradients (experts, router forward, combine + CTC,
        router backward: ~115 launches) replayed from a CUDA graph captured per batch size; the gradient all-reduce
        and the optimiser step stay eager (NCCL and the host-side OneCycle schedule are not captured).  The first call
        for a batch size runs eagerly (lazy allocations, attribute setup), the second captures, later ones replay.
        Steady-state loop only: re-capture (`reset_graphs()`) after the experts' weights or train / eval mode change."""
        net = self.net
        modes = net._experts_train_mode()
        cache = self.__dict__.setdefault("_train_graphs", {})
        key = (int(image.shape[0]), str(image.device), modes)
        ent = cache.get(key)
        if ent is None:
            cache[key] = "warm"
            return self.train_step_stage1(image, labels_index, labels_length, indexs)
        if ent == "warm":
            ent = cache[key] = _capture(self._stage1_device, (image, labels_index, labels_length, indexs))
        loss, taski_loss = _replay(ent, (image, labels_index, labels_length, indexs))
        if any(modes) and net._cache.pack is not None:
            _train_forward_ran(net._cache, list(net.model), modes)
        mdist.allreduce_mean_(net.router_grad_arena())
        self.optimizer.step()
        return loss, taski_loss

    def reset_graphs(self):
        self.__dict__.pop("_train_graphs", None)
        self.__dict__.pop("_infer_graphs", None)

    def _update_representation(self, start_iter, taski, train_loader, valid_loader, pi=15):
        self.pi = pi
        train_loss_avg, train_taski_loss_avg = Averager(), Averager()
        for p in self.net.model.parameters():
            p.requires_grad = False
        self.build_custom_optimizer(None, optimizer="adam", schedule="super", scale=1, the=2)
        start_time = time.time()
        best_score = -1
        n_iter = int(self.opt.num_iter // 2)
        pf = DevicePrefetcher(self.device)

        def stage(batch):
            image_tensors, labels, indexs = batch
            li, ll = self.converter.encode(labels, batch_max_length=self.opt.batch_max_length, device="cpu")
            # images come pinned from a DataLoader(pin_memory=True) (then the copy overlaps the running step); pageable
            # batches are copied synchronously by the driver -- pinning 33 MB per step here would cost more than it saves
            pf.submit((image_tensors, li, ll, _domain_ids(indexs)))
        if start_iter + 1 <= n_iter:
            stage(train_loader.get_batch2())
        for iteration in range(start_iter + 1, n_iter + 1):
            image, labels_index, labels_length, indexs = pf.take()
            if iteration < n_iter:
                stage(train_loader.get_batch2())            # H2D of the next batch overlaps this step's kernels
            loss_clf, taski_loss = self.train_step_stage1(image, labels_index, labels_length, indexs)
            train_loss_avg.add(loss_clf)
            train_taski_loss_avg.add(taski_loss)
            if iteration % (self.opt.val_interval // 5) == 0 or iteration == n_iter or iteration == 1:
                self.val(valid_loader, self.opt, best_score, start_time, iteration, train_loss_avg, train_taski_loss_avg,
                         taski, step=1, val_choose="TF")
                train_loss_avg.reset()
                train_taski_loss_avg.reset()

    # ---- evaluation ----------------------------------------------------------------------------------
    def infer_batch(self, image, val_choose="TF", labels_index=None, labels_length=None, decode="greedy", beam_width=8,
                    beam_topk=16, n_best=1):
        """Hard-routed (TF) or last-expert (FF) inference + device-side decode.
        Returns dict(ids, lens, conf, index, loss) -- ids compact [B,T] (-1 padded).
        decode="greedy": best path (test.py:211-221).  decode="beam": CTC prefix beam search of width beam_width over the
        beam_topk best classes of every frame; ids / lens / conf = exp(score) are the best labeling's, and n_best > 1 adds
        nbest_ids [B,n_best,T], nbest_lens [B,n_best] and nbest_scores [B,n_best] (log-probabilities, best first)."""
        if decode not in ("greedy", "beam"):
            raise ValueError("decode must be 'greedy' or 'beam', got %r" % (decode,))
        beam = decode == "beam"
        net = self.net
        if val_choose == "FF":
            out = net(image, cross=False, is_train=False)
            gate = torch.ones(image.shape[0], 1, device=image.device)
            r = ops.gate_combine([out["logits"]], gate, labels_index, labels_length, want_decode=not beam)
            experts, index = [out["logits"]], None
        else:
            r = net.route_and_combine(image, is_train=False, want_logits=False, targets=labels_index, lengths=labels_length,
                                      want_decode=not beam)
            experts, gate, index = r["expert_logits"], r["combine_gate"], r["index"]
        loss = None
        if labels_index is not None:
            loss = ops.ctc_lattice(r["lpe"], labels_index, labels_length)["loss"]
        if not beam:
            ids, lens, conf = ops.greedy_decode(r["amax"], r["maxprob"])
            return dict(ids=ids, lens=lens, conf=conf, index=index, loss=loss)
        top_ids, top_lp, blank_lp = ops.ctc_topk(experts, gate, r["lse"], beam_topk)
        nb_ids, nb_lens, nb_scores = ops.ctc_beam_search(top_ids, top_lp, blank_lp, beam_width, n_best)
        res = dict(ids=nb_ids[:, 0], lens=nb_lens[:, 0], conf=nb_scores[:, 0].exp(), index=index, loss=loss)
        if n_best > 1:
            res.update(nbest_ids=nb_ids, nbest_lens=nb_lens, nbest_scores=nb_scores)
        return res

    def infer_batch_graphed(self, image, val_choose="TF", decode="greedy", beam_width=8, beam_topk=16, n_best=1):
        """infer_batch replayed from a CUDA graph captured per (batch size, route, decode settings): small batches are launch-bound
        (~95 kernels), and a replay costs one launch.  The graph owns static input / output buffers; the returned
        tensors are views of the static outputs and stay valid until the next replay for the same batch size.
        Eval-mode experts only (train-mode BatchNorm / DropPath state is not captured)."""
        if any(self.net._experts_train_mode()):
            raise RuntimeError("infer_batch_graphed needs eval-mode experts (call model.eval() first)")
        dec = dict(decode=decode, beam_width=beam_width, beam_topk=beam_topk, n_best=n_best)
        key = (int(image.shape[0]), val_choose, str(image.device)) + tuple(dec.values())
        cache = self.__dict__.setdefault("_infer_graphs", {})
        ent = cache.get(key)
        if ent is None:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):             # warm-up on a side stream: lazy allocations, attribute setup, packs
                for _ in range(2):
                    self.infer_batch(image, val_choose, **dec)
            torch.cuda.current_stream().wait_stream(side)
            ent = cache[key] = _capture(lambda x: self.infer_batch(x, val_choose, **dec), (image,))
        return _replay(ent, (image,))

    def validation(self, eval_loader, val_choose="TF"):
        """test.py:139-279 with the decode / confidence on the device.  opt.decode ("greedy", the default, or "beam"),
        opt.beam_width (8) and opt.beam_topk (16) choose the decoder; a config without them decodes greedily."""
        dec = dict(decode=getattr(self.opt, "decode", "greedy"), beam_width=int(getattr(self.opt, "beam_width", 8)),
                   beam_topk=int(getattr(self.opt, "beam_topk", 16)))
        n_correct, norm_ED, length_of_data, infer_time = 0, 0.0, 0, 0.0
        valid_loss_avg = Averager()
        preds_str, confidence, labels = [], [], []
        for image_tensors, labels in eval_loader:
            bs = image_tensors.size(0)
            length_of_data += bs
            image = image_tensors.to(self.device, non_blocking=True)
            labels_index, labels_length = self.converter.encode(labels, batch_max_length=self.opt.batch_max_length)
            t0 = time.time()
            r = self.infer_batch(image, val_choose, labels_index, labels_length, **dec)
            preds_str = self.converter.decode_compact(r["ids"], r["lens"])       # the batch's single D2H sync
            infer_time += time.time() - t0
            valid_loss_avg.add(r["loss"])
            confidence = r["conf"].cpu().tolist()
            for gt, prd in zip(labels, preds_str):
                if getattr(self.opt, "NED", True):
                    if len(gt) == 0 or len(prd) == 0:
                        norm_ED += 0
                    elif len(gt) > len(prd):
                        norm_ED += 1 - edit_distance(prd, gt) / len(gt)
                    else:
                        norm_ED += 1 - edit_distance(prd, gt) / len(prd)
                if prd == gt:
                    n_correct += 1
        n = max(length_of_data, 1)
        return (valid_loss_avg.val(), n_correct / float(n) * 100, norm_ED / float(n) * 100, preds_str, confidence, labels,
                infer_time, length_of_data)

    def val(self, valid_loader, opt, best_score, start_time, iteration, train_loss_avg, train_taski_loss_avg, taski, step,
            val_choose="val"):
        self.model.eval()
        t0 = time.time()
        (valid_loss, current_score, ned_score, preds, confidence_score, labels, infer_time, n) = \
            self.validation(valid_loader, val_choose=val_choose)
        self.model.train()                    # reference quirk 4: puts frozen experts back in train mode (mrn.py:401)
        if current_score > best_score:
            best_score = current_score
            os.makedirs(f"./saved_models/{opt.exp_name}", exist_ok=True)
            if mdist.env_world()[0] == 0:
                torch.save(self.model.state_dict(),
                           f"./saved_models/{opt.exp_name}/{opt.lan_list[taski]}_{taski}_{step}_best_score.pth")
            mdist.barrier()                   # no rank reads the checkpoint before rank 0 has finished writing it
        lr = self.optimizer.param_groups[0]["lr"] if self.optimizer else 0.0
        log = (f"\n[{iteration}/{opt.num_iter}] Train_loss_clf: {train_loss_avg.val():0.5f}, Valid_loss: {valid_loss:0.5f} \n "
               + (f'{"":9s}Train_taski_loss: {train_taski_loss_avg.val():0.5f}\n' if train_taski_loss_avg is not None else "")
               + f'{"":9s}Current_score: {current_score:0.2f}, Ned_score: {ned_score:0.2f}\n'
               + f'{"":9s}Current_lr: {lr:0.7f}, Best_score: {best_score:0.2f}\n'
               + f'{"":9s}Infer_time: {infer_time:0.2f},     Elapsed_time: {(time.time() - t0) / max(n, 1) * 1000:0.2f}\n')
        print(log)
        self.write_log(log + "\n")
        return current_score

    def test(self, AlignCollate_valid, valid_datas, best_scores, ned_scores, taski, val_choose="test"):
        """il_modules/mrn.py:448-515: reload the best checkpoint of the task (strict=True), evaluate every benchmark set
        with the last expert (task 0, "FF") or the hard route (later tasks, "TF"), append the averages.

        valid_datas: list of loaders -- iterables of (images [B,4,32,256], label strings).  (The reference builds them
        from LMDB paths with hierarchical_dataset + AlignCollate_valid; that dataset layer is outside the hot path,
        SURVEY.md §8f.2, so the caller passes the loaders; AlignCollate_valid is accepted and unused.)"""
        val_choose, step = ("FF", 0) if taski == 0 else ("TF", 1)
        os.makedirs(f"./result/{self.opt.exp_name}", exist_ok=True)
        name = self.opt.lan_list[taski]
        path = f"./saved_models/{self.opt.exp_name}/{name}_{taski}_{step}_best_score.pth"
        if not isinstance(self.model, RankLocal):
            self.model = RankLocal(self.net).to(self.device)
        mdist.barrier()
        self.model.load_state_dict(torch.load(path, map_location=self.device), strict=True)
        self.net._cache.key = None
        self.reset_graphs()
        task_accs, ned_accs = [], []
        self.model.eval()
        for loader in valid_datas:
            _, current_score, ned_score, *_ = self.validation(loader, val_choose=val_choose)
            task_accs.append(round(current_score, 2))
            ned_accs.append(round(ned_score, 2))
        if (taski + 1) * 2 == len(task_accs):            # MLT17 / MLT19 pairs (double_write, il_modules/base.py)
            score17 = round(sum(task_accs[0::2]) / len(task_accs[0::2]), 2)
            score19 = round(sum(task_accs[1::2]) / len(task_accs[1::2]), 2)
            best_scores.append(score17)
            ned_scores.append(score19)
            acc_log = f"Task {taski} Avg Incremental Acc:  17: {score17}    19: {score19}\n"
        else:
            best_scores.append(round(sum(task_accs) / max(len(task_accs), 1), 2))
            ned_scores.append(round(sum(ned_accs) / max(len(ned_accs), 1), 2))
            acc_log = (f"Task {taski} Test Average Incremental Accuracy: {best_scores[taski]} \n Task {taski} Incremental "
                       f"Accuracy: {task_accs}\n ned_acc: {ned_accs}\n")
        self.write_log(acc_log)
        print(acc_log)
        return best_scores, ned_scores
