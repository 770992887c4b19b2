"""MRNNet / Model / Model_Extractor with the reference's constructor arguments, methods, attribute names and
state_dict keys (modules/model.py:17-199,314-496), computing through the CUDA library.

Scope (SURVEY.md §8): Prediction="CTC", Transformation="None" with either FeatureExtraction="SVTR" /
SequenceModeling="None" (config/svtr_mrn.py, T = 64) or FeatureExtraction="VGG" / SequenceModeling="BiLSTM"
(config/crnn_mrn.py, T = 63).  Other stages raise NotImplementedError -- there is no PyTorch fallback.

The nn.Module tree exists to own parameters under the reference's names (checkpoints load strict=True,
il_modules/mrn.py:190,465).  Compute never runs per module:
  * experts: one grouped launch sequence over all experts (ops.svtr_experts_forward) fed by an expert-stacked
    SvtrPack that is rebuilt when expert parameters change;
  * router: route / channel_route / dm_router parameters are views into ONE flat fp32 arena (also the gradient,
    Adam and NCCL all-reduce layout).
"""
import copy
from typing import List, Optional

import torch
import torch.nn as nn

from .. import _lib as L
from .. import ops
from .dm_router import DM_Router
from .crnn import BidirectionalLSTM, VGG_FeatureExtractor
from .svtr import SVTR_FeatureExtractor


def _arch(opt):
    """'svtr' (SVTR / None / CTC) or 'crnn' (VGG / BiLSTM / CTC); anything else is outside the implemented path."""
    ok_common = opt.Prediction == "CTC" and opt.Transformation in ("None", None)
    if ok_common and opt.FeatureExtraction == "SVTR" and opt.SequenceModeling != "BiLSTM":
        return "svtr"
    if ok_common and opt.FeatureExtraction == "VGG" and opt.SequenceModeling == "BiLSTM":
        return "crnn"
    raise NotImplementedError(
        "mrn_b200 implements the SVTR / None / CTC (config/svtr_mrn.py) and VGG / BiLSTM / CTC (config/crnn_mrn.py) "
        "hot paths; got %s/%s/%s/%s. No PyTorch fallback is provided."
        % (opt.Transformation, opt.FeatureExtraction, opt.SequenceModeling, opt.Prediction))


def _require_svtr_ctc(opt):
    _arch(opt)


class Model_Extractor(nn.Module):
    """modules/model.py:17-101 (parameter holder)."""

    def __init__(self, opt):
        super().__init__()
        _require_svtr_ctc(opt)
        self.opt = opt
        self.stages = {"Trans": opt.Transformation, "Feat": opt.FeatureExtraction, "Seq": opt.SequenceModeling,
                       "Pred": opt.Prediction}
        self.FeatureExtraction_output = opt.output_channel
        if _arch(opt) == "svtr":
            self.FeatureExtraction = SVTR_FeatureExtractor(opt.input_channel, opt.output_channel)
            self.SequenceModeling = nn.Sequential(nn.Linear(self.FeatureExtraction_output, opt.hidden_size))
        else:
            self.FeatureExtraction = VGG_FeatureExtractor(opt.input_channel, opt.output_channel)
            self.SequenceModeling = nn.Sequential(
                BidirectionalLSTM(self.FeatureExtraction_output, opt.hidden_size, opt.hidden_size),
                BidirectionalLSTM(opt.hidden_size, opt.hidden_size, opt.hidden_size))
        self.SequenceModeling_output = opt.hidden_size


class Model(nn.Module):
    """One expert recogniser (modules/model.py:105-199)."""

    def __init__(self, opt):
        super().__init__()
        self.opt = opt
        self.model = Model_Extractor(opt)
        self.SequenceModeling_output = self.model.SequenceModeling_output
        self.stages = {"Pred": opt.Prediction}
        self.fc = None
        self.Prediction = None
        self._solo: Optional["MRNNet"] = None

    def new_fc(self, hidden_size, nb_classes):
        self.fc = nn.Linear(hidden_size, nb_classes)

    def update_fc(self, hidden_size, nb_classes, device=None):
        fc = nn.Linear(hidden_size, nb_classes)
        if self.fc is not None:
            nb_output = self.fc.out_features
            fc.weight.data[:nb_output] = copy.deepcopy(self.fc.weight.data)
            fc.bias.data[:nb_output] = copy.deepcopy(self.fc.bias.data)
        self.fc = fc

    def build_prediction(self, opt, num_class):
        if opt.Prediction != "CTC":
            raise NotImplementedError("only the CTC head is implemented")
        self.Prediction = self.fc          # same object: state_dict carries fc.* and Prediction.* (model.py:181)

    def weight_align(self, increment):
        weights = self.fc.weight.data
        newnorm = torch.norm(weights[-increment:, :], p=2, dim=1)
        oldnorm = torch.norm(weights[:-increment, :], p=2, dim=1)
        gamma = torch.mean(oldnorm) / torch.mean(newnorm)
        self.fc.weight.data[-increment:, :] *= gamma

    def forward(self, image, text=None, is_train=True):
        """-> {"predict": [B,T,C], "feature": [B,T,256]} (modules/model.py:133-148) via a single-expert pack.
        With opt.autograd and grad mode on, "predict" and "feature" are differentiable with respect to every parameter
        and to the image (training-pack forward, see _expert_autograd_forward)."""
        if _autograd_on(self.opt):
            predict, feature = _expert_autograd_forward(self, image, self.opt, want_features=True)
            return {"predict": predict, "feature": feature}
        feats, logits = _experts_forward([self], image, self.opt, train_mode=self.training)
        return {"predict": logits[0], "feature": feats[:, 0]}

    def copy(self):
        return copy.deepcopy(self)

    def freeze(self):
        for p in self.parameters():
            p.requires_grad = False
        self.eval()
        return self


# ------------------------------------------------------------------------------------------------
class _PackCache:
    """SvtrPack keyed by the experts' parameter versions (rebuilt after an optimizer step / load_state_dict)."""

    def __init__(self):
        self.key = None
        self.pack: Optional[ops.SvtrPack] = None

    def get(self, experts: List[Model], device, prec):
        # parameters only: BN running statistics are owned by the pack between checkpoints (see _sync_bn)
        arch = _arch(experts[0].opt)
        key = (arch, prec, str(device), tuple(id(m) for m in experts),
               sum(int(p._version) for m in experts for p in m.parameters()))
        if key != self.key:
            sd = {}
            for i, m in enumerate(experts):
                for k, v in m.state_dict().items():
                    sd[f"model.{i}.{k}"] = v
            self.pack = (ops.SvtrPack if arch == "svtr" else ops.CrnnPack)(sd, len(experts), device, prec)
            self.key = key
        return self.pack


_solo_cache = _PackCache()


def _precision(opt):
    p = getattr(opt, "precision", "fp32")
    return L.PREC_BF16 if str(p).lower() in ("bf16", "bfloat16") else L.PREC_FP32


def _count_bn_steps(pack, modes):
    steps = getattr(pack, "bn_steps", None)
    if steps is None or len(steps) != len(modes):
        steps = pack.bn_steps = [0] * len(modes)
    for e, t in enumerate(modes):
        steps[e] += int(bool(t))


def _mode_mask(train_mode, n):
    """Per-expert train / eval modes -> bit mask (bit e = expert e in .train()).  A bool applies to every expert."""
    if isinstance(train_mode, (bool, int)):
        return ((1 << n) - 1) if train_mode else 0
    return sum(1 << e for e, t in enumerate(train_mode) if t)


def _experts_forward(experts, image, opt, train_mode, cache=None, drop_scales=None, want_logits=True, chunk=None):
    """train_mode: bool or one bool per expert (the reference can hold experts in different modes: after update_step1
    the newest expert is .eval() while the frozen older ones are still .train(), il_modules/mrn.py:284-287 vs :107)."""
    if not image.is_cuda:
        raise RuntimeError("mrn_b200 needs CUDA tensors: there is no CPU fallback")
    cache = cache or _solo_cache
    pack = cache.get(experts, image.device, _precision(opt))
    modes = [bool(train_mode)] * len(experts) if isinstance(train_mode, (bool, int)) else [bool(t) for t in train_mode]
    mask = _mode_mask(modes, len(experts))
    train_mode = mask != 0
    if pack.arch == "crnn":
        feats, logits = ops.crnn_experts_forward(pack, image.contiguous().float(), bn_batch_stats=mask,
                                                 update_running=mask, want_logits=want_logits)
        if train_mode:
            _train_forward_ran(cache, experts, modes)
        return feats, logits
    if chunk is None:
        chunk = int(getattr(opt, "expert_chunk", 0) or 0)
    if train_mode and drop_scales is None and getattr(opt, "drop_path", True):
        drop_scales = sample_drop_scales(len(experts), image.shape[0], experts[0].model.FeatureExtraction.ConvNet.drop_path_rates(),
                                         image.device)
        if not all(modes):                  # DropPath is the identity for the experts that are in .eval()
            for e, t in enumerate(modes):
                if not t:
                    drop_scales[e].fill_(1.0)
    feats, logits = ops.svtr_experts_forward(pack, image.contiguous().float(), bn_batch_stats=mask,
                                             update_running=mask, drop_scales=drop_scales, chunk=chunk,
                                             want_logits=want_logits)
    if train_mode:
        _train_forward_ran(cache, experts, modes)
    return feats, logits


def _train_forward_ran(cache, experts, modes):
    """Bookkeeping after an expert forward (eager or replayed from a CUDA graph) in which the experts flagged in
    `modes` were in .train(): their BN running statistics changed inside cache.pack.  The solo cache (single-expert
    forwards) belongs to no MRNNet whose state_dict() would sync it, so its experts' buffers are written back at once."""
    cache.pack.bn_dirty = True
    _count_bn_steps(cache.pack, modes)
    if cache is _solo_cache:
        _writeback_bn(experts, cache.pack)


def _autograd_on(opt):
    """opt.autograd (absent = False) and torch grad mode: the forwards build an autograd graph over the kernels."""
    return bool(getattr(opt, "autograd", False)) and torch.is_grad_enabled()


def _writeback_train_pack_bn(expert, tp, n_fwd):
    """A training pack's BatchNorm running statistics -> the expert's buffers, after `n_fwd` train-mode forwards."""
    with torch.no_grad():
        m0, v0, m1, v1 = tp.bn_running_stats()
        for bn, mean, var in zip(_expert_bns(expert, tp.arch), (m0, m1), (v0, v1)):
            bn.running_mean.copy_(mean.reshape(-1))
            bn.running_var.copy_(var.reshape(-1))
            bn.num_batches_tracked += n_fwd


def _train_pack_run(expert, x, opt, net=None, drop=None, want_features=False, param_grads=True):
    """One expert's training-pack forward, the step autograd differentiates (opt.autograd): ops.SvtrTrainPack /
    ops.CrnnTrainPack built from the expert's state_dict, run in the expert's current mode -- in .train() BatchNorm batch
    statistics with the running-statistics update (written back to the expert's buffers once, here) and DropPath `drop`
    [12,2,B] (None: drawn as the default forward draws it).  Returns (logits, features or None, backward);
    backward(dlogits, dfeatures=None, dimage=False) runs the pack's backward and returns (grads, dimage): grads =
    {state_dict key: gradient in the reference layout} (views of the pack's gradient arena), dimage = d loss / d image
    [B,4,32,256] when asked for.  param_grads=False (a frozen expert that only carries the image gradient): the pack has
    no gradient arena, the backward is the input-only one and grads is None."""
    arch = _arch(opt)
    tp = (ops.SvtrTrainPack if arch == "svtr" else ops.CrnnTrainPack)(expert.state_dict(), x.device, _precision(opt),
                                                                      param_grads=param_grads)
    train = bool(expert.training)
    x = x.contiguous().float()
    B = x.shape[0]
    if arch == "crnn":
        out = ops.crnn_train_forward(tp, x, bn_batch_stats=train, update_running=train, want_features=want_features)
    else:
        if drop is None and train and getattr(opt, "drop_path", True):
            rates = expert.model.FeatureExtraction.ConvNet.drop_path_rates()
            drop = sample_drop_scales(1, B, rates, x.device)[0].contiguous()
        out = ops.svtr_train_forward(tp, x, bn_batch_stats=train, update_running=train, drop_scales=drop,
                                     want_features=want_features)
    logits, feats = out if want_features else (out, None)
    if train:
        _writeback_train_pack_bn(expert, tp, 1)
        _solo_cache.key = None              # packs hold BN statistics: rebuild them from the updated buffers
        if net is not None:
            net._cache.key = None

    def backward(dlogits, dfeatures=None, dimage=False):
        if not (param_grads or dimage):
            return None, None
        di = torch.empty(B, 4, 32, 256, device=x.device, dtype=torch.float32) if dimage else None
        if arch == "crnn":
            ops.crnn_train_backward(tp, dlogits, B, bn_batch_stats=train, dfeatures=dfeatures, dimage=di,
                                    param_grads=param_grads)
        else:
            ops.svtr_train_backward(tp, x, dlogits, bn_batch_stats=train, drop_scales=drop, dfeatures=dfeatures, dimage=di,
                                    param_grads=param_grads)
        return (tp.state(tp.grads) if param_grads else None), di
    return logits, feats, backward


def _expert_autograd_forward(expert, image, opt, net=None, want_features=False):
    """Forward of one expert that autograd differentiates (opt.autograd): _train_pack_run and, on backward, the pack's
    backward, mapped back to every parameter by the pack's arena <-> state_dict table, and the image gradient when the
    image requires grad.  Returns logits, or (logits, features) with want_features."""
    if not image.is_cuda:
        raise RuntimeError("mrn_b200 needs CUDA tensors: there is no CPU fallback")
    from ..autograd import ExpertTrain
    if net is not None:
        net._sync_bn()                      # BN statistics the grouped pack still holds -> the module buffers
    named = list(expert.named_parameters())
    return ExpertTrain.apply(lambda x, **kw: _train_pack_run(expert, x, opt, net=net, **kw), [n for n, _ in named],
                             want_features, image, *[p for _, p in named])


_RATES_CACHE = {}


def sample_drop_scales(n_experts, B, rates, device, generator=None):
    """DropPath multipliers [I,12,2,B]: Bernoulli(keep)/keep per sample, block and branch (modules/svtr.py:7-22)."""
    key = (tuple(float(r) for r in rates), str(device))
    rates_t = _RATES_CACHE.get(key)
    if rates_t is None:                     # device-resident once: no host-to-device copy per step (CUDA-graph safe)
        rates_t = _RATES_CACHE[key] = torch.tensor(rates, dtype=torch.float32, device=device).view(1, -1, 1, 1)
    u = torch.rand(n_experts, len(rates), 2, B, device=device, generator=generator)
    keep = (u >= rates_t).float()
    return (keep / (1.0 - rates_t)).contiguous()


def _expert_bns(expert, arch):
    """The expert's two BatchNorm2d modules: VGG's after conv4 and conv5 (crnn), the patch embedding's two (svtr)."""
    cn = expert.model.FeatureExtraction.ConvNet
    return (cn[12], cn[15]) if arch == "crnn" else (cn.patch_embed.proj[1], cn.patch_embed.proj[4])


def _writeback_bn(experts, pack):
    """Train-mode forwards update BN running statistics inside the pack; mirror them into the module buffers so
    state_dict() / checkpoints see what nn.BatchNorm2d in .train() would have produced (reference quirk 4)."""
    m0, v0, m1, v1 = pack.bn_running_stats()
    with torch.no_grad():
        for i, m in enumerate(experts):
            bns = _expert_bns(m, pack.arch)
            steps = getattr(pack, "bn_steps", None)
            n_fwd = steps[i] if steps is not None else 1     # train-mode forwards of this expert since the last write-back
            if n_fwd == 0:
                continue
            for bn, mean, var in ((bns[0], m0, v0), (bns[1], m1, v1)):
                bn.running_mean.data = mean[i].clone()
                bn.running_var.data = var[i].clone()
                bn.num_batches_tracked += n_fwd
    pack.bn_steps = [0] * len(experts)
    pack.bn_dirty = False


class MRNNet(nn.Module):
    """Multiplexed routing network (modules/model.py:314-496)."""

    def __init__(self, opt):
        super().__init__()
        _require_svtr_ctc(opt)
        self.model = nn.ModuleList()
        self.out_dim = None
        self.fc = None
        self.opt = opt
        self.task_sizes = []
        self.patch = 64 if _arch(opt) == "svtr" else 63      # modules/model.py:322-325
        self.router = "dm-router"
        self.layer_num = 1
        self.beta = 1
        self._cache = _PackCache()
        self._frozen_cache = _PackCache()   # the frozen experts' grouped pack when some experts train (opt.autograd_experts)
        self._arena: Optional[torch.Tensor] = None
        self._grad_arena: Optional[torch.Tensor] = None
        self._rws = ops.RouterWorkspace()

    # -- reference API ---------------------------------------------------------------------------
    @property
    def feature_dim(self):
        return 0 if self.out_dim is None else self.out_dim * len(self.model)

    def build_fc(self, hidden_size, nb_classes):
        self.update_fc(hidden_size, nb_classes)

    def update_fc(self, hidden_size, nb_classes):
        """Adds an expert and REBUILDS the router for the new expert count (modules/model.py:428-452)."""
        self.model.append(Model(self.opt))
        self.model[-1].new_fc(hidden_size, nb_classes)
        if self.out_dim is None:
            self.out_dim = self.model[-1].SequenceModeling_output
        self.route = nn.Linear(self.patch, 1)
        self.channel_route = nn.Linear(self.feature_dim, len(self.model))
        block = DM_Router(self.out_dim, self.out_dim * 2, self.patch, len(self.model),
                          autograd=bool(getattr(self.opt, "autograd", False)))
        self.dm_router = nn.Sequential(*[block for _ in range(self.layer_num)])
        self._arena = None
        self._grad_arena = None

    def build_prediction(self, opt, num_class):
        self.model[-1].build_prediction(opt, num_class)

    def load_fc(self, input, output):
        fc = nn.Linear(input, output)
        if self.channel_route is not None:
            nb_output = self.channel_route.out_features
            fc.weight.data[:nb_output, :self.feature_dim - self.out_dim] = copy.deepcopy(self.channel_route.weight.data)
            fc.bias.data[:nb_output] = copy.deepcopy(self.channel_route.bias.data)
        self.fc = fc

    def copy(self):
        return copy.deepcopy(self)

    def freeze(self):
        for p in self.parameters():
            p.requires_grad = False
        self.eval()
        return self

    def softargmax1d(self, input, beta=5):
        return nn.functional.softmax(beta * input, dim=-1)

    def extract_vector(self, x):
        feats, _ = _experts_forward(list(self.model), x, self.opt, self._experts_train_mode(), self._cache, want_logits=False)
        return feats.permute(0, 2, 1, 3).reshape(x.shape[0], self.patch, -1)

    # -- router arena ----------------------------------------------------------------------------
    def router_parameters(self):
        sd = dict(self.named_parameters())
        return [sd[n] for n in ops.ROUTER_PARAM_NAMES]

    def router_arena(self, device=None):
        """Flat fp32 arena holding every router parameter (C-ABI order); parameters become views into it."""
        params = self.router_parameters()
        device = torch.device(device) if device is not None else params[0].device
        n, off = ops.router_param_offsets(len(self.model), self.patch, self.out_dim)
        ok = self._arena is not None and self._arena.device == device and all(
            p.data_ptr() == self._arena.data_ptr() + 4 * off[k] for k, p in enumerate(params))
        if not ok:
            arena = torch.zeros(n, dtype=torch.float32, device=device)      # slots are padded to 8 floats
            for k, p in enumerate(params):
                arena[off[k]:off[k] + p.numel()] = p.data.reshape(-1).to(device)
                p.data = arena[off[k]:off[k] + p.numel()].view(p.shape)
            self._arena = arena
            self._grad_arena = None
        return self._arena

    def router_grad_arena(self):
        arena = self.router_arena()
        if self._grad_arena is None:
            n, off = ops.router_param_offsets(len(self.model), self.patch, self.out_dim)
            self._grad_arena = torch.zeros_like(arena)
            for k, p in enumerate(self.router_parameters()):
                p.grad = self._grad_arena[off[k]:off[k] + p.numel()].view(p.shape)
        return self._grad_arena

    def _sync_bn(self):
        pack = self._cache.pack
        if pack is not None and getattr(pack, "bn_dirty", False) and pack.n_experts == len(self.model):
            _writeback_bn(list(self.model), pack)

    def state_dict(self, *args, **kwargs):
        self._sync_bn()
        return super().state_dict(*args, **kwargs)

    def _experts_train_mode(self):
        """One flag per expert (nn.Module.training of each Model), as a tuple so it can key graph caches."""
        return tuple(bool(m.training) for m in self.model)

    # -- forward ---------------------------------------------------------------------------------
    def forward(self, image, cross=True, text=None, is_train=True):
        """-> {"logits": [B,T,C], "index": gate [B,I] (train) / argmax [B] (eval) / None, "aux_logits": None}
        (modules/model.py:343-359).

        opt.autograd (default off) with grad mode on makes the outputs differentiable (INTEGRATION.md §A):
          * cross=True, is_train=True (soft route): "logits" and "index" (the gate) with respect to route.*,
            channel_route.* and dm_router.0.*.  The experts are frozen: an expert parameter that requires grad raises
            NotImplementedError -- unless opt.autograd_experts is set, in which case every parameter of each expert
            with a parameter that requires grad (a trainable expert) gets its gradient too, along both paths of the
            reference (its logits through the gated combine, its feature through the DM-Router and the gate head);
            trainable experts run their training packs (BatchNorm / DropPath as cross=False), the others the grouped
            forward.  An image that requires grad gets its gradient through every expert: then every expert runs a
            training pack, the frozen ones with the input-only backward (their .grad stays None);
          * cross=True, is_train=False (hard route): "index" is an argmax and "logits" depends only on the frozen
            experts -- outputs as without the switch, no router or image gradient;
          * cross=False: "logits" with respect to every parameter of the newest expert and to the image
            (training-pack forward)."""
        grad = _autograd_on(self.opt)
        if cross is False:
            if grad:
                return dict(logits=_expert_autograd_forward(self.model[-1], image, self.opt, net=self), index=None,
                            aux_logits=None)
            feats, logits = _experts_forward([self.model[-1]], image, self.opt, self.model[-1].training)
            return dict(logits=logits[0], index=None, aux_logits=None)
        if grad and is_train:
            from ..autograd import RoutedSoft
            trainable = tuple(e for e, m in enumerate(self.model) if any(p.requires_grad for p in m.parameters()))
            if trainable and not getattr(self.opt, "autograd_experts", False):
                raise NotImplementedError(
                    "autograd through the routed forward keeps the experts frozen, as MRN stage 1 does "
                    "(il_modules/mrn.py:154-157): set requires_grad=False on every expert parameter, or set "
                    "opt.autograd_experts to train the experts that require grad together with the router")
            expert_params = [p for e in trainable for p in self.model[e].parameters()]
            logits, gate = RoutedSoft.apply(self, image, trainable, *self.router_parameters(), *expert_params)
            return dict(logits=logits, index=gate, aux_logits=None)
        r = self.route_and_combine(image, is_train=is_train, want_logits=True)
        return dict(logits=r["logits"], index=r["index"], aux_logits=None)

    def cross_forward(self, image, text=None, is_train=True):
        r = self.route_and_combine(image, is_train=True, want_logits=True)
        return r["logits"], r["index"]

    def cross_forward_expert(self, image, text=None, is_train=True):
        r = self.route_and_combine(image, is_train=False, want_logits=True)
        return r["logits"], r["index"]

    def pad_zeros_features(self, feature, total):
        raise RuntimeError("padding with ones is fused into mrnb_gate_combine; no padded tensor is materialised")

    def joint_experts_forward(self, image, trainable, input_grad=False):
        """Expert outputs of the soft route when the experts in `trainable` (indices) train with the router
        (opt.autograd_experts): the frozen ones through one grouped forward built over them alone, each trainable one
        through its training pack.  input_grad (the image requires grad): the frozen experts run training packs too,
        without a gradient arena (input-only backward).  DropPath is drawn once for all experts, as the grouped forward
        draws it.  Returns (features [B,I,T,D], [logits_i], {expert index: training-pack backward})."""
        if not image.is_cuda:
            raise RuntimeError("mrn_b200 needs CUDA tensors: there is no CPU fallback")
        full = self._cache.pack
        if full is not None and getattr(full, "bn_dirty", False):
            self._sync_bn()                 # BN statistics the full grouped pack holds -> the module buffers
            self._frozen_cache.key = None
        I, B = len(self.model), image.shape[0]
        modes = self._experts_train_mode()
        drop = None
        if _arch(self.opt) == "svtr" and any(modes) and getattr(self.opt, "drop_path", True):
            rates = self.model[0].model.FeatureExtraction.ConvNet.drop_path_rates()
            drop = sample_drop_scales(I, B, rates, image.device)
            for e, t in enumerate(modes):
                if not t:
                    drop[e].fill_(1.0)
        feats = torch.empty(B, I, self.patch, self.out_dim, device=image.device, dtype=torch.float32)
        logits = [None] * I
        frozen = [e for e in range(I) if e not in trainable]
        if frozen and not input_grad:
            experts = [self.model[e] for e in frozen]
            f, z = _experts_forward(experts, image, self.opt, tuple(modes[e] for e in frozen), self._frozen_cache,
                                    drop_scales=None if drop is None else drop[frozen].contiguous())
            feats[:, frozen] = f
            for k, e in enumerate(frozen):
                logits[e] = z[k]
            if any(modes[e] for e in frozen):
                _writeback_bn(experts, self._frozen_cache.pack)
                self._cache.key = None      # the full grouped pack's BN statistics are stale now
        backward = {}
        for e in (range(I) if input_grad else trainable):
            z, f, backward[e] = _train_pack_run(self.model[e], image, self.opt, net=self, want_features=True,
                                                drop=drop[e].contiguous() if drop is not None and modes[e] else None,
                                                param_grads=e in trainable)
            feats[:, e] = f
            logits[e] = z
        return feats, logits, backward

    def route_and_combine(self, image, is_train=True, want_logits=True, targets=None, lengths=None, want_E=False,
                          want_decode=False, with_backward=False, drop_scales=None, rws=None, experts_out=None):
        """Experts -> DM-Router -> gate -> fused combine.  Soft route when is_train (modules/model.py:397-423),
        hard route otherwise (:366-395).  rws: router workspace to use instead of the module's own.  experts_out:
        (features [B,I,T,D], [logits_i]) computed by the caller (joint_experts_forward) instead of the grouped forward."""
        experts = list(self.model)
        # Hard route (eval): route FIRST, then evaluate only the routed expert's classifier head per sample (SURVEY K8e;
        # modules/model.py:383-393 keeps padded_{index[b]}[b] and discards the other five heads' logits).  The soft
        # route needs every head.
        sparse = (not is_train) and _arch(self.opt) == "svtr" and not int(getattr(self.opt, "expert_chunk", 0) or 0)
        if experts_out is not None:
            assert not sparse, "precomputed expert outputs serve the soft route"
            feats, logits = experts_out
        else:
            feats, logits = _experts_forward(experts, image, self.opt, self._experts_train_mode(), self._cache,
                                             drop_scales=drop_scales, want_logits=not sparse)
        arena = self.router_arena(image.device)
        _, scores, gate, index = ops.router_forward(arena, feats, rws or self._rws, with_backward=with_backward,
                                                    prec=_precision(self.opt), want_out=False)
        if is_train:
            g, idx_out = gate, gate
        else:
            g = torch.nn.functional.one_hot(index.long(), len(experts)).float()
            idx_out = index.long()
            if sparse:
                logits = ops.svtr_heads(self._cache.pack, image.shape[0], index)
        r = ops.gate_combine(logits, g, targets, lengths, want_logits=want_logits, want_E=want_E, want_decode=want_decode)
        r.update(index=idx_out, gate=gate, scores=scores, features=feats, expert_logits=logits, combine_gate=g)
        return r
