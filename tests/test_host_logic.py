"""CPU tests of the host-side mirror of the reference API (no GPU compute): label codec, schedules, module tree /
state_dict contract, loud failure without CUDA."""
import argparse

import pytest
import torch

from mrn_b200 import synth
from oracle import mrn_oracle as O
from oracle.ref_import import reference_available


def make_opt(**kw):
    d = dict(Transformation="None", FeatureExtraction="SVTR", SequenceModeling="None", Prediction="CTC", num_fiducial=20,
             input_channel=4, output_channel=512, hidden_size=256, imgH=32, imgW=256, batch_max_length=25, lr=5e-4,
             num_iter=100, grad_clip=5, exp_name="t", precision="fp32", drop_path=False, lan_list=["a", "b"],
             val_interval=50, start_task=0)
    d.update(kw)
    return argparse.Namespace(**d)


def test_ctc_label_converter_matches_reference_semantics():
    from mrn_b200.utils import CTCLabelConverter
    chars = list("abcdefg") + ["中", "文"]
    conv = CTCLabelConverter(chars)
    assert conv.character[:4] == ["[CTCblank]", "[PAD]", "[UNK]", " "] and conv.dict["a"] == 4       # tools/utils.py:15-31
    idx, lens = conv.encode(["abc", "", "a中z", "g" * 25], batch_max_length=25)
    assert idx.shape == (4, 25) and idx.dtype == torch.int64 and lens.tolist() == [3, 0, 3, 25]
    assert idx[0, :4].tolist() == [4, 5, 6, 1] and idx[1].eq(1).all() and idx[2, :3].tolist() == [4, conv.dict["中"], 2]
    ref_idx, ref_len = O.ctc_encode(["abc", "", "a中z", "g" * 25], conv.dict)
    assert torch.equal(idx, ref_idx) and torch.equal(lens, ref_len)
    raw = torch.tensor([[0, 4, 4, 0, 4, 5, 5, 0, 0, 6], [0] * 10])
    assert conv.decode(raw, [10, 10]) == ["aabc", ""]                                                  # tools/utils.py:62-76
    assert conv.decode_compact(torch.tensor([[4, 4, 5, 6, -1], [-1] * 5]), torch.tensor([4, 0])) == ["aabc", ""]
    if reference_available():
        from oracle.ref_import import reference_modules
        import contextlib, io
        with reference_modules() as ref, contextlib.redirect_stdout(io.StringIO()):
            rc = ref.utils.CTCLabelConverter(chars)
            assert rc.character == conv.character and rc.dict == conv.dict
            ri, rl = rc.encode(["abc", "", "a中z"], batch_max_length=25)
            assert torch.equal(ri.cpu(), idx[:3]) and rl.cpu().tolist() == [3, 0, 3]
            assert rc.decode(raw, [10, 10]) == conv.decode(raw, [10, 10])


def test_one_cycle_and_edit_distance():
    from mrn_b200.il_modules.mrn import one_cycle_lr, edit_distance
    for s in (0, 1, 59, 60, 150, 199):
        assert abs(one_cycle_lr(s, 200, 5e-4) - O.one_cycle_lr(s, 200, 5e-4)) < 1e-15
    assert edit_distance("kitten", "sitting") == 3 and edit_distance("", "abc") == 3 and edit_distance("abc", "abc") == 0


def test_module_tree_keeps_the_reference_state_dict_contract():
    from mrn_b200.il_modules.mrn import RankLocal
    from mrn_b200.modules.model import MRNNet
    cc = (37, 61, 96)
    opt = make_opt()
    net = MRNNet(opt)
    for i, c in enumerate(cc):
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
        # the router is rebuilt for the new expert count at every task (modules/model.py:437-452)
        assert net.channel_route.weight.shape == (i + 1, (i + 1) * 256)
        assert net.dm_router[0].spatial_gating.proj.weight.shape == ((i + 1) * 64, (i + 1) * 64)
    want = synth.svtr_mrn_shapes(cc)
    got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert got == {k: tuple(s) for k, s in want.items()}
    sd = synth.synth_state_dict(cc, 3)
    res = net.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    assert net.model[1].fc is net.model[1].Prediction                  # alias kept (modules/model.py:181)
    wrapped = RankLocal(net).state_dict()
    assert all(k.startswith("module.") for k in wrapped) and len(wrapped) == len(got)   # DataParallel key prefix (mrn.py:412-415)
    # parameters() order of the router == the C-ABI arena order
    from mrn_b200 import ops
    names = [n for n, _ in net.named_parameters() if not n.startswith("model.")]
    assert tuple(names) == ops.ROUTER_PARAM_NAMES
    # SVTR constructor quirk: LayerNorm bias initialised to 1.0 (modules/svtr.py:494-496)
    fresh = MRNNet(opt); fresh.update_fc(256, 10)
    assert float(fresh.model[0].model.FeatureExtraction.ConvNet.blocks1[0].norm1.bias.detach().mean()) == 1.0


def test_crnn_module_tree_keeps_the_reference_state_dict_contract():
    from mrn_b200.modules.model import MRNNet
    cc = (37, 61)
    opt = make_opt(FeatureExtraction="VGG", SequenceModeling="BiLSTM")
    net = MRNNet(opt)
    for c in cc:
        net.update_fc(opt.hidden_size, c)
        net.build_prediction(opt, c)
    assert net.patch == 63 and net.route.weight.shape == (1, 63)       # modules/model.py:322-323
    want = synth.crnn_mrn_shapes(cc)
    got = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    assert list(got) == list(want) and got == {k: tuple(s) for k, s in want.items()}
    res = net.load_state_dict(synth.synth_state_dict(cc, 3, arch="crnn"), strict=True)
    assert not res.missing_keys and not res.unexpected_keys


def test_router_arena_views_share_storage():
    from mrn_b200.modules.model import MRNNet
    from mrn_b200 import ops
    opt = make_opt()
    net = MRNNet(opt)
    for c in (20, 30):
        net.update_fc(256, c); net.build_prediction(opt, c)
    arena = net.router_arena("cpu")
    n, off = ops.router_param_offsets(2)
    assert arena.numel() == n
    net.route.weight.data.fill_(7.0)
    assert float(arena[off[0]]) == 7.0                                  # parameters are views into the arena
    g = net.router_grad_arena()
    g.fill_(2.0)
    assert float(net.dm_router[0].proj_3.bias.grad[0]) == 2.0


def test_no_cpu_fallback_and_unsupported_configs_fail_loudly():
    from mrn_b200.modules.model import MRNNet, Model
    opt = make_opt()
    net = MRNNet(opt)
    net.update_fc(256, 12); net.build_prediction(opt, 12)
    with pytest.raises(RuntimeError, match="no CPU fallback|CUDA"):
        net(torch.zeros(1, 4, 32, 256), True, None, True)
    with pytest.raises(NotImplementedError):
        MRNNet(make_opt(FeatureExtraction="ResNet", SequenceModeling="BiLSTM"))
    with pytest.raises(NotImplementedError):
        MRNNet(make_opt(Transformation="TPS"))
    with pytest.raises(NotImplementedError):
        Model(make_opt(Prediction="Attn"))
    from mrn_b200.il_modules.mrn import MRN
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="CUDA"):
            MRN(opt)


# ---- stage-0 training arenas, driver glue (host logic only) ---------------------------------------------------------
@pytest.mark.parametrize("arch", ["svtr", "crnn"])
def test_train_pack_arena_round_trips_the_expert_state_dict(arch):
    """ops.SvtrTrainPack / CrnnTrainPack: every trainable tensor of the expert lands in the flat arena exactly once (conv
    weights permuted to [Cout,kh,kw,Cin], LSTM directions adjacent) and state() returns the reference layout again."""
    import torch
    from mrn_b200 import ops
    from oracle import mrn_oracle as O
    from oracle import synth
    sd = synth.synth_state_dict((33,), 3, arch=arch)
    esd = {k[len("model.0."):]: v for k, v in sd.items() if k.startswith("model.0.")}
    cls = ops.SvtrTrainPack if arch == "svtr" else ops.CrnnTrainPack
    tp = cls(esd, "cpu")
    keys = [k[len("model.0."):] for k in O.expert_param_keys(sd, 0)]
    back = tp.state()
    assert sorted(back) == sorted(keys)                      # exactly the tensors that receive a gradient in stage 0
    for k in keys:
        assert torch.equal(back[k], esd[k]), k
    n_params = sum(esd[k].numel() for k in keys)
    assert n_params <= tp.numel <= n_params + 8 * len(tp.entries)      # slots padded to 8 floats
    offs = sorted((e[3], e[3] + int(torch.tensor(e[4]).prod())) for e in tp.entries)
    assert all(a1 <= b0 for (a0, a1), (b0, b1) in zip(offs, offs[1:]))       # no overlap
    # gradient arena shares the layout: a write through the view shows up under the reference key
    tp.grads.zero_()
    tp.view(tp.grads, tp.entries[1]).fill_(2.0)
    g = tp.state(tp.grads)
    assert float(g[tp.entries[1][1]].sum()) == 2.0 * g[tp.entries[1][1]].numel()
    assert sum(float(v.abs().sum()) for k, v in g.items() if k != tp.entries[1][1]) == 0.0


def test_domain_ids_flatten_like_the_reference():
    import torch
    from mrn_b200.il_modules.mrn import _domain_ids
    a = _domain_ids([torch.tensor([0, 1, 1]), torch.tensor([2])])
    assert a.dtype == torch.long and a.tolist() == [0, 1, 1, 2]
    assert _domain_ids([3, 0, 1]).tolist() == [3, 0, 1]


def test_rehearsal_memory_index_bookkeeping():
    """build_rehearsal_memory keeps one index array per earlier task, trims them to memory_num / taski and hands the list
    to the dataset layer (il_modules/mrn.py:169-178, il_modules/base.py:292-302)."""
    import numpy as np
    from mrn_b200.il_modules.mrn import MRN

    class FakeLoader:
        def __init__(self):
            self.calls = []

        def rehearsal_prev_model(self, taski):
            return None, 10000 + taski

        def get_dataset(self, taski, memory=None, index_list=None):
            self.calls.append((taski, memory, [np.array(ix) for ix in index_list]))

    learner = MRN.__new__(MRN)                      # host logic only: no device, no model
    learner.opt = argparse.Namespace(memory="random", memory_num=2000)
    learner.memory_index = []
    loader = FakeLoader()
    np.random.seed(111)
    for taski in (1, 2, 3):
        learner.build_rehearsal_memory(loader, taski)
        t, memory, idx = loader.calls[-1]
        assert t == taski and memory == "random" and len(idx) == taski
        per = int(2000 / taski)
        assert all(ix.size == per for ix in idx)
        assert all(len(set(ix.tolist())) == per for ix in idx)                 # drawn without replacement
        assert all(ix.max() < 10000 + k + 1 for k, ix in enumerate(idx))       # task k's array indexes task k's dataset
    first = loader.calls[0][2][0]
    assert (loader.calls[-1][2][0] == first[: int(2000 / 3)]).all()            # earlier arrays are trimmed, not redrawn
    big = MRN.__new__(MRN)
    big.opt = argparse.Namespace(memory="random", memory_num=5000)
    big.memory_index = []
    for taski in (1, 2):
        big.build_rehearsal_memory(loader, taski)
    assert [ix.size for ix in loader.calls[-1][2]] == [5000, 5000]             # memory_num >= 5000: per task, never trimmed


def test_model_eval_and_train_and_freeze_step1_set_the_reference_modes():
    """il_modules/mrn.py:45-50, 289-295: earlier experts eval, newest expert train; freeze_step1 then calls model.train()
    again -- the earlier experts are back in TRAIN mode, the reference's quirk the stage-1 step reproduces -- and freezes
    the newest expert in eval mode while the router modules stay trainable."""
    from mrn_b200.il_modules.mrn import MRN
    from mrn_b200.modules.model import MRNNet
    opt = make_opt()
    net = MRNNet(opt)
    for c in (12, 20):
        net.update_fc(256, c); net.build_prediction(opt, c)
    learner = MRN.__new__(MRN)                      # host logic only: no device
    learner.opt = opt
    learner.model = net
    net.eval()
    learner.model_eval_and_train(1)
    assert net.training and net.model[1].training and not net.model[0].training
    learner.freeze_step1(1)
    assert net.training and net.model[0].training and not net.model[1].training
    assert all(not p.requires_grad for p in net.model[1].parameters())
    assert any(p.requires_grad for n, p in net.named_parameters() if not n.startswith("model."))
