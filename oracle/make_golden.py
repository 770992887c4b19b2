"""Generate tests/golden/*.npz by running the UNMODIFIED reference (simplify23/MRN) in the build container.

Run:  python -m oracle.make_golden          (needs /root/reference; CPU only, ~1 min)

The reference has no golden vectors of its own (SURVEY.md §4), so these fixtures pin the oracle
(oracle/mrn_oracle.py) -- and through it the CUDA path -- to outputs of the reference's own modules:
modules.model.MRNNet / modules.dm_router.DM_Router / torch.nn.CTCLoss / tools.utils.CTCLabelConverter,
driven exactly as il_modules/mrn.py:329-360 and test.py:163-221 drive them.  Weights and inputs are the
deterministic synthetic tensors of oracle/synth.py (rebuilt, not stored).  Large gradients are stored as a
strided subsample plus their Frobenius norm.
"""
import argparse
import contextlib
import io
import os

import numpy as np
import torch

from oracle import synth
from oracle.ref_import import reference_modules

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
SUB = 11    # stride of the subsample kept for tensors above MAX_FULL elements
MAX_FULL = 16384


def keep(t: torch.Tensor, sub: int = SUB, max_full: int = MAX_FULL) -> np.ndarray:
    a = t.detach().cpu().numpy()
    if a.size > max_full:
        return np.ascontiguousarray(a.reshape(-1)[::sub])
    return a.copy()


def build_ref_net(ref, class_counts, sd, arch="svtr"):
    opt = argparse.Namespace(Transformation="None", FeatureExtraction="SVTR" if arch == "svtr" else "VGG",
                             SequenceModeling="None" if arch == "svtr" else "BiLSTM",
                             Prediction="CTC", num_fiducial=20, input_channel=4, output_channel=512,
                             hidden_size=256, imgH=32, imgW=256, batch_max_length=25)
    with contextlib.redirect_stdout(io.StringIO()):
        net = ref.model.MRNNet(opt)
        for C in class_counts:            # il_modules/mrn.py:110-116,96-103
            net.update_fc(opt.hidden_size, C)
            net.build_prediction(opt, C)
    missing = net.load_state_dict(sd, strict=True)   # the state_dict contract (SURVEY.md §8b)
    assert not missing.missing_keys and not missing.unexpected_keys
    return net


def run_case(name, class_counts, B, seed, arch="svtr"):
    I = len(class_counts)
    sd = synth.synth_state_dict(class_counts, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, class_counts, seed)
    rates = [0.1 * i / 11 for i in range(12)]
    drop = synth.synth_drop_scales(I, B, rates, seed)
    g = {}
    with reference_modules() as ref:
        net = build_ref_net(ref, class_counts, sd, arch)
        crit = torch.nn.CTCLoss(reduction="mean", zero_infinity=True)       # il_modules/base.py:131
        ce = torch.nn.CrossEntropyLoss(reduction="mean")                     # il_modules/mrn.py:150
        conv = ref.utils.CTCLabelConverter([chr(0x4E00 + i) for i in range(class_counts[-1] - 4)])

        # ---- eval-mode experts (BN running stats, no DropPath): soft route (train) + hard route (eval)
        net.eval()
        feats = []
        hooks = [m.register_forward_hook(lambda mod, inp, out, L=feats: L.append(out["feature"].detach()))
                 for m in net.model]
        router_out = []
        hooks.append(net.dm_router.register_forward_hook(lambda mod, inp, out: router_out.append(out.detach())))
        for p in net.parameters():
            p.requires_grad_(False)
        for n_, p in net.named_parameters():
            if not n_.startswith("model."):
                p.requires_grad_(True)                                       # router stage (mrn.py:154-157)
        out = net(img, True, None, True)                                     # mrn.py:338
        preds = out["logits"]
        taski_loss = ce(out["index"], dom)                                   # mrn.py:342
        psize = torch.IntTensor([preds.size(1)] * B)
        loss_clf = crit(preds.log_softmax(2).permute(1, 0, 2), tgt, psize, lens)   # mrn.py:345-346
        loss = 15 * loss_clf + taski_loss                                    # mrn.py:360
        net.zero_grad()
        loss.backward()
        g["features"] = keep(torch.stack(feats[:I], 1))
        g["router_out"] = keep(router_out[0])
        g["gate"] = out["index"].detach().numpy()
        g["logits_soft"] = keep(preds)
        g["loss_clf"] = np.float64(loss_clf.item()); g["taski_loss"] = np.float64(taski_loss.item())
        g["loss"] = np.float64(loss.item())
        for n_, p in net.named_parameters():
            if p.grad is not None:
                g["grad." + n_] = keep(p.grad)
                g["gradnorm." + n_] = np.float64(p.grad.double().norm().item())
        total_norm = torch.nn.utils.clip_grad_norm_(net.parameters(), 5)     # mrn.py:364
        g["grad_total_norm"] = np.float64(float(total_norm))
        # one Adam step on the router parameters (mrn.py:52-66,367): lr 5e-4 (config/svtr_mrn.py:33)
        params = [p for p in net.parameters() if p.requires_grad]
        opt_ = torch.optim.Adam(params, lr=5e-4)
        opt_.step()
        for n_, p in net.named_parameters():
            if p.requires_grad:
                g["adam1." + n_] = keep(p.detach())
        net.load_state_dict(sd, strict=True)

        with torch.no_grad():
            ev = net(img, True, None, False)                                 # test.py:165-166
            lg = ev["logits"]
            g["index_hard"] = ev["index"].numpy()
            g["logits_hard"] = keep(lg)
            cost = crit(lg.log_softmax(2).permute(1, 0, 2), tgt, psize, lens)     # test.py:178-183
            g["valid_loss"] = np.float64(cost.item())
            _, pidx = lg.max(2)                                              # test.py:211
            g["decode_raw"] = pidx.numpy()
            strs = conv.decode(pidx, torch.IntTensor([lg.size(1)] * B))      # test.py:212-213
            # ids behind the reference's strings ([PAD]/[UNK] are multi-character entries, so re-derive the ids with
            # the collapse rule of tools/utils.py:66-74 and check they spell exactly the reference's output)
            ids = []
            for b_, row in enumerate(pidx.tolist()):
                r = [c for k_, c in enumerate(row) if c != 0 and not (k_ > 0 and row[k_ - 1] == c)]
                assert "".join(conv.character[c] for c in r) == strs[b_]
                ids.append(r)
            g["decode_ids"] = np.array([r + [-1] * (lg.size(1) - len(r)) for r in ids], dtype=np.int64)
            g["decode_len"] = np.array([len(r) for r in ids], dtype=np.int64)
            pmax, _ = torch.softmax(lg, dim=2).max(dim=2)                    # test.py:219-220
            g["confidence"] = np.array([float(pm.cumprod(dim=0)[-1]) for pm in pmax], dtype=np.float64)   # test.py:257
            ff = net(img, False, None, False)                                # cross=False path, model.py:346-348
            g["logits_last_expert"] = keep(ff["logits"])

        # ---- train-mode experts (BN batch statistics + DropPath with injected masks; reference quirk 4)
        net.train()
        queue = []
        orig_drop = ref.svtr.drop_path

        def injected(x, drop_prob=0., training=False, scale_by_keep=True):
            s = queue.pop(0)
            return x * s.view(-1, 1, 1)
        ref.svtr.drop_path = injected
        try:
            for i in range(I if arch == "svtr" else 0):
                for j in range(12):
                    if rates[j] > 0:                 # Block uses Identity when drop_path == 0 (svtr.py:187)
                        queue.append(drop[i, j, 0]); queue.append(drop[i, j, 1])
            feats.clear(); router_out.clear()
            with torch.no_grad():
                tr = net(img, True, None, True)
            assert not queue
        finally:
            ref.svtr.drop_path = orig_drop
        g["train_features"] = keep(torch.stack(feats[:I], 1))
        g["train_gate"] = tr["index"].numpy()
        g["train_logits_soft"] = keep(tr["logits"])
        cn = net.model[0].model.FeatureExtraction.ConvNet
        bn = cn.patch_embed.proj[1] if arch == "svtr" else cn[12]
        g["train_bn1_running_mean_e0"] = bn.running_mean.numpy().copy()      # momentum 0.1 update
        g["train_bn1_running_var_e0"] = bn.running_var.numpy().copy()
        for h in hooks:
            h.remove()
    g["class_counts"] = np.array(class_counts); g["B"] = np.int64(B); g["seed"] = np.int64(seed)
    g["arch"] = np.array(arch)
    g["sub"] = np.int64(SUB); g["max_full"] = np.int64(MAX_FULL)
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **g)
    print(name, "->", path, os.path.getsize(path) // 1024, "KiB")


def run_stage0_case(name, class_counts, B, seed, bn_train=True, arch="svtr"):
    """One stage-0 iteration of the unmodified reference (il_modules/mrn.py:236-267): the newest expert trained end to
    end through `model(image, cross=False)` with CTC, earlier experts frozen (mrn.py:154-157).  Train mode (BatchNorm
    batch statistics, DropPath masks injected so the run is reproducible)."""
    I = len(class_counts)
    sd = synth.synth_state_dict(class_counts, seed, arch=arch)
    img, tgt, lens, dom = synth.synth_batch(B, class_counts, seed)
    tgt = tgt.clamp(max=class_counts[-1] - 1)
    rates = [0.1 * i / 11 for i in range(12)]
    drop = synth.synth_drop_scales(I, B, rates, seed)
    g = {}
    with reference_modules() as ref:
        net = build_ref_net(ref, class_counts, sd, arch)
        crit = torch.nn.CTCLoss(reduction="mean", zero_infinity=True)       # il_modules/base.py:131
        for i in range(I - 1):
            for p in net.model[i].parameters():
                p.requires_grad = False                                      # mrn.py:154-157
        net.train(bn_train)
        queue = []
        orig_drop = ref.svtr.drop_path

        def injected(x, drop_prob=0., training=False, scale_by_keep=True):
            s = queue.pop(0)
            return x * s.view(-1, 1, 1)
        if bn_train and arch == "svtr":
            ref.svtr.drop_path = injected
            for j in range(12):
                if rates[j] > 0:
                    queue.append(drop[I - 1, j, 0]); queue.append(drop[I - 1, j, 1])
        try:
            preds = net(img, False)["logits"]                                # mrn.py:246
            assert not queue
        finally:
            ref.svtr.drop_path = orig_drop
        psize = torch.IntTensor([preds.size(1)] * B)
        loss = crit(preds.log_softmax(2).permute(1, 0, 2), tgt, psize, lens)  # mrn.py:249-252
        net.zero_grad()
        loss.backward()                                                      # mrn.py:260
        g["logits"] = keep(preds)
        g["loss"] = np.float64(loss.item())
        for n_, p in net.named_parameters():
            if p.grad is not None:
                g["grad." + n_] = keep(p.grad, 101, 2048)
                g["gradnorm." + n_] = np.float64(p.grad.double().norm().item())
        total_norm = torch.nn.utils.clip_grad_norm_(net.parameters(), 5)     # mrn.py:261-263
        g["grad_total_norm"] = np.float64(float(total_norm))
        params = [p for p in net.parameters() if p.requires_grad]            # count_param(), base.py:84-108
        opt_ = torch.optim.Adam(params, lr=5e-4)
        opt_.step()                                                          # mrn.py:264
        for n_, p in net.named_parameters():
            if p.grad is not None:
                g["adam1." + n_] = keep(p.detach(), 101, 2048)
        cn = net.model[I - 1].model.FeatureExtraction.ConvNet
        bn = (cn.patch_embed.proj[1], cn.patch_embed.proj[4]) if arch == "svtr" else (cn[12], cn[15])
        g["bn0_running_mean"] = bn[0].running_mean.numpy().copy(); g["bn0_running_var"] = bn[0].running_var.numpy().copy()
        g["bn1_running_mean"] = bn[1].running_mean.numpy().copy(); g["bn1_running_var"] = bn[1].running_var.numpy().copy()
    g["class_counts"] = np.array(class_counts); g["B"] = np.int64(B); g["seed"] = np.int64(seed)
    g["bn_train"] = np.int64(int(bn_train)); g["arch"] = np.array(arch)
    g["sub"] = np.int64(SUB); g["max_full"] = np.int64(MAX_FULL)
    g["psub"] = np.int64(101); g["pmax_full"] = np.int64(2048)
    os.makedirs(OUT, exist_ok=True)
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **g)
    print(name, "->", path, os.path.getsize(path) // 1024, "KiB")


def run_router_case(name, I, B, seed, sub=SUB):
    """DM_Router alone on random features (modules/dm_router.py:50-67) incl. input gradient."""
    shapes = synth.router_shapes(I)
    sd = {k: synth.synth_tensor(seed, k, s) for k, s in shapes.items()}
    x = synth.randn(seed, "router_x", (B, I, 64, 256))
    with reference_modules() as ref:
        m = ref.dm_router.DM_Router(256, 512, 64, I)
        m.load_state_dict({k[len("dm_router.0."):]: v for k, v in sd.items() if k.startswith("dm_router.0.")}, strict=True)
        xr = x.clone().requires_grad_(True)
        y = m(xr)
        w = synth.randn(seed, "router_dy", y.shape)
        (y * w).sum().backward()
        g = dict(out=keep(y, sub), dx=keep(xr.grad, sub), I=np.int64(I), B=np.int64(B), seed=np.int64(seed),
                 sub=np.int64(sub), max_full=np.int64(MAX_FULL))
        for n_, p in m.named_parameters():
            g["grad." + n_] = keep(p.grad, sub)
            g["gradnorm." + n_] = np.float64(p.grad.double().norm().item())
    path = os.path.join(OUT, name + ".npz")
    np.savez_compressed(path, **g)
    print(name, "->", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    import sys
    torch.manual_seed(0)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    only = sys.argv[1:]
    if not only or "svtr" in only:
        run_case("svtr_mrn_i3_b3", (37, 61, 96), 3, 111)
        run_case("svtr_mrn_i2_b4", (53, 80), 4, 7)
    if not only or "crnn" in only:
        # BASELINE.json configs[0] in miniature: CRNN-MRN (VGG + BiLSTM + CTC), 2 tasks; and a 3-task case
        run_case("crnn_mrn_i2_b4", (53, 80), 4, 21, arch="crnn")
        run_case("crnn_mrn_i3_b2", (37, 61, 96), 2, 33, arch="crnn")
    if not only or "stage0" in only:
        run_stage0_case("svtr_stage0_i2_b3", (37, 61), 3, 17)
        run_stage0_case("svtr_stage0_i1_b2_eval", (45,), 2, 29, bn_train=False)
        run_stage0_case("crnn_stage0_i2_b3", (37, 61), 3, 19, arch="crnn")
        run_stage0_case("crnn_stage0_i1_b2_eval", (45,), 2, 31, bn_train=False, arch="crnn")
    if only and "router" not in only:
        sys.exit(0)
    run_router_case("dm_router_i3_b2", 3, 2, 5)
    run_router_case("dm_router_i6_b1", 6, 1, 9, sub=2 * SUB)      # every 22nd element keeps the file under 1 MB
