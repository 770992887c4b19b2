"""GPU parity tests, building blocks first: every CUDA kernel against the CPU oracle / a torch fp64 statement of the
same op on the same seeded inputs.  All calls go through the C ABI (mrn_b200.ops -> libmrn_b200.so)."""
import math

import numpy as np
import pytest
import torch

from oracle import mrn_oracle as O
from oracle import synth
from conftest import load_golden, gview, rel_err
from persistent_walk import (assert_walk, attn_tc_walk, cdiv, combine_walk, locate, mixer_walk, mlp_walk, tc_gemm2_walk,
                             tc_gemm_bn, tc_gemm_walk)

pytestmark = pytest.mark.gpu


def _ops():
    from mrn_b200 import ops
    return ops


def dev(t):
    return t.cuda().contiguous()


def _kept_ids(rows, n):
    """pytest.params whose id is the one the case had before the trailing parameters were added (its first n values), so
    the existing cases keep their names; the added cases get the default id over all their values."""
    return [pytest.param(*r, id="-".join(str(v) for v in r[:n])) for r in rows]


def _tile_check(err, tol, BN, grid, what, splits=1):
    """err [M, N] absolute error, tol scalar: the 128 x BN output tiles whose error exceeds tol, named with their item
    index t = m_tile * n_tiles + n_tile (split s of a split-K tile: t + s * m_tiles * n_tiles)."""
    M, N = err.shape
    tm, tn = cdiv(M, 128), cdiv(N, BN)
    e = torch.nn.functional.pad(err.nan_to_num(float("inf")), (0, tn * BN - N, 0, tm * 128 - M))
    worst = e.reshape(tm, 128, tn, BN).amax((1, 3)).reshape(-1)
    bad = worst > tol
    coords = lambda t: "m-tile %d, n-tile %d%s" % (t // tn, t % tn, "" if splits == 1 else ", split items t + s * %d" % (tm * tn))
    assert not bool(bad.any()), locate(bad, grid, coords, what, worst / tol)


# ------------------------------------------------------------------------------------------------ GEMMs
@pytest.mark.parametrize("M,N,K,gelu,res", [(256, 192, 64, False, False), (300, 70, 100, True, True),
                                            (1000, 513, 257, False, True), (64, 6, 1536, False, False)])
def test_sgemm_matches_fp64(M, N, K, gelu, res):
    ops = _ops()
    torch.manual_seed(M + N + K)
    a, w, b = torch.randn(M, K), torch.randn(N, K) / math.sqrt(K), torch.randn(N)
    r = torch.randn(M, N) if res else None
    ref = a.double() @ w.double().T + b.double()
    if gelu:
        ref = torch.nn.functional.gelu(ref)
    if res:
        ref = ref + r.double()
    out = ops.linear_f32(dev(a), dev(w), dev(b), dev(r) if res else None, gelu).cpu()
    assert rel_err(out.numpy(), ref.numpy()) < 2e-6


@pytest.mark.parametrize("M,N,K,gelu,res,f32out", [
    (256, 192, 64, False, False, True),      # qkv of stage 1: one k-block, BN=64 tiles
    (384, 128, 256, False, True, True),      # proj + residual, BN=128
    (300, 70, 128, True, False, False),      # M and N tails, bf16 output, GELU
    (1024, 512, 1024, True, False, False),   # fc1-like, 16 k-blocks: exercises the 4-stage ring twice over
    (640, 1899, 256, False, False, True),    # classifier head: N not a multiple of anything
    # persistent walk: >= 4 tiles per CTA (asserted), M tails (M = 77 mod 128), N tails, both tile widths; K = 64 is a
    # one-deep operand ring (its parity flips every k-block), K = 320 is 5 k-blocks on the 2-stage ring (wraps mid-tile)
    (1184 * 128 + 77, 64, 64, False, True, True),      # BN = 64, residual
    (592 * 128 + 77, 70, 320, True, False, False),     # BN = 64, N tail, GELU, bf16 out
    (395 * 128, 384, 320, False, True, True),          # BN = 128, residual
    (395 * 128 + 77, 300, 64, True, False, False),     # BN = 128, N tail, GELU, bf16 out
])
def test_tcgen05_gemm_matches_fp64(M, N, K, gelu, res, f32out):
    ops = _ops()
    torch.manual_seed(M * 7 + N)
    a = dev(torch.randn(M, K).bfloat16())
    w = dev((torch.randn(N, K) / math.sqrt(K)).bfloat16())
    b = dev(torch.randn(N))
    r = dev(torch.randn(M, N)) if res else None
    tiles, grid = tc_gemm_walk(M, N)
    if M > 4096:
        assert_walk(tiles, grid, "tc_gemm_kernel")
    ref = a.double() @ w.double().T + b.double()
    if gelu:
        ref = torch.nn.functional.gelu(ref)
    if res:
        ref = ref + r.double()
    out = torch.full((M, N), float("nan"), device="cuda", dtype=torch.float32 if f32out else torch.bfloat16)
    ops.linear_bf16(a, w, b, r, gelu, f32out, out=out)
    tol = 2e-5 if f32out else 6e-3       # fp32 accumulate of exact bf16 products; bf16 output rounding = 2^-8
    _tile_check((out.double() - ref).abs(), tol * float(ref.abs().max()), tc_gemm_bn(N), grid,
                "tc_gemm %dx%dx%d: tiles over %.0e relative (err / budget)" % (M, N, K, tol))


@pytest.mark.parametrize("a_mn,b_mn", [(0, 0), (0, 1), (1, 0), (1, 1)])
@pytest.mark.parametrize("M,N,K,splitk", [(256, 128, 256, 1), (384, 320, 512, 1), (256, 256, 4096, 8), (200, 70, 192, 1),
                                           # >= 4 tiles per CTA (asserted): K = 320 is 5 k-blocks on the 3-stage ring;
                                           # 13 k-blocks split 4 ways -> splits of 4, 4, 4 and 1 k-blocks
                                           (592 * 128, 256, 320, 1), (37 * 128, 1024, 13 * 64, 4)])
def test_tcgen05_general_gemm_major_modes(a_mn, b_mn, M, N, K, splitk):
    """K-major / MN-major operands straight from HBM (no transposed copies) + split-K atomics."""
    ops = _ops()
    if (a_mn and M % 8) or (b_mn and N % 8):
        pytest.skip("MN-major operands need a 16-byte aligned leading dimension")
    torch.manual_seed(M + 3 * N + K + a_mn * 2 + b_mn)
    a = dev(torch.randn(M, K).bfloat16())
    b = dev((torch.randn(N, K) / math.sqrt(K)).bfloat16())
    tiles, grid = tc_gemm2_walk(M, N, K, splitk)
    if M > 4096 or splitk == 4:
        assert_walk(tiles, grid, "tc_gemm2_kernel")
    ref = a.double() @ b.double().T
    ad = a.T.contiguous() if a_mn else a
    bd = b.T.contiguous() if b_mn else b
    out = ops.tc_gemm_general(ad, a_mn, bd, b_mn, M, N, K, splitk)
    _tile_check((out.double() - ref).abs(), 3e-5 * float(ref.abs().max()), 128 if N >= 128 else 64, grid,
                "tc_gemm2 %dx%dx%d split %d: tiles over 3e-5 relative (err / budget)" % (M, N, K, splitk), splits=splitk)


@pytest.mark.parametrize("D,M,ln,drop,rps", _kept_ids([(64, 1024, True, True, 128), (128, 512, True, False, 128),
                                                          (256, 384, False, True, 128), (128, 2048, False, False, 128)], 4) + [
                                                  # >= 4 tiles per CTA (asserted), DropPath per sample as in the step
                                                  # (512 / 256 / 128 rows per sample at d = 64 / 128 / 256)
                                                  (64, 592 * 128, True, True, 512), (128, 592 * 128, True, True, 256),
                                                  (256, 592 * 128, False, True, 128)])
def test_fused_mlp_tcgen05(D, M, ln, drop, rps):
    """x + rs * (GELU(A W1^T + b1) W2^T + b2) with the hidden activation kept on chip (+ fused next LayerNorm)."""
    ops = _ops()
    torch.manual_seed(D + M)
    a = dev(torch.randn(M, D).bfloat16())
    w1 = dev((torch.randn(4 * D, D) / math.sqrt(D)).bfloat16())
    w2 = dev((torch.randn(D, 4 * D) / math.sqrt(4 * D)).half())          # second GEMM runs f16 x f16
    b1, b2, x = dev(torch.randn(4 * D) * 0.1), dev(torch.randn(D) * 0.1), dev(torch.randn(M, D))
    rs = dev((torch.rand(M // rps) > 0.3).float() / 0.7) if drop else None
    tiles, grid = mlp_walk(M)
    if M > 4096:
        assert_walk(tiles, grid, "mlp_tc_kernel")
    h = torch.nn.functional.gelu(a.double() @ w1.double().T + b1.double()).half().double()       # hidden is an f16 operand
    y = h @ w2.double().T + b2.double()
    if drop:
        y = y * rs.double().repeat_interleave(rps).view(-1, 1)
    ref = x.double() + y
    g, bt = dev(1 + 0.1 * torch.randn(D)), dev(0.1 * torch.randn(D))
    xd = x.clone()
    out_ln = ops.mlp_bf16(a, w1, b1, w2, b2, xd, rs, rps, g if ln else None, bt if ln else None, 1e-6)
    coords = lambda t: "row tile %d" % t
    worst = (xd.double() - ref).abs().reshape(tiles, -1).amax(1) / float(ref.abs().max())
    assert not bool((worst >= 3e-3).any()), locate(worst >= 3e-3, grid, coords, "mlp x: relative error >= 3e-3", worst)
    if ln:
        ref_ln = O._ln(ref, g.double(), bt.double(), 1e-6)
        worst = (out_ln.double() - ref_ln).abs().reshape(tiles, -1).amax(1) / float(ref_ln.abs().max())
        assert not bool((worst >= 8e-3).any()), locate(worst >= 8e-3, grid, coords, "mlp LayerNorm: relative error >= 8e-3", worst)


# ------------------------------------------------------------------------------------------------ LN / attention
@pytest.mark.parametrize("D", [64, 128, 256, 512])
def test_layernorm(D):
    ops = _ops()
    torch.manual_seed(D)
    x, g, b = torch.randn(37, D) * 3 + 1, torch.randn(D), torch.randn(D)
    ref = O._ln(x.double(), g.double(), b.double(), 1e-6)
    out = ops.layernorm(dev(x), dev(g), dev(b), 1e-6).cpu()
    assert rel_err(out.numpy(), ref.numpy()) < 2e-6


@pytest.mark.parametrize("stage,local", [(0, True), (1, True), (1, False), (2, False)])
def test_svtr_attention(stage, local):
    ops = _ops()
    d, heads = O.SVTR_DIMS[stage], O.SVTR_HEADS[stage]
    H, W = O.SVTR_GRID[stage]
    N = H * W
    torch.manual_seed(stage)
    qkv = torch.randn(3, N, 3 * d)
    q, k, v = qkv.double().reshape(3, N, 3, heads, 32).permute(2, 0, 3, 1, 4)
    att = (q * 32 ** -0.5) @ k.transpose(-1, -2)
    if local:
        att = att + O.local_mask(H, W, dtype=torch.float64)
    ref = (torch.softmax(att, -1) @ v).permute(0, 2, 1, 3).reshape(3, N, d)
    out = ops.svtr_attention(dev(qkv), heads, H, W, local).cpu()
    assert rel_err(out.numpy(), ref.numpy()) < 3e-6


_ATTN_STAGES = [(0, True), (1, True), (1, False), (2, False)]


@pytest.mark.parametrize("stage,local,groups,wscale", _kept_ids([(st, lo, 5, 1.5) for st, lo in _ATTN_STAGES], 2)
                         + [(st, lo, 148, ws) for ws in (1.5, 6.0) for st, lo in _ATTN_STAGES])
def test_svtr_attention_tcgen05(stage, local, groups, wscale):
    """Tensor-core attention (QK^T and PV on tcgen05, softmax in registers) vs fp64 on the same bf16 inputs.  At 148
    groups every CTA walks >= 4 items (asserted), so K/V blocks numbered across items, Q handed back between items and
    the next item's first S behind the last P V are exercised; wscale = 6 (peaked scores) moves the running maximum
    across key blocks of different items."""
    ops = _ops()
    d, heads = O.SVTR_DIMS[stage], O.SVTR_HEADS[stage]
    H, W = O.SVTR_GRID[stage]
    N = H * W
    items, grid = attn_tc_walk(groups, N, heads)
    if groups > 5:
        assert_walk(items, grid, "attn_tc_kernel")
    torch.manual_seed(10 + stage)
    qkv = dev((torch.randn(groups, N, 3 * d) * wscale).bfloat16())
    q, k, v = qkv.double().reshape(groups, N, 3, heads, 32).permute(2, 0, 3, 1, 4)
    att = (q * 32 ** -0.5) @ k.transpose(-1, -2)
    if local:
        att = att + O.local_mask(H, W, dtype=torch.float64).cuda()
    ref = torch.softmax(att, -1) @ v                                 # [groups, heads, N, 32]
    out = torch.full((groups, N, d), float("nan"), device="cuda", dtype=torch.bfloat16)
    ops.svtr_attention_bf16(qkv, heads, H, W, local, out=out)
    got = out.double().reshape(groups, N, heads, 32).permute(0, 2, 1, 3)
    # items t = (g * heads + h) * N/128 + query tile (attn_tc.cu:58); bf16 probabilities and bf16 output: 1e-2
    worst = (got - ref).abs().nan_to_num(float("inf")).reshape(items, -1).amax(1) / float(ref.abs().max())
    nqt = N // 128
    coords = lambda t: "group %d, head %d, query tile %d" % (t // (nqt * heads), t // nqt % heads, t % nqt)
    assert not bool((worst >= 1e-2).any()), locate(worst >= 1e-2, grid, coords, "attn_tc: relative error >= 1e-2", worst)


# ------------------------------------------------------------------------------------------------ experts
def _expert_case(cc, B, seed):
    sd = synth.synth_state_dict(cc, seed)
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    return sd, img, tgt, lens, dom


@pytest.mark.parametrize("mode", ["eval", "train"])
def test_svtr_experts_fp32_match_oracle(mode):
    ops = _ops()
    from mrn_b200 import _lib as L
    cc, B, seed = (37, 61, 96), 3, 111
    sd, img, tgt, lens, dom = _expert_case(cc, B, seed)
    I = len(cc)
    drop = synth.synth_drop_scales(I, B, O.svtr_drop_path_rates(), seed) if mode == "train" else None
    with torch.no_grad():
        o = O.mrn_forward(sd, I, img, True, True, bn_mode="batch" if mode == "train" else "eval", drop_scales=drop)
    pack = ops.SvtrPack(sd, I, "cuda", L.PREC_FP32)
    feats, logits = ops.svtr_experts_forward(pack, dev(img), bn_batch_stats=mode == "train", update_running=mode == "train",
                                             drop_scales=dev(drop) if drop is not None else None, chunk=2)
    assert rel_err(feats.cpu().numpy(), o["features"].numpy()) < 1e-4
    for i in range(I):
        assert rel_err(logits[i].cpu().numpy(), o["preds"][i].numpy()) < 1e-4
    g = load_golden("svtr_mrn_i3_b3")          # and directly against the reference's own output
    key = "train_features" if mode == "train" else "features"
    assert rel_err(gview(feats.cpu(), g), g[key]) < 1e-4
    if mode == "train":
        rm = pack.bn_running_stats()[0][0].cpu().numpy()
        assert np.abs(rm - g["train_bn1_running_mean_e0"]).max() < 1e-5


def test_svtr_experts_bf16_within_budget():
    ops = _ops()
    from mrn_b200 import _lib as L
    cc, B, seed = (37, 61, 96), 3, 111
    sd, img, tgt, lens, dom = _expert_case(cc, B, seed)
    with torch.no_grad():
        o = O.mrn_forward(sd, 3, img, True, True)
    pack = ops.SvtrPack(sd, 3, "cuda", L.PREC_BF16)
    feats, logits = ops.svtr_experts_forward(pack, dev(img))
    assert rel_err(feats.cpu().numpy(), o["features"].numpy()) < 2e-2
    for i in range(3):
        assert rel_err(logits[i].cpu().numpy(), o["preds"][i].numpy()) < 2e-2      # north-star bf16 tolerance


# ------------------------------------------------------------------------------------------------ router
def _router_arena(sd, I, device="cuda"):
    ops = _ops()
    n, off = ops.router_param_offsets(I)
    arena = torch.zeros(n, dtype=torch.float32)
    for k, name in enumerate(ops.ROUTER_PARAM_NAMES):
        arena[off[k]:off[k] + sd[name].numel()] = sd[name].reshape(-1).float()
    return arena.to(device), off


@pytest.mark.parametrize("name", ["dm_router_i3_b2", "dm_router_i6_b1"])
def test_dm_router_forward_backward(name):
    ops = _ops()
    g = load_golden(name)
    I, B, seed = int(g["I"]), int(g["B"]), int(g["seed"])
    sd = {k: synth.synth_tensor(seed, k, s) for k, s in synth.router_shapes(I).items()}
    x = synth.randn(seed, "router_x", (B, I, 64, 256))
    dy = synth.randn(seed, "router_dy", (B, I, 64, 256))
    arena, off = _router_arena(sd, I)
    ws = ops.RouterWorkspace()
    out, scores, gate, index = ops.router_forward(arena, dev(x), ws, with_backward=True)
    assert rel_err(gview(out.cpu(), g), g["out"]) < 1e-4
    sdd = {k: v.double() for k, v in sd.items()}
    r_ref = O.gate_scores(sdd, O.dm_router(sdd, x.double()))
    assert rel_err(scores.cpu().numpy(), r_ref.numpy()) < 1e-4
    assert np.abs(gate.cpu().numpy() - torch.softmax(r_ref, -1).numpy()).max() < 1e-4
    grads = torch.empty_like(arena)
    dx = ops.dm_router_backward(arena, dev(x), dev(dy), grads, ws, want_dx=True)
    assert rel_err(gview(dx.cpu(), g), g["dx"]) < 2e-4
    gc = grads.cpu()
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        if not pname.startswith("dm_router.0."):
            continue
        got = gc[off[k]:off[k] + sd[pname].numel()].reshape(sd[pname].shape)
        assert rel_err(gview(got, g), g["grad." + pname[len("dm_router.0."):]]) < 5e-4, pname


@pytest.mark.parametrize("name", ["dm_router_i3_b2", "dm_router_i6_b1"])
def test_dm_router_tensor_core_engine(name):
    """Router contractions on tcgen05 (bf16 operands read K-major / MN-major where they lie, fp32 accumulate, split-K
    weight gradients): within the bf16 budget of the fp32 reference."""
    ops = _ops()
    from mrn_b200 import _lib as L
    g = load_golden(name)
    I, B, seed = int(g["I"]), int(g["B"]), int(g["seed"])
    sd = {k: synth.synth_tensor(seed, k, s) for k, s in synth.router_shapes(I).items()}
    x = synth.randn(seed, "router_x", (B, I, 64, 256))
    dy = synth.randn(seed, "router_dy", (B, I, 64, 256))
    arena, off = _router_arena(sd, I)
    ws = ops.RouterWorkspace()
    out, scores, gate, index = ops.router_forward(arena, dev(x), ws, with_backward=True, prec=L.PREC_BF16)
    assert rel_err(gview(out.cpu(), g), g["out"]) < 2e-2
    grads = torch.empty_like(arena)
    dx = ops.dm_router_backward(arena, dev(x), dev(dy), grads, ws, want_dx=True, prec=L.PREC_BF16)
    assert rel_err(gview(dx.cpu(), g), g["dx"]) < 3e-2
    gc = grads.cpu()
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        if not pname.startswith("dm_router.0."):
            continue
        got = gc[off[k]:off[k + 1]][:sd[pname].numel()].reshape(sd[pname].shape)
        assert rel_err(gview(got, g), g["grad." + pname[len("dm_router.0."):]]) < 3e-2, pname


@pytest.mark.parametrize("prec_name", ["fp32", "bf16"])
@pytest.mark.parametrize("I,B,T", [(6, 3, 64), (3, 5, 64), (6, 2, 63), (6, 256, 64)])
def test_router_training_backward_matches_fp64_autograd(prec_name, I, B, T):
    """mrnb_router_backward (il_modules/mrn.py:342,360: loss = 15 * CTC + CrossEntropy(gate, domain)) against the fp64
    autograd of the oracle for L = sum(dgate_ctc * gate) + CE(gate, domain): EVERY parameter gradient (gate head +
    DM_Router) and the CE loss.  bf16 = the gate-head driven tensor-core path (rank-one d_out, LayerNorm 1 folded into
    proj_1, collapsed last Linear), incl. the T = 63 run padded to 64 frames; fp32 = the generic CUDA-core path.
    B = 256 is the benchmarked batch (split-K factors and tile widths depend on B); the fp64 autograd runs on the device."""
    ops = _ops()
    from mrn_b200 import _lib as L
    seed = 70 + I + T
    prec = L.PREC_BF16 if prec_name == "bf16" else L.PREC_FP32
    tol_gate, tol_g = (2e-2, 5e-2) if prec_name == "bf16" else (1e-4, 5e-4)   # 5e-2: the bf16 router-gradient budget of test_gpu_step.py
    sd = {k: synth.synth_tensor(seed, k, s) for k, s in synth.router_shapes(I, T=T).items()}
    x = synth.randn(seed, "router_x", (B, I, T, 256))
    dgc = synth.randn(seed, "dgate_ctc", (B, I)) * 0.3
    dom = torch.tensor([(3 * b + 1) % I for b in range(B)], dtype=torch.int64)
    sdd = {k: v.cuda().double().requires_grad_(True) for k, v in sd.items()}
    r = O.gate_scores(sdd, O.dm_router(sdd, x.cuda().double()))
    gate_ref = torch.softmax(r, -1)
    ce = torch.nn.functional.cross_entropy(gate_ref, dom.cuda())    # the reference applies CE to the softmaxed gate
    ((gate_ref * dgc.cuda().double()).sum() + ce).backward()
    n, off = ops.router_param_offsets(I, T)
    arena = torch.zeros(n, dtype=torch.float32)
    for k, name in enumerate(ops.ROUTER_PARAM_NAMES):
        arena[off[k]:off[k] + sd[name].numel()] = sd[name].reshape(-1)
    arena = arena.cuda()
    ws = ops.RouterWorkspace()
    out, scores, gate, index = ops.router_forward(arena, dev(x), ws, with_backward=True, prec=prec)
    assert np.abs(gate.cpu().numpy() - gate_ref.detach().cpu().numpy()).max() < tol_gate
    grads = torch.full_like(arena, float("nan"))
    # the CTC part of dL/dgate is an input of the kernel; with the GPU's own gate the two losses differ only through
    # the (tolerated) gate deviation
    taski = ops.router_backward(arena, dev(x), gate, dev(dgc), dom.cuda(), grads, ws, prec=prec)
    assert abs(float(taski) - float(ce.detach())) < 1e-3
    gc = grads.cpu()
    assert torch.isfinite(gc).all()
    gmax = max(float(v.grad.abs().max()) for v in sdd.values())
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        got = gc[off[k]:off[k] + sd[pname].numel()].reshape(sd[pname].shape).double().numpy()
        ref = sdd[pname].grad.cpu().numpy()
        # route.bias has an analytically zero gradient (softmax shift invariance): floor the yardstick
        scale = max(float(np.abs(ref).max()), 1e-3 * gmax)
        err = float(np.abs(got - ref).max()) / scale
        assert err < tol_g, (pname, err)


@pytest.mark.parametrize("prec_name", ["fp32", "bf16"])
@pytest.mark.parametrize("I,B", [(2, 3), (6, 2), (6, 256)])
def test_dm_router_63_frames(prec_name, I, B):
    """CRNN's T = 63 (modules/model.py:322-323).  fp32: the CUDA-core engine on the unpadded problem; bf16: the tcgen05
    engine on the problem padded to 64 frames (zero frame, zero weight rows / columns, masked LayerNorm over frames)
    -- both against the fp64 autograd of the oracle, incl. the un-padded gradient arena and the input gradient.  B = 256
    is the benchmarked batch; the fp64 autograd runs on the device."""
    ops = _ops()
    from mrn_b200 import _lib as L
    T, seed = 63, 40 + I
    prec = L.PREC_BF16 if prec_name == "bf16" else L.PREC_FP32
    tol_o, tol_g = (2e-2, 3e-2) if prec_name == "bf16" else (1e-4, 5e-4)
    shapes = synth.router_shapes(I, T=T)
    sd = {k: synth.synth_tensor(seed, k, s) for k, s in shapes.items()}
    x = synth.randn(seed, "router_x", (B, I, T, 256))
    dy = synth.randn(seed, "router_dy", (B, I, T, 256))
    sdd = {k: v.cuda().double().requires_grad_(True) for k, v in sd.items()}
    xd = x.cuda().double().requires_grad_(True)
    y = O.dm_router(sdd, xd)
    (y * dy.cuda().double()).sum().backward()
    r_ref = O.gate_scores({k: v.detach() for k, v in sdd.items()}, y.detach()).cpu()
    y, xg = y.detach().cpu(), xd.grad.cpu()
    n, off = ops.router_param_offsets(I, T)
    arena = torch.zeros(n, dtype=torch.float32)
    for k, name in enumerate(ops.ROUTER_PARAM_NAMES):
        arena[off[k]:off[k] + sd[name].numel()] = sd[name].reshape(-1)
    arena = arena.cuda()
    ws = ops.RouterWorkspace()
    out, scores, gate, index = ops.router_forward(arena, dev(x), ws, with_backward=True, prec=prec)
    assert out.shape == (B, I, T, 256)
    assert rel_err(out.cpu().numpy(), y.numpy()) < tol_o
    assert rel_err(scores.cpu().numpy(), r_ref.numpy()) < tol_o
    assert np.abs(gate.cpu().numpy() - torch.softmax(r_ref, -1).numpy()).max() < tol_o
    grads = torch.full_like(arena, float("nan"))
    dx = ops.dm_router_backward(arena, dev(x), dev(dy), grads, ws, want_dx=True, prec=prec)
    assert dx.shape == (B, I, T, 256)
    assert rel_err(dx.cpu().numpy(), xg.numpy()) < tol_g
    gc = grads.cpu()
    for k, pname in enumerate(ops.ROUTER_PARAM_NAMES):
        got = gc[off[k]:off[k] + sd[pname].numel()].reshape(sd[pname].shape)
        if not pname.startswith("dm_router.0."):
            assert float(got.abs().max()) == 0.0           # gate-head slots are untouched by dm_router_backward
            continue
        assert rel_err(got.numpy(), sdd[pname].grad.cpu().numpy()) < tol_g, pname


# ------------------------------------------------------------------------------------------------ combine / CTC / decode
def _ragged_logits(cc, B, T, seed, scale=3.0):
    return [synth.randn(seed, f"z{i}", (B, T, c), scale) for i, c in enumerate(cc)]


def _dev_ragged(zs):
    ops = _ops()
    out = []
    for z in zs:
        ld = ops.round_up(z.shape[2], 4)
        buf = torch.zeros(z.shape[0], z.shape[1], ld, device="cuda")
        buf[:, :, :z.shape[2]] = z.cuda()
        out.append(buf[:, :, :z.shape[2]])
    return out


@pytest.mark.parametrize("cc,B,T", [((37, 61, 96), 5, 64), ((1899, 2224, 3844, 4968, 5041, 5153), 4, 64), ((50,), 3, 63),
                                    # the MLT17 class counts at B = 64: ~27 rows per CTA of the TMA-staged combine (asserted)
                                    ((1899, 2224, 3844, 4968, 5041, 5153), 64, 64)])
def test_combine_ctc_decode_match_oracle(cc, B, T):
    ops = _ops()
    seed = 5 + len(cc)
    I = len(cc)
    rows, grid = combine_walk(B, T)
    if B > 5:
        assert_walk(rows, grid, "combine_row_tma_kernel")
    zs = _ragged_logits(cc, B, T, seed)
    gate = torch.softmax(synth.randn(seed, "gate", (B, I), 2.0), -1)
    _, tgt, lens, _ = synth.synth_batch(B, cc, seed)
    tgt[0, :3] = torch.tensor([7, 7, 9]); lens[0] = 3           # repeated label
    if B > 2:
        lens[2] = 0                                             # empty target
    logits_ref = O.combine_soft([z.double() for z in zs], gate.double())
    nll_ref, grad_ref = O.ctc_nll_and_grad(logits_ref, tgt, lens)
    zd = _dev_ragged(zs)
    r = ops.gate_combine(zd, dev(gate), dev(tgt), dev(lens), want_logits=True, want_E=True, want_decode=True)
    worst = (r["logits"].cpu().double() - logits_ref).abs().reshape(B * T, -1).amax(1) / float(logits_ref.abs().max())
    assert not bool((worst >= 1e-6).any()), locate(worst >= 1e-6, grid, lambda t: "sample %d, frame %d" % divmod(t, T),
                                                  "combine logits: relative error >= 1e-6", worst)
    assert rel_err(r["lse"].cpu().numpy(), torch.logsumexp(logits_ref, -1).numpy()) < 1e-6
    pi = 15.0
    c = ops.ctc_lattice(r["lpe"], dev(tgt), dev(lens), r["zlab"], r["E"], grad_scale=pi / B, want_dgate=True, want_occ=True)
    assert rel_err(c["nll"].cpu().numpy(), nll_ref.numpy()) < 1e-5
    loss_ref = float((nll_ref / lens.clamp(min=1)).mean())
    assert abs(float(c["loss"].cpu()) - loss_ref) / abs(loss_ref) < 1e-5
    dg_ref = O.gate_grad_shortcut(logits_ref, [z.double() for z in zs], gate, tgt, lens, pi)
    assert rel_err(c["dgate"].cpu().numpy(), dg_ref.numpy()) < 1e-4
    # dense gradient (expert-training stage)
    dense = ops.ctc_dense_grad(r["logits"], r["lse"], c["occ"], c["nll"], dev(tgt), dev(lens), 1.0 / B)
    scale = (1.0 / (B * lens.clamp(min=1).double())).view(-1, 1, 1)
    # softmax - occupancy cancels on the blank column (occ ~ 0.95): fp32 log-space lattice, same as ATen's kernel
    assert rel_err(dense.cpu().numpy(), (grad_ref * scale).numpy()) < 3e-4
    # decode
    raw_ref, seqs_ref, conf_ref = O.greedy_decode(logits_ref.float())
    assert (r["amax"].cpu().long() == raw_ref).all()
    ids, n, conf = ops.greedy_decode(r["amax"], r["maxprob"])
    for b in range(B):
        assert int(n[b]) == len(seqs_ref[b]) and ids[b, :len(seqs_ref[b])].cpu().tolist() == seqs_ref[b]
    assert rel_err(conf.cpu().numpy(), conf_ref.numpy()) < 1e-4


def test_hard_route_and_ones_plateau_tie_break():
    """Eval route = one-hot gate; a row whose real logits are all < 1 must arg-max onto the FIRST padded column
    (index C_i), as torch.max does on the reference's ones-padding (modules/model.py:361-364)."""
    ops = _ops()
    cc, B, T = (20, 33), 2, 64
    zs = [-(synth.randn(3, "a", (B, T, 20)).abs()) - 0.1, synth.randn(3, "b", (B, T, 33), 3.0)]
    index = torch.tensor([0, 1])
    gate = torch.nn.functional.one_hot(index, 2).float()
    ref = O.combine_hard(zs, index)
    r = ops.gate_combine(_dev_ragged(zs), dev(gate), want_logits=True, want_decode=True)
    assert torch.equal(r["logits"].cpu(), ref)                       # bit exact: no arithmetic on the selected expert
    assert (r["amax"][0].cpu() == 20).all()                          # plateau hit -> first padded column
    assert (r["amax"].cpu().long() == ref.max(2)[1]).all()


def test_ctc_infeasible_target_is_zeroed():
    ops = _ops()
    B, T, Cc = 2, 4, 11
    z = [synth.randn(1, "z", (B, T, Cc))]
    tgt = torch.ones(B, 25, dtype=torch.long); tgt[0, :5] = torch.tensor([3, 3, 3, 3, 3]); tgt[1, :2] = torch.tensor([4, 5])
    lens = torch.tensor([5, 2], dtype=torch.int32)                   # 5 repeated labels need 9 frames > T=4
    gate = torch.ones(B, 1)
    r = ops.gate_combine(_dev_ragged(z), dev(gate), dev(tgt), dev(lens), want_E=True)
    c = ops.ctc_lattice(r["lpe"], dev(tgt), dev(lens), r["zlab"], r["E"], grad_scale=1.0, want_dgate=True)
    nll_ref, _ = O.ctc_nll_and_grad(z[0].double(), tgt, lens)
    assert float(c["nll"][0]) == 0.0 and float(c["dgate"][0].abs().max()) == 0.0
    assert abs(float(c["nll"][1]) - float(nll_ref[1])) < 1e-5


def test_clip_adam_matches_oracle():
    ops = _ops()
    torch.manual_seed(0)
    n = 100003
    p, g = torch.randn(n), torch.randn(n) * 0.3
    ref_p = {"a": p.clone()}
    state = dict(step=0, m={}, v={})
    pd, m, v = dev(p), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    for step in range(1, 4):
        gg = g * step
        norm_ref = O.clip_and_adam(ref_p, {"a": gg.clone()}, state, lr=5e-4)
        norm = ops.clip_adam(pd, dev(gg), m, v, 5e-4, step)
        assert abs(float(norm) - norm_ref) / norm_ref < 1e-5
        assert (pd.cpu() - ref_p["a"]).abs().max() < 2e-6


def test_ctc_nan_logits_propagate_like_torch():
    """zero_infinity zeroes only an INFINITE loss; NaN logits must surface as a NaN loss and NaN gate gradient
    (torch.nn.CTCLoss semantics, il_modules/base.py:131) instead of being silently reported as 0."""
    ops = _ops()
    B, T, Cc = 2, 8, 11
    z = [synth.randn(1, "z", (B, T, Cc))]
    z[0][0, 3, 2] = float("nan")
    tgt = torch.ones(B, 25, dtype=torch.long); tgt[:, :2] = torch.tensor([4, 5])
    lens = torch.tensor([2, 2], dtype=torch.int32)
    gate = torch.ones(B, 1)
    r = ops.gate_combine(_dev_ragged(z), dev(gate), dev(tgt), dev(lens), want_E=True)
    c = ops.ctc_lattice(r["lpe"], dev(tgt), dev(lens), r["zlab"], r["E"], grad_scale=1.0, want_dgate=True)
    ref = torch.nn.functional.ctc_loss(z[0].log_softmax(2).permute(1, 0, 2), tgt[:, :2], torch.full((B,), T), lens.long(),
                                       reduction="none", zero_infinity=True)
    assert torch.isnan(ref[0]) and torch.isnan(c["nll"][0].cpu()) and torch.isnan(c["loss"].cpu()).all()
    assert torch.isnan(c["dgate"][0].cpu()).all()
    assert abs(float(c["nll"][1]) - float(ref[1])) < 1e-4


def test_fused_mlp_is_deterministic_at_headline_size():
    """Regression for the round-1 NaN: the fused-MLP epilogue staging tile used to alias another warp's P tile, so a
    warp running one tile ahead corrupted a slower warp's rows.  At the headline row count every CTA walks ~40 tiles;
    reruns on identical inputs must be bitwise identical and match the fp32 reference."""
    ops = _ops()
    torch.manual_seed(0)
    for d, N in ((64, 512), (128, 256), (256, 128)):
        M = 6 * 256 * N
        x = torch.randn(M, d, device="cuda")
        a16 = ops.cast_bf16(x)
        w1 = torch.randn(4 * d, d, device="cuda") * d ** -0.5
        b1 = torch.randn(4 * d, device="cuda") * 0.1
        w2 = torch.randn(d, 4 * d, device="cuda") * (4 * d) ** -0.5
        b2 = torch.randn(d, device="cuda") * 0.1
        w1h, w2h = ops.cast_bf16(w1), ops.cast_f16(w2)
        ref = x + torch.nn.functional.gelu(a16.float() @ w1h.float().t() + b1) @ w2h.float().t() + b2
        outs = []
        for _ in range(5):
            xx = x.clone()
            ops.mlp_bf16(a16, w1h, b1, w2h, b2, xx, None, 1, None, None)
            outs.append(xx)
        torch.cuda.synchronize()
        for o in outs[1:]:
            assert torch.equal(o, outs[0]), d
        assert float((outs[0] - ref).abs().max() / ref.abs().max()) < 2e-3, d
        del ref, outs


@pytest.mark.parametrize("D,local,ln,drop,wscale,units", _kept_ids([(64, True, True, True, 1.5, 300), (64, False, False, False, 1.5, 300),
                                                                     (128, True, True, False, 1.5, 300), (128, False, True, True, 1.5, 300),
                                                                     (256, False, False, True, 1.5, 300), (64, False, False, False, 4.0, 300),
                                                                     (128, True, False, False, 4.0, 300)], 5) + [
                                                              # >= 4 units per CTA (asserted)
                                                              (64, True, True, True, 1.5, 600), (64, False, False, True, 4.0, 600),
                                                              (128, False, True, True, 1.5, 600), (128, True, True, False, 4.0, 600)])
def test_fused_mixer_tcgen05(D, local, ln, drop, wscale, units):
    """mrnb_mixer_bf16 (qkv GEMM -> attention -> proj + DropPath + residual [+ LayerNorm] in one persistent kernel)
    against the same math in torch fp32 on the bf16-rounded operands (modules/svtr.py:133-152, :201-203).  300 units:
    every CTA walks two or three units; 600 units: at least four, so the persistent pipeline (barrier parities, buffer
    reuse) goes through both parities of every double-buffered resource."""
    ops = _ops()
    torch.manual_seed(D + 7 * local)
    N, heads = 32768 // D, D // 32
    n_units, grid = mixer_walk(units)
    if units > 300:
        assert_walk(n_units, grid, "mixer_tc_kernel")
    H = N // 64
    x = torch.randn(units, N, D, device="cuda")
    a16 = ops.cast_bf16(torch.randn(units, N, D, device="cuda"))
    # wscale = 4: scores spread over tens of log2 units, so the running reference maximum moves between key blocks and the
    # in-place rescale of the TMEM accumulator (lazy rescaling) is exercised
    wqkv = ops.cast_bf16(torch.randn(3 * D, D, device="cuda") * (wscale / D ** 0.5))
    bqkv = torch.randn(3 * D, device="cuda") * 0.2
    wp = ops.cast_bf16(torch.randn(D, D, device="cuda") / D ** 0.5)
    bp = torch.randn(D, device="cuda") * 0.2
    rs = ((torch.rand(units, device="cuda") > 0.2).float() / 0.8).contiguous() if drop else None
    g = (1.0 + 0.1 * torch.randn(D, device="cuda")) if ln else None
    bt = (0.1 * torch.randn(D, device="cuda")) if ln else None
    # reference
    bf = lambda t: t.to(torch.bfloat16).float()
    qkv = bf(a16.float() @ wqkv.float().t() + bqkv).view(units, N, 3, heads, 32).permute(2, 0, 3, 1, 4)
    q, k, v = qkv[0], qkv[1], qkv[2]
    att = (q @ k.transpose(-1, -2)) * 32 ** -0.5
    if local:
        hh, ww = torch.arange(N, device="cuda") // 64, torch.arange(N, device="cuda") % 64
        ok = ((hh[:, None] - hh[None, :]).abs() <= 3) & ((ww[:, None] - ww[None, :]).abs() <= 5)
        att = att.masked_fill(~ok, float("-inf"))
    o = bf((att.softmax(-1) @ v).permute(0, 2, 1, 3).reshape(units, N, D))
    y = o @ wp.float().t() + bp
    ref = x + y * (rs.view(-1, 1, 1) if drop else 1.0)
    xx = x.clone()
    lo = ops.mixer_bf16(a16, wqkv, bqkv, wp, bp, xx, local, rs, g, bt, 1e-6)
    torch.cuda.synchronize()
    if wscale > 2:
        # near one-hot softmax: bf16 rounding of q, k moves individual probabilities by tens of percent, so the yardstick is
        # the unfused tcgen05 pipeline (qkv GEMM -> attention kernel -> proj GEMM), which rounds the same operands
        qkv16 = ops.linear_bf16(a16.view(-1, D), wqkv, bqkv, None, False, out_f32=False)
        att16 = ops.svtr_attention_bf16(qkv16.view(units, N, 3 * D), heads, H, 64, int(local))
        y = ops.linear_bf16(att16.view(-1, D), wp, bp, None, False, out_f32=True).view(units, N, D)
        ref = x + y * (rs.view(-1, 1, 1) if drop else 1.0)
    tol = (5e-2 if wscale > 2 else 3e-2) * float(y.abs().max())
    worst = (xx - ref).abs().nan_to_num(float("inf")).reshape(units, -1).amax(1)
    coords = lambda t: "unit %d" % t
    assert not bool((worst >= tol).any()), locate(worst >= tol, grid, coords, "mixer x: over budget (err / budget)", worst / tol)
    if ln:
        lref = torch.nn.functional.layer_norm(ref, (D,), g, bt, 1e-6)
        ltol = 2e-2 * float(lref.abs().max())      # bf16 output (ulp 2^-6 at |v| ~ 4) of a bf16-operand branch
        worst = (lo.float() - lref).abs().nan_to_num(float("inf")).reshape(units, -1).amax(1)
        assert not bool((worst >= ltol).any()), locate(worst >= ltol, grid, coords, "mixer LayerNorm: over budget (err / budget)",
                                                       worst / ltol)
    # determinism across reruns (persistent pipeline: no cross-warp / cross-unit hazards)
    x2 = x.clone()
    ops.mixer_bf16(a16, wqkv, bqkv, wp, bp, x2, local, rs, g, bt, 1e-6)
    assert torch.equal(x2, xx)
