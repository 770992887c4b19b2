"""Kernel-level parity of the bf16 training attention (the stage-0 step's tensor-core path, svtr_train.cu
attn_tc_forward / attn_tc_backward): the fused score / softmax kernel, the fused dP / dS kernel and the four value-side
head GEMMs (O = P V, dV = P^T dO, dQ = scale dS K, dK = scale dS^T Q), each against fp64 autograd-equivalent math of
softmax(scale q k^T + Local mask) v on the same bf16-rounded q, k, v and the same fp32 dO.

The batch is chosen so that the score kernel and every head GEMM give each CTA at least four work items; a failure names
the (sample, head, 128-row tile) item and its place in its CTA's walk.  The fp64 reference runs on the device: at these
sizes it would take minutes on the host."""
import math

import pytest
import torch

from oracle import mrn_oracle as O
from persistent_walk import assert_walk, attn_sp_walk, cdiv, locate, tc_gemm2_walk

pytestmark = pytest.mark.gpu

SCALE = 32 ** -0.5
U = 2.0 ** -8                 # bf16 unit roundoff (round to nearest, 8 significant bits)
TINY = 2.0 ** -120            # ex2.approx.ftz flushes results below 2^-126 to zero


def _ops():
    from mrn_b200 import ops
    return ops


def _heads_view(t, B, heads):
    """[B, N, heads * 32] -> [B * heads, N, 32]"""
    N = t.shape[1]
    return t.reshape(B, N, heads, 32).permute(0, 2, 1, 3).reshape(B * heads, N, 32)


def _item_max(x, B, heads, N):
    """per-item max of a [B*heads, N, C] tensor over its 128-row tiles -> [B*heads * N/128] in the kernels' walk order
    (t = (b * heads + h) * N/128 + row tile)"""
    return x.reshape(B * heads * (N // 128), -1).amax(1)


@pytest.mark.parametrize("wscale", [1.5, 6.0])
@pytest.mark.parametrize("stage,local", [(0, True), (1, True), (1, False), (2, False)])
def test_attn_train_tcgen05_matches_fp64(stage, local, wscale):
    """Budgets, per element, with u = 2^-8 the bf16 unit roundoff and n = N keys:

    P   kernel: fp32 scores of exact bf16 products, ex2.approx, fp32 sums, P16 = bf16(p).  A score error e shifts the
        probabilities of its row by a factor within exp(+-2e); e <= 2^-18 scale sum|q_i k_i| (32-term fp32 accumulation
        with room for the exponent argument's rounding), e_P = 2^-15 (fp32 row sum, ex2.approx, division) + 3 e_rowmax, so
        |P16 - P| <= E_P = 1.01 P (u + e_P) + 2^-120.
    O   O16 = bf16(P16 v): E_O = 1.02 (E_P |v| + n 2^-23 P |v| + u |O|)   (n 2^-23: n-term fp32 accumulation, allowing
        a truncating adder); also max |dO| per item <= 1e-2 max |O| per item, as for the inference attention.
    dS  dP' = dO16 v^T: |dP' - dP| <= (u + 2^-17) |dO| |v|^T; D' = dO . O16 in fp32: |D' - D| <= |dO| . E_O + 2^-18 |dO| . |O|;
        with d = dP' - D' - (dP - D) bounded by their sum, dS16 = bf16(P16 (dP' - D')):
        E_dS = 1.02 (E_P (|dP - D| + d) + P d + u |dS|).
    dV  dV16 = bf16(P16^T dO16): E_dV = 1.02 (E_P^T |dO| + (u + n 2^-23) P^T |dO| + u |dV|).
    dQ  dQ16 = bf16(scale dS16 k): E_dQ = 1.02 (scale (E_dS |k| + n 2^-23 (|dS| + E_dS) |k|) + u |dQ|); dK likewise with
        dS^T and q.
    Exact: P and dS are 0 outside the Local window, every output element is written (NaN pre-fill), each row of P sums
    to 1 within 1.01 (u + e_P) (at most 2^-7 here, far inside N 2^-9), and a query row with q = 0 is the uniform
    distribution over exactly its visible keys."""
    ops = _ops()
    dev = "cuda"
    d, heads = O.SVTR_DIMS[stage], O.SVTR_HEADS[stage]
    H, W = O.SVTR_GRID[stage]
    N = H * W
    MT = N // 128
    # batch: at least four items per CTA for the score kernel and for the head GEMMs (M = N rows, N = 32 -> BN = 64)
    cap_sp = attn_sp_walk(10 ** 6, N, heads)[1]
    cap_gm = tc_gemm2_walk(N, 32, N, groups=10 ** 6)[1]
    B = cdiv(4 * max(cap_sp, cap_gm), heads * MT)
    sp_items, sp_grid = attn_sp_walk(B, N, heads)
    gm_items, gm_grid = tc_gemm2_walk(N, 32, N, groups=B * heads)
    assert_walk(sp_items, sp_grid, "attn_sp_kernel")
    assert_walk(gm_items, gm_grid, "tc_gemm2_kernel (head GEMMs)")
    G = B * heads

    gen = torch.Generator().manual_seed(1000 * stage + 10 * int(local) + int(wscale))
    qkv = (torch.randn(B, N, 3 * d, generator=gen) * wscale).bfloat16()
    zb, zn = B - 1, 1 * W + 2                      # q = 0 for one token of the last sample (late in every CTA's walk)
    qkv[zb, zn, :d] = 0
    dO = torch.randn(B, N, d, generator=gen)
    qkv, dO = qkv.to(dev), dO.to(dev)
    dO16 = dO.bfloat16()

    # ---- kernels, outputs pre-filled with NaN
    nan16 = lambda *s: torch.full(s, float("nan"), device=dev, dtype=torch.bfloat16)
    P16, O16 = ops.attn_tc_train_forward(qkv, heads, W, local, P=nan16(G, N, N), O=nan16(B, N, d))
    dS16, dqkv16 = ops.attn_tc_train_backward(qkv, O16, P16, dO, dO16, heads, dS=nan16(G, N, N), dqkv=nan16(B, N, 3 * d))
    torch.cuda.synchronize()

    # ---- fp64 reference on the same bf16 q, k, v and fp32 dO
    x = qkv.double()
    q, k, v = (_heads_view(x[..., j * d:(j + 1) * d], B, heads) for j in range(3))
    go = _heads_view(dO.double(), B, heads)
    vis = (O.local_mask(H, W, dtype=torch.float64) == 0).to(dev) if local else torch.ones(N, N, dtype=torch.bool, device=dev)
    S = SCALE * (q @ k.transpose(1, 2))
    P = torch.softmax(S.masked_fill(~vis, float("-inf")), -1)
    Oref = P @ v
    dP = go @ v.transpose(1, 2)
    D = (go * Oref).sum(-1, keepdim=True)
    dS = P * (dP - D)
    dV, dQ, dK = P.transpose(1, 2) @ go, SCALE * (dS @ k), SCALE * (dS.transpose(1, 2) @ q)

    Pk, dSk = P16.double(), dS16.double()
    Ok = _heads_view(O16.double(), B, heads)
    dQk, dKk, dVk = (_heads_view(dqkv16[..., j * d:(j + 1) * d].double(), B, heads) for j in range(3))

    def coords(t):
        g, mt = divmod(t, MT)
        return "sample %d, head %d, row tile %d" % (g // heads, g % heads, mt)

    # ---- exact checks
    written = [("P", P16, sp_grid), ("dS", dS16, sp_grid), ("O", _heads_view(O16, B, heads), gm_grid)]
    written += [(name, _heads_view(dqkv16[..., j * d:(j + 1) * d], B, heads), gm_grid) for j, name in enumerate(("dQ", "dK", "dV"))]
    for name, t, grid in written:
        bad = ~torch.isfinite(t.float().reshape(G * MT, -1)).all(1)
        assert not bool(bad.any()), locate(bad, grid, coords, "%s: elements never written (NaN pre-fill)" % name)
    if local:
        for name, t in (("P", P16), ("dS", dS16)):
            outside = (t != 0) & ~vis
            bad = outside.reshape(G * MT, -1).any(1)
            assert not bool(bad.any()), locate(bad, sp_grid, coords, "%s: non-zero outside the 7 x 11 Local window" % name)
    # q = 0: uniform over exactly the visible keys of that query, in every head of the sample
    for h in range(heads):
        row, vrow = P16[zb * heads + h, zn], vis[zn]
        cnt = int(vrow.sum())
        assert torch.equal(row != 0, vrow), ("q = 0 row: support differs from the visible keys", zb, h, zn)
        vals = row[vrow].float()
        assert bool((vals == vals[0]).all()) and abs(float(vals[0]) * cnt - 1.0) <= U, \
            ("q = 0 row is not uniform over its %d visible keys" % cnt, vals.unique().tolist())

    # ---- budgets
    eS = (2.0 ** -18) * SCALE * (q.abs() @ k.abs().transpose(1, 2)).masked_fill(~vis, 0).amax(-1, keepdim=True)
    eP = 2.0 ** -15 + 3 * eS
    EP = 1.01 * P * (U + eP) + TINY
    acc = N * 2.0 ** -23

    def check(name, got, ref, tol, grid):
        r = (got - ref).abs() / tol
        worst = _item_max(r, B, heads, N)
        assert not bool((worst > 1).any()), locate(worst > 1, grid, coords, "%s outside its budget (err / budget)" % name, worst)

    check("P", Pk, P, EP, sp_grid)
    rs = (Pk.sum(-1) - 1).abs()
    rbad = _item_max((rs / (1.01 * (U + eP[..., 0]) + N * TINY)).unsqueeze(-1), B, heads, N)
    assert not bool((rbad > 1).any()), locate(rbad > 1, sp_grid, coords, "P: row sums off 1", rbad)

    EO = 1.02 * (EP @ v.abs() + acc * (P @ v.abs()) + U * Oref.abs())
    check("O", Ok, Oref, EO, gm_grid)
    orel = _item_max((Ok - Oref).abs(), B, heads, N) / _item_max(Oref.abs(), B, heads, N)
    assert not bool((orel > 1e-2).any()), locate(orel > 1e-2, gm_grid, coords, "O: relative error per item > 1e-2", orel)

    dd = (U + 2.0 ** -17) * (go.abs() @ v.abs().transpose(1, 2)) \
        + ((go.abs() * EO).sum(-1, keepdim=True) + 2.0 ** -18 * (go.abs() * Oref.abs()).sum(-1, keepdim=True))
    EdS = 1.02 * (EP * ((dP - D).abs() + dd) + P * dd + U * dS.abs())
    check("dS", dSk, dS, EdS, sp_grid)
    del dd

    EdV = 1.02 * (EP.transpose(1, 2) @ go.abs() + (U + acc) * (P.transpose(1, 2) @ go.abs()) + U * dV.abs())
    check("dV", dVk, dV, EdV, gm_grid)
    aS = dS.abs() + EdS
    EdQ = 1.02 * (SCALE * (EdS @ k.abs() + acc * (aS @ k.abs())) + U * dQ.abs())
    check("dQ", dQk, dQ, EdQ, gm_grid)
    EdK = 1.02 * (SCALE * (EdS.transpose(1, 2) @ q.abs() + acc * (aS.transpose(1, 2) @ q.abs())) + U * dK.abs())
    check("dK", dKk, dK, EdK, gm_grid)
