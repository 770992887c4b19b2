"""Work-item bookkeeping for the scaled parity tests of the persistent kernels.

Every tensor-core kernel on the hot path is persistent: CTA c walks items t = c, c + grid, c + 2 grid, ...  and carries
barrier phases, TMEM accumulator buffers and operand-ring slots from one item to the next.  A test only reaches that
walk when every CTA gets several items, so each scaled case computes here the item count and the grid its launcher
picks (each function names the host line it mirrors) and asserts items >= 4 * grid: four items per CTA take a
double-buffered accumulator through both buffers and both parities.

When such a case fails, `locate` turns the per-item verdicts into the item's coordinates and its place in its CTA's
walk (ti = t // grid, accumulator buffer ti & 1, barrier parity (ti >> 1) & 1), which is what makes a failure here
fixable from the evidence."""
import torch


def n_sm():
    return torch.cuda.get_device_properties(0).multi_processor_count


def cdiv(a, b):
    return -(-a // b)


def assert_walk(items, grid, what):
    assert items >= 4 * grid, "%s: %d items on a grid of %d -- fewer than 4 per CTA" % (what, items, grid)


# ---- launcher grid rules -----------------------------------------------------------------------------------------
def tc_gemm_bn(N):
    """gemm_tc.cu:721 -- the 128-wide tile for N a multiple of 128 or N > 256, else 64."""
    return 128 if N >= 128 and (N % 128 == 0 or N > 256) else 64


def tc_gemm_walk(M, N, ln=False):
    """(tiles, grid) of tc_gemm_kernel: tiles n fastest, then m (gemm_tc.cu:113); two CTAs per SM, one with the fused
    LayerNorm (gemm_tc.cu:704)."""
    tiles = cdiv(N, tc_gemm_bn(N)) * cdiv(M, 128)
    return tiles, min(tiles, (1 if ln else 2) * n_sm())


def tc_gemm2_walk(M, N, K, splitk=1, groups=1, bn=None):
    """(tiles, grid) of tc_gemm2_kernel: tiles n fastest, then m, then group x split; the split count is the one with
    no empty split (gemm_tc2.cu:380-383); two CTAs per SM for BN <= 128, one for BN = 256 (gemm_tc2.cu:397)."""
    bn = bn or (128 if N >= 128 else 64)
    kb = K // 64
    splits = max(1, min(splitk, kb))
    per = cdiv(kb, splits)
    splits = cdiv(kb, per)
    tiles = cdiv(N, bn) * cdiv(M, 128) * groups * splits
    return tiles, min(tiles, (1 if bn > 128 else 2) * n_sm())


def attn_tc_walk(groups, N, heads):
    """(items, grid) of attn_tc_kernel: items = (query tile, head, group), query tile fastest (attn_tc.cu:57-58); two
    CTAs per SM (attn_tc.cu:321)."""
    items = (N // 128) * heads * groups
    return items, min(items, 2 * n_sm())


def attn_sp_walk(B, N, heads):
    """(items, grid) of attn_sp_kernel (score / softmax and dP / dS): items = (query tile, sample x head), query tile
    fastest; CTAs per SM limited by tensor memory, shared memory and threads (attn_train_tc.cu:245-250)."""
    items = B * heads * (N // 128)
    smem = 1024 + 2 * (128 * 64 * 2 + N * 64 * 2)
    per_sm = min(512 // N, (227 * 1024) // (smem + 5 * 1024), 2048 // (64 + 16 * 32))
    return items, min(items, n_sm() * per_sm)


def mlp_walk(M, groups=1):
    """(tiles, grid) of mlp_tc_kernel: one CTA per SM (mlp_tc.cu:432)."""
    tiles = (M // 128) * groups
    return tiles, min(tiles, n_sm())


def mixer_walk(units):
    """(units, grid) of mixer_tc_kernel: one CTA per SM (mixer_tc.cu:901)."""
    return units, min(units, n_sm())


def combine_walk(B, T):
    """(rows, grid) of combine_row_tma_kernel: one CTA per SM walking rows (ctc.cu:772)."""
    rows = B * T
    return rows, min(rows, n_sm())


# ---- localisation ------------------------------------------------------------------------------------------------
def locate(bad, grid, coords, what, err=None, limit=8):
    """Message naming the failing items.  bad: bool tensor over item indices t (in the kernel's walk order); coords(t) ->
    str of the item's coordinates; err: optional per-item error tensor of the same shape."""
    idx = torch.nonzero(bad.reshape(-1)).flatten().tolist()
    if not idx:
        return ""
    lines = []
    for t in idx[:limit]:
        ti = t // grid
        e = "" if err is None else " err %.3g" % float(err.reshape(-1)[t])
        lines.append("  item t=%d (%s): CTA %d, ti=%d, buffer %d, parity %d%s"
                     % (t, coords(t), t % grid, ti, ti & 1, (ti >> 1) & 1, e))
    tis = sorted({t // grid for t in idx})
    return ("%s: %d of %d items wrong (grid %d; walk positions ti = %s)\n" % (what, len(idx), bad.numel(), grid, tis[:16])
            + "\n".join(lines))
