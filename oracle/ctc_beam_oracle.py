"""fp64 restatement of the CTC prefix beam search (mrn_b200/csrc/ctc_beam.cu) and an exact labeling distribution to
check it against.  The reference has no beam search (test.py:211-221 decodes greedily); these define the semantics
the device kernels implement.
"""
import itertools
import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from .mrn_oracle import ctc_nll_and_grad

NEG_INF = float("-inf")


def ctc_topk(logits: torch.Tensor, K: int):
    """Per-frame candidates of the beam search.  logits: the combined logits [B,T,C] (e.g. combine_soft /
    combine_hard).  Returns (top_ids [B,T,K] int64: the K non-blank classes of highest value, ties to the smaller
    class, -1 past the C-1 real classes; top_lp [B,T,K] = value - logsumexp (-inf in unused slots); blank_lp [B,T])."""
    x = logits.double()
    B, T, C = x.shape
    lse = torch.logsumexp(x, -1)
    vals, idx = torch.sort(x[..., 1:], dim=-1, descending=True, stable=True)    # stable: equal values keep class order
    n = min(K, C - 1)
    top_ids = torch.full((B, T, K), -1, dtype=torch.long, device=x.device)
    top_lp = torch.full((B, T, K), NEG_INF, dtype=torch.float64, device=x.device)
    top_ids[..., :n] = idx[..., :n] + 1
    top_lp[..., :n] = vals[..., :n] - lse[..., None]
    return top_ids, top_lp, x[..., 0] - lse


def _lae(a: float, b: float) -> float:
    if a == NEG_INF:
        return b
    if b == NEG_INF:
        return a
    m = max(a, b)
    return m + math.log1p(math.exp(-abs(a - b)))


def ctc_prefix_beam_search(top_ids, top_lp, blank_lp, W: int, n_best: int = 1,
                           stats: Optional[dict] = None) -> List[Tuple[Tuple[int, ...], float]]:
    """CTC prefix beam search of ONE sample in fp64.  top_ids / top_lp [T,K], blank_lp [T].
    Returns up to n_best (labeling, log-probability) pairs, best first.  A `stats` dict receives "prune_margin": the
    smallest gap over all frames between the W-th kept and the best dropped candidate score (inf if none was dropped),
    i.e. how far the kept beams are from a near-tie that rounding could flip.

    Entries hold (prefix, pb, pnb), score = logaddexp(pb, pnb); the beam starts as {(): pb = 0, pnb = -inf}.  Per frame,
    with e the last label of entry j and only the frame's candidates (blank + the K classes):
      stay j:          pb' = score_j + blank_lp,  pnb' = pnb_j + lp_e if e is a candidate;
      extension j, c:  pnb = (pb_j if c == e else score_j) + lp_c.
    An extension whose prefix is another entry's prefix is log-added into that entry's stay.  The W best candidates by
    (score desc, stay before extension, parent rank, class) form the next beam; candidates scoring -inf are dropped."""
    T, K = len(top_ids), len(top_ids[0])
    beam = [((), 0.0, NEG_INF)]
    for t in range(T):
        cands = [(int(top_ids[t][k]), float(top_lp[t][k])) for k in range(K) if int(top_ids[t][k]) >= 0]
        lp_of = dict(cands)
        blank = float(blank_lp[t])
        slot = {pre: j for j, (pre, _, _) in enumerate(beam)}
        stays = []
        for pre, pb, pnb in beam:
            e = pre[-1] if pre else None
            stays.append([_lae(pb, pnb) + blank, pnb + lp_of[e] if e in lp_of else NEG_INF])
        exts = []
        for j, (pre, pb, pnb) in enumerate(beam):
            sc, e = _lae(pb, pnb), (pre[-1] if pre else None)
            for c, lp in cands:
                v = (pb if c == e else sc) + lp
                new = pre + (c,)
                if new in slot:
                    m = stays[slot[new]]
                    m[1] = _lae(m[1], v)
                else:
                    exts.append((v, 1, j, c, new, NEG_INF, v))
        allc = [(_lae(spb, spnb), 0, j, 0, beam[j][0], spb, spnb) for j, (spb, spnb) in enumerate(stays)] + exts
        allc = [c for c in allc if c[0] > NEG_INF]
        allc.sort(key=lambda c: (-c[0], c[1], c[2], c[3]))
        if stats is not None:
            gap = allc[W - 1][0] - allc[W][0] if len(allc) > W else float("inf")
            stats["prune_margin"] = min(stats.get("prune_margin", float("inf")), gap)
        beam = [(c[4], c[5], c[6]) for c in allc[:W]]
    return [(pre, _lae(pb, pnb)) for pre, pb, pnb in beam[:n_best]]


def ctc_labeling_distribution(logits: torch.Tensor) -> Dict[Tuple[int, ...], float]:
    """Exact log p(labeling | x) of every labeling for one sample, logits [T,C] (tiny T and C only: there are
    sum_n (C-1)^n labelings of length n <= T).  Labelings no alignment of T frames can emit get -inf."""
    T, C = logits.shape
    labs = [lab for n in range(T + 1) for lab in itertools.product(range(1, C), repeat=n)]
    tgt = torch.ones(len(labs), max(T, 1), dtype=torch.long)
    for r, lab in enumerate(labs):
        if lab:
            tgt[r, :len(lab)] = torch.tensor(lab, dtype=torch.long)
    lens = torch.tensor([len(lab) for lab in labs], dtype=torch.int32)
    x = logits.double()[None].expand(len(labs), T, C).contiguous()
    nll, _ = ctc_nll_and_grad(x, tgt, lens, want_grad=False)
    out = {}
    for r, lab in enumerate(labs):
        need = len(lab) + sum(1 for a, b in zip(lab, lab[1:]) if a == b)     # repeats need a blank between them
        out[lab] = -float(nll[r]) if need <= T else NEG_INF                   # ctc_nll_and_grad zeroes infeasible losses
    return out


def collapse(path: Sequence[int]) -> Tuple[int, ...]:
    """Best-path labeling of a frame-wise class sequence: merge repeats, drop blank 0."""
    out, prev = [], None
    for s in path:
        if s != prev and s != 0:
            out.append(int(s))
        prev = s
    return tuple(out)
