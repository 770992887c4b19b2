"""The fp64 CTC prefix beam search (oracle/ctc_beam_oracle.py) against exact labeling probabilities: without pruning
it is exact, and on peaked frames it returns the greedy collapse.  CPU only."""
import math

import pytest
import torch

from oracle import ctc_beam_oracle as BO
from oracle import mrn_oracle as O


def _beam(logits, K, W, n_best):
    ids, lp, blank = BO.ctc_topk(logits[None], K)
    return BO.ctc_prefix_beam_search(ids[0].tolist(), lp[0].tolist(), blank[0].tolist(), W, n_best)


def test_labeling_distribution_sums_to_one_and_matches_brute_force():
    torch.manual_seed(0)
    x = torch.randn(4, 3, dtype=torch.float64) * 2
    dist = BO.ctc_labeling_distribution(x)
    assert len(dist) == 31
    assert abs(sum(math.exp(v) for v in dist.values()) - 1.0) < 1e-12
    for lab in ((), (1,), (2, 2), (1, 2, 1), (1, 1, 1, 1)):
        assert abs(math.exp(dist[lab]) - math.exp(-O.ctc_brute_force(x, list(lab)))) < 1e-12, lab   # (1,1,1,1): 0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_unpruned_beam_is_exact(seed):
    """K = C-1 and W >= the number of reachable prefixes: every labeling keeps all its alignments."""
    torch.manual_seed(seed)
    T, C, W = 4, 3, 32
    x = torch.randn(T, C, dtype=torch.float64) * 1.5
    exact = {k: v for k, v in BO.ctc_labeling_distribution(x).items() if v > float("-inf")}
    got = _beam(x, C - 1, W, W)
    assert len(got) == len(exact)
    for lab, s in got:
        assert abs(s - exact[lab]) < 1e-9, lab
    ranked = sorted(exact.values(), reverse=True)
    for r, (lab, s) in enumerate(got):
        # the beam's order is the exact ranking wherever neighbouring probabilities are separated
        if (r == 0 or ranked[r - 1] - ranked[r] > 1e-9) and (r + 1 == len(ranked) or ranked[r] - ranked[r + 1] > 1e-9):
            assert abs(exact[lab] - ranked[r]) < 1e-9, (r, lab)


def test_beam_merges_prefixes_with_repeats():
    """Labeling (1, 1) needs a blank between the two labels; (1,) collects six of the eight paths."""
    T, C = 3, 2
    x = torch.zeros(T, C, dtype=torch.float64)         # uniform: every path has probability 2^-3
    exact = BO.ctc_labeling_distribution(x)
    got = dict(_beam(x, 1, 8, 8))
    assert abs(math.exp(got[(1,)]) - 6 / 8) < 1e-12 and abs(math.exp(got[(1, 1)]) - 1 / 8) < 1e-12
    for lab, s in got.items():
        assert abs(s - exact[lab]) < 1e-12


@pytest.mark.parametrize("W", [1, 4, 16])
def test_peaked_frames_give_the_greedy_collapse(W):
    torch.manual_seed(5)
    B, T, C = 6, 40, 30
    path = torch.randint(0, C, (B, T))
    path[:, ::3] = 0                                    # some blanks
    path[0, 5:9] = 7                                    # a repeat run
    logits = torch.randn(B, T, C, dtype=torch.float64)
    logits.scatter_(2, path[..., None], 30.0)          # p(path class) ~ 1 - 1e-11 per frame
    ids, lp, blank = BO.ctc_topk(logits, 8)
    for b in range(B):
        best = BO.ctc_prefix_beam_search(ids[b].tolist(), lp[b].tolist(), blank[b].tolist(), W, 1)[0][0]
        assert best == BO.collapse(path[b].tolist())
        _, seqs, _ = O.greedy_decode(logits[b:b + 1])
        assert list(best) == seqs[0]


def test_topk_ties_go_to_the_smaller_class():
    x = torch.tensor([[[0.5, 1.0, 2.0, 1.0, 2.0, 1.0]]], dtype=torch.float64)
    ids, lp, blank = BO.ctc_topk(x, 7)
    assert ids[0, 0].tolist() == [2, 4, 1, 3, 5, -1, -1]
    assert lp[0, 0, 5] == float("-inf") and abs(float(blank[0, 0]) - (0.5 - float(torch.logsumexp(x[0, 0], 0)))) < 1e-15
