"""The inputs of a golden case of the reference's MRN (svtr_mrn_* / crnn_mrn_* under tests/golden/), rebuilt the way
oracle/make_golden.py made them: the synthetic weights and batch of the file's class counts, batch size and seed."""
from conftest import load_golden
from mrn_b200 import synth


def golden_case(name):
    """-> (g, class_counts, B, seed, state_dict, img, tgt, lens, dom); the architecture is the name's prefix."""
    g = load_golden(name)
    cc = tuple(int(c) for c in g["class_counts"])
    B, seed = int(g["B"]), int(g["seed"])
    sd = synth.synth_state_dict(cc, seed, arch=name.split("_", 1)[0])
    img, tgt, lens, dom = synth.synth_batch(B, cc, seed)
    return g, cc, B, seed, sd, img, tgt, lens, dom
