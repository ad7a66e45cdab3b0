"""CPU tests (no GPU) for unitig mode on two-word keys: the restatements of the reference's link graph
(referenceAssembler.all_contigs :90-111) and get_contig (:47-56) in tests/unitig_ref.py, which the GPU tests of
k = 32..63 use as the checker, pinned to the outputs of the unmodified reference; and the vectorised two-word key
codec of the referenceassembler drop-in."""
import json
import os
import random

import numpy as np
import pytest

import oracle
from unitig_ref import py_get_contig, py_link_graph

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _load(name):
    with open(os.path.join(GOLD, name)) as f:
        return json.load(f)


@pytest.mark.parametrize("fixture", ["g200.json", "synth_small.json"])
def test_py_link_graph_equals_reference_links(fixture):
    for case in _load(fixture)["cases"]:
        exp = {i: ([tuple(x) for x in lk[0]], [tuple(x) for x in lk[1]]) for i, lk in enumerate(case["links"])}
        assert py_link_graph(case["contigs"], case["k"]) == exp, (case["k"], case["limit"])


@pytest.mark.parametrize("fixture", ["g200.json", "synth_small.json"])
def test_py_get_contig_equals_reference_probes(fixture):
    for case in _load(fixture)["cases"]:
        d = {km: c for km, c in case["kmers"]}
        for km, text in case["get_contig"]:
            s, c = py_get_contig(d, km)
            assert s == text and km in c, (case["k"], km)


@pytest.mark.parametrize("k", [1, 5, 31, 32, 33, 48, 63, 64])
def test_two_word_key_codec_round_trip(k):
    from referenceassembler import referenceAssembler as ram
    rng = random.Random(k)
    kms = ["".join(rng.choice("ACGT") for _ in range(k)) for _ in range(200)] + ["A" * k, "T" * k]
    lo, hi = ram._encode(kms, k)
    exp = [oracle.encode_str(x) for x in kms]
    assert [(int(h) << 64) | int(a) for a, h in zip(lo, hi)] == exp
    assert ram._decode(lo, k, hi) == kms
    if k <= 32:
        assert not hi.any() and ram._decode(lo, k) == kms
    with pytest.raises(ValueError):
        ram._encode(["N" * k], k)
    assert ram._encode([], k)[0].size == 0 and ram._decode(np.zeros(0, np.uint64), k) == []
