"""Pins oracle/sampler_oracle.py: (1) against the committed fixtures generated from the unmodified reference,
(2) against SURVEY.md Appendix B's known-answer hashes, (3) against the reference class's output over random
configurations (tests/golden/reference_traces.json)."""
import hashlib
import json
import os

import numpy as np
import pytest

from sampler_oracle import oracle_indices
from stoke_b200 import synthetic


def _load(golden_dir):
    with open(os.path.join(golden_dir, "sampler_golden.json")) as f:
        return json.load(f)["cases"]


def _oracle_lists(case):
    sorted_idx = synthetic.sampler_sorted_idx(case["n"])
    return [
        oracle_indices(sorted_idx, case["buckets"], case["bs"], case["w"], r, shuffle=case["shuffle"],
                       seed=case["seed"], epoch=case["epoch"], drop_last=case["drop_last"],
                       allow_bucket_overlap=case["overlap"])
        for r in range(case["w"])
    ]


def _sha(lists):
    h = hashlib.sha256()
    for lst in lists:
        h.update(np.asarray(lst, dtype="<i8").tobytes())
    return h.hexdigest()


def test_oracle_matches_golden(golden_dir):
    cases = _load(golden_dir)
    assert len(cases) >= 70
    for case in cases:
        lists = _oracle_lists(case)
        assert len(lists[0]) == case["len_per_replica"], case
        assert lists[0][:16] == case["rank0_head"], case
        assert _sha(lists) == case["sha256"], case
        if "lists" in case:
            assert lists == case["lists"], case


APPENDIX_B = [
    (dict(n=1000, buckets=4, bs=8, w=2, drop_last=False, overlap=False, shuffle=True, seed=0, epoch=0), 512,
     [57, 161, 45, 182, 909, 603, 394, 171], "63289d0768e349c1"),
    (dict(n=1003, buckets=4, bs=8, w=2, drop_last=True, overlap=True, shuffle=True, seed=0, epoch=3), 496,
     [346, 96, 847, 123, 906, 923, 674, 206], "47405d3a120951fd"),
    (dict(n=1000, buckets=4, bs=8, w=2, drop_last=False, overlap=False, shuffle=False, seed=0, epoch=0), 512,
     [539, 554, 510, 393, 330, 301, 185, 586], "b3c6ada95fe792d5"),
    (dict(n=5000, buckets=5, bs=16, w=8, drop_last=False, overlap=False, shuffle=True, seed=7, epoch=1), 640,
     [4849, 4444, 2271, 3488, 4331, 3582, 682, 3613], "abc7f72f4bb5dc02"),
]


@pytest.mark.parametrize("case,length,head,sha", APPENDIX_B)
def test_oracle_appendix_b(case, length, head, sha):
    lists = _oracle_lists(case)
    assert len(lists[0]) == length
    assert lists[0][:8] == head
    assert _sha(lists)[:16] == sha


def test_oracle_guards():
    idx = synthetic.sampler_sorted_idx(300)
    with pytest.raises(ValueError):
        oracle_indices(idx, 4, 16, 8, 0)  # 75 per bucket < slice 128
    with pytest.raises(ValueError):
        oracle_indices(synthetic.sampler_sorted_idx(380), 4, 8, 2, 0)  # 95 per bucket < 100


def test_oracle_matches_live_reference(golden_dir):
    with open(os.path.join(golden_dir, "reference_traces.json")) as f:
        cases = json.load(f)["sampler_random"]
    assert len(cases) >= 25
    errors = {"ValueError": ValueError, "AssertionError": AssertionError}
    for c in cases:
        args = (synthetic.sampler_sorted_idx(c["n"]), c["buckets"], c["bs"], c["w"], c["rank"], c["shuffle"], c["seed"],
                c["epoch"], c["drop_last"], c["overlap"])
        if "raises" in c:
            with pytest.raises(errors[c["raises"]]):
                oracle_indices(*args)
            continue
        got = oracle_indices(*args)
        assert (len(got), _sha([got])) == (c["len"], c["sha256"]), c
