"""The oracle port against the reference on seeded inputs beyond the goldens of oracle/make_golden.py: every function of
the path the reference itself contains must agree bit for bit with its restatement in oracle/port.py.  Each case is
checked against its stored record (tests/golden/live_cases.npz, see oracle/live_cases.py) everywhere, and also against
the reference itself where its source tree is present (HD_YOLO_REFERENCE)."""
import numpy as np
import pytest
import torch

from conftest import load_golden
from oracle import live_cases, port, ref_shim


@pytest.fixture(scope="module")
def ref():
    return live_cases.reference_impl(ref_shim.load()) if ref_shim.available() else None


def _check(case, ref, *args):
    got = case(port, *args)
    gold = load_golden("live_cases")
    assert sorted(got) == sorted(k for k in gold.files if k.startswith(next(iter(got)).split("_")[0] + "_"))
    for k, v in got.items():
        assert np.array_equal(live_cases.digest(v), gold[k]), f"{k} differs from the record ({gold['source']})"
    if ref is not None:
        want = case(ref, *args)
        assert sorted(want) == sorted(got)
        for k, v in got.items():
            assert torch.equal(v, want[k]), k


@pytest.mark.parametrize("seed,n,nc,conf", live_cases.NMS_CASES)
def test_nms_per_image_and_nms_equal_reference(ref, seed, n, nc, conf):
    _check(live_cases.nms_case, ref, seed, n, nc, conf)


def test_box_helpers_equal_reference(ref):
    _check(live_cases.box_case, ref)


def test_scanner_and_tile_merge_equal_reference(ref):
    _check(live_cases.merge_case, ref)


def test_compute_proposals_equals_reference_head(ref):
    _check(live_cases.proposals_case, ref)
