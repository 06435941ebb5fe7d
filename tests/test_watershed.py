"""Semi-Lagrangian watershed: the native flood (tf_watershed_flood_host, a HOST function of the C-ABI library) and the
oracle restatement against golden vectors produced by the reference's own Cython flood, the native flood against stored
labels on random inputs, and -- where that compiled reference is present (oracle/_ref) -- against it directly on them.

The GPU-marked test runs the public ``Flow.watershed`` (device-side offset preparation + native flood).
"""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

from oracle import build_ref_watershed, watershed_np  # noqa: E402
import make_golden_reference_checks as rc  # noqa: E402
import make_golden_watershed as mgw  # noqa: E402


def native_flood(*a):
    from tobac_flow_b200.watershed import flood_host
    return flood_host(*a)


@pytest.mark.parametrize("name", sorted(mgw.CASES))
def test_flood_matches_reference_golden(golden, name):
    c = mgw.case(**mgw.CASES[name])
    want = golden("watershed")[name + "_labels"]
    got_oracle = watershed_np.watershed(c["fwd"], c["bwd"], c["field"], c["markers"], c["mask"], c["conn"])
    assert np.array_equal(got_oracle, want)
    got_native = watershed_np.watershed(c["fwd"], c["bwd"], c["field"], c["markers"], c["mask"], c["conn"], flood=native_flood)
    assert np.array_equal(got_native, want)


def test_flood_matches_compiled_reference_random(golden):
    """The native flood against stored labels that match the reference's on random inputs (reference_checks.npz) and,
    where the reference's Cython flood has been compiled (oracle/_ref), against it directly."""
    stored = golden("reference_checks")
    for name, got in rc.watershed_random(flood=native_flood).items():
        rc.assert_matches(stored, name, got)
    ref = build_ref_watershed.load()
    if ref is None:
        return
    for seed in rc.WATERSHED_SEEDS:
        c = rc.watershed_case(seed)
        a = watershed_np.watershed(c["fwd"], c["bwd"], c["field"], c["markers"], c["mask"], c["conn"],
                                   flood=lambda *x: ref.watershed_raveled(x[0], x[1], x[2], x[3], x[4], x[5], x[6], x[7],
                                                                          np.zeros(3, np.int32), 0.0, x[8], False))
        b = watershed_np.watershed(c["fwd"], c["bwd"], c["field"], c["markers"], c["mask"], c["conn"], flood=native_flood)
        assert np.array_equal(a, b)


def test_flood_argument_checks():
    from tobac_flow_b200 import _lib
    lib = _lib.load()
    assert lib.tf_watershed_flood_host(None, None, 0, None, 0, None, None, None, None, None, None, 0) < 0


def test_structure_order_and_validation():
    from tobac_flow_b200 import watershed as ws
    fp, off = ws.validate_connectivity(3, 1)
    assert fp.sum() == 7 and list(off) == [1, 1, 1]
    nb = ws.offsets_to_raveled_neighbors((5, 7, 9), fp, off)
    assert list(nb) == [-63, -9, -1, 1, 9, 63]       # stable distance sort keeps C order among the six unit offsets
    assert list(nb) == list(watershed_np.offsets_to_raveled_neighbors((5, 7, 9), fp, off))
    with pytest.raises(ValueError):
        ws.validate_connectivity(3, np.ones((2, 3, 3)))


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(mgw.CASES))
def test_flow_watershed_gpu(golden, name):
    import tobac_flow_b200 as tfb
    c = mgw.case(**mgw.CASES[name])
    fl = tfb.Flow(c["fwd"], c["bwd"])
    got = fl.watershed(c["field"], c["markers"], mask=c["mask"], connectivity=c["conn"])
    assert got.dtype == np.int32 and np.array_equal(got, golden("watershed")[name + "_labels"])
    with pytest.raises(ValueError):
        fl.watershed(c["field"], c["markers"][:, :-1], mask=c["mask"])
