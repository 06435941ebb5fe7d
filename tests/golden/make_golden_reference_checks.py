"""Golden vectors for the cross-checks of the oracle against the unmodified reference that the other golden files do
not cover: get_growth_rate, get_anvil_markers, detect_growth_markers_multichannel, nan_gaussian_filter, the float64 /
integer pair quantisation and the watershed flood on random inputs.

    python tests/golden/make_golden_reference_checks.py

Those checks call the reference itself (refshim.py, oracle/build_ref_watershed.py) only where it is installed; they
compare with ``reference_checks.npz`` everywhere.  The vectors are the oracle's results on exactly the inputs of the
checks, recorded from an oracle that the live comparison had found bit-identical to the reference on these inputs.

Float results are kept as a SHA-256 digest of the whole array (NaN and -0.0 canonicalised, so equal digests mean
``np.array_equal(..., equal_nan=True)``) plus a fixed, seeded sample of elements that makes a failure readable;
integer results are stored whole.
"""
import hashlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)

import make_golden as mg  # noqa: E402
import make_golden_watershed as mgw  # noqa: E402
from oracle import detection_ops as det  # noqa: E402
from oracle import flow_ops as ops  # noqa: E402
from oracle import watershed_np  # noqa: E402

PATH = os.path.join(HERE, "reference_checks.npz")
BACKEND = "cv2" if ops.have_cv2() else "numpy"
SAMPLE = 4096
ANVIL_KW = (dict(), dict(threshold=-12, overlap=0.2, absolute_overlap=1, min_length=1))
MULTICHANNEL_KW = (dict(), dict(overlap=0.2, min_length=2, lower_threshold=0.2, upper_threshold=0.4))
GAUSS_SIGMAS = ((0, 2, 2), (0, 1.5, 1.5))
WATERSHED_SEEDS = range(6)


def multi_inputs():
    """The growth_multi case: the wvd field and the de-quantised flow stored in growth_multi.npz."""
    g = np.load(os.path.join(HERE, "growth_multi.npz"))
    return mg.growth_multi_case(), g["fwd_q256"].astype(np.float32) / 256, g["bwd_q256"].astype(np.float32) / 256


def bt_companion(wvd):
    """A window brightness temperature that cools where the water-vapour difference grows (monotone map + offset)."""
    return (250.0 - 2.2 * (wvd + 25.0)).astype(np.float32)


def nan_gaussian_input(wvd):
    x = wvd[:3].copy()
    x[0, 10:14, 20:30] = np.nan
    x[1, :, 50] = np.nan
    x[2] = np.nan
    return x


def growth_rate_and_anvil(wvd, fwd, bwd):
    dt = np.full(wvd.shape[0], 5.0)
    out = {f"growth_rate_{m}": det.get_growth_rate(wvd, dt, fwd, bwd, method=m, backend=BACKEND)
           for m in ("linear", "cubic")}
    for i, kw in enumerate(ANVIL_KW):
        out[f"anvil_{i}"] = det.get_anvil_markers(wvd, fwd, bwd, backend=BACKEND, **kw)
    return out


def multichannel_and_nan_gaussian(wvd, fwd, bwd):
    dt = np.full(wvd.shape[0], 5.0)
    out = {}
    for i, kw in enumerate(MULTICHANNEL_KW):
        res = det.detect_growth_markers_multichannel(wvd, bt_companion(wvd), dt, dt, fwd, bwd, backend=BACKEND, **kw)
        for j, a in enumerate(res):
            out[f"multichannel_{i}_{j}"] = a
    x = nan_gaussian_input(wvd)
    for i, sigma in enumerate(GAUSS_SIGMAS):
        out[f"nan_gaussian_{i}"] = det.nan_gaussian_filter(x, sigma)
        out[f"nan_gaussian_{i}_keep"] = det.nan_gaussian_filter(x, sigma, propagate_nan=False)
    return out


def quantisation_stacks():
    """Float64 and int32 pairs: numpy keeps float64 and promotes integers, so the reference normalises in float64."""
    from tobac_flow_b200 import synthetic
    bt = synthetic.bt_sequence(3, 120, 160, seed=3, nans=True).astype(np.float64) * 1.0000001
    bt[1, 5:8] = np.nan
    bi = np.nan_to_num(bt * 10).astype(np.int32)
    return bt[0:2], bt[1:3], bi[0:2]


def pair_quantisation():
    return {f"u8_{i}": np.stack(ops.pair_to_u8(s[0], s[1])) for i, s in enumerate(quantisation_stacks())}


def watershed_case(seed):
    return mgw.case(100 + seed, T=4, H=24 + seed, W=31, conn=1 + seed % 2, ties=bool(seed % 2))


def watershed_random(flood=watershed_np.watershed_raveled):
    out = {}
    for seed in WATERSHED_SEEDS:
        c = watershed_case(seed)
        out[f"watershed_{seed}"] = watershed_np.watershed(c["fwd"], c["bwd"], c["field"], c["markers"], c["mask"],
                                                          c["conn"], flood=flood)
    return out


def _canonical(a):
    a = np.ascontiguousarray(a)
    return np.where(np.isnan(a), np.nan, a + 0).astype(a.dtype)


def digest(a):
    a = _canonical(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample(a):
    a = np.asarray(a).reshape(-1)
    idx = np.sort(np.random.default_rng(0).choice(a.size, min(a.size, SAMPLE), replace=False))
    return a[idx]


def entries(name, a):
    a = np.asarray(a)
    if a.dtype.kind == "f":
        return {name + "_sha": np.array(digest(a)), name + "_sample": sample(a)}
    return {name: a}


def assert_matches(g, name, got):
    got = np.asarray(got)
    if name + "_sha" in g.files:
        assert np.array_equal(sample(got), g[name + "_sample"], equal_nan=True), name
        assert digest(got) == str(g[name + "_sha"]), name
    else:
        assert np.array_equal(got, g[name]), name


def main():
    wvd, fwd, bwd = multi_inputs()
    results = {**growth_rate_and_anvil(wvd, fwd, bwd), **multichannel_and_nan_gaussian(wvd, fwd, bwd),
               **pair_quantisation(), **watershed_random()}
    out = {}
    for k, v in results.items():
        out.update(entries(k, v))
    np.savez_compressed(PATH, **out)
    print(os.path.getsize(PATH) // 1024, "KiB", sorted(results))


if __name__ == "__main__":
    main()
