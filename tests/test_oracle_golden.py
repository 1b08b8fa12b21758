"""CPU: pin the oracle (C restatement) to the golden vectors generated from the reference's own compiled
C++ cores (scripts/make_golden.py, scripts/make_golden_reference.py)."""
import json
import os

import numpy as np
import pytest

from oracle import native as on
from oracle import kpconv_np as ok


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def assert_same_point_set(a, b):
    sa, _ = on.sort_rows(np.asarray(a))
    sb, _ = on.sort_rows(np.asarray(b))
    assert sa.shape == sb.shape
    assert np.array_equal(bits(sa), bits(sb))


def per_cloud_sets_equal(pa, la, pb, lb):
    assert np.array_equal(la, lb)
    o = 0
    for n in la:
        assert_same_point_set(pa[o:o + n], pb[o:o + n])
        o += n


def test_subsampling_port_vs_golden_demo(golden):
    g = golden("subsampling_demo.npz")
    p, b = on.port_batch_subsampling(g["points"], g["lengths"], float(g["dl"]))
    per_cloud_sets_equal(p, b, g["sub_points"], g["sub_lengths"])


def test_subsampling_features_classes_vs_golden(golden):
    g = golden("subsampling_demo.npz")
    p, f, c = on.port_grid_subsample(g["w_points"], g["w_features"], g["w_classes"], sampleDl=float(g["w_dl"]))
    # compare as sets of joined rows (order-free)
    ours = np.concatenate([bits(p), bits(f), c.astype(np.uint32)], 1)
    ref = np.concatenate([bits(g["w_sub_points"]), bits(g["w_sub_features"]), g["w_sub_classes"].astype(np.uint32)], 1)
    a, _ = on.sort_rows(ours)
    b, _ = on.sort_rows(ref)
    assert np.array_equal(a, b)


def test_subsampling_port_is_sorted_by_cell_key(golden):
    g = golden("synthetic.npz")
    p, keys = on.port_grid_subsample(g["frag"][:2500], sampleDl=0.06, return_keys=True)
    assert np.all(np.diff(keys.astype(np.int64)) > 0)


@pytest.mark.parametrize("name,pts,lens,nb,r", [
    ("demo", "points", "lengths", "neighbors", 0.125),
    ("frag", "frag", "frag_lengths", "frag_neighbors", 0.075),
    ("lattice", "lattice", None, "lattice_neighbors", 0.075),
])
def test_neighbors_port_vs_golden(golden, name, pts, lens, nb, r):
    g = golden("neighbors_demo.npz" if name == "demo" else "synthetic.npz")
    P = g[pts]
    L = g[lens] if lens else np.array([P.shape[0]], np.int32)
    ref = g[nb]
    canon, changed = on.canonicalize_neighbors(ref, P, P, P.shape[0])
    ours = on.port_batch_neighbors(P, P, L, L, r)
    assert ours.shape == ref.shape
    assert np.array_equal(ours, canon)
    # inside a tie group the reference holds the same index SET
    assert np.array_equal(np.sort(ref, 1), np.sort(ours, 1))
    if name == "lattice":
        assert changed > 0, "the lattice fixture is meant to exercise exact d2 ties"


def test_neighbors_pool_and_upsample_vs_golden(golden):
    g = golden("neighbors_demo.npz")
    q, qb, s, sb = g["pool_points"], g["pool_lengths"], g["points"], g["lengths"]
    ours = on.port_batch_neighbors(q, s, qb, sb, float(g["radius"]))
    canon, _ = on.canonicalize_neighbors(g["pool_neighbors"], q, s, s.shape[0])
    assert np.array_equal(ours, canon)
    ours = on.port_batch_neighbors(s, q, sb, qb, 2 * float(g["radius"]))
    canon, _ = on.canonicalize_neighbors(g["up_neighbors"], s, q, q.shape[0])
    assert np.array_equal(ours, canon)


def test_ordered_neighbors_vs_golden(golden):
    g = golden("neighbors_demo.npz")
    ours = on.port_ordered_neighbors(g["ord_points"], g["ord_points"], float(g["ord_radius"]))
    canon, _ = on.canonicalize_neighbors(g["ord_neighbors"], g["ord_points"], g["ord_points"], -1)
    assert np.array_equal(ours, canon)
    assert (g["ord_neighbors"] == -1).any()


def test_port_vs_compiled_reference_random():
    """The reference cores' canonical outputs on these seeded clouds, as digests (scripts/make_golden_reference.py)."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")) as fh:
        want = json.load(fh)["random_trials"]
    rng = np.random.default_rng(0)
    for trial in range(3):
        n1, n2 = rng.integers(200, 1500, 2)
        P = rng.uniform(-1, 1, (n1 + n2, 3)).astype(np.float32)
        L = np.array([n1, n2], np.int32)
        r = float(rng.uniform(0.1, 0.3))
        assert on.digest(on.port_batch_neighbors(P, P, L, L, r)) == want[trial]["neighbors"]
        pp, pb = on.port_batch_subsampling(P, L, r)
        assert pb.tolist() == want[trial]["sub_lengths"]
        o = 0
        for n, w in zip(pb, want[trial]["sub_points"]):
            assert on.digest(on.sort_rows(bits(pp[o:o + n]))[0]) == w
            o += n


def test_empty_and_single_point_inputs():
    P = np.zeros((1, 3), np.float32)
    nb = on.port_batch_neighbors(P, P, [1], [1], 0.1)
    assert nb.tolist() == [[0]]
    p, b = on.port_batch_subsampling(P, [1], 0.1)
    assert p.shape == (1, 3) and b.tolist() == [1]
    # strict '<' on the squared distance: a support exactly at distance r is NOT a neighbour
    Q = np.array([[0, 0, 0]], np.float32)
    S = np.array([[0.5, 0, 0], [0.25, 0, 0]], np.float32)
    nb = on.port_batch_neighbors(Q, S, [1], [2], 0.5)
    assert nb.tolist() == [[1]]


def test_kpconv_restatement_fp32_vs_fp64():
    """How much of the 1e-4 budget fp32 summation order consumes on its own."""
    rng = np.random.default_rng(1)
    N, H, K, Cin, Cout = 300, 20, 15, 16, 24
    q = rng.uniform(0, 1, (N, 3)).astype(np.float32)
    idx = rng.integers(0, N + 1, (N, H)).astype(np.int32)
    f = rng.normal(size=(N, Cin)).astype(np.float32)
    Kp = (rng.normal(size=(K, 3)) * 0.1).astype(np.float32)
    W = rng.normal(size=(K, Cin, Cout)).astype(np.float32)
    for infl in ok.INFLUENCES:
        for mode in ok.MODES:
            a = ok.kpconv_ops(q, q, idx, f, Kp, W, 0.15, infl, mode, dtype=np.float32)
            b = ok.kpconv_ops(q, q, idx, f, Kp, W, 0.15, infl, mode, dtype=np.float64)
            assert np.abs(a - b).max() / np.abs(b).max() < 2e-5
    with pytest.raises(ValueError):
        ok.kpconv_ops(q, q, idx, f, Kp, W, 0.15, "cubic", "sum")
    with pytest.raises(ValueError):
        ok.kpconv_ops(q, q, idx, f, Kp, W, 0.15, "linear", "mean")


def test_kpconv_first_layer_counts_real_neighbours():
    """With all-ones input features the normalisation equals the number of real neighbours (:249-253)."""
    rng = np.random.default_rng(2)
    N, H, K = 50, 8, 15
    q = rng.uniform(0, 0.2, (N, 3)).astype(np.float32)
    idx = rng.integers(0, N + 1, (N, H)).astype(np.int32)
    f = np.ones((N, 1), np.float32)
    Kp = np.zeros((K, 3), np.float32)
    W = np.ones((K, 1, 1), np.float32)
    out = ok.kpconv_ops(q, q, idx, f, Kp, W, 10.0, "constant", "sum")
    real = (idx < N).sum(1)
    expect = np.where(real > 0, K * real / np.maximum(real, 1), 0.0)
    assert np.allclose(out[:, 0], expect)
