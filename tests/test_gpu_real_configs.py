"""GPU parity at BASELINE.json's REAL configurations (the shapes bench.py measures), not at reduced sizes:

* configs[1] / configs[3] -- bench.py's exact workload: 8 stacked room_fragment(f, 30000), 40 neighbour columns.
  Pyramid: every matrix bit-exact against the oracle pyramid built with the REFERENCE's compiled C++ cores
  (canonicalised, stored as digests in tests/golden/reference_digests.json) and against the C port's pyramid, which
  shows where a difference starts. Encoder: the float64 restatement of the whole
  encoder for one 30k-point fragment (<= 1e-4 per level), and a sampled-row oracle check of every fused op of the
  full 8 x 30k batch.
* configs[4] -- 1 M points: grid subsampling and radius neighbours bit-exact against the reference C++ cores.
* configs[2] -- KITTI parameters (first_subsampling_dl 0.30, results_kitti/Log_11011605/parameters.txt) against
  the full float64 restatement, and the 120k-point scan against the restatement on >= 2000 sampled query rows of
  every KPConv (rigid, offset head and deformable) and every unary / pool.

Tolerances: bit-exact on indices and barycenters; 1e-4 max-norm relative per tensor on fp32 features (north_star).
Reference files followed: datasets/common.py:1301-1413, tf_custom_ops/tf_neighbors/neighbors/neighbors.cpp:211-332,
tf_custom_ops/tf_subsampling/grid_subsampling/grid_subsampling.cpp:5-149, kernels/convolution_ops.py:161-499,
models/network_blocks.py:1052-1118.
"""
import json
import os

import numpy as np
import pytest
import torch

from oracle import native as on
from oracle import kpconv_np as ok

from _trace import record_ops, check_sampled_rows

pytestmark = pytest.mark.gpu

RTOL = 1e-4
BENCH_LIMITS = [40, 40, 40, 40, 40]          # bench.py LIMITS


def t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def rel_err(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


# ---- the reference's C++ cores, canonicalised -----------------------------------------------------------
# The reference emits subsampled cells in std::unordered_map iteration order and breaks exact-d2 ties by KD-tree
# visit order (SURVEY 7, hard parts 1-2). Canonical forms: cells ascend in the reference's cell key per cloud (= the
# C port's order), neighbours ascend in (d2, index). Feeding every level with canonically ordered points makes the
# reference's in-input-order fp32 barycenter sums identical to ours, level after level. The canonical outputs of the
# reference's compiled cores on the workloads below are stored as digests (scripts/make_golden_reference.py); the C
# port (pinned to the reference by tests/test_oracle_golden.py) is the live oracle that localises a difference.

def reference_digests(name):
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_digests.json")) as fh:
        return json.load(fh)[name]


def assert_pyramid_matches_reference(inputs, name):
    """Every level of `inputs` equals the reference cores' canonical pyramid, through its stored digests."""
    want = reference_digests(name)
    for l, w in enumerate(want):
        assert on.digest(bits(inputs["points"][l])) == w["points"], "points level %d" % l
        assert inputs["lengths"][l].tolist() == w["lengths"], "lengths level %d" % l
        for key in ("neighbors", "pools", "upsamples"):
            a = inputs[key][l]
            (rows, cols), _ = w[key]
            if rows == 0:
                assert a.shape[0] == 0
                continue
            sup = {"neighbors": l, "pools": l, "upsamples": l + 1}[key]
            # ours is always `limit` wide, the reference slice min(max, limit): the extra columns are shadow
            assert a.shape[1] >= cols and (a[:, cols:] == inputs["points"][sup].shape[0]).all(), (key, l)
            assert on.digest(a[:, :cols]) == w[key], (key, l)


def assert_pyramid_equal(inputs, ref, L):
    for l in range(L):
        assert np.array_equal(bits(inputs["points"][l]), bits(ref["points"][l])), "points level %d" % l
        assert np.array_equal(inputs["lengths"][l], ref["lengths"][l]), "lengths level %d" % l
        for key in ("neighbors", "pools", "upsamples"):
            a, b = inputs[key][l], ref[key][l]
            if b.shape[0] == 0:
                assert a.shape[0] == 0
                continue
            sup = {"neighbors": l, "pools": l, "upsamples": l + 1}[key]
            shadow = ref["points"][sup].shape[0]
            if b.shape[1] < a.shape[1]:             # ours is always `limit` wide, the reference slice min(max, limit)
                b = np.concatenate([b, np.full((b.shape[0], a.shape[1] - b.shape[1]), shadow, np.int32)], 1)
            assert a.shape == b.shape, (key, l, a.shape, b.shape)
            assert np.array_equal(a, b), (key, l)


def _inputs_to_numpy(out, n_points, in_dim=1):
    inputs = {k: [x.cpu().numpy() for x in v] for k, v in out["inputs"].items() if k not in ("features", "orders")}
    inputs["features"] = np.ones((n_points, in_dim), np.float32)
    return inputs


# ----------------------------------------------------------------------------------------------------------
#  configs[1] / [3]: bench.py's workload
# ----------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def bench_workload(cuda):
    """Exactly what bench.py builds for rank 0: fragments 0..7 x 30000 points, ARCH_ENCODER, seed-0 parameters."""
    from d3feat_b200 import synth
    from d3feat_b200.encoder import KPFCNN
    cfg = synth.Config(architecture=synth.ARCH_ENCODER)
    params = synth.make_params(cfg, seed=0)
    clouds = [synth.room_fragment(f, 30000) for f in range(8)]
    P = np.concatenate(clouds, 0)
    L = np.array([c.shape[0] for c in clouds], np.int32)
    enc = KPFCNN(cfg, params, BENCH_LIMITS, device=cuda)
    return cfg, params, clouds, P, L, enc


def test_bench_workload_pyramid_bit_exact_vs_reference_cores(cuda, bench_workload):
    cfg, params, clouds, P, L, enc = bench_workload
    assert P.shape[0] == 240000
    out = enc(P, L, decoder=False)
    inputs = _inputs_to_numpy(out, P.shape[0])
    ref = ok.descriptor_input_pyramid(cfg, P, L, BENCH_LIMITS, on.port_batch_neighbors, on.port_batch_subsampling)
    assert [p.shape[0] for p in ref["points"]] == [p.shape[0] for p in inputs["points"]]
    assert_pyramid_equal(inputs, ref, 5)
    assert_pyramid_matches_reference(inputs, "bench_workload_pyramid")


def test_bench_workload_encoder_one_fragment_vs_float64(cuda, bench_workload):
    """One 30k-point fragment (BASELINE configs[1] literally) through the full 5-level encoder, 40 columns, vs the
    float64 restatement on the same pyramid: every level's skip features and the final [N4, 2048] features."""
    cfg, params, clouds, P, L, enc = bench_workload
    c = clouds[3]
    l1 = np.array([c.shape[0]], np.int32)
    out = enc(c, l1, decoder=False)
    inputs = _inputs_to_numpy(out, c.shape[0])
    F_ref = ok.EncoderOracle(cfg, params, np.float64).encoder(inputs)
    assert [f.shape[1] for f in out["F"]] == [128, 256, 512, 1024, 2048]
    for l, (a, b) in enumerate(zip(out["F"], F_ref)):
        assert a.shape == b.shape
        assert rel_err(a.cpu().numpy(), b) < RTOL, "level %d" % l


def test_bench_workload_every_op_sampled_rows_vs_float64(cuda, bench_workload):
    """The full 8 x 30k batch (the shape bench.py times): the float64 restatement of every fused op on 2000 sampled
    output rows, on that op's real inputs."""
    cfg, params, clouds, P, L, enc = bench_workload
    with record_ops() as tr:
        out = enc(P, L, decoder=False)
        torch.cuda.synchronize()
    assert out["F"][-1].shape[1] == 2048
    rep = check_sampled_rows(tr, 2000, np.random.default_rng(0), RTOL, min_kpconv=10)
    assert sum(1 for r in rep if r[0] in ("unary", "unary_pair")) >= 18
    # the single-shot result equals the pipelined one bit for bit (BatchPipeline is what bench.py times)
    from d3feat_b200.encoder import BatchPipeline
    pipe = BatchPipeline(enc, decoder=False)
    pipe.prime(t(P, cuda), t(L, cuda))
    res = pipe.step(None, None)
    pipe.drain()
    assert torch.equal(res, out["F"][-1])


# ----------------------------------------------------------------------------------------------------------
#  configs[4]: 1 M-point microbench, bit-exact vs the reference C++ cores
# ----------------------------------------------------------------------------------------------------------

def test_micro_1m_bit_exact_vs_reference_cores(cuda):
    from d3feat_b200 import synth, tf_custom_ops as ops
    want = reference_digests("micro_1m")
    P = synth.surface_cloud(0, 1000000)
    n = np.array([P.shape[0]], np.int32)
    sp, sb = ops.batch_grid_subsampling(t(P, cuda), t(n, cuda), 0.03)
    M = want["M"]                                              # the reference's std::unordered_map cell count
    assert sp.shape[0] == M and int(sb.item()) == M
    ours = bits(sp.cpu().numpy())
    a, _ = on.sort_rows(ours)
    assert on.digest(a) == want["sub_points"]                  # same barycenters, bit for bit
    # radius neighbours of the subsampled cloud (r = 0.075), every row, vs the reference's KD-tree search on the
    # canonically ordered (ascending reference cell key) barycenters, canonicalised
    m = np.array([M], np.int32)
    nbm = ops.batch_ordered_neighbors(sp, sp, t(m, cuda), t(m, cuda), 0.075).cpu().numpy()
    assert on.digest(nbm) == want["neighbors"]                 # same maximum count, same rows


# ----------------------------------------------------------------------------------------------------------
#  configs[2]: KITTI-shaped scan, deformable blocks
# ----------------------------------------------------------------------------------------------------------

def test_kitti_reference_parameters_dl030_vs_float64(cuda):
    """The reference's KITTI parameters (first_subsampling_dl = 0.30 -> conv radius 0.75 m, deformable blocks in the
    last two levels with the doubled search radius): whole encoder vs the float64 restatement."""
    from d3feat_b200 import synth
    from d3feat_b200.encoder import KPFCNN
    cfg = synth.Config(architecture=synth.ARCH_KITTI_DEFORM, first_subsampling_dl=0.30, first_features_dim=32)
    cloud = synth.lidar_scan(2, 16000, dl=0.30)
    L = np.array([cloud.shape[0]], np.int32)
    params = synth.make_params(cfg, 2)
    limits = [40, 40, 40, 60, 40]
    out = KPFCNN(cfg, params, limits, device=cuda)(cloud, L)
    inputs = _inputs_to_numpy(out, cloud.shape[0])
    ref = ok.descriptor_input_pyramid(cfg, cloud, L, limits, on.port_batch_neighbors, on.port_batch_subsampling)
    assert_pyramid_equal(inputs, ref, len(ref["points"]))
    assert_pyramid_matches_reference(inputs, "kitti_dl030_pyramid")
    F_ref = ok.EncoderOracle(cfg, params, np.float64).encoder(inputs)
    for l, (a, b) in enumerate(zip(out["F"], F_ref)):
        assert rel_err(a.cpu().numpy(), b) < RTOL, "level %d" % l


def test_kitti_120k_every_op_sampled_rows_vs_float64(cuda):
    """120 000 level-0 points (BASELINE configs[2]'s size; reached with a 4 cm first voxel, a 64-beam scan voxelised at
    0.30 m keeps < 25k points): pyramid bit-exact vs the reference cores, and every KPConv -- rigid, offset head,
    deformable -- unary and pool on 2000 sampled rows vs the float64 restatement."""
    from d3feat_b200 import synth
    from d3feat_b200.encoder import KPFCNN
    cfg = synth.Config(architecture=synth.ARCH_KITTI_DEFORM, first_subsampling_dl=0.04, first_features_dim=32)
    cloud = synth.lidar_scan(1, 120000, dl=0.04)
    L = np.array([cloud.shape[0]], np.int32)
    params = synth.make_params(cfg, 1)
    limits = [40, 40, 40, 60, 40]
    enc = KPFCNN(cfg, params, limits, device=cuda)
    with record_ops() as tr:
        out = enc(cloud, L)
        torch.cuda.synchronize()
    inputs = _inputs_to_numpy(out, cloud.shape[0])
    ref = ok.descriptor_input_pyramid(cfg, cloud, L, limits, on.port_batch_neighbors, on.port_batch_subsampling)
    assert_pyramid_equal(inputs, ref, len(ref["points"]))
    assert_pyramid_matches_reference(inputs, "kitti_120k_pyramid")
    rep = check_sampled_rows(tr, 2000, np.random.default_rng(1), RTOL, min_kpconv=10)
    assert any(r[0] == "kpconv_deform" for r in rep)
    # reproducible: no atomics on float data anywhere on the path
    F2 = enc(cloud, L)["F"]
    for a, b in zip(out["F"], F2):
        assert torch.equal(a, b)


# ----------------------------------------------------------------------------------------------------------
#  num_kernel_points other than 15 (utils/config.py allows any K) and the pipeline's stream contract
# ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("K,Cin,Cout,deform", [(7, 32, 32, False), (19, 16, 24, False), (13, 32, 48, True)])
def test_kpconv_any_number_of_kernel_points(cuda, K, Cin, Cout, deform):
    from d3feat_b200 import convolution_ops as co
    from test_gpu_kpconv import make_case
    rng = np.random.default_rng(K)
    q, s, idx, f, Kp, W = make_case(rng, 700, 700, 45, Cin, Cout, K=K, extent=0.1)
    args = [t(x, cuda) for x in (q, s, idx, f, Kp)]
    if deform:
        off = (rng.normal(size=(700, K, 3)) * 0.03).astype(np.float32)
        out = co.KPConv_deform_ops(*args, t(off, cuda), None, t(W, cuda), 0.1, "linear", "sum").cpu().numpy()
        ref = ok.kpconv_deform_ops(q, s, idx, f, Kp, off, None, W, 0.1, "linear", "sum", dtype=np.float64)
    else:
        for mode in ("sum", "closest"):
            out = co.KPConv_ops(*args, t(W, cuda), 0.1, "linear", mode).cpu().numpy()
            ref = ok.kpconv_ops(q, s, idx, f, Kp, W, 0.1, "linear", mode, dtype=np.float64)
            assert rel_err(out, ref) < RTOL, mode
    assert rel_err(out, ref) < RTOL


def test_batch_pipeline_result_is_ordered_on_the_callers_stream(cuda):
    """BatchPipeline.step() returns a tensor produced on its private stream; the caller's current stream must see
    finished data without any explicit synchronisation (ADVICE r1)."""
    from d3feat_b200 import synth
    from d3feat_b200.encoder import KPFCNN, BatchPipeline
    cfg = synth.Config(architecture=synth.ARCH_ENCODER)
    params = synth.make_params(cfg, 5)
    enc = KPFCNN(cfg, params, [35, 33, 34, 36, 30], device=cuda)
    c = synth.room_fragment(90, 20000)
    L = np.array([c.shape[0]], np.int32)
    want = enc(c, L, decoder=False)["F"][-1].clone()
    torch.cuda.synchronize()
    pipe = BatchPipeline(enc, decoder=False)
    pipe.prime(t(c, cuda), t(L, cuda))
    got = []
    for i in range(4):
        res = pipe.step(t(c, cuda), t(L, cuda))
        got.append(res.clone())              # consumer kernel on the caller's (default) stream, no sync in between
    pipe.drain()
    for g in got:
        assert torch.equal(g, want)


# ----------------------------------------------------------------------------------------------------------
#  the sync-free form: static pyramid + device-side row counts + CUDA graph replay (encoder.GraphPipeline)
# ----------------------------------------------------------------------------------------------------------

def test_static_pyramid_equals_exact_pyramid(cuda):
    """d3f_pyramid_build, static form (no device->host read, capacity-sized launches, level sizes in device memory):
    counts, points and every index matrix -- including the shadow index = the actual support count -- equal the exact
    form's on the rows that exist."""
    from d3feat_b200 import synth, pyramid as pyr
    from d3feat_b200.encoder import KPFCNN
    cfg = synth.Config(architecture=synth.ARCH_ENCODER)
    enc = KPFCNN(cfg, synth.make_params(cfg, 0), BENCH_LIMITS, device=cuda)
    clouds = [synth.room_fragment(110, 9000), synth.room_fragment(111, 7000)]
    P = np.concatenate(clouds, 0)
    L = np.array([c.shape[0] for c in clouds], np.int32)
    exact = enc.build_inputs(P, L)
    sizes = [int(p.shape[0]) for p in exact["points"]]
    bb = np.concatenate([P.min(0) - 0.1, P.max(0) + 0.1]).astype(np.float32)
    buf = pyr.PyramidBuffers(cfg, BENCH_LIMITS, pyr.bucket_capacities(sizes, 1.2), 2, cuda, bbox=bb)
    buf.points0[:P.shape[0]].copy_(t(P, cuda))
    buf.lengths0.copy_(t(L, cuda))
    buf.n0.fill_(P.shape[0])
    st = enc.build_inputs_static(buf)
    assert st["counts"][:5].cpu().tolist() == sizes and int(st["status"].item()) == 0
    for l in range(5):
        n = sizes[l]
        assert st["points"][l].shape[0] == buf.caps[l] >= n
        assert torch.equal(st["points"][l][:n], exact["points"][l])
        assert torch.equal(st["lengths"][l], exact["lengths"][l])
        assert torch.equal(st["neighbors"][l][:n], exact["neighbors"][l])
        if l < 4:
            assert torch.equal(st["pools"][l][:sizes[l + 1]], exact["pools"][l])
            assert torch.equal(st["upsamples"][l][:n], exact["upsamples"][l])


def test_graph_pipeline_matches_exact_path_and_flags_overflow(cuda):
    """Five batches of different sizes through ONE captured bucket (3-slot ring, pyramid(i+1) || encoder(i)): every
    result equals the one-batch-at-a-time exact path (the deep GEMMs may pick another deterministic split-K plan for the
    capacity-sized launch, hence 2e-5 instead of bit equality), no host synchronisation is needed to get there, and a
    batch that does not fit the bucket is reported through the status word."""
    from d3feat_b200 import synth
    from d3feat_b200.encoder import KPFCNN, GraphPipeline
    cfg = synth.Config(architecture=synth.ARCH_ENCODER)
    enc = KPFCNN(cfg, synth.make_params(cfg, 5), [35, 33, 34, 36, 30], device=cuda)
    batches = []
    for i, n in enumerate([12000, 11000, 12000, 9500, 11800]):
        clouds = [synth.room_fragment(120 + 2 * i, n), synth.room_fragment(121 + 2 * i, n - 700)]
        batches.append((np.concatenate(clouds, 0), np.array([c.shape[0] for c in clouds], np.int32)))
    want = [enc(P, L, decoder=False)["F"] for P, L in batches]
    pipe = GraphPipeline.for_batch(enc, t(batches[0][0], cuda), t(batches[0][1], cuda), slack=1.2)
    pipe.prime(t(batches[0][0], cuda), t(batches[0][1], cuda))
    got = []
    for i in range(len(batches)):
        nxt = batches[i + 1] if i + 1 < len(batches) else None
        res, counts = pipe.step(t(nxt[0], cuda), t(nxt[1], cuda)) if nxt else pipe.step()
        got.append((res.clone(), counts.clone()))        # consumed on the caller's stream, no explicit sync
    pipe.check()
    assert pipe.kernels_per_step > 100
    for i, ((res, counts), F) in enumerate(zip(got, want)):
        n = int(counts[4].item())
        assert n == F[-1].shape[0], i
        assert rel_err(res[:n].cpu().numpy(), F[-1].cpu().numpy()) < 2e-5, i
    # a batch with far more level-1 cells than the bucket was sized for: flagged, not silently truncated
    rng = np.random.default_rng(0)
    ext = pipe.bbox[3:] - pipe.bbox[:3]
    spread = (pipe.bbox[:3] + 0.05 * ext + rng.uniform(0.0, 0.9, (batches[0][0].shape[0], 3)) * ext).astype(np.float32)
    pipe.prime(t(spread, cuda), t(batches[0][1], cuda))
    pipe.step()
    with pytest.raises(RuntimeError):
        pipe.check()

