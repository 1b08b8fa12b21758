"""Generate the self-contained reference fixtures of the test suite from a checkout of the original D3Feat project
and the reference's compiled C++ cores (oracle/_ref, `make -C oracle ref REF=<checkout>`):

    python scripts/make_golden_reference.py <D3Feat checkout>

tests/golden/released/      small files copied verbatim from the released models: parameters.txt and the
                            tensor-bundle .index of every snapshot, the kernel-point .ply files of the KITTI run, the
                            raw payload bytes of that snapshot's kernel-point tensors (snap-61_kernel_points.npz) and
                            the first 2048 vertices of demo_data/cloud_bin_0.ply (vertex count in the header adjusted).
tests/golden/reference_digests.json
                            (shape, sha256) of the reference cores' outputs, canonically ordered, for the inputs the
                            tests regenerate from seeds: too large to store, compared exactly through their digests.
"""
import json
import os
import shutil
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import native as on  # noqa: E402
from oracle import kpconv_np as ok  # noqa: E402
from d3feat_b200 import synth  # noqa: E402
from d3feat_b200 import tf_checkpoint as ck  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")
SNAPSHOTS = (("results_kitti/Log_11011605", 61), ("results/Log_contraloss", 54), ("results/Log_circleloss", 48))
KITTI_KP = "results_kitti/Log_11011605/kernel_points/epoch61"
DEMO_HEAD = 2048


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


# The reference emits subsampled cells in std::unordered_map iteration order and breaks exact-d2 ties by KD-tree visit
# order. Canonical forms: cells ascend in the reference's cell key per cloud (= the C port's order), neighbours ascend
# in (d2, index). Feeding every level with canonically ordered points makes the reference's in-input-order fp32
# barycenter sums identical to the port's, level after level.

def canonical_ref_subsampling(points, lengths, dl):
    rp, rb = on.ref_batch_subsampling(points, lengths, dl)
    pp, pb = on.port_batch_subsampling(points, lengths, dl)
    assert np.array_equal(rb, pb)
    o = 0
    for n in rb:                                   # same point SET per cloud, bit for bit
        assert np.array_equal(on.sort_rows(bits(rp[o:o + n]))[0], on.sort_rows(bits(pp[o:o + n]))[0])
        o += n
    return pp, pb


def canonical_ref_neighbors(q, s, qb, sb, r):
    return on.canonicalize_neighbors(on.ref_batch_neighbors(q, s, qb, sb, r), q, s, s.shape[0])[0]


def released_files(ref):
    out = os.path.join(GOLDEN, "released")
    for log, snap in SNAPSHOTS:
        os.makedirs(os.path.join(out, log, "snapshots"), exist_ok=True)
        shutil.copyfile(os.path.join(ref, log, "parameters.txt"), os.path.join(out, log, "parameters.txt"))
        shutil.copyfile(os.path.join(ref, log, "snapshots", "snap-%d.index" % snap),
                        os.path.join(out, log, "snapshots", "snap-%d.index" % snap))
    os.makedirs(os.path.join(out, KITTI_KP), exist_ok=True)
    for f in sorted(os.listdir(os.path.join(ref, KITTI_KP))):
        if f.endswith(".ply"):
            shutil.copyfile(os.path.join(ref, KITTI_KP, f), os.path.join(out, KITTI_KP, f))
    prefix = os.path.join(ref, SNAPSHOTS[0][0], "snapshots", "snap-%d" % SNAPSHOTS[0][1])
    _, entries = ck.read_index(prefix)
    data = np.memmap(prefix + ".data-00000-of-00001", dtype=np.uint8, mode="r")
    payload = {n.replace("/", "|"): np.array(data[e["offset"]:e["offset"] + e["size"]])
               for n, e in entries.items() if n.endswith("kernel_points")}
    np.savez_compressed(os.path.join(out, "snap-61_kernel_points.npz"), **payload)
    raw = open(os.path.join(ref, "demo_data", "cloud_bin_0.ply"), "rb").read()
    end = raw.index(b"end_header\n") + len(b"end_header\n")
    head = raw[:end].replace(b"element vertex 258342\n", b"element vertex %d\n" % DEMO_HEAD)
    assert head != raw[:end]
    os.makedirs(os.path.join(out, "demo_data"), exist_ok=True)
    with open(os.path.join(out, "demo_data", "cloud_bin_0_head.ply"), "wb") as fh:
        fh.write(head + raw[end:end + 12 * DEMO_HEAD])


def pyramid(cfg, P, L, limits):
    ref = ok.descriptor_input_pyramid(cfg, P, L, limits, canonical_ref_neighbors, canonical_ref_subsampling)
    return on.pyramid_digests(ref)


def digests():
    d = {}
    # tests/test_oracle_golden.py::test_port_vs_compiled_reference_random
    rng = np.random.default_rng(0)
    trials = []
    for trial in range(3):
        n1, n2 = rng.integers(200, 1500, 2)
        P = rng.uniform(-1, 1, (n1 + n2, 3)).astype(np.float32)
        L = np.array([n1, n2], np.int32)
        r = float(rng.uniform(0.1, 0.3))
        nb = on.canonicalize_neighbors(on.ref_batch_neighbors(P, P, L, L, r), P, P, P.shape[0])[0]
        rp, rb = on.ref_batch_subsampling(P, L, r)
        o, clouds = 0, []
        for n in rb:
            clouds.append(on.digest(on.sort_rows(bits(rp[o:o + n]))[0]))
            o += n
        trials.append(dict(neighbors=on.digest(nb), sub_lengths=rb.tolist(), sub_points=clouds))
    d["random_trials"] = trials
    # tests/test_gpu_real_configs.py::test_micro_1m_bit_exact_vs_reference_cores
    P = synth.surface_cloud(0, 1000000)
    n = np.array([P.shape[0]], np.int32)
    rp, rb = on.ref_batch_subsampling(P, n, 0.03)
    M = int(rb[0])
    pp, _ = canonical_ref_subsampling(P, n, 0.03)
    m = np.array([M], np.int32)
    nb = canonical_ref_neighbors(pp, pp, m, m, 0.075)
    d["micro_1m"] = dict(M=M, sub_points=on.digest(on.sort_rows(bits(rp))[0]), neighbors=on.digest(nb))
    # tests/test_gpu_real_configs.py: bench.py's workload, the KITTI parameters, the 120k-point scan
    cfg = synth.Config(architecture=synth.ARCH_ENCODER)
    clouds = [synth.room_fragment(f, 30000) for f in range(8)]
    P = np.concatenate(clouds, 0)
    L = np.array([c.shape[0] for c in clouds], np.int32)
    d["bench_workload_pyramid"] = pyramid(cfg, P, L, [40, 40, 40, 40, 40])
    cfg = synth.Config(architecture=synth.ARCH_KITTI_DEFORM, first_subsampling_dl=0.30, first_features_dim=32)
    cloud = synth.lidar_scan(2, 16000, dl=0.30)
    d["kitti_dl030_pyramid"] = pyramid(cfg, cloud, np.array([cloud.shape[0]], np.int32), [40, 40, 40, 60, 40])
    cfg = synth.Config(architecture=synth.ARCH_KITTI_DEFORM, first_subsampling_dl=0.04, first_features_dim=32)
    cloud = synth.lidar_scan(1, 120000, dl=0.04)
    d["kitti_120k_pyramid"] = pyramid(cfg, cloud, np.array([cloud.shape[0]], np.int32), [40, 40, 40, 60, 40])
    with open(os.path.join(GOLDEN, "reference_digests.json"), "w") as fh:
        json.dump(d, fh, indent=1)
        fh.write("\n")


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    assert on.have_ref(), "oracle/_ref missing: make -C oracle ref REF=<D3Feat checkout>"
    released_files(os.path.abspath(sys.argv[1]))
    digests()


if __name__ == "__main__":
    main()
