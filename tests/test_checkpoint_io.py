"""Formats either side of the hot path (SURVEY.md §8 f3/f4): TF checkpoint bundles, parameters.txt, PLY, and the
per-fragment output arrays. CPU only.

Known answers from the reference's own artefacts (tests/golden/released/, files of the released models copied verbatim
by scripts/make_golden_reference.py): the 10 kernel-point tensors inside results_kitti/Log_11011605/snapshots/snap-61
must equal the kernel_points/epoch61/*.ply files the trainer wrote from the same variables, bit for bit, and the
variable names of all three released snapshots must be exactly the names the host mirror looks up.
"""
import glob
import os

import numpy as np
import pytest

from d3feat_b200 import io_utils, synth
from d3feat_b200 import tf_checkpoint as ck

REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "released")


def released_snapshot(tmp_path, log, snap, payload=None):
    """Prefix of a tensor bundle made of the released snapshot's real .index and a data shard of the real length in
    which only the tensors of `payload` ({name: raw bytes}) hold their real bytes (the rest is left as a hole)."""
    prefix = str(tmp_path / ("snap-%d" % snap))
    with open(os.path.join(REF, log, "snapshots", "snap-%d.index" % snap), "rb") as fh:
        index = fh.read()
    with open(prefix + ".index", "wb") as fh:
        fh.write(index)
    _, entries = ck.read_index(prefix)
    with open(prefix + ".data-00000-of-00001", "wb") as fh:
        fh.truncate(max(e["offset"] + e["size"] for e in entries.values()))
        for name, raw in (payload or {}).items():
            fh.seek(entries[name]["offset"])
            fh.write(raw.tobytes())
    return prefix


def model_variables(prefix):
    """{name: (shape, dtype)} of the variables load_params returns, from the bundle's index alone."""
    _, entries = ck.read_index(prefix)
    return {n[len(ck.MODEL_SCOPE):]: (tuple(e["shape"]), np.dtype(ck._DTYPES[e["dtype"]])) for n, e in entries.items()
            if n.startswith(ck.MODEL_SCOPE) and not n.endswith(ck._OPTIMIZER_SLOTS)}


def test_crc32c_known_answers():
    assert ck.crc32c(b"123456789") == 0xE3069283          # the standard CRC-32C check value
    assert ck.crc32c(b"") == 0
    assert ck.crc32c(b"6789", ck.crc32c(b"12345")) == 0xE3069283


def test_bundle_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    tensors = {"KernelPointNetwork/layer_0/simple_0/weights": rng.normal(size=(15, 1, 64)).astype(np.float32),
               "KernelPointNetwork/layer_0/simple_0/kernel_points": rng.normal(size=(15, 3)).astype(np.float32),
               "KernelPointNetwork/layer_0/simple_0/weights/Momentum": np.zeros((15, 1, 64), np.float32),
               "global_step": np.array(7, np.int64), "flags": np.array([True, False]),
               "big": rng.normal(size=(300, 300))}
    for i in range(150):                                    # several index blocks
        tensors["KernelPointNetwork/pad/v%03d" % i] = np.full((i % 5 + 1,), i, np.int32)
    prefix = str(tmp_path / "snap-1")
    ck.write_checkpoint(prefix, tensors, block_entries=16)
    back = ck.read_checkpoint(prefix, verify_crc_below=1 << 30)
    assert set(back) == set(tensors)
    for k, v in tensors.items():
        assert back[k].dtype == v.dtype and back[k].shape == v.shape and np.array_equal(back[k], v), k
    params = ck.load_params(prefix)
    assert "layer_0/simple_0/weights" in params and "layer_0/simple_0/weights/Momentum" not in params
    assert "global_step" not in params
    assert set(ck.read_checkpoint(prefix, names=["global_step"])) == {"global_step"}
    with pytest.raises(ck.CheckpointError):
        ck.read_checkpoint(prefix, names=["nope"])


def test_bundle_corruption_is_detected(tmp_path):
    prefix = str(tmp_path / "snap-2")
    ck.write_checkpoint(prefix, {"a/b": np.arange(10, dtype=np.float32)})
    raw = bytearray(open(prefix + ".data-00000-of-00001", "rb").read())
    raw[5] ^= 0xFF
    open(prefix + ".data-00000-of-00001", "wb").write(bytes(raw))
    with pytest.raises(ck.CheckpointError, match="checksum"):
        ck.read_checkpoint(prefix)
    idx = bytearray(open(prefix + ".index", "rb").read())
    idx[3] ^= 0x01
    open(prefix + ".index", "wb").write(bytes(idx))
    with pytest.raises(ck.CheckpointError):
        ck.read_index(prefix)
    open(prefix + ".index", "wb").write(b"not a table")
    with pytest.raises(ck.CheckpointError, match="magic"):
        ck.read_index(prefix)


def test_released_snapshots_known_answers(tmp_path):
    log = os.path.join(REF, "results_kitti", "Log_11011605")
    z = np.load(os.path.join(REF, "snap-61_kernel_points.npz"))
    prefix = released_snapshot(tmp_path, "results_kitti/Log_11011605", 61,
                               {k.replace("|", "/"): z[k] for k in z.files})
    names = [k.replace("|", "/") for k in z.files]
    params = {n[len(ck.MODEL_SCOPE):]: a for n, a in ck.read_checkpoint(prefix, names=names).items()}   # CRC-checked
    plys = sorted(glob.glob(os.path.join(log, "kernel_points", "epoch61", "*.ply")))
    assert len(plys) == 10 and len(params) == 10
    for f in plys:
        base = os.path.basename(f)[:-4]                                      # layer_1_resnetb_0_conv2
        names = [n for n in params if n.endswith("kernel_points") and n.replace("/", "_").startswith(base + "_k")]
        assert len(names) == 1, base
        want = io_utils.read_ply_points(f)
        assert np.array_equal(params[names[0]].view(np.uint32), want.view(np.uint32)), base
    # variable names / shapes == what the host mirror asks for, for every released model
    for log, snap in (("results_kitti/Log_11011605", 61), ("results/Log_contraloss", 54), ("results/Log_circleloss", 48)):
        cfg = io_utils.load_config(os.path.join(REF, log))
        got = model_variables(released_snapshot(tmp_path, log, snap))
        want = synth.make_params(cfg, 0)
        assert set(got) == set(want), log
        assert all(got[k] == (tuple(np.shape(want[k])), np.float32) for k in got), log
        assert cfg.num_layers == 5 and cfg.first_features_dim == 64 and cfg.num_kernel_points == 15


def test_config_and_ply_readers_on_reference_files():
    cfg = io_utils.load_config(os.path.join(REF, "results", "Log_contraloss"))
    assert cfg.architecture[0] == "simple" and cfg.architecture[-1] == "last_unary" and len(cfg.architecture) == 19
    assert abs(cfg.first_subsampling_dl - 0.03) < 1e-9 and cfg.KP_influence == "linear" and cfg.modulated is False
    # demo_data/cloud_bin_0.ply (CloudCompare header, 258342 vertices) cut to its first 2048 vertices
    pts = io_utils.read_ply_points(os.path.join(REF, "demo_data", "cloud_bin_0_head.ply"))
    assert pts.shape == (2048, 3) and pts.dtype == np.float32 and np.isfinite(pts).all()


def test_ply_ascii_and_big_endian(tmp_path):
    pts = np.random.default_rng(1).normal(size=(20, 3)).astype(np.float32)
    a = tmp_path / "a.ply"
    a.write_text("ply\nformat ascii 1.0\nelement vertex 20\nproperty float x\nproperty float y\nproperty float z\n"
                 "end_header\n" + "\n".join("%.9g %.9g %.9g" % tuple(p) for p in pts) + "\n")
    assert np.array_equal(io_utils.read_ply_points(str(a)), pts)
    b = tmp_path / "b.ply"
    head = (b"ply\nformat binary_big_endian 1.0\nelement vertex 20\nproperty uchar red\nproperty double x\n"
            b"property float y\nproperty float z\nelement face 0\nproperty list uchar int vertex_indices\nend_header\n")
    rec = np.zeros(20, dtype=[("red", "u1"), ("x", ">f8"), ("y", ">f4"), ("z", ">f4")])
    rec["x"], rec["y"], rec["z"] = pts[:, 0], pts[:, 1], pts[:, 2]
    b.write_bytes(head + rec.tobytes())
    assert np.array_equal(io_utils.read_ply_points(str(b)), pts)


def test_keypoint_selection_and_writers(tmp_path):
    rng = np.random.default_rng(2)
    N = 500
    pts = rng.normal(size=(N, 3)).astype(np.float32)
    desc = rng.normal(size=(N, 32)).astype(np.float32)
    sc = rng.uniform(size=(N, 1)).astype(np.float32)
    ids = io_utils.select_keypoints(sc)
    assert np.array_equal(ids, np.argsort(sc, axis=0).squeeze())                 # utils/tester.py:210
    assert np.array_equal(io_utils.select_keypoints(sc, 250), np.argsort(sc, axis=0)[-250:].squeeze())   # :283
    paths = io_utils.write_fragment(str(tmp_path), "7-scenes-redkitchen", 3, pts, desc, sc)
    assert [os.path.relpath(p, tmp_path) for p in paths] == [
        "descriptors/7-scenes-redkitchen/cloud_bin_3.D3Feat.npy", "keypoints/7-scenes-redkitchen/cloud_bin_3.npy",
        "scores/7-scenes-redkitchen/cloud_bin_3.npy"]
    d, k, s = (np.load(p) for p in paths)
    assert d.shape == (N, 32) and k.shape == (N, 3) and s.shape == (N, 1) and d.dtype == np.float32
    assert (np.diff(s[:, 0]) >= 0).all()                    # ascending: evaluate.py takes the LAST 250 rows
    assert np.array_equal(k[-1], pts[np.argmax(sc)]) and np.array_equal(d[-1], desc[np.argmax(sc)])

