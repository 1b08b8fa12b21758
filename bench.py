#!/usr/bin/env python
"""Benchmark of the D3Feat hot path (BASELINE.json): points/sec through the KPFCNN encoder.

    python bench.py --gpus N --steps K --warmup W            # this repository's CUDA path
    python bench.py --impl reference --gpus N ...            # the reference's CPU path (oracle/_ref + restatement)
    python bench.py --workload single30k|kitti120k|micro1m   # the other BASELINE configs (side lines, same JSON shape)
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed (.npy)

Default workload `batch8x30k`: a step = one pass of the hot path (4 grid subsamplings + 13 radius searches + 10 KPConv +
23 unary convs + BN/LeakyReLU/pools) over one batch of 8 stacked synthetic 3DMatch-shaped fragments of 30 000 points
per GPU (BASELINE configs[1] stacked as in configs[3]). value = level-0 points / second, whole job. For N > 1 every
rank runs its own fragments (weak scaling) and the step ends with the NCCL all-gather of the per-fragment descriptors.

Both arms print the SAME `config` (arm-specific notes live under `detail`). The reference arm runs exactly the
workload it prints -- full-size fragments; when K + W full steps would not finish within a few minutes it runs fewer
timed steps and says so (`steps_run`), it never shrinks the fragments.
"""
import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = ("batch8x30k", "single30k", "kitti120k", "micro1m")
REF_ARM_BUDGET_S = 200.0          # the reference arm cuts STEPS (never points) to stay inside this
DUMP_BUDGET_BYTES = 64 << 20      # --dump-outputs writes at most this much


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="batch8x30k", choices=WORKLOADS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipeline", action="store_true", help="one batch at a time on one stream")
    ap.add_argument("--no-graph", action="store_true", help="do not replay the step as a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the arrays the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def dump_outputs(d, arrays):
    """Write {name: array} as d/<name>.npy in float32 (float64 for integers that float32 cannot hold exactly). The
    inputs are seeded, so two builds given the same arguments can be compared file by file. An array larger than its
    even share of DUMP_BUDGET_BYTES is cut to a fixed, seeded sample of rows, whose indices go to <name>_rows.npy."""
    os.makedirs(d, exist_ok=True)
    share = DUMP_BUDGET_BYTES // max(len(arrays), 1)
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype.kind in "iu":
            a = a.astype(np.float32 if a.size == 0 or np.abs(a).max() < (1 << 24) else np.float64)
        elif a.dtype != np.float64:
            a = a.astype(np.float32)
        if a.nbytes > share:
            row_bytes = a.nbytes // a.shape[0] + 8
            rows = np.sort(np.random.default_rng(0).choice(a.shape[0], share // row_bytes, replace=False))
            np.save(os.path.join(d, name + "_rows.npy"), rows.astype(np.float64))
            a = a[rows]
        np.save(os.path.join(d, name + ".npy"), np.ascontiguousarray(a))


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ----------------------------------------------------------------------------------------------------
#  algorithmic bytes (SURVEY.md 8d) -- the figures `roofline.achieved` is computed from
# ----------------------------------------------------------------------------------------------------

def kpconv_algorithmic_bytes(Nq, H, K, Cin, Cout):
    """bytes = Nq*H*(4 + 12 + 4*Cin) + 4*Nq*Cout + 4*K*Cin*Cout + 12*Nq."""
    return Nq * H * (4 + 12 + 4 * Cin) + 4 * Nq * Cout + 4 * K * Cin * Cout + 12 * Nq


def unary_algorithmic_bytes(N, Cin, Cout, residual=False):
    return 4 * N * (Cin + Cout + (Cout if residual else 0)) + 4 * Cin * Cout


def neighbors_algorithmic_bytes(Nq, Ns, cols):
    """12*(Nq + Ns) + 4*Nq*cols (the 27-cell candidate reads are cache traffic, not counted)."""
    return 12 * (Nq + Ns) + 4 * Nq * cols


def subsample_algorithmic_bytes(N, M):
    """12*N in + 12*M out + 8*N keys."""
    return 12 * N + 12 * M + 8 * N


# ----------------------------------------------------------------------------------------------------
#  workloads
# ----------------------------------------------------------------------------------------------------

def make_workload(name, rank):
    """(config object, neighbour caps, list of level-0 clouds of this rank, JSON description)."""
    from d3feat_b200 import synth
    if name in ("batch8x30k", "single30k"):
        nfrag = 8 if name == "batch8x30k" else 1
        cfg = synth.Config(architecture=synth.ARCH_ENCODER)
        limits = [40, 40, 40, 40, 40]      # "max 40 neighbors" (north_star); calibrated caps are 35-40 on real fragments
        clouds = [synth.room_fragment(rank * nfrag + i, 30000) for i in range(nfrag)]
        desc = dict(workload="%d stacked 3DMatch-shaped synthetic fragment%s x 30000 pts per GPU, full 5-level KPFCNN "
                             "encoder" % (nfrag, "s" if nfrag > 1 else ""),
                    baseline_config="configs[1] stacked as in configs[3]" if nfrag > 1 else "configs[1]",
                    fragments_per_gpu=nfrag, points_per_fragment=30000, levels=5, K=15, neighbor_cols=limits,
                    first_subsampling_dl=0.03, params_seed=0)
        return cfg, limits, clouds, desc, 0
    if name == "kitti120k":
        cfg = synth.Config(architecture=synth.ARCH_KITTI_DEFORM, first_subsampling_dl=0.04, first_features_dim=32)
        limits = [40, 40, 40, 60, 40]
        clouds = [synth.lidar_scan(1 + rank, 120000, dl=0.04)]
        desc = dict(workload="KITTI-shaped synthetic 64-beam scan, 120000 level-0 pts per GPU, 5-level encoder with "
                             "deformable KPConv in the last three blocks",
                    baseline_config="configs[2]", fragments_per_gpu=1, points_per_fragment=120000, levels=5, K=15,
                    neighbor_cols=limits, first_subsampling_dl=0.04, params_seed=1,
                    note="a 64-beam scan voxelised at the reference's 0.30 m keeps < 25k points; the 120k level-0 "
                         "points configs[2] names are reached with a 4 cm first voxel")
        return cfg, limits, clouds, desc, 1
    raise ValueError(name)


# ----------------------------------------------------------------------------------------------------
#  reference arm / CPU baseline: the reference's own C++ cores (oracle/_ref) for the pyramid and the numpy
#  restatement of the TF graph for the encoder, on the host cores
# ----------------------------------------------------------------------------------------------------

def cpu_one_fragment(cfg, params, pts, limits, use_ref):
    from oracle import native as on
    from oracle import kpconv_np as ok
    nb = on.ref_batch_neighbors if use_ref else on.port_batch_neighbors
    sb = on.ref_batch_subsampling if use_ref else on.port_batch_subsampling
    lens = np.array([pts.shape[0]], np.int32)
    inputs = ok.descriptor_input_pyramid(cfg, pts, lens, limits, nb, sb)
    inputs["features"] = np.ones((pts.shape[0], 1), np.float32)
    F = ok.EncoderOracle(cfg, params, np.float32).encoder(inputs)
    return F[-1]


def cpu_reference_run(cfg, params, clouds, limits, steps, warmup, budget_s):
    """Each step processes ALL `clouds` (the same fragments one GPU step processes), one fragment per host thread, with
    every host core in use: T = min(nproc, fragments) worker threads (the reference's tf.data map runs its pyramids
    concurrently the same way, datasets/common.py:600,744) and nproc // T BLAS threads inside each numpy call.
    Returns (per-step seconds, info)."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import native as on
    use_ref = on.have_ref()
    if not use_ref:
        on.port()
    nproc = os.cpu_count() or 1
    T = max(1, min(nproc, len(clouds)))
    blas = max(1, nproc // T)
    try:
        from threadpoolctl import threadpool_limits
        limiter = threadpool_limits(limits=blas)
    except Exception:                      # threadpoolctl missing: BLAS keeps its default
        limiter, blas = None, None
    times = []
    t_start = time.perf_counter()
    with ThreadPoolExecutor(T) as ex:
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            last = list(ex.map(lambda p: cpu_one_fragment(cfg, params, p, limits, use_ref), clouds))
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
            done_timed = len(times)
            elapsed = time.perf_counter() - t_start
            if done_timed >= 3 and elapsed + 1.5 * dt > budget_s:
                break                      # cut STEPS, never the fragment size
    if limiter is not None:
        limiter.restore_original_limits()
    kind = "reference" if use_ref else "port"
    n_pts = int(sum(c.shape[0] for c in clouds))
    sample = ("%d fragment(s), %d level-0 pts per step, %d worker threads x %s BLAS threads on %d cores, %d timed steps "
              "after %d warm-up (median); pyramid = %s, encoder = numpy fp32 restatement of the TF1 graph "
              "(TensorFlow not installable)") % (
        len(clouds), n_pts, T, str(blas), nproc, len(times), warmup,
        "reference C++ cores (oracle/_ref)" if use_ref else "C restatement (oracle/liboracle.so)")
    return times, dict(kind=kind, cores=nproc, threads=T, sample=sample, points_per_step=n_pts,
                       outputs=dict(features=np.concatenate(last, 0)))


def cpu_micro_run(P, steps, warmup):
    """configs[4] on the host: the reference's grid_subsampling + batch_nanoflann_neighbors (single thread each, as one
    TF op executes)."""
    from oracle import native as on
    use_ref = on.have_ref()
    sub = on.ref_batch_subsampling if use_ref else on.port_batch_subsampling
    nbf = on.ref_batch_neighbors if use_ref else on.port_batch_neighbors
    n = np.array([P.shape[0]], np.int32)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        sp, sb = sub(P, n, 0.03)
        nb = nbf(sp, sp, sb, sb, 0.075)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    return times, dict(kind="reference" if use_ref else "port", cores=os.cpu_count() or 1, threads=1,
                       sample="1 000 000 raw points per step: grid subsampling dl 0.03 then radius neighbours r 0.075 of "
                              "the subsampled cloud, single host thread (one TF op), %d timed steps after %d warm-up "
                              "(median)" % (len(times), warmup), points_per_step=int(P.shape[0]),
                       outputs=dict(subsampled_points=sp, subsampled_lengths=sb, neighbors=nb))


# ----------------------------------------------------------------------------------------------------
#  clocks
# ----------------------------------------------------------------------------------------------------

class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + self.Q,
                                       "--format=csv,noheader,nounits", "-lms", os.environ.get("D3F_BENCH_LMS", "20")],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            pass
        else:      # a benchmark that raises before stop() must not leave the sampler polling
            atexit.register(self.p.kill)

    def stop(self):
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[])
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = [float(r[1]) for r in rows if r[1].strip().replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if r[2].strip().replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = set()
        for r in rows:
            for i, n in enumerate(names):
                if r[5 + i].strip().lower().startswith("active"):
                    reasons.add(n)
        out.update(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None,
                   reasons=sorted(reasons), samples=len(rows))
        return out


def stats_ms(ts):
    a = np.asarray(ts, np.float64)
    return dict(median=float(np.median(a)), mean=float(a.mean()), max=float(a.max()), min=float(a.min()))


def measured_traffic(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel from the committed `ncu --set
    full` capture (profiles/r2_traffic.json, written by scripts/ncu_summarize.py from the .ncu-rep); null when no
    capture of the current kernel is committed -- never a hand-copied constant."""
    p = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get(key)
    if not d:
        return None, None
    return int(d["dram_bytes_per_launch"]), d.get("source")


# ----------------------------------------------------------------------------------------------------
def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "micro1m":
        return main_micro(args, world, rank, local_rank)
    from d3feat_b200 import synth
    cfg, LIMITS, clouds, wdesc, pseed = make_workload(args.workload, rank)
    params = synth.make_params(cfg, seed=pseed)
    config = dict(wdesc, parallelism="fragments sharded, dp%d" % args.gpus)
    base = dict(metric="points/sec through KPFCNN encoder", unit="points/s", n_gpus=args.gpus, steps=args.steps,
                warmup=args.warmup, higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", config=config)

    if args.impl == "reference":
        if rank != 0:
            return
        # the same fragments ALL ranks of the CUDA arm process in one step (N x fragments_per_gpu), on this host's cores
        all_clouds = []
        for r in range(max(args.gpus, 1)):
            all_clouds += make_workload(args.workload, r)[2]
        times, info = cpu_reference_run(cfg, params, all_clouds, LIMITS, args.steps, min(args.warmup, 2),
                                        REF_ARM_BUDGET_S)
        st = stats_ms([t * 1000.0 for t in times])
        value = info["points_per_step"] / (st["median"] / 1000.0)
        line = dict(base, impl="reference", value=value, ms_per_step=st["median"], ms_per_step_mean=st["mean"],
                    ms_per_step_max=st["max"], steps_run=len(times),
                    cpu_baseline=dict(value=value, unit="points/s", cores=info["cores"], kind=info["kind"],
                                      sample=info["sample"]),
                    e2e=dict(value=value, unit="points/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                    gpu_launches=0)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, info["outputs"])
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    from d3feat_b200 import _lib
    from d3feat_b200 import convolution_ops as co
    from d3feat_b200.encoder import KPFCNN
    from d3feat_b200.distributed import all_gather_descriptors_padded

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()

    # ---- workload: this rank's fragments (seeded by global fragment id) --------------------------------
    P = np.concatenate(clouds, 0)
    L = np.array([c.shape[0] for c in clouds], np.int32)
    n_points = int(P.shape[0])
    P_pin = torch.from_numpy(P).pin_memory()
    L_pin = torch.from_numpy(L).pin_memory()
    P_dev, L_dev = P_pin.to(dev), L_pin.to(dev)
    enc = KPFCNN(cfg, params, LIMITS, device=dev)
    bbox = np.concatenate([P.min(0), P.max(0)]).astype(np.float32)

    gather_cap = max(64, n_points // 128)    # rows reserved per rank for the coarsest-level descriptors (~1.5x actual)

    # (result, device level counts or None) of the most recent step: what --dump-outputs writes
    last_out = [None]

    def step_resident():
        out = enc(P_dev, L_dev, bbox=bbox, decoder=False)
        desc = out["F"][-1]
        last_out[0] = (desc, None)
        if world > 1:      # the one exchange step: NCCL all-gather of the per-fragment descriptors (sync-free)
            desc, _ = all_gather_descriptors_padded(desc, out["inputs"]["lengths"][-1], gather_cap)
        return desc

    def host_outputs():
        """This rank's coarsest-level encoder features of the most recent step, rows beyond the level count dropped
        (the graph pipeline returns a capacity-sized buffer)."""
        res, counts = last_out[0]
        if counts is not None:
            res = res[:int(counts[len(LIMITS) - 1].item())]
        return dict(features=res.cpu().numpy())

    def step_e2e():
        # the call a user makes: host buffers in, descriptors out (host) -- H2D and D2H inside the timed region
        p = P_pin.to(dev, non_blocking=True)
        l = L_pin.to(dev, non_blocking=True)
        out = enc(p, l, decoder=False)          # bbox computed on the device (one small D2H read)
        desc = out["F"][-1]
        if world > 1:      # the gathered matrix stays in HBM (that is where a matcher consumes it) ...
            gathered[0], _ = all_gather_descriptors_padded(desc, out["inputs"]["lengths"][-1], gather_cap)
        return desc.cpu()  # ... the host gets this rank's own descriptors

    gathered = [None]      # the most recent all-gathered descriptor matrix (kept alive until the next step replaces it)
    flush_buf = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)     # > 126 MB L2

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(ms):
        if world > 1:
            tms = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            return float(tms.item())
        return ms

    def timed(fn, steps, warmup):
        """One batch at a time. Per-step device time from CUDA events on the launching (current) stream."""
        for _ in range(warmup):
            fn()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        n0 = _lib.launch_count()
        for a, b in evs:
            flush_buf.fill_(1)            # L2 flush between timed iterations (outside the event bracket)
            a.record()
            fn()
            b.record()
        barrier()
        launches = (_lib.launch_count() - n0) // max(steps, 1)
        st = stats_ms([a.elapsed_time(b) for a, b in evs])
        return st, launches

    def make_pipeline(post):
        """(pipeline, step(points, lengths, bbox, pre) -> result tensor). Default: GraphPipeline (static pyramid + device
        row counts, the step = two CUDA graph replays); --no-graph: BatchPipeline (eager launches, 4 size read-backs)."""
        from d3feat_b200.encoder import BatchPipeline, GraphPipeline
        if args.no_graph:
            pipe = BatchPipeline(enc, decoder=False, post=post)
            return pipe, (lambda p, l, bb, pre: pipe.step(p, l, bb, pre=pre)), (lambda p, l, bb: pipe.prime(p, l, bb))
        pipe = GraphPipeline.for_batch(enc, P_dev, L_dev, decoder=False, post=post,
                                       encoder_streams=int(os.environ.get("D3F_ENC_STREAMS", "2")))

        def step(p, l, bb, pre):
            res, counts = pipe.step(p, l, pre=pre)
            last_counts[0] = counts
            return res
        return pipe, step, (lambda p, l, bb: pipe.prime(p, l))

    last_counts = [None]

    def timed_latency(steps, warmup):
        """One batch at a time through the same pipeline object (prime -> step -> result on the caller's stream):
        the un-overlapped latency of a batch."""
        pipe, step, prime = make_pipeline(None)

        def one():
            prime(P_dev, L_dev, bbox)
            return step(None, None, None, None)
        for _ in range(warmup):
            one()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            flush_buf.fill_(1)
            a.record()
            one()
            b.record()
        pipe.drain()
        barrier()
        if hasattr(pipe, "check"):
            pipe.check()
        return stats_ms([a.elapsed_time(b) for a, b in evs])

    def timed_pipelined(steps, warmup, e2e):
        """K steps of the two-stream pipeline: encoder(i) on one stream while the pyramid of batch i+1 is built on
        the other (encoder.BatchPipeline). The timed region holds exactly K encoders and K pyramids (the first
        encoder consumes the primed pyramid, the last step builds one more), the L2 flush of every step, and for
        e2e the H2D copy of each batch's points and the D2H copy of each batch's descriptors. Per-step device time =
        the interval between consecutive end-of-step events on the encoder stream (the stream every step's last
        kernel / D2H copy is enqueued on); their sum is the device time of the whole region."""
        def post(inputs, desc):
            if world > 1:      # the one exchange step: NCCL all-gather of the per-fragment descriptors (sync-free);
                # the gathered matrix stays in HBM, the step returns this rank's own descriptors
                rows = inputs.get("rows")
                gathered[0], _ = all_gather_descriptors_padded(desc, inputs["lengths"][-1], max(gather_cap, desc.shape[0]),
                                                               rows_dev=rows[-1] if rows else None)
            return desc

        pipe, step, prime = make_pipeline(post)
        src_p, src_l, src_bbox = (P_pin, L_pin, None) if e2e else (P_dev, L_dev, bbox)
        host_out = None
        host_counts = torch.zeros((8,), dtype=torch.int32).pin_memory()

        def one(k_flush, mark=None):
            nonlocal host_out
            res = step(src_p, src_l, src_bbox, (lambda: flush_buf.fill_(1)) if k_flush else None)
            with torch.cuda.stream(pipe.s_enc):
                if e2e:       # the rank's descriptors (and, graph mode, the device-side level counts) go to the host
                    if host_out is None:
                        host_out = torch.empty(res.shape, dtype=res.dtype, pin_memory=True)
                        e2e_bytes[0] = int(host_out.numel() * 4) + (32 if last_counts[0] is not None else 0)
                    host_out.copy_(res, non_blocking=True)
                    if last_counts[0] is not None:
                        host_counts.copy_(last_counts[0], non_blocking=True)
                if mark is not None:
                    mark.record(pipe.s_enc)
            last_out[0] = (res, last_counts[0])
            return res

        prime(src_p, src_l, src_bbox)
        for _ in range(warmup):
            one(False)
        # untimed settling: a fresh process can see one-off stalls (allocator growth, the previous process's context
        # still being torn down); keep warming up until five consecutive steps run within 1.5x of the fastest seen
        # (with several ranks every step holds a collective, so the count must be the same everywhere: fixed)
        best, calm = float("inf"), 0
        for it in range(40):
            t_s = time.perf_counter()
            one(False)
            dt = time.perf_counter() - t_s
            best = min(best, dt)
            calm = calm + 1 if dt < 1.5 * best else 0
            if (world == 1 and calm >= 5) or (world > 1 and it >= 9):
                break
        pipe.drain()
        barrier()
        n0 = _lib.launch_count()
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        t0 = time.perf_counter()
        marks[0].record(pipe.s_enc)
        for i in range(steps):
            one(True, marks[i + 1])
        pipe.drain()
        barrier()
        wall = (time.perf_counter() - t0) * 1000.0 / steps      # synchronised on both sides
        # consecutive encoders alternate between w streams and finish in bursts: a step's time is the completion
        # interval averaged over a window of w steps (w = 1: plain consecutive intervals; fewer steps than streams:
        # the whole region)
        w = min(len(getattr(pipe, "s_encs", [None])), steps)
        per_step = [marks[i].elapsed_time(marks[i + w]) / w for i in range(steps - w + 1)]
        launches = (_lib.launch_count() - n0) // max(steps, 1)
        if hasattr(pipe, "check"):
            pipe.check()                                          # no batch overflowed the shape bucket
            launches = int(pipe.kernels_per_step)                 # kernels inside the two replayed graphs of a step
        st = stats_ms(per_step)
        st["wall_mean"] = wall
        return st, launches

    e2e_bytes = [None]
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if args.no_pipeline:
        seq, _ = timed(step_resident, args.steps, max(args.warmup, 3))      # un-pipelined latency of one batch
    else:
        seq = timed_latency(args.steps, max(args.warmup, 3))
    if args.no_pipeline:
        st, launches = timed(step_resident, args.steps, 1)
        clocks = sampler.stop() if sampler else None
        outputs = host_outputs() if args.dump_outputs else None
        st_e2e, _ = timed(step_e2e, args.steps, 1)
    else:
        st, launches = timed_pipelined(args.steps, max(args.warmup, 3), False)
        clocks = sampler.stop() if sampler else None
        outputs = host_outputs() if args.dump_outputs else None
        st_e2e, _ = timed_pipelined(args.steps, max(args.warmup, 3), True)
    # headline = the MEDIAN step (max over ranks); mean and max are reported beside it: a single host stall moves the
    # mean of 20 steps by tens of percent and says nothing about the path
    ms = reduce_max(st["median"])
    ms_e2e = reduce_max(st_e2e["median"])
    total_points = n_points * world
    value = total_points / (ms / 1000.0)
    e2e_value = total_points / (ms_e2e / 1000.0)
    # bytes of the host tensor(s) the e2e step returns (per rank)
    d2h = e2e_bytes[0] if e2e_bytes[0] is not None else int(step_e2e().numel() * 4)

    # ---- roofline: the dominant KPConv timed alone + the whole step against SURVEY 8(d)'s algorithmic bytes --------
    roof = None
    if rank == 0:
        calls = []
        orig_kp, orig_kd, orig_un, orig_up = co.KPConv_ops, co.KPConv_deform_ops, co.unary_convolution, \
            co.unary_pair_convolution

        def hook_kp(q, s, idx, f, Kp, W, *a, **k):
            calls.append(("kpconv", (q, s, idx, f, Kp, W) + a, k))
            return orig_kp(q, s, idx, f, Kp, W, *a, **k)

        def hook_kd(q, s, idx, f, Kp, off, mod, W, *a, **k):
            calls.append(("kpconv_deform", (q, s, idx, f, Kp, off, mod, W) + a, k))
            return orig_kd(q, s, idx, f, Kp, off, mod, W, *a, **k)

        def hook_un(x, w, **k):
            calls.append(("unary", (x, w), k))
            return orig_un(x, w, **k)

        def hook_up(x1, w1, a1, x2, w2, a2, alpha, **k):
            calls.append(("unary_pair", (x1, w1, x2, w2), {}))
            return orig_up(x1, w1, a1, x2, w2, a2, alpha, **k)

        co.KPConv_ops, co.KPConv_deform_ops, co.unary_convolution, co.unary_pair_convolution = \
            hook_kp, hook_kd, hook_un, hook_up
        try:
            out = enc(P_dev, L_dev, bbox=bbox, decoder=False)
        finally:
            co.KPConv_ops, co.KPConv_deform_ops, co.unary_convolution, co.unary_pair_convolution = \
                orig_kp, orig_kd, orig_un, orig_up
        inp = out["inputs"]
        enc_bytes, best = 0, None
        for kind, a, k in calls:
            if kind in ("kpconv", "kpconv_deform"):
                idx, f, W = a[2], a[3], (a[5] if kind == "kpconv" else a[7])
                b = kpconv_algorithmic_bytes(int(idx.shape[0]), int(idx.shape[1]), int(W.shape[0]), int(W.shape[1]),
                                             int(W.shape[2]))
                if kind == "kpconv" and int(W.shape[1]) > 1 and (best is None or b > best[0]):
                    best = (b, a, k)
            elif kind == "unary":
                b = unary_algorithmic_bytes(int(a[0].shape[0]), int(a[1].shape[0]), int(a[1].shape[1]),
                                            k.get("residual") is not None)
            else:
                b = (unary_algorithmic_bytes(int(a[0].shape[0]), int(a[1].shape[0]), int(a[1].shape[1])) +
                     4 * int(a[2].shape[0]) * int(a[2].shape[1]) + 4 * int(a[3].shape[0]) * int(a[3].shape[1]))
            enc_bytes += b
        sizes = [int(p.shape[0]) for p in inp["points"]]
        pyr_bytes = 0
        for l in range(len(sizes)):
            pyr_bytes += neighbors_algorithmic_bytes(sizes[l], sizes[l], LIMITS[l])
            if l + 1 < len(sizes):
                pyr_bytes += subsample_algorithmic_bytes(sizes[l], sizes[l + 1])
                pyr_bytes += neighbors_algorithmic_bytes(sizes[l + 1], sizes[l], LIMITS[l])
                pyr_bytes += neighbors_algorithmic_bytes(sizes[l], sizes[l + 1], LIMITS[l])
        abytes, a, k = best
        for _ in range(3):
            orig_kp(*a, **k)
        reps = 10
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for ea, eb in evs:
            flush_buf.fill_(1)
            ea.record()
            orig_kp(*a, **k)
            eb.record()
        torch.cuda.synchronize()
        kst = stats_ms([ea.elapsed_time(eb) for ea, eb in evs])
        kms = kst["median"]
        Nq, H = int(a[2].shape[0]), int(a[2].shape[1])
        Cin, Cout = int(a[5].shape[1]), int(a[5].shape[2])
        peak, peak_src = peaks()
        ach = abytes / (kms * 1e-3) / 1e9
        traffic, traffic_src = measured_traffic("kpconv_%d_%d" % (Cin, Cout))
        whole = (enc_bytes + pyr_bytes) / (st["median"] * 1e-3) / 1e9
        roof = dict(bound="hbm", kernel="KPConv %d->%d on Nq=%d queries x H=%d (d3f_kpconv_forward, the largest KPConv "
                                        "of the step)" % (Cin, Cout, Nq, H),
                    achieved=ach, peak=peak, unit="GB/s", frac=ach / peak, traffic=traffic, traffic_source=traffic_src,
                    peak_source=peak_src, algorithmic_bytes_per_launch=abytes, ms_per_launch=kms,
                    ms_per_launch_max=kst["max"], Nq=Nq, H=H,
                    whole_step=dict(algorithmic_bytes=int(enc_bytes + pyr_bytes), encoder_bytes=int(enc_bytes),
                                    pyramid_bytes=int(pyr_bytes), achieved=whole, frac=whole / peak,
                                    note="SURVEY 8(d) gather model summed over every KPConv / unary / neighbour search "
                                         "/ subsampling of one step, divided by the median step time"),
                    whole_step_frac=whole / peak)

    cpu = None
    if rank == 0 and args.gpus == 1 and not args.no_cpu_baseline:
        # same fragments as the timed CUDA step, 1 warm-up + 3 timed steps, median
        times, info = cpu_reference_run(cfg, params, clouds, LIMITS, 3, 1, 120.0)
        cst = stats_ms([t * 1000.0 for t in times])
        cpu = dict(value=info["points_per_step"] / (cst["median"] / 1000.0), unit="points/s", cores=info["cores"],
                   kind=info["kind"], sample=info["sample"], ms_per_step=cst["median"], ms_per_step_max=cst["max"])

    if rank == 0:
        line = dict(base, value=value, ms_per_step=ms, ms_per_step_mean=st["mean"], ms_per_step_max=st["max"],
                    wall_ms_per_step=st.get("wall_mean", st["mean"]),
                    e2e=dict(value=e2e_value, unit="points/s", h2d_bytes_per_step=int(P.nbytes + L.nbytes) * world,
                             d2h_bytes_per_step=d2h * world, ms_per_step=ms_e2e, ms_per_step_mean=st_e2e["mean"],
                             ms_per_step_max=st_e2e["max"]),
                    gpu_launches=int(launches), clocks=clocks, roofline=roof, cpu_baseline=cpu)
        line["detail"] = dict(
            statistic="value / e2e = points per MEDIAN step (max over ranks); mean and max beside it",
            l2="256 MiB L2 flush at the start of every timed step",
            e2e_output="every rank returns its own fragments' descriptors to its host; with N > 1 the all-gathered "
                       "matrix stays in HBM",
            pipeline=("one batch at a time, eager launches" if args.no_pipeline else
                      ("two streams: pyramid(i+1) || encoder(i), eager launches (encoder.BatchPipeline)" if args.no_graph
                       else "two streams: pyramid(i+1) || encoder(i); each half is ONE CUDA graph replay per step, level "
                            "sizes stay on the device, no host synchronisation (encoder.GraphPipeline)")))
        line["single_batch_latency_ms"] = seq["median"]
        line["single_batch_latency_ms_max"] = seq["max"]
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


# ----------------------------------------------------------------------------------------------------
#  configs[4]: 1 M-point radius-neighbour + grid-subsample microbench
# ----------------------------------------------------------------------------------------------------
def main_micro(args, world, rank, local_rank):
    from d3feat_b200 import synth
    P = synth.surface_cloud(rank, 1000000)
    config = dict(workload="radius-neighbour (r 0.075) + grid-subsample (dl 0.03) microbench, 1 000 000 raw points per "
                           "GPU, hash-grid kernels", baseline_config="configs[4]", points=1000000, dl=0.03,
                  radius=0.075, parallelism="replicas, dp%d" % args.gpus)
    base = dict(metric="points/sec through grid subsampling + radius neighbours", unit="points/s", n_gpus=args.gpus,
                steps=args.steps, warmup=args.warmup, higher_is_better=True, scaling="weak", vs_baseline=None,
                dtype="f32", data="synthetic", config=config)
    if args.impl == "reference":
        if rank != 0:
            return
        times, info = cpu_micro_run(P, min(args.steps, 5), min(args.warmup, 1))
        st = stats_ms([t * 1000.0 for t in times])
        value = info["points_per_step"] / (st["median"] / 1000.0)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, info["outputs"])
        print(json.dumps(dict(base, impl="reference", value=value, ms_per_step=st["median"], steps_run=len(times),
                              cpu_baseline=dict(value=value, unit="points/s", cores=info["cores"], kind=info["kind"],
                                                sample=info["sample"]),
                              e2e=dict(value=value, unit="points/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                              gpu_launches=0)))
        return
    import torch
    from d3feat_b200 import _lib, tf_custom_ops as ops
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    _lib.lib()
    P_pin = torch.from_numpy(P).pin_memory()
    P_dev = P_pin.to(dev)
    n_dev = torch.tensor([P.shape[0]], dtype=torch.int32, device=dev)
    bbox = np.concatenate([P.min(0), P.max(0)]).astype(np.float32)
    flush_buf = torch.empty((256 << 20,), dtype=torch.uint8, device=dev)
    res = {}

    def sub(p):
        return ops.batch_grid_subsampling(p, n_dev, 0.03, bbox=bbox)

    def nbr(sp, sb):
        return ops.batch_ordered_neighbors(sp, sp, sb, sb, 0.075, bbox=bbox)

    def step(p):
        sp, sb = sub(p)
        nb = nbr(sp, sb)
        res["M"], res["cols"] = int(sp.shape[0]), int(nb.shape[1])
        if args.dump_outputs:
            res["out"] = (sp, sb, nb)
        return sp, sb, nb

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        n0 = _lib.launch_count()
        for a, b in evs:
            flush_buf.fill_(1)
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        return stats_ms([a.elapsed_time(b) for a, b in evs]), (_lib.launch_count() - n0) // max(steps, 1)

    sampler = ClockSampler(local_rank) if rank == 0 else None
    st, launches = timed(lambda: step(P_dev), args.steps, max(args.warmup, 3))
    clocks = sampler.stop() if sampler else None
    outputs = None
    if args.dump_outputs and rank == 0:
        outputs = dict(zip(("subsampled_points", "subsampled_lengths", "neighbors"), (t.cpu().numpy() for t in res["out"])))

    def e2e():
        sp, sb, nb = step(P_pin.to(dev, non_blocking=True))
        return sp.cpu(), nb.cpu()
    st_e2e, _ = timed(e2e, max(3, args.steps // 2), 2)
    sp, sb, nb = step(P_dev)
    M, cols = res["M"], res["cols"]
    st_sub, _ = timed(lambda: sub(P_dev), args.steps, 2)
    st_nb, _ = timed(lambda: nbr(sp, sb), args.steps, 2)
    peak, peak_src = peaks()
    nb_bytes = neighbors_algorithmic_bytes(M, M, cols)
    sub_bytes = subsample_algorithmic_bytes(P.shape[0], M)
    ach = nb_bytes / (st_nb["median"] * 1e-3) / 1e9
    traffic, traffic_src = measured_traffic("radius_query_1m")
    roof = dict(bound="hbm", kernel="radius neighbours of %d subsampled points, %d columns (hash-grid build + query)" % (
                    M, cols), achieved=ach, peak=peak, unit="GB/s", frac=ach / peak, traffic=traffic,
                traffic_source=traffic_src, peak_source=peak_src, algorithmic_bytes_per_launch=int(nb_bytes),
                ms_per_launch=st_nb["median"],
                subsample=dict(algorithmic_bytes=int(sub_bytes), ms=st_sub["median"],
                               achieved=sub_bytes / (st_sub["median"] * 1e-3) / 1e9,
                               frac=sub_bytes / (st_sub["median"] * 1e-3) / 1e9 / peak),
                whole_step_frac=(nb_bytes + sub_bytes) / (st["median"] * 1e-3) / 1e9 / peak)
    cpu = None
    if rank == 0 and args.gpus == 1 and not args.no_cpu_baseline:
        times, info = cpu_micro_run(P, 3, 1)
        cst = stats_ms([t * 1000.0 for t in times])
        cpu = dict(value=info["points_per_step"] / (cst["median"] / 1000.0), unit="points/s", cores=info["cores"],
                   kind=info["kind"], sample=info["sample"], ms_per_step=cst["median"])
    if rank == 0:
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        n = P.shape[0] * world
        print(json.dumps(dict(base, value=n / (st["median"] * 1e-3), ms_per_step=st["median"],
                              ms_per_step_mean=st["mean"], ms_per_step_max=st["max"],
                              e2e=dict(value=n / (st_e2e["median"] * 1e-3), unit="points/s",
                                       h2d_bytes_per_step=int(P.nbytes) * world,
                                       d2h_bytes_per_step=int(12 * M + 4 * M * cols) * world,
                                       ms_per_step=st_e2e["median"]),
                              gpu_launches=int(launches), clocks=clocks, roofline=roof, cpu_baseline=cpu,
                              detail=dict(subsampled_points=M, neighbor_cols=cols,
                                          l2="256 MiB L2 flush at the start of every timed step"))))


if __name__ == "__main__":
    main()
