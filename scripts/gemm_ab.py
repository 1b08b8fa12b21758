"""GPU: A/B of the two operand paths of tc_gemm_kernel at the encoder's GEMM shapes (the list of gemm_probe.py).

    python scripts/gemm_ab.py [--reps 30]

Default path: the split A operand in tensor memory; D3F_TC_A_SMEM=1: both A images in shared memory. The two are
timed alternately, one GEMM per CUDA-event pair, each rep after a 256 MiB L2 flush. Prints the median time of each and
the time per k-chunk: median / (waves x k-chunks per CTA), waves = ceil(CTAs / 148), which is what one k-chunk costs
an SM when every SM runs one CTA of the grid at a time."""
import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from d3feat_b200 import convolution_ops as co

SHAPES = [(4177, 3840, 256), (1204, 7680, 512), (26112, 480, 32), (240000, 32, 128), (240000, 64, 128), (60336, 64, 256),
          (1204, 1024, 2048), (240000, 480, 32), (240000, 64, 32), (240000, 128, 32), (60336, 960, 64), (60336, 128, 64),
          (60336, 480, 32)]


def tiles(M, K, N):
    bn = 128 if N > 64 else (64 if N > 32 else 32)
    if bn == 128 and K <= 256 and M >= 8192:
        bn = 64
    npad = (N + bn - 1) // bn * bn
    return (M + 127) // 128 * (npad // bn), (K + 31) // 32


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    co.USE_TENSOR_CORES = True
    os.environ["D3F_TC_STREAM"] = "0"
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
    paths = (("tmem", "0"), ("smem", "1"))
    print("%-22s %9s %9s %8s | %7s %7s | %6s" % ("M x K -> N", "CTAs", "chunks", "waves", "tmem us", "smem us", "ratio"))
    for M, K, N in SHAPES:
        x = torch.randn(M, K, device=dev)
        w = torch.randn(K, N, device=dev) / K ** 0.5
        times = {p: [] for p, _ in paths}
        for _, flag in paths:                      # warm both: module load, weight packing
            os.environ["D3F_TC_A_SMEM"] = flag
            co.unary_convolution(x, w)
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for p, flag in paths:
                os.environ["D3F_TC_A_SMEM"] = flag
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                co.unary_convolution(x, w)
                e1.record()
                torch.cuda.synchronize()
                times[p].append(e0.elapsed_time(e1) * 1e3)
        ctas, nk = tiles(M, K, N)
        waves = (ctas + 147) // 148
        med = {p: float(np.median(v)) for p, v in times.items()}
        spread = {p: float(np.percentile(v, 90) - np.percentile(v, 10)) for p, v in times.items()}
        print("%6d x %5d -> %5d %9d %9d %8d | %7.1f %7.1f | %6.3f   us/chunk/SM tmem %.3f smem %.3f   "
              "p10-p90 spread tmem %.1f smem %.1f us" % (
                  M, K, N, ctas, nk, waves, med["tmem"], med["smem"], med["tmem"] / med["smem"],
                  med["tmem"] / (waves * nk), med["smem"] / (waves * nk), spread["tmem"], spread["smem"]))
    os.environ["D3F_TC_A_SMEM"] = "0"


if __name__ == "__main__":
    main()
