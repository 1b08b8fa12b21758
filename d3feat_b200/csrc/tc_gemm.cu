// Tensor-core GEMM for sm_100a: tcgen05.mma (kind::tf32) with the accumulator in TMEM, fp32-accurate through
// a 3xTF32 split:   A = Ah + Al,  B = Bh + Bl  (Ah/Bh = operand rounded to TF32, Al/Bl = exact remainder)
//                   D += Ah*Bh + Al*Bh + Ah*Bl          (dropped Al*Bl term ~ 2^-22 relative)
//
//   C[M,N] = epilogue( rowscale[m] * (A[M,K] @ W[K,N]) )
//
// * A is the activation matrix (row-major fp32 in global memory). Producer warp w copies the raw rows it owns,
//   [32w, 32w+32), into a swizzled shared-memory slot (cp.async, 128-bit, coalesced); lane l reads its own row back,
//   splits it into (hi, lo) in registers and writes both to tensor memory (tcgen05.st): TMEM lane = row, one
//   column per k-element. The MMAs take A from TMEM, so shared memory carries only the raw copy of A and the B
//   images. (D3F_TC_A_SMEM=1 keeps the round-2 path for A/B timing: both A images in shared memory, in the K-major
//   SWIZZLE_128B layout of the UMMA descriptor.)
// * W is static: it is packed once (pack_weight_kernel) into K-major [Npad, Kpad] hi/lo images, fetched by TMA.
// * One elected thread of warp 4 issues the MMAs (M = 128, N = BN, K = 8 per instruction, three per K step); a
//   1-4 stage mbarrier ring overlaps the producers with the tensor pipe; tcgen05.commit releases stages / signals the
//   epilogue.
// * Epilogue: warps 0-3 read their 32 TMEM lanes (tcgen05.ld 32x32b), apply rowscale / BN / bias / residual /
//   LeakyReLU and store rows straight to global memory.
#include <stdlib.h>

#include "ops.cuh"
#include "tc_common.cuh"

namespace d3f {

constexpr int kTcBM = 128;       // rows per CTA (UMMA M)
constexpr int kTcBK = 32;        // fp32 per k-chunk = one 128 B swizzle row
constexpr int kTcProducerThreads = 128;
constexpr int kTcThreads = 160;  // 4 producer/epilogue warps + 1 MMA warp

// ---------------------------------------------------------------------------------------------------
// W[K,N] row-major -> packed[Kpad/32][2][Npad][32]: for every 32-wide k-chunk a (hi, lo) pair of ready-made shared
// memory images: row n holds the 32 k-values of output column n as 128 bytes whose 16-byte chunks are XOR-swizzled
// with (n & 7) -- exactly the K-major SWIZZLE_128B layout the UMMA descriptor reads. A BN-row tile of a k-chunk is
// therefore ONE contiguous block per image and is fetched by a single TMA bulk copy (cp.async.bulk).
__global__ void __launch_bounds__(256) pack_weight_kernel(const float* __restrict__ W, int K, int N, int Kpad,
                                                          int Npad, float* __restrict__ packed) {
  long long total = (long long)Npad * Kpad;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int k = (int)(i / Npad), n = (int)(i % Npad);      // consecutive threads: consecutive n (coalesced reads of W)
    float x = (n < N && k < K) ? W[(size_t)k * N + n] : 0.f;
    float hi, lo;
    split_tf32(x, hi, lo);
    int kc = k >> 5, kl = k & 31;
    size_t slab = (size_t)kc * 2 * Npad * 32;
    size_t off = (size_t)n * 32 + (size_t)((((kl >> 2) ^ (n & 7)) << 2) | (kl & 3));
    packed[slab + off] = hi;
    packed[slab + (size_t)Npad * 32 + off] = lo;
  }
}

int tc_padded_k(int K) { return (K + kTcBK - 1) / kTcBK * kTcBK; }
int tc_block_n(int N) { return N > 64 ? 128 : (N > 32 ? 64 : 32); }
int tc_padded_n(int N) { int bn = tc_block_n(N); return (N + bn - 1) / bn * bn; }
size_t tc_packed_floats(int K, int N) { return 2 * (size_t)tc_padded_k(K) * tc_padded_n(N); }

int tc_pack_weight(const float* W, int K, int N, float* packed, cudaStream_t stream) {
  D3F_REQUIRE(K >= 1 && N >= 1 && W && packed, D3F_ERR_INVALID, "pack_weight: bad arguments");
  int Kpad = tc_padded_k(K), Npad = tc_padded_n(N);
  long long total = (long long)Npad * Kpad;
  int blocks = (int)min((total + 255) / 256, (long long)kNumSMs * 8);
  pack_weight_kernel<<<blocks, 256, 0, stream>>>(W, K, N, Kpad, Npad, packed);
  D3F_LAUNCH_CHECK("pack_weight_kernel");
  return D3F_OK;
}

// ---------------------------------------------------------------------------------------------------
// The tensor pipe truncates (round-toward-zero) when it writes the fp32 accumulator back to TMEM: measured bias
// ~ -1.1e-8 * K relative for all-positive data (scripts/tc_accuracy_probe.py). The k-chunks are therefore
// rotated over kAcc independent TMEM accumulators (2 x 128 or 4 x 64 / 4 x 32 columns) that the epilogue adds
// in registers with round-to-nearest: the truncation chain per accumulator is kAcc times shorter.
// ACC = 0: the default rotation (2 x 128, 4 x 64 / 4 x 32 columns; 2 x 64 for the two-CTA <64,2> ring with the A
// operand in TMEM, where 4 x 64 + 128 A columns would not leave room for a second CTA -- K of that variant stays
// <= 1024 in the encoder: bias < 5.6e-6). ACC = 1: a single accumulator for GEMMs of <= 4 k-chunks (K <= 128: bias
// < 1.5e-6), so that four small CTAs share an SM.
// A_SMEM = false (default): the split A operand lives in TMEM, 64 columns per ring stage ([hi 32 | lo 32]) after
// the accumulators. A_SMEM = true: both A images in shared memory (the round-2 operand path, kept for A/B timing).
// TMEM allocation (a power of two >= 32) / ring stages / shared memory / CTAs per SM, A in TMEM vs A in smem:
//   <32,1,1>   32 + 64 -> 128 | 1 |  25 KB | 4        (A_SMEM:  32 | 1 |  41 KB | 4)
//   <64,1,1>   64 + 64 -> 128 | 1 |  33 KB | 4        (A_SMEM:  64 | 1 |  49 KB | 4)
//   <32,2,0>  128 + 128 -> 256 | 2 |  49 KB | 2       (A_SMEM: 128 | 2 |  81 KB | 2)
//   <64,2,0>  128 + 128 -> 256 | 2 |  65 KB | 2       (A_SMEM: 256 | 2 |  97 KB | 2)
//   <128,2,0> 256 + 128 -> 512 | 2 |  97 KB | 1       (A_SMEM: 256 | 2 | 129 KB | 1)
//   <32,4,0>  128 + 256 -> 512 | 4 |  97 KB | 1       (A_SMEM: 128 | 4 | 161 KB | 1)
//   <64,4,0>  256 + 256 -> 512 | 4 | 129 KB | 1       (A_SMEM: 256 | 4 | 193 KB | 1)
//   <128,3,0> 256 + 192 -> 512 | 3 | 145 KB | 1       (A_SMEM: 256 | 3 | 193 KB | 1)
// (CTAs per SM: the launch bounds' register budget; shared memory and TMEM admit at least as many.)
template <int BN, int STAGES, int ACC, bool A_SMEM>
struct TcAcc {
  static constexpr int kAcc = ACC > 0 ? ACC : (BN >= 128 ? 2 : ((BN == 64 && STAGES == 2 && !A_SMEM) ? 2 : 4));
  static constexpr int kACol = kAcc * BN;                    // first TMEM column of the A ring
  static constexpr int kUsed = kACol + (A_SMEM ? 0 : 64 * STAGES);
  static constexpr int kCols = kUsed <= 32 ? 32 : kUsed <= 64 ? 64 : kUsed <= 128 ? 128 : kUsed <= 256 ? 256 : 512;
  static_assert(kUsed <= 512, "TMEM plan exceeds 512 columns");
};

// ring depth = prefetch distance + 1. Skinny-K GEMMs (<= 4 k-chunks) take 2 stages so that two CTAs share an SM and
// overlap each other's load / MMA / epilogue phases; long-K GEMMs take the deepest ring that fits (one CTA per SM).
// A stage holds the raw (A in TMEM) or the hi and lo (A_SMEM) images of the A tile, then the B hi and lo images.
template <int BN, int STAGES, bool A_SMEM>
struct TcSmem {
  static constexpr int kStages = STAGES;
  static constexpr int kABytes = kTcBM * 128;  // one image of the A tile
  static constexpr int kBBytes = BN * 128;
  static constexpr int kBOff = (A_SMEM ? 2 : 1) * kABytes;
  static constexpr int kStageBytes = kBOff + 2 * kBBytes;
  static constexpr int kTotal = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;
};

template <int BN, int STAGES, int ACC, bool A_SMEM>
__global__ void __launch_bounds__(kTcThreads, STAGES == 1 ? 4 : ((STAGES == 2 && BN <= 64) ? 2 : 1))
tc_gemm_kernel(const float* __restrict__ A, const float* __restrict__ A2, int K1, const float* __restrict__ Bp,
               float* __restrict__ C, int Mcap, int N, int K, int Kpad, int Npad, int chunks_per_split, Epilogue ep) {
  // the split-K slabs are laid out with the launch capacity; the rows that exist come from device memory if given
  const int M = ep.m_dev ? min(Mcap, max(__ldg(ep.m_dev) - ep.m_off, 0)) : Mcap;
  if ((int)blockIdx.y * kTcBM >= M) return;   // CTA-uniform, before any barrier / TMEM allocation
  extern __shared__ uint8_t smem_raw[];
  using S = TcSmem<BN, STAGES, A_SMEM>;
  using P = TcAcc<BN, STAGES, ACC, A_SMEM>;
  constexpr int kStages = S::kStages;
  // 1024 B alignment: SWIZZLE_128B atoms are 8 rows x 128 B and the swizzle uses absolute address bits
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = (uint64_t*)(smem + kStages * S::kStageBytes);
  // bars[0..S) full, bars[S..2S) empty, bars[2S] accumulator ready; then the TMEM base address
  uint32_t* tmem_slot = (uint32_t*)(bars + 2 * kStages + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = blockIdx.y * kTcBM, n0 = blockIdx.x * BN;
  // split-K: CTA z owns the k-chunks [kt0, kt0 + nk) and writes raw partial sums to its own [M,N] slab of C
  const int kt0 = blockIdx.z * chunks_per_split;
  const int nk = min(Kpad / kTcBK - kt0, chunks_per_split);
  C += (size_t)blockIdx.z * Mcap * N;

  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(smem_u32(&bars[s]), kTcProducerThreads + 1);   // + the TMA issuer's arrive.expect_tx
      mbar_init(smem_u32(&bars[kStages + s]), 1);
    }
    mbar_init(smem_u32(&bars[2 * kStages]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)P::kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < 4) {
    // ===================== producers: global --cp.async--> swizzled raw stage --hi/lo split--> operand =========
    // The raw fp32 A tile is copied asynchronously kStages-1 k-chunks ahead (rows beyond M / K zero-filled), the
    // pre-split B images by TMA. When a thread's copy group of chunk kt has landed (cp.async.wait_group is per
    // thread) the A values are split into (hi, lo):
    //   A in TMEM: warp w copies the 32 rows it owns, [32w, 32w+32) (eight lanes per 128-byte row segment); after
    //     wait_group + __syncwarp lane l reads its own row 32w + l back (eight 16-byte chunks; the swizzle puts the
    //     rows of a quarter-warp in distinct bank groups) and writes hi / lo to TMEM lane 32w + l, columns
    //     [kACol + 64 s, +32) / [kACol + 64 s + 32, +32). Warp w may only touch TMEM lanes [32w, 32w+32).
    //   A_SMEM: every thread owns fixed 16-byte pieces of the stage and splits them in place (hi overwrites the raw
    //     value, lo goes to the second image), in the K-major SWIZZLE_128B layout the UMMA descriptor reads.
    const int chunk = A_SMEM ? (tid & 7) : (lane & 7);      // 16-byte chunk inside the 128-byte row
    constexpr int kRowStep = A_SMEM ? 16 : 4;                 // rows one copy instruction covers
    const int rbase = A_SMEM ? (tid >> 3) : warp * 32 + (lane >> 3);
    auto issue_chunk = [&](int kt) {
      const int s = kt % kStages;
      const uint32_t ph = (uint32_t)(kt / kStages) & 1u;
      mbar_wait(smem_u32(&bars[kStages + s]), ph ^ 1u);      // stage free (its MMAs retired)
      if constexpr (!A_SMEM) tc_fence_after();               // the TMEM A stage is rewritten after this wait
      uint8_t* st = smem + s * S::kStageBytes;
      // the A operand is [A | A2] along K when A2 is given (K1 = columns of A, a multiple of the k-chunk): a whole
      // k-chunk comes from one of the two row-major matrices
      int k0 = (kt0 + kt) * kTcBK + chunk * 4;
      const float* src = A;
      int ld = K;
      if (A2 != nullptr) {
        ld = K1;
        if (k0 >= K1) {
          src = A2;
          ld = K - K1;
          k0 -= K1;
        }
      }
#pragma unroll
      for (int it = 0; it < (A_SMEM ? kTcBM : 32) / kRowStep; ++it) {
        const int row = rbase + it * kRowStep;
        const int gm = m0 + row;
        const uint32_t off = (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
        const bool ok = gm < M && k0 < ld;
        cp_async16_zfill(smem_u32(st + off), src + (size_t)(ok ? gm : 0) * ld + (ok ? k0 : 0), ok);
      }
      if (tid == 0) {
        // B operand of this k-chunk: two contiguous pre-swizzled images (hi, lo) of BN rows x 128 B -> two TMA bulk
        // copies that complete on the stage's "full" barrier
        const uint32_t full = smem_u32(&bars[s]);
        const float* slab = Bp + (size_t)(kt0 + kt) * 2 * Npad * 32 + (size_t)n0 * 32;
        mbar_arrive_expect_tx(full, 2u * S::kBBytes);
        tma_bulk_g2s(smem_u32(st + S::kBOff), slab, S::kBBytes, full);
        tma_bulk_g2s(smem_u32(st + S::kBOff + S::kBBytes), slab + (size_t)Npad * 32, S::kBBytes, full);
      }
    };
    for (int i = 0; i < kStages - 1; ++i) {
      if (i < nk) issue_chunk(i);
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (int kt = 0; kt < nk; ++kt) {
      const int s = kt % kStages;
      uint8_t* st = smem + s * S::kStageBytes;
      if constexpr (kStages == 1) {
        // one stage: copy, split, hand over; the next chunk's copy waits for this chunk's MMAs. The overlap comes
        // from the other CTAs on the SM (four fit).
        issue_chunk(kt);
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
      } else {
        asm volatile("cp.async.wait_group %0;" ::"n"(kStages >= 2 ? kStages - 2 : 0) : "memory");   // chunk kt landed
      }
      const uint32_t st_s = smem_u32(st);
      if constexpr (A_SMEM) {
        // all of this thread's pieces are read before anything is written back: the loads are independent of the
        // in-place stores (which the compiler could not prove), so the eight shared-memory round trips overlap
        float4 x[kTcBM / 16];
#pragma unroll
        for (int it = 0; it < kTcBM / 16; ++it) {
          const int row = it * 16 + rbase;
          const uint32_t off = (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
          x[it] = lds128(st_s + off);
        }
#pragma unroll
        for (int it = 0; it < kTcBM / 16; ++it) {
          const int row = it * 16 + rbase;
          const uint32_t off = (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
          float4 hi, lo;
          split_tf32(x[it].x, hi.x, lo.x);
          split_tf32(x[it].y, hi.y, lo.y);
          split_tf32(x[it].z, hi.z, lo.z);
          split_tf32(x[it].w, hi.w, lo.w);
          sts128(st_s + off, hi);
          sts128(st_s + S::kABytes + off, lo);
        }
        fence_proxy_async();   // generic-proxy writes -> visible to the tensor core (async proxy)
      } else {
        __syncwarp();          // the other lanes' pieces of this warp's rows have landed too
        const int row = warp * 32 + lane;
        float hi[32], lo[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float4 x = lds128(st_s + (uint32_t)row * 128u + (uint32_t)((c ^ (row & 7)) << 4));
          split_tf32(x.x, hi[4 * c + 0], lo[4 * c + 0]);
          split_tf32(x.y, hi[4 * c + 1], lo[4 * c + 1]);
          split_tf32(x.z, hi[4 * c + 2], lo[4 * c + 2]);
          split_tf32(x.w, hi[4 * c + 3], lo[4 * c + 3]);
        }
        const uint32_t ta = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(P::kACol + 64 * s);
        tmem_st32(ta, hi);
        tmem_st32(ta + 32u, lo);
        tc_fence_before();     // the completed TMEM stores -> ordered before the MMA issuer's wait on full[s]
      }
      mbar_arrive(smem_u32(&bars[s]));
      if constexpr (kStages > 1) {
        // refill the stage that MMA(kt-1) is about to release, kStages-1 chunks ahead
        if (kt + kStages - 1 < nk) issue_chunk(kt + kStages - 1);
        asm volatile("cp.async.commit_group;" ::: "memory");        // possibly empty: keeps the group count uniform
      }
    }

    // ===================== epilogue: TMEM -> registers -> smem transpose -> coalesced global ============
    // Each warp owns TMEM lanes / tile rows [32w, 32w+32). A thread reads its row's 32 columns from TMEM, the
    // warp transposes them through a padded 32x33 shared tile (the stage buffers are free: every MMA that
    // read them has retired when the accumulator barrier fires), then lane <-> column: the per-column BN /
    // bias parameters sit in registers and every residual load / store is one coalesced 128-byte row segment.
    mbar_wait(smem_u32(&bars[2 * kStages]), 0);
    tc_fence_after();
    const int row = warp * 32 + lane;      // TMEM lane == tile row; warp w may only touch lanes [32w, 32w+32)
    const int gm = m0 + row;
    const float rs = (ep.rowscale != nullptr && gm < M) ? ep.rowscale[gm] : 1.f;
    const int nacc = nk < P::kAcc ? nk : P::kAcc;
    const uint32_t tile = smem_u32(smem) + (uint32_t)warp * (32 * 33 * 4);
    const int rows_here = min(32, M - (m0 + warp * 32));   // rows of this warp that exist (<= 0: none)
    const bool has_bn = ep.bn_scale != nullptr, has_bias = ep.bias != nullptr, has_res = ep.residual != nullptr;
    const bool has_leaky = ep.leaky_alpha >= 0.f;
    // output row of tile row (warp*32 + lane): identity, or the caller's row map (KPConv walks its queries in
    // the hash grid's cell order and scatters the rows back)
    const int my_orow = (gm < M) ? (ep.row_map ? ep.row_map[gm] : gm) : 0;
    const bool full_tile = rows_here == 32 && ep.row_map == nullptr && (!has_leaky || (ep.leaky_alpha >= 0.f && ep.leaky_alpha <= 1.f));
    const float alpha_eff = has_leaky ? ep.leaky_alpha : 1.f;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      const int gn = n0 + c0 + lane;
      const bool col_ok = gn < N;
      // residual rows of this column chunk: all 32 coalesced loads are in flight before anything waits on them
      float res[32];
      if (has_res && full_tile && n0 + c0 + 32 <= N) {
        const float* rp = ep.residual + (size_t)(m0 + warp * 32) * N + gn;
#pragma unroll
        for (int rr = 0; rr < 32; ++rr) res[rr] = rp[(size_t)rr * N];
      } else if (has_res) {
#pragma unroll
        for (int rr = 0; rr < 32; ++rr) {
          const int orow = __shfl_sync(0xffffffffu, my_orow, rr);
          res[rr] = (col_ok && rr < rows_here) ? ep.residual[(size_t)orow * N + gn] : 0.f;
        }
      }
      float v[32];
      tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
#pragma unroll 1
      for (int a = 1; a < nacc; ++a) {
        float w[32];
        tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(a * BN + c0), w);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += w[j];
      }
#pragma unroll
      for (int j = 0; j < 32; ++j) sts32(tile + (uint32_t)(lane * 33 + j) * 4u, v[j] * rs);
      __syncwarp();
      const float sc = (has_bn && col_ok) ? ep.bn_scale[gn] : 1.f;
      const float sh = (has_bn && col_ok) ? ep.bn_shift[gn] : 0.f;
      const float bi = (has_bias && col_ok) ? ep.bias[gn] : 0.f;
      if (full_tile && n0 + c0 + 32 <= N) {
        // interior tile (all but the last row block / column chunk), rows in place: no per-element predicates, no
        // shuffles, one pointer bump per row. LeakyReLU with 0 <= alpha <= 1 is max(y, alpha y); alpha = 1: identity.
        // (ncu of the level-0 unaries: 10.7k warp instructions per 128 x 64 tile, two thirds of them in this loop's
        // address / predicate scaffolding; the kernel sat at 61 % issue-slot utilisation.)
        float* cp = C + (size_t)(m0 + warp * 32) * N + gn;
#pragma unroll
        for (int rr = 0; rr < 32; ++rr) {
          float y = fmaf(lds32(tile + (uint32_t)(rr * 33 + lane) * 4u), sc, sh) + bi;
          if (has_res) y += res[rr];
          y = fmaxf(y, y * alpha_eff);
          cp[(size_t)rr * N] = y;
        }
      } else {
#pragma unroll
        for (int rr = 0; rr < 32; ++rr) {
          const int orow = __shfl_sync(0xffffffffu, my_orow, rr);
          if (col_ok && rr < rows_here) {
            float y = fmaf(lds32(tile + (uint32_t)(rr * 33 + lane) * 4u), sc, sh) + bi;
            if (has_res) y += res[rr];
            if (has_leaky) y = y > 0.f ? y : y * ep.leaky_alpha;
            C[(size_t)orow * N + gn] = y;
          }
        }
      }
      __syncwarp();
    }
    tc_fence_before();
  } else {
    // ===================== MMA issuer (warp 4, one elected lane) ========================================
    const uint32_t idesc = make_idesc_tf32(kTcBM, BN);
    for (int kt = 0; kt < nk; ++kt) {
      const int s = kt % kStages;
      const uint32_t ph = (uint32_t)(kt / kStages) & 1u;
      mbar_wait(smem_u32(&bars[s]), ph);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t sa = smem_u32(smem + s * S::kStageBytes);
        const uint64_t b_hi = make_smem_desc(sa + S::kBOff), b_lo = make_smem_desc(sa + S::kBOff + S::kBBytes);
        const uint32_t d = tmem_base + (uint32_t)((kt % P::kAcc) * BN);
#pragma unroll
        for (int j = 0; j < kTcBK / 8; ++j) {
          const uint64_t adv = (uint64_t)((j * 32) >> 4);   // +32 B per K = 8 step inside the swizzle atom
          const uint32_t acc = (kt >= P::kAcc || j != 0) ? 1u : 0u;
          if constexpr (A_SMEM) {
            const uint64_t a_hi = make_smem_desc(sa), a_lo = make_smem_desc(sa + S::kABytes);
            umma_tf32(d, a_hi + adv, b_hi + adv, idesc, acc);
            umma_tf32(d, a_lo + adv, b_hi + adv, idesc, 1u);
            umma_tf32(d, a_hi + adv, b_lo + adv, idesc, 1u);
          } else {
            // A stage s: hi at columns [kACol + 64 s, +32), lo at [+32, +64); K = 8 columns per MMA
            const uint32_t a_hi = tmem_base + (uint32_t)(P::kACol + 64 * s + 8 * j);
            umma_tf32_ts(d, a_hi, b_hi + adv, idesc, acc);
            umma_tf32_ts(d, a_hi + 32u, b_hi + adv, idesc, 1u);
            umma_tf32_ts(d, a_hi, b_lo + adv, idesc, 1u);
          }
        }
        umma_commit(smem_u32(&bars[kStages + s]));                 // stage free once these MMAs retire
        if (kt == nk - 1) umma_commit(smem_u32(&bars[2 * kStages]));  // accumulator complete
      }
      __syncwarp();
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base),
                 "r"((uint32_t)P::kCols)
                 : "memory");
  }
}

// fixed-order reduction of the split-K partials + the block epilogue
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ part, int splits, int Mcap, int N,
                                                            Epilogue ep, float* __restrict__ C) {
  const int M = ep.m_dev ? min(Mcap, max(__ldg(ep.m_dev) - ep.m_off, 0)) : Mcap;
  const long long slab = (long long)Mcap * N;
  long long total = (long long)M * N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    int m = (int)(i / N), n = (int)(i % N);
    float y = 0.f;
    for (int z = 0; z < splits; ++z) y += part[(size_t)z * slab + i];
    if (ep.rowscale) y *= ep.rowscale[m];
    if (ep.bn_scale) y = fmaf(y, ep.bn_scale[n], ep.bn_shift[n]);
    if (ep.bias) y += ep.bias[n];
    const size_t orow = ep.row_map ? (size_t)ep.row_map[m] : (size_t)m;
    if (ep.residual) y += ep.residual[orow * N + n];
    if (ep.leaky_alpha >= 0.f) y = y > 0.f ? y : y * ep.leaky_alpha;
    C[orow * N + n] = y;
  }
}

template <int BN, bool A_SMEM, int STAGES, int ACC = 0>
static int launch_tc_s(const float* A, const float* A2, int K1, const float* Bp, float* C, int M, int N, int K,
                       const Epilogue& ep, cudaStream_t stream, int splits, float* split_ws) {
  using S = TcSmem<BN, STAGES, A_SMEM>;
  static bool configured = false;   // idempotent attribute set; benign if two host threads race
  if (!configured) {
    D3F_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<BN, STAGES, ACC, A_SMEM>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
    configured = true;
  }
  int Kpad = tc_padded_k(K), Npad = tc_padded_n(N);
  const int nk = Kpad / kTcBK;
  if (splits <= 1) {
    dim3 grid(Npad / BN, ceil_div(M, kTcBM), 1);
    tc_gemm_kernel<BN, STAGES, ACC, A_SMEM><<<grid, kTcThreads, S::kTotal, stream>>>(A, A2, K1, Bp, C, M, N, K, Kpad, Npad, nk, ep);
    D3F_LAUNCH_CHECK("tc_gemm_kernel");
    return D3F_OK;
  }
  const int cps = ceil_div(nk, splits);
  splits = ceil_div(nk, cps);
  Epilogue raw;
  raw.rowscale = nullptr; raw.bn_scale = nullptr; raw.bn_shift = nullptr; raw.bias = nullptr; raw.residual = nullptr;
  raw.leaky_alpha = -1.f; raw.row_map = nullptr; raw.m_dev = ep.m_dev; raw.m_off = ep.m_off;
  dim3 grid(Npad / BN, ceil_div(M, kTcBM), splits);
  tc_gemm_kernel<BN, STAGES, ACC, A_SMEM><<<grid, kTcThreads, S::kTotal, stream>>>(A, A2, K1, Bp, split_ws, M, N, K, Kpad, Npad, cps, raw);
  D3F_LAUNCH_CHECK("tc_gemm_kernel");
  long long total = (long long)M * N;
  int blocks = (int)min((total + 255) / 256, (long long)kNumSMs * 8);
  splitk_reduce_kernel<<<blocks, 256, 0, stream>>>(split_ws, splits, M, N, ep, C);
  D3F_LAUNCH_CHECK("splitk_reduce_kernel");
  return D3F_OK;
}

// ---------------------------------------------------------------------------------------------------
// Streaming variant for the long-K, huge-M GEMMs of levels 0/1: the KPConv contractions [Nq, 15 Cin] x [15 Cin, Cout]
// on 60k-240k rows with Cout <= 64 (VERDICT item 5, "operand pipeline"). OPT-IN (D3F_TC_STREAM=1): measured
// (scripts/gemm_probe.py, profiles/r2_notes.md section 7) it gains 10 % on the 240k-row contraction (0.157 -> 0.142 ms)
// and nothing on the 60k-row ones, while it owns all 512 TMEM columns and ~200 KB of shared memory of every SM.
// ONE persistent CTA per SM walks its tiles and the product is issued TRANSPOSED:
//     D[2 BN, 256] += Wimg[2 BN, 8] . Ximg[256, 8]^T        one tcgen05.mma per K = 8 step instead of three
//   rows    0..BN-1 = W_hi of the tile's output channels, BN..2BN-1 = W_lo   (the two packed images are adjacent in smem)
//   columns 0..127  = X_hi of the tile's 128 rows,        128..255 = X_lo    (the split images are adjacent in smem)
//   out[q][c] = D[c][q] + D[c][128+q] + D[BN+c][q]          (3xTF32; the lo*lo quadrant is ignored)
// so the same shared-memory images serve with the operand roles swapped.
//   * 8 producer warps: cp.async of the raw fp32 X pieces three k-chunks ahead, in-place hi/lo split, W images by TMA;
//     the ring never drains between tiles;
//   * 1 MMA warp: 4 MMAs per k-chunk into one of two 256-column TMEM accumulators (double-buffered by tile parity);
//   * 4 epilogue warps (one TMEM lane quadrant each): 32 queries at a time, TMEM -> registers -> two partial tiles in
//     shared memory (W_hi rows, W_lo rows) -> summed, epilogue applied, coalesced rows; overlaps the next tile's k-loop.
// Barriers: full[s] / empty[s] per ring stage (chunk counter runs across tiles), acc_full[b] / acc_empty[b] per TMEM set.
// One accumulator per tile: the write-back truncation (see TcAcc) is ~1.1e-8 K, so the host keeps K <= 1024 here.
// What the three measured variants say (same 0.74-0.86 us per k-chunk and SM in all of them: twelve M=128 MMAs or
// four M=64/128 x N=256 MMAs per chunk, 3 or 6 chunks of loads in flight): neither the tensor pipe nor the bytes in
// flight bound these GEMMs -- the 3xTF32 split does. Per 16 KB chunk the SM moves 16 KB (cp.async write) + 16 KB (LDS)
// + 32 KB (STS hi, lo) + 40 KB (operand reads of the MMAs) through shared memory: 104 KB at 128 B/clk = 0.41 us.
constexpr int kStProdWarps = 8;
constexpr int kStProdThreads = kStProdWarps * 32;
constexpr int kStThreads = (kStProdWarps + 4 + 1) * 32;   // + 4 epilogue warps + the MMA warp

template <int BN>
struct StSmem {
  static constexpr int kStages = 4;
  static constexpr int kABytes = kTcBM * 128;               // one image (hi or lo) of the 128-row X tile
  static constexpr int kBBytes = BN * 128;                  // one image of the BN-row W tile
  static constexpr int kStageBytes = 2 * kABytes + 2 * kBBytes;
  static constexpr int kPStride = BN + 1;                   // padded row of a partial tile
  static constexpr int kPBytes = 2 * 32 * kPStride * 4;     // [W_hi | W_lo part][32 queries][BN + 1]
  static constexpr int kTotal = kStages * kStageBytes + kPBytes + 1024 /*align*/ + 256 /*barriers*/;
  static constexpr int kCols = 512;                         // two accumulators of 256 columns
};

template <int BN>
__global__ void __launch_bounds__(kStThreads, 1)
tc_gemm_stream_kernel(const float* __restrict__ A, const float* __restrict__ A2, int K1, const float* __restrict__ Bp,
                      float* __restrict__ C, int Mcap, int N, int K, int Kpad, int Npad, Epilogue ep) {
  const int M = ep.m_dev ? min(Mcap, max(__ldg(ep.m_dev) - ep.m_off, 0)) : Mcap;
  const int nk = Kpad / kTcBK;
  const int ntn = Npad / BN;
  const int tiles = ceil_div(M, kTcBM) * ntn;                // n-tiles of one row block are neighbours: X stays in L2
  if ((int)blockIdx.x >= tiles) return;                      // CTA-uniform, before any barrier / TMEM allocation
  const int my_tiles = (tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  extern __shared__ uint8_t smem_raw[];
  using S = StSmem<BN>;
  constexpr int kStages = S::kStages;
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* part_smem = smem + kStages * S::kStageBytes;
  uint64_t* bars = (uint64_t*)(part_smem + ((S::kPBytes + 15) / 16) * 16);
  uint64_t* full = bars;                       // [kStages] split images + weight images of a chunk complete
  uint64_t* empty = full + kStages;            // [kStages] the MMAs that read the stage retired
  uint64_t* acc_full = empty + kStages;        // [2]
  uint64_t* acc_empty = acc_full + 2;          // [2]
  uint32_t* tmem_slot = (uint32_t*)(acc_empty + 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(smem_u32(&full[s]), kStProdThreads + 1);     // + the TMA issuer's arrive.expect_tx
      mbar_init(smem_u32(&empty[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&acc_full[b]), 1);
      mbar_init(smem_u32(&acc_empty[b]), 4);                 // one arrive per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kStProdWarps + 4) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)S::kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kStProdWarps) {
    // ===================== producers ======================================================================
    const int chunk = tid & 7;      // 16-byte chunk inside the 128-byte row
    const int rsub = tid >> 3;      // 0..31: row inside a 32-row slab
    const int total = my_tiles * nk;
    int i_tile = (int)blockIdx.x, i_kt = 0, i_g = 0;         // the next chunk to copy: (tile, k-chunk), running number
    auto issue_chunk = [&]() {
      const int s = i_g % kStages;
      const uint32_t ph = (uint32_t)(i_g / kStages) & 1u;
      mbar_wait(smem_u32(&empty[s]), ph ^ 1u);               // stage free (its MMAs retired)
      uint8_t* st = smem + s * S::kStageBytes;
      const int m0 = (i_tile / ntn) * kTcBM, n0 = (i_tile % ntn) * BN;
      int k0 = i_kt * kTcBK + chunk * 4;
      const float* src = A;
      int ld = K;
      if (A2 != nullptr) {
        ld = K1;
        if (k0 >= K1) {
          src = A2;
          ld = K - K1;
          k0 -= K1;
        }
      }
#pragma unroll
      for (int it = 0; it < kTcBM / 32; ++it) {
        const int row = it * 32 + rsub;
        const int gm = m0 + row;
        const uint32_t off = (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
        const bool ok = gm < M && k0 < ld;
        cp_async16_zfill(smem_u32(st + off), src + (size_t)(ok ? gm : 0) * ld + (ok ? k0 : 0), ok);
      }
      if (tid == 0) {
        const uint32_t fb = smem_u32(&full[s]);
        const float* slab = Bp + (size_t)i_kt * 2 * Npad * 32 + (size_t)n0 * 32;
        mbar_arrive_expect_tx(fb, 2u * S::kBBytes);
        tma_bulk_g2s(smem_u32(st + 2 * S::kABytes), slab, S::kBBytes, fb);
        tma_bulk_g2s(smem_u32(st + 2 * S::kABytes + S::kBBytes), slab + (size_t)Npad * 32, S::kBBytes, fb);
      }
      ++i_g;
      if (++i_kt == nk) {
        i_kt = 0;
        i_tile += (int)gridDim.x;
      }
    };
    for (int i = 0; i < kStages - 1; ++i) {
      if (i < total) issue_chunk();
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (int g = 0; g < total; ++g) {
      const int s = g % kStages;
      asm volatile("cp.async.wait_group %0;" ::"n"(kStages - 2) : "memory");   // this thread's pieces of chunk g landed
      const uint32_t st_s = smem_u32(smem + s * S::kStageBytes);
      float4 x[kTcBM / 32];
#pragma unroll
      for (int it = 0; it < kTcBM / 32; ++it) {
        const int row = it * 32 + rsub;
        x[it] = lds128(st_s + (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4));
      }
#pragma unroll
      for (int it = 0; it < kTcBM / 32; ++it) {
        const int row = it * 32 + rsub;
        const uint32_t off = (uint32_t)row * 128u + (uint32_t)((chunk ^ (row & 7)) << 4);
        float4 hi, lo;
        split_tf32(x[it].x, hi.x, lo.x);
        split_tf32(x[it].y, hi.y, lo.y);
        split_tf32(x[it].z, hi.z, lo.z);
        split_tf32(x[it].w, hi.w, lo.w);
        sts128(st_s + off, hi);
        sts128(st_s + S::kABytes + off, lo);
      }
      fence_proxy_async();   // generic-proxy writes -> visible to the tensor core (async proxy)
      mbar_arrive(smem_u32(&full[s]));
      if (i_g < total) issue_chunk();
      asm volatile("cp.async.commit_group;" ::: "memory");        // possibly empty: keeps the group count uniform
    }
  } else if (warp < kStProdWarps + 4) {
    // ===================== epilogue warps: accumulator b of tile i while the k-loop of tile i+1 runs =========
    // quadrant ew holds D rows [ew * RQ, (ew + 1) * RQ): ew = 0, 1 -> W_hi rows of channels (ew & 1) * RQ + lane,
    // ew = 2, 3 -> the W_lo rows of the same channels (M = 64: 16 rows per quadrant in lanes 0..15; M = 128: 32)
    constexpr int RQ = BN / 2;
    constexpr int PS = S::kPStride;
    const int ew = warp - kStProdWarps;                      // == warp % 4: the TMEM lane quadrant this warp may read
    const int et = tid - kStProdThreads;                     // 0..127 inside the epilogue group
    const int wpart = ew >> 1;
    const int ch = (ew & 1) * RQ + lane;                     // channel of this lane's accumulator row (lane < RQ)
    const uint32_t part = smem_u32(part_smem);
    const bool has_bn = ep.bn_scale != nullptr, has_bias = ep.bias != nullptr, has_res = ep.residual != nullptr;
    const bool has_leaky = ep.leaky_alpha >= 0.f;
    for (int i = 0; i < my_tiles; ++i) {
      const int t = (int)blockIdx.x + i * (int)gridDim.x;
      const int m0 = (t / ntn) * kTcBM, n0 = (t % ntn) * BN;
      const int b = i & 1;
      mbar_wait(smem_u32(&acc_full[b]), (uint32_t)(i >> 1) & 1u);
      tc_fence_after();
      const uint32_t tacc = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(b * 256);
#pragma unroll 1
      for (int q0 = 0; q0 < kTcBM; q0 += 32) {
        if (m0 + q0 >= M) break;                             // uniform over the epilogue group
        float v[32];
        tmem_ld32(tacc + (uint32_t)q0, v);                   // . x X_hi
        if (wpart == 0) {
          float w[32];
          tmem_ld32(tacc + (uint32_t)(128 + q0), w);         // W_hi x X_lo
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] += w[j];
        }
        if (lane < RQ) {
#pragma unroll
          for (int j = 0; j < 32; ++j) sts32(part + (uint32_t)((wpart * 32 + j) * PS + ch) * 4u, v[j]);
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");
        // 32 queries x BN channels: a warp writes 8 rows, lanes run along the channels (coalesced row segments)
#pragma unroll 1
        for (int rr = 0; rr < 8; ++rr) {
          const int r = (et >> 5) * 8 + rr;
          const int gm = m0 + q0 + r;
          if (gm >= M) break;                                // warp-uniform
          const float rs = ep.rowscale != nullptr ? ep.rowscale[gm] : 1.f;
          const size_t orow = ep.row_map ? (size_t)ep.row_map[gm] : (size_t)gm;
#pragma unroll
          for (int c = lane; c < BN; c += 32) {
            const int gn = n0 + c;
            if (gn < N) {
              float y = lds32(part + (uint32_t)(r * PS + c) * 4u) + lds32(part + (uint32_t)((32 + r) * PS + c) * 4u);
              y *= rs;
              if (has_bn) y = fmaf(y, ep.bn_scale[gn], ep.bn_shift[gn]);
              if (has_bias) y += ep.bias[gn];
              if (has_res) y += ep.residual[orow * N + gn];
              if (has_leaky) y = y > 0.f ? y : y * ep.leaky_alpha;
              C[orow * N + gn] = y;
            }
          }
        }
        asm volatile("bar.sync 1, 128;" ::: "memory");      // the partial tiles are free again
      }
      // every lane's tcgen05.ld has completed (wait::ld inside tmem_ld32): hand the accumulator back
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&acc_empty[b]));
    }
  } else {
    // ===================== MMA issuer (one elected lane) ====================================================
    const uint32_t idesc = make_idesc_tf32(2 * BN, 256);
    int g = 0;
    for (int i = 0; i < my_tiles; ++i) {
      const int b = i & 1;
      mbar_wait(smem_u32(&acc_empty[b]), ((uint32_t)(i >> 1) & 1u) ^ 1u);   // accumulator b drained (tile i - 2)
      tc_fence_after();
      for (int kt = 0; kt < nk; ++kt, ++g) {
        const int s = g % kStages;
        mbar_wait(smem_u32(&full[s]), (uint32_t)(g / kStages) & 1u);
        tc_fence_after();
        if (lane == 0) {
          const uint32_t sa = smem_u32(smem + s * S::kStageBytes);
          const uint64_t x_img = make_smem_desc(sa);                        // 256 rows: X_hi | X_lo
          const uint64_t w_img = make_smem_desc(sa + 2 * S::kABytes);       // 2 BN rows: W_hi | W_lo
          const uint32_t d = tmem_base + (uint32_t)(b * 256);
#pragma unroll
          for (int j = 0; j < kTcBK / 8; ++j) {
            const uint64_t adv = (uint64_t)((j * 32) >> 4);   // +32 B per K = 8 step inside the swizzle atom
            umma_tf32(d, w_img + adv, x_img + adv, idesc, (kt != 0 || j != 0) ? 1u : 0u);
          }
          umma_commit(smem_u32(&empty[s]));                       // stage free once these MMAs retire
          if (kt == nk - 1) umma_commit(smem_u32(&acc_full[b]));  // accumulator complete
        }
        __syncwarp();
      }
    }
    tc_fence_before();
  }
  __syncthreads();
  if (warp == kStProdWarps + 4) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)S::kCols)
                 : "memory");
  }
}

template <int BN>
static int launch_tc_stream(const float* A, const float* A2, int K1, const float* Bp, float* C, int M, int N, int K,
                            const Epilogue& ep, cudaStream_t stream) {
  using S = StSmem<BN>;
  static bool configured = false;   // idempotent attribute set; benign if two host threads race
  if (!configured) {
    D3F_CUDA(cudaFuncSetAttribute(tc_gemm_stream_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, S::kTotal));
    configured = true;
  }
  const int Kpad = tc_padded_k(K), Npad = tc_padded_n(N);
  const long long tiles = (long long)ceil_div(M, kTcBM) * (Npad / BN);
  const int grid = (int)(tiles < kNumSMs ? tiles : kNumSMs);
  tc_gemm_stream_kernel<BN><<<grid, kStThreads, S::kTotal, stream>>>(A, A2, K1, Bp, C, M, N, K, Kpad, Npad, ep);
  D3F_LAUNCH_CHECK("tc_gemm_stream_kernel");
  return D3F_OK;
}

// D3F_TC_SKINNY=0 disables the single-stage variant (A/B measurements); D3F_TC_SKINNY_CHUNKS caps its k-chunks
static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}
static bool force_deep_ring() {
  static const bool off = env_int("D3F_TC_SKINNY", 1) == 0;
  return off;
}
static const int kSkinnyChunks = [] { int c = env_int("D3F_TC_SKINNY_CHUNKS", 4); return c < 1 ? 1 : (c > 4 ? 4 : c); }();

template <int BN, bool A_SMEM>
static int launch_tc(const float* A, const float* A2, int K1, const float* Bp, float* C, int M, int N, int K,
                     const Epilogue& ep, cudaStream_t stream, int splits = 1, float* split_ws = nullptr) {
  const int nk_per_cta = ceil_div(tc_padded_k(K) / kTcBK, splits > 1 ? splits : 1);
  const long long ctas = (long long)ceil_div(M, kTcBM) * (tc_padded_n(N) / BN) * (splits > 1 ? splits : 1);
  // measured on B200 (scripts/gemm_probe.py): with more CTAs than SMs, two co-resident CTAs (2 stages each) beat one
  // CTA with a deep ring; with few CTAs the deep ring wins
  // memory-bound skinny GEMMs with many output tiles (the level-0/1 unary convolutions): single-stage, single
  // accumulator CTAs, four per SM -- their load / MMA / epilogue phases overlap across CTAs
  if constexpr (BN <= 64) {
    if (nk_per_cta <= kSkinnyChunks && splits <= 1 && ctas > 4ll * kNumSMs && !force_deep_ring())
      return launch_tc_s<BN, A_SMEM, 1, 1>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
  }
  if (nk_per_cta <= 4 || (BN <= 64 && ctas > kNumSMs)) return launch_tc_s<BN, A_SMEM, 2>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
  return launch_tc_s<BN, A_SMEM, (BN >= 128 ? 3 : 4)>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
}

bool tc_gemm_supported(const float* A, int K) {
  return (K % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
}

// A[M,K] fp32 row-major, Bp = packed weight (tc_pack_weight), C[M,N]
// split-K plan for GEMMs that cannot fill the GPU with output tiles: returns the number of K splits (1 = none)
// Deterministic split-K plan for GEMMs whose output tiles cannot fill the GPU. The k-loop of a CTA is latency bound
// (about a microsecond per k-chunk), so the cost of a plan is (waves of CTAs) x (k-chunks per CTA) plus the extra
// pass of the reduction; the cheapest of s = 1..8 wins. Returns the number of K splits (1 = none).
int tc_gemm_splits(int M, int N, int K) {
  const int bn = tc_block_n(N);
  const long long ctas = (long long)ceil_div(M, kTcBM) * (tc_padded_n(N) / bn);
  const int nk = tc_padded_k(K) / kTcBK;
  if (ctas >= 96 || nk < 16) return 1;
  int best = 1;
  long long best_cost = (long long)ceil_div((int)ctas, kNumSMs) * nk * 8;   // in eighths of a k-chunk
  for (int s = 2; s <= 8 && s <= nk / 4; ++s) {
    const int cps = ceil_div(nk, s);
    const int eff = ceil_div(nk, cps);   // splits actually launched
    if (eff != s) continue;
    long long cost = (long long)ceil_div((int)(ctas * s), kNumSMs) * cps * 8 + 40 + 6 * s;   // + reduce launch, traffic
    if (cost < best_cost) {
      best_cost = cost;
      best = s;
    }
  }
  return best;
}
// Workspace bound that holds for every M' <= M of the same GEMM family (the chunks of one KPConv share a buffer): the
// planner only splits below 96 output tiles and never more than 8 ways, and a partial slab is at most one 128 x bn
// tile per CTA, so 8 x min(tiles, 95) tiles always suffice.
size_t tc_gemm_split_ws_floats(int M, int N, int K) {
  const int bn = tc_block_n(N);
  const long long ctas = (long long)ceil_div(M, kTcBM) * (tc_padded_n(N) / bn);
  const int nk = tc_padded_k(K) / kTcBK;
  if (nk < 16) return 0;
  // rows/cols covered by one CTA tile: 128 x bn. Worst case over all M' <= M: min(ctas, 95) tiles x 8 splits.
  const long long tiles = ctas < 95 ? ctas : 95;
  return (size_t)(8 * tiles * kTcBM * bn);
}

int tc_gemm(const float* A, const float* Bp, float* C, int M, int N, int K, const Epilogue& ep, cudaStream_t stream,
            float* split_ws, const float* A2, int K1) {
  if (M <= 0 || N <= 0) return D3F_OK;
  D3F_REQUIRE(tc_gemm_supported(A, K), D3F_ERR_INVALID, "tc_gemm: needs K %% 4 == 0 and 16-byte aligned A");
  if (A2 != nullptr)
    D3F_REQUIRE(K1 > 0 && K1 < K && K1 % kTcBK == 0 && tc_gemm_supported(A2, K - K1), D3F_ERR_INVALID,
                "tc_gemm: split A operand needs K1 %% %d == 0 and a 16-byte aligned second matrix", kTcBK);
  int bn = tc_block_n(N);
  // skinny-K, huge-M GEMMs (the level-0/1 unary convolutions) are bound by per-CTA fixed costs and the C write:
  // 64-wide column tiles let two CTAs share an SM and overlap each other's load / MMA / epilogue phases. The packed
  // image is the same (Npad is a multiple of 128, hence of 64).
  if (bn == 128 && K <= 256 && M >= 8192) bn = 64;
  const int splits = split_ws != nullptr ? tc_gemm_splits(M, N, K) : 1;
  // the streaming variant: enough row tiles to keep one persistent CTA per SM busy for several tiles
  const bool stream_ok = env_int("D3F_TC_STREAM", 0) != 0;          // read per call: tests switch it on and off
  const int stream_min_nk = env_int("D3F_TC_STREAM_MIN_CHUNKS", 8);
  if (stream_ok && bn <= 64 && splits <= 1 && (long long)ceil_div(M, kTcBM) * (tc_padded_n(N) / bn) >= 2ll * kNumSMs &&
      K <= 1024 && tc_padded_k(K) / kTcBK >= stream_min_nk) {
    if (bn == 64) return launch_tc_stream<64>(A, A2, K1, Bp, C, M, N, K, ep, stream);
    return launch_tc_stream<32>(A, A2, K1, Bp, C, M, N, K, ep, stream);
  }
  // D3F_TC_A_SMEM=1: the A operand through shared memory (both split images), for A/B timing of the two paths
  if (env_int("D3F_TC_A_SMEM", 0) != 0) {
    switch (bn) {
      case 128: return launch_tc<128, true>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
      case 64: return launch_tc<64, true>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
      default: return launch_tc<32, true>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
    }
  }
  switch (bn) {
    case 128: return launch_tc<128, false>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
    case 64: return launch_tc<64, false>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
    default: return launch_tc<32, false>(A, A2, K1, Bp, C, M, N, K, ep, stream, splits, split_ws);
  }
}

}  // namespace d3f
