// tcgen05 / TMEM / TMA weight-gradient GEMM:  D[N1,N2] (+)= sum_m A[m,N1] * B[m,N2]   (bf16 or split bf16 pairs in, fp32 out)
//
// Split pairs (NFDPM_BF16X2, the fp32-faithful mode): the kernel runs on the operands' bf16 columns (2 per logical column,
// groups of [32 hi | 32 lo]), so the accumulator tile holds, for every logical (n1, n2), the four partial products
// hi*hi, hi*lo, lo*hi, lo*lo at (row, row + 32) x (column, column + 32) of its group; the in-kernel slab reduction adds the
// four (their sum is the exact product of the represented values hi + lo) while it sums the split-M slabs.
//
// Both operands are read straight from their row-major activation layouts ([M, ld], channel fastest): the reduction
// index m is the STRIDED dimension, i.e. both UMMA operands are "MN-major".  No transposed copies are made:
//   TMA     box = 64 columns (128 bytes) x 64 rows of m, 128B swizzle -> smem rows of 128 bytes, one per m
//   UMMA    shared-memory descriptors in MN-major SWIZZLE_128B form: 64 contiguous MN elements per row,
//           8-row (K) groups 1024 bytes apart (SBO), 64-column MN chunks one TMA box apart (LBO);
//           instruction descriptor with the A/B "major" bits set (transpose), M=128, N=BN<=256, K=16
// Output tile 128 (N1) x BN (N2); the M reduction is split across CTAs (tiles x splits <= #SMs) and every CTA writes
// its fp32 partial tile to a workspace slab; reduce_rows_kernel sums the slabs in a fixed order (deterministic, no
// float atomics — `torch.use_deterministic_algorithms(True)` stays honest, reference utils.py:45-60).
//   warp 0: TMA producer (4-stage ring) | warp 1: MMA issuer, TMEM owner | warps 2..5: epilogue (TMEM -> global)
#include <stdlib.h>

#include "tc_common.cuh"

namespace nfdpm {

constexpr int TN_BK = 64;                       // rows of m per pipeline stage
constexpr int TN_STAGES = 4;
constexpr int TN_A_BYTES = 2 * TN_BK * 128;     // two 64-column boxes (N1 tile = 128)
constexpr int TN_B_BYTES_MAX = 4 * TN_BK * 128; // up to four 64-column boxes (BN <= 256)
constexpr int TN_STAGE_BYTES = TN_A_BYTES + TN_B_BYTES_MAX;
constexpr int TN_THREADS = 64 + 128;

// MN-major, SWIZZLE_128B: LBO = bytes between 64-element MN chunks (one TMA box), SBO = 1024 (8 k-rows of 128 B)
__device__ __forceinline__ uint64_t make_smem_desc_mn(uint32_t saddr) {
  return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((TN_BK * 128) >> 4) << 16) | (64ull << 32) | (1ull << 46) |
         (2ull << 61);
}
__device__ __forceinline__ uint32_t make_idesc_mn(int M, int N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// One item of the split reduction: logical output row n1, columns n2..n2+3 (row rr / column cc of tile (t1, t2)), summed
// over the `splits` slabs of ws in slab order (split pairs: then hh, hl, lh, ll) and stored in the output's layout.
__device__ __forceinline__ void tn_reduce_item(const float* __restrict__ ws, float* __restrict__ D, int n1, int n2, int t1,
                                               int rr, int t2, int cc, int BN, int N2, int64_t slab, int splits, int x3,
                                               int out_mode, int out_c, int N2L, int accumulate) {
  int tap = 0, co = 0;
  if (out_mode == NFDPM_TN_OUT_TAPS) {              // n1 = tap*out_c + co  ->  [co][n2][tap]  (ZeroConv weight)
    tap = n1 / out_c;
    co = n1 - tap * out_c;
    if (tap >= 9) return;
  } else if (out_mode == NFDPM_TN_OUT_STRIP && n2 >= out_c) {   // keep the first out_c columns
    return;
  }
  // accumulator coordinates of the (hi, hi) entry; the other three components sit 32 rows / columns further
  const int mrow = x3 ? t1 * 128 + ((rr >> 5) << 6) + (rr & 31) : n1;
  const int mcol = x3 ? t2 * BN + ((cc >> 5) << 6) + (cc & 31) : n2;
  const float* src = ws + (int64_t)mrow * N2 + mcol;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (x3) {
    for (int s2 = 0; s2 < splits; ++s2) {            // slab order, then hh, hl, lh, ll: fixed => bitwise reproducible
      const float* p = src + s2 * slab;
      const float4 v0 = __ldcg(reinterpret_cast<const float4*>(p));
      const float4 v1 = __ldcg(reinterpret_cast<const float4*>(p + 32));
      const float4 v2 = __ldcg(reinterpret_cast<const float4*>(p + 32 * (int64_t)N2));
      const float4 v3 = __ldcg(reinterpret_cast<const float4*>(p + 32 * (int64_t)N2 + 32));
      acc.x += ((v0.x + v1.x) + v2.x) + v3.x;
      acc.y += ((v0.y + v1.y) + v2.y) + v3.y;
      acc.z += ((v0.z + v1.z) + v2.z) + v3.z;
      acc.w += ((v0.w + v1.w) + v2.w) + v3.w;
    }
  } else {
    int s2 = 0;
    for (; s2 + 4 <= splits; s2 += 4) {              // four slab loads in flight, added in slab order
      float4 v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) v[j] = __ldcg(reinterpret_cast<const float4*>(src + (s2 + j) * slab));
#pragma unroll
      for (int j = 0; j < 4; ++j) { acc.x += v[j].x; acc.y += v[j].y; acc.z += v[j].z; acc.w += v[j].w; }
    }
    for (; s2 < splits; ++s2) {
      const float4 v = __ldcg(reinterpret_cast<const float4*>(src + s2 * slab));
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  if (out_mode == NFDPM_TN_OUT_PLAIN) {
    float4* d = reinterpret_cast<float4*>(D + (int64_t)n1 * N2L + n2);
    if (accumulate) {
      const float4 o = *d;
      acc.x += o.x; acc.y += o.y; acc.z += o.z; acc.w += o.w;
    }
    *d = acc;
  } else {
    // layout-changing outputs (the weight tensors' own layouts): four scalar stores
    const float av[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int64_t o;
      if (out_mode == NFDPM_TN_OUT_TAPS) {
        o = ((int64_t)co * N2L + n2 + j) * 9 + tap;
      } else {
        if (n2 + j >= out_c) break;
        o = (int64_t)n1 * out_c + n2 + j;
      }
      D[o] = accumulate ? D[o] + av[j] : av[j];
    }
  }
}

__global__ void __launch_bounds__(TN_THREADS, 1) gemm_tn_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                   const __grid_constant__ CUtensorMap tmB,
                                                                   float* __restrict__ ws, int M, int N1, int N2, int BN,
                                                                   int num_n2, int splits, int kb_per_split,
                                                                   float* __restrict__ D, int accumulate,
                                                                   int* __restrict__ counters, int out_mode, int out_c,
                                                                   int x3, int N1L, int N2L) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * TN_STAGES + 1];
  __shared__ uint32_t s_tmem_base;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t bar_full = smem_u32(&bars[0]), bar_empty = smem_u32(&bars[TN_STAGES]);
  const uint32_t bar_done = smem_u32(&bars[2 * TN_STAGES]);

  const int tile = blockIdx.x / splits, split = blockIdx.x - tile * splits;
  const int t1 = tile / num_n2, t2 = tile - t1 * num_n2;
  const int num_kb = (M + TN_BK - 1) / TN_BK;
  const int kb0 = split * kb_per_split;
  const int kb1 = min(num_kb, kb0 + kb_per_split);
  const int nb_boxes = BN >> 6;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < TN_STAGES; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&s_tmem_base), 256);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;

  if (warp == 0) {
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx_bytes = (uint32_t)(TN_A_BYTES + nb_boxes * TN_BK * 128);
    for (int kb = kb0; kb < kb1; ++kb) {
      mbar_wait(bar_empty + 8 * stage, phase ^ 1);
      if (lane == 0) {
        const uint32_t sa = ring + stage * TN_STAGE_BYTES, sb = sa + TN_A_BYTES;
        mbar_arrive_expect_tx(bar_full + 8 * stage, tx_bytes);
        for (int j = 0; j < 2; ++j)
          tma_load_2d(sa + j * (TN_BK * 128), &tmA, t1 * 128 + j * 64, kb * TN_BK, bar_full + 8 * stage);
        for (int j = 0; j < nb_boxes; ++j)
          tma_load_2d(sb + j * (TN_BK * 128), &tmB, t2 * BN + j * 64, kb * TN_BK, bar_full + 8 * stage);
      }
      __syncwarp();
      if (++stage == TN_STAGES) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t idesc = make_idesc_mn(128, BN);
    for (int kb = kb0; kb < kb1; ++kb) {
      mbar_wait(bar_full + 8 * stage, phase);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t sa = ring + stage * TN_STAGE_BYTES, sb = sa + TN_A_BYTES;
        const uint64_t adesc = make_smem_desc_mn(sa), bdesc = make_smem_desc_mn(sb);
#pragma unroll
        for (int k = 0; k < TN_BK / 16; ++k)            // 16 k-rows = 2048 bytes = 128 descriptor units
          umma_bf16(tmem_base, adesc + 128 * k, bdesc + 128 * k, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
        umma_commit(bar_empty + 8 * stage);
        if (kb == kb1 - 1) umma_commit(bar_done);
      }
      __syncwarp();
      if (++stage == TN_STAGES) { stage = 0; phase ^= 1; }
    }
  } else {
    // epilogue: TMEM lane = row of the tile = n1 index
    const int q = warp & 3;
    const int n1 = t1 * 128 + q * 32 + lane;
    float* dst = ws + ((int64_t)split * N1 + n1) * N2 + t2 * BN;
    const bool have = kb1 > kb0;                           // an empty split (tail) contributes zeros
    if (have) {
      mbar_wait(bar_done, 0);
      tc_fence_after();
    }
    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
    for (int c0 = 0; c0 < BN; c0 += 16) {
      uint32_t r[16];
      if (have) {
        tmem_ld16(taddr + c0, r);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) r[j] = 0u;
      }
      if (n1 < N1 && t2 * BN + c0 < N2) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(dst + c0 + 4 * j) =
              make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                          __uint_as_float(r[4 * j + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 256);
  }
  if (counters == nullptr) return;          // the caller reduces the slabs with a separate kernel

  // ---- in-kernel split reduction.  All CTAs of the grid are co-resident (grid <= #SMs, one CTA per SM), so the
  // CTAs of a tile can wait for each other: publish the slab, wait until all `splits` slabs of the tile exist, then
  // every CTA sums a band of the tile's rows over the slabs IN SLAB ORDER (deterministic) straight into D.
  int* arrive = counters + 2 * tile;
  int* done = arrive + 1;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    atomicAdd(arrive, 1);
    const uint64_t t0 = global_timer_ns();
    while (atomicAdd(arrive, 0) < splits) {
      __nanosleep(64);
      if (global_timer_ns() - t0 > 2000000000ull) __trap();
    }
    __threadfence();
  }
  __syncthreads();
  // logical geometry of the tile: with split pairs 128 accumulator rows / BN columns are 64 / BN/2 logical ones
  const int RL = x3 ? 64 : 128, CL = x3 ? (BN >> 1) : BN;
  const int band = (RL + splits - 1) / splits;
  const int r_lo = split * band;
  const int r_hi = min(min(RL, r_lo + band), N1L - t1 * RL);      // logical rows of this CTA's band that exist
  const int cols = min(CL, N2L - t2 * CL);
  const int64_t slab = (int64_t)N1 * N2;
  if (r_hi > r_lo && cols > 0) {
    const int c4 = cols >> 2, n_items = (r_hi - r_lo) * c4;
    for (int it = threadIdx.x; it < n_items; it += TN_THREADS) {
      const int r = it / c4, c = it - r * c4;
      const int rr = r_lo + r, cc = 4 * c;
      tn_reduce_item(ws, D, t1 * RL + rr, t2 * CL + cc, t1, rr, t2, cc, BN, N2, slab, splits, x3, out_mode, out_c, N2L,
                     accumulate);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (atomicAdd(done, 1) == splits - 1) {    // last CTA of the tile: re-arm the counters for the next launch
      *arrive = 0;
      *done = 0;
      __threadfence();
    }
  }
}

// The split reduction of gemm_tn_tc_kernel as a kernel of its own, for grids whose CTAs are not all co-resident (more
// tiles x splits than SMs, e.g. the split-pair weight gradients of the ZeroConv and the first coupling conv at levels
// wider than ~260 channels): the same items, the same slab order, hence the same bits as the in-kernel reduction.
__global__ void __launch_bounds__(256) gemm_tn_reduce_kernel(const float* __restrict__ ws, float* __restrict__ D, int N1L,
                                                             int N2L, int N2, int BN, int64_t slab, int splits, int x3,
                                                             int out_mode, int out_c, int accumulate) {
  const int RL = x3 ? 64 : 128, CL = x3 ? (BN >> 1) : BN, c4 = N2L >> 2;
  const int64_t n_items = (int64_t)N1L * c4;
  for (int64_t it = (int64_t)blockIdx.x * 256 + threadIdx.x; it < n_items; it += (int64_t)gridDim.x * 256) {
    const int n1 = (int)(it / c4), n2 = (int)(it - (int64_t)n1 * c4) * 4;
    const int t1 = n1 / RL, t2 = n2 / CL;
    tn_reduce_item(ws, D, n1, n2, t1, n1 - t1 * RL, t2, n2 - t2 * CL, BN, N2, slab, splits, x3, out_mode, out_c, N2L,
                   accumulate);
  }
}

static int sm_count() {
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
      sms = 148;
  }
  return sms;
}

// tiling shared by the launcher and the workspace query
void gemm_tn_tc_plan(int M, int N1, int N2, int* BN, int* tiles, int* splits, int* kb_per_split) {
  const int bn = N2 >= 256 ? 256 : (N2 + 63) / 64 * 64;
  const int n2t = (N2 + bn - 1) / bn, n1t = (N1 + 127) / 128;
  const int t = n1t * n2t;
  const int num_kb = (M + TN_BK - 1) / TN_BK;
  // split the M reduction over the SMs, but keep >= 16 k-blocks (1024 rows) per CTA: below that the slab traffic and
  // the wait of the in-kernel reduction cost more than the parallelism buys (measured: 17-25 us at M = 2048 with 18 splits)
  static int min_kb = -1;
  if (min_kb < 0) {
    const char* e = getenv("NFDPM_TN_MIN_KB");
    min_kb = e ? atoi(e) : 1;
    if (min_kb < 1) min_kb = 1;
  }
  int s = sm_count() / t;
  if (s < 1) s = 1;
  if (s > num_kb / min_kb) s = num_kb / min_kb;
  if (s < 1) s = 1;
  const int per = (num_kb + s - 1) / s;
  s = (num_kb + per - 1) / per;
  *BN = bn; *tiles = t; *splits = s; *kb_per_split = per;
}

bool gemm_tn_tc_ok(const void* A, int64_t lda, const void* Bm, int64_t ldb, int N1, int N2) {
  return (lda % 8 == 0) && (ldb % 8 == 0) && (N2 % 16 == 0) && (N2 % 4 == 0) && ((uintptr_t)A % 16 == 0) &&
         ((uintptr_t)Bm % 16 == 0) && N1 > 0;
}

// x3: A and Bm are split bf16 pairs (lda / ldb / N1 / N2 count logical columns; a row is 2 x ld bf16)
int gemm_tn_tc(const void* A, int64_t lda, const void* Bm, int64_t ldb, float* ws, int M, int N1L, int N2L, int* splits_out,
               float* D, int accumulate, int* counters, int out_mode, int out_c, int x3, cudaStream_t st) {
  // the kernel's own dimensions: bf16 columns of the operands (whole groups of 64 for split pairs)
  const int N1 = x3 ? 2 * ((N1L + 31) / 32 * 32) : N1L, N2 = x3 ? 2 * ((N2L + 31) / 32 * 32) : N2L;
  const int kmul = x3 ? 2 : 1;
  int BN, tiles, splits, per;
  gemm_tn_tc_plan(M, N1, N2, &BN, &tiles, &splits, &per);
  const int num_n2 = (N2 + BN - 1) / BN;
  // the tensor maps cover the physical row width (lda / ldb): padding columns inside it are real memory, columns
  // beyond it and rows >= M are zero-filled by TMA
  CUtensorMap tmA, tmB;
  if (make_map(&tmA, A, M, lda * kmul, lda * kmul, TN_BK)) return 1;
  if (make_map(&tmB, Bm, M, ldb * kmul, ldb * kmul, TN_BK)) return 1;
  static bool attr_set = false;
  const size_t smem = 1024 + (size_t)TN_STAGES * TN_STAGE_BYTES;
  if (!attr_set) {
    NFDPM_CUDA(cudaFuncSetAttribute(gemm_tn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_set = true;
  }
  NFDPM_REQUIRE((out_mode == NFDPM_TN_OUT_PLAIN && !x3) || counters != nullptr,
                "nfdpm_gemm_tn: layout-changing outputs and split-pair operands need the in-kernel reduction (counters)");
  const bool coresident = !(tiles > 500 || tiles * splits > sm_count());
  if (!coresident && (out_mode != NFDPM_TN_OUT_PLAIN || x3)) {
    // slabs to ws, then the same reduction as a separate kernel (plain fp32 / bf16 outputs keep reduce_rows_kernel)
    gemm_tn_tc_kernel<<<tiles * splits, TN_THREADS, smem, st>>>(tmA, tmB, ws, M, N1, N2, BN, num_n2, splits, per, D,
                                                               accumulate, nullptr, out_mode, out_c, x3, N1L, N2L);
    NFDPM_CHECK_LAUNCH("gemm_tn_tc_kernel");
    const int64_t items = (int64_t)N1L * (N2L >> 2);
    const int64_t g = (items + 255) / 256;
    gemm_tn_reduce_kernel<<<(int)(g < 148 * 8 ? g : 148 * 8), 256, 0, st>>>(ws, D, N1L, N2L, N2, BN, (int64_t)N1 * N2,
                                                                            splits, x3, out_mode, out_c, accumulate);
    NFDPM_CHECK_LAUNCH("gemm_tn_reduce_kernel");
    *splits_out = 0;
    return 0;
  }
  if (!coresident) counters = nullptr;     // co-residency not guaranteed: reduce separately
  gemm_tn_tc_kernel<<<tiles * splits, TN_THREADS, smem, st>>>(tmA, tmB, ws, M, N1, N2, BN, num_n2, splits, per, D,
                                                             accumulate, counters, out_mode, out_c, x3, N1L, N2L);
  NFDPM_CHECK_LAUNCH("gemm_tn_tc_kernel");
  *splits_out = counters != nullptr ? 0 : splits;     // 0: already reduced into D
  return 0;
}

}  // namespace nfdpm
