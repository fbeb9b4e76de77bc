// tcgen05 / TMEM / TMA GEMM for the coupling networks:  D[M,N] = epilogue(A[M,K] * Bw[N,K]^T)
//   A  [M,K] row-major (pixel-major activations), Bw [N,K] row-major (packed conv weights), fp32 accumulation in tensor
//   memory.  Operands are bf16 (NFDPM_BF16: one tcgen05.mma per K=16 slice, 2^-9 operand rounding) or SPLIT bf16 pairs
//   (NFDPM_BF16X2, common.cuh: v = hi + lo, three tcgen05.mma per slice pair, 2^-17 — the fp32-faithful mode that meets the
//   reference's 1e-4 parity bar on the tensor cores).  Output fp32, bf16 or split pairs (the next GEMM's A operand).
//
// Persistent, warp-specialised CTA (one per SM, 64 + 32 * TCG_EPI_WARPS = 576 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 2D loads of a 128x64 A box and a BNx64 B box (128B swizzle)
//               into a shared-memory ring (TcPlan: 3 x 48 KB stages, or as many 16 KB + BN x 128 B stages as fit - 4 at
//               BN = 256 - for multi-tile K >= 256 shapes), completion on mbarriers
//   warp 1      MMA issuer: one lane issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) x4 per stage,
//               tcgen05.commit releases the smem stage / publishes the accumulator; also owns TMEM alloc/dealloc
//   warps 2..17 epilogue (four per TMEM lane quadrant): software-pipelined tcgen05.ld (32x32b.x16) of the accumulator
//               quadrant, fused ActNorm+ReLU as one FMA + max per element (utils.py:69,84-87), convert, conflict-free
//               16-byte stores into a 128B-swizzled staging buffer, then ONE thread issues cp.async.bulk.tensor stores
//               (full 128-byte lines; r1 profile: per-thread row-strided global stores capped output at 2.3 TB/s).  The
//               staging buffer holds the whole tile (classic plan) or one 64-column pass (deep plan).
//               Two TMEM accumulator stages (2 x 256 columns) let the epilogue of tile i overlap the main loop of
//               tile i+1.  (r1 profile: with 4 epilogue warps and scalar parameter loads the kernel was
//               issue-bound in the epilogue at 30% tensor-pipe activity.)
// Tiles are scheduled by tc_sched.h (persistent stride + half-width tiles in the last round when that balances it).
// BN (<= 256, multiple of 16) is a runtime value: it only enters through the B tensor map box, the expected
// transaction bytes and the instruction descriptor.
//
// Every mbarrier wait is bounded (2 s on %globaltimer) and traps instead of hanging the GPU.
#include <stdlib.h>

#include "tc_common.cuh"
#include "tc_sched.h"

namespace nfdpm {

// Epilogue warps of THIS kernel: four per TMEM lane quadrant.  ncu r1 (source page): with two per quadrant the 8 epilogue
// warps were busy ~73 % of the kernel (IPC 0.9/SM, latency-bound on tcgen05.ld -> FFMA -> F2FP -> STS chains) and the
// tensor pipe idled at 41 % waiting for a drained accumulator stage: the kernel was EPILOGUE-bound, not operand-bound
// (which is why the cta_group::2 variant, gemm_tc2.cu, did not help).  More warps = more chains in flight.
constexpr int TCG_EPI_WARPS = 16;
constexpr int TCG_EPQ = TCG_EPI_WARPS / 4;            // epilogue warps per quadrant = chunk stride
constexpr int TC_THREADS = 64 + 32 * TCG_EPI_WARPS;
__device__ __forceinline__ void epi_barrier_g() { asm volatile("bar.sync 1, %0;" ::"n"(32 * TCG_EPI_WARPS) : "memory"); }
constexpr int TC_ACC_COLS = 256;     // TMEM columns per accumulator stage

// persistent tile schedule (tc_sched.h: shared with the host-side unit test)
__device__ __forceinline__ bool tc_work(int it, int num_tiles, int num_n, int BN, int split, TcWork& w) {
  return tc_work_for((int)blockIdx.x, (int)gridDim.x, it, num_tiles, num_n, BN, split, w);
}

// Shared-memory plan chosen by the host: TcPlan (tc_sched.h)

// profiling hook (nfdpm_gemm_debug): per-CTA cycle counters [grid][16] int64; NULL = off
__device__ long long* g_tc_dbg = nullptr;

template <int EPI, typename OutT, bool X3>
__global__ void __launch_bounds__(TC_THREADS, 1) gemm_nt_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                   const __grid_constant__ CUtensorMap tmB,
                                                                   const __grid_constant__ CUtensorMap tmD, int M, int N, int K,
                                                                   int BN, int split, const TcPlan plan,
                                                                   const float* __restrict__ ep_scale,
                                                                   const float* __restrict__ ep_bias) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * TC_MAX_STAGES + 4];
  __shared__ uint32_t s_tmem_base;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // 1024-byte aligned tile ring (swizzle-128B requirement), then the epilogue parameters
  const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int n_stages = plan.n_stages;
  const uint32_t stage_bytes = (uint32_t)plan.stage_bytes;
  const uint32_t cstage = ring + n_stages * stage_bytes;               // 1024-aligned output staging tile
  float* s_ep = reinterpret_cast<float*>(smem_raw + (ring - smem_u32(smem_raw)) + n_stages * stage_bytes + plan.cstage_bytes);
  const uint32_t bar_full = smem_u32(&bars[0]), bar_empty = smem_u32(&bars[TC_MAX_STAGES]);
  const uint32_t bar_tfull = smem_u32(&bars[2 * TC_MAX_STAGES]), bar_tempty = smem_u32(&bars[2 * TC_MAX_STAGES + 2]);

  const int num_n = (N + BN - 1) / BN;
  const int num_m = (M + TC_BM - 1) / TC_BM;
  const int num_tiles = num_m * num_n;
  const int num_kb = K / TC_BK;          // K counts bf16 columns of the operand rows (2 x logical K for split pairs)

  const int n_pad = num_n * BN;        // columns covered by the tiles (>= N); parameters are zero beyond N
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    tma_prefetch_desc(&tmD);
    for (int s = 0; s < n_stages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_tfull + 8 * a, 1);
      mbar_init(bar_tempty + 8 * a, 32 * TCG_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&s_tmem_base), 512);
  tc_fence_before();
  __syncthreads();                     // barriers initialised, tensor memory allocated
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;
  // everything above overlaps the tail of the previous kernel in the stream (PDL); global memory is touched below
  const long long t_entry = clock64();
  const unsigned long long g_entry = global_timer_ns();
  pdl_trigger();
  pdl_wait();
  const long long t_dep = clock64();
  long long* const dbg = g_tc_dbg;
  long long w0 = 0, w1 = 0, w2 = 0, w3 = 0, w4 = 0;       // wait / work cycle counters of this warp (profiling hook)
  const long long t_start = clock64();
  if (warp >= 2 && EPI != NFDPM_EPI_RAW) {
    // the epilogue warps stage the folded ActNorm parameters while the producer / MMA warps already run the main loop
    // (r1 counters: staging them with all warps in front of the role split cost 0.6 us per launch)
    for (int i = threadIdx.x - 64; i < n_pad; i += 32 * TCG_EPI_WARPS) {
      const float e = (i < N) ? expf(ep_scale[i]) : 0.f;
      s_ep[i] = e;                                   // y = max(0, e*acc + e*b)
      if (EPI == NFDPM_EPI_ACTNORM_RELU) s_ep[n_pad + i] = (i < N) ? e * ep_bias[i] : 0.f;
    }
    epi_barrier_g();
  }

  if (warp == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    TcWork wk;
    for (int it = 0; tc_work(it, num_tiles, num_n, BN, split, wk); ++it) {
      const int m_blk = wk.m_blk;
      const uint32_t tx_bytes = (uint32_t)(TC_A_BYTES + wk.bn * TC_BK * 2);
      const bool two_b = split && wk.bn == BN;            // split mode: the B box holds BN/2 rows
      for (int kb = 0; kb < num_kb; ++kb) {
        const long long c0 = dbg ? clock64() : 0;
        mbar_wait(bar_empty + 8 * stage, phase ^ 1);
        if (dbg) w0 += clock64() - c0;
        if (lane == 0) {
          const uint32_t sa = ring + stage * stage_bytes, sb = sa + TC_A_BYTES;
          mbar_arrive_expect_tx(bar_full + 8 * stage, tx_bytes);
          tma_load_2d(sa, &tmA, kb * TC_BK, m_blk * TC_BM, bar_full + 8 * stage);
          tma_load_2d(sb, &tmB, kb * TC_BK, wk.n0, bar_full + 8 * stage);
          if (two_b) tma_load_2d(sb + (uint32_t)(BN >> 1) * TC_BK * 2, &tmB, kb * TC_BK, wk.n0 + (BN >> 1), bar_full + 8 * stage);
        }
        __syncwarp();
        if (++stage == n_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    TcWork wk;
    for (int it = 0; tc_work(it, num_tiles, num_n, BN, split, wk); ++it) {
      const uint32_t idesc = make_idesc(TC_BM, wk.bn);
      const long long c0 = dbg ? clock64() : 0;
      mbar_wait(bar_tempty + 8 * acc, acc_phase ^ 1);     // epilogue has drained this accumulator stage
      if (dbg) w1 += clock64() - c0;
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + acc * TC_ACC_COLS;
      for (int kb = 0; kb < num_kb; ++kb) {
        const long long c1 = dbg ? clock64() : 0;
        mbar_wait(bar_full + 8 * stage, phase);           // TMA bytes have landed
        if (dbg) w0 += clock64() - c1;
        tc_fence_after();
        if (lane == 0) {
          const uint32_t sa = ring + stage * stage_bytes, sb = sa + TC_A_BYTES;
          const uint64_t adesc = make_smem_desc(sa), bdesc = make_smem_desc(sb);
          umma_stage<X3>(tmem_d, adesc, bdesc, idesc, kb == 0);
          umma_commit(bar_empty + 8 * stage);             // smem stage reusable once these MMAs retire
          if (kb == num_kb - 1) umma_commit(bar_tfull + 8 * acc);   // accumulator complete
        }
        __syncwarp();
        if (++stage == n_stages) { stage = 0; phase ^= 1; }
      }
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
  } else {
    // ===================== epilogue (warps 2..17) =====================
    const int q = warp & 3;                               // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;                     // which of the TCG_EPQ warps of the quadrant
    int acc = 0;
    uint32_t acc_phase = 0;
    TcWork wk;
    for (int it = 0; tc_work(it, num_tiles, num_n, BN, split, wk); ++it) {
      const int m_blk = wk.m_blk, n_base = wk.n0, n_chunks = wk.bn >> 4;
      const long long c0 = dbg ? clock64() : 0;
      mbar_wait(bar_tfull + 8 * acc, acc_phase);
      tc_fence_after();
      const long long c1 = dbg ? clock64() : 0;
      w0 += c1 - c0;
      const int trow = q * 32 + lane;                      // row inside the tile == TMEM lane
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + acc * TC_ACC_COLS;
      const long long c2 = dbg ? clock64() : 0;
      w1 += c2 - c1;
      auto process = [&](const uint32_t (&r)[16], int c0, int c_stage) {
        const int n0 = n_base + c0;
        float v[16];
        if (EPI == NFDPM_EPI_ACTNORM_RELU) {
          const float4* pe = reinterpret_cast<const float4*>(s_ep + n0);
          const float4* pb = reinterpret_cast<const float4*>(s_ep + n_pad + n0);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 e = pe[j], b = pb[j];
            v[4 * j + 0] = fmaxf(0.f, fmaf(__uint_as_float(r[4 * j + 0]), e.x, b.x));
            v[4 * j + 1] = fmaxf(0.f, fmaf(__uint_as_float(r[4 * j + 1]), e.y, b.y));
            v[4 * j + 2] = fmaxf(0.f, fmaf(__uint_as_float(r[4 * j + 2]), e.z, b.z));
            v[4 * j + 3] = fmaxf(0.f, fmaf(__uint_as_float(r[4 * j + 3]), e.w, b.w));
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
        }
        TcStage<OutT>::put16(cstage, trow, c_stage, v);
      };
      // This warp owns chunks half, half + TCG_EPQ, ... (16 columns each); the TMEM load of its next chunk is in flight
      // while the current one is processed.  The chunks are written to the staging buffer in PASSES of cpw chunks per
      // warp (= cpw * 64 columns): [staging free] -> convert -> [fence, barrier] -> one thread issues the pass's TMA box
      // stores.  Classic plan: one pass = the whole tile; deep plan: cpw = 1, one 64-column box group per pass.
      constexpr int CPB = TcStage<OutT>::kColsPerBox;
      const int cpw = plan.cpw;
      const int k_total = ((n_chunks + TCG_EPQ - 1) / TCG_EPQ + cpw - 1) / cpw * cpw;   // same trip count for every warp
      auto chunk_step = [&](uint32_t (&cur)[16], uint32_t (&nxt)[16], int k) {
        const int ch = half + TCG_EPQ * k;
        const int pass = k / cpw;
        const int col0 = pass * cpw * (16 * TCG_EPQ);        // first tile column of this pass
        if (k - pass * cpw == 0) {
          // the previous pass's (or tile's) TMA stores must have finished READING the staging buffer
          if (warp == 2 && lane == 0) tma_store_wait_read();
          epi_barrier_g();
        }
        if (ch < n_chunks) {
          tmem_ld_wait();
          if (ch + TCG_EPQ < n_chunks) tmem_ld16(taddr + (ch + TCG_EPQ) * 16, nxt);
          process(cur, ch * 16, ch * 16 - col0);
        }
        if (k - pass * cpw == cpw - 1) {
          if (k == k_total - 1) {
            // accumulator drained: hand the TMEM stage back to the MMA warp before doing the stores
            tc_fence_before();
            mbar_arrive(bar_tempty + 8 * acc);
          }
          fence_proxy_async();                             // generic-proxy smem writes -> visible to the TMA engine
          epi_barrier_g();
          if (warp == 2 && lane == 0) {
            const int cols = min(wk.bn - col0, cpw * (16 * TCG_EPQ));
            const int n_boxes = (cols + CPB - 1) / CPB;
            for (int j = 0; j < n_boxes; ++j)              // rows >= M and columns >= N are clipped by the tensor map
              tma_store_2d(&tmD, cstage + (uint32_t)j * 16384u, (n_base + col0 + j * CPB) * TcMemCols<OutT>::v, m_blk * TC_BM);
            tma_store_commit();
          }
        }
      };
      uint32_t ra[16], rb[16];
      if (half < n_chunks) tmem_ld16(taddr + half * 16, ra);
      for (int k = 0; k < k_total; k += 2) {
        chunk_step(ra, rb, k);
        if (k + 1 < k_total) chunk_step(rb, ra, k + 1);
      }
      const long long c3 = dbg ? clock64() : 0;
      w2 += c3 - c2;
      if (dbg) w4 += 1;
      acc ^= 1;
      if (acc == 0) acc_phase ^= 1;
    }
    // the staging tile must have been READ before the CTA gives its shared memory back; the writes themselves are
    // complete and visible to the next kernel at grid completion (what griddepcontrol.wait / stream order wait for)
    if (warp == 2 && lane == 0) tma_store_wait_read();
  }
  if (dbg != nullptr && lane == 0 && warp <= 2) {
    long long* o = dbg + (int64_t)blockIdx.x * 16;
    const long long total = clock64() - t_start;
    if (warp == 0) { o[0] = total; o[1] = w0; }                       // producer: cycles waiting for a free smem stage
    if (warp == 1) { o[2] = total; o[3] = w0; o[4] = w1; }            // MMA: waiting for TMA bytes / for a drained accumulator
    if (warp == 2) { o[5] = total; o[6] = w0; o[7] = w1; o[8] = w2; o[9] = w3; o[10] = w4; }   // epilogue: wait tfull /
                                                                      // wait staging free / TMEM->smem / barrier / tiles
    if (warp == 2) {                                                  // CTA lifetime: entry -> dependency resolved -> roles start -> end
      o[11] = t_dep - t_entry; o[12] = t_start - t_dep; o[13] = (long long)g_entry; o[14] = (long long)global_timer_ns();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ---------------------------------------------------------------- host side
template <int EPI, typename OutT, bool X3>
static int launch_tc(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD, int M, int N, int Kmem, int BN,
                     int split, const TcPlan& plan, const float* es, const float* eb, int grid, size_t smem, cudaStream_t st) {
  static bool attr_set = false;
  if (!attr_set) {
    NFDPM_CUDA(cudaFuncSetAttribute(gemm_nt_tc_kernel<EPI, OutT, X3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    TC_SMEM_MAX));
    attr_set = true;
  }
  NFDPM_CUDA(launch_pdl(gemm_nt_tc_kernel<EPI, OutT, X3>, dim3(grid), dim3(TC_THREADS), smem, st, tmA, tmB, tmD, M, N, Kmem,
                        BN, split, plan, es, eb));
  return 0;
}

// lda / ldb / ldd and K count LOGICAL elements; a split-pair row occupies 2 x ld bf16.
int gemm_nt_tc(const void* A, int64_t lda, const void* Bw, int64_t ldb, void* D, int64_t ldd, int M, int N, int K,
               int in_dtype, int out_dtype, int epilogue, const float* ep_scale, const float* ep_bias, cudaStream_t st) {
  const bool x3 = in_dtype == NFDPM_BF16X2, out_x2 = out_dtype == NFDPM_BF16X2;
  NFDPM_REQUIRE(N % 16 == 0, "nfdpm_gemm_nt(tensor core): N=%d must be a multiple of 16", N);
  NFDPM_REQUIRE(!out_x2 || (N % 32 == 0 && ldd % 32 == 0), "nfdpm_gemm_nt: split-pair output needs N and ldd multiples of 32");
  NFDPM_REQUIRE(((uintptr_t)A % 16 == 0) && ((uintptr_t)Bw % 16 == 0) && ((uintptr_t)D % 16 == 0),
                "nfdpm_gemm_nt(tensor core): operands must be 16-byte aligned");
  NFDPM_REQUIRE(epilogue == NFDPM_EPI_RAW || N <= 2048, "nfdpm_gemm_nt(tensor core): fused ActNorm epilogue supports N <= 2048");
  // the plan's knobs (tc_sched.h tc_nt_plan), read once per process
  static int bn_cap = -1, narrow_below = -1, split_on = -1, deep_on = -1, sms = 0;
  if (bn_cap < 0) {
    const char* e = getenv("NFDPM_TC_BN");
    bn_cap = e ? atoi(e) : 256;
    if (bn_cap != 64 && bn_cap != 128) bn_cap = 256;
    e = getenv("NFDPM_TC_NARROW");
    narrow_below = e ? atoi(e) : 74;
    e = getenv("NFDPM_TC_SPLIT");                       // 0 keeps whole tiles in the last round
    split_on = (e && atoi(e) == 0) ? 0 : 1;
    e = getenv("NFDPM_TC_DEEP");                        // 0: classic plan everywhere, 2: deep plan for every shape
    deep_on = e ? atoi(e) : 1;
  }
  if (sms == 0) {
    int dev = 0;
    NFDPM_CUDA(cudaGetDevice(&dev));
    NFDPM_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  }
  const int kmul = x3 ? 2 : 1;                           // bf16 columns per logical K
  const int Kmem = K * kmul;
  const TcNtPlan p = tc_nt_plan(M, N, Kmem, out_dtype == NFDPM_F32, out_dtype == NFDPM_BF16, epilogue != NFDPM_EPI_RAW, sms,
                                bn_cap, narrow_below, split_on, deep_on);
  const int BN = p.BN, split = p.split, grid = p.grid;
  const TcPlan plan = p.plan;
  const size_t smem = (size_t)p.smem;
  CUtensorMap tmA, tmB, tmD;
  if (make_map(&tmA, A, M, Kmem, lda * kmul, TC_BM)) return 1;
  if (make_map(&tmB, Bw, N, Kmem, ldb * kmul, split ? BN / 2 : BN)) return 1;
  if (out_x2) { if (make_map(&tmD, D, M, 2 * (int64_t)N, 2 * ldd, TC_BM)) return 1; }
  else if (make_map(&tmD, D, M, N, ldd, TC_BM, out_dtype == NFDPM_F32)) return 1;
#define GO(EPI, T, X) return launch_tc<EPI, T, X>(tmA, tmB, tmD, M, N, Kmem, BN, split, plan, ep_scale, ep_bias, grid, smem, st)
  const bool raw = epilogue == NFDPM_EPI_RAW;
  if (x3) {
    if (out_dtype == NFDPM_F32) { if (raw) GO(NFDPM_EPI_RAW, float, true); else GO(NFDPM_EPI_ACTNORM_RELU, float, true); }
    if (out_x2) { if (raw) GO(NFDPM_EPI_RAW, bf16x2_t, true); else GO(NFDPM_EPI_ACTNORM_RELU, bf16x2_t, true); }
    return fail("nfdpm_gemm_nt: split-pair operands produce fp32 or split-pair output (out_dtype %d)", out_dtype);
  }
  if (out_dtype == NFDPM_F32) { if (raw) GO(NFDPM_EPI_RAW, float, false); else GO(NFDPM_EPI_ACTNORM_RELU, float, false); }
  if (out_dtype == NFDPM_BF16) { if (raw) GO(NFDPM_EPI_RAW, __nv_bfloat16, false); else GO(NFDPM_EPI_ACTNORM_RELU, __nv_bfloat16, false); }
  return fail("nfdpm_gemm_nt: bf16 operands produce fp32 or bf16 output (out_dtype %d)", out_dtype);
#undef GO
}

}  // namespace nfdpm

// profiling hook: per-CTA cycle counters of nfdpm_gemm_nt's tcgen05 kernel into a device int64 [148][16] buffer (NULL = off)
extern "C" int nfdpm_gemm_debug(void* buf) {
  long long* p = reinterpret_cast<long long*>(buf);
  NFDPM_CUDA(cudaMemcpyToSymbol(nfdpm::g_tc_dbg, &p, sizeof(p)));
  return 0;
}
