// Persistent tile schedule and host launch plan of the tcgen05 GEMM (gemm_tc.cu), as plain functions so that the
// host-side unit test (tests/test_sched_cpu.py, compiled with g++) exercises exactly the code the kernel and launcher run.
//
// One unit of work of a CTA: a BM x bn output tile at column n0.  Every CTA runs the same number of full tiles
// (tile = cta + it * grid); when the tile count is not a multiple of the grid (512 tiles on 148 SMs: 68 CTAs would run a 4th
// tile while 80 idle for a whole tile time), the REMAINING tiles are split into two half-width tiles each and handed to
// 2 * rem CTAs (`split` mode: the B tensor-map box is BN/2 rows, a full tile takes two B loads per stage), so the last wave
// costs half a tile on (almost) every SM instead of a whole tile on some.
#pragma once
#if defined(__CUDACC__)
#define TC_SCHED_HD __host__ __device__ __forceinline__
#else
#define TC_SCHED_HD inline
#endif

namespace nfdpm {

struct TcWork { int m_blk, n0, bn; };

// it-th unit of work of CTA `cta` of `grid`; false when the CTA is done
TC_SCHED_HD bool tc_work_for(int cta, int grid, int it, int num_tiles, int num_n, int BN, int split, TcWork& w) {
  int tile = cta + it * grid, half = -1;
  if (split) {
    const int full_per = num_tiles / grid;
    if (it > full_per) return false;
    if (it == full_per) {
      const int rem = num_tiles - full_per * grid;
      if (cta >= 2 * rem) return false;
      tile = full_per * grid + (cta >> 1);
      half = cta & 1;
    }
  }
  if (tile >= num_tiles) return false;
  w.m_blk = tile / num_n;
  const int n_blk = tile - w.m_blk * num_n;
  w.n0 = n_blk * BN + (half > 0 ? (BN >> 1) : 0);
  w.bn = half >= 0 ? (BN >> 1) : BN;
  return true;
}

// may the last round be split?  (half tiles must be whole 64-column store groups and whole UMMA N steps; every N block full)
TC_SCHED_HD bool tc_split_ok(int tiles, int grid, int BN, int N) {
  const int rem = tiles % grid;
  return tiles > grid && rem > 0 && 2 * rem <= grid && BN % 128 == 0 && N % BN == 0;
}

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;              // 64 bf16 = 128 bytes = one swizzle-128B row
constexpr int TC_STAGES = 3;           // classic layout: 3 x 48 KB ring + a whole-tile (64 KB) output staging buffer
constexpr int TC_MAX_STAGES = 6;       // deep layout: as many (16 KB + BN x 128 B) stages as fit next to a 64-column staging buffer
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;          // 16 KB
constexpr int TC_B_BYTES_MAX = 256 * TC_BK * 2;        // 32 KB
constexpr int TC_STAGE_BYTES = TC_A_BYTES + TC_B_BYTES_MAX;
constexpr int TC_CSTAGE_BYTES = 64 * 1024;   // output staging: 128 rows x 256 bf16 / 128 fp32, as 16 KB swizzled boxes
constexpr int TC_SMEM_MAX = 226 * 1024;      // dynamic shared memory the kernel is allowed (gemm_tc.cu launch_tc)

// Shared-memory plan of the kernel:
//   classic  n_stages = 3, stage_bytes = 48 KB, the epilogue converts the WHOLE tile into a 64 KB staging buffer (cpw = all
//            chunks of a warp in one pass) and stores it with one burst of TMA box stores;
//   deep     stage_bytes = 16 KB + BN x 128 B, the staging buffer holds one 64-column PASS (16 KB bf16 / 32 KB fp32, cpw = 1
//            chunk per warp per pass) and the space goes to the operand ring: 4 x 48 KB stages at BN = 256 (r1 counters: with
//            3 stages the MMA warp waited for TMA bytes ~25 % of its loop - two stages in flight while one is consumed is
//            about one L2 round trip at the MMA rate).
struct TcPlan { int n_stages, stage_bytes, cstage_bytes, cpw; };

// Everything the host decides for one gemm_nt_tc launch.
struct TcNtPlan {
  int BN, num_n, tiles, grid, split;
  TcPlan plan;
  int smem;                            // dynamic shared memory in bytes (1 KB alignment slack + ring + staging + ActNorm scratch)
};

// The launch plan of gemm_nt_tc for D[M, N] with Kmem bf16 columns per operand row (2 x K for split pairs), output kind
// (out_f32: fp32; out_bf16: bf16; neither: split pairs) and epilogue, on `sms` SMs.  bn_cap, narrow_below, split_on and
// deep_on are the NFDPM_TC_BN / NFDPM_TC_NARROW / NFDPM_TC_SPLIT / NFDPM_TC_DEEP knobs (defaults 256, 74, 1, 1).
inline TcNtPlan tc_nt_plan(int M, int N, int Kmem, bool out_f32, bool out_bf16, bool actnorm, int sms, int bn_cap,
                           int narrow_below, int split_on, int deep_on) {
  TcNtPlan p;
  // N tile: multiple of 16 that splits N evenly; <= 256 columns for bf16 / split output, <= 128 for fp32 output (the
  // classic staging tile holds 128 x 256 bf16 or 128 x 128 fp32 / split pairs)
  int bn_max = out_f32 ? 128 : 256;
  if (bn_max > bn_cap) bn_max = bn_cap;
  // few rows (deep levels): narrower tiles put more CTAs to work (measured at M = 2048, N = 512: 6.1 vs 7.2 us; round 2,
  // per-StepFlow chain over the three levels with narrowing below 48 / 74 / 100 / 148 tiles: 172.3 / 170.1 / 170.9 / 175.4 us
  // in the split-pair mode, 110.4 / 108.7 / 108.9 / 112.3 us in bf16)
  const int m_tiles = (M + TC_BM - 1) / TC_BM;
  while (bn_max > 64 && N >= 2 * bn_max / 2 && m_tiles * ((N + bn_max - 1) / bn_max) <= narrow_below && N % (bn_max / 2) == 0) bn_max >>= 1;
  const int cpb = out_bf16 ? 64 : 32;    // logical columns per 128-byte TMA store box
  const int nblk = (N + bn_max - 1) / bn_max;
  // one N block: any multiple of 16 (columns >= N are clipped by the D tensor map); several N blocks: BN must be a
  // whole number of store boxes, otherwise a tile's last box would spill into its neighbour's columns
  p.BN = (nblk == 1) ? (N + 15) / 16 * 16 : ((N + nblk - 1) / nblk + cpb - 1) / cpb * cpb;
  p.num_n = (N + p.BN - 1) / p.BN;
  p.tiles = m_tiles * p.num_n;
  p.grid = p.tiles < sms ? p.tiles : sms;
  // last-wave balancing (TcWork): split the tiles beyond the last full round into half-width tiles when that puts
  // them on (almost) every SM
  p.split = (split_on && tc_split_ok(p.tiles, p.grid, p.BN, N)) ? 1 : 0;
  const int extra = actnorm ? 2 * p.num_n * p.BN * 4 : 0;      // folded ActNorm scale and bias, zero beyond N
  // classic: the 64 KB staging buffer holds 256 bf16 / 128 fp32 / 128 split-pair columns of the tile per pass
  p.plan = {TC_STAGES, TC_STAGE_BYTES, TC_CSTAGE_BYTES, out_bf16 ? 4 : 2};
  // the deep ring pays when the main loop is long enough to be fed from L2 continuously (measured, tools/bench_gemms.py:
  // M=32768 N=K=512 22.2 -> 21.7 us, N=112 fp32-out 11.0 -> 10.5 us); with ONE tile per CTA (deep levels) the pass-wise
  // epilogue has no next main loop to hide behind and costs 0.5 us, so those keep the classic plan.  deep_on = 0 keeps
  // the classic plan everywhere, = 2 forces the deep plan for every shape
  if (deep_on == 2 || (deep_on == 1 && Kmem / TC_BK >= 4 && p.tiles > p.grid)) {
    p.plan.stage_bytes = TC_A_BYTES + p.BN * TC_BK * 2;
    p.plan.cstage_bytes = 128 * 64 * (out_bf16 ? 2 : 4);     // one 64-column pass
    p.plan.cpw = 1;
    const int avail = TC_SMEM_MAX - 1024 - p.plan.cstage_bytes - extra;   // 226 KB dynamic + static barriers
    p.plan.n_stages = avail / p.plan.stage_bytes;
    if (p.plan.n_stages > TC_MAX_STAGES) p.plan.n_stages = TC_MAX_STAGES;
  }
  p.smem = 1024 + p.plan.n_stages * p.plan.stage_bytes + p.plan.cstage_bytes + extra;
  return p;
}

}  // namespace nfdpm
