// ZeroConv 3x3 GEMM with the affine-coupling epilogue FUSED (north star item 4): the taps-as-N product
//     pm[m, tap*C+co] = sum_ci h2[m,ci] * W3[co,ci,tap]
// is accumulated in tensor memory (tcgen05.mma, bf16 operands via TMA), dumped to SHARED memory and consumed on the
// spot by the step-boundary arithmetic of flow_boundary.cu — 3x3 gather-add, bias, exp(3 logs), sigmoid affine coupling
// (forward: transforms.py:179-184 incl. the per-image log-det; inverse: :196-200), then the next StepFlow's fused
// ActNorm + 1x1 conv (transforms.py:80,132 / :144,93), the NCHW state store and the im2col rows of the next coupling
// network.  pm (36*C*P bytes per image, 9x the flow state) never reaches L2/HBM, and one launch replaces two.
//
// A CTA owns WHOLE images so the 3x3 neighbourhood never crosses CTAs:
//   P = 256 (16x16): 1 image  = 2 UMMA M-tiles sharing the B operand      P | 128: 128/P images = 1 M-tile
// Roles (512 threads): warp 0 TMA producer, warp 1 MMA issuer + TMEM owner, warps 2..15 stage the flow state and the
// parameters while the main loop runs; afterwards all 16 warps dump TMEM -> smem and run the boundary phases.
#include <algorithm>

#include "boundary_body.cuh"   // store8<A1T>, NFDPM_A1_DISPATCH (includes tc_common.cuh)

namespace nfdpm {

constexpr int G3_THREADS = 512;
constexpr int G3_BK = 64;

struct G3Args {
  float* pm_out; int64_t ld_pm_out;      // optional copy of pm for the training stash (may be null)
  const float* in; int64_t in_bs;        // flow state entering the coupling [B,C,P]
  const float* bias3; const float* logs3;
  float* ld_part;                        // [B] per-image sum of log(s + 1e-6), either direction (may be null)
  const float* mt; const float* beta;    // next mix (null = none)
  float* y; int64_t y_bs;                // NCHW sink (may be null)
  float* xs; int64_t xs_bs;              // pre-mix stash sink (may be null)
  void* a1; int64_t lda1;                // im2col sink (may be null)
  int B, C, H, W, inverse;
  int K, ldp;                            // GEMM reduction length in bf16 columns of the operand rows (multiple of 64; 2 x the
                                         // logical length for split pairs), padded 9C (multiple of 16)
  int ipc;                               // images per CTA
  int ipp;                               // images per boundary pass (smem budget for the pm rows)
  int stages, stage_bytes, a_bytes, b_box_rows, n_bbox;
  int pm_region;                         // bytes of max(ring, pm staging)
  FastDiv dCP, dP, dPCh, dCh, dW, dOgP, dPNg, dNg, dCp, dLdp;   // index divisors (multiply-high, common.cuh)
};

template <typename A1T, bool X3>
__global__ void __launch_bounds__(G3_THREADS, 1) gemm3_boundary_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                       const __grid_constant__ CUtensorMap tmB,
                                                                       const G3Args a) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t bars[2 * 3 + 1];
  __shared__ uint32_t s_tmem_base;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
  const int C = a.C, H = a.H, W = a.W, P = H * W, Ch = C >> 1, PS = P + 1, Cp = (C + 3) & ~3;
  const int ldp = a.ldp, lds = ldp + 4;                     // padded pm row stride in shared memory (floats)
  const uint32_t ring = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* base = smem_raw + (ring - smem_u32(smem_raw));
  float* pm_s = reinterpret_cast<float*>(base);             // aliases the operand ring (used after the main loop)
  float* x_s = reinterpret_cast<float*>(base + a.pm_region); // [ipc][C][PS]
  float* u_s = x_s + a.ipc * C * PS;                        // [ipc][C][PS] (aliases x_s when there is no mix)
  float* m_s = (a.mt != nullptr) ? u_s + a.ipc * C * PS : u_s;     // [C][Cp] + beta[Cp]
  float* par_s = m_s + ((a.mt != nullptr) ? (C * Cp + Cp) : 0);    // [2C]
  float* ls_s = par_s + 2 * C;                              // [ipp][P*Ch]
  const int W2p = W + 2, PP = (H + 2) * W2p;
  // after the coupling passes the pm rows are dead: their memory holds the zero-bordered im2col source and its column table
  float* pad_s = reinterpret_cast<float*>(base);            // [ipc][Ch][PP]
  int* kt_s = reinterpret_cast<int*>(pad_s + ((a.ipc * Ch * PP + 3) & ~3));   // [9*Ch] im2col column -> offset in pad_s
  if (a.mt == nullptr) u_s = x_s;
  const uint32_t bar_full = smem_u32(&bars[0]), bar_empty = smem_u32(&bars[3]), bar_done = smem_u32(&bars[6]);

  const int img0 = blockIdx.x * a.ipc;
  const int n_img = min(a.ipc, a.B - img0);                 // images this CTA really owns
  const int n_mt = (a.ipc * P) > 128 ? 2 : 1;               // UMMA M-tiles
  const int row0 = img0 * P;                                // first row of h2 / pm
  const int num_kb = a.K / G3_BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < a.stages; ++s) {
      mbar_init(bar_full + 8 * s, 1);
      mbar_init(bar_empty + 8 * s, 1);
    }
    mbar_init(bar_done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(smem_u32(&s_tmem_base), 512);
  pdl_trigger();
  pdl_wait();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = s_tmem_base;

  if (warp == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    const uint32_t tx = (uint32_t)(a.a_bytes + a.n_bbox * a.b_box_rows * 128);
    for (int kb = 0; kb < num_kb; ++kb) {
      mbar_wait(bar_empty + 8 * stage, phase ^ 1);
      if (lane == 0) {
        const uint32_t sa = ring + stage * a.stage_bytes, sb = sa + a.a_bytes;
        mbar_arrive_expect_tx(bar_full + 8 * stage, tx);
        for (int t = 0; t < n_mt; ++t) tma_load_2d(sa + t * 16384, &tmA, kb * G3_BK, row0 + t * 128, bar_full + 8 * stage);
        for (int j = 0; j < a.n_bbox; ++j)
          tma_load_2d(sb + j * a.b_box_rows * 128, &tmB, kb * G3_BK, j * a.b_box_rows, bar_full + 8 * stage);
      }
      __syncwarp();
      if (++stage == a.stages) { stage = 0; phase ^= 1; }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    int stage = 0;
    uint32_t phase = 0;
    const int n0 = ldp > 256 ? 224 : ldp, n1 = ldp - n0;    // N split (each a multiple of 16, <= 256)
    const uint32_t idesc0 = make_idesc(128, n0), idesc1 = make_idesc(128, n1 > 0 ? n1 : 16);
    for (int kb = 0; kb < num_kb; ++kb) {
      mbar_wait(bar_full + 8 * stage, phase);
      tc_fence_after();
      if (lane == 0) {
        const uint32_t sa = ring + stage * a.stage_bytes, sb = sa + a.a_bytes;
        for (int t = 0; t < n_mt; ++t) {
          const uint64_t adesc = make_smem_desc(sa + t * 16384);
          const uint64_t b0 = make_smem_desc(sb), b1 = make_smem_desc(sb + n0 * 128);
          const uint32_t d = tmem_base + t * 256;
          umma_stage<X3>(d, adesc, b0, idesc0, kb == 0);
          if (n1 > 0) umma_stage<X3>(d + n0, adesc, b1, idesc1, kb == 0);
        }
        umma_commit(bar_empty + 8 * stage);
        if (kb == num_kb - 1) umma_commit(bar_done);
      }
      __syncwarp();
      if (++stage == a.stages) { stage = 0; phase ^= 1; }
    }
  } else {
    // ===================== warps 2..15: stage parameters and the flow state while the GEMM runs =====================
    const int t2 = tid - 64, nt2 = G3_THREADS - 64;
    if (a.mt != nullptr) {
      for (int i = t2; i < C * Cp; i += nt2) {
        const int r = fdiv(i, a.dCp), c = i - r * Cp;
        m_s[i] = (c < C) ? a.mt[r * C + c] : 0.f;
      }
      for (int i = t2; i < Cp; i += nt2) m_s[C * Cp + i] = (i < C) ? a.beta[i] : 0.f;
    }
    for (int i = t2; i < C; i += nt2) {
      par_s[i] = a.bias3[i];
      par_s[C + i] = expf(3.f * a.logs3[i]);
    }
    // batches of four loads in flight before the dependent shared-memory stores
    const int nx = n_img * C * P;
    for (int base = t2; base < nx; base += 4 * nt2) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * nt2;
        float val = 0.f;
        if (i < nx) {
          const int im = fdiv(i, a.dCP), r = i - im * C * P;
          val = a.in[(int64_t)(img0 + im) * a.in_bs + r];
        }
        v[u] = val;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * nt2;
        if (i < nx) {
          const int im = fdiv(i, a.dCP), r = i - im * C * P;
          const int c = fdiv(r, a.dP), p = r - c * P;
          x_s[(im * C + c) * PS + p] = v[u];
        }
      }
    }
  }
  // accumulator complete (every thread observes the commit), operand ring free for reuse
  mbar_wait(bar_done, 0);
  tc_fence_after();
  __syncthreads();

  const int rows_pp = a.ipp * P;                            // pm rows per pass (multiple of 32)
  const int n_pass = (a.ipc + a.ipp - 1) / a.ipp;
  const int q = warp & 3, cw = warp >> 2;                   // TMEM lane quadrant, column-slice owner (4 per quadrant)
  for (int pass = 0; pass < n_pass; ++pass) {
    const int im_lo = pass * a.ipp;
    const int im_n = min(a.ipp, n_img - im_lo);             // images of this pass (<= 0: nothing left)
    if (im_n <= 0) break;
    // ---- TMEM -> smem: rows [r_lo, r_lo + rows_pp) of the CTA tile
    const int r_lo = pass * rows_pp;
    for (int t = 0; t < n_mt; ++t) {
      const int trow = t * 128 + q * 32;                    // first tile row of this warp's lanes
      if (trow < r_lo || trow >= r_lo + rows_pp) continue;
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + t * 256;
      float* dst = pm_s + (size_t)(trow - r_lo + lane) * lds;
      for (int c0 = cw * 16; c0 < ldp; c0 += 64) {
        uint32_t r[16];
        tmem_ld16(taddr + c0, r);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<float4*>(dst + c0 + 4 * j) =
              make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]),
                          __uint_as_float(r[4 * j + 3]));
      }
    }
    __syncthreads();
    if (a.pm_out != nullptr) {                              // training stash: coalesced copy of the pm rows
      const int n = im_n * P * ldp;
      float* o = a.pm_out + (int64_t)(row0 + r_lo) * a.ld_pm_out;
      for (int i = tid; i < n; i += G3_THREADS) {
        const int r = fdiv(i, a.dLdp), c = i - r * ldp;
        o[(int64_t)r * a.ld_pm_out + c] = pm_s[(size_t)r * lds + c];
      }
    }
    // ---- affine coupling: item = (image, pixel, j), j fastest
    {
      const int n_it = im_n * P * Ch;
      for (int it = tid; it < n_it; it += G3_THREADS) {
        const int im = fdiv(it, a.dPCh), r = it - im * P * Ch;
        const int p = fdiv(r, a.dCh), j = r - p * Ch;
        const int py = fdiv(p, a.dW), px = p - py * W;
        const float* pmi = pm_s + (size_t)(im * P) * lds;
        float ls = 0.f, tt = 0.f;
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          const int yy = py + tap / 3 - 1, xx = px + tap % 3 - 1;
          if (yy >= 0 && yy < H && xx >= 0 && xx < W) {
            const float* rr = pmi + (size_t)(yy * W + xx) * lds + tap * C + j;
            ls += rr[0];
            tt += rr[Ch];
          }
        }
        const float log_s = (ls + par_s[j]) * par_s[C + j];
        const float sh_t = (tt + par_s[Ch + j]) * par_s[C + Ch + j];
        const float s = 1.f / (1.f + expf(-(log_s + 2.f)));
        float* xb = x_s + ((im_lo + im) * C + Ch + j) * PS + p;
        if (a.inverse) {
          *xb = *xb / (s + 1e-6f) - sh_t;
          if (a.ld_part != nullptr) ls_s[it] = logf(s + 1e-6f);
        } else {
          *xb = (*xb + sh_t) * s;
          ls_s[it] = logf(s + 1e-6f);
        }
      }
    }
    __syncthreads();
    if (a.ld_part != nullptr && warp < im_n) {
      // deterministic per-image sum: one warp per image, fixed lane-strided order + shuffle tree
      float acc = 0.f;
      const float* l = ls_s + warp * P * Ch;
#pragma unroll 8
      for (int i = lane; i < P * Ch; i += 32) acc += l[i];
      acc = warp_sum(acc);
      if (lane == 0) a.ld_part[img0 + im_lo + warp] = acc;
    }
    __syncthreads();                                         // pm_s / ls_s are rewritten by the next pass
  }

  if (a.a1 != nullptr) {
    for (int i = tid; i < a.ipc * Ch * PP; i += G3_THREADS) pad_s[i] = 0.f;
    for (int k = tid; k < 9 * Ch; k += G3_THREADS) {
      const int c = k / 9, tap = k - c * 9;
      kt_s[k] = c * PP + (tap / 3) * W2p + (tap % 3);
    }
    if (a.mt == nullptr) __syncthreads();                    // (with a mix, its barrier orders the zero fill)
  }
  // ---- pre-mix stash (the next StepFlow's input)
  if (a.xs != nullptr) {
    for (int i = tid; i < n_img * C * P; i += G3_THREADS) {
      const int im = fdiv(i, a.dCP), r = i - im * C * P;
      const int c = fdiv(r, a.dP), p = r - c * P;
      a.xs[(int64_t)(img0 + im) * a.xs_bs + r] = x_s[(im * C + c) * PS + p];
    }
  }
  // ---- channel mix, item = (image, group of 4 outputs, pixel), lanes over pixels
  if (a.mt != nullptr) {
    const int n_og = Cp >> 2;
    for (int it = tid; it < n_img * n_og * P; it += G3_THREADS) {
      const int im = fdiv(it, a.dOgP), r = it - im * n_og * P;
      const int og = fdiv(r, a.dP), p = r - og * P;
      const float4 b4 = *reinterpret_cast<const float4*>(m_s + C * Cp + og * 4);
      float a0 = b4.x, a1 = b4.y, a2 = b4.z, a3 = b4.w;
      const float* xi = x_s + (size_t)im * C * PS + p;
#pragma unroll 4
      for (int c = 0; c < C; ++c) {
        const float xv = xi[c * PS];
        const float4 w = *reinterpret_cast<const float4*>(m_s + c * Cp + og * 4);
        a0 = fmaf(w.x, xv, a0);
        a1 = fmaf(w.y, xv, a1);
        a2 = fmaf(w.z, xv, a2);
        a3 = fmaf(w.w, xv, a3);
      }
      const int o = og * 4;
      float* ui = u_s + (size_t)im * C * PS + p;
      ui[o * PS] = a0;
      if (o + 1 < C) ui[(o + 1) * PS] = a1;
      if (o + 2 < C) ui[(o + 2) * PS] = a2;
      if (o + 3 < C) ui[(o + 3) * PS] = a3;
    }
    __syncthreads();
  }
  // ---- interior of the zero-bordered copy of the channels the next coupling network reads
  if (a.a1 != nullptr) {
    for (int i = tid; i < n_img * C * P; i += G3_THREADS) {
      const int im = fdiv(i, a.dCP), r = i - im * C * P;
      const int c = fdiv(r, a.dP), p = r - c * P;
      if (c < Ch) {
        const int py = fdiv(p, a.dW), px = p - py * W;
        pad_s[(im * Ch + c) * PP + (py + 1) * W2p + px + 1] = u_s[(im * C + c) * PS + p];
      }
    }
  }
  // ---- NCHW sink
  if (a.y != nullptr) {
    for (int i = tid; i < n_img * C * P; i += G3_THREADS) {
      const int im = fdiv(i, a.dCP), r = i - im * C * P;
      const int c = fdiv(r, a.dP), p = r - c * P;
      a.y[(int64_t)(img0 + im) * a.y_bs + r] = u_s[(im * C + c) * PS + p];
    }
  }
  if (a.a1 != nullptr) __syncthreads();
  // ---- im2col sink, item = (image, pixel, 8-column group), group fastest
  if (a.a1 != nullptr) {
    const int Kc = Ch * 9;
    const int n_g = (int)(a.lda1 >> 3);
    for (int it = tid; it < n_img * P * n_g; it += G3_THREADS) {
      const int im = fdiv(it, a.dPNg), r = it - im * P * n_g;
      const int p = fdiv(r, a.dNg), g = r - p * n_g;
      const int py = fdiv(p, a.dW), px = p - py * W;
      const float* win = pad_s + (size_t)im * Ch * PP + py * W2p + px;
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = g * 8 + e;
        v[e] = (k < Kc) ? win[kt_s[k]] : 0.f;
      }
      store8<A1T>(reinterpret_cast<A1T*>(a.a1), (int64_t)(img0 + im) * P + p, a.lda1, g * 8, v);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// shape plan shared by the launcher and the support query
static bool g3_plan(int B, int C, int H, int W, int K, int64_t ldp, bool mix, G3Args* a, size_t* smem) {
  const int P = H * W;
  if (C % 2 || K % G3_BK || ldp % 16 || ldp < 9 * C || ldp > 512) return false;
  int ipc;
  if (P == 256) ipc = 1;
  else if (P <= 128 && 128 % P == 0) ipc = 128 / P;
  else return false;
  const int rows = ipc * P;
  if (rows > 128 && ldp > 256) return false;                // two M-tiles need 2 x ldp <= 512 TMEM columns
  const int a_bytes = rows > 128 ? 32768 : 16384;
  const int n_bbox = ldp > 256 ? 2 : 1;
  const int b_rows = (int)(ldp / n_bbox);
  if (b_rows % 8) return false;
  const int stage_bytes = a_bytes + (int)ldp * 128;
  const int lds = (int)ldp + 4;
  // images per pass: the pm rows of a pass must fit ~120 KB
  int ipp = ipc;
  while (ipp > 1 && (size_t)ipp * P * lds * 4 > 122880) ipp = (ipp + 1) / 2;
  if ((ipp * P) % 32 != 0 && ipp != ipc) return false;
  if (ipp > G3_THREADS / 32) return false;                  // one warp per image in the log-det reduction
  if ((size_t)ipp * P * lds * 4 > 122880) return false;
  const size_t pm_bytes = (size_t)ipp * P * lds * 4;
  const size_t PS = P + 1, Cp = (C + 3) & ~3;
  size_t body = (size_t)ipc * C * PS * (mix ? 2 : 1) + (mix ? C * Cp + Cp : 0) + 2 * C + (size_t)ipp * P * (C / 2);
  body *= sizeof(float);
  // the im2col source (zero-bordered copy + column table) reuses the pm rows' memory
  const size_t pad_bytes = sizeof(float) * ((((size_t)ipc * (C / 2) * (H + 2) * (W + 2) + 3) & ~(size_t)3) + 9 * (size_t)(C / 2));
  int stages = 3;
  while (stages > 2 && 1024 + std::max((size_t)stages * stage_bytes, pm_bytes) + body > 224 * 1024) --stages;
  size_t region = std::max(std::max((size_t)stages * stage_bytes, pm_bytes), pad_bytes);
  region = (region + 15) & ~(size_t)15;
  if (1024 + region + body > 224 * 1024) return false;
  if (a) {
    a->ipc = ipc; a->ipp = ipp; a->stages = stages; a->stage_bytes = stage_bytes; a->a_bytes = a_bytes;
    a->b_box_rows = b_rows; a->n_bbox = n_bbox; a->pm_region = (int)region;
  }
  if (smem) *smem = 1024 + region + body;
  return true;
}

}  // namespace nfdpm

using namespace nfdpm;

// K counts bf16 columns of the operand rows (2 x the logical reduction length for split pairs)
extern "C" int nfdpm_gemm3_boundary_ok(int B, int C, int H, int W, int K, int64_t ldp) {
  return g3_plan(B, C, H, W, K, ldp, true, nullptr, nullptr) ? 1 : 0;
}

extern "C" int nfdpm_gemm3_boundary(const void* h2, int h_dtype, int64_t ldh, const void* w3p, float* pm_out, int64_t ld_pm_out,
                                    const float* in, int64_t in_bs, const float* bias3, const float* logs3, float* ld_part,
                                    const float* mt, const float* beta, float* y, int64_t y_bs, float* xs, int64_t xs_bs,
                                    void* a1, int a1_dtype, int64_t lda1, int B, int C, int H, int W, int K, int64_t ldp,
                                    int inverse, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(h2 && w3p && in && bias3 && logs3, "nfdpm_gemm3_boundary: null pointer");
  NFDPM_REQUIRE((mt == nullptr) == (beta == nullptr), "nfdpm_gemm3_boundary: mt/beta must both be set or both NULL");
  NFDPM_REQUIRE(y != nullptr || a1 != nullptr || xs != nullptr, "nfdpm_gemm3_boundary: no sink");
  NFDPM_REQUIRE(a1 == nullptr || (lda1 % 8 == 0 && lda1 >= 9 * (int64_t)(C / 2) && ((uintptr_t)a1 % 16) == 0),
                "nfdpm_gemm3_boundary: bad im2col sink");
  NFDPM_REQUIRE(a1 == nullptr || a1_dtype == NFDPM_F32 || a1_dtype == NFDPM_BF16 || (a1_dtype == NFDPM_BF16X2 && lda1 % 32 == 0),
                "nfdpm_gemm3_boundary: bad a1 dtype");
  NFDPM_REQUIRE(h_dtype == NFDPM_BF16 || (h_dtype == NFDPM_BF16X2 && ldh % 32 == 0 && K % 32 == 0),
                "nfdpm_gemm3_boundary: h2 / w3p must be bf16 or split pairs (dtype %d)", h_dtype);
  const bool x3 = h_dtype == NFDPM_BF16X2;
  const int kmul = x3 ? 2 : 1;
  NFDPM_REQUIRE(ldh >= K && ldh % 8 == 0 && ((uintptr_t)h2 % 16) == 0 && ((uintptr_t)w3p % 16) == 0,
                "nfdpm_gemm3_boundary: bad GEMM operands");
  NFDPM_REQUIRE(pm_out == nullptr || ld_pm_out >= ldp, "nfdpm_gemm3_boundary: bad pm_out");
  G3Args a;
  size_t smem = 0;
  NFDPM_REQUIRE(g3_plan(B, C, H, W, K * kmul, ldp, mt != nullptr, &a, &smem),
                "nfdpm_gemm3_boundary: unsupported shape B=%d C=%d H=%d W=%d K=%d ldp=%lld (use nfdpm_gemm_nt + "
                "nfdpm_flow_boundary)", B, C, H, W, K, (long long)ldp);
  a.pm_out = pm_out; a.ld_pm_out = ld_pm_out; a.in = in; a.in_bs = in_bs; a.bias3 = bias3; a.logs3 = logs3;
  a.ld_part = ld_part; a.mt = mt; a.beta = beta; a.y = y; a.y_bs = y_bs; a.xs = xs; a.xs_bs = xs_bs; a.a1 = a1;
  a.lda1 = lda1; a.B = B; a.C = C; a.H = H; a.W = W; a.inverse = inverse; a.K = K * kmul; a.ldp = (int)ldp;
  {
    const int P = H * W, Ch = C / 2, Cp = (C + 3) & ~3, n_g = lda1 >= 8 ? (int)(lda1 >> 3) : 1;
    a.dCP = make_fastdiv(C * P); a.dP = make_fastdiv(P); a.dPCh = make_fastdiv(P * Ch); a.dCh = make_fastdiv(Ch);
    a.dW = make_fastdiv(W); a.dOgP = make_fastdiv((Cp >> 2) * P); a.dPNg = make_fastdiv(P * n_g); a.dNg = make_fastdiv(n_g);
    a.dCp = make_fastdiv(Cp); a.dLdp = make_fastdiv((int)ldp);
  }
  const int64_t M = (int64_t)B * H * W;
  CUtensorMap tmA, tmB;
  if (make_map(&tmA, h2, M, K * kmul, ldh * kmul, 128)) return 1;
  if (make_map(&tmB, w3p, ldp, K * kmul, K * kmul, a.b_box_rows)) return 1;
  const int grid = (B + a.ipc - 1) / a.ipc;
  cudaStream_t st = as_stream(stream);
  const int a1dt = a1 != nullptr ? a1_dtype : NFDPM_F32;
#define LAUNCH(T, X)                                                                                                   \
  do {                                                                                                                 \
    static bool attr_set = false;                                                                                      \
    if (!attr_set) {                                                                                                   \
      NFDPM_CUDA(cudaFuncSetAttribute(gemm3_boundary_kernel<T, X>, cudaFuncAttributeMaxDynamicSharedMemorySize, 225 * 1024)); \
      attr_set = true;                                                                                                 \
    }                                                                                                                  \
    NFDPM_CUDA(launch_pdl(gemm3_boundary_kernel<T, X>, dim3(grid), dim3(G3_THREADS), smem, st, tmA, tmB, a));          \
  } while (0)
#define GO_X3(T) LAUNCH(T, true)
#define GO_BF(T) LAUNCH(T, false)
  if (x3) NFDPM_A1_DISPATCH(a1dt, GO_X3);
  else NFDPM_A1_DISPATCH(a1dt, GO_BF);
#undef GO_X3
#undef GO_BF
#undef LAUNCH
  return 0;
}
