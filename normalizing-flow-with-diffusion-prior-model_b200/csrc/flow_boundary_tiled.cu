// Step boundary for images that one CTA cannot (or should not) own: the same arithmetic as flow_boundary_kernel
// (flow_boundary.cu / boundary_body.cuh: [affine coupling with the taps-as-N rows] -> [fused ActNorm + 1x1 conv] -> NCHW state
// and/or im2col rows of the next coupling network), but a CTA owns a BAND of R image rows instead of a whole image:
//   * images with more than 256 pixels (the 64x64 and 32x32 levels of a 128x128 input) get the fused boundary at all,
//   * small batches (config 4: 8 images per GPU) spread over B * ceil(H / R) CTAs instead of B.
// The im2col rows of a pixel need the mixed state of its 3x3 neighbourhood, so a band RECOMPUTES one halo row above and one
// below (coupling + mix of the halo pixels; their pm rows are in L2): no inter-CTA exchange, at (R + 2) / R of the elementwise
// arithmetic.  The band is addressed as Rv = R + 2*halo "virtual" rows starting at image row r0 - halo; rows outside the image
// are skipped, so every index division is by a launch constant (multiply-high, common.cuh).
// The per-image log-det is written as one partial per band: ld_part[t * B + b] (nfdpm_accumulate sums the rows in order);
// the inverse writes the same partial, from the s it divides by.
#include "boundary_body.cuh"
#include <stdlib.h>

namespace nfdpm {

struct TileGeom {
  int R, T, halo, Rv, Pv;              // own rows per band, bands per image, halo rows (0/1), R + 2*halo, Rv * W
  FastDiv dPv, dT;
  int bulk_m;                          // the mix matrix + beta arrive by cp.async.bulk (C % 4 == 0, 16-byte aligned)
};

//   x_s [C][Pv+1] | u_s [C][Pv+1] (mix only) | m_s [C][Cp] + beta [Cp] (mix only) | par_s [2C] | ls_s [R*W*C/2] (coupling only)
//   | pad_s [C/2][(R+2)*(W+2)] | kt_s [9*C/2]   (im2col sink only)
static __host__ __device__ size_t tiled_scratch_floats(int C, int W, int R, int halo, bool coupling, bool mix, size_t* pad_off,
                                                       size_t* kt_off) {
  const size_t Pv = (size_t)(R + 2 * halo) * W, PS = Pv + 1, Cp = (C + 3) & ~3, Ch = C / 2;
  size_t fl = (size_t)C * PS * (mix ? 2 : 1);
  if (mix) fl += (size_t)C * Cp + Cp;
  if (coupling) fl += 2 * (size_t)C + (size_t)R * W * Ch;
  fl = (fl + 3) & ~(size_t)3;
  if (pad_off) *pad_off = fl;
  if (halo) fl += (Ch * (size_t)(R + 2) * (W + 2) + 3) & ~(size_t)3;
  if (kt_off) *kt_off = fl;
  if (halo) fl += (9 * Ch + 3) & ~(size_t)3;
  return fl;
}

template <bool COUPLING, typename A1T>
__global__ void __launch_bounds__(1024) flow_boundary_tiled_kernel(const BoundaryArgs a, const TileGeom g) {
  extern __shared__ __align__(16) float sm[];
  __shared__ __align__(8) uint64_t m_bar;
  const int tid = threadIdx.x, nt = blockDim.x;
  pdl_trigger();
  if (g.bulk_m && tid == 0) {
    mbar_init(smem_u32(&m_bar), 1);
    fence_barrier_init();
  }
  pdl_wait();
  const int b = fdiv((int)blockIdx.x, g.dT), t = (int)blockIdx.x - b * g.T;
  const int C = a.C, H = a.H, W = a.W, P = H * W, Ch = C >> 1;
  const int R = g.R, halo = g.halo, Pv = g.Pv, PS = Pv + 1, Cp = (C + 3) & ~3;
  const int r0 = t * R, v0 = r0 - halo;                 // first own row, image row of virtual row 0
  const int W2p = W + 2, PP = (R + 2) * W2p;
  const bool mix = a.mt != nullptr;
  const bool want_a1 = a.a1 != nullptr;                 // host: halo == 1 exactly when there is an im2col sink
  size_t pad_off, kt_off;
  tiled_scratch_floats(C, W, R, halo, COUPLING, mix, &pad_off, &kt_off);
  float* x_s = sm;
  float* u_s = mix ? x_s + C * PS : x_s;
  float* m_s = x_s + C * PS * (mix ? 2 : 1);           // [C][Cp] + beta [Cp] (mix only)
  float* par_s = m_s + (mix ? (C * Cp + Cp) : 0);
  float* ls_s = par_s + (COUPLING ? 2 * C : 0);
  float* pad_s = sm + pad_off;
  int* kt_s = reinterpret_cast<int*>(sm + kt_off);

  // ---- phase 0: parameters and the band of the image, channel-major (lanes over pixels: coalesced runs of Pv floats)
  if (mix && g.bulk_m) {
    // [C][C] matrix + beta [C]: two contiguous blocks, fetched by the bulk-copy engine while the CTA stages the band
    // (C = 192: 147 KB per CTA, which took 36 dependent load rounds per thread as a loop)
    if (tid == 0) {
      const uint32_t bar = smem_u32(&m_bar);
      const uint32_t nb = (uint32_t)C * C * 4;
      mbar_arrive_expect_tx(bar, nb + (uint32_t)C * 4);
      for (uint32_t off = 0; off < nb; off += 32768)
        bulk_load(smem_u32(m_s) + off, reinterpret_cast<const char*>(a.mt) + off, min(nb - off, 32768u), bar);
      bulk_load(smem_u32(m_s + C * Cp), a.beta, (uint32_t)C * 4, bar);
    }
  } else if (mix) {
    for (int i = tid; i < C * Cp; i += nt) {
      const int r = fdiv(i, a.dCp), c = i - r * Cp;
      m_s[i] = (c < C) ? __ldg(a.mt + r * C + c) : 0.f;
    }
    for (int i = tid; i < Cp; i += nt) m_s[C * Cp + i] = (i < C) ? __ldg(a.beta + i) : 0.f;
  }
  if (COUPLING) {
    for (int i = tid; i < C; i += nt) {
      par_s[i] = __ldg(a.bias3 + i);
      par_s[C + i] = expf(3.f * __ldg(a.logs3 + i));
    }
  }
  if (want_a1) {
    for (int i = tid; i < Ch * PP; i += nt) pad_s[i] = 0.f;
    for (int k = tid; k < 9 * Ch; k += nt) {
      const int c = k / 9, tap = k - c * 9;
      kt_s[k] = c * PP + (tap / 3) * W2p + (tap % 3);
    }
  }
  const float* inb = a.in + (int64_t)b * a.in_bs;
  if (a.squeeze_in) {
    const int W2 = 2 * W;
    for (int i = tid; i < (C >> 2) * Pv; i += nt) {
      const int cc = fdiv(i, g.dPv), q = i - cc * Pv;
      const int v = fdiv(q, a.dW), px = q - v * W, py = v0 + v;
      float2 t0 = make_float2(0.f, 0.f), t1 = t0;
      if (py >= 0 && py < H) {
        const float* s = inb + ((int64_t)cc * 2 * H + 2 * py) * W2 + 2 * px;
        t0 = *reinterpret_cast<const float2*>(s);
        t1 = *reinterpret_cast<const float2*>(s + W2);
      }
      x_s[(cc * 4 + 0) * PS + q] = t0.x;
      x_s[(cc * 4 + 1) * PS + q] = t0.y;
      x_s[(cc * 4 + 2) * PS + q] = t1.x;
      x_s[(cc * 4 + 3) * PS + q] = t1.y;
    }
  } else {
    for (int i = tid; i < C * Pv; i += nt) {
      const int c = fdiv(i, g.dPv), q = i - c * Pv;
      const int py = v0 + fdiv(q, a.dW);
      x_s[c * PS + q] = (py >= 0 && py < H) ? __ldg(inb + (int64_t)c * P + (int64_t)v0 * W + q) : 0.f;
    }
  }
  __syncthreads();

  // ---- phase 1: affine coupling of every pixel of the band (halo included), item = (pixel, j), j fastest
  if (COUPLING) {
    const float* pmb = a.pm + (int64_t)b * P * a.ldp;
    const int64_t ldp = a.ldp;
    for (int it = tid; it < Pv * Ch; it += nt) {
      const int q = fdiv(it, a.dCh), j = it - q * Ch;
      const int v = fdiv(q, a.dW), px = q - v * W, py = v0 + v;
      if (py < 0 || py >= H) continue;
      const int p = py * W + px;
      float lv[9], tv[9];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int yy = py + tap / 3 - 1, xx = px + tap % 3 - 1;
        const bool ok = (yy >= 0) && (yy < H) && (xx >= 0) && (xx < W);
        const float* r = pmb + (int64_t)(ok ? yy * W + xx : p) * ldp + tap * C + j;
        const float l0 = __ldg(r), t0 = __ldg(r + Ch);
        lv[tap] = ok ? l0 : 0.f;
        tv[tap] = ok ? t0 : 0.f;
      }
      float ls = 0.f, tt = 0.f;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        ls += lv[tap];
        tt += tv[tap];
      }
      const float log_s = (ls + par_s[j]) * par_s[C + j];
      const float sh_t = (tt + par_s[Ch + j]) * par_s[C + Ch + j];
      const float s = 1.f / (1.f + expf(-(log_s + 2.f)));
      const float xb = x_s[(Ch + j) * PS + q];
      if (a.inverse) {
        x_s[(Ch + j) * PS + q] = xb / (s + 1e-6f) - sh_t;
        if (a.ld_part != nullptr && v >= halo && v < halo + R) ls_s[(q - halo * W) * Ch + j] = logf(s + 1e-6f);
      } else {
        x_s[(Ch + j) * PS + q] = (xb + sh_t) * s;
        if (v >= halo && v < halo + R) ls_s[(q - halo * W) * Ch + j] = logf(s + 1e-6f);
      }
    }
    __syncthreads();
    if (a.ld_part != nullptr && tid < 32) {
      const int n_own = (min(H, r0 + R) - r0) * W * Ch;            // own rows are contiguous from r0: entries [0, n_own) are set
      float acc = 0.f;
#pragma unroll 8
      for (int i = tid; i < n_own; i += 32) acc += ls_s[i];
      acc = warp_sum(acc);
      if (tid == 0) a.ld_part[(int64_t)t * a.B + b] = acc;
    }
  }

  // ---- phase 1b: stash of the pre-mix state (own pixels)
  if (a.xs != nullptr) {
    float* xb = a.xs + (int64_t)b * a.xs_bs + (int64_t)v0 * W;
    for (int i = tid; i < C * Pv; i += nt) {
      const int c = fdiv(i, g.dPv), q = i - c * Pv;
      const int v = fdiv(q, a.dW);
      if (v >= halo && v < halo + R && v0 + v < H) xb[(int64_t)c * P + q] = x_s[c * PS + q];
    }
  }

  // ---- phase 2: channel mix of the band, item = (group of 4 outputs, pixel), lanes over pixels
  if (mix) {
    if (g.bulk_m) mbar_wait(smem_u32(&m_bar), 0);
    const int n_og = Cp >> 2;
    for (int it = tid; it < n_og * Pv; it += nt) {
      const int og = fdiv(it, g.dPv), q = it - og * Pv;
      const float4 b4 = *reinterpret_cast<const float4*>(m_s + C * Cp + og * 4);
      float a0 = b4.x, a1 = b4.y, a2 = b4.z, a3 = b4.w;
#pragma unroll 4
      for (int c = 0; c < C; ++c) {
        const float xv_ = x_s[c * PS + q];
        const float4 w = *reinterpret_cast<const float4*>(m_s + c * Cp + og * 4);
        a0 = fmaf(w.x, xv_, a0);
        a1 = fmaf(w.y, xv_, a1);
        a2 = fmaf(w.z, xv_, a2);
        a3 = fmaf(w.w, xv_, a3);
      }
      const int o = og * 4;
      u_s[o * PS + q] = a0;
      if (o + 1 < C) u_s[(o + 1) * PS + q] = a1;
      if (o + 2 < C) u_s[(o + 2) * PS + q] = a2;
      if (o + 3 < C) u_s[(o + 3) * PS + q] = a3;
    }
    __syncthreads();
  }
  if (want_a1) {
    // interior of the zero-bordered copy: pad row v <-> image row r0 - 1 + v (rows outside the image stay zero)
    for (int i = tid; i < Ch * Pv; i += nt) {
      const int c = fdiv(i, g.dPv), q = i - c * Pv;
      const int v = fdiv(q, a.dW), px = q - v * W, py = v0 + v;
      if (py >= 0 && py < H) pad_s[c * PP + v * W2p + px + 1] = u_s[c * PS + q];
    }
  }

  // ---- phase 3a: NCHW sink (own pixels)
  if (a.y != nullptr) {
    float* yb = a.y + (int64_t)b * a.y_bs + (int64_t)v0 * W;
    for (int i = tid; i < C * Pv; i += nt) {
      const int c = fdiv(i, g.dPv), q = i - c * Pv;
      const int v = fdiv(q, a.dW);
      if (v >= halo && v < halo + R && v0 + v < H) yb[(int64_t)c * P + q] = u_s[c * PS + q];
    }
  }
  // ---- phase 3b: im2col sink (own pixels), item = (pixel, 8-column group), group fastest
  if (want_a1) {
    __syncthreads();
    const int K = Ch * 9;
    const int n_g = (int)(a.lda1 >> 3);
    A1T* a1b = reinterpret_cast<A1T*>(a.a1);
    for (int it = tid; it < R * W * n_g; it += nt) {
      const int po = fdiv(it, a.dNg), gg = it - po * n_g;
      const int vo = fdiv(po, a.dW), px = po - vo * W, py = r0 + vo;
      if (py >= H) continue;
      const float* win = pad_s + vo * W2p + px;          // top-left of the 3x3 window: pad row of image row py - 1
      float vv[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = gg * 8 + e;
        vv[e] = (k < K) ? win[kt_s[k]] : 0.f;
      }
      store8<A1T>(a1b, (int64_t)b * P + py * W + px, a.lda1, gg * 8, vv);
    }
  }
}

// rows per band: about 256 own pixels per CTA, fewer when that would leave most SMs without a CTA
static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return (v && *v) ? atoi(v) : dflt;
}
static int choose_rows(int B, int C, int H, int W, bool coupling, bool mix, bool want_a1) {
  static const int pix = env_int("NFDPM_TILE_PIX", 256), ctas = env_int("NFDPM_TILE_CTAS", 112);   // tuning knobs
  int R = pix / W;
  if (R < 1) R = 1;
  if (R > H) R = H;
  while (R > 1 && (int64_t)B * ((H + R - 1) / R) < ctas) --R;
  const int halo = want_a1 ? 1 : 0;
  while (R > 1 && tiled_scratch_floats(C, W, R, halo, coupling, mix, nullptr, nullptr) * sizeof(float) > 200 * 1024) --R;
  return R;
}

}  // namespace nfdpm

using namespace nfdpm;

extern "C" int nfdpm_flow_boundary_tiles(int B, int C, int H, int W, int coupling, int mix, int want_a1) {
  if (B <= 0 || C <= 0 || H <= 0 || W <= 0) return 0;
  const int R = choose_rows(B, C, H, W, coupling != 0, mix != 0, want_a1 != 0);
  if (tiled_scratch_floats(C, W, R, want_a1 ? 1 : 0, coupling != 0, mix != 0, nullptr, nullptr) * sizeof(float) > 200 * 1024) return 0;
  return (H + R - 1) / R;
}

extern "C" int nfdpm_flow_boundary_tiled(const float* in, int64_t in_bs, int squeeze_in, const float* pm, int64_t ldp,
                                         const float* bias3, const float* logs3, float* ld_part, const float* mt,
                                         const float* beta, float* y, int64_t y_bs, float* xs, int64_t xs_bs, void* a1,
                                         int a1_dtype, int64_t lda1, int B, int C, int H, int W, int inverse, int tiles,
                                         nfdpm_stream_t stream) {
  NFDPM_REQUIRE(in != nullptr, "nfdpm_flow_boundary_tiled: null input");
  NFDPM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && C % 2 == 0, "nfdpm_flow_boundary_tiled: bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
  NFDPM_REQUIRE((mt == nullptr) == (beta == nullptr), "nfdpm_flow_boundary_tiled: mt/beta must both be set or both NULL");
  NFDPM_REQUIRE(pm == nullptr || (bias3 && logs3 && ldp >= 9 * (int64_t)C), "nfdpm_flow_boundary_tiled: coupling source needs bias3/logs3/ldp");
  NFDPM_REQUIRE(!squeeze_in || (C % 4 == 0 && in_bs % 2 == 0 && ((uintptr_t)in % 8) == 0), "nfdpm_flow_boundary_tiled: squeeze source needs C %% 4 == 0 and 8-byte alignment");
  NFDPM_REQUIRE(a1 == nullptr || (lda1 % 8 == 0 && lda1 >= 9 * (int64_t)(C / 2) && ((uintptr_t)a1 % 16) == 0), "nfdpm_flow_boundary_tiled: bad im2col sink");
  NFDPM_REQUIRE(a1 == nullptr || a1_dtype == NFDPM_F32 || a1_dtype == NFDPM_BF16 || (a1_dtype == NFDPM_BF16X2 && lda1 % 32 == 0), "nfdpm_flow_boundary_tiled: bad a1 dtype");
  NFDPM_REQUIRE(y != nullptr || a1 != nullptr || xs != nullptr, "nfdpm_flow_boundary_tiled: no sink");
  NFDPM_REQUIRE((int64_t)B * C * H * W < (1ll << 31), "nfdpm_flow_boundary_tiled: tensor too large for 32-bit indices");
  const int want = nfdpm_flow_boundary_tiles(B, C, H, W, pm != nullptr, mt != nullptr, a1 != nullptr);
  NFDPM_REQUIRE(want > 0, "nfdpm_flow_boundary_tiled: one image row does not fit in shared memory (C=%d, W=%d)", C, W);
  NFDPM_REQUIRE(tiles == want, "nfdpm_flow_boundary_tiled: tiles=%d, nfdpm_flow_boundary_tiles() says %d", tiles, want);
  const int R = choose_rows(B, C, H, W, pm != nullptr, mt != nullptr, a1 != nullptr);
  BoundaryArgs a;
  a.in = in; a.in_bs = in_bs; a.pm = pm; a.ldp = ldp; a.bias3 = bias3; a.logs3 = logs3; a.ld_part = ld_part;
  a.mt = mt; a.beta = beta; a.y = y; a.y_bs = y_bs; a.xs = xs; a.xs_bs = xs_bs; a.a1 = a1; a.lda1 = lda1;
  a.B = B; a.C = C; a.H = H; a.W = W; a.squeeze_in = squeeze_in; a.inverse = inverse;
  boundary_fill_div(a);
  TileGeom g;
  g.R = R; g.T = tiles; g.halo = a1 != nullptr ? 1 : 0; g.Rv = R + 2 * g.halo; g.Pv = g.Rv * W;
  g.dPv = make_fastdiv(g.Pv); g.dT = make_fastdiv(tiles);
  g.bulk_m = (mt != nullptr && C % 4 == 0 && ((uintptr_t)mt % 16) == 0 && ((uintptr_t)beta % 16) == 0) ? 1 : 0;
  const size_t smem = tiled_scratch_floats(C, W, R, g.halo, pm != nullptr, mt != nullptr, nullptr, nullptr) * sizeof(float);
  int64_t items = (int64_t)g.Pv * (C / 2);
  if (a1 != nullptr && (int64_t)R * W * (lda1 / 8) > items) items = (int64_t)R * W * (lda1 / 8);
  if (mt != nullptr && (int64_t)g.Pv * ((C + 3) / 4) > items) items = (int64_t)g.Pv * ((C + 3) / 4);
  int threads = (int)((items + 31) / 32 * 32);
  if (threads > 1024) threads = 1024;
  if (threads < 128) threads = 128;
  cudaStream_t st = as_stream(stream);
  const int a1dt = a1 != nullptr ? a1_dtype : NFDPM_F32;
#define LAUNCH(CP, T)                                                                                               \
  do {                                                                                                              \
    static bool attr_set = false;                                                                                   \
    if (!attr_set) {                                                                                                \
      NFDPM_CUDA(cudaFuncSetAttribute(flow_boundary_tiled_kernel<CP, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      200 * 1024));                                                                 \
      attr_set = true;                                                                                              \
    }                                                                                                               \
    NFDPM_CUDA(launch_pdl(flow_boundary_tiled_kernel<CP, T>, dim3((unsigned)(B * tiles)), dim3(threads), smem, st, a, g)); \
  } while (0)
#define GO_CP(T) LAUNCH(true, T)
#define GO_NC(T) LAUNCH(false, T)
  if (pm != nullptr) NFDPM_A1_DISPATCH(a1dt, GO_CP);
  else NFDPM_A1_DISPATCH(a1dt, GO_NC);
#undef GO_CP
#undef GO_NC
#undef LAUNCH
  NFDPM_CHECK_LAUNCH("flow_boundary_tiled_kernel");
  return 0;
}
