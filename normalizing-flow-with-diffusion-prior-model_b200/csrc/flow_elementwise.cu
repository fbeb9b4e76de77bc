// HBM-bound kernels of the Glow flow path: fused ActNorm + invertible 1x1 conv ("channel mix", K-A /
// K-A^-1), stand-alone ActNorm, squeeze / unsqueeze, channel-block copies, data-dependent ActNorm
// statistics, the Gaussian prior with per-channel constants (K-G) and the accumulator finalize.
//
// Roofline: all of these read x once and write y once => 8 bytes per element (fp32 in + out);
// DESIGN.md §kernels lists the algorithmic bytes per image per StepFlow (8*C*P).
#include "common.cuh"
#include "wide_mix.cuh"

namespace nfdpm {

// ------------------------------------------------------------------------------------------------
// K-A register path: C <= 16 known at compile time.  One thread owns 4 consecutive pixels of one image
// and ALL C channels: C independent 128-bit loads in flight per thread, C*C*4 FMAs, C 128-bit stores.
// Warp lanes cover 32*4 consecutive pixels => every (warp, channel) access is one 512-byte run.
template <int C>
__global__ void __launch_bounds__(256) chanmix_small_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                            const float* __restrict__ mt,
                                                            const float* __restrict__ beta, int P4 /* P/4 */,
                                                            int64_t n_groups, int64_t xbs, int64_t ybs) {
  __shared__ float s_m[C * C + C];
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) s_m[i] = mt[i];
  for (int i = threadIdx.x; i < C; i += blockDim.x) s_m[C * C + i] = beta[i];
  __syncthreads();
  for (int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; g < n_groups; g += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = g / P4;
    const int p = (int)(g - b * P4) * 4;
    const float* xp = x + b * xbs + p;
    float* yp = y + b * ybs + p;
    const int64_t P = (int64_t)P4 * 4;
    float4 xi[C];
#pragma unroll
    for (int i = 0; i < C; ++i) xi[i] = ldg_stream4(xp + i * P);
    float4 acc[C];
#pragma unroll
    for (int o = 0; o < C; ++o) {
      const float bo = s_m[C * C + o];
      acc[o] = make_float4(bo, bo, bo, bo);
    }
#pragma unroll
    for (int i = 0; i < C; ++i) {
#pragma unroll
      for (int o = 0; o < C; ++o) {
        const float w = s_m[i * C + o];
        acc[o].x = fmaf(w, xi[i].x, acc[o].x);
        acc[o].y = fmaf(w, xi[i].y, acc[o].y);
        acc[o].z = fmaf(w, xi[i].z, acc[o].z);
        acc[o].w = fmaf(w, xi[i].w, acc[o].w);
      }
    }
#pragma unroll
    for (int o = 0; o < C; ++o) stg_stream4(yp + o * P, acc[o]);
  }
}

// K-A generic path: any C (<= 192).  CTA = 256 threads = TPG pixel groups x (256/TPG) output slices; the x tile
// [C][TPG*V] and the CxC matrix live in shared memory; each thread produces 4 output channels x V pixels at a
// time.  V = 4 (128-bit access) when P % 4 == 0, else V = 1.  TPG = 64 normally, 16 for wide C (smem budget).
template <int V, int TPG>
__global__ void __launch_bounds__(256) chanmix_generic_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                              const float* __restrict__ mt,
                                                              const float* __restrict__ beta, int C, int P,
                                                              int64_t n_groups, int64_t xbs, int64_t ybs) {
  extern __shared__ __align__(16) float sm[];
  const int Cp = (C + 3) & ~3;
  float* s_m = sm;                 // [C][Cp]  (row = input channel, col = output channel, zero padded)
  float* s_b = s_m + C * Cp;       // [Cp]
  float* s_x = s_b + Cp;           // [C][TPG*V]
  constexpr int NQ = 256 / TPG;    // output slices
  for (int i = threadIdx.x; i < C * Cp; i += 256) {
    const int r = i / Cp, c = i - r * Cp;
    s_m[i] = (c < C) ? mt[r * C + c] : 0.f;
  }
  for (int i = threadIdx.x; i < Cp; i += 256) s_b[i] = (i < C) ? beta[i] : 0.f;
  const int pg = threadIdx.x % TPG;   // pixel group within tile (consecutive lanes -> consecutive pixels)
  const int q = threadIdx.x / TPG;    // output slice
  const int PV = P / V;
  for (int64_t tile = blockIdx.x; tile * TPG < n_groups; tile += gridDim.x) {
    __syncthreads();  // s_m ready (first iteration) / previous tile consumed
    // ---- stage x tile
    for (int idx = threadIdx.x; idx < C * TPG; idx += 256) {
      const int i = idx / TPG, gl = idx - i * TPG;
      const int64_t g = tile * TPG + gl;
      if constexpr (V == 4) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g < n_groups) {
          const int64_t b = g / PV;
          const int p = (int)(g - b * PV) * 4;
          v = ldg_stream4(x + b * xbs + (int64_t)i * P + p);
        }
        *reinterpret_cast<float4*>(s_x + (i * TPG + gl) * 4) = v;
      } else {
        float v = 0.f;
        if (g < n_groups) {
          const int64_t b = g / PV;
          const int p = (int)(g - b * PV);
          v = __ldg(x + b * xbs + (int64_t)i * P + p);
        }
        s_x[i * TPG + gl] = v;
      }
    }
    __syncthreads();
    const int64_t g = tile * TPG + pg;
    const bool live = g < n_groups;
    int64_t b = 0;
    int p = 0;
    if (live) {
      b = g / PV;
      p = (int)(g - b * PV) * V;
    }
    for (int o0 = q * 4; o0 < C; o0 += 4 * NQ) {
      float acc[4][V];
#pragma unroll
      for (int j = 0; j < 4; ++j)
#pragma unroll
        for (int v = 0; v < V; ++v) acc[j][v] = s_b[o0 + j];
      for (int i = 0; i < C; ++i) {
        const float4 w = *reinterpret_cast<const float4*>(s_m + i * Cp + o0);
        float xv[V];
        if constexpr (V == 4) {
          const float4 t4 = *reinterpret_cast<const float4*>(s_x + (i * TPG + pg) * 4);
          xv[0] = t4.x; xv[1] = t4.y; xv[2] = t4.z; xv[3] = t4.w;
        } else {
          xv[0] = s_x[i * TPG + pg];
        }
#pragma unroll
        for (int v = 0; v < V; ++v) {
          acc[0][v] = fmaf(w.x, xv[v], acc[0][v]);
          acc[1][v] = fmaf(w.y, xv[v], acc[1][v]);
          acc[2][v] = fmaf(w.z, xv[v], acc[2][v]);
          acc[3][v] = fmaf(w.w, xv[v], acc[3][v]);
        }
      }
      if (live) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (o0 + j < C) {
            float* yp = y + b * ybs + (int64_t)(o0 + j) * P + p;
            if constexpr (V == 4) stg_stream4(yp, make_float4(acc[j][0], acc[j][1], acc[j][2], acc[j][3]));
            else *yp = acc[j][0];
          }
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
__global__ void actnorm_apply_kernel(const float* __restrict__ x, float* __restrict__ y, const float* __restrict__ s,
                                     const float* __restrict__ bsv, int C, int P, int64_t n, int inverse) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)((i / P) % C);
    const float sc = __ldg(s + c), bi = __ldg(bsv + c);
    const float v = x[i];
    y[i] = inverse ? v * expf(-sc) - bi : expf(sc) * (v + bi);
  }
}

// Squeeze: out[b, c*4+h1*2+w1, h, w] = in[b, c, 2h+h1, 2w+w1].  One thread per (b, c, h, w-pair) of the
// OUTPUT grid reading a 2x2 input patch... mapped so that input reads are 8-byte and output writes are
// coalesced along w for each of the four output channels.
__global__ void squeeze_kernel(const float* __restrict__ x, float* __restrict__ y, int C, int H, int W, int64_t n,
                               int64_t xbs, int64_t ybs) {
  const int Ho = H >> 1, Wo = W >> 1;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(i % Wo);
    int64_t r = i / Wo;
    const int h = (int)(r % Ho);
    r /= Ho;
    const int c = (int)(r % C);
    const int64_t b = r / C;
    const float* xp = x + b * xbs + ((int64_t)c * H + 2 * h) * W + 2 * w;
    const float2 top = *reinterpret_cast<const float2*>(xp);
    const float2 bot = *reinterpret_cast<const float2*>(xp + W);
    float* yp = y + b * ybs + ((int64_t)(c * 4) * Ho + h) * Wo + w;
    const int64_t cs = (int64_t)Ho * Wo;
    yp[0] = top.x;
    yp[cs] = top.y;
    yp[2 * cs] = bot.x;
    yp[3 * cs] = bot.y;
  }
}

// Unsqueeze: out[b, c, 2h+c1, 2w+c2] = in[b, c*4+c1*2+c2, h, w]; x is [B,C,H,W] with C = 4*Co.
__global__ void unsqueeze_kernel(const float* __restrict__ x, float* __restrict__ y, int Co, int H, int W, int64_t n,
                                 int64_t xbs, int64_t ybs) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int w = (int)(i % W);
    int64_t r = i / W;
    const int h = (int)(r % H);
    r /= H;
    const int c = (int)(r % Co);
    const int64_t b = r / Co;
    const int64_t cs = (int64_t)H * W;
    const float* xp = x + b * xbs + ((int64_t)(c * 4) * H + h) * W + w;
    float* yp = y + b * ybs + ((int64_t)c * 2 * H + 2 * h) * (2 * W) + 2 * w;
    *reinterpret_cast<float2*>(yp) = make_float2(xp[0], xp[cs]);
    *reinterpret_cast<float2*>(yp + 2 * W) = make_float2(xp[2 * cs], xp[3 * cs]);
  }
}

__global__ void copy_channels_kernel(const float* __restrict__ src, float* __restrict__ dst, int64_t per_b /*Cn*P*/,
                                     int64_t n, int64_t sbs, int64_t dbs) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t b = i / per_b, r = i - b * per_b;
    dst[b * dbs + r] = src[b * sbs + r];
  }
}

// ------------------------------------------------------------------------------------------------
// Data-dependent ActNorm statistics: one CTA per channel, fp64 two-pass (mean, then centred sum of
// squares) so the result matches torch's fp32 Welford to ~1e-7 regardless of the mean/std ratio.
__global__ void __launch_bounds__(256) channel_stats_kernel(const float* __restrict__ x, int layout, int B, int C,
                                                            int P, int64_t xs, float* __restrict__ scale_out,
                                                            float* __restrict__ bias_out) {
  __shared__ double sh[8];
  __shared__ double s_mean;
  const int c = blockIdx.x;
  const int64_t n = (int64_t)B * P;
  auto at = [&](int64_t m) -> float {
    if (layout == 0) {
      const int64_t b = m / P, p = m - b * P;
      return x[b * xs + (int64_t)c * P + p];
    }
    return x[m * xs + c];
  };
  double s = 0.0;
  for (int64_t m = threadIdx.x; m < n; m += 256) s += (double)at(m);
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += sh[i];
    s_mean = t / (double)n;
  }
  __syncthreads();
  const double mean = s_mean;
  double q = 0.0;
  for (int64_t m = threadIdx.x; m < n; m += 256) {
    const double d = (double)at(m) - mean;
    q += d * d;
  }
  q = warp_sum(q);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = q;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += sh[i];
    const double var = t / (double)(n - 1);  // unbiased, torch.std default (transforms.py:76)
    const float sd = (float)sqrt(var);
    scale_out[c] = -logf(sd + 1e-6f);
    bias_out[c] = -(float)mean;
  }
}

// ------------------------------------------------------------------------------------------------
// K-G: Gaussian log-density with per-channel constants.  One CTA per image.
__global__ void __launch_bounds__(256) gauss_logp_const_kernel(const float* __restrict__ z,
                                                               const float* __restrict__ bias,
                                                               const float* __restrict__ logs,
                                                               float* __restrict__ out, int C, int P) {
  __shared__ float sh[256];
  const int b = blockIdx.x;
  const float* zp = z + (int64_t)b * C * P;
  const float LOG2PI = 1.8378770664093453f;
  float acc = 0.f;
  for (int i = threadIdx.x; i < C * P; i += 256) {
    const int c = i / P;
    float mean = 0.f, lg = 0.f;
    if (bias != nullptr) {
      mean = __ldg(bias + c) * expf(3.f * __ldg(logs + c));
      lg = __ldg(bias + C + c) * expf(3.f * __ldg(logs + C + c));
    }
    const float d = zp[i] - mean;
    acc += -0.5f * (LOG2PI + 2.f * lg + d * d * expf(-2.f * lg));
  }
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[b] = sh[0];
}

// out = mean + exp(lg)*T*eps per channel; T = temp_b[b] or `temperature`; eps from `eps` or, with `seeds`, drawn by
// philox_normal(seeds[b], stream_id, c*P + p) and copied to eps_out (may be NULL)
__global__ void gauss_sample_const_kernel(const float* __restrict__ eps, const int64_t* __restrict__ seeds,
                                          uint32_t stream_id, const float* __restrict__ bias,
                                          const float* __restrict__ logs, float temperature,
                                          const float* __restrict__ temp_b, float* __restrict__ eps_out,
                                          float* __restrict__ out, int C, int P, int64_t n) {
  const int64_t CP = (int64_t)C * P;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)((i / P) % C);
    float mean = 0.f, lg = 0.f;
    if (bias != nullptr) {
      mean = __ldg(bias + c) * expf(3.f * __ldg(logs + c));
      lg = __ldg(bias + C + c) * expf(3.f * __ldg(logs + C + c));
    }
    float e, T = temperature;
    if (seeds != nullptr || temp_b != nullptr) {
      const int64_t b = i / CP;
      if (temp_b != nullptr) T = temp_b[b];
      if (seeds != nullptr) {
        e = philox_normal((uint64_t)seeds[b], stream_id, (uint32_t)(i - b * CP));
        if (eps_out != nullptr) eps_out[i] = e;
      } else {
        e = eps[i];
      }
    } else {
      e = eps[i];
    }
    out[i] = __fmaf_rn(__fmul_rn(expf(lg), T), e, mean);   // the roundings spelled out: the same bits in every branch
  }
}

// acc[b] += sum_r part[r*B+b] + sum_j cmul[j]*cval[j]
template <typename T>
__global__ void accumulate_kernel(T* __restrict__ acc, const float* __restrict__ part, int R, int B,
                                  const float* __restrict__ cval, const float* __restrict__ cmul, int nc) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double s = 0.0;
  for (int j = 0; j < nc; ++j) s += (double)cmul[j] * (double)cval[j];
  for (int r = 0; r < R; ++r) s += (double)part[(int64_t)r * B + b];
  acc[b] = (T)((double)acc[b] + s);
}

static int grid_for(int64_t n, int tpb, int cap = 148 * 16) {
  int64_t g = cdiv64(n, tpb);
  if (g < 1) g = 1;
  return (int)(g > cap ? cap : g);
}

}  // namespace nfdpm

using namespace nfdpm;

extern "C" int nfdpm_channel_mix(const float* x, float* y, const float* mt, const float* beta, int B, int C, int P,
                                 int64_t xbs, int64_t ybs, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x && y && mt && beta, "nfdpm_channel_mix: null pointer");
  NFDPM_REQUIRE(B > 0 && C > 0 && P > 0, "nfdpm_channel_mix: bad shape B=%d C=%d P=%d", B, C, P);
  NFDPM_REQUIRE(C <= kWideMixMax, "nfdpm_channel_mix: C=%d > %d unsupported", C, kWideMixMax);
  cudaStream_t st = as_stream(stream);
  if (C > kWideMixMin) return chanmix_wide(x, y, mt, beta, B, C, P, xbs, ybs, st);
  const bool vec = (P % 4 == 0) && (xbs % 4 == 0) && (ybs % 4 == 0) && (((uintptr_t)x | (uintptr_t)y) % 16 == 0);
  if (vec && (C == 4 || C == 8 || C == 12 || C == 16)) {
    const int64_t ng = (int64_t)B * (P / 4);
    const int grid = grid_for(ng, 256, 148 * 8);
    switch (C) {
      case 4: chanmix_small_kernel<4><<<grid, 256, 0, st>>>(x, y, mt, beta, P / 4, ng, xbs, ybs); break;
      case 8: chanmix_small_kernel<8><<<grid, 256, 0, st>>>(x, y, mt, beta, P / 4, ng, xbs, ybs); break;
      case 12: chanmix_small_kernel<12><<<grid, 256, 0, st>>>(x, y, mt, beta, P / 4, ng, xbs, ybs); break;
      default: chanmix_small_kernel<16><<<grid, 256, 0, st>>>(x, y, mt, beta, P / 4, ng, xbs, ybs); break;
    }
    NFDPM_CHECK_LAUNCH("chanmix_small_kernel");
    return 0;
  }
  const int V = vec ? 4 : 1;
  const int Cp = (C + 3) & ~3;
  const int TPG = (C > 64) ? 16 : 64;
  const size_t smem = sizeof(float) * ((size_t)C * Cp + Cp + (size_t)C * TPG * V);
  NFDPM_REQUIRE(smem <= 227 * 1024, "nfdpm_channel_mix: C=%d needs %zu bytes of shared memory", C, smem);
  const int64_t ng = (int64_t)B * P / V;
  const int grid = grid_for(cdiv64(ng, TPG), 1, 148 * 4);
  // the opt-in shared-memory limit is raised once per instantiation (never during a stream capture)
#define LAUNCH(VV, TT)                                                                                           \
  do {                                                                                                           \
    static bool attr_set = false;                                                                                \
    if (!attr_set) {                                                                                             \
      NFDPM_CUDA(cudaFuncSetAttribute(chanmix_generic_kernel<VV, TT>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      227 * 1024));                                                              \
      attr_set = true;                                                                                           \
    }                                                                                                            \
    chanmix_generic_kernel<VV, TT><<<grid, 256, smem, st>>>(x, y, mt, beta, C, P, ng, xbs, ybs);                 \
  } while (0)
  if (V == 4) { if (TPG == 64) LAUNCH(4, 64); else LAUNCH(4, 16); }
  else { if (TPG == 64) LAUNCH(1, 64); else LAUNCH(1, 16); }
#undef LAUNCH
  NFDPM_CHECK_LAUNCH("chanmix_generic_kernel");
  return 0;
}

extern "C" int nfdpm_actnorm_apply(const float* x, float* y, const float* scale, const float* bias, int B, int C,
                                   int P, int inverse, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x && y && scale && bias, "nfdpm_actnorm_apply: null pointer");
  NFDPM_REQUIRE(B > 0 && C > 0 && P > 0, "nfdpm_actnorm_apply: bad shape");
  const int64_t n = (int64_t)B * C * P;
  actnorm_apply_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(x, y, scale, bias, C, P, n, inverse);
  NFDPM_CHECK_LAUNCH("actnorm_apply_kernel");
  return 0;
}

extern "C" int nfdpm_channel_stats(const float* x, int layout, int B, int C, int P, int64_t xs, float* scale_out,
                                   float* bias_out, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x && scale_out && bias_out, "nfdpm_channel_stats: null pointer");
  NFDPM_REQUIRE(B > 0 && C > 0 && P > 0 && (int64_t)B * P > 1, "nfdpm_channel_stats: need at least 2 samples per channel");
  NFDPM_REQUIRE(layout == 0 || layout == 1, "nfdpm_channel_stats: bad layout %d", layout);
  channel_stats_kernel<<<C, 256, 0, as_stream(stream)>>>(x, layout, B, C, P, xs, scale_out, bias_out);
  NFDPM_CHECK_LAUNCH("channel_stats_kernel");
  return 0;
}

extern "C" int nfdpm_squeeze(const float* x, float* y, int B, int C, int H, int W, int64_t xbs, int64_t ybs,
                             nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x && y, "nfdpm_squeeze: null pointer");
  NFDPM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "nfdpm_squeeze: bad shape");
  NFDPM_REQUIRE(H % 2 == 0 && W % 2 == 0, "nfdpm_squeeze: H=%d, W=%d must be even", H, W);
  NFDPM_REQUIRE(xbs % 2 == 0 && ((uintptr_t)x % 8) == 0, "nfdpm_squeeze: input must be 8-byte aligned");
  const int64_t n = (int64_t)B * C * (H / 2) * (W / 2);
  squeeze_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(x, y, C, H, W, n, xbs, ybs);
  NFDPM_CHECK_LAUNCH("squeeze_kernel");
  return 0;
}

extern "C" int nfdpm_unsqueeze(const float* x, float* y, int B, int C, int H, int W, int64_t xbs, int64_t ybs,
                               nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x && y, "nfdpm_unsqueeze: null pointer");
  NFDPM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "nfdpm_unsqueeze: bad shape");
  NFDPM_REQUIRE(C % 4 == 0, "nfdpm_unsqueeze: C=%d must be a multiple of 4", C);
  NFDPM_REQUIRE(ybs % 2 == 0 && ((uintptr_t)y % 8) == 0, "nfdpm_unsqueeze: output must be 8-byte aligned");
  const int64_t n = (int64_t)B * (C / 4) * H * W;
  unsqueeze_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(x, y, C / 4, H, W, n, xbs, ybs);
  NFDPM_CHECK_LAUNCH("unsqueeze_kernel");
  return 0;
}

extern "C" int nfdpm_copy_channels(const float* src, float* dst, int B, int Cn, int P, int64_t sbs, int64_t dbs,
                                   nfdpm_stream_t stream) {
  NFDPM_REQUIRE(src && dst, "nfdpm_copy_channels: null pointer");
  NFDPM_REQUIRE(B > 0 && Cn > 0 && P > 0, "nfdpm_copy_channels: bad shape");
  const int64_t per_b = (int64_t)Cn * P, n = per_b * B;
  copy_channels_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(src, dst, per_b, n, sbs, dbs);
  NFDPM_CHECK_LAUNCH("copy_channels_kernel");
  return 0;
}

extern "C" int nfdpm_gauss_logp_const(const float* z, const float* bias, const float* logs, float* logp_part, int B,
                                      int C, int P, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(z && logp_part, "nfdpm_gauss_logp_const: null pointer");
  NFDPM_REQUIRE((bias == nullptr) == (logs == nullptr), "nfdpm_gauss_logp_const: bias/logs must both be set or both NULL");
  NFDPM_REQUIRE(B > 0 && C > 0 && P > 0, "nfdpm_gauss_logp_const: bad shape");
  gauss_logp_const_kernel<<<B, 256, 0, as_stream(stream)>>>(z, bias, logs, logp_part, C, P);
  NFDPM_CHECK_LAUNCH("gauss_logp_const_kernel");
  return 0;
}

extern "C" int nfdpm_gauss_sample_const_ex(const float* eps, const int64_t* seeds, uint32_t stream_id, const float* bias,
                                           const float* logs, float temperature, const float* temp_b, float* eps_out,
                                           float* out, int B, int C, int P, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(out, "nfdpm_gauss_sample_const_ex: null pointer");
  NFDPM_REQUIRE((eps == nullptr) != (seeds == nullptr), "nfdpm_gauss_sample_const_ex: give exactly one of eps / seeds");
  NFDPM_REQUIRE(seeds != nullptr || (stream_id == 0 && eps_out == nullptr),
                "nfdpm_gauss_sample_const_ex: stream_id / eps_out need seeds");
  NFDPM_REQUIRE((bias == nullptr) == (logs == nullptr), "nfdpm_gauss_sample_const_ex: bias/logs must both be set or both NULL");
  NFDPM_REQUIRE(B > 0 && C > 0 && P > 0, "nfdpm_gauss_sample_const_ex: bad shape");
  NFDPM_REQUIRE((int64_t)C * P <= 0xFFFFFFFFll, "nfdpm_gauss_sample_const_ex: more than 2^32 drawn elements per image");
  const int64_t n = (int64_t)B * C * P;
  gauss_sample_const_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(eps, seeds, stream_id, bias, logs, temperature,
                                                                              temp_b, eps_out, out, C, P, n);
  NFDPM_CHECK_LAUNCH("gauss_sample_const_kernel");
  return 0;
}

extern "C" int nfdpm_gauss_sample_const(const float* eps, const float* bias, const float* logs, float temperature,
                                        float* out, int B, int C, int P, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(eps && out, "nfdpm_gauss_sample_const: null pointer");
  return nfdpm_gauss_sample_const_ex(eps, nullptr, 0u, bias, logs, temperature, nullptr, nullptr, out, B, C, P, stream);
}

extern "C" int nfdpm_accumulate(void* acc, int acc_dtype, const float* part, int R, int B, const float* cval,
                                const float* cmul, int nc, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(acc, "nfdpm_accumulate: null accumulator");
  NFDPM_REQUIRE(B > 0 && R >= 0 && nc >= 0, "nfdpm_accumulate: bad sizes");
  NFDPM_REQUIRE(R == 0 || part, "nfdpm_accumulate: null partials");
  NFDPM_REQUIRE(nc == 0 || (cval && cmul), "nfdpm_accumulate: null constants");
  const int grid = (B + 127) / 128;
  if (acc_dtype == NFDPM_F64)
    accumulate_kernel<double><<<grid, 128, 0, as_stream(stream)>>>((double*)acc, part, R, B, cval, cmul, nc);
  else if (acc_dtype == NFDPM_F32)
    accumulate_kernel<float><<<grid, 128, 0, as_stream(stream)>>>((float*)acc, part, R, B, cval, cmul, nc);
  else
    return fail("nfdpm_accumulate: accumulator dtype %d not supported (fp32/fp64 only)", acc_dtype);
  NFDPM_CHECK_LAUNCH("accumulate_kernel");
  return 0;
}
