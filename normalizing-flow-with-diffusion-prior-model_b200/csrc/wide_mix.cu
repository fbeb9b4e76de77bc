// Channel-mix kernels of the wide levels, 192 < C <= 1024 channels (the final levels of L6 / L7 models on RGB input):
//   chanmix_wide_kernel        K-A / K-A^-1 (and, transposed, dx = W^T du of the backward): the C x C matrix streams
//                              through shared memory in chunks of kKC input channels, output channels tiled over CTAs
//   mix_bwd_part_wide_kernel   the per-image partials of d(W^), d(b^) of nfdpm_mix_bwd, 32 x 32 elements per CTA
//   mix_reduce_wide_kernel / mix_inv_sb_wide_kernel / mix_inv_gemm_wide_kernel
//                              nfdpm_mix_inv_param_grad with its two C^3 products spread over CTAs
// The single-pass kernels keep the whole matrix (or a C x C temporary) in shared memory, which caps them at 192 channels.
// These levels carry under 1 % of a model's FLOPs (DESIGN.md §8): the kernels aim at a grid that covers the GPU at a few
// pixels per image.  Every sum runs in a fixed order (no atomics): the results are bitwise reproducible.
#include "wide_mix.cuh"

namespace nfdpm {

static constexpr int kKC = 32;   // input channels per shared-memory chunk of the matrix
static constexpr int kOT = 32;   // output channels per CTA of chanmix_wide_kernel (one per lane)
static constexpr int kPG = 4;    // pixel groups per CTA of chanmix_wide_kernel (one per warp)

// The im2col-row gradient of the coupling network (nfdpm_mix_bwd's da1, NULL: none) and the image geometry
struct Col2im {
  const float* da1; int64_t lda1;
  int Ch, H, W;
};

// v = du[b, c, p]; for c < Ch adds the col2im of da1 as mix_bwd_kernel does: du + ((0 + tap 0) + tap 1 ...) over the
// taps that fall inside the image
__device__ __forceinline__ float with_col2im(float v, const Col2im& ci, int64_t b, int c, int p) {
  if (ci.da1 == nullptr || c >= ci.Ch) return v;
  const int P = ci.H * ci.W, py = p / ci.W, px = p - py * ci.W;
  const float* dab = ci.da1 + b * P * ci.lda1 + c * 9;
  float acc = 0.f;
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const int yy = py - (tap / 3 - 1), xx = px - (tap % 3 - 1);
    if (yy >= 0 && yy < ci.H && xx >= 0 && xx < ci.W) acc += __ldg(dab + (int64_t)(yy * ci.W + xx) * ci.lda1 + tap);
  }
  return v + acc;
}

// out[b, r, p] = init(r) + sum_k M(r, k) in[b, k, p], k ascending (fmaf chain, as chanmix_generic_kernel and the dx loop
// of mix_bwd_kernel).  M(r, k) = mt[k*C + r] (K-A: r is the output channel, init = beta[r]) or, TR, mt[r*C + k] (dx = W^T du:
// init 0, the input carries the col2im).  CTA = kOT output channels (lanes) x kPG groups of V consecutive pixels (warps);
// grid (pixel-group tiles, output-channel tiles).
template <int V, bool TR>
__global__ void __launch_bounds__(128) chanmix_wide_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                           const float* __restrict__ mt, const float* __restrict__ beta,
                                                           int C, int P, int64_t n_groups, int64_t xbs, int64_t ybs,
                                                           const Col2im ci) {
  __shared__ float s_m[kKC][kOT + 1];          // [k][r]
  __shared__ float s_x[kKC][kPG * V];          // [k][group * V + v]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int o0 = blockIdx.y * kOT, o = o0 + lane;
  const int64_t g0 = (int64_t)blockIdx.x * kPG, g = g0 + warp;
  const int PV = P / V;
  const float init = (beta != nullptr && o < C) ? __ldg(beta + o) : 0.f;
  float acc[V];
#pragma unroll
  for (int v = 0; v < V; ++v) acc[v] = init;
  for (int i0 = 0; i0 < C; i0 += kKC) {
    const int kn = min(kKC, C - i0);
    __syncthreads();                           // the previous chunk is consumed
    for (int idx = threadIdx.x; idx < kKC * kOT; idx += 128) {
      const int k = TR ? idx % kKC : idx / kOT, r = TR ? idx / kKC : idx % kOT;   // lanes walk the unit-stride index
      float v = 0.f;
      if (k < kn && o0 + r < C)
        v = TR ? __ldg(mt + (int64_t)(o0 + r) * C + i0 + k) : __ldg(mt + (int64_t)(i0 + k) * C + o0 + r);
      s_m[k][r] = v;
    }
    for (int idx = threadIdx.x; idx < kKC * kPG * V; idx += 128) {
      const int k = idx / (kPG * V), e = idx - k * (kPG * V), gl = e / V;
      const int64_t gg = g0 + gl;
      float v = 0.f;
      if (k < kn && gg < n_groups) {
        const int64_t b = gg / PV;
        const int p = (int)(gg - b * PV) * V + (e - gl * V);
        v = with_col2im(__ldg(x + b * xbs + (int64_t)(i0 + k) * P + p), ci, b, i0 + k, p);
      }
      s_x[k][e] = v;
    }
    __syncthreads();
    for (int k = 0; k < kn; ++k) {
      const float w = s_m[k][lane];
#pragma unroll
      for (int v = 0; v < V; ++v) acc[v] = fmaf(w, s_x[k][warp * V + v], acc[v]);
    }
  }
  if (g < n_groups && o < C) {
    const int64_t b = g / PV;
    float* yp = y + b * ybs + (int64_t)o * P + (g - b * PV) * V;
    if constexpr (V == 4) stg_stream4(yp, make_float4(acc[0], acc[1], acc[2], acc[3]));
    else *yp = acc[0];
  }
}

// part[b][o*C + i] = sum_p du[b, o, p] x[b, i, p] and part[b][C*C + o] = sum_p du[b, o, p], du with the col2im, p ascending
// from 0 (the order of mix_bwd_kernel's per-thread branch).  Column i = C of the last tile is the all-ones row:
// fmaf(d, 1, acc) rounds d + acc once, as acc += d does.  CTA = 32 (o) x 32 (i) elements of one image, 4 per thread;
// pixels stream through shared memory in chunks of 32.  Grid (i tiles over C + 1, o tiles, images).
__global__ void __launch_bounds__(256) mix_bwd_part_wide_kernel(const float* __restrict__ du, int64_t du_bs,
                                                                const float* __restrict__ x, int64_t x_bs,
                                                                float* __restrict__ part, int C, int P, const Col2im ci) {
  constexpr int PK = 32;
  __shared__ float s_d[32][PK + 1];   // [o][p]
  __shared__ float s_x[32][PK + 1];   // [i][p]
  const int b = blockIdx.z, o0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const float* dub = du + (int64_t)b * du_bs;
  const float* xb = x + (int64_t)b * x_bs;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int p0 = 0; p0 < P; p0 += PK) {
    const int pn = min(PK, P - p0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < 32 * PK; idx += 256) {
      const int r = idx / PK, pl = idx % PK;    // lanes walk pixels
      float dv = 0.f, xv = 0.f;
      if (pl < pn) {
        const int p = p0 + pl;
        if (o0 + r < C) dv = with_col2im(__ldg(dub + (int64_t)(o0 + r) * P + p), ci, b, o0 + r, p);
        if (i0 + r < C) xv = __ldg(xb + (int64_t)(i0 + r) * P + p);
        else if (i0 + r == C) xv = 1.f;
      }
      s_d[r][pl] = dv;
      s_x[r][pl] = xv;
    }
    __syncthreads();
    for (int pl = 0; pl < pn; ++pl) {
      const float xv = s_x[tx][pl];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = fmaf(s_d[ty + 8 * j][pl], xv, acc[j]);
    }
  }
  float* pb = part + (int64_t)b * ((int64_t)C * C + C);
  const int i = i0 + tx;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int o = o0 + ty + 8 * j;
    if (o < C && i < C) pb[(int64_t)o * C + i] = acc[j];
    else if (o < C && i == C) pb[(int64_t)C * C + o] = acc[j];
  }
}

// out[e] = sum_b part[b*n + e], b ascending (mix_reduce_partials' order, spread over the grid)
__global__ void __launch_bounds__(256) mix_reduce_wide_kernel(const float* __restrict__ part, int B, int n,
                                                              float* __restrict__ out) {
  for (int e = blockIdx.x * 256 + threadIdx.x; e < n; e += gridDim.x * 256) {
    float acc = 0.f;
    int b = 0;
    for (; b + 8 <= B; b += 8) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __ldcg(part + (int64_t)(b + j) * n + e);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc += v[j];
    }
    for (; b < B; ++b) acc += __ldcg(part + (int64_t)b * n + e);
    out[e] = acc;
  }
}

// d_bias = -g;  d_scale_c = -e^{-s_c} sum_j G_cj winv_cj (+ P dld_sum).  One warp per channel, lanes over j, fixed
// shuffle tree.
__global__ void __launch_bounds__(256) mix_inv_sb_wide_kernel(const float* __restrict__ Gg, int C,
                                                              const float* __restrict__ s, const float* __restrict__ winv,
                                                              const float* __restrict__ dld_sum, float P,
                                                              float* __restrict__ d_scale, float* __restrict__ d_bias) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  if (d_bias != nullptr && lane == 0) d_bias[c] = -Gg[(int64_t)C * C + c];
  if (d_scale == nullptr) return;
  float acc = 0.f;
  for (int j = lane; j < C; j += 32) acc = fmaf(Gg[(int64_t)c * C + j], winv[(int64_t)c * C + j], acc);
  acc = warp_sum(acc);
  if (lane == 0) {
    float v = -expf(-s[c]) * acc;
    if (dld_sum != nullptr) v += dld_sum[0] * P;
    d_scale[c] = v;
  }
}

// out[r*C + n] = epilogue(sum_k A[r*sar + k*sak] Bm[k*sbk + n*sbn]), k ascending from 0 (the orders of
// mix_inv_param_grad_kernel).  TMAT: T = diag(e^-s) G W^-T, out = e^{-s_r} acc.  Otherwise dW = -W^-T T (+ P dld_sum
// W^-T): out = -acc + P dld_sum winv[n*C + r].  CTA = 32 x 32 outputs, 4 per thread; k in chunks of 32.
template <bool TMAT>
__global__ void __launch_bounds__(256) mix_inv_gemm_wide_kernel(const float* __restrict__ A, int64_t sar, int64_t sak,
                                                                const float* __restrict__ Bm, int64_t sbk, int64_t sbn,
                                                                float* __restrict__ out, int C, const float* __restrict__ s,
                                                                const float* __restrict__ winv,
                                                                const float* __restrict__ dld_sum, float P) {
  __shared__ float s_a[32][kKC + 1];   // [r][k]
  __shared__ float s_b[32][kKC + 1];   // [n][k]
  const int r0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  for (int k0 = 0; k0 < C; k0 += kKC) {
    const int kn = min(kKC, C - k0);
    __syncthreads();
    for (int idx = threadIdx.x; idx < 32 * kKC; idx += 256) {
      int r = idx % 32, k = idx / 32;          // lanes walk r when A's unit stride is r ...
      if (sak == 1) { k = idx % 32; r = idx / 32; }   // ... and k when it is k
      s_a[r][k] = (k < kn && r0 + r < C) ? A[(r0 + r) * sar + (k0 + k) * sak] : 0.f;
      int n = idx % 32, kb = idx / 32;
      if (sbk == 1) { kb = idx % 32; n = idx / 32; }
      s_b[n][kb] = (kb < kn && n0 + n < C) ? Bm[(k0 + kb) * sbk + (n0 + n) * sbn] : 0.f;
    }
    __syncthreads();
    for (int k = 0; k < kn; ++k) {
      const float bv = s_b[tx][k];
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = fmaf(s_a[ty + 8 * j][k], bv, acc[j]);
    }
  }
  const int n = n0 + tx;
  if (n >= C) return;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int r = r0 + ty + 8 * j;
    if (r >= C) continue;
    float v;
    if constexpr (TMAT) {
      v = expf(s ? -s[r] : 0.f) * acc[j];
    } else {
      v = -acc[j];
      if (dld_sum != nullptr) v += dld_sum[0] * P * winv[(int64_t)n * C + r];
    }
    out[(int64_t)r * C + n] = v;
  }
}

static int grid_blocks(int64_t n, int per_block, int cap) {
  const int64_t g = (n + per_block - 1) / per_block;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

int chanmix_wide(const float* x, float* y, const float* mt, const float* beta, int B, int C, int P, int64_t xbs,
                 int64_t ybs, cudaStream_t st) {
  const bool vec = (P % 4 == 0) && (xbs % 4 == 0) && (ybs % 4 == 0) && (((uintptr_t)y) % 16 == 0);
  const int V = vec ? 4 : 1;
  const int64_t ng = (int64_t)B * P / V;
  const dim3 grid((unsigned)cdiv64(ng, kPG), (unsigned)cdiv64(C, kOT));
  const Col2im none{nullptr, 0, 0, 1, 1};
  if (V == 4) chanmix_wide_kernel<4, false><<<grid, 128, 0, st>>>(x, y, mt, beta, C, P, ng, xbs, ybs, none);
  else chanmix_wide_kernel<1, false><<<grid, 128, 0, st>>>(x, y, mt, beta, C, P, ng, xbs, ybs, none);
  NFDPM_CHECK_LAUNCH("chanmix_wide_kernel");
  return 0;
}

int mix_bwd_wide(const float* du, int64_t du_bs, const float* da1, int64_t lda1, const float* x, int64_t x_bs,
                 const float* mt, float* dx, int64_t dx_bs, float* part, int B, int C, int H, int W, cudaStream_t st) {
  NFDPM_REQUIRE(B <= 65535, "nfdpm_mix_bwd: B=%d > 65535 images at %d channels", B, C);
  const int P = H * W;
  const Col2im ci{da1, lda1, C / 2, H, W};
  const bool vec = (P % 4 == 0) && (dx_bs % 4 == 0) && (((uintptr_t)dx) % 16 == 0);
  const int V = vec ? 4 : 1;
  const int64_t ng = (int64_t)B * P / V;
  const dim3 grid((unsigned)cdiv64(ng, kPG), (unsigned)cdiv64(C, kOT));
  if (V == 4) chanmix_wide_kernel<4, true><<<grid, 128, 0, st>>>(du, dx, mt, nullptr, C, P, ng, du_bs, dx_bs, ci);
  else chanmix_wide_kernel<1, true><<<grid, 128, 0, st>>>(du, dx, mt, nullptr, C, P, ng, du_bs, dx_bs, ci);
  NFDPM_CHECK_LAUNCH("chanmix_wide_kernel");
  const dim3 pgrid((unsigned)cdiv64(C + 1, 32), (unsigned)cdiv64(C, 32), (unsigned)B);
  mix_bwd_part_wide_kernel<<<pgrid, 256, 0, st>>>(du, du_bs, x, x_bs, part, C, P, ci);
  NFDPM_CHECK_LAUNCH("mix_bwd_part_wide_kernel");
  return 0;
}

int mix_inv_param_grad_wide(const float* part, int B, int C, const float* s, const float* winv, const float* dld_sum,
                            float P, float* d_weight, float* d_scale, float* d_bias, float* scratch, cudaStream_t st) {
  const int n = C * C + C;
  mix_reduce_wide_kernel<<<grid_blocks(n, 256, 148 * 8), 256, 0, st>>>(part, B, n, scratch);
  NFDPM_CHECK_LAUNCH("mix_reduce_wide_kernel");
  if (d_scale != nullptr || d_bias != nullptr) {
    mix_inv_sb_wide_kernel<<<(C + 7) / 8, 256, 0, st>>>(scratch, C, s, winv, dld_sum, P, d_scale, d_bias);
    NFDPM_CHECK_LAUNCH("mix_inv_sb_wide_kernel");
  }
  if (d_weight == nullptr) return 0;
  // T = diag(e^-s) G W^-T into d_weight, then dW = -W^-T T (+ the log-det term) into the G part of scratch, which is
  // free by then, then copied over T: the scratch stays C*C + C floats
  const dim3 grid((unsigned)cdiv64(C, 32), (unsigned)cdiv64(C, 32));
  mix_inv_gemm_wide_kernel<true><<<grid, 256, 0, st>>>(scratch, C, 1, winv, 1, C, d_weight, C, s, winv, dld_sum, P);
  NFDPM_CHECK_LAUNCH("mix_inv_gemm_wide_kernel");
  mix_inv_gemm_wide_kernel<false><<<grid, 256, 0, st>>>(winv, 1, C, d_weight, C, 1, scratch, C, s, winv, dld_sum, P);
  NFDPM_CHECK_LAUNCH("mix_inv_gemm_wide_kernel");
  NFDPM_CUDA(cudaMemcpyAsync(d_weight, scratch, sizeof(float) * (size_t)C * C, cudaMemcpyDeviceToDevice, st));
  return 0;
}

}  // namespace nfdpm
