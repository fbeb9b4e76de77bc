// Backward kernels of the Glow flow path (training, SURVEY k14): what autograd would compute for
// normalizing_flow/transforms.py:80-81,131-132,179-184,286-289, utils.py:43-44,68-69, prior.py:36-37,79-83.
//   coupling_bwd_kernel        affine coupling + log-det: d(out), d(ld) -> d(K-A output), d(pm), d(bias3), d(logs3)
//   actnorm_relu_bwd_kernel    rows: dpre = dh*(h>0)*exp(s); per-channel ds, db partials
//   mix_bwd_kernel             fused ActNorm+1x1 conv backward (+ col2im of the im2col-row gradient): dx, dW^, db^ partials
//   mix_param_grad_kernel      folds dW^, db^ and the log-det terms into d(weight), d(scale), d(bias)
//   gemm_tn_kernel             weight gradients: D[N1,N2] = sum_m A[m,N1]*B[m,N2] (split over M, deterministic partials)
//   split_prior_bwd_kernel / gauss_const_bwd_kernel / col2im_add_kernel / reduce_rows_kernel
// All reductions are two-stage with a fixed order (no float atomics): bitwise reproducible.
#include <stdlib.h>

#include "tc_common.cuh"

namespace nfdpm {

template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v);
template <> __device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// 8-element vector load / store helpers: columns k0..k0+7 (k0 % 8 == 0) of row `row` of a row-major [rows, ld] matrix
// (16-byte bf16, 2 x 16-byte fp32, 2 x 16-byte hi/lo for split pairs; ld counts logical columns)
template <typename T> struct Vec8;
template <> struct Vec8<float> {
  static __device__ __forceinline__ void load(const float* base, int64_t row, int64_t ld, int k0, float (&v)[8]) {
    const float* p = base + row * ld + k0;
    const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
  }
  static __device__ __forceinline__ void store(float* base, int64_t row, int64_t ld, int k0, const float (&v)[8]) {
    float* p = base + row * ld + k0;
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
  }
};
__device__ __forceinline__ void unpack_bf16x8(const uint4 u, float (&v)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[2 * i] = __uint_as_float(w[i] << 16);
    v[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
}
template <> struct Vec8<__nv_bfloat16> {
  static __device__ __forceinline__ void load(const __nv_bfloat16* base, int64_t row, int64_t ld, int k0, float (&v)[8]) {
    unpack_bf16x8(*reinterpret_cast<const uint4*>(base + row * ld + k0), v);
  }
  static __device__ __forceinline__ void store(__nv_bfloat16* base, int64_t row, int64_t ld, int k0, const float (&v)[8]) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      w[i] = *reinterpret_cast<uint32_t*>(&t);
    }
    *reinterpret_cast<uint4*>(base + row * ld + k0) = make_uint4(w[0], w[1], w[2], w[3]);
  }
};
template <> struct Vec8<bf16x2_t> {
  static __device__ __forceinline__ void load(const bf16x2_t* base, int64_t row, int64_t ld, int k0, float (&v)[8]) {
    const __nv_bfloat16* p = reinterpret_cast<const __nv_bfloat16*>(base) + 2 * row * ld + split_col(k0);
    float lo[8];
    unpack_bf16x8(*reinterpret_cast<const uint4*>(p), v);
    unpack_bf16x8(*reinterpret_cast<const uint4*>(p + 32), lo);
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] += lo[i];
  }
  static __device__ __forceinline__ void store(bf16x2_t* base, int64_t row, int64_t ld, int k0, const float (&v)[8]) {
    split_store8(reinterpret_cast<__nv_bfloat16*>(base) + 2 * row * ld, k0, v);
  }
};
// scalar element (row, k) of the same matrices
template <typename T> __device__ __forceinline__ void st_rc(T* base, int64_t row, int64_t ld, int64_t k, float v) {
  put_rc<T>(base, row, ld, k, v);
}

// ------------------------------------------------------------------------------------------------ coupling backward
struct CouplingBwdArgs {
  const float* dy; int64_t dy_bs;      // grad wrt coupling output [B,C,P]
  const float* dld;                    // grad wrt log_det_jac [B] (may be null)
  const float* u; int64_t u_bs;        // coupling input (K-A output) [B,C,P]
  const float* pm; int64_t ldp;        // taps-as-N rows [B*P, ldp]
  const float* bias3; const float* logs3;
  float* du; int64_t du_bs;            // out: grad wrt coupling input (first half = dy_a, im2col part added by mix_bwd)
  void* dpm; int64_t ld_dpm;           // out: [B*P, ld_dpm] (fp32 or bf16; columns >= 9C are zero)
  float* dpar;                         // out: [B][2C] per-image partials: dbias3[C], dlogs3[C]
  int B, C, H, W;
  float* dbias; float* dlogs; int* counter;   // optional: the last CTA sums the partials (image order) into these
  FastDiv dP, dW, dCh, dNg, d2C;              // H*W, W, C/2, ld_dpm/8, 2C
  int pm_bulk;                                // stage the image's pm rows in shared memory with the bulk-copy engine
};

// Shared-memory floats of coupling_bwd_kernel without the optional pm block (coupling_bwd_smem)
__host__ __device__ __forceinline__ size_t coupling_bwd_floats(int C, int H, int W, size_t* pad_off, size_t* kt_off) {
  const size_t P = (size_t)H * W, PS = P + 1, Ch = C / 2, PP = (size_t)(H + 2) * (W + 2);
  size_t fl = (size_t)C * PS + Ch * PS + 4 * P * Ch + 2 * C;          // g_s, ub_s, r_s, par_s
  fl = (fl + 3) & ~(size_t)3;
  if (pad_off) *pad_off = fl;
  fl += ((size_t)C * PP + 3) & ~(size_t)3;                            // dP_pad: zero-bordered [C][(H+2)(W+2)]
  if (kt_off) *kt_off = fl;
  fl += (9 * (size_t)C + 3) & ~(size_t)3;                             // kt_s: dpm column -> offset inside dP_pad
  return fl;
}

// One CTA per image.  Same structure as the forward step boundary (boundary_body.cuh): the image's pm block arrives by
// bulk copy while the gradients are staged; index divisions are multiply-high; the dpm rows (the transposed-conv scatter
// dpm[p, tap*C+co] = dP[co][p - shift(tap)]) are gathered from a zero-bordered copy of dP through a column table.
// INV: backward of the inverse x_b = y_b/(s+1e-6) - t (a.u = the inverse's input y, a.dy = grad wrt its output x; no
// log-det term): du_b = dx_b/(s+eps), ds = -dx_b*y_b/(s+eps)^2, dt = -dx_b.
template <typename TD, bool INV>
__global__ void __launch_bounds__(1024) coupling_bwd_kernel(const CouplingBwdArgs a) {
  extern __shared__ __align__(128) float sm_raw[];
  __shared__ __align__(8) uint64_t pm_bar;
  const int C = a.C, H = a.H, W = a.W, P = H * W, Ch = C >> 1, PS = P + 1;
  const int W2p = W + 2, PP = (H + 2) * W2p;
  const int b = blockIdx.x, tid = threadIdx.x, nt = blockDim.x;
  const size_t n_pm = a.pm_bulk ? (size_t)P * a.ldp : 0;
  float* sm = sm_raw + n_pm;
  size_t pad_off, kt_off;
  coupling_bwd_floats(C, H, W, &pad_off, &kt_off);
  float* g_s = sm;                  // [C][PS] dy, second half becomes du_b
  float* ub_s = g_s + C * PS;       // [Ch][PS] u_b
  float* r_s = ub_s + Ch * PS;      // [4][P*Ch] reduction terms
  float* par_s = r_s + 4 * P * Ch;  // [2C]
  float* dP_pad = sm + pad_off;     // [C][PP] grad wrt gathered conv output, zero border
  int* kt_s = reinterpret_cast<int*>(sm + kt_off);   // [9C]
  if (a.pm_bulk && tid == 0) {
    const uint32_t bar = smem_u32(&pm_bar);
    mbar_init(bar, 1);
    fence_barrier_init();
    const char* src = reinterpret_cast<const char*>(a.pm + (size_t)b * n_pm);
    mbar_arrive_expect_tx(bar, (uint32_t)(n_pm * 4));
    for (size_t off = 0; off < n_pm * 4; off += 32768) {
      const uint32_t len = (uint32_t)((n_pm * 4 - off) < 32768 ? (n_pm * 4 - off) : 32768);
      bulk_load(smem_u32(sm_raw) + (uint32_t)off, src + off, len, bar);
    }
  }
  // ---- stage dy and u_b: every global load of a batch is issued before the first dependent shared-memory store
  const float* dyb = a.dy + (int64_t)b * a.dy_bs;
  const float* ub = a.u + (int64_t)b * a.u_bs;
  const int nx = C * P;
  for (int base = tid; base < nx || base == tid; base += 4 * nt) {   // (every thread runs the first pass: tables below)
    float v[4], w[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = base + u * nt;
      v[u] = (i < nx) ? dyb[i] : 0.f;
      w[u] = (i < nx && i >= Ch * P) ? ub[i] : 0.f;
    }
    if (base == tid) {                                               // parameters and tables ride on the first batch
      for (int i = tid; i < C; i += nt) {
        par_s[i] = a.bias3[i];
        par_s[C + i] = expf(3.f * a.logs3[i]);
      }
      for (int i = tid; i < C * PP; i += nt) dP_pad[i] = 0.f;
      for (int k = tid; k < 9 * C; k += nt) {
        const int tap = k / C, co = k - tap * C;                     // (runs once per thread at most a few times)
        kt_s[k] = co * PP + (2 - tap / 3) * W2p + (2 - tap % 3);     // pm row (py,px) at tap feeds pixel (py-dy, px-dx)
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = base + u * nt;
      if (i < nx) {
        const int c = fdiv(i, a.dP), p = i - c * P;
        g_s[c * PS + p] = v[u];
        if (c >= Ch) ub_s[(c - Ch) * PS + p] = w[u];
      }
    }
  }
  __syncthreads();
  const float gld = (a.dld != nullptr) ? a.dld[b] : 0.f;
  if (a.pm_bulk) mbar_wait(smem_u32(&pm_bar), 0);
  const float* pmb = a.pm_bulk ? sm_raw : a.pm + (int64_t)b * P * a.ldp;
  const bool pm_smem = a.pm_bulk != 0;
  for (int it = tid; it < P * Ch; it += nt) {
    const int p = fdiv(it, a.dCh), j = it - p * Ch;
    const int py = fdiv(p, a.dW), px = p - py * W;
    float lv[9], tv[9];
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int yy = py + tap / 3 - 1, xx = px + tap % 3 - 1;
      const bool ok = (yy >= 0) && (yy < H) && (xx >= 0) && (xx < W);
      const float* r = pmb + (int64_t)(ok ? yy * W + xx : p) * a.ldp + tap * C + j;
      const float l0 = pm_smem ? r[0] : __ldg(r), t0 = pm_smem ? r[Ch] : __ldg(r + Ch);
      lv[tap] = ok ? l0 : 0.f;
      tv[tap] = ok ? t0 : 0.f;
    }
    float ls = 0.f, tt = 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      ls += lv[tap];
      tt += tv[tap];
    }
    const float g_l = par_s[C + j], g_t = par_s[C + Ch + j];
    const float log_s = (ls + par_s[j]) * g_l;
    const float t = (tt + par_s[Ch + j]) * g_t;
    const float s = 1.f / (1.f + expf(-(log_s + 2.f)));
    const float dyv = g_s[(Ch + j) * PS + p];
    float ds, dt, dub;
    if (INV) {
      const float r = 1.f / (s + 1e-6f);
      dub = dyv * r;
      ds = -dub * ub_s[j * PS + p] * r;
      dt = -dyv;
    } else {
      ds = dyv * (ub_s[j * PS + p] + t) + gld / (s + 1e-6f);
      dt = dyv * s;
      dub = dyv * s;
    }
    const float dls = ds * s * (1.f - s);
    g_s[(Ch + j) * PS + p] = dub;                // du_b
    const int pq = (py + 1) * W2p + px + 1;
    dP_pad[j * PP + pq] = dls * g_l;
    dP_pad[(Ch + j) * PP + pq] = dt * g_t;
    r_s[0 * P * Ch + j * P + p] = dls * g_l;         // -> dbias3[j]
    r_s[1 * P * Ch + j * P + p] = dt * g_t;          // -> dbias3[Ch+j]
    r_s[2 * P * Ch + j * P + p] = 3.f * dls * log_s; // -> dlogs3[j]
    r_s[3 * P * Ch + j * P + p] = 3.f * dt * t;      // -> dlogs3[Ch+j]
  }
  __syncthreads();
  // outputs: du (coalesced over pixels)
  float* dub = a.du + (int64_t)b * a.du_bs;
  for (int i = tid; i < C * P; i += nt) {
    const int c = fdiv(i, a.dP), p = i - c * P;
    dub[i] = g_s[c * PS + p];
  }
  // dpm rows: dpm[p', tap*C+co] = dP[co][p' - shift(tap)] = dP_pad[kt_s[col] + py'*(W+2) + px'] (zero outside the image and
  // in the padding columns).  A thread produces 8 consecutive columns (one 16-byte bf16 / two 16-byte fp32 stores).
  const int ldp = (int)a.ld_dpm;
  TD* dpmb = reinterpret_cast<TD*>(a.dpm);
  const int64_t row0 = (int64_t)b * P;
  if ((ldp & 7) == 0 && (((uintptr_t)dpmb) & 15) == 0) {
    const int n_g = ldp >> 3, K = 9 * C;
    for (int it = tid; it < P * n_g; it += nt) {
      const int pp = fdiv(it, a.dNg), g = it - pp * n_g;
      const int py = fdiv(pp, a.dW), px = pp - py * W;
      const float* win = dP_pad + py * W2p + px;
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int col = g * 8 + e;
        v[e] = (col < K) ? win[kt_s[col]] : 0.f;
      }
      Vec8<TD>::store(dpmb, row0 + pp, ldp, g * 8, v);
    }
  } else {
    for (int i = tid; i < P * ldp; i += nt) {
      const int pp = i / ldp, col = i - pp * ldp;
      float v = 0.f;
      if (col < 9 * C) {
        const int py = fdiv(pp, a.dW), px = pp - py * W;
        v = dP_pad[kt_s[col] + py * W2p + px];
      }
      st_rc<TD>(dpmb, row0 + pp, ldp, col, v);
    }
  }
  // per-image parameter partials: one warp per (kind, j) row of r_s, fixed order
  const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
  for (int row = warp; row < 4 * Ch; row += nw) {
    float acc = 0.f;
    const float* rp = r_s + row * P;      // row = kind*Ch + j  (r_s laid out [kind][j][p])
#pragma unroll 8
    for (int p = lane; p < P; p += 32) acc += rp[p];
    acc = warp_sum(acc);
    if (lane == 0) {
      const int kind = fdiv(row, a.dCh), j = row - kind * Ch;
      // kind 0: dbias[j], 1: dbias[Ch+j], 2: dlogs[j], 3: dlogs[Ch+j]
      const int dst = (kind < 2 ? 0 : C) + ((kind & 1) ? Ch : 0) + j;
      a.dpar[(int64_t)b * 2 * C + dst] = acc;
    }
  }
  if (a.counter != nullptr) {
    // the CTA that finishes last reduces all per-image partials in image order (deterministic) and re-arms the counter
    __shared__ int s_last;
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(a.counter, 1) == (int)gridDim.x - 1);
    __syncthreads();
    if (s_last) {
      __threadfence();
      // [row group][2C] partial sums over interleaved images, then a fixed-order combine: deterministic and parallel
      // (a single thread per column walking all B rows is ~B dependent L2 round trips)
      const int n2c = 2 * C;
      int RG = nt / n2c;
      if (RG > 32) RG = 32;
      if (RG < 1) RG = 1;
      float* red = sm;                       // the image buffers are dead by now: RG * 2C floats
      for (int idx = tid; idx < RG * n2c; idx += nt) {
        const int rg = fdiv(idx, a.d2C), i = idx - rg * n2c;
        float acc = 0.f;
        int bb = rg;
        for (; bb + 31 * RG < a.B; bb += 32 * RG) {        // 32 loads in flight, added in image order
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __ldcg(a.dpar + (int64_t)(bb + j * RG) * n2c + i);
#pragma unroll
          for (int j = 0; j < 32; ++j) acc += v[j];
        }
        for (; bb + 7 * RG < a.B; bb += 8 * RG) {          // eight loads in flight, added in image order
          float v[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) v[j] = __ldcg(a.dpar + (int64_t)(bb + j * RG) * n2c + i);
#pragma unroll
          for (int j = 0; j < 8; ++j) acc += v[j];
        }
        for (; bb < a.B; bb += RG) acc += __ldcg(a.dpar + (int64_t)bb * n2c + i);
        red[idx] = acc;
      }
      __syncthreads();
      for (int i = tid; i < n2c; i += nt) {
        float acc = 0.f;
        for (int rg = 0; rg < RG; ++rg) acc += red[rg * n2c + i];
        if (i < C) a.dbias[i] = acc; else a.dlogs[i - C] = acc;
      }
      if (tid == 0) *a.counter = 0;
    }
  }
}

// Tiled variant for images (or channel counts) that do not fit one CTA: CTA = (image, tile of TP pixels), direct global
// access; the gradient wrt the gathered conv output goes to dP [M, C] and dpm_expand_kernel scatters it into the
// taps-as-N rows afterwards (a pixel's dpm row needs dP of its 8 neighbours, which may live in other tiles).
template <bool INV>
__global__ void __launch_bounds__(256) coupling_bwd_tiled_kernel(const CouplingBwdArgs a, float* __restrict__ dP, int TP) {
  extern __shared__ __align__(16) float sm[];        // r_s [4][Ch][TP] + par_s [2C]
  const int C = a.C, H = a.H, W = a.W, P = H * W, Ch = C >> 1;
  const int T = (P + TP - 1) / TP;
  const int b = blockIdx.x / T, t = blockIdx.x - b * T;
  const int p0 = t * TP, np = min(TP, P - p0);
  float* r_s = sm;
  float* par_s = r_s + 4 * Ch * TP;
  const int tid = threadIdx.x, nt = blockDim.x;
  for (int i = tid; i < C; i += nt) {
    par_s[i] = a.bias3[i];
    par_s[C + i] = expf(3.f * a.logs3[i]);
  }
  __syncthreads();
  const float* dyb = a.dy + (int64_t)b * a.dy_bs;
  const float* ub = a.u + (int64_t)b * a.u_bs;
  float* dub = a.du + (int64_t)b * a.du_bs;
  for (int i = tid; i < Ch * np; i += nt) {           // first half passes through
    const int c = i / np, pl = i - c * np;
    dub[(int64_t)c * P + p0 + pl] = dyb[(int64_t)c * P + p0 + pl];
  }
  const float gld = (a.dld != nullptr) ? a.dld[b] : 0.f;
  const float* pmb = a.pm + (int64_t)b * P * a.ldp;
  for (int it = tid; it < np * Ch; it += nt) {
    const int pl = it / Ch, j = it - pl * Ch;
    const int p = p0 + pl;
    const int py = p / W, px = p - py * W;
    float ls = 0.f, tt = 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int yy = py + tap / 3 - 1, xx = px + tap % 3 - 1;
      const bool ok = (yy >= 0) && (yy < H) && (xx >= 0) && (xx < W);
      const float* r = pmb + (int64_t)(ok ? yy * W + xx : p) * a.ldp + tap * C + j;
      const float l0 = __ldg(r), t0 = __ldg(r + Ch);
      ls += ok ? l0 : 0.f;
      tt += ok ? t0 : 0.f;
    }
    const float g_l = par_s[C + j], g_t = par_s[C + Ch + j];
    const float log_s = (ls + par_s[j]) * g_l;
    const float tv = (tt + par_s[Ch + j]) * g_t;
    const float s = 1.f / (1.f + expf(-(log_s + 2.f)));
    const float dyv = dyb[(int64_t)(Ch + j) * P + p];
    float ds, dt, duv;
    if (INV) {
      const float r = 1.f / (s + 1e-6f);
      duv = dyv * r;
      ds = -duv * ub[(int64_t)(Ch + j) * P + p] * r;
      dt = -dyv;
    } else {
      ds = dyv * (ub[(int64_t)(Ch + j) * P + p] + tv) + gld / (s + 1e-6f);
      dt = dyv * s;
      duv = dyv * s;
    }
    const float dls = ds * s * (1.f - s);
    dub[(int64_t)(Ch + j) * P + p] = duv;
    float* dpr = dP + ((int64_t)b * P + p) * C;
    dpr[j] = dls * g_l;
    dpr[Ch + j] = dt * g_t;
    r_s[(0 * Ch + j) * TP + pl] = dls * g_l;
    r_s[(1 * Ch + j) * TP + pl] = dt * g_t;
    r_s[(2 * Ch + j) * TP + pl] = 3.f * dls * log_s;
    r_s[(3 * Ch + j) * TP + pl] = 3.f * dt * tv;
  }
  __syncthreads();
  const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
  for (int row = warp; row < 4 * Ch; row += nw) {
    float acc = 0.f;
    const float* rp = r_s + row * TP;
    for (int pl = lane; pl < np; pl += 32) acc += rp[pl];
    acc = warp_sum(acc);
    if (lane == 0) {
      const int kind = row / Ch, j = row - kind * Ch;
      const int dst = (kind < 2 ? 0 : C) + ((kind & 1) ? Ch : 0) + j;
      a.dpar[(int64_t)blockIdx.x * 2 * C + dst] = acc;
    }
  }
}

// dpm[m, tap*C+co] = dP[m - shift(tap), co] inside the image, 0 outside and in the padding columns
template <typename TD>
__global__ void dpm_expand_kernel(const float* __restrict__ dP, TD* __restrict__ dpm, int64_t ld, int C, int H, int W,
                                  int64_t n) {
  const int P = H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i / ld;
    const int col = (int)(i - m * ld);
    float v = 0.f;
    if (col < 9 * C) {
      const int tap = col / C, co = col - tap * C;
      const int64_t b = m / P;
      const int p = (int)(m - b * P);
      const int py = p / W, px = p - py * W;
      const int yy = py - (tap / 3 - 1), xx = px - (tap % 3 - 1);
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = __ldg(dP + (b * P + yy * W + xx) * C + co);
    }
    st_rc<TD>(dpm, m, ld, col, v);
  }
}

// ------------------------------------------------------------------------------------------------ ActNorm+ReLU backward
// rows [M, ld], channel fastest.  CTA = `rows_per_cta` rows x all N columns; a thread owns 8 consecutive columns
// (16-byte bf16 / 32-byte fp32 vectors, fully coalesced rows), the CTA's 256 threads cover 256/(N/8) rows at a time and
// loop over the rest; per-column partial sums are combined across the row groups in shared memory in a fixed order.
template <typename TD, typename TH, typename TO>
__global__ void __launch_bounds__(256) actnorm_relu_bwd_kernel(const TD* __restrict__ dh, const TH* __restrict__ h,
                                                               const float* __restrict__ scale, TO* __restrict__ dpre,
                                                               float* __restrict__ part, int M, int N, int64_t ld_dh,
                                                               int64_t ld_h, int64_t ld_o, int rows_per_cta) {
  extern __shared__ __align__(16) float red[];           // [row groups][2][N]
  const int cg = N >> 3;                                  // column groups of 8 (N % 8 == 0, cg <= 256)
  const int rg = 256 / cg;                                // row groups processed concurrently
  const int tid = threadIdx.x;
  const int g = tid % cg, r0 = tid / cg;
  const int m0 = blockIdx.x * rows_per_cta, m1 = min(M, m0 + rows_per_cta);
  float ds[8], db[8], e[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { ds[j] = 0.f; db[j] = 0.f; }
  if (r0 < rg) {
#pragma unroll
    for (int j = 0; j < 8; ++j) e[j] = expf(__ldg(scale + g * 8 + j));
#pragma unroll 4
    for (int m = m0 + r0; m < m1; m += rg) {
      float gv[8], hv[8], o[8];
      Vec8<TD>::load(dh, m, ld_dh, g * 8, gv);
      Vec8<TH>::load(h, m, ld_h, g * 8, hv);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float gg = (hv[j] > 0.f) ? gv[j] : 0.f;
        ds[j] = fmaf(gg, hv[j], ds[j]);
        o[j] = gg * e[j];
        db[j] += o[j];
      }
      Vec8<TO>::store(dpre, m, ld_o, g * 8, o);
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      red[(r0 * 2 + 0) * N + g * 8 + j] = ds[j];
      red[(r0 * 2 + 1) * N + g * 8 + j] = db[j];
    }
  }
  __syncthreads();
  for (int i = tid; i < 2 * N; i += 256) {
    float acc = 0.f;
    for (int r = 0; r < rg; ++r) acc += red[r * 2 * N + i];
    part[(int64_t)blockIdx.x * 2 * N + i] = acc;
  }
}

// out[n] (+)= sum_r part[r*stride + n]
// Column sums of a [R, stride] partial matrix in a fixed order: CTA = 32 columns x 8 row lanes; lane ry sums rows
// ry, ry+8, ... and the 8 lane sums are added in order (deterministic; coalesced 128-byte row segments).
__device__ __forceinline__ float colsum_32x8(const float* __restrict__ part, int R, int64_t stride, int col, bool valid,
                                             float (*sh)[33]) {
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5;
  float s = 0.f;
  if (valid)
    for (int r = ry; r < R; r += 8) s += part[(int64_t)r * stride + col];
  sh[ry][cx] = s;
  __syncthreads();
  float t = 0.f;
  if (ry == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) t += sh[i][cx];
  }
  return t;   // valid for ry == 0
}

// out0[i] = sum_r part[r*stride + i] (i < n0);  out1[i - n0] = ... (n0 <= i < n0 + n1): one launch for a (scale, bias) or
// (bias, logs) pair whose partials sit side by side
__global__ void __launch_bounds__(256) reduce_rows2_kernel(const float* __restrict__ part, float* __restrict__ out0,
                                                           float* __restrict__ out1, int R, int n0, int n1, int64_t stride) {
  __shared__ float sh[8][33];
  const int i = blockIdx.x * 32 + (threadIdx.x & 31);
  const float s = colsum_32x8(part, R, stride, i, i < n0 + n1, sh);
  if ((threadIdx.x >> 5) == 0 && i < n0 + n1) {
    if (i < n0) out0[i] = s; else out1[i - n0] = s;
  }
}

__global__ void __launch_bounds__(256) reduce_rows_kernel(const float* __restrict__ part, float* __restrict__ out, int R,
                                                          int n, int64_t stride, int accumulate) {
  __shared__ float sh[8][33];
  const int i = blockIdx.x * 32 + (threadIdx.x & 31);
  const float s = colsum_32x8(part, R, stride, i, i < n, sh);
  if ((threadIdx.x >> 5) == 0 && i < n) out[i] = accumulate ? out[i] + s : s;
}

// ------------------------------------------------------------------------------------------------ K-A backward
struct MixBwdArgs {
  const float* du; int64_t du_bs;     // grad wrt K-A output [B,C,P] (first half still lacks the im2col part)
  const float* da1; int64_t lda1;     // grad wrt im2col rows [B*P, lda1] (may be null)
  const float* x; int64_t x_bs;       // K-A input [B,C,P]
  const float* mt;                    // fwd_mt[i*C+o] = W^[o][i]
  float* dx; int64_t dx_bs;           // out
  float* part;                        // out: [B*T][C*C + C]: dW^x[o*C+i] = sum_p du[o]x[i];  db^[o] = sum_p du[o]
  int B, C, H, W;
  int TP;                             // pixels per CTA tile (T = ceil(P/TP) tiles per image)
  FastDiv dC, dCh, dW, dT, dNpFull, dNpLast;   // C, C/2, W, tiles per image, pixels of a full / of the last tile
};

__global__ void __launch_bounds__(1024) mix_bwd_kernel(const MixBwdArgs a) {
  // CTA = (image b, pixel tile t): pixels [p0, p0 + np) of the image; images up to 256 pixels are one tile
  extern __shared__ __align__(16) float sm[];
  const int C = a.C, H = a.H, W = a.W, P = H * W, Ch = C >> 1;
  const int T = (int)a.dT.d;
  const int b = fdiv((int)blockIdx.x, a.dT), t = blockIdx.x - b * T;
  const int p0 = t * a.TP, np = min(a.TP, P - p0), PS = a.TP + 1;
  float* d_s = sm;                 // [C][PS] du (complete)
  float* x_s = d_s + C * PS;       // [C][PS]
  float* w_s = x_s + C * PS;       // [C][C]  w_s[o*C+i] = W^[o][i]
  const int tid = threadIdx.x, nt = blockDim.x;
  // index divisions are multiply-high (run-time divisors; exact for these ranges)
  const FastDiv dNp = (t == T - 1) ? a.dNpLast : a.dNpFull;
  const float* dub = a.du + (int64_t)b * a.du_bs;
  const float* xb = a.x + (int64_t)b * a.x_bs;
  // staging: the global loads of a batch are issued before the first dependent shared-memory store
  const int nx = C * np;
  for (int base = tid; base < nx || base == tid; base += 4 * nt) {   // (every thread runs the first pass: w_s below)
    float dv[4], xv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = base + u * nt;
      dv[u] = xv[u] = 0.f;
      if (i < nx) {
        const int c = fdiv(i, dNp), pl = i - c * np;
        dv[u] = dub[(int64_t)c * P + p0 + pl];
        xv[u] = xb[(int64_t)c * P + p0 + pl];
      }
    }
    if (base == tid) {
      for (int i = tid; i < C * C; i += nt) {
        const int o = fdiv(i, a.dC), ii = i - o * C;
        w_s[i] = a.mt[ii * C + o];
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = base + u * nt;
      if (i < nx) {
        const int c = fdiv(i, dNp), pl = i - c * np;
        d_s[c * PS + pl] = dv[u];
        x_s[c * PS + pl] = xv[u];
      }
    }
  }
  __syncthreads();
  if (a.da1 != nullptr) {
    // col2im: A1[m, c*9+tap] = u[c][m + shift(tap)]  =>  du[c][p] += sum_tap dA1[p - shift(tap), c*9+tap]
    const float* dab = a.da1 + (int64_t)b * P * a.lda1;
    for (int it = tid; it < np * Ch; it += nt) {
      const int pl = fdiv(it, a.dCh), c = it - pl * Ch;
      const int p = p0 + pl;
      const int py = fdiv(p, a.dW), px = p - py * W;
      float v[9];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {                            // all nine loads in flight, added in tap order
        const int yy = py - (tap / 3 - 1), xx = px - (tap % 3 - 1);
        const bool ok = yy >= 0 && yy < H && xx >= 0 && xx < W;
        const float l = __ldg(dab + (int64_t)(ok ? yy * W + xx : p) * a.lda1 + c * 9 + tap);
        v[tap] = ok ? l : 0.f;
      }
      float acc = 0.f;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int yy = py - (tap / 3 - 1), xx = px - (tap % 3 - 1);
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) acc += v[tap];
      }
      d_s[c * PS + pl] += acc;
    }
    __syncthreads();
  }
  // dx[i][p] = sum_o W^[o][i] du[o][p]
  float* dxb = a.dx + (int64_t)b * a.dx_bs;
  for (int it = tid; it < C * np; it += nt) {
    const int i = fdiv(it, dNp), pl = it - i * np;
    float acc = 0.f;
#pragma unroll 4
    for (int o = 0; o < C; ++o) acc = fmaf(w_s[o * C + i], d_s[o * PS + pl], acc);
    dxb[(int64_t)i * P + p0 + pl] = acc;
  }
  // partials of d(W^) and d(b^), fixed summation order.  Many pixels: one warp per element, lanes over pixels + shuffle
  // tree, FOUR elements per warp in flight (their shuffle chains interleave; each element's own order is unchanged).
  // Few pixels (deep levels, C up to 48..192 -> thousands of elements): one THREAD per element, sequential over p.
  float* pb = a.part + (int64_t)blockIdx.x * (C * C + C);
  const int n_e = C * C + C;
  if (np >= 64) {
    const int warp = tid >> 5, lane = tid & 31, nw = nt >> 5;
    for (int e0 = warp * 4; e0 < n_e; e0 += nw * 4) {
      float acc[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int e = e0 + k;
        acc[k] = 0.f;
        if (e < C * C) {
          const int o = fdiv(e, a.dC), i = e - o * C;
          for (int pl = lane; pl < np; pl += 32) acc[k] = fmaf(d_s[o * PS + pl], x_s[i * PS + pl], acc[k]);
        } else if (e < n_e) {
          const int o = e - C * C;
          for (int pl = lane; pl < np; pl += 32) acc[k] += d_s[o * PS + pl];
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
        for (int k = 0; k < 4; ++k) acc[k] += __shfl_xor_sync(0xffffffffu, acc[k], o);
      }
      if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (e0 + k < n_e) pb[e0 + k] = acc[k];
      }
    }
  } else {
    for (int e = tid; e < n_e; e += nt) {
      float acc = 0.f;
      if (e < C * C) {
        const int o = fdiv(e, a.dC), i = e - o * C;   // lanes share o (broadcast) and walk i: rows PS apart -> no conflicts
#pragma unroll 4
        for (int pl = 0; pl < np; ++pl) acc = fmaf(d_s[o * PS + pl], x_s[i * PS + pl], acc);
      } else {
        const int o = e - C * C;
#pragma unroll 4
        for (int pl = 0; pl < np; ++pl) acc += d_s[o * PS + pl];
      }
      pb[e] = acc;
    }
  }
}

// dW, ds, db of one StepFlow from the per-image partials and the log-det terms.  One CTA per StepFlow.
struct MixParamItem {
  const float* part; int B;        // [B][C*C + C]
  const float* W; const float* s; const float* bv; const float* winv;
  const float* dld_sum;            // [1] sum_b d(ld)[b]
  float P;                         // H*W multiplier of the log-det constants
  float* dW; float* ds; float* db; // out (overwritten)
  float* scratch;                  // [C*C + C] reduced partials
  int C;
};
constexpr int kParamBatch = 16;
struct MixParamBatch { MixParamItem it[kParamBatch]; };

// sum of the B per-image partial rows of one item into it.scratch (eight loads in flight, added in order: deterministic)
__device__ __forceinline__ void mix_reduce_partials(const MixParamItem& it, int tid) {
  const int n = it.C * it.C + it.C;
  for (int e = tid; e < n; e += blockDim.x) {
    float acc = 0.f;
    int b = 0;
    for (; b + 8 <= it.B; b += 8) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __ldcg(it.part + (int64_t)(b + j) * n + e);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc += v[j];
    }
    for (; b < it.B; ++b) acc += __ldcg(it.part + (int64_t)b * n + e);
    it.scratch[e] = acc;
  }
}

__global__ void __launch_bounds__(256) mix_param_grad_kernel(const MixParamBatch batch) {
  const MixParamItem it = batch.it[blockIdx.x];
  const int C = it.C, tid = threadIdx.x;
  mix_reduce_partials(it, tid);
  __syncthreads();
  const float G = it.dld_sum[0] * it.P;
  // dW^_total[o][i] = dW^x[o][i] + db^[o]*b[i];  W^[o][i] = W[o][i]*exp(s[i])
  for (int e = tid; e < C * C; e += 256) {
    const int o = e / C, i = e - o * C;
    const float bi = it.bv ? it.bv[i] : 0.f, es = expf(it.s ? it.s[i] : 0.f);
    const float dwh = it.scratch[e] + it.scratch[C * C + o] * bi;
    if (it.dW) it.dW[e] = dwh * es + G * it.winv[i * C + o];
  }
  for (int i = tid; i < C; i += 256) {
    const float bi = it.bv ? it.bv[i] : 0.f, es = expf(it.s ? it.s[i] : 0.f);
    float ds = 0.f, db = 0.f;
    for (int o = 0; o < C; ++o) {
      const float wh = it.W[o * C + i] * es;
      const float dwh = it.scratch[o * C + i] + it.scratch[C * C + o] * bi;
      ds = fmaf(dwh, wh, ds);
      db = fmaf(wh, it.scratch[C * C + o], db);
    }
    if (it.ds) it.ds[i] = ds + G;
    if (it.db) it.db[i] = db;
  }
}

// The inverse mix x = M u - b, M = diag(e^-s) W^-1, from the partials of a mix_bwd run with mt = inv_mt (G = sum dx u^T,
// g = sum dx):  db = -g,  ds_c = -sum_j G_cj M_cj,  dW = -W^-T (diag(e^-s) G) W^-T.  One CTA per StepFlow; shared memory
// holds diag(e^-s) G W^-T [C][C].
__global__ void __launch_bounds__(256) mix_inv_param_grad_kernel(const MixParamBatch batch) {
  extern __shared__ float t_s[];
  const MixParamItem it = batch.it[blockIdx.x];
  const int C = it.C, tid = threadIdx.x;
  mix_reduce_partials(it, tid);
  __syncthreads();
  const float* G = it.scratch;
  const float* g = it.scratch + C * C;
  for (int c = tid; c < C; c += 256) {
    if (it.db) it.db[c] = -g[c];
    if (it.ds) {
      float acc = 0.f;
      for (int j = 0; j < C; ++j) acc = fmaf(G[c * C + j], it.winv[c * C + j], acc);
      it.ds[c] = -expf(-it.s[c]) * acc;
    }
  }
  if (it.dW == nullptr) return;
  for (int e = tid; e < C * C; e += 256) {
    const int c = e / C, k = e - c * C;
    float acc = 0.f;
    for (int d = 0; d < C; ++d) acc = fmaf(G[c * C + d], it.winv[k * C + d], acc);
    t_s[e] = expf(it.s ? -it.s[c] : 0.f) * acc;
  }
  __syncthreads();
  for (int e = tid; e < C * C; e += 256) {
    const int a = e / C, k = e - a * C;
    float acc = 0.f;
    for (int c = 0; c < C; ++c) acc = fmaf(it.winv[c * C + a], t_s[c * C + k], acc);
    it.dW[e] = -acc;
  }
}

// ------------------------------------------------------------------------------------------------ wgrad GEMM (TN)
// D[N1, N2] = sum_m A[m, N1] * B[m, N2];  tile 128 x 128, 256 threads, 8x8 per thread; grid.z splits M, each split
// writes its own partial slab (reduced by reduce_rows_kernel) -> deterministic.
template <typename TA, typename TB>
__global__ void __launch_bounds__(256) gemm_tn_kernel(const TA* __restrict__ A, int64_t lda, const TB* __restrict__ Bm,
                                                      int64_t ldb, float* __restrict__ part, int M, int N1, int N2,
                                                      int rows_per_split) {
  constexpr int BT = 128, BKm = 16;
  __shared__ __align__(16) float As[BKm][BT + 4];
  __shared__ __align__(16) float Bs[BKm][BT + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int n1_0 = blockIdx.y * BT, n2_0 = blockIdx.x * BT;
  const int m_lo = blockIdx.z * rows_per_split, m_hi = min(M, m_lo + rows_per_split);
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  for (int m0 = m_lo; m0 < m_hi; m0 += BKm) {
    // 16 rows x 128 cols per operand = 2048 elements, 8 per thread; column fastest -> coalesced
    for (int e = tid; e < BKm * BT; e += 256) {
      const int r = e >> 7, c = e & 127;
      const int m = m0 + r;
      As[r][c] = (m < m_hi && n1_0 + c < N1) ? ldf<TA>(A + (int64_t)m * lda + n1_0 + c) : 0.f;
      Bs[r][c] = (m < m_hi && n2_0 + c < N2) ? ldf<TB>(Bm + (int64_t)m * ldb + n2_0 + c) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < BKm; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[k][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[k][64 + tx * 4]);
      const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* pz = part + (int64_t)blockIdx.z * N1 * N2;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = n1_0 + (i >> 2) * 64 + ty * 4 + (i & 3);
    if (r >= N1) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int c = n2_0 + (j >> 2) * 64 + tx * 4 + (j & 3);
      if (c < N2) pz[(int64_t)r * N2 + c] = acc[i][j];
    }
  }
}

// ------------------------------------------------------------------------------------------------ priors
// Split prior backward, one thread per pixel (same tiling as the forward kernel): writes dz into channels C/2..C of
// dstate, dh rows [M, ldh] (columns C..ldh zero) and per-image partials [B][2C] (dbias[C], dlogs[C]).
__global__ void __launch_bounds__(256) split_prior_bwd_kernel(const float* __restrict__ dlp, const float* __restrict__ h,
                                                              int64_t ldh, const float* __restrict__ bias,
                                                              const float* __restrict__ logs, const float* __restrict__ x,
                                                              int64_t xbs, float* __restrict__ dstate, int64_t dbs,
                                                              float* __restrict__ dh, float* __restrict__ dpar, int B,
                                                              int C, int P) {
  extern __shared__ __align__(16) float s_par[];   // [2C]
  __shared__ float red[256];
  const int Ch = C >> 1, b = blockIdx.x, tid = threadIdx.x;
  for (int i = tid; i < C; i += 256) {
    s_par[i] = (h != nullptr) ? bias[i] : 0.f;
    s_par[C + i] = (h != nullptr) ? expf(3.f * logs[i]) : 1.f;
  }
  __syncthreads();
  const float g = dlp[b];
  // per-channel partial sums are accumulated channel by channel (fixed order) to stay deterministic
  for (int j = 0; j < Ch; ++j) {
    float s_bm = 0.f, s_bl = 0.f, s_lm = 0.f, s_ll = 0.f;
    for (int p = tid; p < P; p += 256) {
      const int64_t m = (int64_t)b * P + p;
      float mean = 0.f, lg = 0.f;
      if (h != nullptr) {
        mean = (h[m * ldh + j] + s_par[j]) * s_par[C + j];
        lg = (h[m * ldh + Ch + j] + s_par[Ch + j]) * s_par[C + Ch + j];
      }
      const float z = x[b * xbs + (int64_t)(Ch + j) * P + p];
      const float d = z - mean, iv = expf(-2.f * lg);
      const float dz = -d * iv * g, dmean = d * iv * g, dlg = (-1.f + d * d * iv) * g;
      dstate[b * dbs + (int64_t)(Ch + j) * P + p] += dz;
      if (h != nullptr) {
        const float dhm = dmean * s_par[C + j], dhl = dlg * s_par[C + Ch + j];
        dh[m * ldh + j] = dhm;
        dh[m * ldh + Ch + j] = dhl;
        s_bm += dhm; s_bl += dhl;
        s_lm += 3.f * dmean * mean; s_ll += 3.f * dlg * lg;
      }
    }
    if (h != nullptr) {
      float* vals[4] = {&s_bm, &s_bl, &s_lm, &s_ll};
      const int dst[4] = {j, Ch + j, C + j, C + Ch + j};
      for (int k = 0; k < 4; ++k) {
        red[tid] = *vals[k];
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
          if (tid < s) red[tid] += red[tid + s];
          __syncthreads();
        }
        if (tid == 0) dpar[(int64_t)b * 2 * C + dst[k]] = red[0];
        __syncthreads();
      }
    }
  }
  if (h != nullptr) {
    for (int i = tid; i < P * (int)(ldh - C); i += 256) {
      const int p = i / (int)(ldh - C), c = C + i % (int)(ldh - C);
      dh[((int64_t)b * P + p) * ldh + c] = 0.f;
    }
  }
}

// Gaussian prior with per-channel constants: dz and per-image partials [B][4C]: dbias[2C], dlogs[2C] of the 2C-channel conv
__global__ void __launch_bounds__(256) gauss_const_bwd_kernel(const float* __restrict__ dl, const float* __restrict__ z,
                                                              const float* __restrict__ bias, const float* __restrict__ logs,
                                                              float* __restrict__ dz, float* __restrict__ dpar, int C, int P) {
  __shared__ float red[256];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float g = dl[b];
  for (int c = 0; c < C; ++c) {
    float mean = 0.f, lg = 0.f, em = 1.f, el = 1.f;
    if (bias != nullptr) {
      em = expf(3.f * logs[c]); el = expf(3.f * logs[C + c]);
      mean = bias[c] * em; lg = bias[C + c] * el;
    }
    const float iv = expf(-2.f * lg);
    float sm_ = 0.f, sl_ = 0.f;
    for (int p = tid; p < P; p += 256) {
      const int64_t i = ((int64_t)b * C + c) * P + p;
      const float d = z[i] - mean;
      dz[i] = -d * iv * g;
      sm_ += d * iv * g;
      sl_ += (-1.f + d * d * iv) * g;
    }
    if (bias != nullptr) {
      float v[2] = {sm_, sl_};
      for (int k = 0; k < 2; ++k) {
        red[tid] = v[k];
        __syncthreads();
        for (int s = 128; s > 0; s >>= 1) {
          if (tid < s) red[tid] += red[tid + s];
          __syncthreads();
        }
        if (tid == 0) {
          const float tot = red[0];
          // mean_c = bias_c*em: dbias_c = tot*em, dlogs_c = 3*tot*mean ; same for the log-sd half
          const int cc = k == 0 ? c : C + c;
          const float e = k == 0 ? em : el, val = k == 0 ? mean : lg;
          dpar[(int64_t)b * 4 * C + cc] = tot * e;
          dpar[(int64_t)b * 4 * C + 2 * C + cc] = 3.f * tot * val;
        }
        __syncthreads();
      }
    }
  }
}

// Backward of the reparameterised draw z = mean + exp(lg)*T*eps with (mean, lg) = ((h + bias)*exp(3*logs)) split into
// channel halves (Split prior, C = 2 x latent channels).  With h == nullptr mean / lg are the per-channel constants
// bias*exp(3*logs) (GaussianPrior).  d mean = dz, d lg = dz*exp(lg)*T*eps.  One CTA per image, channels in chunks of up to
// 256: thread t owns channel j0 + t % cw and every rg-th pixel (rg = 256 / cw row groups), so the dh / h rows are read and
// written along consecutive channels; per-channel partials are combined over the row groups in a fixed order
// (deterministic).  Writes dh rows [M, ldh] (columns C..ldh zero) when h is given, and dpar [B][2C] (dbias[C], dlogs[C]).
__global__ void __launch_bounds__(256) split_sample_bwd_kernel(const float* __restrict__ dz, int64_t dz_bs,
                                                               const float* __restrict__ eps, float temperature,
                                                               const float* __restrict__ h, int64_t ldh,
                                                               const float* __restrict__ bias, const float* __restrict__ logs,
                                                               float* __restrict__ dh, float* __restrict__ dpar, int C, int P) {
  __shared__ float red[4][256];
  const int Ch = C >> 1, b = blockIdx.x, tid = threadIdx.x;
  for (int j0 = 0; j0 < Ch; j0 += 256) {
    const int cw = min(256, Ch - j0), rg = 256 / cw;
    const int jl = tid % cw, r = tid / cw, j = j0 + jl;
    float s_bm = 0.f, s_bl = 0.f, s_lm = 0.f, s_ll = 0.f;
    if (r < rg) {
      const float em = expf(3.f * logs[j]), el = expf(3.f * logs[Ch + j]);
      const float bm = bias[j], bl = bias[Ch + j];
      for (int p = r; p < P; p += rg) {
        const int64_t m = (int64_t)b * P + p;
        const float hm = (h != nullptr) ? h[m * ldh + j] : 0.f, hl = (h != nullptr) ? h[m * ldh + Ch + j] : 0.f;
        const float mean = (hm + bm) * em, lg = (hl + bl) * el;
        const float g = dz[b * dz_bs + (int64_t)j * P + p];
        const float dlg = g * expf(lg) * temperature * eps[((int64_t)b * Ch + j) * P + p];
        const float dhm = g * em, dhl = dlg * el;
        if (h != nullptr) {
          dh[m * ldh + j] = dhm;
          dh[m * ldh + Ch + j] = dhl;
        }
        s_bm += dhm; s_bl += dhl;
        s_lm += 3.f * g * mean; s_ll += 3.f * dlg * lg;
      }
    }
    red[0][tid] = s_bm; red[1][tid] = s_bl; red[2][tid] = s_lm; red[3][tid] = s_ll;
    __syncthreads();
    for (int i = tid; i < 4 * cw; i += 256) {
      const int k = i / cw, jj = i % cw;
      float acc = 0.f;
      for (int q = 0; q < rg; ++q) acc += red[k][q * cw + jj];
      const int dst[4] = {j0 + jj, Ch + j0 + jj, C + j0 + jj, C + Ch + j0 + jj};
      dpar[(int64_t)b * 2 * C + dst[k]] = acc;
    }
    __syncthreads();
  }
  if (h != nullptr) {
    for (int i = tid; i < P * (int)(ldh - C); i += 256) {
      const int p = i / (int)(ldh - C), c = C + i % (int)(ldh - C);
      dh[((int64_t)b * P + p) * ldh + c] = 0.f;
    }
  }
}

// dstate[b, c, p] += sum_tap dA[(b,p - shift(tap)), c*9+tap]   for c < Cin  (col2im of a 3x3 "same" conv input gradient)
__global__ void col2im_add_kernel(const float* __restrict__ da, int64_t lda, float* __restrict__ dstate, int64_t dbs, int Cin,
                                  int H, int W, int64_t n) {
  const int P = H * W;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int p = (int)(i % P);
    int64_t r = i / P;
    const int c = (int)(r % Cin);
    const int64_t b = r / Cin;
    const int py = p / W, px = p - py * W;
    float acc = 0.f;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int yy = py - (tap / 3 - 1), xx = px - (tap % 3 - 1);
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) acc += da[(b * P + yy * W + xx) * lda + c * 9 + tap];
    }
    dstate[b * dbs + (int64_t)c * P + p] += acc;
  }
}

// tcgen05 path (gemm_tn_tc.cu)
void gemm_tn_tc_plan(int M, int N1, int N2, int* BN, int* tiles, int* splits, int* kb_per_split);
bool gemm_tn_tc_ok(const void* A, int64_t lda, const void* Bm, int64_t ldb, int N1, int N2);
int gemm_tn_tc(const void* A, int64_t lda, const void* Bm, int64_t ldb, float* ws, int M, int N1, int N2, int* splits_out,
               float* D, int accumulate, int* counters, int out_mode, int out_c, int x3, cudaStream_t st);

}  // namespace nfdpm

using namespace nfdpm;

static size_t coupling_bwd_smem(int C, int H, int W) {
  return sizeof(float) * coupling_bwd_floats(C, H, W, nullptr, nullptr);
}
static int coupling_bwd_tile(int C, int P) {
  int tp = P < 128 ? P : 128;
  while (tp > 8 && sizeof(float) * (4 * (size_t)(C / 2) * tp + 2 * C) > 96 * 1024) tp = (tp + 1) / 2;
  if (tp >= P) tp = (P + 1) / 2;       // the tiled path always has >= 2 tiles (tiles == 1 means "single-kernel path")
  return tp;
}
/* 1: the image fits one CTA (single kernel, dp_scratch unused); otherwise the number of pixel tiles per image: dpar has
 * B*tiles rows, dp_scratch [B*H*W*C] floats is required and the last-CTA reduction (counter) is not used. */
extern "C" int nfdpm_coupling_bwd_tiles(int C, int H, int W) {
  const int P = H * W;
  if (coupling_bwd_smem(C, H, W) <= 200 * 1024) return 1;
  const int tp = coupling_bwd_tile(C, P);
  return (P + tp - 1) / tp;
}

template <bool INV>
static int coupling_bwd_launch(const float* dy, int64_t dy_bs, const float* dld, const float* u, int64_t u_bs,
                               const float* pm, int64_t ldp, const float* bias3, const float* logs3, float* du,
                               int64_t du_bs, void* dpm, int dpm_dtype, int64_t ld_dpm, float* dpar, float* dbias,
                               float* dlogs, int32_t* counter, float* dp_scratch, int B, int C, int H, int W,
                               cudaStream_t st) {
  const char* name = INV ? "nfdpm_coupling_inv_bwd" : "nfdpm_coupling_bwd";
  NFDPM_REQUIRE(dy && u && pm && bias3 && logs3 && du && dpm && dpar, "%s: null pointer", name);
  NFDPM_REQUIRE(B > 0 && C > 0 && C % 2 == 0 && H > 0 && W > 0 && ldp >= 9 * (int64_t)C && ld_dpm >= 9 * (int64_t)C,
                "%s: bad shape", name);
  NFDPM_REQUIRE(dpm_dtype == NFDPM_F32 || dpm_dtype == NFDPM_BF16 || (dpm_dtype == NFDPM_BF16X2 && ld_dpm % 32 == 0),
                "%s: bad dpm dtype", name);
  NFDPM_REQUIRE(counter == nullptr || (dbias && dlogs), "%s: the fused reduction needs dbias/dlogs", name);
  const int P = H * W, Ch = C / 2;
  static bool attr_set = false;
  if (!attr_set) {
    NFDPM_CUDA(cudaFuncSetAttribute(coupling_bwd_kernel<float, INV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    NFDPM_CUDA(cudaFuncSetAttribute(coupling_bwd_kernel<__nv_bfloat16, INV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    NFDPM_CUDA(cudaFuncSetAttribute(coupling_bwd_kernel<bf16x2_t, INV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    NFDPM_CUDA(cudaFuncSetAttribute(coupling_bwd_tiled_kernel<INV>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    attr_set = true;
  }
  size_t smem = coupling_bwd_smem(C, H, W);
  if (smem <= 200 * 1024) {
    CouplingBwdArgs a{dy, dy_bs, dld, u, u_bs, pm, ldp, bias3, logs3, du, du_bs, dpm, ld_dpm, dpar, B, C, H, W, dbias, dlogs,
                      counter};
    a.dP = make_fastdiv(P); a.dW = make_fastdiv(W); a.dCh = make_fastdiv(Ch);
    a.dNg = make_fastdiv(ld_dpm >= 8 ? (int)(ld_dpm >> 3) : 1); a.d2C = make_fastdiv(2 * C);
    const size_t pm_bytes = (size_t)P * (size_t)ldp * sizeof(float);
    a.pm_bulk = (ldp % 4 == 0 && ((uintptr_t)pm % 16) == 0 && smem + pm_bytes <= 200 * 1024) ? 1 : 0;
    if (a.pm_bulk) smem += pm_bytes;
    int threads = (P * Ch + 31) / 32 * 32;
    threads = threads > 1024 ? 1024 : (threads < 128 ? 128 : threads);
    if (dpm_dtype == NFDPM_F32) coupling_bwd_kernel<float, INV><<<B, threads, smem, st>>>(a);
    else if (dpm_dtype == NFDPM_BF16X2) coupling_bwd_kernel<bf16x2_t, INV><<<B, threads, smem, st>>>(a);
    else coupling_bwd_kernel<__nv_bfloat16, INV><<<B, threads, smem, st>>>(a);
    NFDPM_CHECK_LAUNCH("coupling_bwd_kernel");
    return 0;
  }
  NFDPM_REQUIRE(dp_scratch != nullptr && counter == nullptr,
                "%s: this image needs the tiled path (dp_scratch, no fused reduction): see nfdpm_coupling_bwd_tiles", name);
  const int TP = coupling_bwd_tile(C, P), T = (P + TP - 1) / TP;
  CouplingBwdArgs a{dy, dy_bs, dld, u, u_bs, pm, ldp, bias3, logs3, du, du_bs, dpm, ld_dpm, dpar, B, C, H, W, nullptr,
                    nullptr, nullptr};
  a.dP = make_fastdiv(P); a.dW = make_fastdiv(W); a.dCh = make_fastdiv(Ch);
  a.dNg = make_fastdiv(ld_dpm >= 8 ? (int)(ld_dpm >> 3) : 1); a.d2C = make_fastdiv(2 * C);
  a.pm_bulk = 0;
  const size_t smem_t = sizeof(float) * (4 * (size_t)Ch * TP + 2 * C);
  coupling_bwd_tiled_kernel<INV><<<B * T, 256, smem_t, st>>>(a, dp_scratch, TP);
  NFDPM_CHECK_LAUNCH("coupling_bwd_tiled_kernel");
  const int64_t n = (int64_t)B * P * ld_dpm;
  int64_t g = (n + 255) / 256;
  if (g > 148 * 32) g = 148 * 32;
  if (dpm_dtype == NFDPM_F32) dpm_expand_kernel<float><<<(int)g, 256, 0, st>>>(dp_scratch, (float*)dpm, ld_dpm, C, H, W, n);
  else if (dpm_dtype == NFDPM_BF16X2) dpm_expand_kernel<bf16x2_t><<<(int)g, 256, 0, st>>>(dp_scratch, (bf16x2_t*)dpm, ld_dpm, C, H, W, n);
  else dpm_expand_kernel<__nv_bfloat16><<<(int)g, 256, 0, st>>>(dp_scratch, (__nv_bfloat16*)dpm, ld_dpm, C, H, W, n);
  NFDPM_CHECK_LAUNCH("dpm_expand_kernel");
  return 0;
}

extern "C" int nfdpm_coupling_bwd(const float* dy, int64_t dy_bs, const float* dld, const float* u, int64_t u_bs,
                                  const float* pm, int64_t ldp, const float* bias3, const float* logs3, float* du,
                                  int64_t du_bs, void* dpm, int dpm_dtype, int64_t ld_dpm, float* dpar, float* dbias,
                                  float* dlogs, int32_t* counter, float* dp_scratch, int B, int C, int H, int W,
                                  nfdpm_stream_t stream) {
  return coupling_bwd_launch<false>(dy, dy_bs, dld, u, u_bs, pm, ldp, bias3, logs3, du, du_bs, dpm, dpm_dtype, ld_dpm, dpar,
                                    dbias, dlogs, counter, dp_scratch, B, C, H, W, as_stream(stream));
}

extern "C" int nfdpm_coupling_inv_bwd(const float* dx, int64_t dx_bs, const float* y, int64_t y_bs, const float* pm,
                                      int64_t ldp, const float* bias3, const float* logs3, float* dy, int64_t dyo_bs,
                                      void* dpm, int dpm_dtype, int64_t ld_dpm, float* dpar, float* dbias, float* dlogs,
                                      int32_t* counter, float* dp_scratch, int B, int C, int H, int W,
                                      nfdpm_stream_t stream) {
  return coupling_bwd_launch<true>(dx, dx_bs, nullptr, y, y_bs, pm, ldp, bias3, logs3, dy, dyo_bs, dpm, dpm_dtype, ld_dpm,
                                   dpar, dbias, dlogs, counter, dp_scratch, B, C, H, W, as_stream(stream));
}

extern "C" int nfdpm_actnorm_relu_bwd(const void* dh, int dh_dtype, int64_t ld_dh, const void* h, int h_dtype, int64_t ld_h,
                                      const float* scale, void* dpre, int o_dtype, int64_t ld_o, float* part, int M,
                                      int N, int rows_per_cta, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(dh && h && scale && dpre && part, "nfdpm_actnorm_relu_bwd: null pointer");
  NFDPM_REQUIRE(M > 0 && N > 0 && rows_per_cta > 0, "nfdpm_actnorm_relu_bwd: bad shape");
  NFDPM_REQUIRE(N % 8 == 0 && N <= 2048 && ld_dh % 8 == 0 && ld_h % 8 == 0 && ld_o % 8 == 0,
                "nfdpm_actnorm_relu_bwd: N and the leading dimensions must be multiples of 8 (N <= 2048)");
  NFDPM_REQUIRE(((uintptr_t)dh % 16 == 0) && ((uintptr_t)h % 16 == 0) && ((uintptr_t)dpre % 16 == 0),
                "nfdpm_actnorm_relu_bwd: operands must be 16-byte aligned");
  const int grid = (M + rows_per_cta - 1) / rows_per_cta;
  const int cg = N / 8;
  NFDPM_REQUIRE(cg <= 256, "nfdpm_actnorm_relu_bwd: N too large");
  const int rg = 256 / cg;
  const size_t smem = sizeof(float) * (size_t)rg * 2 * N;
  cudaStream_t st = as_stream(stream);
#define GO(TD, TH, TO) actnorm_relu_bwd_kernel<TD, TH, TO><<<grid, 256, smem, st>>>((const TD*)dh, (const TH*)h, scale, (TO*)dpre, part, M, N, ld_dh, ld_h, ld_o, rows_per_cta)
  if (h_dtype == NFDPM_BF16X2 || o_dtype == NFDPM_BF16X2) {
    // fp32-faithful training: fp32 dh from the split-pair dgrad GEMM, split-pair stash h, split-pair dpre for the next GEMMs
    NFDPM_REQUIRE(dh_dtype == NFDPM_F32 && h_dtype == NFDPM_BF16X2 && o_dtype == NFDPM_BF16X2 && ld_h % 32 == 0 && ld_o % 32 == 0,
                  "nfdpm_actnorm_relu_bwd: the split-pair form is (fp32 dh, split h) -> split dpre with ld %% 32 == 0");
    GO(float, bf16x2_t, bf16x2_t);
    NFDPM_CHECK_LAUNCH("actnorm_relu_bwd_kernel");
    return 0;
  }
  const int key = (dh_dtype == NFDPM_BF16 ? 4 : 0) | (h_dtype == NFDPM_BF16 ? 2 : 0) | (o_dtype == NFDPM_BF16 ? 1 : 0);
  NFDPM_REQUIRE((dh_dtype == NFDPM_F32 || dh_dtype == NFDPM_BF16) && (h_dtype == NFDPM_F32 || h_dtype == NFDPM_BF16) &&
                (o_dtype == NFDPM_F32 || o_dtype == NFDPM_BF16), "nfdpm_actnorm_relu_bwd: bad dtypes");
  switch (key) {
    case 0: GO(float, float, float); break;
    case 1: GO(float, float, __nv_bfloat16); break;
    case 2: GO(float, __nv_bfloat16, float); break;
    case 3: GO(float, __nv_bfloat16, __nv_bfloat16); break;
    case 4: GO(__nv_bfloat16, float, float); break;
    case 5: GO(__nv_bfloat16, float, __nv_bfloat16); break;
    case 6: GO(__nv_bfloat16, __nv_bfloat16, float); break;
    default: GO(__nv_bfloat16, __nv_bfloat16, __nv_bfloat16); break;
  }
#undef GO
  NFDPM_CHECK_LAUNCH("actnorm_relu_bwd_kernel");
  return 0;
}

extern "C" int nfdpm_reduce_rows2(const float* part, float* out0, float* out1, int R, int n0, int n1, int64_t stride,
                                  nfdpm_stream_t stream) {
  NFDPM_REQUIRE(part && out0 && out1 && R > 0 && n0 > 0 && n1 > 0 && stride >= n0 + n1, "nfdpm_reduce_rows2: bad arguments");
  reduce_rows2_kernel<<<(n0 + n1 + 31) / 32, 256, 0, as_stream(stream)>>>(part, out0, out1, R, n0, n1, stride);
  NFDPM_CHECK_LAUNCH("reduce_rows2_kernel");
  return 0;
}

extern "C" int nfdpm_reduce_rows(const float* part, float* out, int R, int n, int64_t stride, int accumulate,
                                 nfdpm_stream_t stream) {
  NFDPM_REQUIRE(part && out && R > 0 && n > 0 && stride >= n, "nfdpm_reduce_rows: bad arguments");
  reduce_rows_kernel<<<(n + 31) / 32, 256, 0, as_stream(stream)>>>(part, out, R, n, stride, accumulate);
  NFDPM_CHECK_LAUNCH("reduce_rows_kernel");
  return 0;
}

static int mix_bwd_tile(int C, int P) {
  static int cap = -1;
  if (cap < 0) {
    const char* e = getenv("NFDPM_MIXBWD_TP");
    cap = e ? atoi(e) : 256;
    if (cap < 8) cap = 256;
  }
  int tp = P < cap ? P : cap;
  while (tp > 8 && sizeof(float) * (2 * (size_t)C * (tp + 1) + (size_t)C * C) > 200 * 1024) tp = (tp + 1) / 2;
  return tp;
}
/* number of pixel tiles per image of nfdpm_mix_bwd (rows of `part` per image) */
extern "C" int nfdpm_mix_bwd_tiles(int C, int H, int W) {
  const int P = H * W, tp = mix_bwd_tile(C, P);
  return (P + tp - 1) / tp;
}

extern "C" int nfdpm_mix_bwd(const float* du, int64_t du_bs, const float* da1, int64_t lda1, const float* x, int64_t x_bs,
                             const float* mt, float* dx, int64_t dx_bs, float* part, int B, int C, int H, int W,
                             nfdpm_stream_t stream) {
  NFDPM_REQUIRE(du && x && mt && dx && part, "nfdpm_mix_bwd: null pointer");
  NFDPM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "nfdpm_mix_bwd: bad shape");
  NFDPM_REQUIRE(da1 == nullptr || (C % 2 == 0 && lda1 >= 9 * (int64_t)(C / 2)), "nfdpm_mix_bwd: bad im2col gradient");
  const int P = H * W, TP = mix_bwd_tile(C, P), T = (P + TP - 1) / TP;
  const size_t smem = sizeof(float) * (2 * (size_t)C * (TP + 1) + (size_t)C * C);
  NFDPM_REQUIRE(smem <= 200 * 1024, "nfdpm_mix_bwd: %d channels do not fit shared memory (%zu bytes)", C, smem);
  MixBwdArgs a{du, du_bs, da1, lda1, x, x_bs, mt, dx, dx_bs, part, B, C, H, W, TP};
  a.dC = make_fastdiv(C); a.dCh = make_fastdiv(C / 2 > 0 ? C / 2 : 1); a.dW = make_fastdiv(W); a.dT = make_fastdiv(T);
  a.dNpFull = make_fastdiv(TP); a.dNpLast = make_fastdiv(P - (T - 1) * TP);
  static bool attr_set = false;
  if (!attr_set) {
    NFDPM_CUDA(cudaFuncSetAttribute(mix_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set = true;
  }
  int threads = (TP * C + 31) / 32 * 32;
  if (TP < 64 && threads < 512) threads = 512;       // per-element partial sums at deep levels
  threads = threads > 1024 ? 1024 : (threads < 128 ? 128 : threads);
  mix_bwd_kernel<<<B * T, threads, smem, as_stream(stream)>>>(a);
  NFDPM_CHECK_LAUNCH("mix_bwd_kernel");
  return 0;
}

extern "C" int nfdpm_mix_param_grad(const nfdpm_mix_grad_item* items, int n, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(items && n > 0, "nfdpm_mix_param_grad: no items");
  for (int base = 0; base < n; base += kParamBatch) {
    MixParamBatch pb;
    const int cnt = (n - base < kParamBatch) ? n - base : kParamBatch;
    for (int i = 0; i < cnt; ++i) {
      const nfdpm_mix_grad_item& s = items[base + i];
      NFDPM_REQUIRE(s.part && s.weight && s.winv && s.dld_sum && s.scratch && s.C > 0 && s.B > 0,
                    "nfdpm_mix_param_grad: item %d incomplete", base + i);
      pb.it[i] = MixParamItem{s.part, s.B, s.weight, s.scale, s.bias, s.winv, s.dld_sum, s.P, s.d_weight, s.d_scale,
                              s.d_bias, s.scratch, s.C};
    }
    mix_param_grad_kernel<<<cnt, 256, 0, as_stream(stream)>>>(pb);
    NFDPM_CHECK_LAUNCH("mix_param_grad_kernel");
  }
  return 0;
}

extern "C" int nfdpm_mix_inv_param_grad(const nfdpm_mix_grad_item* items, int n, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(items && n > 0, "nfdpm_mix_inv_param_grad: no items");
  for (int i = 0; i < n; ++i) {
    const nfdpm_mix_grad_item& s = items[i];
    NFDPM_REQUIRE(s.part && s.winv && s.scratch && s.C > 0 && s.B > 0 && (s.d_scale == nullptr || s.scale != nullptr),
                  "nfdpm_mix_inv_param_grad: item %d incomplete", i);
    NFDPM_REQUIRE(sizeof(float) * (size_t)s.C * s.C <= 200 * 1024, "nfdpm_mix_inv_param_grad: %d channels do not fit", s.C);
  }
  static bool attr_set = false;
  if (!attr_set) {
    NFDPM_CUDA(cudaFuncSetAttribute(mix_inv_param_grad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set = true;
  }
  for (int base = 0; base < n; base += kParamBatch) {
    MixParamBatch pb;
    const int cnt = (n - base < kParamBatch) ? n - base : kParamBatch;
    int cmax = 0;
    for (int i = 0; i < cnt; ++i) {
      const nfdpm_mix_grad_item& s = items[base + i];
      pb.it[i] = MixParamItem{s.part, s.B, s.weight, s.scale, s.bias, s.winv, nullptr, s.P, s.d_weight, s.d_scale,
                              s.d_bias, s.scratch, s.C};
      if (s.C > cmax) cmax = s.C;
    }
    mix_inv_param_grad_kernel<<<cnt, 256, sizeof(float) * (size_t)cmax * cmax, as_stream(stream)>>>(pb);
    NFDPM_CHECK_LAUNCH("mix_inv_param_grad_kernel");
  }
  return 0;
}

extern "C" int64_t nfdpm_gemm_tn_workspace(int M, int N1, int N2, int* splits_out) {
  // enough splits to fill the GPU (~296 CTAs) but at least 256 rows per split
  const int tiles = ((N1 + 127) / 128) * ((N2 + 127) / 128);
  int splits = (296 + tiles - 1) / tiles;
  const int max_splits = (M + 255) / 256;
  if (splits > max_splits) splits = max_splits;
  if (splits < 1) splits = 1;
  if (splits_out) *splits_out = splits;
  // the tensor-core path (bf16 operands) splits M differently: size the workspace for whichever is larger
  int bn, t, s_tc, per;
  gemm_tn_tc_plan(M, N1, N2, &bn, &t, &s_tc, &per);
  const int smax = splits > s_tc ? splits : s_tc;
  // split-pair operands: the accumulator covers 2 x 2 bf16 columns per logical element (whole groups of 64)
  const int n1m = 2 * ((N1 + 31) / 32 * 32), n2m = 2 * ((N2 + 31) / 32 * 32);
  int s_x3;
  gemm_tn_tc_plan(M, n1m, n2m, &bn, &t, &s_x3, &per);
  const int64_t plain = (int64_t)smax * N1 * N2, x3 = (int64_t)s_x3 * n1m * n2m;
  return plain > x3 ? plain : x3;
}

extern "C" int nfdpm_gemm_tn(const void* A, int a_dtype, int64_t lda, const void* Bm, int b_dtype, int64_t ldb, float* D,
                             int64_t ldd, int M, int N1, int N2, float* ws, int accumulate, int32_t* counters,
                             int out_mode, int out_c, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(A && Bm && D && ws, "nfdpm_gemm_tn: null pointer");
  NFDPM_REQUIRE(M > 0 && N1 > 0 && N2 > 0 && lda >= N1 && ldb >= N2 && ldd == N2, "nfdpm_gemm_tn: bad shape (ldd must equal N2)");
  NFDPM_REQUIRE(out_mode >= NFDPM_TN_OUT_PLAIN && out_mode <= NFDPM_TN_OUT_STRIP && (out_mode == NFDPM_TN_OUT_PLAIN || out_c > 0),
                "nfdpm_gemm_tn: bad output mode");
  cudaStream_t st = as_stream(stream);
  const int n = N1 * N2;
  if (a_dtype == NFDPM_BF16X2 || b_dtype == NFDPM_BF16X2) {
    NFDPM_REQUIRE(a_dtype == b_dtype && lda % 32 == 0 && ldb % 32 == 0 && N2 % 4 == 0 && lda >= (N1 + 31) / 32 * 32 &&
                  ldb >= (N2 + 31) / 32 * 32 && ((uintptr_t)A % 16 == 0) && ((uintptr_t)Bm % 16 == 0) && counters != nullptr,
                  "nfdpm_gemm_tn: split-pair operands need both operands split, ld %% 32 == 0 covering whole column groups, "
                  "N2 %% 4 == 0 and counters");
    int s_tc = 1;
    return gemm_tn_tc(A, lda, Bm, ldb, ws, M, N1, N2, &s_tc, D, accumulate, counters, out_mode, out_c, 1, st);
  }
  if (a_dtype == NFDPM_BF16 && b_dtype == NFDPM_BF16 && gemm_tn_tc_ok(A, lda, Bm, ldb, N1, N2)) {
    int s_tc = 1;
    if (gemm_tn_tc(A, lda, Bm, ldb, ws, M, N1, N2, &s_tc, D, accumulate, counters, out_mode, out_c, 0, st)) return 1;
    if (s_tc > 0) {                                     // not reduced in-kernel
      reduce_rows_kernel<<<(n + 31) / 32, 256, 0, st>>>(ws, D, s_tc, n, n, accumulate);
      NFDPM_CHECK_LAUNCH("reduce_rows_kernel");
    }
    return 0;
  }
  NFDPM_REQUIRE(out_mode == NFDPM_TN_OUT_PLAIN, "nfdpm_gemm_tn: layout-changing outputs need bf16 operands + counters");
  int splits = 1;
  nfdpm_gemm_tn_workspace(M, N1, N2, &splits);
  int rows = (M + splits - 1) / splits;
  rows = (rows + 15) / 16 * 16;
  splits = (M + rows - 1) / rows;
  dim3 grid((N2 + 127) / 128, (N1 + 127) / 128, splits);
#define GO(TA, TB) gemm_tn_kernel<TA, TB><<<grid, 256, 0, st>>>((const TA*)A, lda, (const TB*)Bm, ldb, ws, M, N1, N2, rows)
  if (a_dtype == NFDPM_F32 && b_dtype == NFDPM_F32) GO(float, float);
  else if (a_dtype == NFDPM_F32 && b_dtype == NFDPM_BF16) GO(float, __nv_bfloat16);
  else if (a_dtype == NFDPM_BF16 && b_dtype == NFDPM_BF16) GO(__nv_bfloat16, __nv_bfloat16);
  else if (a_dtype == NFDPM_BF16 && b_dtype == NFDPM_F32) GO(__nv_bfloat16, float);
  else return fail("nfdpm_gemm_tn: bad dtypes");
#undef GO
  NFDPM_CHECK_LAUNCH("gemm_tn_kernel");
  reduce_rows_kernel<<<(n + 31) / 32, 256, 0, st>>>(ws, D, splits, n, n, accumulate);
  NFDPM_CHECK_LAUNCH("reduce_rows_kernel");
  return 0;
}

extern "C" int nfdpm_split_prior_bwd(const float* dlp, const float* h, int64_t ldh, const float* bias, const float* logs,
                                     const float* x, int64_t xbs, float* dstate, int64_t dbs, float* dh, float* dpar,
                                     int B, int C, int H, int W, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(dlp && x && dstate, "nfdpm_split_prior_bwd: null pointer");
  NFDPM_REQUIRE(h == nullptr || (bias && logs && dh && dpar && ldh >= C), "nfdpm_split_prior_bwd: learned prior needs bias/logs/dh/dpar");
  NFDPM_REQUIRE(B > 0 && C > 0 && C % 2 == 0 && H > 0 && W > 0, "nfdpm_split_prior_bwd: bad shape");
  split_prior_bwd_kernel<<<B, 256, sizeof(float) * 2 * C, as_stream(stream)>>>(dlp, h, ldh, bias, logs, x, xbs, dstate, dbs,
                                                                                dh, dpar, B, C, H * W);
  NFDPM_CHECK_LAUNCH("split_prior_bwd_kernel");
  return 0;
}

extern "C" int nfdpm_gauss_const_bwd(const float* dl, const float* z, const float* bias, const float* logs, float* dz,
                                     float* dpar, int B, int C, int P, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(dl && z && dz, "nfdpm_gauss_const_bwd: null pointer");
  NFDPM_REQUIRE((bias == nullptr) == (logs == nullptr) && (bias == nullptr || dpar), "nfdpm_gauss_const_bwd: bias/logs/dpar mismatch");
  NFDPM_REQUIRE(B > 0 && C > 0 && P > 0, "nfdpm_gauss_const_bwd: bad shape");
  gauss_const_bwd_kernel<<<B, 256, 0, as_stream(stream)>>>(dl, z, bias, logs, dz, dpar, C, P);
  NFDPM_CHECK_LAUNCH("gauss_const_bwd_kernel");
  return 0;
}

extern "C" int nfdpm_split_sample_bwd(const float* dz, int64_t dz_bs, const float* eps, float temperature, const float* h,
                                      int64_t ldh, const float* bias, const float* logs, float* dh, float* dpar, int B, int C,
                                      int H, int W, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(dz && eps && bias && logs && dpar, "nfdpm_split_sample_bwd: null pointer");
  NFDPM_REQUIRE(h == nullptr || (dh && ldh >= C), "nfdpm_split_sample_bwd: the conditional form needs dh with ldh >= C");
  NFDPM_REQUIRE(B > 0 && C > 0 && C % 2 == 0 && H > 0 && W > 0, "nfdpm_split_sample_bwd: bad shape");
  split_sample_bwd_kernel<<<B, 256, 0, as_stream(stream)>>>(dz, dz_bs, eps, temperature, h, ldh, bias,
                                                                                 logs, dh, dpar, C, H * W);
  NFDPM_CHECK_LAUNCH("split_sample_bwd_kernel");
  return 0;
}

extern "C" int nfdpm_col2im_add(const float* da, int64_t lda, float* dstate, int64_t dbs, int B, int Cin, int H, int W,
                                nfdpm_stream_t stream) {
  NFDPM_REQUIRE(da && dstate, "nfdpm_col2im_add: null pointer");
  NFDPM_REQUIRE(B > 0 && Cin > 0 && H > 0 && W > 0 && lda >= 9 * (int64_t)Cin, "nfdpm_col2im_add: bad shape");
  const int64_t n = (int64_t)B * Cin * H * W;
  int64_t g = (n + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  col2im_add_kernel<<<(int)g, 256, 0, as_stream(stream)>>>(da, lda, dstate, dbs, Cin, H, W, n);
  NFDPM_CHECK_LAUNCH("col2im_add_kernel");
  return 0;
}
