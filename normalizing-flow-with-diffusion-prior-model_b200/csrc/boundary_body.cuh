// The arithmetic of one step boundary for ONE image, shared by flow_boundary_kernel (one CTA per image) and the fused
// deep-level StepFlow kernel (deep_step.cu).  See flow_boundary.cu for the description.  Internal header.
#pragma once
#include "tc_common.cuh"

namespace nfdpm {


struct BoundaryArgs {
  const float* in; int64_t in_bs;       // source state [B,C,P] (or [B,C/4,2H,2W] when squeeze_in)
  const float* pm; int64_t ldp;         // SRC_COUPLING: taps-as-N rows [B*P, ldp]
  const float* bias3; const float* logs3;
  float* ld_part;                       // coupling, either direction: [B] per-image sum of log(s + 1e-6) (may be null)
  const float* mt; const float* beta;   // mix (null = identity)
  float* y; int64_t y_bs;               // NCHW sink (may be null)
  float* xs; int64_t xs_bs;             // NCHW sink of the PRE-mix state (training stash of the next step's input; may be null)
  void* a1; int64_t lda1;               // im2col sink (may be null)
  int B, C, H, W;
  int squeeze_in, inverse;
  FastDiv dP, dW, dCp, dCh, dNg;        // H*W, W, round4(C), C/2, lda1/8 (boundary_fill_div)
};

// host: fill the divisors once every other field is set
static inline void boundary_fill_div(BoundaryArgs& a) {
  a.dP = make_fastdiv(a.H * a.W);
  a.dW = make_fastdiv(a.W);
  a.dCp = make_fastdiv((a.C + 3) & ~3);
  a.dCh = make_fastdiv(a.C / 2 > 0 ? a.C / 2 : 1);
  a.dNg = make_fastdiv(a.lda1 >= 8 ? (int)(a.lda1 >> 3) : 1);
}

// profiling hook of this translation unit (nfdpm_flow_boundary_debug): per-CTA phase timeline [B][16] int64, NULL = off
static __device__ long long* g_bd_dbg = nullptr;

// eight consecutive columns k0..k0+7 (k0 % 8 == 0) of row `row` of the im2col sink [rows, ld] (ld counts logical columns)
template <typename T> __device__ __forceinline__ void store8(T* base, int64_t row, int64_t ld, int k0, const float (&v)[8]);
template <> __device__ __forceinline__ void store8<float>(float* base, int64_t row, int64_t ld, int k0, const float (&v)[8]) {
  float* p = base + row * ld + k0;
  *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  *reinterpret_cast<float4*>(p + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
template <> __device__ __forceinline__ void store8<__nv_bfloat16>(__nv_bfloat16* base, int64_t row, int64_t ld, int k0,
                                                                  const float (&v)[8]) {
  uint32_t w[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 t = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    w[i] = *reinterpret_cast<uint32_t*>(&t);
  }
  *reinterpret_cast<uint4*>(base + row * ld + k0) = make_uint4(w[0], w[1], w[2], w[3]);
}
template <> __device__ __forceinline__ void store8<bf16x2_t>(bf16x2_t* base, int64_t row, int64_t ld, int k0,
                                                             const float (&v)[8]) {
  split_store8(reinterpret_cast<__nv_bfloat16*>(base) + 2 * row * ld, k0, v);
}

// host: run `GO(type)` with the element type of an im2col sink of dtype code `dt` (NFDPM_F32 when there is no sink)
#define NFDPM_A1_DISPATCH(dt, GO)                    \
  do {                                               \
    if ((dt) == NFDPM_BF16) { GO(__nv_bfloat16); }   \
    else if ((dt) == NFDPM_BF16X2) { GO(bf16x2_t); } \
    else { GO(float); }                              \
  } while (0)


// Shared-memory scratch of the body in floats (nfdpm_flow_boundary_smem() returns it in bytes):
//   x_s [C][P+1] | u_s [C][P+1] (mix only) | m_s [C][Cp] + beta [Cp] (mix only) | par_s [2C] | ls_s [P*C/2] (coupling only)
//   | pad_s [C/2][(H+2)*(W+2)]  zero-bordered copy of the channels the next coupling network reads (im2col source)
//   | kt_s  [9*C/2] int         im2col column k -> offset of its (channel, tap) inside pad_s
__host__ __device__ __forceinline__ size_t boundary_scratch_floats(int C, int H, int W, bool coupling, bool mix, size_t* pad_off,
                                                                   size_t* kt_off) {
  const size_t P = (size_t)H * W, PS = P + 1, Cp = (C + 3) & ~3, Ch = C / 2;
  size_t fl = (size_t)C * PS * (mix ? 2 : 1);
  if (mix) fl += (size_t)C * Cp + Cp;
  if (coupling) fl += 2 * (size_t)C + P * Ch;
  fl = (fl + 3) & ~(size_t)3;
  if (pad_off) *pad_off = fl;
  fl += (Ch * (size_t)(H + 2) * (W + 2) + 3) & ~(size_t)3;
  if (kt_off) *kt_off = fl;
  fl += (9 * Ch + 3) & ~(size_t)3;
  return fl;
}

// `sm`: shared-memory scratch of nfdpm_flow_boundary_smem() bytes; all `nt` threads of the CTA must call this together.
// PM_SMEM: the taps-as-N rows of image b are (or will be: pm_bar) in shared memory at `pm_img` (row stride `pm_ld` floats)
// instead of a.pm in global memory; pm_bar != 0: shared-memory address of an mbarrier (phase 0) that completes when a bulk
// copy has landed them (flow_boundary.cu).
template <bool COUPLING, typename A1T, bool PM_SMEM = false>
__device__ __forceinline__ void flow_boundary_body(const BoundaryArgs& a, const int b, float* sm, const int tid, const int nt,
                                                   const float* pm_img = nullptr, const int pm_ld = 0,
                                                   const uint32_t pm_bar = 0) {
  const int C = a.C, H = a.H, W = a.W, P = H * W, Ch = C >> 1;
  long long* const dbg = g_bd_dbg;
  auto stamp = [&](int slot) {
    if (dbg != nullptr && tid == 0) dbg[(int64_t)b * 16 + slot] = clock64();
  };
  stamp(0);
  const int PS = P + 1;                       // padded pixel stride: conflict-free for lanes over channels
  const int Cp = (C + 3) & ~3;
  const int W2p = W + 2, PP = (H + 2) * W2p;  // zero-bordered image of one channel
  const bool mix = a.mt != nullptr;
  const bool want_a1 = a.a1 != nullptr;
  size_t pad_off, kt_off;
  boundary_scratch_floats(C, H, W, COUPLING, mix, &pad_off, &kt_off);
  float* x_s = sm;                            // [C][PS]  source / coupling result
  float* u_s = x_s + C * PS;                  // [C][PS]  mixed result (aliases x_s when there is no mix)
  float* m_s = mix ? u_s + C * PS : u_s;      // [C][Cp] + beta [Cp]
  float* par_s = m_s + (mix ? (C * Cp + Cp) : 0);                 // [2C] bias3, exp(3 logs3)
  float* ls_s = par_s + (COUPLING ? 2 * C : 0);                   // [P*Ch] log-det terms
  float* pad_s = sm + pad_off;                                    // [Ch][PP]
  int* kt_s = reinterpret_cast<int*>(sm + kt_off);                // [9*Ch]
  if (!mix) u_s = x_s;

  // ---- phase 0: parameters + the image, channel-major (lanes over pixels -> coalesced).  Every global load of a batch is
  // issued before the first dependent shared-memory store: the warps issue in order, so load -> store -> load chains would
  // serialise one L2 round trip per element (r1 timeline: 2.1 us for 3 elements per thread).
  const float* inb = a.in + (int64_t)b * a.in_bs;
  const int nx = C * P;
  float xv[4];
  if (!a.squeeze_in) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = tid + u * nt;
      xv[u] = (i < nx) ? inb[i] : 0.f;
    }
  }
  {
    const int n_m = mix ? C * Cp : 0;
    float mv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = tid + u * nt;
      mv[u] = 0.f;
      if (i < n_m) {
        const int r = fdiv(i, a.dCp), c = i - r * Cp;
        if (c < C) mv[u] = a.mt[r * C + c];
      }
    }
    const float bev = (mix && tid < C) ? a.beta[tid] : 0.f;
    const float b3v = (COUPLING && tid < C) ? a.bias3[tid] : 0.f;
    const float l3v = (COUPLING && tid < C) ? a.logs3[tid] : 0.f;
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = tid + u * nt;
      if (i < n_m) m_s[i] = mv[u];
    }
    for (int i = tid + 4 * nt; i < n_m; i += nt) {                // shapes with more than 4 matrix entries per thread
      const int r = fdiv(i, a.dCp), c = i - r * Cp;
      m_s[i] = (c < C) ? a.mt[r * C + c] : 0.f;
    }
    if (mix) {
      if (tid < Cp) m_s[C * Cp + tid] = bev;
      for (int i = tid + nt; i < Cp; i += nt) m_s[C * Cp + i] = (i < C) ? a.beta[i] : 0.f;
    }
    if (COUPLING) {
      if (tid < C) {
        par_s[tid] = b3v;
        par_s[C + tid] = expf(3.f * l3v);
      }
      for (int i = tid + nt; i < C; i += nt) {
        par_s[i] = a.bias3[i];
        par_s[C + i] = expf(3.f * a.logs3[i]);
      }
    }
  }
  if (want_a1) {
    for (int i = tid; i < Ch * PP; i += nt) pad_s[i] = 0.f;       // borders stay zero; the interior is filled below
    for (int k = tid; k < 9 * Ch; k += nt) {
      const int c = k / 9, tap = k - c * 9;
      kt_s[k] = c * PP + (tap / 3) * W2p + (tap % 3);
    }
  }
  if (a.squeeze_in) {
    // in is [C/4, 2H, 2W]; channel c = cc*4 + h1*2 + w1 reads in[cc, 2y+h1, 2x+w1]
    const int W2 = 2 * W;
    for (int i = tid; i < (C >> 2) * P; i += nt) {
      const int cc = fdiv(i, a.dP), p = i - cc * P;
      const int py = fdiv(p, a.dW), px = p - py * W;
      const float* s = inb + ((int64_t)cc * 2 * H + 2 * py) * W2 + 2 * px;
      const float2 t0 = *reinterpret_cast<const float2*>(s), t1 = *reinterpret_cast<const float2*>(s + W2);
      x_s[(cc * 4 + 0) * PS + p] = t0.x;
      x_s[(cc * 4 + 1) * PS + p] = t0.y;
      x_s[(cc * 4 + 2) * PS + p] = t1.x;
      x_s[(cc * 4 + 3) * PS + p] = t1.y;
    }
  } else {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = tid + u * nt;
      if (i < nx) {
        const int c = fdiv(i, a.dP), p = i - c * P;
        x_s[c * PS + p] = xv[u];
      }
    }
    for (int base = tid + 4 * nt; base < nx; base += 4 * nt) {
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * nt;
        v[u] = (i < nx) ? inb[i] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int i = base + u * nt;
        if (i < nx) {
          const int c = fdiv(i, a.dP), p = i - c * P;
          x_s[c * PS + p] = v[u];
        }
      }
    }
  }
  __syncthreads();
  stamp(1);

  // ---- phase 1: affine coupling, item = (pixel, j) with j fastest (pm rows read contiguously)
  if (COUPLING) {
    if (PM_SMEM && pm_bar != 0) mbar_wait(pm_bar, 0);             // the bulk copy of the image's pm rows has landed
    const float* pmb = PM_SMEM ? pm_img : a.pm + (int64_t)b * P * a.ldp;
    const int64_t ldp = PM_SMEM ? (int64_t)pm_ld : a.ldp;
    for (int it = tid; it < P * Ch; it += nt) {
      const int p = fdiv(it, a.dCh), j = it - p * Ch;
      const int py = fdiv(p, a.dW), px = p - py * W;
      // all 18 loads are issued before the first use (each pm element is consumed exactly once: plain streaming reads)
      float lv[9], tv[9];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const int yy = py + tap / 3 - 1, xx = px + tap % 3 - 1;
        const bool ok = (yy >= 0) && (yy < H) && (xx >= 0) && (xx < W);
        const float* r = pmb + (int64_t)(ok ? yy * W + xx : p) * ldp + tap * C + j;
        const float l0 = PM_SMEM ? r[0] : __ldg(r), t0 = PM_SMEM ? r[Ch] : __ldg(r + Ch);
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
      const float xb = x_s[(Ch + j) * PS + p];
      if (a.inverse) {
        x_s[(Ch + j) * PS + p] = xb / (s + 1e-6f) - sh_t;
        // the forward's term: the same s (from the same pass-through half) that the inverse divides by
        if (a.ld_part != nullptr) ls_s[it] = logf(s + 1e-6f);
      } else {
        x_s[(Ch + j) * PS + p] = (xb + sh_t) * s;
        ls_s[it] = logf(s + 1e-6f);
      }
    }
    __syncthreads();
    stamp(2);
    if (a.ld_part != nullptr && tid < 32) {
      // deterministic per-image sum: fixed lane-strided order + shuffle tree
      float acc = 0.f;
#pragma unroll 8
      for (int i = tid; i < P * Ch; i += 32) acc += ls_s[i];        // (unrolled: the loads pipeline, the order is unchanged)
      acc = warp_sum(acc);
      if (tid == 0) a.ld_part[b] = acc;
    }
  }

  stamp(3);
  // ---- phase 1b: stash the pre-mix state (the next StepFlow's input, needed by its backward)
  if (a.xs != nullptr) {
    float* xb = a.xs + (int64_t)b * a.xs_bs;
    for (int i = tid; i < C * P; i += nt) {
      const int c = fdiv(i, a.dP), p = i - c * P;
      xb[i] = x_s[c * PS + p];
    }
  }

  stamp(4);
  // ---- phase 2: channel mix, item = (group of 4 outputs, pixel), lanes over pixels
  if (mix) {
    const int n_og = Cp >> 2;
    for (int it = tid; it < n_og * P; it += nt) {
      const int og = fdiv(it, a.dP), p = it - og * P;
      const float4 b4 = *reinterpret_cast<const float4*>(m_s + C * Cp + og * 4);
      float a0 = b4.x, a1 = b4.y, a2 = b4.z, a3 = b4.w;
#pragma unroll 4
      for (int c = 0; c < C; ++c) {                                // same summation order; unrolled so the loads pipeline
        const float xv_ = x_s[c * PS + p];
        const float4 w = *reinterpret_cast<const float4*>(m_s + c * Cp + og * 4);
        a0 = fmaf(w.x, xv_, a0);
        a1 = fmaf(w.y, xv_, a1);
        a2 = fmaf(w.z, xv_, a2);
        a3 = fmaf(w.w, xv_, a3);
      }
      const int o = og * 4;
      u_s[o * PS + p] = a0;
      if (o + 1 < C) u_s[(o + 1) * PS + p] = a1;
      if (o + 2 < C) u_s[(o + 2) * PS + p] = a2;
      if (o + 3 < C) u_s[(o + 3) * PS + p] = a3;
    }
    __syncthreads();
  }
  if (want_a1) {
    // interior of the zero-bordered copy: the channels the next coupling network reads (without a mix: x_a, which passes
    // through the coupling unchanged)
    for (int i = tid; i < Ch * P; i += nt) {
      const int c = fdiv(i, a.dP), p = i - c * P;
      const int py = fdiv(p, a.dW), px = p - py * W;
      pad_s[c * PP + (py + 1) * W2p + px + 1] = u_s[c * PS + p];
    }
  }

  stamp(5);
  // ---- phase 3a: NCHW sink (lanes over pixels)
  if (a.y != nullptr) {
    float* yb = a.y + (int64_t)b * a.y_bs;
    for (int i = tid; i < C * P; i += nt) {
      const int c = fdiv(i, a.dP), p = i - c * P;
      yb[i] = u_s[c * PS + p];
    }
  }
  stamp(6);
  if (want_a1) __syncthreads();
  // ---- phase 3b: im2col sink, item = (pixel, 8-column group), group fastest -> 128-byte runs per row.  Column k = c*9 + tap
  // of pixel (py, px) is pad_s[kt_s[k] + py*(W+2) + px]: no bounds tests, no divisions by 9 in the inner loop.
  if (want_a1) {
    const int K = Ch * 9;
    const int n_g = (int)(a.lda1 >> 3);
    A1T* a1b = reinterpret_cast<A1T*>(a.a1);
    for (int it = tid; it < P * n_g; it += nt) {
      const int p = fdiv(it, a.dNg), g = it - p * n_g;
      const int py = fdiv(p, a.dW), px = p - py * W;
      const float* win = pad_s + py * W2p + px;
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int k = g * 8 + e;
        v[e] = (k < K) ? win[kt_s[k]] : 0.f;
      }
      store8<A1T>(a1b, (int64_t)b * P + p, a.lda1, g * 8, v);
    }
  }
  stamp(7);
}

}  // namespace nfdpm
