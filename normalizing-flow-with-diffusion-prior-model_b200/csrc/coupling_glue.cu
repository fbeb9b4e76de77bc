// Memory-bound kernels around the coupling-network GEMMs:
//   im2col3x3           NCHW fp32 -> pixel-major im2col rows (fp32 or bf16) for the first 3x3 conv
//   pack_matrix         weight layout/cast for the GEMM B operands
//   coupling_apply      3x3 gather-add of the taps-as-N ZeroConv output + bias/exp(3 logs) + sigmoid affine
//                       transform (forward / inverse) + per-image log-det partial sums
//   split_prior_logp    Split: latent copy-out + learned Gaussian prior log-density
//   split_prior_sample  Split.invert without a latent
#include "common.cuh"

namespace nfdpm {

constexpr int TPB = 256;  // pixels per CTA in the per-pixel kernels (must match nfdpm_ld_tiles)


// One thread per (pixel m, input channel c): writes the 9 taps of that channel, columns c*9 .. c*9+8.
// Threads of a warp share c and walk consecutive pixels => coalesced NCHW reads.  Pad columns are zeroed
// by the threads with c == Cin-1... (done by a dedicated range below to keep the hot loop branch-free).
template <typename T>
__global__ void im2col3x3_kernel(const float* __restrict__ x, T* __restrict__ out, int Cin, int H, int W,
                                 int64_t M, int64_t xbs, int64_t ld) {
  const int P = H * W;
  const int K = Cin * 9;
  const int64_t n = M * Cin;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t m = i % M;
    const int c = (int)(i / M);
    const int64_t b = m / P;
    const int p = (int)(m - b * P);
    const int py = p / W, px = p - py * W;
    const float* xc = x + b * xbs + (int64_t)c * P;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
      const int yy = py + ky - 1;
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int xx = px + kx - 1;
        float v = 0.f;
        if (yy >= 0 && yy < H && xx >= 0 && xx < W) v = __ldg(xc + yy * W + xx);
        put_rc<T>(out, m, ld, c * 9 + ky * 3 + kx, v);
      }
    }
    if (c == Cin - 1)
      for (int k = K; k < ld; ++k) put_rc<T>(out, m, ld, k, 0.f);
  }
}

template <typename T>
__global__ void pack_matrix_kernel(const float* __restrict__ in, T* __restrict__ out, int na, int nb, int nk,
                                   int64_t sa, int64_t sb, int64_t sk, int64_t ld, int rows_out) {
  const int64_t n = (int64_t)rows_out * ld;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / ld;
    const int k = (int)(i - r * ld);
    float v = 0.f;
    if (r < (int64_t)na * nb && k < nk) {
      const int a = (int)(r / nb), b = (int)(r - (int64_t)a * nb);
      v = __ldg(in + a * sa + b * sb + k * sk);
    }
    put_rc<T>(out, r, ld, k, v);
  }
}

// Batched pack: every weight layout of every StepFlow in ONE launch (the parameters change once per optimiser step; 7
// separate packs per StepFlow were ~440 launches per training step).  jobs: device table, 10 x int64 per job:
//   [0] in  [1] out  [2] sa  [3] sb  [4] sk  [5] ld_out  [6] na | nb<<32  [7] nk | rows_out<<32
//   [8] out_dtype | first_block<<32  [9] nk2 | sk2<<32   (column k -> (k / nk2)*sk + (k % nk2)*sk2; nk2 = 1: plain)
constexpr int PACK_ELEMS = 4096;      // one CTA = a 64 (rows) x 64 (columns) tile of the output matrix
__global__ void __launch_bounds__(256) pack_batch_kernel(const int64_t* __restrict__ jobs, int n_jobs) {
  __shared__ int s_job;
  __shared__ float tile[64][65];
  if (threadIdx.x == 0) {
    int lo = 0, hi = n_jobs - 1;                       // last job whose first_block <= blockIdx.x
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if ((int)(jobs[mid * 10 + 8] >> 32) <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    s_job = lo;
  }
  __syncthreads();
  const int64_t* j = jobs + (int64_t)s_job * 10;
  const float* in = reinterpret_cast<const float*>(j[0]);
  const int64_t sa = j[2], sb = j[3], sk = j[4], ld = j[5];
  const int na = (int)(j[6] & 0xffffffff), nb = (int)(j[6] >> 32);
  const int nk = (int)(j[7] & 0xffffffff), rows_out = (int)(j[7] >> 32);
  const int dtype = (int)(j[8] & 0xffffffff), first = (int)(j[8] >> 32);
  const int nk2 = (int)(j[9] & 0xffffffff);
  const int64_t sk2 = j[9] >> 32;
  const int ct = (int)((ld + 63) >> 6);                // column tiles per row band
  const int tb = blockIdx.x - first;
  const int r0 = (tb / ct) << 6, c0 = (tb % ct) << 6;
  // gather 64 x 64 source elements into shared memory.  Lanes walk the direction that is contiguous in the SOURCE:
  // columns when sk == 1, rows when the source is row-contiguous (transposing jobs: sa == 1, nb == 1) -> coalesced reads
  const bool rows_fast = (sk != 1) && (sa == 1) && (nb == 1);
  for (int e = threadIdx.x; e < 4096; e += 256) {
    const int rr = rows_fast ? (e & 63) : (e >> 6), cc = rows_fast ? (e >> 6) : (e & 63);
    const int64_t r = r0 + rr;
    const int k = c0 + cc;
    float v = 0.f;
    if (r < (int64_t)na * nb && k < nk && r < rows_out) {
      const int a = (int)(r / nb), b = (int)(r - (int64_t)a * nb);
      const int k1 = k / nk2, k2 = k - k1 * nk2;
      v = __ldg(in + a * sa + b * sb + k1 * sk + k2 * sk2);
    }
    tile[rr][cc] = v;
  }
  __syncthreads();
  for (int e = threadIdx.x; e < 4096; e += 256) {
    const int rr = e >> 6, cc = e & 63;
    const int64_t r = r0 + rr;
    const int k = c0 + cc;
    if (r < rows_out && k < ld) {
      const float v = tile[rr][cc];
      if (dtype == NFDPM_F32) reinterpret_cast<float*>(j[1])[r * ld + k] = v;
      else if (dtype == NFDPM_BF16X2) put_rc<bf16x2_t>(reinterpret_cast<bf16x2_t*>(j[1]), r, ld, k, v);
      else reinterpret_cast<__nv_bfloat16*>(j[1])[r * ld + k] = __float2bfloat16_rn(v);
    }
  }
}

// Tile geometry shared by the per-pixel kernels: CTA `blockIdx.x` owns up to TPB consecutive flattened pixels.
//   P >  TPB: grid = B * T, T = ceil(P/TPB); CTA (b, t) owns pixels [t*TPB, min(P,(t+1)*TPB)) of image b
//   P <= TPB: grid = ceil(B / ipc), ipc = TPB / P whole images per CTA
struct PixTile {
  int64_t first_m;
  int n_valid;
};
__device__ __forceinline__ PixTile pix_tile(int B, int P) {
  PixTile t;
  if (P > TPB) {
    const int T = (P + TPB - 1) / TPB;
    const int b = blockIdx.x / T, ti = blockIdx.x - b * T;
    t.first_m = (int64_t)b * P + (int64_t)ti * TPB;
    t.n_valid = min(TPB, P - ti * TPB);
  } else {
    const int ipc = TPB / P;
    const int b0 = blockIdx.x * ipc;
    t.first_m = (int64_t)b0 * P;
    t.n_valid = min(ipc, B - b0) * P;
  }
  return t;
}
static int pix_grid(int B, int P) {
  if (P > TPB) return B * ((P + TPB - 1) / TPB);
  const int ipc = TPB / P;
  return (B + ipc - 1) / ipc;
}

// Affine coupling epilogue.  One thread per pixel; loops over the C/2 transformed channels two at a time
// (8-byte loads of the taps-as-N rows).  INVERSE selects x_b = y_b/(s+1e-6) - t.  In either direction a non-null ld_part
// receives the per-image sum of log(s + 1e-6): the inverse divides by exactly the s the forward multiplies by.
template <bool INVERSE, int VEC>
__global__ void __launch_bounds__(TPB) coupling_apply_kernel(const float* __restrict__ pm, int64_t ldp,
                                                             const float* __restrict__ bias3,
                                                             const float* __restrict__ logs3,
                                                             const float* x, float* y,  // may alias (in place)
                                                             float* __restrict__ ld_part, int B, int C, int H,
                                                             int W, int64_t xbs, int64_t ybs) {
  __shared__ float sh[TPB];
  extern __shared__ __align__(16) float s_par[];  // [2*C]: bias3, exp(3*logs3)
  const int P = H * W, Ch = C >> 1;
  for (int i = threadIdx.x; i < C; i += TPB) {
    s_par[i] = bias3[i];
    s_par[C + i] = expf(3.f * logs3[i]);
  }
  __syncthreads();
  const PixTile tile = pix_tile(B, P);
  const int t = threadIdx.x;
  const bool live = t < tile.n_valid;
  float ld_acc = 0.f;
  if (live) {
    const int64_t m = tile.first_m + t;
    const int64_t b = m / P;
    const int p = (int)(m - b * P);
    const int py = p / W, px = p - py * W;
    // neighbour row offsets (in rows of pm) and validity, tap = ky*3 + kx
    int64_t roff[9];
    bool ok[9];
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const int yy = py + ky - 1, xx = px + kx - 1;
        ok[ky * 3 + kx] = (yy >= 0 && yy < H && xx >= 0 && xx < W);
        roff[ky * 3 + kx] = (m + (ky - 1) * W + (kx - 1)) * ldp;
      }
    const float* xb = x + b * xbs + p;
    float* yb = y + b * ybs + p;
    if (x != y) {
      for (int j = 0; j < Ch; ++j) yb[(int64_t)j * P] = xb[(int64_t)j * P];
    }
    for (int j = 0; j < Ch; j += VEC) {
      float ls[VEC], tt[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) ls[v] = tt[v] = 0.f;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        if (ok[tap]) {
          const float* r = pm + roff[tap] + tap * C + j;
          if constexpr (VEC == 2) {
            const float2 a = *reinterpret_cast<const float2*>(r);
            const float2 c2 = *reinterpret_cast<const float2*>(r + Ch);
            ls[0] += a.x; ls[1] += a.y;
            tt[0] += c2.x; tt[1] += c2.y;
          } else {
            ls[0] += r[0];
            tt[0] += r[Ch];
          }
        }
      }
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const int jj = j + v;
        const float log_s = (ls[v] + s_par[jj]) * s_par[C + jj];
        const float sh_t = (tt[v] + s_par[Ch + jj]) * s_par[C + Ch + jj];
        const float s = 1.f / (1.f + expf(-(log_s + 2.f)));
        const float xv = xb[(int64_t)(Ch + jj) * P];
        if (INVERSE) {
          yb[(int64_t)(Ch + jj) * P] = xv / (s + 1e-6f) - sh_t;
          if (ld_part != nullptr) ld_acc += logf(s + 1e-6f);
        } else {
          yb[(int64_t)(Ch + jj) * P] = (xv + sh_t) * s;
          ld_acc += logf(s + 1e-6f);
        }
      }
    }
  }
  if (ld_part != nullptr) {
    tile_image_reduce<TPB>(ld_acc, sh, tile.first_m, tile.n_valid, P,
                           [&](int64_t b, int ti, float s) { ld_part[(int64_t)ti * B + b] = s; });
  }
}

// Split prior: mean/logs from the raw ZeroConv GEMM rows h [M, ldh] (column = co), z = x[:, C/2:].
template <bool SAMPLE>
__global__ void __launch_bounds__(TPB) split_prior_kernel(const float* __restrict__ h, int64_t ldh,
                                                          const float* __restrict__ bias,
                                                          const float* __restrict__ logs,
                                                          const float* __restrict__ x, int64_t xbs,
                                                          float* __restrict__ z_out, float* __restrict__ logp_part,
                                                          const float* __restrict__ eps, float temperature,
                                                          float* __restrict__ y, int64_t ybs, int B, int C, int P) {
  __shared__ float sh[TPB];
  extern __shared__ __align__(16) float s_par[];  // [2*C]
  const int Ch = C >> 1;
  for (int i = threadIdx.x; i < C; i += TPB) {
    s_par[i] = (h != nullptr) ? bias[i] : 0.f;
    s_par[C + i] = (h != nullptr) ? expf(3.f * logs[i]) : 1.f;
  }
  __syncthreads();
  const PixTile tile = pix_tile(B, P);
  const int t = threadIdx.x;
  const bool live = t < tile.n_valid;
  const float LOG2PI = 1.8378770664093453f;
  float acc = 0.f;
  if (live) {
    const int64_t m = tile.first_m + t;
    const int64_t b = m / P;
    const int p = (int)(m - b * P);
    const float* hr = (h != nullptr) ? h + m * ldh : nullptr;
    for (int j = 0; j < Ch; ++j) {
      float mean = 0.f, lg = 0.f;
      if (hr != nullptr) {
        mean = (hr[j] + s_par[j]) * s_par[C + j];
        lg = (hr[Ch + j] + s_par[Ch + j]) * s_par[C + Ch + j];
      }
      if (SAMPLE) {
        const float e = eps[(b * Ch + j) * (int64_t)P + p];
        y[b * ybs + (int64_t)(Ch + j) * P + p] = mean + (expf(lg) * temperature) * e;
      } else {
        const float z = x[b * xbs + (int64_t)(Ch + j) * P + p];
        if (z_out != nullptr) z_out[(b * Ch + j) * (int64_t)P + p] = z;
        const float d = z - mean;
        acc += -0.5f * (LOG2PI + 2.f * lg + d * d * expf(-2.f * lg));
      }
    }
  }
  if (!SAMPLE && logp_part != nullptr) {
    tile_image_reduce<TPB>(acc, sh, tile.first_m, tile.n_valid, P,
                           [&](int64_t b, int ti, float s) { logp_part[(int64_t)ti * B + b] = s; });
  }
}

// Layout converters for stand-alone coupling-net module calls (off the hot path).
//   rows_to_nchw: out[b,n,p] = f(h[(b*P+p)*ldh + n]);  mode 0: v; 1 (ZeroConv2d, utils.py:44): (v+p1[n])*exp(3*p2[n]);
//                 2 (ActNorm, transforms.py:80): exp(p1[n])*(v+p2[n])
__global__ void rows_to_nchw_kernel(const float* __restrict__ h, int64_t ldh, int mode, const float* __restrict__ p1,
                                    const float* __restrict__ p2, float* __restrict__ out, int Nc, int P, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int p = (int)(i % P);
    const int64_t r = i / P;
    const int c = (int)(r % Nc);
    const int64_t b = r / Nc;
    float v = h[(b * P + p) * ldh + c];
    if (mode == 1) v = (v + __ldg(p1 + c)) * expf(3.f * __ldg(p2 + c));
    else if (mode == 2) v = expf(__ldg(p1 + c)) * (v + __ldg(p2 + c));
    out[i] = v;
  }
}
template <typename T>
__global__ void nchw_to_rows_kernel(const float* __restrict__ x, T* __restrict__ out, int Cc, int P, int64_t xbs,
                                    int64_t ld, int64_t n /* B*P*ld */) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % ld);
    const int64_t m = i / ld;
    const int64_t b = m / P;
    const int p = (int)(m - b * P);
    put_rc<T>(out, m, ld, c, c < Cc ? x[b * xbs + (int64_t)c * P + p] : 0.f);
  }
}

static int grid_for(int64_t n, int tpb, int cap = 148 * 16) {
  int64_t g = cdiv64(n, tpb);
  if (g < 1) g = 1;
  return (int)(g > cap ? cap : g);
}

}  // namespace nfdpm

using namespace nfdpm;

extern "C" int nfdpm_ld_tiles(int P) { return P > TPB ? (P + TPB - 1) / TPB : 1; }

extern "C" int nfdpm_im2col3x3(const float* x, void* out, int out_dtype, int B, int Cin, int H, int W, int64_t xbs,
                               int64_t ld, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x && out, "nfdpm_im2col3x3: null pointer");
  NFDPM_REQUIRE(B > 0 && Cin > 0 && H > 0 && W > 0, "nfdpm_im2col3x3: bad shape");
  NFDPM_REQUIRE(ld >= (int64_t)Cin * 9, "nfdpm_im2col3x3: ld_out=%lld < 9*Cin=%d", (long long)ld, Cin * 9);
  const int64_t M = (int64_t)B * H * W;
  const int grid = grid_for(M * Cin, 256);
  if (out_dtype == NFDPM_F32)
    im2col3x3_kernel<float><<<grid, 256, 0, as_stream(stream)>>>(x, (float*)out, Cin, H, W, M, xbs, ld);
  else if (out_dtype == NFDPM_BF16)
    im2col3x3_kernel<__nv_bfloat16><<<grid, 256, 0, as_stream(stream)>>>(x, (__nv_bfloat16*)out, Cin, H, W, M, xbs, ld);
  else if (out_dtype == NFDPM_BF16X2 && ld % 32 == 0)
    im2col3x3_kernel<bf16x2_t><<<grid, 256, 0, as_stream(stream)>>>(x, (bf16x2_t*)out, Cin, H, W, M, xbs, ld);
  else
    return fail("nfdpm_im2col3x3: out_dtype %d unsupported", out_dtype);
  NFDPM_CHECK_LAUNCH("im2col3x3_kernel");
  return 0;
}

extern "C" int nfdpm_pack_matrix(const float* in, void* out, int out_dtype, int na, int nb, int nk, int64_t sa,
                                 int64_t sb, int64_t sk, int64_t ld, int rows_out, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(in && out, "nfdpm_pack_matrix: null pointer");
  NFDPM_REQUIRE(na > 0 && nb > 0 && nk > 0 && ld >= nk && rows_out >= na * nb, "nfdpm_pack_matrix: bad shape");
  const int grid = grid_for((int64_t)rows_out * ld, 256);
  if (out_dtype == NFDPM_F32)
    pack_matrix_kernel<float><<<grid, 256, 0, as_stream(stream)>>>(in, (float*)out, na, nb, nk, sa, sb, sk, ld, rows_out);
  else if (out_dtype == NFDPM_BF16)
    pack_matrix_kernel<__nv_bfloat16><<<grid, 256, 0, as_stream(stream)>>>(in, (__nv_bfloat16*)out, na, nb, nk, sa, sb, sk, ld, rows_out);
  else if (out_dtype == NFDPM_BF16X2 && ld % 32 == 0)
    pack_matrix_kernel<bf16x2_t><<<grid, 256, 0, as_stream(stream)>>>(in, (bf16x2_t*)out, na, nb, nk, sa, sb, sk, ld, rows_out);
  else
    return fail("nfdpm_pack_matrix: out_dtype %d unsupported", out_dtype);
  NFDPM_CHECK_LAUNCH("pack_matrix_kernel");
  return 0;
}

extern "C" int nfdpm_pack_elems(void) { return PACK_ELEMS; }
/* blocks of one job = ceil(rows_out/64) * ceil(ld_out/64) */

extern "C" int nfdpm_pack_batch(const int64_t* jobs_dev, int n_jobs, int n_blocks, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(jobs_dev && n_jobs > 0 && n_blocks > 0, "nfdpm_pack_batch: bad arguments");
  pack_batch_kernel<<<n_blocks, 256, 0, as_stream(stream)>>>(jobs_dev, n_jobs);
  NFDPM_CHECK_LAUNCH("pack_batch_kernel");
  return 0;
}

extern "C" int nfdpm_coupling_apply(const float* pm, int64_t ldp, const float* bias3, const float* logs3,
                                    const float* x, float* y, float* ld_part, int B, int C, int H, int W,
                                    int64_t xbs, int64_t ybs, int inverse, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(pm && bias3 && logs3 && x && y, "nfdpm_coupling_apply: null pointer");
  NFDPM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "nfdpm_coupling_apply: bad shape");
  NFDPM_REQUIRE(C % 2 == 0, "nfdpm_coupling_apply: C=%d must be even", C);
  NFDPM_REQUIRE(ldp >= 9 * (int64_t)C, "nfdpm_coupling_apply: ldp too small");
  const int P = H * W;
  const int grid = pix_grid(B, P);
  const size_t smem = sizeof(float) * 2 * C;
  cudaStream_t st = as_stream(stream);
  const bool vec2 = ((C / 2) % 2 == 0) && (ldp % 2 == 0) && ((uintptr_t)pm % 8 == 0);
#define LAUNCH(INV, VEC)                                                                                         \
  coupling_apply_kernel<INV, VEC><<<grid, TPB, smem, st>>>(pm, ldp, bias3, logs3, x, y, ld_part, B, C, H, W, xbs, ybs)
  if (inverse) { if (vec2) LAUNCH(true, 2); else LAUNCH(true, 1); }
  else { if (vec2) LAUNCH(false, 2); else LAUNCH(false, 1); }
#undef LAUNCH
  NFDPM_CHECK_LAUNCH("coupling_apply_kernel");
  return 0;
}

extern "C" int nfdpm_split_prior_logp(const float* h, int64_t ldh, const float* bias, const float* logs,
                                      const float* x, int64_t xbs, float* z_out, float* logp_part, int B, int C,
                                      int H, int W, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x, "nfdpm_split_prior_logp: null input");
  NFDPM_REQUIRE(h == nullptr || (bias && logs && ldh >= C), "nfdpm_split_prior_logp: learned prior needs bias/logs/ldh");
  NFDPM_REQUIRE(B > 0 && C > 0 && C % 2 == 0 && H > 0 && W > 0, "nfdpm_split_prior_logp: bad shape");
  const int P = H * W;
  split_prior_kernel<false><<<pix_grid(B, P), TPB, sizeof(float) * 2 * C, as_stream(stream)>>>(
      h, ldh, bias, logs, x, xbs, z_out, logp_part, nullptr, 0.f, nullptr, 0, B, C, P);
  NFDPM_CHECK_LAUNCH("split_prior_kernel<logp>");
  return 0;
}

extern "C" int nfdpm_split_prior_sample(const float* h, int64_t ldh, const float* bias, const float* logs,
                                        const float* eps, float temperature, float* y, int64_t ybs, int B, int C,
                                        int H, int W, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(eps && y, "nfdpm_split_prior_sample: null pointer");
  NFDPM_REQUIRE(h == nullptr || (bias && logs && ldh >= C), "nfdpm_split_prior_sample: learned prior needs bias/logs/ldh");
  NFDPM_REQUIRE(B > 0 && C > 0 && C % 2 == 0 && H > 0 && W > 0, "nfdpm_split_prior_sample: bad shape");
  const int P = H * W;
  split_prior_kernel<true><<<pix_grid(B, P), TPB, sizeof(float) * 2 * C, as_stream(stream)>>>(
      h, ldh, bias, logs, nullptr, 0, nullptr, nullptr, eps, temperature, y, ybs, B, C, P);
  NFDPM_CHECK_LAUNCH("split_prior_kernel<sample>");
  return 0;
}

extern "C" int nfdpm_rows_to_nchw(const float* h, int64_t ldh, int mode, const float* p1, const float* p2, float* out,
                                  int B, int Nc, int P, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(h && out, "nfdpm_rows_to_nchw: null pointer");
  NFDPM_REQUIRE(mode >= 0 && mode <= 2 && (mode == 0 || (p1 && p2)), "nfdpm_rows_to_nchw: bad mode/params");
  NFDPM_REQUIRE(B > 0 && Nc > 0 && P > 0 && ldh >= Nc, "nfdpm_rows_to_nchw: bad shape");
  const int64_t n = (int64_t)B * Nc * P;
  rows_to_nchw_kernel<<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(h, ldh, mode, p1, p2, out, Nc, P, n);
  NFDPM_CHECK_LAUNCH("rows_to_nchw_kernel");
  return 0;
}

extern "C" int nfdpm_nchw_to_rows(const float* x, void* out, int out_dtype, int B, int Cc, int P, int64_t xbs,
                                  int64_t ld, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(x && out, "nfdpm_nchw_to_rows: null pointer");
  NFDPM_REQUIRE(B > 0 && Cc > 0 && P > 0 && ld >= Cc, "nfdpm_nchw_to_rows: bad shape");
  const int64_t n = (int64_t)B * P * ld;
  if (out_dtype == NFDPM_F32)
    nchw_to_rows_kernel<float><<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(x, (float*)out, Cc, P, xbs, ld, n);
  else if (out_dtype == NFDPM_BF16)
    nchw_to_rows_kernel<__nv_bfloat16><<<grid_for(n, 256), 256, 0, as_stream(stream)>>>(x, (__nv_bfloat16*)out, Cc, P, xbs, ld, n);
  else
    return fail("nfdpm_nchw_to_rows: out_dtype %d unsupported", out_dtype);
  NFDPM_CHECK_LAUNCH("nchw_to_rows_kernel");
  return 0;
}
