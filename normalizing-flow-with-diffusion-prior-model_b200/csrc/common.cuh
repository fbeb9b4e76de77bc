// Shared helpers for libnfdpm_b200 (sm_100a).  Internal header, not part of the C ABI.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <curand_philox4x32_x.h>   // header-only device code: no libcurand link

#include "../../include/nfdpm_b200.h"

namespace nfdpm {

// thread-local last error (nfdpm_last_error_string)
char* err_buf();
int fail(const char* fmt, ...);

#define NFDPM_REQUIRE(cond, ...)                \
  do {                                          \
    if (!(cond)) return nfdpm::fail(__VA_ARGS__); \
  } while (0)

// Check the launch itself (not execution): cheap, does not synchronise.
#define NFDPM_CHECK_LAUNCH(name)                                                         \
  do {                                                                                   \
    cudaError_t e__ = cudaGetLastError();                                                \
    if (e__ != cudaSuccess) return nfdpm::fail("%s: launch failed: %s", name, cudaGetErrorString(e__)); \
  } while (0)

#define NFDPM_CUDA(call)                                                                  \
  do {                                                                                    \
    cudaError_t e__ = (call);                                                             \
    if (e__ != cudaSuccess) {                                                             \
      (void)cudaGetLastError(); /* do not leave a sticky error for the next call */       \
      return nfdpm::fail("%s: %s", #call, cudaGetErrorString(e__));                       \
    }                                                                                     \
  } while (0)

static inline cudaStream_t as_stream(nfdpm_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }

bool pdl_enabled();   // env NFDPM_PDL (default on)
// <<<grid, block, smem, stream>>> with the programmatic-stream-serialization attribute (PDL) when enabled
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ---------------------------------------------------------------- split bf16 pairs (NFDPM_BF16X2)
// A logical fp32 value v is carried as hi = bf16(v), lo = bf16(v - hi): v = hi + lo up to 2^-17 |v|.  A row of K logical
// columns (K % 32 == 0) occupies 2K bf16: the group g = k / 32 owns 64 consecutive bf16, [hi(32g..32g+31) | lo(32g..32g+31)],
// i.e. one 128-byte swizzle row of a TMA box holds both planes of 32 logical columns and the four K=16 UMMA slices of a
// [rows][64] operand tile are hi(0..15), hi(16..31), lo(0..15), lo(16..31).  The tensor-core kernels then form
// A*B ~= Ahi*Bhi + Alo*Bhi + Ahi*Blo (three tcgen05.mma per slice pair into ONE fp32 TMEM accumulator): the dropped
// lo*lo term and the rounding of lo are both <= 2^-17 relative, against 2^-9 for plain bf16 operands.
struct __align__(4) bf16x2_t { __nv_bfloat16 hi, lo; };          // storage unit: 4 bytes per logical element
__host__ __device__ __forceinline__ int64_t split_col(int64_t k) { return ((k >> 5) << 6) + (k & 31); }   // bf16 index of hi(k); lo(k) is +32
__device__ __forceinline__ void split_pair(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16_rn(v);
  lo = __float2bfloat16_rn(v - __bfloat162float(hi));
}
// eight consecutive logical columns k0..k0+7 (k0 % 8 == 0) of the split row starting at `row` (bf16 units): two 16-byte stores
__device__ __forceinline__ void split_store8(__nv_bfloat16* row, int64_t k0, const float (&v)[8]) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    __nv_bfloat162 th = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    const float2 back = __bfloat1622float2(th);
    __nv_bfloat162 tl = __floats2bfloat162_rn(v[2 * i] - back.x, v[2 * i + 1] - back.y);
    h[i] = *reinterpret_cast<uint32_t*>(&th);
    l[i] = *reinterpret_cast<uint32_t*>(&tl);
  }
  __nv_bfloat16* p = row + split_col(k0);
  *reinterpret_cast<uint4*>(p) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(p + 32) = make_uint4(l[0], l[1], l[2], l[3]);
}

// element (r, k) of a row-major [rows, ld] matrix of fp32 / bf16 / split pairs (ld counts LOGICAL columns)
template <typename T> __device__ __forceinline__ void put_rc(T* out, int64_t r, int64_t ld, int64_t k, float v);
template <> __device__ __forceinline__ void put_rc<float>(float* out, int64_t r, int64_t ld, int64_t k, float v) { out[r * ld + k] = v; }
template <> __device__ __forceinline__ void put_rc<__nv_bfloat16>(__nv_bfloat16* out, int64_t r, int64_t ld, int64_t k, float v) {
  out[r * ld + k] = __float2bfloat16_rn(v);
}
template <> __device__ __forceinline__ void put_rc<bf16x2_t>(bf16x2_t* out, int64_t r, int64_t ld, int64_t k, float v) {
  __nv_bfloat16* p = reinterpret_cast<__nv_bfloat16*>(out) + 2 * r * ld + split_col(k);
  split_pair(v, p[0], p[32]);
}

// streaming 128-bit access: read-once / write-once tensors should not pollute L1
__device__ __forceinline__ float4 ldg_stream4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_stream4(float* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
               "f"(v.w)
               : "memory");
}

// Programmatic dependent launch (PDL): a kernel launched with launch_pdl() may start while its predecessor in the
// stream is still draining; it must call pdl_wait() before touching global memory the predecessor writes (the call
// returns once the predecessor grid has completed and flushed), and pdl_trigger() lets ITS successor start early.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// Division by a run-time constant as multiply-high: the kernels below are issue-bound on index arithmetic (r1 timeline: a
// 32-bit division costs ~35 instructions and there were ~14 per thread).  Exact for n * d < 2^32.
struct FastDiv {
  uint32_t d, m;                          // m = ceil(2^32 / d); m == 0 encodes d == 1
};
static inline FastDiv make_fastdiv(int d) {
  FastDiv f;
  f.d = (uint32_t)d;
  f.m = d > 1 ? (uint32_t)(((1ull << 32) + (uint32_t)d - 1) / (uint32_t)d) : 0u;
  return f;
}
__device__ __forceinline__ int fdiv(int n, const FastDiv f) { return f.m ? (int)__umulhi((uint32_t)n, f.m) : n; }

// Counter-based standard normal draw: a pure function of (seed of the image, draw site, element index), so a sample does not
// depend on its batch, its position in it, earlier draws or graph replays.  The contract (include/nfdpm_b200.h, DESIGN §4;
// tests/test_seeded_sampling_cpu.py holds a numpy oracle of it):
//   key     = (lo32(seed), hi32(seed)), seed = the image's int64 seed reinterpreted as uint64
//   counter = (e >> 2, stream, 0, 0), e = c*P + p the element's index in the image's drawn tensor [C_draw, H, W]
//   w0..w3  = Philox4x32-10(counter, key)
//   u_i     = fp32((w_i >> 8) + 0.5) * 2^-24: in (0, 1]; the +0.5 is exact below 2^23 and rounds to even above, so
//             u = 1 is possible (probability 2^-24) and gives a zero normal, never a NaN or an infinity
//   r = sqrtf(-2 logf(u_even)); sincospif(2 u_odd) -> n_even = r*cos, n_odd = r*sin, for (w0, w1) and (w2, w3)
//   element e takes n[e & 3]
__device__ __forceinline__ float philox_normal(uint64_t seed, uint32_t stream, uint32_t e) {
  const uint4 w = curand_Philox4x32_10(make_uint4(e >> 2, stream, 0u, 0u),
                                       make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const bool hi = (e & 2u) != 0u;
  const uint32_t we = hi ? w.z : w.x, wo = hi ? w.w : w.y;
  const float ue = ((float)(we >> 8) + 0.5f) * 0x1p-24f;
  const float uo = ((float)(wo >> 8) + 0.5f) * 0x1p-24f;
  const float r = sqrtf(-2.f * logf(ue));
  float s, c;
  sincospif(2.f * uo, &s, &c);
  return (e & 1u) ? r * s : r * c;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Deterministic per-image reduction of one value per thread, for kernels whose CTA owns TPB consecutive
// flattened pixels m = b*P + p of ONE tile:  val[t] -> sums[img] for the images the tile overlaps.
// `first_m` = flattened index of thread 0, `n_valid` = number of valid threads.  Results are written by
// out(b, tile_in_image, sum).  Fixed summation order => bitwise reproducible.
template <int TPB, typename Out>
__device__ __forceinline__ void tile_image_reduce(float v, float* sh /*[TPB]*/, int64_t first_m, int n_valid, int P,
                                                  Out out) {
  const int t = threadIdx.x;
  sh[t] = (t < n_valid) ? v : 0.f;
  __syncthreads();
  if (P >= TPB) {
    // the tile lies inside one image (tiles are cut per image when P > TPB; P == TPB is one image)
    // tree reduction in a fixed order
    for (int s = TPB / 2; s > 0; s >>= 1) {
      if (t < s) sh[t] += sh[t + s];
      __syncthreads();
    }
    if (t == 0) out(first_m / P, (int)((first_m % P) / TPB), sh[0]);
  } else {
    // several whole images per tile: one thread sums one image sequentially
    const int n_img = (n_valid + P - 1) / P;
    if (t < n_img) {
      float s = 0.f;
      const int lo = t * P, hi = min(lo + P, n_valid);
      for (int i = lo; i < hi; ++i) s += sh[i];
      out(first_m / P + t, 0, s);
    }
  }
}

}  // namespace nfdpm
