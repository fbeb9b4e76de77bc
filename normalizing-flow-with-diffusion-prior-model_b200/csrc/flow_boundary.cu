// Fused "step boundary" kernel: everything that happens to the flow state between the last GEMM of one StepFlow
// and the first GEMM of the next one, in ONE launch, one CTA per image:
//
//   source   SRC_PLAIN     x = in[b]                       (optionally with squeeze addressing, transforms.py:226)
//            SRC_COUPLING  x = affine coupling of in[b] with the taps-as-N ZeroConv rows pm (forward:
//                          transforms.py:179-184 incl. the per-image log-det partial; inverse: :196-200)
//   mix      u = Mt^T x + beta     fused ActNorm + invertible 1x1 conv of the NEXT step (forward, transforms.py:80,132)
//                                  or of THIS step (inverse, :144,:93); optional
//   sinks    y[b]  <- u            NCHW fp32 flow state (optional)
//            a1    <- im2col3x3(u[:C/2])  pixel-major rows for the next coupling network's first GEMM (optional)
//
// All global traffic is coalesced: the image is staged channel-major in shared memory, pm rows are read with the
// channel index fastest across lanes (each pm element is consumed exactly once), im2col rows are written as 16-byte
// (bf16) / 32-byte (fp32) pieces with the column group fastest across lanes.
// Replaces, per StepFlow: nfdpm_coupling_apply + nfdpm_channel_mix + nfdpm_im2col3x3 (+ nfdpm_squeeze at level entry).
#include "boundary_body.cuh"

namespace nfdpm {

// PM_BULK: the image's taps-as-N rows (one contiguous block of P*ldp floats) are fetched by the bulk-copy engine
// (cp.async.bulk, completion on an mbarrier) into shared memory while the CTA stages the state and the parameters; the
// coupling then gathers its 18 values per item from shared memory instead of issuing 18 scattered L2 loads per thread
// (r1 timeline: 4.2 / 2.0 / 1.1 us of the 12.3 / 7.7 / 6.1 us kernel at the three levels of config 2).
template <bool COUPLING, typename A1T, bool PM_BULK>
__global__ void __launch_bounds__(1024) flow_boundary_kernel(const BoundaryArgs a) {
  extern __shared__ __align__(128) float sm[];
  __shared__ __align__(8) uint64_t pm_bar;
  pdl_trigger();      // PDL: the next kernel of the chain may be scheduled as soon as SMs free up ...
  if (PM_BULK && threadIdx.x == 0) {
    mbar_init(smem_u32(&pm_bar), 1);
    fence_barrier_init();
  }
  pdl_wait();         // ... and this one reads nothing before its predecessor has completed
  if (PM_BULK) {
    const size_t n = (size_t)a.H * a.W * a.ldp;                 // floats of this image's pm block
    if (threadIdx.x == 0) {
      const uint32_t bar = smem_u32(&pm_bar);
      const char* src = reinterpret_cast<const char*>(a.pm + (size_t)blockIdx.x * n);
      mbar_arrive_expect_tx(bar, (uint32_t)(n * 4));
      for (size_t off = 0; off < n * 4; off += 32768) {
        const uint32_t len = (uint32_t)((n * 4 - off) < 32768 ? (n * 4 - off) : 32768);
        bulk_load(smem_u32(sm) + (uint32_t)off, src + off, len, bar);
      }
    }
    flow_boundary_body<COUPLING, A1T, true>(a, blockIdx.x, sm + n, threadIdx.x, blockDim.x, sm, (int)a.ldp,
                                            smem_u32(&pm_bar));
  } else {
    flow_boundary_body<COUPLING, A1T, false>(a, blockIdx.x, sm, threadIdx.x, blockDim.x);
  }
}

}  // namespace nfdpm

using namespace nfdpm;

// profiling hook: per-image phase timeline of nfdpm_flow_boundary into a device int64 [B][16] buffer (NULL = off)
extern "C" int nfdpm_flow_boundary_debug(void* buf) {
  long long* p = reinterpret_cast<long long*>(buf);
  NFDPM_CUDA(cudaMemcpyToSymbol(nfdpm::g_bd_dbg, &p, sizeof(p)));
  return 0;
}

extern "C" size_t nfdpm_flow_boundary_smem(int C, int H, int W, int coupling, int mix) {
  return boundary_scratch_floats(C, H, W, coupling != 0, mix != 0, nullptr, nullptr) * sizeof(float);
}

static int flow_boundary_impl(const float* in, int64_t in_bs, int squeeze_in, const float* pm, int64_t ldp,
                              const float* bias3, const float* logs3, float* ld_part, const float* mt,
                              const float* beta, float* y, int64_t y_bs, float* xs, int64_t xs_bs, void* a1, int a1_dtype,
                              int64_t lda1, int B, int C, int H, int W, int inverse, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(in != nullptr, "nfdpm_flow_boundary: null input");
  NFDPM_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0 && C % 2 == 0, "nfdpm_flow_boundary: bad shape B=%d C=%d H=%d W=%d", B, C, H, W);
  NFDPM_REQUIRE((mt == nullptr) == (beta == nullptr), "nfdpm_flow_boundary: mt/beta must both be set or both NULL");
  NFDPM_REQUIRE(pm == nullptr || (bias3 && logs3 && ldp >= 9 * (int64_t)C), "nfdpm_flow_boundary: coupling source needs bias3/logs3/ldp");
  NFDPM_REQUIRE(!squeeze_in || (C % 4 == 0 && in_bs % 2 == 0 && ((uintptr_t)in % 8) == 0), "nfdpm_flow_boundary: squeeze source needs C %% 4 == 0 and 8-byte alignment");
  NFDPM_REQUIRE(a1 == nullptr || (lda1 % 8 == 0 && lda1 >= 9 * (int64_t)(C / 2) && ((uintptr_t)a1 % 16) == 0), "nfdpm_flow_boundary: bad im2col sink");
  NFDPM_REQUIRE(a1 == nullptr || a1_dtype == NFDPM_F32 || a1_dtype == NFDPM_BF16 || (a1_dtype == NFDPM_BF16X2 && lda1 % 32 == 0), "nfdpm_flow_boundary: bad a1 dtype");
  NFDPM_REQUIRE(y != nullptr || a1 != nullptr || xs != nullptr, "nfdpm_flow_boundary: no sink");
  size_t smem = nfdpm_flow_boundary_smem(C, H, W, pm != nullptr, mt != nullptr);
  NFDPM_REQUIRE(smem <= 200 * 1024, "nfdpm_flow_boundary: image too large for the fused path (%zu bytes of shared memory); "
                "use the unfused kernels", smem);
  BoundaryArgs a;
  a.in = in; a.in_bs = in_bs; a.pm = pm; a.ldp = ldp; a.bias3 = bias3; a.logs3 = logs3; a.ld_part = ld_part;
  a.mt = mt; a.beta = beta; a.y = y; a.y_bs = y_bs; a.xs = xs; a.xs_bs = xs_bs; a.a1 = a1; a.lda1 = lda1;
  a.B = B; a.C = C; a.H = H; a.W = W; a.squeeze_in = squeeze_in; a.inverse = inverse;
  boundary_fill_div(a);
  cudaStream_t st = as_stream(stream);
  const int a1dt = a1 != nullptr ? a1_dtype : NFDPM_F32;
  // one CTA per image: give it as many warps as its largest phase has work items (latency hiding), up to 1024 threads
  int64_t items = (int64_t)H * W * (C / 2);
  if (a1 != nullptr && (int64_t)H * W * (lda1 / 8) > items) items = (int64_t)H * W * (lda1 / 8);
  int threads = (int)((items + 31) / 32 * 32);
  if (threads > 1024) threads = 1024;
  if (threads < 128) threads = 128;
  // coupling source: stage the image's pm block in shared memory with the bulk-copy engine when it fits and is aligned
  const size_t pm_bytes = (size_t)H * W * (size_t)ldp * sizeof(float);
  const bool bulk = pm != nullptr && ldp % 4 == 0 && ((uintptr_t)pm % 16) == 0 && smem + pm_bytes <= 200 * 1024;
  if (bulk) smem += pm_bytes;
#define LAUNCH(CP, T, BK)                                                                                          \
  do {                                                                                                             \
    static bool attr_set = false;                                                                                  \
    if (!attr_set) {                                                                                               \
      NFDPM_CUDA(cudaFuncSetAttribute(flow_boundary_kernel<CP, T, BK>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                      200 * 1024));                                                                \
      attr_set = true;                                                                                             \
    }                                                                                                              \
    NFDPM_CUDA(launch_pdl(flow_boundary_kernel<CP, T, BK>, dim3(B), dim3(threads), smem, st, a));                  \
  } while (0)
#define GO_BULK(T) LAUNCH(true, T, true)
#define GO_CP(T) LAUNCH(true, T, false)
#define GO_NC(T) LAUNCH(false, T, false)
  if (pm != nullptr && bulk) NFDPM_A1_DISPATCH(a1dt, GO_BULK);
  else if (pm != nullptr) NFDPM_A1_DISPATCH(a1dt, GO_CP);
  else NFDPM_A1_DISPATCH(a1dt, GO_NC);
#undef GO_BULK
#undef GO_CP
#undef GO_NC
#undef LAUNCH
  NFDPM_CHECK_LAUNCH("flow_boundary_kernel");
  return 0;
}

extern "C" int nfdpm_flow_boundary(const float* in, int64_t in_bs, int squeeze_in, const float* pm, int64_t ldp,
                                   const float* bias3, const float* logs3, float* ld_part, const float* mt,
                                   const float* beta, float* y, int64_t y_bs, void* a1, int a1_dtype, int64_t lda1,
                                   int B, int C, int H, int W, int inverse, nfdpm_stream_t stream) {
  return flow_boundary_impl(in, in_bs, squeeze_in, pm, ldp, bias3, logs3, ld_part, mt, beta, y, y_bs, nullptr, 0, a1,
                            a1_dtype, lda1, B, C, H, W, inverse, stream);
}

extern "C" int nfdpm_flow_boundary_stash(const float* in, int64_t in_bs, int squeeze_in, const float* pm, int64_t ldp,
                                         const float* bias3, const float* logs3, float* ld_part, const float* mt,
                                         const float* beta, float* y, int64_t y_bs, float* xs, int64_t xs_bs, void* a1,
                                         int a1_dtype, int64_t lda1, int B, int C, int H, int W, nfdpm_stream_t stream) {
  return flow_boundary_impl(in, in_bs, squeeze_in, pm, ldp, bias3, logs3, ld_part, mt, beta, y, y_bs, xs, xs_bs, a1,
                            a1_dtype, lda1, B, C, H, W, 0, stream);
}

// ld_part (may be null): per-image sum of log(s + 1e-6), the partial flow_boundary writes in inverse mode
extern "C" int nfdpm_flow_boundary_inv_stash_ld(const float* in, int64_t in_bs, const float* pm, int64_t ldp,
                                                const float* bias3, const float* logs3, float* ld_part, const float* mt,
                                                const float* beta, float* y, int64_t y_bs, float* xs, int64_t xs_bs,
                                                void* a1, int a1_dtype, int64_t lda1, int B, int C, int H, int W,
                                                nfdpm_stream_t stream) {
  NFDPM_REQUIRE(in && pm && bias3 && logs3 && mt && beta && y && xs, "nfdpm_flow_boundary_inv_stash_ld: null pointer");
  return flow_boundary_impl(in, in_bs, 0, pm, ldp, bias3, logs3, ld_part, mt, beta, y, y_bs, xs, xs_bs, a1, a1_dtype, lda1,
                            B, C, H, W, 1, stream);
}

extern "C" int nfdpm_flow_boundary_inv_stash(const float* in, int64_t in_bs, const float* pm, int64_t ldp,
                                             const float* bias3, const float* logs3, const float* mt, const float* beta,
                                             float* y, int64_t y_bs, float* xs, int64_t xs_bs, void* a1, int a1_dtype,
                                             int64_t lda1, int B, int C, int H, int W, nfdpm_stream_t stream) {
  NFDPM_REQUIRE(in && pm && bias3 && logs3 && mt && beta && y && xs, "nfdpm_flow_boundary_inv_stash: null pointer");
  return nfdpm_flow_boundary_inv_stash_ld(in, in_bs, pm, ldp, bias3, logs3, nullptr, mt, beta, y, y_bs, xs, xs_bs, a1,
                                          a1_dtype, lda1, B, C, H, W, stream);
}
