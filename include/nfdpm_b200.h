/*
 * nfdpm_b200.h — C ABI of libnfdpm_b200.so: hand-written sm_100a kernels for the Glow flow
 * hot path of NFDPM (reference: davitpapikyan/Normalizing-Flow-with-Diffusion-Prior-Model).
 *
 * The reference is pure Python on PyTorch; it has no FFI of its own.  The "interface each entry
 * point replaces" is therefore the reference's Python call site (file:line below, relative to the
 * reference root), and the binding a maintainer adds is a ctypes stub (see INTEGRATION.md and
 * normalizing-flow-with-diffusion-prior-model_b200/normalizing_flow/_native.py).
 *
 * Conventions (all entry points):
 *   - plain C types only: raw DEVICE pointers, explicit sizes/strides (in ELEMENTS), stream last;
 *   - return 0 on success, non-zero on failure (nfdpm_last_error_string() explains, thread-local);
 *   - never allocate, never synchronise, never touch the legacy default stream implicitly: all
 *     work is enqueued on `stream`; scratch memory is passed in by the caller;
 *   - flow tensors are NCHW fp32 ("[B,C,P]" below, P = H*W) with an explicit batch stride so
 *     channel halves of a wider tensor can be read/written in place (chunk/concat without copies);
 *   - coupling-network activations are pixel-major rows "[M,ld]" (M = B*P, channel fastest),
 *     fp32 (NFDPM_F32, exact CUDA-core path), bf16 (NFDPM_BF16, tcgen05 tensor-core path) or split bf16 pairs
 *     (NFDPM_BF16X2, tcgen05 path with fp32-faithful products);
 *   - no CPU fallback exists anywhere in the library.
 */
#ifndef NFDPM_B200_H_
#define NFDPM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NFDPM_VERSION 100

/* element / accumulator type codes */
#define NFDPM_F32 0
#define NFDPM_F64 1
#define NFDPM_BF16 2
/* Split bf16 pairs, the operand format of the fp32-faithful tensor-core mode: a logical value v is stored as
 * hi = bf16(v) and lo = bf16(v - hi) (v = hi + lo to 2^-17 relative).  A row of ld logical columns (ld % 32 == 0)
 * occupies 2*ld bf16 = 4*ld bytes; group g = k/32 owns 64 consecutive bf16: [hi(32g .. 32g+31) | lo(32g .. 32g+31)].
 * The GEMM kernels compute A*B as Ahi*Bhi + Alo*Bhi + Ahi*Blo with fp32 accumulation in tensor memory (three
 * tcgen05.mma per K slice), which reproduces the reference's fp32 convolutions (utils.py:36,64, transforms.py:266)
 * to ~1e-6 relative instead of bf16's ~2e-3.  Sizes / leading dimensions of such matrices count LOGICAL elements. */
#define NFDPM_BF16X2 3

/* GEMM epilogues */
#define NFDPM_EPI_RAW 0          /* D = acc                                   */
#define NFDPM_EPI_ACTNORM_RELU 1 /* D = max(0, exp(scale[n]) * (acc + bias[n])) (utils.py:69,84-87) */

typedef void* nfdpm_stream_t; /* cudaStream_t */

int nfdpm_version(void);
const char* nfdpm_last_error_string(void);
/* Number of SMs of the current device (grid sizing on the host side); <0 on error. */
int nfdpm_sm_count(void);

/* ---------------------------------------------------------------------------------------------
 * K-LU + fold: per-step parameter preparation, batched over n steps in ONE launch per 16 items.
 * Replaces torch.slogdet(weight.double()) (normalizing_flow/transforms.py:131) and
 * weight.inverse() (transforms.py:144), and folds ActNorm (transforms.py:80, :93) into the 1x1 mix:
 *   forward  y = W*diag(exp(s))*(x + b)        -> fwd_mt[i*C+o] = W[o][i]*exp(s[i]),  fwd_beta[o] = sum_i fwd_mt[i][o]*b[i]
 *   inverse  x = diag(exp(-s))*W^-1*y - b      -> inv_mt[i*C+o] = exp(-s[o])*Winv[o][i], inv_beta[o] = -b[o]
 *   logdet[0] = log|det W| (fp64 partial-pivot LU, rounded to fp32) + sum(s)
 * weight==NULL means identity, scale/bias==NULL mean zeros.  Any output pointer may be NULL.
 * lu_ws: 2*C*C doubles of scratch per item (required when weight != NULL).
 */
typedef struct {
  const float* weight; /* [C,C] row = output channel (InvConv2d.weight squeezed) */
  const float* scale;  /* [C] ActNorm.scale */
  const float* bias;   /* [C] ActNorm.bias  */
  int32_t C;
  int32_t pad_;
  float* fwd_mt;
  float* fwd_beta;
  float* inv_mt;
  float* inv_beta;
  float* winv;   /* [C,C] row-major W^-1 (fp32) */
  float* logdet; /* [1] */
  double* lu_ws; /* [2*C*C] */
} nfdpm_mix_item;
int nfdpm_mix_prepare(const nfdpm_mix_item* items_host, int n, nfdpm_stream_t stream);

/* K-A / K-A^-1: y[b,o,p] = sum_i mt[i*C+o]*x[b,i,p] + beta[o]  (fused ActNorm + 1x1 conv,
 * transforms.py:80 + :132 forward; :144 + :93 inverse).  x,y: [B,C,P] with batch strides.
 * C <= 1024; above 192 the matrix streams through shared memory in chunks (same summation order) and x, y must not
 * overlap. */
int nfdpm_channel_mix(const float* x, float* y, const float* mt, const float* beta, int B, int C, int P,
                      int64_t x_bstride, int64_t y_bstride, nfdpm_stream_t stream);

/* Stand-alone ActNorm (transforms.py:80 / :93): inverse==0: y = exp(s[c])*(x+b[c]); else y = x*exp(-s[c]) - b[c]. */
int nfdpm_actnorm_apply(const float* x, float* y, const float* scale, const float* bias, int B, int C, int P,
                        int inverse, nfdpm_stream_t stream);

/* Data-dependent ActNorm statistics (transforms.py:74-78): scale_out[c] = -log(std_unbiased + 1e-6),
 * bias_out[c] = -mean.  layout 0: x is [B,C,P] (NCHW, batch stride xs); layout 1: x is rows [M=B*P, ld=xs],
 * channel fastest.  Written straight into the parameter storage. */
int nfdpm_channel_stats(const float* x, int layout, int B, int C, int P, int64_t xs, float* scale_out,
                        float* bias_out, nfdpm_stream_t stream);

/* Squeeze / unsqueeze (transforms.py:226 / :238): out channel = c*4 + h1*2 + w1.
 * squeeze: x [B,C,H,W] -> y [B,4C,H/2,W/2]; unsqueeze: x [B,C,H,W] -> y [B,C/4,2H,2W]. */
int nfdpm_squeeze(const float* x, float* y, int B, int C, int H, int W, int64_t x_bstride, int64_t y_bstride,
                  nfdpm_stream_t stream);
int nfdpm_unsqueeze(const float* x, float* y, int B, int C, int H, int W, int64_t x_bstride, int64_t y_bstride,
                    nfdpm_stream_t stream);
/* chunk / concat without torch: copy a [B,Cn,P] channel block between strided tensors (transforms.py:285, :308). */
int nfdpm_copy_channels(const float* src, float* dst, int B, int Cn, int P, int64_t src_bstride,
                        int64_t dst_bstride, nfdpm_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Coupling network (normalizing_flow/utils.py:83-89) as three GEMMs over pixel-major rows.
 *   conv3x3(C/2->512): A1 = im2col(x_a) [M, ld>=9*C/2], column = c*9 + ky*3 + kx (== the layout of
 *                      nn.Conv2d.weight.view(512,-1)), zero padded up to ld        -> nfdpm_im2col3x3
 *   conv1x1(512->512): plain GEMM
 *   ZeroConv3x3(512->C): "taps as N": PM[m, tap*C+co] = sum_ci h2[m,ci]*W3[co,ci,tap] (one GEMM, N=9C);
 *                      the 3x3 gather-add over neighbouring pixels happens in nfdpm_coupling_apply.
 */
 /* (out_dtype of nfdpm_im2col3x3 / nfdpm_pack_matrix / nfdpm_pack_batch and the a1_dtype of the step-boundary entry points:
 *  NFDPM_F32, NFDPM_BF16 or NFDPM_BF16X2; for split pairs ld_out % 32 == 0.) */
int nfdpm_im2col3x3(const float* x, void* out, int out_dtype, int B, int Cin, int H, int W, int64_t x_bstride,
                    int64_t ld_out, nfdpm_stream_t stream);

/* Generic gather + cast used to lay out weights for the GEMMs (no arithmetic):
 *   out[(a*nb + b)*ld_out + k] = in[a*sa + b*sb + k*sk]  for a<na, b<nb, k<nk; columns nk..ld_out-1 and
 *   rows na*nb..rows_out-1 are zero-filled. */
int nfdpm_pack_matrix(const float* in, void* out, int out_dtype, int na, int nb, int nk, int64_t sa, int64_t sb,
                      int64_t sk, int64_t ld_out, int rows_out, nfdpm_stream_t stream);

/* nfdpm_pack_matrix for MANY matrices in one launch (all weight layouts of all StepFlows after an optimiser step).
 * jobs_dev: device table of 10 x int64 per job: in, out, sa, sb, sk, ld_out, na|nb<<32, nk|rows_out<<32,
 * out_dtype|first_block<<32, nk2|sk2<<32 (column k reads offset (k/nk2)*sk + (k%nk2)*sk2; nk2 = 1 is the plain form).
 * Job i owns blocks [first_block_i, first_block_{i+1}): ceil(rows_out/64) * ceil(ld_out/64) tiles of 64 x 64 elements. */
int nfdpm_pack_elems(void);
int nfdpm_pack_batch(const int64_t* jobs_dev, int n_jobs, int n_blocks, nfdpm_stream_t stream);

/* D[M,N] = epilogue(A[M,K] * Bw[N,K]^T).  A, Bw: in_dtype (NFDPM_F32 -> CUDA-core fp32 kernel,
 * NFDPM_BF16 / NFDPM_BF16X2 -> tcgen05/TMEM kernel, fp32 accumulate); D: out_dtype (F32, BF16, or BF16X2 from
 * BF16X2 operands).  K must be a multiple of 16 (F32) / 64 (BF16) / 32 (BF16X2, with lda, ldb, ldd % 32 == 0) and
 * lda, ldb, ldd multiples of 8.  Replaces nn.Conv2d.forward at
 * utils.py:69 (x2) and ZeroConv2d's conv at utils.py:44, transforms.py:266. */
int nfdpm_gemm_nt(const void* A, int64_t lda, const void* Bw, int64_t ldb, void* D, int64_t ldd, int M, int N,
                  int K, int in_dtype, int out_dtype, int epilogue, const float* ep_scale, const float* ep_bias,
                  nfdpm_stream_t stream);

/* Affine-coupling epilogue (transforms.py:179-184 forward, :196-200 inverse).
 *   pm   [M, ldp]: taps-as-N output of the ZeroConv GEMM (column = tap*C + co, tap = ky*3+kx)
 *   net[co] = (sum_tap pm[m + (ky-1)*W + (kx-1), tap*C+co] (zero outside the image) + bias3[co]) * exp(3*logs3[co])
 *   log_s = net[0:C/2], t = net[C/2:C], s = sigmoid(log_s + 2)
 *   forward: y_b = (x_b + t)*s;   inverse: y_b = x_b/(s + 1e-6) - t;   both: ld_part = sum log(s + 1e-6)
 * x,y [B,C,P] NCHW (batch strides); the first C/2 channels are copied through when y != x.
 * ld_part (either direction, may be NULL): fp32 [T][B] partial sums, T = nfdpm_ld_tiles(P); entry t*B+b.  The inverse's
 * partial equals the forward's bit for bit for the same pm: it is -log|det| of the inverse at its output. */
int nfdpm_ld_tiles(int P);
int nfdpm_coupling_apply(const float* pm, int64_t ldp, const float* bias3, const float* logs3, const float* x,
                         float* y, float* ld_part, int B, int C, int H, int W, int64_t x_bstride,
                         int64_t y_bstride, int inverse, nfdpm_stream_t stream);

/* Split prior (transforms.py:266-268, 286-289; prior.py:36-37).  h [M, ldh] = raw ZeroConv GEMM output
 * (N = C, column = co; NULL when the prior is not learned -> mean = logs = 0), bias/logs = split.conv.{bias,logs}.
 *   mean = ((h+bias)*exp(3*logs))[0:C/2], lg = (...)[C/2:C];  z = x[:, C/2:C]
 *   logp_part[t*B+b] = sum -0.5*(log(2pi) + 2*lg + (z-mean)^2*exp(-2*lg))      (may be NULL)
 *   z_out [B,C/2,P] contiguous copy of z (may be NULL). */
int nfdpm_split_prior_logp(const float* h, int64_t ldh, const float* bias, const float* logs, const float* x,
                           int64_t x_bstride, float* z_out, float* logp_part, int B, int C, int H, int W,
                           nfdpm_stream_t stream);
/* Split.invert without a latent (transforms.py:305-307, prior.py:49-50): writes
 * mean + exp(lg)*temperature*eps into channels C/2..C of y [B,C,P]; eps [B,C/2,P] contiguous. */
int nfdpm_split_prior_sample(const float* h, int64_t ldh, const float* bias, const float* logs, const float* eps,
                             float temperature, float* y, int64_t y_bstride, int B, int C, int H, int W,
                             nfdpm_stream_t stream);
/* nfdpm_split_prior_sample with per-image temperatures and seeded draws.  Exactly one of eps / seeds is given.
 *   temp_b   fp32 [B]: the temperature of image b (NULL: `temperature` for every image)
 *   seeds    int64 [B]: the draw of image b is a pure function of (seeds[b], stream_id, element index), independent of the
 *            batch, the image's position in it and any earlier draw (contract below); NULL: read eps as above
 *   stream_id the draw site (Glow: the level of the Split; a stand-alone Split or GlowBlock: 0; GaussianPrior: 0xFFFFFFFF);
 *            must be 0 without seeds
 *   eps_out  [B,C/2,P] contiguous (may be NULL; needs seeds): receives the drawn standard normals
 * Draw contract (Philox4x32-10 of <curand_philox4x32_x.h>, full-precision logf / sincospif):
 *   key = (lo32(s), hi32(s)) with s = seeds[b] as uint64;  counter = (e >> 2, stream_id, 0, 0), e = c*P + p the element's
 *   index in the image's drawn tensor [C_draw, H, W];  u_i = fp32((w_i >> 8) + 0.5) * 2^-24 for the four output words
 *   (in (0, 1]: the +0.5 rounds to even from 2^23 on);  r = sqrtf(-2 logf(u_even)), sincospif(2 u_odd):
 *   n_even = r*cos, n_odd = r*sin for the pairs (w0, w1), (w2, w3);  element e takes n[e & 3].
 * With NULL new arguments the result is nfdpm_split_prior_sample's bit for bit. */
int nfdpm_split_prior_sample_ex(const float* h, int64_t ldh, const float* bias, const float* logs, const float* eps,
                                const int64_t* seeds, uint32_t stream_id, float temperature, const float* temp_b,
                                float* eps_out, float* y, int64_t y_bstride, int B, int C, int H, int W,
                                nfdpm_stream_t stream);

/* GaussianPrior (prior.py:70-99): the reference convolves an all-zero map, so mean/logs are the
 * per-channel constants (bias*exp(3*logs))[0:C] and [C:2C] of the 2C-channel ZeroConv2d.
 * bias/logs NULL -> standard normal.  logp_part: fp32 [B]. */
int nfdpm_gauss_logp_const(const float* z, const float* bias, const float* logs, float* logp_part, int B, int C,
                           int P, nfdpm_stream_t stream);
int nfdpm_gauss_sample_const(const float* eps, const float* bias, const float* logs, float temperature, float* out,
                             int B, int C, int P, nfdpm_stream_t stream);
/* nfdpm_gauss_sample_const with temp_b / seeds / stream_id / eps_out as in nfdpm_split_prior_sample_ex (the drawn tensor
 * of image b is out[b], [C, P]; GaussianPrior.sample draws with stream_id 0xFFFFFFFF).  NULL new arguments: the old bits. */
int nfdpm_gauss_sample_const_ex(const float* eps, const int64_t* seeds, uint32_t stream_id, const float* bias,
                                const float* logs, float temperature, const float* temp_b, float* eps_out, float* out, int B,
                                int C, int P, nfdpm_stream_t stream);

/* Fused step boundary (one CTA per image; P = H*W <= 256 and the image must fit in shared memory, see
 * nfdpm_flow_boundary_smem): source -> [affine coupling with pm] -> [channel mix] -> NCHW state and/or im2col rows.
 * Equivalent to nfdpm_coupling_apply + nfdpm_channel_mix + nfdpm_im2col3x3 (+ nfdpm_squeeze when squeeze_in) in ONE
 * launch with coalesced traffic; replaces the same reference lines (transforms.py:80,132,144,93,179-184,196-200,226).
 *   in  [B,C,P] (batch stride in_bs) or, with squeeze_in, [B,C/4,2H,2W];  pm == NULL: no coupling;
 *   mt == NULL: no mix;  y == NULL / a1 == NULL: sink disabled;  ld_part [B] (coupling in either direction, may be
 *   NULL: the sum of log(s + 1e-6), as in nfdpm_coupling_apply);
 *   a1: rows [B*P, lda1] of dtype a1_dtype (F32/BF16), column = c*9 + ky*3 + kx over the first C/2 channels. */
size_t nfdpm_flow_boundary_smem(int C, int H, int W, int coupling, int mix);
int nfdpm_flow_boundary(const float* in, int64_t in_bs, int squeeze_in, const float* pm, int64_t ldp,
                        const float* bias3, const float* logs3, float* ld_part, const float* mt, const float* beta,
                        float* y, int64_t y_bs, void* a1, int a1_dtype, int64_t lda1, int B, int C, int H, int W,
                        int inverse, nfdpm_stream_t stream);

/* Forward-only nfdpm_flow_boundary with one more sink for training: xs [B,C,P] receives the PRE-mix state (the
 * coupling output == the next StepFlow's input x, which its backward needs for d(weight) = du x^T). */
int nfdpm_flow_boundary_stash(const float* in, int64_t in_bs, int squeeze_in, const float* pm, int64_t ldp,
                              const float* bias3, const float* logs3, float* ld_part, const float* mt, const float* beta,
                              float* y, int64_t y_bs, float* xs, int64_t xs_bs, void* a1, int a1_dtype, int64_t lda1,
                              int B, int C, int H, int W, nfdpm_stream_t stream);
/* The INVERSE step boundary (coupling^-1 from pm, then the inverse mix mt/beta = inv_mt/inv_beta) with the sinks the
 * backward of Glow.invert needs: xs [B,C,P] receives the coupling^-1 output u (the inverse mix's input), y the step's
 * output, a1 (may be NULL) the next network's im2col rows.  No squeeze source, no log-det.  One CTA per image. */
int nfdpm_flow_boundary_inv_stash(const float* in, int64_t in_bs, const float* pm, int64_t ldp, const float* bias3,
                                  const float* logs3, const float* mt, const float* beta, float* y, int64_t y_bs, float* xs,
                                  int64_t xs_bs, void* a1, int a1_dtype, int64_t lda1, int B, int C, int H, int W,
                                  nfdpm_stream_t stream);
/* nfdpm_flow_boundary_inv_stash with a log-det sink: ld_part [B] (may be NULL) receives each image's sum of log(s + 1e-6),
 * the partial nfdpm_flow_boundary writes in inverse mode (same arithmetic and reduction order).  The density of a
 * recorded Glow.invert. */
int nfdpm_flow_boundary_inv_stash_ld(const float* in, int64_t in_bs, const float* pm, int64_t ldp, const float* bias3,
                                     const float* logs3, float* ld_part, const float* mt, const float* beta, float* y,
                                     int64_t y_bs, float* xs, int64_t xs_bs, void* a1, int a1_dtype, int64_t lda1, int B,
                                     int C, int H, int W, nfdpm_stream_t stream);

/* ZeroConv GEMM + step boundary in ONE launch (tensor-core mode): pm = h2[M,K] * w3p[ldp,K]^T is accumulated in tensor
 * memory, staged in shared memory and consumed by the arithmetic of nfdpm_flow_boundary (coupling source), so the
 * taps-as-N rows never reach L2/HBM.  Same reference lines as nfdpm_gemm_nt (utils.py:44) + nfdpm_flow_boundary.
 * h2, w3p: h_dtype = NFDPM_BF16 or NFDPM_BF16X2 (K, ldh count logical columns); CTAs own whole images: needs H*W == 256 or
 * H*W dividing 128, ldp <= 512 (nfdpm_gemm3_boundary_ok, whose K counts bf16 columns: 2 x logical K for split pairs).
 * pm_out (optional, fp32 [M, ld_pm_out]): copy of pm for the training stash; xs: pre-mix stash as in ..._stash;
 * ld_part [B] in either direction, as in nfdpm_flow_boundary. */
int nfdpm_gemm3_boundary_ok(int B, int C, int H, int W, int K, int64_t ldp);
int nfdpm_gemm3_boundary(const void* h2, int h_dtype, int64_t ldh, const void* w3p, float* pm_out, int64_t ld_pm_out, const float* in,
                         int64_t in_bs, const float* bias3, const float* logs3, float* ld_part, const float* mt,
                         const float* beta, float* y, int64_t y_bs, float* xs, int64_t xs_bs, void* a1, int a1_dtype,
                         int64_t lda1, int B, int C, int H, int W, int K, int64_t ldp, int inverse,
                         nfdpm_stream_t stream);

/* profiling hook: per-CTA wait/work cycle counters of the tcgen05 GEMM kernel (device int64 [grid][16], NULL = off) */
int nfdpm_gemm_debug(void* counters);
/* profiling hook: per-image phase timeline of nfdpm_flow_boundary (device int64 [B][16], NULL = off) */
int nfdpm_flow_boundary_debug(void* timeline);

/* Layout converters for stand-alone ZeroConv2d / Conv2dActNorm module calls (normalizing_flow/utils.py:43-44, :68-69).
 *   rows_to_nchw: out[b,n,p] = f(h[(b*P+p)*ldh + n]); mode 0: identity; 1: (v+p1[n])*exp(3*p2[n]) (ZeroConv2d gain);
 *                 2: exp(p1[n])*(v+p2[n]) (ActNorm).   nchw_to_rows: rows[m, c] = x[b,c,p], columns Cc..ld-1 zero. */
int nfdpm_rows_to_nchw(const float* h, int64_t ldh, int mode, const float* p1, const float* p2, float* out, int B,
                       int Nc, int P, nfdpm_stream_t stream);
int nfdpm_nchw_to_rows(const float* x, void* out, int out_dtype, int B, int Cc, int P, int64_t x_bstride, int64_t ld,
                       nfdpm_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Backward (training) — what autograd computes for the reference lines cited at each forward entry point.
 * All reductions are two-stage in a fixed order (deterministic).
 */
/* Affine coupling + log-det backward (transforms.py:179-184).  dy [B,C,P] grad of the coupling output, dld [B] grad of
 * log_det_jac (may be NULL), u [B,C,P] coupling input, pm as in the forward.  Outputs: du [B,C,P] (first half = dy_a;
 * the coupling-net part is added by nfdpm_mix_bwd), dpm [B*P, ld_dpm] (F32, BF16 or BF16X2, columns >= 9C zero-filled: the
 * K operand of the ZeroConv dgrad GEMM), dpar [B][2C] per-image partials (dbias3[C], dlogs3[C]).  With `counter` (one
 * zero-initialised int32, re-armed by the kernel) the last CTA sums dpar over the images in order into dbias[C] /
 * dlogs[C]; with counter == NULL reduce dpar with nfdpm_reduce_rows2. */
int nfdpm_coupling_bwd(const float* dy, int64_t dy_bs, const float* dld, const float* u, int64_t u_bs, const float* pm,
                       int64_t ldp, const float* bias3, const float* logs3, float* du, int64_t du_bs, void* dpm,
                       int dpm_dtype, int64_t ld_dpm, float* dpar, float* dbias, float* dlogs, int32_t* counter,
                       float* dp_scratch, int B, int C, int H, int W, nfdpm_stream_t stream);
/* 1: one CTA per image (dp_scratch unused).  > 1: the image is processed in pixel tiles: dpar has B*tiles rows (reduce
 * with nfdpm_reduce_rows2), dp_scratch [B*H*W*C] floats is required and counter must be NULL. */
int nfdpm_coupling_bwd_tiles(int C, int H, int W);
/* Backward of the INVERSE coupling x_b = y_b/(s+1e-6) - t, x_a = y_a (transforms.py:196-200): y is the inverse's input,
 * dx the gradient of its output.  dy_a = dx_a (the coupling-network part is added later through col2im),
 * dy_b = dx_b/(s+1e-6); ds = -dx_b*y_b/(s+1e-6)^2, dt = -dx_b.  dpm, dpar, dbias/dlogs/counter, dp_scratch and the
 * one-CTA-per-image / pixel-tiled choice (nfdpm_coupling_bwd_tiles) are exactly those of nfdpm_coupling_bwd; no log-det. */
int nfdpm_coupling_inv_bwd(const float* dx, int64_t dx_bs, const float* y, int64_t y_bs, const float* pm, int64_t ldp,
                           const float* bias3, const float* logs3, float* dy, int64_t dy_bs, void* dpm, int dpm_dtype,
                           int64_t ld_dpm, float* dpar, float* dbias, float* dlogs, int32_t* counter, float* dp_scratch,
                           int B, int C, int H, int W, nfdpm_stream_t stream);
/* nfdpm_coupling_inv_bwd plus the gradient of the log-det the inverse accumulates, sum log(s+1e-6): dld [B] (may be NULL:
 * identical to nfdpm_coupling_inv_bwd) adds dld/(s+1e-6) to ds, the forward's term of nfdpm_coupling_bwd. */
int nfdpm_coupling_inv_bwd_ld(const float* dx, int64_t dx_bs, const float* dld, const float* y, int64_t y_bs,
                              const float* pm, int64_t ldp, const float* bias3, const float* logs3, float* dy, int64_t dy_bs,
                              void* dpm, int dpm_dtype, int64_t ld_dpm, float* dpar, float* dbias, float* dlogs,
                              int32_t* counter, float* dp_scratch, int B, int C, int H, int W, nfdpm_stream_t stream);
/* ActNorm+ReLU backward on rows (utils.py:69,84-87): dpre = dh*(h>0)*exp(scale); part[cta][2N] partial d(scale), d(bias);
 * ctas = ceil(M/rows_per_cta).  dtypes: any mix of F32 / BF16, or the fp32-faithful form (F32 dh, BF16X2 h) -> BF16X2 dpre. */
int nfdpm_actnorm_relu_bwd(const void* dh, int dh_dtype, int64_t ld_dh, const void* h, int h_dtype, int64_t ld_h,
                           const float* scale, void* dpre, int o_dtype, int64_t ld_o, float* part, int M, int N,
                           int rows_per_cta, nfdpm_stream_t stream);
/* out[i] (+)= sum_{r<R} part[r*stride + i], i < n */
int nfdpm_reduce_rows(const float* part, float* out, int R, int n, int64_t stride, int accumulate, nfdpm_stream_t stream);
/* out0[i] = sum_r part[r*stride + i] for i < n0, out1[i-n0] likewise for n0 <= i < n0+n1 (a parameter pair in one launch) */
int nfdpm_reduce_rows2(const float* part, float* out0, float* out1, int R, int n0, int n1, int64_t stride,
                       nfdpm_stream_t stream);
/* Fused ActNorm + 1x1 conv backward (transforms.py:80,132) incl. col2im of the im2col-row gradient da1 (may be NULL):
 * dx = W^T du; part [B][C*C + C]: per-image sum_p du[o]x[i] and sum_p du[o]. */
/* pixel tiles per image of nfdpm_mix_bwd: `part` has B*tiles rows of C*C + C floats (1 for C > 192).  C <= 1024;
 * above 192 channels dx must not overlap du. */
int nfdpm_mix_bwd_tiles(int C, int H, int W);
int nfdpm_mix_bwd(const float* du, int64_t du_bs, const float* da1, int64_t lda1, const float* x, int64_t x_bs,
                  const float* mt, float* dx, int64_t dx_bs, float* part, int B, int C, int H, int W,
                  nfdpm_stream_t stream);
/* d(InvConv2d.weight), d(ActNorm.scale), d(ActNorm.bias) of n StepFlows from the nfdpm_mix_bwd partials plus the
 * log-det terms  P*sum(dld)*W^-T  and  P*sum(dld)  (transforms.py:81,131). */
typedef struct {
  const float* part; int32_t B; int32_t C;
  const float* weight; const float* scale; const float* bias; const float* winv;
  const float* dld_sum; float P; int32_t pad_;
  float* d_weight; float* d_scale; float* d_bias; float* scratch; /* scratch: C*C + C floats */
} nfdpm_mix_grad_item;
int nfdpm_mix_param_grad(const nfdpm_mix_grad_item* items_host, int n, nfdpm_stream_t stream);
/* Parameter gradients of the INVERSE mix x = M u - b, M = diag(e^-s) W^-1 (transforms.py:92-94,142-145), from the
 * partials of an nfdpm_mix_bwd run with mt = inv_mt (its x = the inverse input u, its du = grad wrt the output x):
 * d_bias = -g, d_scale_c = -sum_j G_cj M_cj, d_weight = -W^-T diag(e^-s) G W^-T.  weight may be NULL; winv is W^-1 (the
 * identity for a lone ActNorm); any of d_weight / d_scale / d_bias may be NULL.  dld_sum (may be NULL: no log-det term)
 * is sum_b d(ld)[b] for the constant P*(sum s + log|det W|) the inverse accumulates: it adds P*dld_sum*W^-T to d_weight
 * and P*dld_sum to d_scale.  C <= 1024 (scratch stays C*C + C floats). */
int nfdpm_mix_inv_param_grad(const nfdpm_mix_grad_item* items_host, int n, nfdpm_stream_t stream);
/* Weight gradients: D[N1,N2] (+)= sum_m A[m,N1]*B[m,N2] (A, B row-major, F32, BF16 or both BF16X2; D fp32 with ldd == N2).
 * Split pairs (needs counters): the tensor-core accumulator holds hi*hi, hi*lo, lo*hi, lo*lo of every logical element and the
 * in-kernel reduction adds the four: the exact product of the represented values.
 * ws: nfdpm_gemm_tn_workspace(M,N1,N2,NULL) floats.  counters (may be NULL): >= 1024 int32, ZERO before the first use
 * and private to one stream; with it the bf16 tensor-core path sums its split-M partial slabs inside the GEMM kernel
 * (the CTAs of an output tile wait for each other; fixed slab order, so the result stays bitwise reproducible) instead
 * of in a second launch.  The kernel re-arms the counters itself.  out_mode != PLAIN (needs counters + bf16 operands)
 * writes the sum directly in the weight tensor's own layout, saving the unpack launch.  With out_mode PLAIN and either split
 * pairs or bf16 operands with counters, the reduction stores float4 rows: D must then be 16-byte aligned. */
int64_t nfdpm_gemm_tn_workspace(int M, int N1, int N2, int* splits_out);
#define NFDPM_TN_OUT_PLAIN 0 /* D[n1*N2 + n2]                                                               */
#define NFDPM_TN_OUT_TAPS 1  /* n1 = tap*out_c + co -> D[(co*N2 + n2)*9 + tap]: ZeroConv weight [out_c,N2,3,3] */
#define NFDPM_TN_OUT_STRIP 2 /* D[n1*out_c + n2] for n2 < out_c: drops the K-padding columns of the im2col rows  */
int nfdpm_gemm_tn(const void* A, int a_dtype, int64_t lda, const void* Bm, int b_dtype, int64_t ldb, float* D, int64_t ldd,
                  int M, int N1, int N2, float* ws, int accumulate, int32_t* counters, int out_mode, int out_c,
                  nfdpm_stream_t stream);
/* Split prior backward (transforms.py:286-289, prior.py:36-37): dstate[:, C/2:] += dz; dh rows [M, ldh]; dpar [B][2C]. */
int nfdpm_split_prior_bwd(const float* dlp, const float* h, int64_t ldh, const float* bias, const float* logs,
                          const float* x, int64_t xbs, float* dstate, int64_t dbs, float* dh, float* dpar, int B, int C,
                          int H, int W, nfdpm_stream_t stream);
/* GaussianPrior backward (prior.py:79-83): dz [B,C,P]; dpar [B][4C] per-image partials: d(bias)[2C], d(logs)[2C]. */
int nfdpm_gauss_const_bwd(const float* dl, const float* z, const float* bias, const float* logs, float* dz, float* dpar,
                          int B, int C, int P, nfdpm_stream_t stream);
/* Backward of the reparameterised prior draw z = mean + exp(lg)*T*eps (transforms.py:305-307, prior.py:49-50,97-99):
 * (mean, lg) = (h + bias)*exp(3*logs) split into channel halves; C = 2 x latent channels.  dz: [B, C/2, P] with batch
 * stride dz_bs; eps: [B, C/2, P] contiguous.  d mean = dz, d lg = dz*exp(lg)*T*eps.  Writes dh rows [M, ldh] (columns
 * C..ldh zero) for the conv's wgrad / dgrad GEMMs and dpar [B][2C]: per-image d(bias)[C], d(logs)[C].  h == NULL: mean / lg
 * are the per-channel constants bias*exp(3*logs) (GaussianPrior) and dh is not written. */
int nfdpm_split_sample_bwd(const float* dz, int64_t dz_bs, const float* eps, float temperature, const float* h, int64_t ldh,
                           const float* bias, const float* logs, float* dh, float* dpar, int B, int C, int H, int W,
                           nfdpm_stream_t stream);
/* nfdpm_split_sample_bwd plus the gradient of the draw's log-density sum -(log 2pi + 2 lg + T^2 eps^2)/2 (the logp term of
 * a sampled Split in Glow.invert): d lg -= dlp[b] per element, nothing on the mean.  dlp [B] may be NULL (identical to
 * nfdpm_split_sample_bwd). */
int nfdpm_split_sample_bwd_lp(const float* dz, int64_t dz_bs, const float* dlp, const float* eps, float temperature,
                              const float* h, int64_t ldh, const float* bias, const float* logs, float* dh, float* dpar,
                              int B, int C, int H, int W, nfdpm_stream_t stream);
/* nfdpm_split_sample_bwd_lp with a per-image temperature: temp_b fp32 [B] (may be NULL: `temperature` for every image, the
 * old bits).  eps is the draw the forward used (eps_out of a seeded draw). */
int nfdpm_split_sample_bwd_ex(const float* dz, int64_t dz_bs, const float* eps, float temperature, const float* temp_b,
                              const float* dlp, const float* h, int64_t ldh, const float* bias, const float* logs, float* dh,
                              float* dpar, int B, int C, int H, int W, nfdpm_stream_t stream);
/* dstate[b,c,p] += col2im(da)[b,c,p] for c < Cin (input gradient of a 3x3 "same" conv expressed as im2col rows). */
int nfdpm_col2im_add(const float* da, int64_t lda, float* dstate, int64_t dbs, int B, int Cin, int H, int W,
                     nfdpm_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Fused optimiser step = trainer.py:165-167 (clip_grad_value_, clip_grad_norm_, Adam/AdamW step; utils.py:120-137) in
 * three launches over all parameter tensors.
 *   refs    device table, one 32-byte record per tensor: { float* param; float* grad (NULL = skip); int64 state_off;
 *           int32 numel; int32 clip (member of the clip group) }
 *   chunks  device table of n_chunks int32 pairs { tensor index, element offset }, one per nfdpm_opt_chunk() elements
 *   exp_avg / exp_avg_sq  flat fp32 state (indexed by state_off), partial [n_chunks] scratch,
 *   scal    [3] device floats: clip coefficient (out), gradient norm of the clip group (out), step count (in/out, += 1)
 * Gradients of the clip group are modified in place (clamped, then scaled) exactly like the two torch utilities. */
int nfdpm_opt_chunk(void);
int nfdpm_fused_clip_adam(const void* refs, const int32_t* chunks, int n_chunks, float* exp_avg, float* exp_avg_sq,
                          float* partial, float* scal, float clip_value, float max_norm, double lr, double beta1,
                          double beta2, double eps, double weight_decay, int decoupled, nfdpm_stream_t stream);

/* acc[b] += sum_{r<R} part[r*B+b] + sum_{j<nc} cmul[j]*cval[j]   (fixed order -> deterministic).
 * acc is the caller's running log_det_jac / logp (`+=` in place, transforms.py:81,131,184,288), fp32 or fp64.
 * cval/cmul: device fp32 arrays (e.g. logdet constants and their H*W multipliers); may be NULL with nc=0. */
int nfdpm_accumulate(void* acc, int acc_dtype, const float* part, int R, int B, const float* cval,
                     const float* cmul, int nc, nfdpm_stream_t stream);

/* Row-band variant of nfdpm_flow_boundary (csrc/flow_boundary_tiled.cu): the same arithmetic and arguments, but a CTA owns a
 * band of image rows (plus one recomputed halo row above and below when there is an im2col sink), so images of any size
 * take the fused boundary and small batches spread over B * tiles CTAs.  `in` and `y` / `xs` must NOT alias (a band reads
 * halo rows another band writes).  nfdpm_flow_boundary_tiles() returns the number of bands per image for a shape and
 * sink combination (0: one row does not fit in shared memory); the log-det (either direction) is written as `tiles`
 * partial rows: ld_part[t * B + b].  Replaces, like nfdpm_flow_boundary: transforms.py:179-184 / :196-200 (coupling), :80 + :132 /
 * :144 + :93 (ActNorm + 1x1 conv), :226 (squeeze) and the im2col of utils.py:64's 3x3 conv. */
int nfdpm_flow_boundary_tiles(int B, int C, int H, int W, int coupling, int mix, int want_a1);
int nfdpm_flow_boundary_tiled(const float* in, int64_t in_bs, int squeeze_in, const float* pm, int64_t ldp,
                              const float* bias3, const float* logs3, float* ld_part, const float* mt, const float* beta,
                              float* y, int64_t y_bs, float* xs, int64_t xs_bs, void* a1, int a1_dtype, int64_t lda1, int B,
                              int C, int H, int W, int inverse, int tiles, nfdpm_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Data formats either side of the flow (SURVEY §8f): the diffusion prior's latent formater and the
 * image pre/post-processing of the training / sampling loops.  Pure HBM-bound byte work.
 *
 * CatFormater (diffusion_prior/latent_formaters.py:163-236): process_latents squeezes / unsqueezes every
 * latent part to the resolution of the middle part and concatenates along channels; postprocess is the
 * inverse.  ONE launch moves all parts.  Part i is the contiguous latent [B,C,H,W]; `degree` = number of
 * squeezes (>0) or unsqueezes (<0) that bring it to Ht x Wt; its slice of cat is [ch_offset, ch_offset+ch_count).
 * to_cat != 0: latents -> cat [B,Ct,Ht,Wt] (process_latents); to_cat == 0: cat -> latents (postprocess). */
#define NFDPM_MAX_LATENT_PARTS 8
typedef struct {
  float* ptr;
  int32_t C, H, W;
  int32_t degree;
  int32_t ch_offset;
  int32_t ch_count;
} nfdpm_latent_part;
int nfdpm_latent_format(const nfdpm_latent_part* parts_host, int n_parts, float* cat, int B, int Ct, int Ht, int Wt,
                        int to_cat, nfdpm_stream_t stream);

/* postprocess_batch (normalizing_flow/utils.py:199-210) on the device:
 *   out[i] = (uint8) clip(floor((x[i] + 0.5) * n_bins) * out_scale, 0, 255),  out_scale = (float)(256.0 / n_bins).
 * The caller copies the uint8 result to the host (1 byte per value instead of 4). */
int nfdpm_postprocess_u8(const float* x, uint8_t* out, int64_t n, float n_bins, float out_scale, nfdpm_stream_t stream);

/* preprocess_batch (normalizing_flow/utils.py:175-196) fused with the dequantisation-noise add of the training
 * step (normalizing_flow/trainer.py:155):  y = floor(x*255 / 2^(8-n_bits)) / n_bins - 0.5  [+ noise / n_bins]
 * (floor only when n_bits < 8; noise may be NULL).  Same fp32 operation order as the reference: bit-identical. */
int nfdpm_preprocess(const float* x, const float* noise, float* y, int64_t n, int n_bits, float n_bins,
                     nfdpm_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* NFDPM_B200_H_ */
