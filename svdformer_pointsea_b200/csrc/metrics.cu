// Evaluation epilogue of the Chamfer distance for sm_100a: per-cloud CD terms, F-score and the
// density-aware Chamfer distance in ONE launch.
//
// Replaces the torch expressions the reference runs after every chamfer_3DDist call in evaluation
//   calc_cd    utils/loss_utils.py:98-115   cd_p = (mean sqrt d1 + mean sqrt d2) / 2, cd_t = mean d1 + mean d2
//   fscore     metrics/CD/fscore.py:3-16    precision_i = mean(d_i < thr), f = 2 p1 p2 / (p1 + p2), NaN -> 0
//   calc_dcd   utils/loss_utils.py:117-155  count_1[x] = #{gt points whose nearest neighbour is x} (scatter_add on
//              idx1), weight = 1 / (count^n_lambda + 1e-6) * frac, loss_1 = mean(1 - exp(-alpha d1) * weight), ...
// (about 30 torch kernels and four (B,n)-sized temporaries per call) by a single kernel: one CTA per
// cloud, the two hit-count histograms live in shared memory (global scratch beyond 40960 points), and one
// pass over dist/idx produces all eight per-cloud numbers.
//   out (B,8) f32 = { mean sqrt d1, mean sqrt d2, mean d1, mean d2, precision_1, precision_2, fscore, dcd }
// Sums are accumulated in fp64 (torch reduces in fp32 with its own tree order; the callers' tolerance is
// 1e-5 relative, asserted in tests/test_gpu_parity.py).  Element-wise fp32 steps follow the reference's order.
//
// Backward (chamfer_metrics_bwd_kernel): per-cloud upstream gradients of the five differentiable outputs (and of the
// raw dist outputs) -> per-point gradients of dist1 / dist2, which ps_chamfer_bwd turns into point gradients.  Same
// layout as the forward; the hit-count histograms are rebuilt rather than kept from the forward.
#include "common.cuh"

namespace ps {
namespace {

constexpr int MT_THREADS = 1024;
constexpr int MT_SMEM_POINTS = 40960;  // n1 + n2 ints that fit the shared-memory histograms (160 KB)

__device__ __forceinline__ double block_sum(double v, double* red) {
  __syncthreads();  // red may still be read from the previous call
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  if (threadIdx.x < 32) {
    t = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
  }
  return t;  // valid in thread 0
}

// Hit-count histograms of one cloud: count1 (n2 entries) = hits per cloud-2 point from idx1, count2 = count1 + n2
// (n1 entries) = hits per cloud-1 point from idx2.  In shared memory (zeroed here) or in the cloud's slice of a
// zero-filled global scratch.  Ends with a barrier: one CTA owns the cloud, so block-level visibility is enough for
// global counts too.
__device__ __forceinline__ void hit_histograms(const int* __restrict__ i1, const int* __restrict__ i2, int* count1,
                                               int n1, int n2, int use_smem) {
  int* count2 = count1 + n2;
  if (use_smem) {
    for (int j = threadIdx.x; j < n1 + n2; j += MT_THREADS) count1[j] = 0;
    __syncthreads();
  }
  for (int j = threadIdx.x; j < n1; j += MT_THREADS) atomicAdd(&count1[__ldg(i1 + j)], 1);
  for (int j = threadIdx.x; j < n2; j += MT_THREADS) atomicAdd(&count2[__ldg(i2 + j)], 1);
  __syncthreads();
}

// calc_dcd's weight of a point whose nearest neighbour was hit cnt times: (cnt ** n_lambda + 1e-6) ** (-1) * frac
__device__ __forceinline__ float dcd_weight(int cnt, float n_lambda, float frac) {
  float w = (float)cnt;
  if (n_lambda == 0.5f) w = sqrtf(w);                                // count.float() ** n_lambda (torch's pow
  else if (n_lambda == 2.0f) w = __fmul_rn(w, w);                    // special-cases 0.5 and 2)
  else if (n_lambda != 1.0f) w = powf(w, n_lambda);
  return __fmul_rn(__frcp_rn(__fadd_rn(w, 1e-6f)), frac);
}

// One side of calc_dcd: sum over j of 1 - exp(-alpha * d[j]) * weight(count[idx[j]])
__device__ __forceinline__ float dcd_term(float d, int cnt, float alpha, float n_lambda, float frac) {
  const float e = expf(__fmul_rn(-d, alpha));                       // torch.exp(-dist * alpha)
  return __fsub_rn(1.0f, __fmul_rn(e, dcd_weight(cnt, n_lambda, frac)));
}

__global__ void __launch_bounds__(MT_THREADS) chamfer_metrics_kernel(
    const float* __restrict__ dist1, const float* __restrict__ dist2, const int* __restrict__ idx1,
    const int* __restrict__ idx2, float* __restrict__ out, int* __restrict__ gcount, int n1, int n2,
    float thr, float alpha, float n_lambda, float frac1, float frac2, int use_smem) {
  extern __shared__ int scount[];
  __shared__ double red[32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* d1 = dist1 + (size_t)b * n1;
  const float* d2 = dist2 + (size_t)b * n2;
  const bool dcd = idx1 != nullptr && idx2 != nullptr;
  int* count1 = use_smem ? scount : gcount + (size_t)b * (n1 + n2);
  int* count2 = count1 + n2;
  if (dcd) hit_histograms(idx1 + (size_t)b * n1, idx2 + (size_t)b * n2, count1, n1, n2, use_smem);
  double s_sqrt1 = 0, s1 = 0, hit1 = 0, l1 = 0, s_sqrt2 = 0, s2 = 0, hit2 = 0, l2 = 0;
  for (int j = tid; j < n1; j += MT_THREADS) {
    const float d = __ldg(d1 + j);
    s_sqrt1 += (double)sqrtf(d);
    s1 += (double)d;
    hit1 += d < thr ? 1.0 : 0.0;
    if (dcd) l1 += (double)dcd_term(d, count1[__ldg(idx1 + (size_t)b * n1 + j)], alpha, n_lambda, frac1);
  }
  for (int j = tid; j < n2; j += MT_THREADS) {
    const float d = __ldg(d2 + j);
    s_sqrt2 += (double)sqrtf(d);
    s2 += (double)d;
    hit2 += d < thr ? 1.0 : 0.0;
    if (dcd) l2 += (double)dcd_term(d, count2[__ldg(idx2 + (size_t)b * n2 + j)], alpha, n_lambda, frac2);
  }
  double v[8] = {s_sqrt1, s_sqrt2, s1, s2, hit1, hit2, l1, l2};
#pragma unroll
  for (int i = 0; i < 8; i++) v[i] = block_sum(v[i], red);
  if (tid == 0) {
    float* o = out + (size_t)b * 8;
    o[0] = (float)(v[0] / n1);
    o[1] = (float)(v[1] / n2);
    o[2] = (float)(v[2] / n1);
    o[3] = (float)(v[3] / n2);
    const float p1 = (float)(v[4] / n1), p2 = (float)(v[5] / n2);
    o[4] = p1;
    o[5] = p2;
    const float f = __fdiv_rn(__fmul_rn(__fmul_rn(2.0f, p1), p2), __fadd_rn(p1, p2));  // fscore.py:14
    o[6] = (f != f) ? 0.f : f;                                                           // fscore.py:15
    o[7] = dcd ? __fdiv_rn(__fadd_rn((float)(v[6] / n1), (float)(v[7] / n2)), 2.0f) : 0.f;  // (loss1 + loss2) / 2
  }
}

// bits of ps_chamfer_metrics_bwd's `terms`: the per-cloud upstream gradients present in gcoef5 (B,5)
constexpr unsigned T_SQRT1 = 1u, T_SQRT2 = 2u, T_MEAN1 = 4u, T_MEAN2 = 8u, T_DCD = 16u, T_ALL = 31u;

// Gradient w.r.t. the distances of one side (n points):
//   gd[j] = graw[j] + (g_sqrt / n) / (2 sqrt d[j]) + g_mean / n + ((g_dcd * 0.5 / n) * w(count[idx[j]])) * exp(-alpha d[j]) * alpha
// which is torch's backward of mean, sqrt (grad / (2 result)), (loss1 + loss2) / 2, 1 - e * w and exp(-d * alpha), in
// torch's order of operations.  A term whose bit is clear is skipped, so it cannot contribute a NaN.  The upstream
// gradients are read here, not passed in: values live across the first side's loop would be spilled around the
// calls of the division slow path.
__device__ __forceinline__ void dist_grad_side(const float* __restrict__ d, const int* __restrict__ idx,
                                               const int* count, const float* __restrict__ graw, float* __restrict__ gd,
                                               int n, const float* __restrict__ gc, unsigned terms, unsigned sqrt_bit,
                                               unsigned mean_bit, float alpha, float n_lambda, float frac) {
  const bool sq = terms & sqrt_bit, mean = terms & mean_bit, dcd = terms & T_DCD;
  const float fn = (float)n;
  const float cs = sq ? __fdiv_rn(__ldg(gc + __ffs(sqrt_bit) - 1), fn) : 0.f;
  const float cm = mean ? __fdiv_rn(__ldg(gc + __ffs(mean_bit) - 1), fn) : 0.f;
  const float cd = dcd ? __fdiv_rn(__fmul_rn(__ldg(gc + 4), 0.5f), fn) : 0.f;
  for (int j = threadIdx.x; j < n; j += MT_THREADS) {
    float acc = graw ? __ldg(graw + j) : 0.f;
    const float dj = (sq || dcd) ? __ldg(d + j) : 0.f;
    if (sq) acc = __fadd_rn(acc, __fdiv_rn(cs, __fmul_rn(2.0f, sqrtf(dj))));
    if (mean) acc = __fadd_rn(acc, cm);
    if (dcd) {
      const float e = expf(__fmul_rn(-dj, alpha));
      const float w = dcd_weight(count[__ldg(idx + j)], n_lambda, frac);
      acc = __fadd_rn(acc, __fmul_rn(__fmul_rn(__fmul_rn(cd, w), e), alpha));
    }
    gd[j] = acc;
  }
}

__global__ void __launch_bounds__(MT_THREADS) chamfer_metrics_bwd_kernel(
    const float* __restrict__ dist1, const float* __restrict__ dist2, const int* __restrict__ idx1,
    const int* __restrict__ idx2, const float* __restrict__ gcoef5, unsigned terms, const float* __restrict__ graw1,
    const float* __restrict__ graw2, float* __restrict__ graddist1, float* __restrict__ graddist2,
    int* __restrict__ gcount, int n1, int n2, float alpha, float n_lambda, float frac1, float frac2, int use_smem) {
  extern __shared__ int scount[];
  const int b = blockIdx.x;
  const size_t o1 = (size_t)b * n1, o2 = (size_t)b * n2;
  const bool dcd = terms & T_DCD;
  int* count1 = nullptr;  // histograms exist only with the dcd term
  if (dcd) {
    count1 = use_smem ? scount : gcount + (size_t)b * (n1 + n2);
    hit_histograms(idx1 + o1, idx2 + o2, count1, n1, n2, use_smem);
  }
  const float* gc = gcoef5 + (size_t)b * 5;  // only read for set bits: gcoef5 may be NULL when terms == 0
  dist_grad_side(dist1 + o1, dcd ? idx1 + o1 : nullptr, count1, graw1 ? graw1 + o1 : nullptr, graddist1 + o1, n1, gc,
                 terms, T_SQRT1, T_MEAN1, alpha, n_lambda, frac1);
  dist_grad_side(dist2 + o2, dcd ? idx2 + o2 : nullptr, dcd ? count1 + n2 : nullptr, graw2 ? graw2 + o2 : nullptr, graddist2 + o2, n2,
                 gc, terms, T_SQRT2, T_MEAN2, alpha, n_lambda, frac2);
}

// Storage of the hit-count histograms of B clouds: dynamic shared memory (*smem bytes) when n1 + n2 fits, otherwise a
// zero-filled global scratch owned by `mem` (*gcount).
int histogram_storage(int B, int n1, int n2, int dev, cudaStream_t stream, ScratchGuard& mem, size_t* smem, int** gcount) {
  if ((long long)n1 + n2 <= MT_SMEM_POINTS) {
    *smem = (size_t)(n1 + n2) * sizeof(int);
    return PS_OK;
  }
  const size_t bytes = (size_t)B * ((size_t)n1 + n2) * sizeof(int);
  if (int rc = mem.alloc(bytes, dev, stream)) return rc;
  *gcount = static_cast<int*>(mem.ptr);
  return fill32_async(*gcount, 0u, bytes, stream);
}

}  // namespace
}  // namespace ps

using namespace ps;

extern "C" int ps_chamfer_metrics(const float* dist1, const float* dist2, const int* idx1, const int* idx2,
                                  float* out8, int B, int n1, int n2, float fscore_threshold, float dcd_alpha,
                                  float dcd_n_lambda, float dcd_frac1, float dcd_frac2, int dev, void* stream_) {
  PS_REQUIRE(B >= 0 && n1 > 0 && n2 > 0, "ps_chamfer_metrics: bad sizes B=%d n1=%d n2=%d", B, n1, n2);
  if (B == 0) return PS_OK;
  PS_REQUIRE(dist1 && dist2 && out8, "ps_chamfer_metrics: null pointer");
  PS_REQUIRE((idx1 == nullptr) == (idx2 == nullptr), "ps_chamfer_metrics: idx1 and idx2 must both be given (DCD) or both be NULL");
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_chamfer_metrics: cannot select device %d", dev);
  cudaStream_t stream = (cudaStream_t)stream_;
  const int use_smem = (long long)n1 + n2 <= MT_SMEM_POINTS;
  ScratchGuard gcount_mem;
  int* gcount = nullptr;
  size_t smem = 0;
  if (idx1 != nullptr)
    if (int rc = histogram_storage(B, n1, n2, dev, stream, gcount_mem, &smem, &gcount)) return rc;
  PS_CUDA(cudaFuncSetAttribute(chamfer_metrics_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(MT_SMEM_POINTS * sizeof(int))));
  chamfer_metrics_kernel<<<B, MT_THREADS, smem, stream>>>(dist1, dist2, idx1, idx2, out8, gcount, n1, n2, fscore_threshold,
                                                          dcd_alpha, dcd_n_lambda, dcd_frac1, dcd_frac2, use_smem);
  PS_LAUNCH_CHECK();
  return gcount_mem.release();
}

extern "C" int ps_chamfer_metrics_bwd(const float* dist1, const float* dist2, const int* idx1, const int* idx2,
                                      const float* gcoef5, unsigned terms, const float* graw1, const float* graw2,
                                      float* graddist1, float* graddist2, int B, int n1, int n2, float dcd_alpha,
                                      float dcd_n_lambda, float dcd_frac1, float dcd_frac2, int dev, void* stream_) {
  PS_REQUIRE(B >= 0 && n1 > 0 && n2 > 0, "ps_chamfer_metrics_bwd: bad sizes B=%d n1=%d n2=%d", B, n1, n2);
  PS_REQUIRE((terms & ~T_ALL) == 0u, "ps_chamfer_metrics_bwd: unknown terms bits 0x%x", terms & ~T_ALL);
  if (B == 0) return PS_OK;
  PS_REQUIRE(dist1 && dist2 && graddist1 && graddist2, "ps_chamfer_metrics_bwd: null pointer");
  PS_REQUIRE(gcoef5 || terms == 0u, "ps_chamfer_metrics_bwd: null pointer gcoef5 with terms 0x%x", terms);
  PS_REQUIRE((idx1 && idx2) || !(terms & T_DCD), "ps_chamfer_metrics_bwd: null pointer idx1/idx2 with the dcd term (bit 4)");
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_chamfer_metrics_bwd: cannot select device %d", dev);
  cudaStream_t stream = (cudaStream_t)stream_;
  const int use_smem = (long long)n1 + n2 <= MT_SMEM_POINTS;
  ScratchGuard gcount_mem;
  int* gcount = nullptr;
  size_t smem = 0;
  if (terms & T_DCD)
    if (int rc = histogram_storage(B, n1, n2, dev, stream, gcount_mem, &smem, &gcount)) return rc;
  PS_CUDA(cudaFuncSetAttribute(chamfer_metrics_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(MT_SMEM_POINTS * sizeof(int))));
  chamfer_metrics_bwd_kernel<<<B, MT_THREADS, smem, stream>>>(dist1, dist2, idx1, idx2, gcoef5, terms, graw1, graw2,
                                                              graddist1, graddist2, gcount, n1, n2, dcd_alpha, dcd_n_lambda,
                                                              dcd_frac1, dcd_frac2, use_smem);
  PS_LAUNCH_CHECK();
  return gcount_mem.release();
}
