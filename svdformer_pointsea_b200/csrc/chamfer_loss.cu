// The four Chamfer training losses of utils/loss_utils.py:10-31 as one forward and one backward.
//
// Forward: the Chamfer forward with its fused loss sums (chamfer_fwd_impl with sums6, as ps_chamfer_fwd_sums), then
// one single-thread kernel that combines the sums in double and rounds once to the fp32 loss.  The loss stays on the
// device, so the call needs no host sync and can be captured in a CUDA graph.
//
// Backward: each point's distance gradient is derived inline from the upstream gradient of the loss and the forward's
// own `dist`, with the operations torch's autograd applies to the reference expression:
//   DivBackward of "/ 2"     g * 0.5                          (sqrt kinds)
//   MeanBackward             g * (1.0f / n)                   (torch's CUDA division by a scalar multiplies by the
//                                                              fp32 reciprocal, computed on the host)
//   SqrtBackward             g / (2 * sqrtf(d))               (inf / NaN at d = 0, exactly where torch has them)
// and then the arithmetic of ps_chamfer_bwd (g + g, __fmul_rn(g, a - b)).  Two passes, as chamfer_bwd_kernel: plain
// stores of each point's own term, then atomics for the scattered terms.  A NULL gradient buffer is skipped in both
// passes; a non-NULL one is fully overwritten (zero where no term reaches it).
#include "comm.cuh"

namespace ps {

// the loss of `kind` from the six sums of ps_chamfer_sums (counts in s[4], s[5]; an empty batch gives NaN, as
// torch.mean of an empty tensor)
__global__ void chamfer_loss_finalize_kernel(const double* __restrict__ s, float* __restrict__ loss, int kind) {
  double v;
  switch (kind) {
    case PS_LOSS_CD: v = s[2] / s[4] + s[3] / s[5]; break;
    case PS_LOSS_CD_SQRT: v = (s[0] / s[4] + s[1] / s[5]) * 0.5; break;
    case PS_LOSS_SINGLE: v = s[2] / s[4]; break;
    default: v = s[0] / s[4]; break;  // PS_LOSS_SINGLE_SQRT
  }
  *loss = (float)v;
}

struct ChamferLossBwdParams {
  const float *xyz1, *xyz2, *dist1, *dist2;
  const int *idx1, *idx2;
  const float* grad_loss;
  float *g1, *g2;
  float inv1, inv2;  // 1.0f / n1, 1.0f / n2
  int N, M, kind;
  size_t tot1, lo, hi;  // this pass covers elements [lo, hi) of side 1 (< tot1) followed by side 2
};

template <bool SCATTER>
__global__ void __launch_bounds__(256) chamfer_loss_bwd_kernel(const ChamferLossBwdParams p) {
  size_t i = p.lo + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= p.hi) return;
  const bool side2 = i >= p.tot1;
  if (side2) i -= p.tot1;
  const float* a = side2 ? p.xyz2 : p.xyz1;
  const float* bt = side2 ? p.xyz1 : p.xyz2;
  float* ga = side2 ? p.g2 : p.g1;
  float* gb = side2 ? p.g1 : p.g2;
  const int na = side2 ? p.M : p.N, nb = side2 ? p.N : p.M;
  const bool single = p.kind == PS_LOSS_SINGLE || p.kind == PS_LOSS_SINGLE_SQRT;
  if (side2 && single) {  // no term on side 2: only pass A reaches here, to zero the buffer
    ga[i * 3 + 0] = 0.f;
    ga[i * 3 + 1] = 0.f;
    ga[i * 3 + 2] = 0.f;
    return;
  }
  const bool sqrt_kind = p.kind == PS_LOSS_CD_SQRT || p.kind == PS_LOSS_SINGLE_SQRT;
  float g0 = __ldg(p.grad_loss);
  if (p.kind == PS_LOSS_CD_SQRT) g0 = __fmul_rn(g0, 0.5f);
  g0 = __fmul_rn(g0, side2 ? p.inv2 : p.inv1);
  if (sqrt_kind) {
    const float d = __ldg((side2 ? p.dist2 : p.dist1) + i);
    g0 = __fdiv_rn(g0, __fmul_rn(2.f, __fsqrt_rn(d)));
  }
  const size_t b = i / na;
  const int j = __ldg((side2 ? p.idx2 : p.idx1) + i);
  const float* pa = a + i * 3;
  const float* pb = bt + (b * nb + j) * 3;
  const float g = g0 + g0;
  const float vx = __fmul_rn(g, __ldg(pa + 0) - __ldg(pb + 0));
  const float vy = __fmul_rn(g, __ldg(pa + 1) - __ldg(pb + 1));
  const float vz = __fmul_rn(g, __ldg(pa + 2) - __ldg(pb + 2));
  if (!SCATTER) {
    ga[i * 3 + 0] = vx;
    ga[i * 3 + 1] = vy;
    ga[i * 3 + 2] = vz;
  } else {
    float* o = gb + (b * nb + j) * 3;
    atomicAdd(o + 0, -vx);
    atomicAdd(o + 1, -vy);
    atomicAdd(o + 2, -vz);
  }
}

static bool loss_kind_ok(int kind) { return kind >= PS_LOSS_CD && kind <= PS_LOSS_SINGLE_SQRT; }

}  // namespace ps

using namespace ps;

extern "C" int ps_chamfer_loss_fwd(const float* xyz1, const float* xyz2, float* dist1, float* dist2, int* idx1,
                                   int* idx2, double* sums6, float* loss, int kind, int B, int N, int M, int dev,
                                   void* stream_) {
  PS_REQUIRE(loss_kind_ok(kind), "ps_chamfer_loss_fwd: unknown kind %d", kind);
  PS_REQUIRE(sums6 && loss, "ps_chamfer_loss_fwd: null pointer sums6 / loss");
  // validates sizes and the remaining pointers before any CUDA call; B = 0 zeroes sums6 (the loss becomes NaN)
  if (int rc = chamfer_fwd_impl(xyz1, xyz2, dist1, dist2, idx1, idx2, sums6, nullptr, B, N, M, dev, stream_,
                                "ps_chamfer_loss_fwd"))
    return rc;
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_chamfer_loss_fwd: cannot select device %d", dev);
  chamfer_loss_finalize_kernel<<<1, 1, 0, (cudaStream_t)stream_>>>(sums6, loss, kind);
  PS_LAUNCH_CHECK();
  return PS_OK;
}

extern "C" int ps_chamfer_loss_bwd(const float* xyz1, const float* xyz2, const float* dist1, const float* dist2,
                                   const int* idx1, const int* idx2, const float* grad_loss, float* gradxyz1,
                                   float* gradxyz2, int kind, int B, int N, int M, int dev, void* stream_) {
  PS_REQUIRE(B >= 0 && N > 0 && M > 0, "ps_chamfer_loss_bwd: bad sizes B=%d N=%d M=%d", B, N, M);
  PS_REQUIRE(loss_kind_ok(kind), "ps_chamfer_loss_bwd: unknown kind %d", kind);
  PS_REQUIRE(gradxyz1 || gradxyz2, "ps_chamfer_loss_bwd: gradxyz1 and gradxyz2 are both null");
  if (B == 0) return PS_OK;
  PS_REQUIRE(xyz1 && xyz2 && dist1 && dist2 && idx1 && idx2 && grad_loss, "ps_chamfer_loss_bwd: null pointer");
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_chamfer_loss_bwd: cannot select device %d", dev);
  cudaStream_t stream = (cudaStream_t)stream_;
  const size_t tot1 = (size_t)B * N, tot2 = (size_t)B * M;
  const bool two_sided = kind == PS_LOSS_CD || kind == PS_LOSS_CD_SQRT;
  ChamferLossBwdParams p{xyz1, xyz2, dist1, dist2, idx1, idx2, grad_loss, gradxyz1, gradxyz2,
                         1.0f / (float)tot1, 1.0f / (float)tot2, N, M, kind, tot1, 0, 0};
  // pass A: the points of each non-NULL buffer (side 1 first, so the range is contiguous)
  p.lo = gradxyz1 ? 0 : tot1;
  p.hi = gradxyz2 ? tot1 + tot2 : tot1;
  chamfer_loss_bwd_kernel<false><<<ceil_div(p.hi - p.lo, 256), 256, 0, stream>>>(p);
  PS_LAUNCH_CHECK();
  // pass B: side 1 scatters into gradxyz2, side 2 (two-sided kinds) into gradxyz1
  p.lo = gradxyz2 ? 0 : tot1;
  p.hi = (two_sided && gradxyz1) ? tot1 + tot2 : tot1;
  if (p.hi > p.lo) {
    chamfer_loss_bwd_kernel<true><<<ceil_div(p.hi - p.lo, 256), 256, 0, stream>>>(p);
    PS_LAUNCH_CHECK();
  }
  return PS_OK;
}
