// Scatter-max for sm_100a: torch_scatter.scatter(src, index, dim, out, dim_size, reduce="max"), the call PointSea's
// renderer makes to draw its depth maps (models_PointSea/mv_utils_zs.py:130).
//
// Values are combined in place with integer atomics that preserve the order of IEEE floats, so no scratch buffer is
// needed and the result does not depend on the order of the updates (it is bit-exact against any correct max):
//   sign bit clear: atomicMax on the bits as int       (+0 < ... < +inf < NaN)
//   sign bit set:   atomicMin on the bits as unsigned  (-0 > ... > -inf)
// A positive pattern is larger than every negative one in both comparisons, so the two kinds mix correctly.  The
// branch is on the sign bit, not on v >= 0: -0.0 on the signed path would read INT_MIN and lose to every negative
// value.  NaN is canonicalised to one positive pattern, so it wins (torch's scatter_reduce "amax" propagates NaN) and a
// negative NaN never reaches the unsigned path.  A NaN already in a caller's `out=` is kept too: a positive pattern
// beats every value, and an atomic that replaces a negative pattern sees it in its return value and puts the canonical
// NaN back (an atomicMax that nothing can beat).  This costs no pass over `out`.
//
// One atomic per element.  Combining the lanes of a warp that hit the same output element first (__match_any_sync,
// then one atomic per group) was measured against it on PointSea's render shapes and is not used: it is 1.3-2.5x slower
// when the pixels of a warp differ, which is what projected clouds give, and wins only when whole warps hit one pixel
// (DESIGN.md §4.9).
//
// The argmax pass (optional) runs after the value pass: atomicMin of the position along E of every element equal to
// the result (NaN matching NaN), so the lowest position wins, deterministically.
#include "common.cuh"

namespace ps {
namespace {

constexpr int SC_THREADS = 256;
constexpr unsigned NEG_FLT_MAX_BITS = 0xff7fffffu;  // -FLT_MAX: torch_scatter's initial value of a fresh max
constexpr unsigned CANONICAL_NAN = 0x7fc00000u;

// Flat position p of a (outer, E, inner) tensor -> (o, e, i).  Sizes are 64-bit; when the tensor has fewer than 2^32
// elements the divisions are done in 32 bits (a 64-bit division is a long software sequence).
struct Split3 {
  long long o, e, i;
};
__device__ __forceinline__ Split3 split3(long long p, long long E, long long inner, bool small) {
  Split3 s;
  const long long row = E * inner;
  if (small) {
    const unsigned up = (unsigned)p, ur = (unsigned)row, ui = (unsigned)inner;
    const unsigned o = up / ur, r = up - o * ur, e = r / ui;
    s.o = o;
    s.e = e;
    s.i = r - e * ui;
  } else {
    s.o = p / row;
    const long long r = p - s.o * row;
    s.e = r / inner;
    s.i = r - s.e * inner;
  }
  return s;
}

__device__ __forceinline__ unsigned canonical_bits(float v) { return v != v ? CANONICAL_NAN : __float_as_uint(v); }

__global__ void __launch_bounds__(SC_THREADS) scatter_prep_kernel(float* __restrict__ out, long long* __restrict__ arg,
                                                                  long long m, long long E, int fresh) {
  const long long stride = (long long)gridDim.x * SC_THREADS;
  for (long long j = (long long)blockIdx.x * SC_THREADS + threadIdx.x; j < m; j += stride) {
    if (fresh) out[j] = __uint_as_float(NEG_FLT_MAX_BITS);
    if (arg) arg[j] = E;
  }
}

// torch_scatter's masked_fill(out == lowest, 0): also turns a max of exactly -FLT_MAX into 0
__global__ void __launch_bounds__(SC_THREADS) scatter_zero_empty_kernel(float* __restrict__ out, long long m) {
  const long long stride = (long long)gridDim.x * SC_THREADS;
  for (long long j = (long long)blockIdx.x * SC_THREADS + threadIdx.x; j < m; j += stride)
    if (__float_as_uint(out[j]) == NEG_FLT_MAX_BITS) out[j] = 0.f;
}

__global__ void __launch_bounds__(SC_THREADS) scatter_max_kernel(const float* __restrict__ src,
                                                                 const long long* __restrict__ index,
                                                                 float* __restrict__ out, long long n, long long E,
                                                                 long long inner, long long D, bool small) {
  const long long stride = (long long)gridDim.x * SC_THREADS;
  for (long long p = (long long)blockIdx.x * SC_THREADS + threadIdx.x; p < n; p += stride) {
    const long long d = __ldg(index + p);
    if ((unsigned long long)d >= (unsigned long long)D) continue;
    const Split3 s = split3(p, E, inner, small);
    float* dst = out + (s.o * D + d) * inner + s.i;
    const unsigned bits = canonical_bits(__ldg(src + p));
    const unsigned old = (bits >> 31) ? atomicMin(reinterpret_cast<unsigned*>(dst), bits)
                                      : (unsigned)atomicMax(reinterpret_cast<int*>(dst), (int)bits);
    if (old > 0xff800000u) atomicMax(reinterpret_cast<int*>(dst), (int)CANONICAL_NAN);  // replaced a negative NaN
  }
}

__global__ void __launch_bounds__(SC_THREADS) scatter_argmax_kernel(const float* __restrict__ src,
                                                                    const long long* __restrict__ index,
                                                                    const float* __restrict__ out,
                                                                    long long* __restrict__ arg, long long n,
                                                                    long long E, long long inner, long long D,
                                                                    bool small) {
  const long long stride = (long long)gridDim.x * SC_THREADS;
  for (long long p = (long long)blockIdx.x * SC_THREADS + threadIdx.x; p < n; p += stride) {
    const long long d = __ldg(index + p);
    if ((unsigned long long)d >= (unsigned long long)D) continue;
    const Split3 s = split3(p, E, inner, small);
    const long long dst = (s.o * D + d) * inner + s.i;
    const float v = __ldg(src + p), r = out[dst];
    if (v == r || (v != v && r != r))
      atomicMin(reinterpret_cast<unsigned long long*>(arg + dst), (unsigned long long)s.e);
  }
}

int grid_for(long long work, int dev) {
  const long long blocks = (work + SC_THREADS - 1) / SC_THREADS, cap = (long long)sm_count(dev) * (2048 / SC_THREADS);
  return (int)(blocks < cap ? blocks : cap);
}

bool mul_overflows(long long a, long long b, long long c, long long* r) {
  long long t;
  return __builtin_mul_overflow(a, b, &t) || __builtin_mul_overflow(t, c, r);
}

}  // namespace
}  // namespace ps

using namespace ps;

extern "C" int ps_scatter_max(const float* src, const long long* index, float* out, long long* argmax, long long outer,
                              long long E, long long inner, long long D, int fresh, int dev, void* stream_) {
  long long n = 0, m = 0;
  PS_REQUIRE(outer >= 0 && E >= 0 && inner >= 0 && D >= 0 && !mul_overflows(outer, E, inner, &n) &&
                 !mul_overflows(outer, D, inner, &m),
             "ps_scatter_max: bad sizes outer=%lld E=%lld inner=%lld D=%lld", outer, E, inner, D);
  if (m == 0) return PS_OK;  // nothing to write (with D == 0 every index is out of range)
  if (n == 0 && !fresh && !argmax) return PS_OK;
  PS_REQUIRE(out && (n == 0 || (src && index)), "ps_scatter_max: null pointer");
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_scatter_max: cannot select device %d", dev);
  cudaStream_t stream = (cudaStream_t)stream_;
  const bool small = n <= 0xffffffffLL;
  if (fresh || argmax) {
    scatter_prep_kernel<<<grid_for(m, dev), SC_THREADS, 0, stream>>>(out, argmax, m, E, fresh);
    PS_LAUNCH_CHECK();
  }
  if (n > 0) {
    scatter_max_kernel<<<grid_for(n, dev), SC_THREADS, 0, stream>>>(src, index, out, n, E, inner, D, small);
    PS_LAUNCH_CHECK();
  }
  if (fresh) {
    scatter_zero_empty_kernel<<<grid_for(m, dev), SC_THREADS, 0, stream>>>(out, m);
    PS_LAUNCH_CHECK();
  }
  if (argmax && n > 0) {
    scatter_argmax_kernel<<<grid_for(n, dev), SC_THREADS, 0, stream>>>(src, index, out, argmax, n, E, inner, D, small);
    PS_LAUNCH_CHECK();
  }
  return PS_OK;
}
