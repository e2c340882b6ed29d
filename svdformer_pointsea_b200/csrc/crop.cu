// Online cropping of ShapeNet-55/34 (utils/helpers.py:62-123, seprate_point_cloud) for sm_100a.
//
// The reference loops over the batch: per cloud it computes torch.norm(center - points, p=2, dim=-1), runs a full
// torch.argsort over it and gathers the two halves of the sorted order (the points nearest the centre are the crop, the
// rest is the kept input).  Here one CTA per cloud does all of it in one launch:
//   * the distance is the fp32 value torch's norm returns: sqrt((x^2 + z^2) + y^2) with every step rounded on its own
//     (the order torch's reduction combines a length-3 row in, DESIGN.md §2), so the sort key has torch's rounding;
//   * the key (distance bits << 32 | point index) is unique, so any correct sort gives torch's stable order, ties
//     broken by the lower index.  Distances are never negative, so their bits order as unsigned integers; every NaN
//     becomes one pattern above +inf (torch's sort puts NaN last and keeps NaNs in index order);
//   * the keys are bitonic-sorted in shared memory (8 bytes per point: 128 KB at 16384 points);
//   * sorted position j < count goes to the crop row, the others to the kept row, both in ascending distance; with
//     pad_zeros the kept row is the whole cloud in its original order, cropped points multiplied by 0 (NaN and inf
//     give NaN and negative values -0.0, exactly as `points * 0`).
#include "common.cuh"

#include <cstring>

namespace ps {
namespace {

constexpr int CS_T = 1024;
constexpr int CS_MIN_N = 33, CS_MAX_N = 16384;

// torch.norm(d, p=2, dim=-1) over a length-3 row on CUDA (DESIGN.md §2)
__device__ __forceinline__ float torch_norm3(float dx, float dy, float dz) {
  return __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dz, dz)), __fmul_rn(dy, dy)));
}

// meta[b] = {centre x, y, z, count as int bits}
__global__ void __launch_bounds__(CS_T, 1) crop_split_kernel(const float* __restrict__ xyz, const float4* __restrict__ meta,
                                                           float* __restrict__ keep, float* __restrict__ crop, int N,
                                                           int npow2, long long keep_stride, long long crop_stride,
                                                           int pad_zeros) {
  extern __shared__ u64 keys[];
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* cloud = xyz + (size_t)b * N * 3;
  const float4 m = meta[b];
  for (int k = tid; k < npow2; k += CS_T) {
    u64 key = ~0ull;  // padding sorts after every point
    if (k < N) {
      const float d = torch_norm3(__fsub_rn(m.x, cloud[3 * k]), __fsub_rn(m.y, cloud[3 * k + 1]),
                                  __fsub_rn(m.z, cloud[3 * k + 2]));
      const unsigned bits = d != d ? 0x7fc00000u : __float_as_uint(d);
      key = ((u64)bits << 32) | (unsigned)k;
    }
    keys[k] = key;
  }
  __syncthreads();
  for (int size = 2; size <= npow2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < npow2 / 2; t += CS_T) {
        const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
        const u64 a = keys[lo], c = keys[hi];
        if ((a > c) == ((lo & size) == 0)) { keys[lo] = c; keys[hi] = a; }
      }
      __syncthreads();
    }
  }
  const int count = __float_as_int(m.w);
  float* kr = keep + (size_t)b * keep_stride * 3;
  float* cr = crop + (size_t)b * crop_stride * 3;
  for (int j = tid; j < N; j += CS_T) {
    const int k = (int)(unsigned)keys[j];
    const float px = cloud[3 * k], py = cloud[3 * k + 1], pz = cloud[3 * k + 2];
    if (j < count) { cr[3 * j] = px; cr[3 * j + 1] = py; cr[3 * j + 2] = pz; }
    if (pad_zeros) {
      float* o = kr + 3 * k;
      if (j < count) { o[0] = __fmul_rn(px, 0.f); o[1] = __fmul_rn(py, 0.f); o[2] = __fmul_rn(pz, 0.f); }
      else { o[0] = px; o[1] = py; o[2] = pz; }
    } else if (j >= count) {
      float* o = kr + 3 * (j - count);
      o[0] = px; o[1] = py; o[2] = pz;
    }
  }
}

}  // namespace
}  // namespace ps

using namespace ps;

extern "C" int ps_crop_split(const float* xyz, const float* centers_host, const int* num_crop_host, float* keep,
                             float* crop, int B, int N, int keep_stride, int crop_stride, int pad_zeros, int dev,
                             void* stream_) {
  PS_REQUIRE(B >= 0 && N >= 0 && keep_stride >= 0 && crop_stride >= 0,
             "ps_crop_split: bad sizes B=%d N=%d keep_stride=%d crop_stride=%d", B, N, keep_stride, crop_stride);
  if (B == 0) return PS_OK;
  PS_REQUIRE(xyz && centers_host && num_crop_host, "ps_crop_split: null pointer");
  if (N < CS_MIN_N || N > CS_MAX_N)
    return set_error(PS_ERR_UNSUPPORTED, "ps_crop_split: N=%d outside %d..%d (one CTA sorts one cloud)", N, CS_MIN_N,
                     CS_MAX_N);
  bool any_keep = false, any_crop = false;  // an output with only empty rows is never written and may be NULL
  for (int b = 0; b < B; b++) {
    const int c = num_crop_host[b];
    PS_REQUIRE(c >= 0 && c <= N, "ps_crop_split: count %d of cloud %d outside [0, %d]", c, b, N);
    PS_REQUIRE(crop_stride >= c && keep_stride >= (pad_zeros ? N : N - c),
               "ps_crop_split: cloud %d (count %d) does not fit rows of keep_stride=%d / crop_stride=%d", b, c,
               keep_stride, crop_stride);
    any_keep = any_keep || pad_zeros || c < N;
    any_crop = any_crop || c > 0;
  }
  PS_REQUIRE((keep || !any_keep) && (crop || !any_crop), "ps_crop_split: null pointer");
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_crop_split: cannot select device %d", dev);
  cudaStream_t stream = (cudaStream_t)stream_;
  float4* host_meta = new float4[B];
  for (int b = 0; b < B; b++) {
    host_meta[b] = make_float4(centers_host[3 * b], centers_host[3 * b + 1], centers_host[3 * b + 2], 0.f);
    memcpy(&host_meta[b].w, &num_crop_host[b], sizeof(int));
  }
  ScratchGuard meta;
  int rc = meta.alloc((size_t)B * sizeof(float4), dev, stream);
  // pageable source: the copy has taken the bytes when it returns, so the staging array can go at once
  if (rc == PS_OK && cudaMemcpyAsync(meta.ptr, host_meta, (size_t)B * sizeof(float4), cudaMemcpyHostToDevice, stream) !=
                         cudaSuccess)
    rc = set_error(PS_ERR_CUDA, "ps_crop_split: upload of centres and counts failed: %s",
                   cudaGetErrorString(cudaGetLastError()));
  delete[] host_meta;
  if (rc) return rc;
  int npow2 = 1;
  while (npow2 < N) npow2 <<= 1;
  const size_t smem = (size_t)npow2 * sizeof(u64);
  PS_CUDA(cudaFuncSetAttribute(crop_split_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  crop_split_kernel<<<B, CS_T, smem, stream>>>(xyz, static_cast<const float4*>(meta.ptr), keep, crop, N, npow2,
                                               keep_stride, crop_stride, pad_zeros);
  PS_LAUNCH_CHECK();
  return meta.release();
}
