// Furthest point sampling for sm_100a: one thread-block cluster per cloud.
//
// Replaces furthest_point_sampling_kernel (pointnet2_ops/_ext-src/src/sampling_gpu.cu:69-173).
//
// The reference keeps the running min-distance array `temp` in GLOBAL memory and re-reads the
// coordinates every iteration (sampling_gpu.cu:95-110), with one 512-thread block per cloud and
// a 9-level __syncthreads tree per iteration.  Here:
//   * a cluster of C CTAs x T threads owns one cloud; every thread owns P = 2*PP points whose
//     coordinates AND running min distance live in registers for the whole kernel (global memory
//     is read once); distances are evaluated two points at a time with FADD2/FMUL2/FFMA2;
//   * few fat threads (T = 128 or 256, up to 32 points each) rather than many thin ones: the
//     per-warp cost of the exchange (~90 instructions) is what limits the iteration rate, so it
//     is paid by 4-8 warps per SM instead of 16;
//   * per iteration a warp resolves its best with two REDUX ops (max of the distance bits, then
//     min of the tie-break rank);
//   * MODE 0 (C == 1): warp winners meet in shared memory, one __syncthreads per iteration;
//   * MODE 1 (C <= 4): every warp winner is pushed straight into the slot arrays of ALL CTAs of
//     the cluster with st.async (distributed shared memory); the bytes are counted on the
//     DESTINATION CTA's mbarrier, on which every warp of that CTA sleeps (try_wait) until all
//     (T/32)*C candidates of the iteration have landed, then reduces them redundantly.  No
//     barrier.cluster in the loop: its .release costs a MEMBAR.ALL.GPU per iteration (measured,
//     profiles/fps_r1_notes.md);
//   * MODE 2 (C >= 8): CTA-level reduce first (one __syncthreads), then one st.async per CTA pair.
//   * MODE 3 (C <= 4, the default there): same direct all-to-all as MODE 1, but with plain remote
//     vector stores (st.shared::cluster.v4) and TAG POLLING instead of st.async + mbarrier: each 16-byte half
//     of an entry carries the iteration number, and lane e of every warp spins on entry e of its OWN CTA's
//     slot array (local ld.volatile) until both halves show the current tag.  The async-proxy path costs
//     ~520 cycles even inside one CTA (profiles/microbench_r1.jsonl); a remote store is visible after ~1/2 of
//     the 215-cycle DSMEM round trip and a local poll costs ~40.  With 4 fat warps per CTA the polling load on
//     the LSU is small (the first attempt polled with 16 warps and lost to the barrier).  The spin is bounded:
//     a protocol failure traps (the launch fails with an error) instead of hanging the GPU or returning garbage.
//   The message carries the winner's coordinates, so the next iteration never touches global
//   memory.  Two slot buffers suffice: a writer can only be at iteration j+2 after consuming all
//   candidates of j+1, and a reader sends its j+1 candidate only after reading the slots of j.
//
// Bit-exact tie-breaking.  The reference's winner among equal distances is decided by its
// per-thread strict `>` scan (lowest k within thread tid = k mod bs) followed by the shared-
// memory tree whose __update keeps the LEFT operand on ties (sampling_gpu.cu:59-65,115-168):
// the tied thread with the smallest bit-reversed tid wins.  That order is
//     rank(k) = bitrev_L(k mod bs) * nper + floor(k / bs),  bs = 2^L = opt_n_threads(N),
//     nper = ceil(N / bs),
// and we select (distance desc, rank asc).  Points are DEALT TO THREADS IN RANK ORDER: thread g
// owns ranks [g*P, (g+1)*P), so the rank of its i-th point is g*P + i, the lowest i on a tie is
// the lowest rank, and no bit reversal is needed inside the loop.  Points with |p|^2 <= 1e-3
// (compared in double, as the reference does, sampling_gpu.cu:100-101) never update and are never
// selected; they are carried as distance -1, which orders below every real distance when the
// fp32 bit patterns are compared as signed integers.
#include "common.cuh"

#include <atomic>
#include <cmath>
#include <cstdlib>

namespace ps {

struct __align__(16) FpsEntry {  // two 16-byte vectors, each written by ONE st.async.v4
  int tb;          // distance bits (signed compare)
  unsigned rank;   // tie-break rank, smaller wins
  float x;
  unsigned pad_a;
  float y, z;
  int k;           // point index
  unsigned pad_b;
};

struct FpsArgs {
  const float* xyz;
  int* idx;
  float* new_xyz;  // optional (B, npoint, 3): coordinates of the sampled points (fused fps_subsample)
  int N, npoint;
  int L;     // log2(bs) of the reference launch
  int nper;  // ceil(N / bs)
  const int* run_flag = nullptr;  // optional (B): a cloud whose flag is 0 has been sampled by fps_pruned_kernel already
  // ragged batches (fps_small_kernel<..., true>): cloud b is the first part[b].x points of row b (rows of `stride`
  // points), with its own log2(bs) = part[b].y and nper = part[b].z
  const int4* part = nullptr;
  long long stride = 0;
};

// rank -> point index (may be >= N for the padding ranks of the last rows)
__device__ __forceinline__ int fps_rank_to_k(unsigned rank, int L, int nper) {
  const unsigned cls = rank / (unsigned)nper, m = rank % (unsigned)nper;
  const unsigned r = L ? (__brev(cls) >> (32 - L)) : 0u;
  return (int)(r + (m << L));
}

// lexicographic "a better than b": larger tb, then smaller rank
__device__ __forceinline__ bool fps_better(int tb_a, unsigned r_a, int tb_b, unsigned r_b) {
  return tb_a > tb_b || (tb_a == tb_b && r_a < r_b);
}

// Warp-wide argbest over (tb desc, rank asc); returns the winning lane.
__device__ __forceinline__ int warp_argbest(int tb, unsigned rank, int& tb_max) {
  tb_max = __reduce_max_sync(0xffffffffu, tb);
  const unsigned r = (tb == tb_max) ? rank : 0xffffffffu;
  const unsigned rmin = __reduce_min_sync(0xffffffffu, r);
  const unsigned m = __ballot_sync(0xffffffffu, r == rmin);
  return __ffs(m) - 1;
}

// ---- st.async + mbarrier: the remote store and its completion signal travel together -------------
__device__ __forceinline__ void fps_mbar_init(unsigned bar, unsigned cnt) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(cnt) : "memory");
}
__device__ __forceinline__ void fps_mbar_expect_tx(unsigned bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
// default (.acquire.cta) wait, as for TMA loads: the cluster-scope acquire would add a CCTL.IVALL
// (L1 invalidate) per iteration, and only shared memory is read after the wait.
__device__ __forceinline__ bool fps_mbar_try_wait(unsigned bar, unsigned parity) {
  unsigned ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
  return ok != 0;
}
__device__ __forceinline__ void st_async_v4(unsigned raddr, unsigned rbar, unsigned a, unsigned b, unsigned c, unsigned d) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];"
               ::"r"(raddr), "r"(a), "r"(b), "r"(c), "r"(d), "r"(rbar) : "memory");
}

__device__ __forceinline__ int4 ld_volatile_shared_v4(const void* p) {
  int4 v;
  asm volatile("ld.volatile.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(smem_u32(p)) : "memory");
  return v;
}
constexpr int FPS_SPIN_LIMIT = 1 << 22;  // ~0.1 s of polling: far beyond any legitimate wait

template <int PP, int T, int MODE>
__global__ void __launch_bounds__(T, 1) fps_kernel(const FpsArgs a) {
  constexpr int P = 2 * PP;
  constexpr int WARPS = T / 32;
  constexpr bool CLUSTER = MODE != 0;
  constexpr bool POLL = MODE == 3;
  constexpr bool DIRECT = MODE == 1 || MODE == 3;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  // layout: px[P*T] py[P*T] pz[P*T] pk[P*T] | mbar[2] (16 B) | slots[2][E] | wslots[2][WARPS] (MODE 2)
  float* px = reinterpret_cast<float*>(smem_raw);
  float* py = px + P * T;
  float* pz = py + P * T;
  int* pk = reinterpret_cast<int*>(pz + P * T);
  u64* mbar = reinterpret_cast<u64*>(pk + P * T);
  FpsEntry* slots = reinterpret_cast<FpsEntry*>(mbar + 2);

  const unsigned C = CLUSTER ? cluster_nctarank() : 1u;
  const unsigned crank = CLUSTER ? cluster_ctarank() : 0u;
  const int b = CLUSTER ? (int)cluster_id_x() : (int)blockIdx.x;
  if (a.run_flag && __ldg(a.run_flag + b) == 0) return;  // the whole cluster leaves together: nothing was armed yet
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int E = DIRECT ? WARPS * (int)C : (CLUSTER ? (int)C : WARPS);
  FpsEntry* wslots = slots + 2 * E;  // CTA-level staging (MODE 2)

  const int N = a.N;
  const float* cloud = a.xyz + (size_t)b * N * 3;
  int* out = a.idx + (size_t)b * a.npoint;
  const int g = (int)crank * T + tid;
  const unsigned rank0 = (unsigned)g * P;  // this thread owns ranks [rank0, rank0 + P)
  const unsigned R = (unsigned)a.nper << a.L;

  u64 x2[PP], y2[PP], z2[PP];
  float t[P];
#pragma unroll
  for (int i = 0; i < P; i++) {
    float xv = 0.f, yv = 0.f, zv = 0.f;
    int k = 0;
    t[i] = -1.0f;
    if (rank0 + i < R) {
      k = fps_rank_to_k(rank0 + i, a.L, a.nper);
      if (k < N) {
        xv = __ldg(cloud + (size_t)k * 3 + 0);
        yv = __ldg(cloud + (size_t)k * 3 + 1);
        zv = __ldg(cloud + (size_t)k * 3 + 2);
        const float mag = dist2_ref(xv, yv, zv);
        t[i] = ((double)mag <= 1e-3) ? -1.0f : 1e10f;
      }
    }
    px[i * T + tid] = xv;
    py[i * T + tid] = yv;
    pz[i * T + tid] = zv;
    pk[i * T + tid] = k;
    if (i & 1) {
      x2[i / 2] = pack2(lo2(x2[i / 2]), xv); y2[i / 2] = pack2(lo2(y2[i / 2]), yv); z2[i / 2] = pack2(lo2(z2[i / 2]), zv);
    } else {
      x2[i / 2] = pack2(xv, 0.f); y2[i / 2] = pack2(yv, 0.f); z2[i / 2] = pack2(zv, 0.f);
    }
  }
  if (POLL) {  // tags of both buffers start at 0 (iteration tags are >= 1)
    for (int e = tid; e < 2 * E; e += T) { slots[e].pad_a = 0u; slots[e].pad_b = 0u; }
  }
  if (CLUSTER && !POLL && tid == 0) {
    // one local arrive (the expect_tx) + E*32 bytes of st.async traffic complete a phase
    fps_mbar_init(smem_u32(&mbar[0]), 1);
    fps_mbar_init(smem_u32(&mbar[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fps_mbar_expect_tx(smem_u32(&mbar[0]), (unsigned)E * 32u);
    fps_mbar_expect_tx(smem_u32(&mbar[1]), (unsigned)E * 32u);
  }
  const float p0x = __ldg(cloud + 0), p0y = __ldg(cloud + 1), p0z = __ldg(cloud + 2);
  float lx = p0x, ly = p0y, lz = p0z;
  float* oxyz = a.new_xyz ? a.new_xyz + (size_t)b * a.npoint * 3 : nullptr;
  if (g == 0 && a.npoint > 0) { out[0] = 0; if (oxyz) { oxyz[0] = p0x; oxyz[1] = p0y; oxyz[2] = p0z; } }
  if (CLUSTER) { cluster_arrive_release(); cluster_wait_acquire(); }  // peers resident, mbarriers armed
  else __syncthreads();

  for (int j = 1; j < a.npoint; j++) {
    // ---- per-thread update + best: d = |p - last|^2 two points at a time (FADD2/FMUL2/FFMA2) --
    const u64 nlx = pack2(-lx, -lx), nly = pack2(-ly, -ly), nlz = pack2(-lz, -lz);
    float run[PP];  // running maximum after each pair (non-decreasing)
    float best = -1.0f;
#pragma unroll
    for (int i = 0; i < PP; i++) {
      const u64 d = dist2x2(x2[i], y2[i], z2[i], nlx, nly, nlz);
      t[2 * i] = fminf(lo2(d), t[2 * i]);
      t[2 * i + 1] = fminf(hi2(d), t[2 * i + 1]);  // padding / skipped points stay at -1
      best = max3(best, t[2 * i], t[2 * i + 1]);    // one FMNMX3 per two points
      run[i] = best;
    }
    // lowest i holding the maximum == lowest rank among this thread's ties: the first pair whose
    // running maximum already equals the final one contains it (one compare per PAIR, not per point)
    int bp = 0;
    float e0 = t[0];
#pragma unroll
    for (int i = PP - 1; i >= 0; i--)
      if (run[i] == best) { bp = i; e0 = t[2 * i]; }
    const int bi = 2 * bp + (e0 == best ? 0 : 1);
    const int tb = __float_as_int(best);
    const unsigned rk = rank0 + (unsigned)bi;
    int tbw;
    const int wl = warp_argbest(tb, rk, tbw);
    const int buf = j & 1;

    if constexpr (MODE == 0 && WARPS <= 4) {
      // Single CTA of 4 warps (8 warps: the REDUX path below measured faster): the winning lane writes the warp's entry itself (no payload broadcast), and after the
      // barrier EVERY lane folds the WARPS entries in registers — broadcast LDS.128 and WARPS-1 compares
      // instead of a second round of REDUX / ballot / shuffles on the critical path of the iteration.
      FpsEntry* ws = slots + buf * WARPS;
      if (lane == wl) {
        const int pi = bi * T + tid;
        *reinterpret_cast<int4*>(&ws[warp]) = make_int4(tbw, (int)rk, __float_as_int(px[pi]), 0);
        *reinterpret_cast<int4*>(reinterpret_cast<char*>(&ws[warp]) + 16) = make_int4(__float_as_int(py[pi]), __float_as_int(pz[pi]), pk[pi], 0);
      }
      __syncthreads();
      int4 ba = *reinterpret_cast<const int4*>(&ws[0]);
      int4 bb = *reinterpret_cast<const int4*>(reinterpret_cast<const char*>(&ws[0]) + 16);
#pragma unroll
      for (int w = 1; w < WARPS; w++) {
        const int4 ca = *reinterpret_cast<const int4*>(&ws[w]);
        const int4 cb = *reinterpret_cast<const int4*>(reinterpret_cast<const char*>(&ws[w]) + 16);
        if (fps_better(ca.x, (unsigned)ca.y, ba.x, (unsigned)ba.y)) { ba = ca; bb = cb; }
      }
      lx = __int_as_float(ba.z); ly = __int_as_float(bb.x); lz = __int_as_float(bb.y);
      int kf = bb.z;
      if (ba.x < 0) {  // no eligible point anywhere: the reference's tree returns thread 0's besti = 0
        kf = 0; lx = p0x; ly = p0y; lz = p0z;
      }
      if (g == 0) { out[j] = kf; if (oxyz) { oxyz[j * 3 + 0] = lx; oxyz[j * 3 + 1] = ly; oxyz[j * 3 + 2] = lz; } }
      continue;
    }

    // winner's payload to every lane of the warp
    float wx = 0.f, wy = 0.f, wz = 0.f;
    int wk = 0;
    if (lane == wl) { const int pi = bi * T + tid; wx = px[pi]; wy = py[pi]; wz = pz[pi]; wk = pk[pi]; }
    const unsigned s_rk = __shfl_sync(0xffffffffu, rk, wl);
    const unsigned s_x = __shfl_sync(0xffffffffu, __float_as_uint(wx), wl);
    const unsigned s_y = __shfl_sync(0xffffffffu, __float_as_uint(wy), wl);
    const unsigned s_z = __shfl_sync(0xffffffffu, __float_as_uint(wz), wl);
    const unsigned s_k = __shfl_sync(0xffffffffu, (unsigned)wk, wl);

    if (POLL) {
      // lane c stores the warp's candidate into slot (crank*WARPS+warp) of CTA c; both halves carry the tag j
      if ((unsigned)lane < C) {
        const unsigned e = crank * WARPS + warp;
        const unsigned ra = mapa_shared(smem_u32(&slots[buf * E + e]), (unsigned)lane);
        st_cluster_v4(ra, (unsigned)tbw, s_rk, s_x, (unsigned)j);
        st_cluster_v4(ra + 16, s_y, s_z, s_k, (unsigned)j);
      }
    } else if (DIRECT) {
      // lane c pushes the warp's candidate to slot (crank*WARPS+warp) of CTA c: C pushes in flight
      if ((unsigned)lane < C) {
        const unsigned e = crank * WARPS + warp;
        const unsigned ra = mapa_shared(smem_u32(&slots[buf * E + e]), (unsigned)lane);
        const unsigned rb = mapa_shared(smem_u32(&mbar[buf]), (unsigned)lane);
        st_async_v4(ra, rb, (unsigned)tbw, s_rk, s_x, 0u);
        st_async_v4(ra + 16, rb, s_y, s_z, s_k, 0u);
      }
    } else {
      FpsEntry* ws = (CLUSTER ? wslots : slots) + buf * WARPS;
      if (lane == 0) {
        FpsEntry en;
        en.tb = tbw; en.rank = s_rk; en.x = __uint_as_float(s_x); en.y = __uint_as_float(s_y);
        en.z = __uint_as_float(s_z); en.k = (int)s_k; en.pad_a = en.pad_b = 0u;
        ws[warp] = en;
      }
      __syncthreads();
      if (CLUSTER && warp == 0) {
        // warp 0 reduces the warp winners and forwards the CTA winner to every CTA
        FpsEntry en;
        en.tb = (int)0x80000000; en.rank = 0xffffffffu; en.x = en.y = en.z = 0.f; en.k = 0;
        if (lane < WARPS) en = ws[lane];
        int tbc;
        const int cl = warp_argbest(en.tb, en.rank, tbc);
        const unsigned c_rk = __shfl_sync(0xffffffffu, en.rank, cl);
        const unsigned c_x = __shfl_sync(0xffffffffu, __float_as_uint(en.x), cl);
        const unsigned c_y = __shfl_sync(0xffffffffu, __float_as_uint(en.y), cl);
        const unsigned c_z = __shfl_sync(0xffffffffu, __float_as_uint(en.z), cl);
        const unsigned c_k = __shfl_sync(0xffffffffu, (unsigned)en.k, cl);
        if ((unsigned)lane < C) {
          const unsigned ra = mapa_shared(smem_u32(&slots[buf * E + crank]), (unsigned)lane);
          const unsigned rb = mapa_shared(smem_u32(&mbar[buf]), (unsigned)lane);
          st_async_v4(ra, rb, (unsigned)tbc, c_rk, c_x, 0u);
          st_async_v4(ra + 16, rb, c_y, c_z, c_k, 0u);
        }
      }
    }
    if (CLUSTER && !POLL) {
      // buffer `buf` is used by iterations buf, buf+2, ... (buf=1: j=1,3,..; buf=0: j=2,4,..)
      const unsigned parity = (unsigned)((j - 1) >> 1) & 1u;
      while (!fps_mbar_try_wait(smem_u32(&mbar[buf]), parity)) {}
      // re-arm for iteration j+2.  Safe before our other warps have observed this phase: the next
      // phase cannot complete until they have sent their j+1 and j+2 candidates.
      if (tid == 0) fps_mbar_expect_tx(smem_u32(&mbar[buf]), (unsigned)E * 32u);
    }

    // ---- final reduce over the E candidates (identical in every warp of every CTA) --------
    const FpsEntry* sl = slots + buf * E;
    constexpr int MAXE = DIRECT ? (WARPS * 4 + 31) / 32 : 1;  // entries per lane (C <= 4 when DIRECT)
    int4 va[MAXE], vb[MAXE];
    if (POLL) {
      // lane e spins on entry e of this CTA's own slot array until both halves carry tag j.  Two buffers are
      // enough: a peer can only write iteration j+2 into this buffer after it has seen OUR iteration j+1
      // entry, which this warp sends after leaving this loop.
      int spins = 0;
      bool ok;
      do {
        ok = true;
#pragma unroll
        for (int u = 0; u < MAXE; u++) {
          const int e = lane + 32 * u;
          va[u] = make_int4((int)0x80000000, -1, 0, j);
          vb[u] = make_int4(0, 0, 0, j);
          if (e < E) {
            va[u] = ld_volatile_shared_v4(&sl[e]);
            vb[u] = ld_volatile_shared_v4(reinterpret_cast<const char*>(&sl[e]) + 16);
          }
          ok = ok && va[u].w == j && vb[u].w == j;
        }
      } while (!__all_sync(0xffffffffu, ok) && ++spins < FPS_SPIN_LIMIT);
      if (spins >= FPS_SPIN_LIMIT) __trap();  // bounded: a protocol failure aborts the launch (an error on the stream), never wrong samples or a hang
    } else {
#pragma unroll
      for (int u = 0; u < MAXE; u++) {
        const int e = lane + 32 * u;
        va[u] = make_int4((int)0x80000000, -1, 0, 0);
        vb[u] = make_int4(0, 0, 0, 0);
        if (e < E) {
          va[u] = *reinterpret_cast<const int4*>(&sl[e]);
          vb[u] = *reinterpret_cast<const int4*>(reinterpret_cast<const char*>(&sl[e]) + 16);
        }
      }
    }
#pragma unroll
    for (int u = 1; u < MAXE; u++)
      if (fps_better(va[u].x, (unsigned)va[u].y, va[0].x, (unsigned)va[0].y)) { va[0] = va[u]; vb[0] = vb[u]; }
    int tbf;
    const int fl = warp_argbest(va[0].x, (unsigned)va[0].y, tbf);
    lx = __shfl_sync(0xffffffffu, __int_as_float(va[0].z), fl);
    ly = __shfl_sync(0xffffffffu, __int_as_float(vb[0].x), fl);
    lz = __shfl_sync(0xffffffffu, __int_as_float(vb[0].y), fl);
    int kf = __shfl_sync(0xffffffffu, vb[0].z, fl);
    if (tbf < 0) {  // no eligible point anywhere: the reference's tree returns thread 0's besti = 0
      kf = 0; lx = p0x; ly = p0y; lz = p0z;
    }
    if (g == 0) { out[j] = kf; if (oxyz) { oxyz[j * 3 + 0] = lx; oxyz[j * 3 + 1] = ly; oxyz[j * 3 + 2] = lz; } }
  }
  if (CLUSTER) { cluster_arrive_release(); cluster_wait_acquire(); }  // no CTA exits while peers may still write to it
}

// ------------------------------------------------------------------------------------------------
// Lean exchange for small clusters (2-4 CTAs, N <= 16384): fps_kernel MODE 1 with 8-byte messages.
//
// In MODE 1 a warp's candidate travels with its coordinates (32 bytes, two st.async.v4 per destination, five payload
// shuffles before, two LDS.128 + four shuffles after the final reduce), because a CTA only holds its own points.  A
// 16384-point cloud is 192 KB: every CTA of the cluster can hold ALL of it in shared memory, ordered by rank — then a
// candidate is just (distance bits, rank), one st.async.v2 per destination, and the winner's coordinates are a local
// broadcast load.  Same protocol otherwise (two slot buffers, byte-counting mbarrier on the destination, every warp
// reduces the E candidates redundantly), same dealing of ranks to threads, same selection order.
__device__ __forceinline__ void st_async_v2(unsigned raddr, unsigned rbar, unsigned a, unsigned b) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v2.b32 [%0], {%1, %2}, [%3];"
               ::"r"(raddr), "r"(a), "r"(b), "r"(rbar) : "memory");
}

template <int PP, int T>
__global__ void __launch_bounds__(T, 1) fps_lean_kernel(const FpsArgs a, int Rpad) {
  constexpr int P = 2 * PP;
  constexpr int WARPS = T / 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* ax = reinterpret_cast<float*>(smem_raw);  // the whole cloud by rank
  float* ay = ax + Rpad;
  float* az = ay + Rpad;
  u64* mbar = reinterpret_cast<u64*>(az + Rpad);
  int2* slots = reinterpret_cast<int2*>(mbar + 2);  // [2][E]
  const unsigned C = cluster_nctarank();
  const unsigned crank = cluster_ctarank();
  const int b = (int)cluster_id_x();
  if (a.run_flag && __ldg(a.run_flag + b) == 0) return;  // the whole cluster leaves together: nothing was armed yet
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int E = WARPS * (int)C;
  const int N = a.N;
  const float* cloud = a.xyz + (size_t)b * N * 3;
  int* out = a.idx + (size_t)b * a.npoint;
  float* oxyz = a.new_xyz ? a.new_xyz + (size_t)b * a.npoint * 3 : nullptr;
  const int g = (int)crank * T + tid;
  const unsigned rank0 = (unsigned)g * P;
  const unsigned R = (unsigned)a.nper << a.L;

  for (unsigned r = tid; r < (unsigned)Rpad; r += T) {
    float xv = 0.f, yv = 0.f, zv = 0.f;
    if (r < R) {
      const int k = fps_rank_to_k(r, a.L, a.nper);
      if (k < N) { xv = __ldg(cloud + (size_t)k * 3 + 0); yv = __ldg(cloud + (size_t)k * 3 + 1); zv = __ldg(cloud + (size_t)k * 3 + 2); }
    }
    ax[r] = xv; ay[r] = yv; az[r] = zv;
  }
  if (tid == 0) {
    fps_mbar_init(smem_u32(&mbar[0]), 1);
    fps_mbar_init(smem_u32(&mbar[1]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    fps_mbar_expect_tx(smem_u32(&mbar[0]), (unsigned)E * 8u);
    fps_mbar_expect_tx(smem_u32(&mbar[1]), (unsigned)E * 8u);
  }
  __syncthreads();
  u64 x2[PP], y2[PP], z2[PP];
  float t[P];
#pragma unroll
  for (int i = 0; i < P; i++) {
    const unsigned r = rank0 + i;
    float xv = 0.f, yv = 0.f, zv = 0.f;
    t[i] = -1.0f;
    if (r < R && fps_rank_to_k(r, a.L, a.nper) < N) {
      xv = ax[r]; yv = ay[r]; zv = az[r];
      t[i] = ((double)dist2_ref(xv, yv, zv) <= 1e-3) ? -1.0f : 1e10f;
    }
    if (i & 1) {
      x2[i / 2] = pack2(lo2(x2[i / 2]), xv); y2[i / 2] = pack2(lo2(y2[i / 2]), yv); z2[i / 2] = pack2(lo2(z2[i / 2]), zv);
    } else {
      x2[i / 2] = pack2(xv, 0.f); y2[i / 2] = pack2(yv, 0.f); z2[i / 2] = pack2(zv, 0.f);
    }
  }
  const float p0x = __ldg(cloud + 0), p0y = __ldg(cloud + 1), p0z = __ldg(cloud + 2);
  float lx = p0x, ly = p0y, lz = p0z;
  if (g == 0 && a.npoint > 0) out[0] = 0;
  cluster_arrive_release(); cluster_wait_acquire();  // peers resident, mbarriers armed
  // lane c pushes the warp's candidate to slot (crank*WARPS+warp) of CTA c: the remote addresses of both buffers are
  // loop constants
  unsigned ra[2] = {0u, 0u}, rb[2] = {0u, 0u};
  if ((unsigned)lane < C) {
    const unsigned e = crank * WARPS + warp;
#pragma unroll
    for (int u = 0; u < 2; u++) {
      ra[u] = mapa_shared(smem_u32(&slots[u * E + e]), (unsigned)lane);
      rb[u] = mapa_shared(smem_u32(&mbar[u]), (unsigned)lane);
    }
  }

  for (int j = 1; j < a.npoint; j++) {
    const u64 nlx = pack2(-lx, -lx), nly = pack2(-ly, -ly), nlz = pack2(-lz, -lz);
    float run[PP];
    float best = -1.0f;
#pragma unroll
    for (int i = 0; i < PP; i++) {
      const u64 d = dist2x2(x2[i], y2[i], z2[i], nlx, nly, nlz);
      t[2 * i] = fminf(lo2(d), t[2 * i]);
      t[2 * i + 1] = fminf(hi2(d), t[2 * i + 1]);  // padding / skipped points stay at -1
      best = max3(best, t[2 * i], t[2 * i + 1]);
      run[i] = best;
    }
    int bp = 0;
    float e0 = t[0];
#pragma unroll
    for (int i = PP - 1; i >= 0; i--)
      if (run[i] == best) { bp = i; e0 = t[2 * i]; }
    const unsigned rk = rank0 + (unsigned)(2 * bp + (e0 == best ? 0 : 1));
    const int tb = __float_as_int(best);
    const int wm = __reduce_max_sync(0xffffffffu, tb);
    const unsigned wk = __reduce_min_sync(0xffffffffu, tb == wm ? rk : 0xffffffffu);
    const int buf = j & 1;
    // (selects, not ra[buf]: a dynamically indexed register array lives in local memory, and its two loads sat in
    // front of the remote store in every iteration)
    if ((unsigned)lane < C) st_async_v2(buf ? ra[1] : ra[0], buf ? rb[1] : rb[0], (unsigned)wm, wk);
    const unsigned parity = (unsigned)((j - 1) >> 1) & 1u;
    while (!fps_mbar_try_wait(smem_u32(&mbar[buf]), parity)) {}
    if (tid == 0) fps_mbar_expect_tx(smem_u32(&mbar[buf]), (unsigned)E * 8u);  // re-arm for iteration j + 2 (see fps_kernel)
    int2 sv = lane < E ? slots[buf * E + lane] : make_int2((int)0x80000000, -1);
    if (E > 32) {  // 16 CTAs of 128 threads: two candidates per lane
      const int2 s2 = lane + 32 < E ? slots[buf * E + 32 + lane] : make_int2((int)0x80000000, -1);
      if (fps_better(s2.x, (unsigned)s2.y, sv.x, (unsigned)sv.y)) sv = s2;
    }
    const int gm = __reduce_max_sync(0xffffffffu, sv.x);
    unsigned gk = __reduce_min_sync(0xffffffffu, sv.x == gm ? (unsigned)sv.y : 0xffffffffu);
    if (gm < 0) {  // no eligible point anywhere: the reference's tree returns thread 0's besti = 0
      gk = 0xffffffffu;
      lx = p0x; ly = p0y; lz = p0z;
    } else {
      lx = ax[gk]; ly = ay[gk]; lz = az[gk];
    }
    if (g == 0) out[j] = (int)gk;  // raw rank; turned into the point index after the loop
  }
  cluster_arrive_release(); cluster_wait_acquire();  // no CTA exits while peers may still write to it
  if (crank == 0) {
    __syncthreads();
    for (int j = tid; j < a.npoint; j += T) {
      const unsigned gk = j ? (unsigned)out[j] : 0u;
      int k = 0;
      float ox = p0x, oy = p0y, oz = p0z;
      if (j && gk != 0xffffffffu) { k = fps_rank_to_k(gk, a.L, a.nper); ox = ax[gk]; oy = ay[gk]; oz = az[gk]; }
      out[j] = k;
      if (oxyz) { oxyz[j * 3 + 0] = ox; oxyz[j * 3 + 1] = oy; oxyz[j * 3 + 2] = oz; }
    }
  }
}

template <int PP, int T>
static int launch_fps_lean(const FpsArgs& a, int B, int C, cudaStream_t stream) {
  const int R = a.nper << a.L;
  const int Rpad = (R + 3) & ~3;
  const int E = (T / 32) * C;
  const size_t smem = (size_t)3 * Rpad * sizeof(float) + 16 + (size_t)2 * E * sizeof(int2);
  auto kern = fps_lean_kernel<PP, T>;
  PS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (C > 8) PS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(B * C);
  cfg.blockDim = dim3(T);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = C;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  PS_CUDA(cudaLaunchKernelEx(&cfg, kern, a, Rpad));
  PS_LAUNCH_CHECK();
  return PS_OK;
}

template <int T>
static int dispatch_lean(int PP, const FpsArgs& a, int B, int C, cudaStream_t s) {
  switch (PP) {
    case 1: return launch_fps_lean<1, T>(a, B, C, s);
    case 2: return launch_fps_lean<2, T>(a, B, C, s);
    case 4: return launch_fps_lean<4, T>(a, B, C, s);
    case 8: return launch_fps_lean<8, T>(a, B, C, s);
    case 16: return launch_fps_lean<16, T>(a, B, C, s);
  }
  return set_error(PS_ERR_UNSUPPORTED, "ps_fps: no kernel for %d point pairs per thread", PP);
}

// ------------------------------------------------------------------------------------------------
// Small clouds (N <= 4096: the FPS calls inside the models — 2048 -> 512, 512 -> 128, sample_and_group_knn): ONE CTA
// of T = 128 .. 512 threads per cloud with a lean arg-max.  fps_kernel<PP,T,0> pays ~565-725 cycles per iteration before
// any distance work (two REDUX + ballot, five payload shuffles, a 32-byte entry per warp, a second round of the same
// after the barrier); here a warp publishes only (distance bits, rank) — 8 bytes — and the winner's coordinates are
// looked up in the CTA's own shared-memory copy of the cloud by its rank, as fps_pruned_kernel does: two REDUX, one
// store, one barrier, one load, two REDUX, three broadcast loads.  Same dealing of points to threads in rank order,
// same selection (distance desc, rank asc), same -1 convention for skipped / padding points as fps_kernel.
template <int PP, int T, bool RAGGED = false>
__global__ void __launch_bounds__(T, 1) fps_small_kernel(const FpsArgs a) {
  constexpr int P = 2 * PP;
  constexpr int WARPS = T / 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* px = reinterpret_cast<float*>(smem_raw);  // [P][T]: point i of thread t at i * T + t
  float* py = px + P * T;
  float* pz = py + P * T;
  __shared__ int2 slots[2][WARPS];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (a.run_flag && __ldg(a.run_flag + b) == 0) return;
  int N = a.N, L = a.L, nper = a.nper;
  const float* cloud = a.xyz + (size_t)b * N * 3;
  if constexpr (RAGGED) {
    const int4 pt = a.part[b];
    N = pt.x; L = pt.y; nper = pt.z;
    cloud = a.xyz + (size_t)b * a.stride * 3;
  }
  int* out = a.idx + (size_t)b * a.npoint;
  float* oxyz = a.new_xyz ? a.new_xyz + (size_t)b * a.npoint * 3 : nullptr;
  const unsigned rank0 = (unsigned)tid * P;  // this thread owns ranks [rank0, rank0 + P)
  const unsigned R = (unsigned)nper << L;

  u64 x2[PP], y2[PP], z2[PP];
  float t[P];
#pragma unroll
  for (int i = 0; i < P; i++) {
    float xv = 0.f, yv = 0.f, zv = 0.f;
    t[i] = -1.0f;
    if (rank0 + i < R) {
      const int k = fps_rank_to_k(rank0 + i, L, nper);
      if (k < N) {
        xv = __ldg(cloud + (size_t)k * 3 + 0);
        yv = __ldg(cloud + (size_t)k * 3 + 1);
        zv = __ldg(cloud + (size_t)k * 3 + 2);
        t[i] = ((double)dist2_ref(xv, yv, zv) <= 1e-3) ? -1.0f : 1e10f;
      }
    }
    px[i * T + tid] = xv; py[i * T + tid] = yv; pz[i * T + tid] = zv;
    if (i & 1) {
      x2[i / 2] = pack2(lo2(x2[i / 2]), xv); y2[i / 2] = pack2(lo2(y2[i / 2]), yv); z2[i / 2] = pack2(lo2(z2[i / 2]), zv);
    } else {
      x2[i / 2] = pack2(xv, 0.f); y2[i / 2] = pack2(yv, 0.f); z2[i / 2] = pack2(zv, 0.f);
    }
  }
  const float p0x = __ldg(cloud + 0), p0y = __ldg(cloud + 1), p0z = __ldg(cloud + 2);
  float lx = p0x, ly = p0y, lz = p0z;
  if (tid == 0 && a.npoint > 0) out[0] = 0;
  __syncthreads();

  for (int j = 1; j < a.npoint; j++) {
    const u64 nlx = pack2(-lx, -lx), nly = pack2(-ly, -ly), nlz = pack2(-lz, -lz);
    float run[PP];
    float best = -1.0f;
#pragma unroll
    for (int i = 0; i < PP; i++) {
      const u64 d = dist2x2(x2[i], y2[i], z2[i], nlx, nly, nlz);
      t[2 * i] = fminf(lo2(d), t[2 * i]);
      t[2 * i + 1] = fminf(hi2(d), t[2 * i + 1]);  // padding / skipped points stay at -1
      best = max3(best, t[2 * i], t[2 * i + 1]);
      run[i] = best;
    }
    int bp = 0;
    float e0 = t[0];
#pragma unroll
    for (int i = PP - 1; i >= 0; i--)
      if (run[i] == best) { bp = i; e0 = t[2 * i]; }
    const unsigned rk = rank0 + (unsigned)(2 * bp + (e0 == best ? 0 : 1));
    const int tb = __float_as_int(best);
    const int wm = __reduce_max_sync(0xffffffffu, tb);
    const unsigned wk = __reduce_min_sync(0xffffffffu, tb == wm ? rk : 0xffffffffu);
    const int buf = j & 1;
    if (lane == 0) slots[buf][warp] = make_int2(wm, (int)wk);
    __syncthreads();
    const int2 sv = lane < WARPS ? slots[buf][lane] : make_int2((int)0x80000000, -1);
    const int gm = __reduce_max_sync(0xffffffffu, sv.x);
    unsigned gk = __reduce_min_sync(0xffffffffu, sv.x == gm ? (unsigned)sv.y : 0xffffffffu);
    if (gm < 0) {  // no eligible point anywhere: the reference's tree returns thread 0's besti = 0
      gk = 0xffffffffu;
      lx = p0x; ly = p0y; lz = p0z;
    } else {
      const unsigned wt = gk / (unsigned)P, wi = gk % (unsigned)P;
      lx = px[wi * T + wt]; ly = py[wi * T + wt]; lz = pz[wi * T + wt];
    }
    if (tid == 0) out[j] = (int)gk;  // raw rank; turned into the point index after the loop
  }
  __syncthreads();
  for (int j = tid; j < a.npoint; j += T) {
    const unsigned gk = j ? (unsigned)out[j] : 0u;
    int k = 0;
    float ox = p0x, oy = p0y, oz = p0z;
    if (j && gk != 0xffffffffu) {
      k = fps_rank_to_k(gk, L, nper);
      const unsigned wt = gk / (unsigned)P, wi = gk % (unsigned)P;
      ox = px[wi * T + wt]; oy = py[wi * T + wt]; oz = pz[wi * T + wt];
    }
    out[j] = k;
    if (oxyz) { oxyz[j * 3 + 0] = ox; oxyz[j * 3 + 1] = oy; oxyz[j * 3 + 2] = oz; }
  }
}

template <int PP, int T, bool RAGGED = false>
static int launch_fps_small(const FpsArgs& a, int B, cudaStream_t stream) {
  const size_t smem = (size_t)3 * 2 * PP * T * sizeof(float);
  auto kern = fps_small_kernel<PP, T, RAGGED>;
  if (smem + 1024 > 48 * 1024) PS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));  // + static slots
  kern<<<B, T, smem, stream>>>(a);
  PS_LAUNCH_CHECK();
  return PS_OK;
}

// Generic fallback for clouds too large for the register-resident kernel: one CTA per cloud,
// running min distances in a global scratch array (still the exact reference order).
constexpr int FPS_GT = 512;
__device__ __forceinline__ unsigned fps_k_to_rank(int k, int L, int nper) {
  const unsigned low = (unsigned)k & ((1u << L) - 1u);
  const unsigned rev = L ? (__brev(low) >> (32 - L)) : 0u;
  return rev * (unsigned)nper + ((unsigned)k >> L);
}
__global__ void __launch_bounds__(FPS_GT, 1) fps_generic_kernel(const FpsArgs a, float* temp_all) {
  constexpr int WARPS = FPS_GT / 32;
  __shared__ FpsEntry ws[2][WARPS];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = a.N;
  const float* cloud = a.xyz + (size_t)b * N * 3;
  float* temp = temp_all + (size_t)b * N;
  int* out = a.idx + (size_t)b * a.npoint;
  for (int k = tid; k < N; k += FPS_GT) {
    const float mag = dist2_ref(cloud[k * 3 + 0], cloud[k * 3 + 1], cloud[k * 3 + 2]);
    temp[k] = ((double)mag <= 1e-3) ? -1.0f : 1e10f;
  }
  float lx = cloud[0], ly = cloud[1], lz = cloud[2];
  float* oxyz = a.new_xyz ? a.new_xyz + (size_t)b * a.npoint * 3 : nullptr;
  if (tid == 0 && a.npoint > 0) { out[0] = 0; if (oxyz) { oxyz[0] = lx; oxyz[1] = ly; oxyz[2] = lz; } }
  __syncthreads();
  for (int j = 1; j < a.npoint; j++) {
    // stride FPS_GT is a multiple of bs, so k mod bs is constant per thread and the first maximum
    // in k order is the lowest rank
    float best = -1.0f;
    int bk = tid < N ? tid : 0;
    for (int k = tid; k < N; k += FPS_GT) {
      const float d = dist2_ref(cloud[k * 3 + 0] - lx, cloud[k * 3 + 1] - ly, cloud[k * 3 + 2] - lz);
      const float t = fminf(d, temp[k]);
      temp[k] = t;
      if (t > best) { best = t; bk = k; }
    }
    int tbw;
    const unsigned rk = fps_k_to_rank(bk, a.L, a.nper);
    const int wl = warp_argbest(__float_as_int(best), rk, tbw);
    const int buf = j & 1;
    if (lane == wl) {
      FpsEntry en;
      en.tb = __float_as_int(best); en.rank = rk; en.k = bk;
      en.x = cloud[bk * 3 + 0]; en.y = cloud[bk * 3 + 1]; en.z = cloud[bk * 3 + 2];
      en.pad_a = en.pad_b = 0u;
      ws[buf][warp] = en;
    }
    __syncthreads();
    FpsEntry en;
    en.tb = (int)0x80000000; en.rank = 0xffffffffu; en.x = en.y = en.z = 0.f; en.k = 0;
    if (lane < WARPS) en = ws[buf][lane];
    int tbf;
    const int fl = warp_argbest(en.tb, en.rank, tbf);
    lx = __shfl_sync(0xffffffffu, en.x, fl);
    ly = __shfl_sync(0xffffffffu, en.y, fl);
    lz = __shfl_sync(0xffffffffu, en.z, fl);
    int kf = __shfl_sync(0xffffffffu, en.k, fl);
    if (tbf < 0) { kf = 0; lx = cloud[0]; ly = cloud[1]; lz = cloud[2]; }
    if (tid == 0) { out[j] = kf; if (oxyz) { oxyz[j * 3 + 0] = lx; oxyz[j * 3 + 1] = ly; oxyz[j * 3 + 2] = lz; } }
  }
}

// ------------------------------------------------------------------------------------------------
// Bucket-pruned FPS: ONE CTA per cloud, no cluster exchange, same samples bit for bit.
//
// An iteration of the register-resident kernel above is ~270 cycles of distance updates plus ~800 cycles of
// cluster-wide exchange (DESIGN.md 4.3): the exchange cannot shrink, so the way out is to need no cluster.  What
// forces four SMs per 16384-point cloud is the full update of every running minimum each iteration — yet a new
// sample only lowers the minima of points closer to it than to every earlier sample, a handful after the first few
// dozen iterations.  Here the points are sorted into BUCKETS of 32 spatial neighbours (counting sort by the Morton
// index of a 16^3 grid over the cloud's bounding box), coordinates live in shared memory (192 KB for 16384 points),
// the running minima in registers (lane l of a warp holds point l of each of the warp's FP_RPW buckets), and lane s
// also keeps bucket s's bounding box, its maximum running minimum and the (rank, position) of that maximum.  Per
// iteration every warp tests its buckets against the new sample — a bucket whose box is farther away than its
// largest running minimum cannot change (fminf(d, t) == t for all its points; the bound carries a 2^-20 safety
// margin over the rounding of both sides) — and only the AFFECTED buckets are updated (32 lanes = 32 points, two
// REDUX for the bucket's new maximum).  The arg-max is then bucket maxima -> warp (two REDUX) -> 16 slots in shared
// memory -> one __syncthreads -> every warp folds the 16 slots.  Buckets are dealt to warps round-robin so that the
// few affected buckets of an iteration (spatial neighbours) land in different warps.
// Selection order is unchanged: (running minimum desc, reference tie-break rank asc); skipped points (|p|^2 <= 1e-3)
// are left out of the buckets altogether; the winner's index comes back from its rank (fps_rank_to_k).
// Pruning cannot change a result, only the time: a cloud on which it does not bite (e.g. all points in one grid cell
// next to a far outlier) is detected at iteration FP_CHECK by the number of bucket updates so far and handed to the
// cluster kernel through run_flag (launched right behind, it returns at once for the clouds already done).
constexpr int FP_MAXN = 16384;                      // 512 buckets: FP_RPW per warp, 512 / FP_RPW warps
constexpr int FP_G = 16, FP_CELLS = FP_G * FP_G * FP_G;
constexpr int FP_CHECK = 192;                       // iteration at which the pruning rate is judged

__device__ __forceinline__ unsigned fp_spread4(unsigned v) { return (v & 1u) | ((v & 2u) << 2) | ((v & 4u) << 4) | ((v & 8u) << 6); }
// order-preserving map float -> unsigned (for REDUX min / max over floats of either sign)
__device__ __forceinline__ unsigned fp_ord(float f) { const unsigned u = __float_as_uint(f); return (u & 0x80000000u) ? ~u : (u | 0x80000000u); }
__device__ __forceinline__ float fp_unord(unsigned k) { return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k); }

struct FpsPruneArgs {
  unsigned short* inv;  // (B, FP_MAXN) scratch: sorted position -> point index
  int* flag;            // (B): 0 = sampled here, 1 = hand the cloud to the cluster kernel
  int check;            // 0: never give up (forced)
  int max_updates;      // bucket updates allowed in the first FP_CHECK iterations
};

// FP_RPW: buckets per warp (16: 32 warps, 32: 16 warps); lane s < FP_RPW owns bucket s's box and maximum.
// DISPATCH: how a warp reaches the code of an affected bucket (its running minima sit in registers, so every bucket
// has its own copy of the update): 0 = one uniform test per bucket, 1 = jump table over the set bits of the mask,
// 2 = no updates at all (timing of the arg-max skeleton only; results are wrong).
// Measured (B200, B = 32, 16384 -> 2048, us per iteration; profiles/fps_pruned_r2.jsonl): skeleton 0.244 (16 warps) /
// 0.351 (32 warps); with updates 0.835 (16 warps, jump table), 0.897 (tests), 0.809 / 0.784 (32 warps) on a uniform
// cube, 0.586 on a sphere surface — against 0.546 for the 4-CTA cluster kernel.  A CPU simulation of the same
// pruning (uniform cube) counts 18 affected buckets per iteration and 2.6 on the busiest warp: each bucket update
// costs ~400 cycles of single-warp latency (bit scan + branch tree + LDC/BRX ~150, LDS + distance + two dependent
// REDUX ~250), so the critical path is 480 + 2.6 x 400 cycles and the kernel only wins on THROUGHPUT (148 clouds:
// 1.68 ms against 2.95 ms), which is where the launcher uses it.
template <int FP_RPW, int DISPATCH>
__global__ void __launch_bounds__(512 / FP_RPW * 32, 1) fps_pruned_kernel(const FpsArgs a, const FpsPruneArgs q) {
  constexpr int FP_WARPS = 512 / FP_RPW;
  constexpr int FP_T = FP_WARPS * 32;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sx = reinterpret_cast<float*>(smem_raw);
  float* sy = sx + FP_MAXN;
  float* sz = sy + FP_MAXN;
  int* cnt = reinterpret_cast<int*>(sz + FP_MAXN);  // FP_CELLS counters / cursors
  __shared__ unsigned red[6][FP_WARPS];
  __shared__ int wtot[FP_WARPS];
  __shared__ int2 slots[2][FP_WARPS];
  __shared__ int aff_total;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int N = a.N;
  const float* cloud = a.xyz + (size_t)b * N * 3;
  int* out = a.idx + (size_t)b * a.npoint;
  float* oxyz = a.new_xyz ? a.new_xyz + (size_t)b * a.npoint * 3 : nullptr;
  unsigned short* inv = q.inv + (size_t)b * FP_MAXN;
  const float INF = __int_as_float(0x7f800000);

  // ---- bounding box of the eligible points -------------------------------------------------------
  unsigned bb[6] = {0xffffffffu, 0xffffffffu, 0xffffffffu, 0u, 0u, 0u};  // ordered keys: min x,y,z / max x,y,z
  for (int k = tid; k < N; k += FP_T) {
    const float x = __ldg(cloud + (size_t)k * 3 + 0), y = __ldg(cloud + (size_t)k * 3 + 1), z = __ldg(cloud + (size_t)k * 3 + 2);
    if ((double)dist2_ref(x, y, z) <= 1e-3) continue;
    const unsigned kx = fp_ord(x), ky = fp_ord(y), kz = fp_ord(z);
    bb[0] = min(bb[0], kx); bb[1] = min(bb[1], ky); bb[2] = min(bb[2], kz);
    bb[3] = max(bb[3], kx); bb[4] = max(bb[4], ky); bb[5] = max(bb[5], kz);
  }
#pragma unroll
  for (int i = 0; i < 6; i++) {
    const unsigned v = i < 3 ? __reduce_min_sync(0xffffffffu, bb[i]) : __reduce_max_sync(0xffffffffu, bb[i]);
    if (lane == 0) red[i][warp] = v;
  }
  for (int c = tid; c < FP_CELLS; c += FP_T) cnt[c] = 0;
  if (tid == 0) aff_total = 0;
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 6; i++) {
    const unsigned v = lane < FP_WARPS ? red[i][lane] : (i < 3 ? 0xffffffffu : 0u);
    bb[i] = i < 3 ? __reduce_min_sync(0xffffffffu, v) : __reduce_max_sync(0xffffffffu, v);
  }
  const float p0x = __ldg(cloud + 0), p0y = __ldg(cloud + 1), p0z = __ldg(cloud + 2);
  if (bb[3] == 0u) {
    // no eligible point at all: the reference's tree returns thread 0's initial besti = 0 every time
    for (int j = tid; j < a.npoint; j += FP_T) { out[j] = 0; if (oxyz) { oxyz[j * 3 + 0] = p0x; oxyz[j * 3 + 1] = p0y; oxyz[j * 3 + 2] = p0z; } }
    if (tid == 0) q.flag[b] = 0;
    return;
  }
  const float lox = fp_unord(bb[0]), loy = fp_unord(bb[1]), loz = fp_unord(bb[2]);
  const float ex = fp_unord(bb[3]) - lox, ey = fp_unord(bb[4]) - loy, ez = fp_unord(bb[5]) - loz;
  const float gx = ex > 0.f ? (float)FP_G / ex : 0.f, gy = ey > 0.f ? (float)FP_G / ey : 0.f, gz = ez > 0.f ? (float)FP_G / ez : 0.f;
  auto cell_of = [&](float x, float y, float z) {
    const unsigned cx = min((unsigned)FP_G - 1u, (unsigned)max(0, (int)((x - lox) * gx)));
    const unsigned cy = min((unsigned)FP_G - 1u, (unsigned)max(0, (int)((y - loy) * gy)));
    const unsigned cz = min((unsigned)FP_G - 1u, (unsigned)max(0, (int)((z - loz) * gz)));
    return (int)(fp_spread4(cx) | (fp_spread4(cy) << 1) | (fp_spread4(cz) << 2));
  };

  // ---- counting sort by grid cell (Morton order of the cells) ------------------------------------
  for (int k = tid; k < N; k += FP_T) {
    const float x = __ldg(cloud + (size_t)k * 3 + 0), y = __ldg(cloud + (size_t)k * 3 + 1), z = __ldg(cloud + (size_t)k * 3 + 2);
    if ((double)dist2_ref(x, y, z) <= 1e-3) continue;
    atomicAdd(&cnt[cell_of(x, y, z)], 1);
  }
  __syncthreads();
  {
    constexpr int PER = FP_CELLS / FP_T;  // 8 consecutive counters per thread
    int v[PER], run = 0;
#pragma unroll
    for (int i = 0; i < PER; i++) { v[i] = cnt[tid * PER + i]; run += v[i]; }
    int incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
    if (lane == 31) wtot[warp] = incl;
    __syncthreads();
    int wbase = 0;
    for (int w = 0; w < warp; w++) wbase += wtot[w];
    int base = wbase + incl - run;
#pragma unroll
    for (int i = 0; i < PER; i++) { cnt[tid * PER + i] = base; base += v[i]; }
  }
  int nvalid = 0;
  for (int w = 0; w < FP_WARPS; w++) nvalid += wtot[w];
  __syncthreads();
  for (int k = tid; k < N; k += FP_T) {
    const float x = __ldg(cloud + (size_t)k * 3 + 0), y = __ldg(cloud + (size_t)k * 3 + 1), z = __ldg(cloud + (size_t)k * 3 + 2);
    if ((double)dist2_ref(x, y, z) <= 1e-3) continue;
    const int pos = atomicAdd(&cnt[cell_of(x, y, z)], 1);
    sx[pos] = x; sy[pos] = y; sz[pos] = z;
    inv[pos] = (unsigned short)k;
  }
  __syncthreads();  // also orders this block's writes to `inv` before its reads below

  // ---- per-lane state: running minima, ranks; per-bucket state in lane s ---------------------------
  float t[FP_RPW];
  unsigned rk2[FP_RPW / 2];
  float blx = INF, bly = INF, blz = INF, bhx = -INF, bhy = -INF, bhz = -INF;
  int bmax = (int)0x80000000;   // bits of the bucket's largest running minimum (signed compare), none: INT_MIN
  unsigned bkey = 0xffffffffu;  // (rank << 14 | position) of that maximum, lowest rank among equals
#pragma unroll
  for (int s = 0; s < FP_RPW; s++) {
    const int pos = (s * FP_WARPS + warp) * 32 + lane;
    const bool valid = pos < nvalid;
    unsigned rank = 0x3fffu;
    float x = 0.f, y = 0.f, z = 0.f;
    if (valid) { rank = fps_k_to_rank((int)inv[pos], a.L, a.nper); x = sx[pos]; y = sy[pos]; z = sz[pos]; }
    t[s] = valid ? 1e10f : -1.0f;
    if (s & 1) rk2[s / 2] |= rank << 16; else rk2[s / 2] = rank;
    const unsigned any = __ballot_sync(0xffffffffu, valid);
    const unsigned nx = __reduce_min_sync(0xffffffffu, valid ? fp_ord(x) : 0xffffffffu), ny = __reduce_min_sync(0xffffffffu, valid ? fp_ord(y) : 0xffffffffu);
    const unsigned nz = __reduce_min_sync(0xffffffffu, valid ? fp_ord(z) : 0xffffffffu), mx = __reduce_max_sync(0xffffffffu, valid ? fp_ord(x) : 0u);
    const unsigned my = __reduce_max_sync(0xffffffffu, valid ? fp_ord(y) : 0u), mz = __reduce_max_sync(0xffffffffu, valid ? fp_ord(z) : 0u);
    if (lane == s && any) {
      blx = fp_unord(nx); bly = fp_unord(ny); blz = fp_unord(nz); bhx = fp_unord(mx); bhy = fp_unord(my); bhz = fp_unord(mz);
      bmax = __float_as_int(1e10f);  // every non-empty bucket is updated in the first iteration, which also sets bkey
    }
  }

  float lx = p0x, ly = p0y, lz = p0z;
  if (tid == 0 && a.npoint > 0) { out[0] = 0; if (oxyz) { oxyz[0] = p0x; oxyz[1] = p0y; oxyz[2] = p0z; } }
  int updates = 0;
  const float SHRINK = 1.0f - 9.5367431640625e-07f;  // 1 - 2^-20

  for (int j = 1; j < a.npoint; j++) {
    // ---- which of this warp's buckets can change: box distance (a lower bound) vs largest running minimum ----
    const float dx = fmaxf(fmaxf(blx - lx, lx - bhx), 0.f), dy = fmaxf(fmaxf(bly - ly, ly - bhy), 0.f), dz = fmaxf(fmaxf(blz - lz, lz - bhz), 0.f);
    const float lb = (dx * dx + dy * dy + dz * dz) * SHRINK;
    unsigned mask = __ballot_sync(0xffffffffu, bmax >= 0 && !(lb > __int_as_float(bmax)));
    updates += __popc(mask);
    auto row = [&](const int s, float& ts) {  // s is a literal at every call site
      const int pos = (s * FP_WARPS + warp) * 32 + lane;
      const float d = dist2_ref(sx[pos] - lx, sy[pos] - ly, sz[pos] - lz);
      const float tv = ts < 0.f ? ts : fminf(d, ts);  // padding lanes stay at -1
      ts = tv;
      const int tb = __float_as_int(tv);
      const int m = __reduce_max_sync(0xffffffffu, tb);
      const unsigned rank = (s & 1) ? (rk2[s / 2] >> 16) : (rk2[s / 2] & 0xffffu);
      const unsigned key = tb == m ? ((rank << 14) | (unsigned)pos) : 0xffffffffu;
      const unsigned kmin = __reduce_min_sync(0xffffffffu, key);
      if (lane == s) { bmax = m; bkey = kmin; }
    };
    if (DISPATCH == 0) {
      if (mask) {
#pragma unroll
        for (int s = 0; s < FP_RPW; s++)
          if (mask & (1u << s)) row(s, t[s]);  // warp-uniform
      }
    } else if (DISPATCH == 1) {
      while (mask) {
        const int s = __ffs(mask) - 1;
        mask &= mask - 1;
#define FP_CASE(S) case S: if (S < FP_RPW) row(S, t[S < FP_RPW ? S : 0]); break;
        switch (s) {
          FP_CASE(0) FP_CASE(1) FP_CASE(2) FP_CASE(3) FP_CASE(4) FP_CASE(5) FP_CASE(6) FP_CASE(7)
          FP_CASE(8) FP_CASE(9) FP_CASE(10) FP_CASE(11) FP_CASE(12) FP_CASE(13) FP_CASE(14) FP_CASE(15)
          FP_CASE(16) FP_CASE(17) FP_CASE(18) FP_CASE(19) FP_CASE(20) FP_CASE(21) FP_CASE(22) FP_CASE(23)
          FP_CASE(24) FP_CASE(25) FP_CASE(26) FP_CASE(27) FP_CASE(28) FP_CASE(29) FP_CASE(30) FP_CASE(31)
        }
#undef FP_CASE
      }
    }
    // ---- arg-max: buckets -> warp -> block ----------------------------------------------------------
    const int wm = __reduce_max_sync(0xffffffffu, bmax);
    const unsigned wk = __reduce_min_sync(0xffffffffu, bmax == wm ? bkey : 0xffffffffu);
    const int buf = j & 1;
    if (lane == 0) {
      slots[buf][warp] = make_int2(wm, (int)wk);
      if (q.check && j == FP_CHECK) atomicAdd(&aff_total, updates);
    }
    __syncthreads();
    const int2 sv = lane < FP_WARPS ? slots[buf][lane] : make_int2((int)0x80000000, -1);
    const int gm = __reduce_max_sync(0xffffffffu, sv.x);
    const unsigned gk = __reduce_min_sync(0xffffffffu, sv.x == gm ? (unsigned)sv.y : 0xffffffffu);
    const int wpos = (int)(gk & 0x3fffu);
    lx = sx[wpos]; ly = sy[wpos]; lz = sz[wpos];
    if (tid == 0) out[j] = (int)gk;  // raw (rank, position); turned into the point index after the loop (off the critical path)
    if (q.check && j == FP_CHECK) {
      if (aff_total > q.max_updates) {  // uniform: no warp adds after this barrier
        if (tid == 0) q.flag[b] = 1;
        return;
      }
    }
  }
  __syncthreads();  // thread 0's writes to out[] are visible to the block
  for (int j = 1 + tid; j < a.npoint; j += FP_T) {
    const unsigned gk = (unsigned)out[j];
    out[j] = fps_rank_to_k(gk >> 14, a.L, a.nper);
    if (oxyz) { const int wpos = (int)(gk & 0x3fffu); oxyz[j * 3 + 0] = sx[wpos]; oxyz[j * 3 + 1] = sy[wpos]; oxyz[j * 3 + 2] = sz[wpos]; }
  }
  if (tid == 0) q.flag[b] = 0;
}

// opt_n_threads of the reference (include/cuda_utils.h:15-19), evaluated the same way
// (double log ratio truncated) so bs matches even where the quotient is inexact.
static int ref_block_log2(int n) {
  const int pow_2 = (int)(std::log(static_cast<double>(n)) / std::log(2.0));
  int bs = 1 << pow_2;
  if (bs > 512) bs = 512;
  if (bs < 1) bs = 1;
  int L = 0;
  while ((1 << L) < bs) L++;
  return L;
}

template <int PP, int T, int MODE>
static int launch_fps(const FpsArgs& a, int B, int C, cudaStream_t stream) {
  constexpr int P = 2 * PP, WARPS = T / 32;
  const int E = (MODE == 1 || MODE == 3) ? WARPS * C : (MODE == 0 ? WARPS : C);
  const size_t smem = (size_t)4 * P * T * sizeof(float) + 16 + (size_t)2 * E * sizeof(FpsEntry) +
                      (MODE == 2 ? (size_t)2 * WARPS * sizeof(FpsEntry) : 0);
  auto kern = fps_kernel<PP, T, MODE>;
  if (smem > 48 * 1024) PS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (MODE == 0) {
    kern<<<B, T, smem, stream>>>(a);
  } else {
    if (C > 8) PS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(B * C);
    cfg.blockDim = dim3(T);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = C;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    PS_CUDA(cudaLaunchKernelEx(&cfg, kern, a));
  }
  PS_LAUNCH_CHECK();
  return PS_OK;
}

template <int T, int MODE>
static int dispatch_pp(int PP, const FpsArgs& a, int B, int C, cudaStream_t s) {
  switch (PP) {
    case 1: return launch_fps<1, T, MODE>(a, B, C, s);
    case 2: return launch_fps<2, T, MODE>(a, B, C, s);
    case 4: return launch_fps<4, T, MODE>(a, B, C, s);
    case 8: return launch_fps<8, T, MODE>(a, B, C, s);
    case 16: return launch_fps<16, T, MODE>(a, B, C, s);
  }
  return set_error(PS_ERR_UNSUPPORTED, "ps_fps: no kernel for %d point pairs per thread", PP);
}

struct FpsPlan { int C, T, PP; double cost; };  // cost: modelled SM cycles per iteration, waves included

// How many clusters of `c` CTAs (one CTA per SM, as every fps_kernel configuration runs) the device
// keeps resident at once: clusters must sit inside one GPC, so this is less than SMs / c for the
// large sizes.  Probed once per (device, size) with cudaOccupancyMaxActiveClusters on a stand-in
// kernel of the same footprint.
__global__ void __launch_bounds__(256, 1) fps_capacity_probe_kernel(int* p) {
  extern __shared__ int probe_smem[];
  if (p) p[0] = probe_smem[0];
}
static int cluster_capacity(int dev, int c, int nsm) {
  static std::atomic<int> cache[64][5];  // zero-initialised; concurrent first calls compute the same value
  int slot = 0;
  while ((1 << slot) < c) slot++;
  if (dev >= 0 && dev < 64) { const int c0 = cache[dev][slot].load(std::memory_order_relaxed); if (c0) return c0; }
  int cap = nsm / c;
  if (c > 1) {
    const int smem = 120 * 1024;  // forces one CTA per SM
    cudaFuncSetAttribute(fps_capacity_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (c > 8) cudaFuncSetAttribute(fps_capacity_probe_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(c * nsm);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = c; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, fps_capacity_probe_kernel, &cfg) == cudaSuccess && n > 0) cap = n;
    else cudaGetLastError();
  }
  if (cap < 1) cap = 1;
  if (dev >= 0 && dev < 64) cache[dev][slot].store(cap, std::memory_order_relaxed);
  return cap;
}

// Per-iteration cost model in SM cycles, cost = base + slope * PP (PP = point pairs per thread), fitted to B200
// measurements at B = 32 (tools/fps_time.py with PS_FPS_CLUSTER / PS_FPS_THREADS forced; profiles/fps_r1_notes.md):
// one warp per scheduler cannot hide its own dependency chains, so the per-pair cost is ~20 cycles rather than
// the ~7 issue slots it needs, and every configuration carries 550-800 cycles of exchange + reduction latency.
//   C=1 T=128: 565 + 23.5 PP     C=1 T=256: 725 + 43 PP
//   C=2 T=128: 758 + 19.7 PP     C=2 T=256: 800 + 38 PP
//   C=4 T=128: 800 + 16.7 PP     C=4 T=256: 860 + 33 PP
//   C=8      : (T/128) * (13 PP + 90) + 940   (two-level exchange; B=4 N=16384 measured 1132 cycles at PP=8)
//   C=16     : (T/128) * (13 PP + 90) + 1300  (only reachable when the cloud needs 16 CTAs)
// Lean 8-byte exchange (fps_lean_kernel; clouds that fit every CTA's shared memory, N <= 16384; second session of round
// 2, tools/fps_sweep.sh): C=2: 550 + 20 PP, C=4: 560 + 20 PP (PP=16: 880 = 0.449 us; PP=8: 720 = 0.366 us),
// C=8: 600 + 20 PP (PP=8: 757), C=16: 810 + 20 PP (PP=4: 892); T=256 doubles the per-pair term and adds ~70.
static bool fps_lean_fits(int c, int t, long long R, bool poll) {
  return c >= 2 && (t / 32) * c <= 64 && !poll && (size_t)3 * (size_t)R * sizeof(float) <= 200 * 1024;
}
static double fps_iter_cost(int c, int t, int pp, bool lean = false) {
  if (lean) {
    const double base = c == 2 ? 550.0 : (c == 4 ? 560.0 : (c == 8 ? 600.0 : 810.0));
    return base + (t / 128) * 20.0 * pp + (t == 256 ? 70.0 : 0.0);
  }
  if (c == 1) return t == 128 ? 565.0 + 23.5 * pp : 725.0 + 43.0 * pp;
  if (c == 2) return t == 128 ? 758.0 + 19.7 * pp : 800.0 + 38.0 * pp;
  if (c == 4) return t == 128 ? 800.0 + 16.7 * pp : 860.0 + 33.0 * pp;
  return (t / 128) * (13.0 * pp + 90.0) + (c == 8 ? 940.0 : 1300.0);
}
static bool fps_lean_enabled(bool poll) {
  bool lean = !poll;
  if (const char* e = getenv("PS_FPS_LEAN")) lean = lean && atoi(e) != 0;
  return lean;
}
static bool plan_fps(int B, int N, int L, int nper, int nsm, int dev, bool lean_on, FpsPlan& best) {
  const long long R = (long long)nper << L;
  int force_c = 0, force_t = 0;
  if (const char* e = getenv("PS_FPS_CLUSTER")) force_c = atoi(e);
  if (const char* e = getenv("PS_FPS_THREADS")) force_t = atoi(e);
  double best_cost = 1e30;
  bool found = false;
  for (int c = 1; c <= 16; c *= 2) {
    if (force_c && c != force_c) continue;
    for (int t = 128; t <= 256; t *= 2) {
      if (force_t && t != force_t) continue;
      int pp = 1;
      while ((long long)2 * pp * c * t < R) pp *= 2;
      if (pp > 16) continue;
      const int waves = ceil_div(B, cluster_capacity(dev, c, nsm));  // clusters that do not fit wait for a free GPC slot
      const double cost = waves * fps_iter_cost(c, t, pp, lean_on && fps_lean_fits(c, t, R, false));
      if (cost < best_cost - 1e-9) { best_cost = cost; best = {c, t, pp, cost}; found = true; }
    }
  }
  return found;
}

}  // namespace ps

using namespace ps;

extern "C" int ps_fps(const float* xyz, int* idx, int B, int N, int npoint, int dev, void* stream_) {
  return ps_fps_sample(xyz, idx, nullptr, B, N, npoint, dev, stream_);
}

extern "C" int ps_fps_sample(const float* xyz, int* idx, float* new_xyz, int B, int N, int npoint, int dev, void* stream_) {
  return ps_fps_sample_ex(xyz, idx, new_xyz, B, N, npoint, 0, dev, stream_);
}

extern "C" int ps_fps_sample_ex(const float* xyz, int* idx, float* new_xyz, int B, int N, int npoint, int flags, int dev,
                                void* stream_) {
  PS_REQUIRE(B >= 0 && N > 0 && npoint >= 0, "ps_fps: bad sizes B=%d N=%d npoint=%d", B, N, npoint);
  PS_REQUIRE((flags & ~PS_FPS_CORUN) == 0, "ps_fps: unknown flags 0x%x", flags);
  if (B == 0 || npoint == 0) return PS_OK;
  PS_REQUIRE(xyz && idx, "ps_fps: null pointer");
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_fps: cannot select device %d", dev);
  cudaStream_t stream = (cudaStream_t)stream_;
  const int nsm = sm_count(dev);

  FpsArgs a;
  a.xyz = xyz; a.idx = idx; a.new_xyz = new_xyz; a.N = N; a.npoint = npoint;
  a.L = ref_block_log2(N);
  a.nper = ceil_div(N, 1 << a.L);

  // exchange for small clusters: tag polling on plain remote stores (MODE 3) or st.async + mbarrier (lean / MODE 1)
  bool poll = false;
  if (const char* e = getenv("PS_FPS_EXCHANGE")) poll = (e[0] == 'p');
  bool lean_on = fps_lean_enabled(poll);
  FpsPlan pl;
  bool planned = plan_fps(B, N, a.L, a.nper, nsm, dev, lean_on, pl);
  // PS_FPS_CORUN: the caller runs another kernel next to this one (the sharded losses put the FPS chain under a Chamfer
  // term).  The lean exchange keeps the whole cloud in every CTA's shared memory (192 KB at 16384 points), i.e. it owns
  // its SMs.  That is the better neighbour while it leaves SMs over (C4 loss part, shard of 8 clouds: 1.56 against
  // 1.94 ms; 16 clouds: a tie); a batch whose clusters cover the GPU starves the neighbour instead (32 clouds: 3.58
  // against 3.29 ms), so there the 32-byte messages (64 KB per CTA, shares its SMs) are used (tools/c4loss_time.py)
  if ((flags & PS_FPS_CORUN) && lean_on && planned && B > 16 && 2 * pl.C * B > nsm) {
    lean_on = false;
    planned = plan_fps(B, N, a.L, a.nper, nsm, dev, lean_on, pl);
  }

  // Bucket-pruned single-CTA kernel (N <= 16384) where it wins: one SM per cloud at 0.6-0.85 us per iteration against
  // 2-4 SMs per cloud at 0.45 us for the cluster kernel (B200, profiles/fps_pruned_r2.jsonl), i.e. when the batch needs
  // so many waves of clusters that the planner's best estimate exceeds the pruned kernel's ~1700 cycles per iteration.  It leaves a per-cloud flag for the cluster kernel launched behind it, which only
  // samples the clouds the pruning did not bite on.  PS_FPS_PRUNE=0 off, 1 forced for every N it accepts (no give-up), 2 as 1
  // but with the give-up path.
  ScratchGuard prune_mem;
  {
    int mode = -1;
    if (const char* e = getenv("PS_FPS_PRUNE")) mode = atoi(e);
    // ~1650 cycles per iteration for the pruned kernel on a uniform cube (fewer on surfaces), one SM per cloud
    const bool wins = planned && N >= 8192 && npoint >= 2 * FP_CHECK && pl.cost > 1700.0 * ceil_div(B, nsm);
    const bool eligible = N <= FP_MAXN && npoint > 1 && (mode > 0 || (mode < 0 && wins));
    if (eligible) {
      const size_t inv_bytes = ((size_t)B * FP_MAXN * sizeof(unsigned short) + 255) & ~(size_t)255;
      if (int rc = prune_mem.alloc(inv_bytes + (size_t)B * sizeof(int), dev, stream)) return rc;
      FpsPruneArgs q;
      q.inv = static_cast<unsigned short*>(prune_mem.ptr);
      q.flag = reinterpret_cast<int*>(static_cast<char*>(prune_mem.ptr) + inv_bytes);
      q.check = (mode == 1 || npoint <= FP_CHECK + 1) ? 0 : 1;  // PS_FPS_PRUNE=2: pruned kernel first whatever the planner says, give-up path on
      // an unpruned scan updates every bucket every iteration; a working pruning touches all of them in the first
      // few iterations and a few per cent later (uniform cube: ~12 % of bucket x iteration pairs up to FP_CHECK)
      q.max_updates = (int)(0.5 * FP_CHECK * ceil_div(N, 32));
      const size_t smem = (size_t)3 * FP_MAXN * sizeof(float) + (size_t)FP_CELLS * sizeof(int);
      auto kern = fps_pruned_kernel<32, 1>;
      PS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      kern<<<B, 512, smem, stream>>>(a, q);
      PS_LAUNCH_CHECK();
      if (!q.check) return prune_mem.release();
      a.run_flag = q.flag;
    }
  }

  // small clouds: one CTA per cloud with the lean arg-max (fps_small_kernel); PS_FPS_SMALL=0 keeps the cluster planner
  {
    const long long R = (long long)a.nper << a.L;
    bool small = R <= 4096 && a.run_flag == nullptr;
    if (const char* e = getenv("PS_FPS_SMALL")) small = small && atoi(e) != 0;
    if (getenv("PS_FPS_CLUSTER") || getenv("PS_FPS_THREADS")) small = false;  // a forced plan means the cluster kernels
    if (small) {
      const int T = R <= 1024 ? 128 : (R <= 2048 ? 256 : 512);
      int PP = 1;
      while (2ll * PP * T < R) PP *= 2;
      if (T == 128) return PP == 1 ? launch_fps_small<1, 128>(a, B, stream) : (PP == 2 ? launch_fps_small<2, 128>(a, B, stream) : launch_fps_small<4, 128>(a, B, stream));
      if (T == 256) return PP <= 2 ? launch_fps_small<2, 256>(a, B, stream) : launch_fps_small<4, 256>(a, B, stream);
      return PP <= 2 ? launch_fps_small<2, 512>(a, B, stream) : launch_fps_small<4, 512>(a, B, stream);
    }
  }

  if (!planned) {
    // beyond the register-resident kernels (N > 131072): one CTA per cloud with global scratch
    ScratchGuard temp_mem;
    if (int rc = temp_mem.alloc((size_t)B * N * sizeof(float), dev, stream)) return rc;
    fps_generic_kernel<<<B, FPS_GT, 0, stream>>>(a, static_cast<float*>(temp_mem.ptr));
    PS_LAUNCH_CHECK();
    return temp_mem.release();
  }
  // lean 8-byte exchange where every CTA of the cluster can hold the whole cloud (PS_FPS_LEAN=0: the 32-byte messages)
  if (lean_on && fps_lean_fits(pl.C, pl.T, (long long)a.nper << a.L, poll))
    return pl.T == 128 ? dispatch_lean<128>(pl.PP, a, B, pl.C, stream) : dispatch_lean<256>(pl.PP, a, B, pl.C, stream);
  if (pl.T == 128) {
    if (pl.C == 1) return dispatch_pp<128, 0>(pl.PP, a, B, pl.C, stream);
    if (pl.C <= 4) return poll ? dispatch_pp<128, 3>(pl.PP, a, B, pl.C, stream) : dispatch_pp<128, 1>(pl.PP, a, B, pl.C, stream);
    return dispatch_pp<128, 2>(pl.PP, a, B, pl.C, stream);
  }
  if (pl.C == 1) return dispatch_pp<256, 0>(pl.PP, a, B, pl.C, stream);
  if (pl.C <= 4) return poll ? dispatch_pp<256, 3>(pl.PP, a, B, pl.C, stream) : dispatch_pp<256, 1>(pl.PP, a, B, pl.C, stream);
  return dispatch_pp<256, 2>(pl.PP, a, B, pl.C, stream);
}

// Ragged batch: cloud b is the first n_host[b] points of row b, sampled exactly as ps_fps_sample samples that cloud on
// its own (its own bs = opt_n_threads(n) and nper, hence its own tie-break ranks).  One launch of the single-CTA kernel
// for the whole batch, sized by its largest cloud; a smaller cloud leaves the ranks beyond its own as padding.
extern "C" int ps_fps_sample_ragged(const float* xyz, const int* n_host, int* idx, float* new_xyz, int B, int stride,
                                    int npoint, int dev, void* stream_) {
  PS_REQUIRE(B >= 0 && stride >= 0 && npoint >= 0, "ps_fps_sample_ragged: bad sizes B=%d stride=%d npoint=%d", B, stride,
             npoint);
  if (B == 0 || npoint == 0) return PS_OK;
  PS_REQUIRE(xyz && n_host && idx, "ps_fps_sample_ragged: null pointer");
  long long Rmax = 0;
  for (int b = 0; b < B; b++) {
    const int n = n_host[b];
    PS_REQUIRE(n >= 1 && n <= stride, "ps_fps_sample_ragged: size %d of cloud %d outside [1, stride=%d]", n, b, stride);
    const int L = ref_block_log2(n);
    const long long R = (long long)ceil_div(n, 1 << L) << L;
    if (R > Rmax) Rmax = R;
  }
  if (Rmax > 8192)
    return set_error(PS_ERR_UNSUPPORTED, "ps_fps_sample_ragged: a cloud of %lld padded points exceeds the 8192 one CTA holds",
                     Rmax);
  DeviceGuard guard(dev);
  if (!guard.ok) return set_error(PS_ERR_CUDA, "ps_fps_sample_ragged: cannot select device %d", dev);
  cudaStream_t stream = (cudaStream_t)stream_;
  int4* host_part = new int4[B];
  for (int b = 0; b < B; b++) {
    const int L = ref_block_log2(n_host[b]);
    host_part[b] = make_int4(n_host[b], L, ceil_div(n_host[b], 1 << L), 0);
  }
  ScratchGuard part;
  int rc = part.alloc((size_t)B * sizeof(int4), dev, stream);
  // pageable source: the copy has taken the bytes when it returns, so the staging array can go at once
  if (rc == PS_OK && cudaMemcpyAsync(part.ptr, host_part, (size_t)B * sizeof(int4), cudaMemcpyHostToDevice, stream) !=
                         cudaSuccess)
    rc = set_error(PS_ERR_CUDA, "ps_fps_sample_ragged: upload of the cloud sizes failed: %s",
                   cudaGetErrorString(cudaGetLastError()));
  delete[] host_part;
  if (rc) return rc;
  FpsArgs a;
  a.xyz = xyz; a.idx = idx; a.new_xyz = new_xyz; a.N = 0; a.npoint = npoint; a.L = 0; a.nper = 0;
  a.part = static_cast<const int4*>(part.ptr);
  a.stride = stride;
  if (Rmax <= 512) rc = launch_fps_small<2, 128, true>(a, B, stream);
  else if (Rmax <= 1024) rc = launch_fps_small<4, 128, true>(a, B, stream);
  else if (Rmax <= 2048) rc = launch_fps_small<4, 256, true>(a, B, stream);
  else if (Rmax <= 4096) rc = launch_fps_small<4, 512, true>(a, B, stream);
  else rc = launch_fps_small<8, 512, true>(a, B, stream);
  if (rc) return rc;
  return part.release();
}
