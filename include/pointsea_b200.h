/*
 * pointsea_b200.h — C ABI of the B200-native point-geometry hot path.
 *
 * Drop-in boundary for shiyuan0806/SVDFormer_PointSea.  Every entry point replaces one
 * launcher the reference binds through pybind11 (cited per function, paths relative to the
 * reference tree).  The reference-side binding a maintainer adds is a ctypes / pybind stub
 * that forwards `tensor.data_ptr()` + sizes + the current CUDA stream; see INTEGRATION.md.
 *
 * Conventions
 *   - plain C: raw DEVICE pointers, int sizes, the CUDA device ordinal and a cudaStream_t
 *     passed as void*.  No torch / ATen types cross this boundary.
 *   - all tensors are dense, contiguous, fp32 / int32, laid out exactly as the reference's
 *     (B,N,3) clouds, (B,C,N) features and (B,S,K) index tensors.
 *   - the caller owns every buffer (the reference's pybind layer allocates with torch::zeros;
 *     our Python layer allocates with torch.empty).  The library never retains a pointer.
 *     Scratch, where a kernel needs it, is stream-ordered (cudaMallocAsync on `stream`).
 *   - work is enqueued on `stream` and the call returns immediately (no host sync).
 *   - return value: PS_OK (0) or a negative PS_ERR_* code; ps_last_error() gives a
 *     thread-local message.  Nothing ever calls exit() (the reference's CUDA_CHECK_ERRORS
 *     does: pointnet2_ops/_ext-src/include/cuda_utils.h:30-39) and no error is silently
 *     dropped (the reference's Chamfer returns an int Python ignores: chamfer3D.cu:145-150).
 *   - thread-safe: callable concurrently from several host threads on the same or different
 *     devices (nn.DataParallel replica threads).  The only process-wide state is per-device
 *     and internally synchronised: a private scratch memory pool and cached device attributes
 *     (runtime.cu), and the mutex-guarded staging slots / CUDA-graph caches of the one-launch
 *     step entry points (step.cu, host_pipeline.cu).  Error text and the launch counter are
 *     thread-local.
 */
#ifndef POINTSEA_B200_H
#define POINTSEA_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define PS_OK 0
#define PS_ERR_INVALID_ARG (-1) /* null pointer, negative size, unsupported size */
#define PS_ERR_CUDA (-2)        /* a CUDA runtime call or launch failed */
#define PS_ERR_UNSUPPORTED (-3) /* shape outside what the kernels cover (message says which) */

/* Library version: major*10000 + minor*100 + patch. */
int ps_version(void);
/* Thread-local, NUL-terminated description of the last error on this host thread. */
const char* ps_last_error(void);
/* SM count and compute capability of `dev` (used by the host layer to fail loudly off sm_100). */
int ps_device_info(int dev, int* sm_count, int* cc_major, int* cc_minor);

/* ---- Chamfer distance -------------------------------------------------------------------
 * Replaces chamfer_cuda_forward  (metrics/CD/chamfer3D/chamfer3D.cu:136-154, kernel :12-134;
 * pybind `chamfer_3D.forward`, chamfer_cuda.cpp:17-19,31).
 *   xyz1 (B,N,3) f32, xyz2 (B,M,3) f32
 *   dist1 (B,N) f32 = min_j |xyz1_i - xyz2_j|^2 ; idx1 (B,N) i32 = lowest argmin j
 *   dist2 (B,M), idx2 (B,M): the same with the roles swapped.
 * Arithmetic is the reference's SASS order d = fma(dz,dz, fma(dx,dx, dy*dy)), dx = target - query.
 */
int ps_chamfer_fwd(const float* xyz1, const float* xyz2, float* dist1, float* dist2, int* idx1,
                   int* idx2, int B, int N, int M, int dev, void* stream);

/* Replaces chamfer_cuda_backward (chamfer3D.cu:176-195, kernel :155-174; pybind `.backward`).
 *   gradxyz1 (B,N,3), gradxyz2 (B,M,3) are OVERWRITTEN (the reference needs them pre-zeroed by
 *   the caller, dist_chamfer_3D.py:56-60; here zero-filling is not required).
 */
int ps_chamfer_bwd(const float* xyz1, const float* xyz2, const float* graddist1,
                   const float* graddist2, const int* idx1, const int* idx2, float* gradxyz1,
                   float* gradxyz2, int B, int N, int M, int dev, void* stream);

/* Fused reduction of Chamfer's outputs as the callers reduce them (utils/loss_utils.py:10-31 `mean`,
 * `mean(sqrt)`; :98-103 per-cloud means): out6 (6 doubles, device) = { sum sqrt(dist1),
 * sum sqrt(dist2), sum dist1, sum dist2, n1, n2 }.  One launch; these partial sums and counts are
 * what the multi-GPU path all-reduces. */
int ps_chamfer_sums(const float* dist1, const float* dist2, double* out6, long long n1, long long n2,
                    int dev, void* stream);

/* ps_chamfer_fwd with the callers' reductions (utils/loss_utils.py:10-31: mean / mean-of-sqrt per side) fused
 * into the forward's epilogue launch: sums6 (device, 6 doubles, layout of ps_chamfer_sums) comes out of the pass
 * that writes dist/idx, without re-reading them.  The sums are accumulated in a fixed order (bit-reproducible). */
int ps_chamfer_fwd_sums(const float* xyz1, const float* xyz2, float* dist1, float* dist2, int* idx1, int* idx2,
                        double* sums6, int B, int N, int M, int dev, void* stream);

/* ---- Chamfer training losses (utils/loss_utils.py:10-31) as one forward and one backward ----------------------
 * n1 = B*N and n2 = B*M are the element counts torch.mean divides by.  Other kind values are rejected. */
#define PS_LOSS_CD 0          /* chamfer:                  mean(d1) + mean(d2)               */
#define PS_LOSS_CD_SQRT 1     /* chamfer_sqrt:             (mean(sqrt d1) + mean(sqrt d2)) / 2 */
#define PS_LOSS_SINGLE 2      /* chamfer_single_side:      mean(d1)                          */
#define PS_LOSS_SINGLE_SQRT 3 /* chamfer_single_side_sqrt: mean(sqrt d1)                     */
/* ps_chamfer_fwd_sums (dist/idx and sums6, device, 6 doubles of scratch) followed by one single-thread launch that
 * writes loss (device, 1 float): the sums combined in double and rounded once.  No host sync.  B = 0 gives NaN, as
 * torch.mean of an empty tensor. */
int ps_chamfer_loss_fwd(const float* xyz1, const float* xyz2, float* dist1, float* dist2, int* idx1, int* idx2,
                        double* sums6, float* loss, int kind, int B, int N, int M, int dev, void* stream);
/* Backward of ps_chamfer_loss_fwd: grad_loss (device, 1 float) is the upstream gradient of the loss.  Each point's
 * distance gradient is derived from dist1/dist2 with torch's autograd of the reference expression (g*0.5 for the
 * sqrt kinds' "/ 2", g * (1.0f/n), g / (2*sqrtf(d)) for the sqrt kinds: inf/NaN at d = 0 as in torch), then turned
 * into point gradients with ps_chamfer_bwd's arithmetic.  gradxyz1 (B,N,3) / gradxyz2 (B,M,3): OVERWRITTEN (zero
 * where no term reaches them); either may be NULL (its writes and scatters are skipped), not both.  Two launches:
 * plain stores, then atomics; the second is skipped when no scattered term lands in a non-NULL buffer. */
int ps_chamfer_loss_bwd(const float* xyz1, const float* xyz2, const float* dist1, const float* dist2, const int* idx1,
                        const int* idx2, const float* grad_loss, float* gradxyz1, float* gradxyz2, int kind, int B,
                        int N, int M, int dev, void* stream);

/* ---- the single collective of the batch-sharded path (SURVEY 8e), over peer memory ---------------------------
 * The reference has no multi-process path (nn.DataParallel gathers on one GPU); its loss reductions
 * (utils/loss_utils.py:10-19,50-57) are what has to be summed across ranks.  A ps_comm is a set of per-rank
 * MAILBOXES in device memory that the peers store into directly over NVLink: the kernel that produces the sums
 * publishes them, a one-warp kernel adds the world's contributions in rank order (bit-identical on every rank).
 * No host call per step, so a whole step replays as one CUDA graph.  Setup (once):
 *   ps_comm_create on every rank -> ps_comm_export (an opaque ps_comm_handle_bytes()-byte handle, CUDA IPC) ->
 *   exchange the handles by any host channel (torch.distributed.all_gather_object, MPI, a file) ->
 *   ps_comm_connect(handles of all ranks, rank order).  Ranks living in ONE process (threads, tests) use
 *   ps_comm_connect_local instead.  Every rank must issue the same sequence of collective calls. */
typedef struct ps_comm ps_comm;
int ps_comm_create(int rank, int world, int dev, ps_comm** out);
int ps_comm_handle_bytes(void);
int ps_comm_export(ps_comm* comm, void* handle);
int ps_comm_connect(ps_comm* comm, const void* handles /* world x ps_comm_handle_bytes() */);
int ps_comm_connect_local(ps_comm* const* comms, int world);
/* out[0..n) (device) = sum over ranks of in[0..n) (device), n <= 30, one launch on `stream`. */
int ps_comm_allreduce(ps_comm* comm, const double* in, double* out, int n, void* stream);
/* Diagnostics (synchronises the device): messages published / consumed, and whether a wait timed out
 * (a lost peer gives NaN results and this flag after ~4 s instead of hanging the GPU). */
int ps_comm_status(ps_comm* comm, long long* published, long long* consumed, int* timed_out);
int ps_comm_destroy(ps_comm* comm);

/* One training-style Chamfer step on DEVICE buffers as ONE launch: forward + loss sums (+ publish to the peers)
 * + backward (+ wait: world-wide sums).  Equivalent to ps_chamfer_fwd_sums, ps_chamfer_bwd and — with a
 * communicator — ps_comm_allreduce of the sums, captured into a CUDA graph keyed by the arguments and replayed
 * with a single cudaGraphLaunch (fresh buffer addresses retarget the cached graph in place).  graddist1 ==
 * graddist2 == NULL: forward + sums only.  comm == NULL: sums_global6 is not written.  Buffers as in
 * ps_chamfer_fwd / ps_chamfer_bwd; sums_local6 / sums_global6: device, 6 doubles each. */
int ps_chamfer_step(const float* xyz1, const float* xyz2, const float* graddist1, const float* graddist2,
                    float* dist1, float* dist2, int* idx1, int* idx2, float* gradxyz1, float* gradxyz2,
                    double* sums_local6, double* sums_global6, ps_comm* comm, int B, int N, int M, int dev,
                    void* stream);
/* Same arguments, nothing launched: captures and instantiates the graph of this exact call ahead of time, so the
 * first real step costs a replay (ranks that share a device, or a timed loop, call this first). */
int ps_chamfer_step_prepare(const float* xyz1, const float* xyz2, const float* graddist1, const float* graddist2,
                            float* dist1, float* dist2, int* idx1, int* idx2, float* gradxyz1, float* gradxyz2,
                            double* sums_local6, double* sums_global6, ps_comm* comm, int B, int N, int M, int dev);
/* Graph-cache counters of ps_chamfer_step / of the host-buffer entry points on `dev`: exact replays, in-place
 * retargets (cudaGraphExecUpdate) and instantiations so far. */
int ps_chamfer_step_stats(int dev, long long* hits, long long* updates, long long* instantiations);
int ps_chamfer_host_stats(int dev, long long* hits, long long* updates, long long* instantiations);

/* Host-buffer form of one Chamfer step (forward, and backward when graddist1/2 are given): every
 * pointer here is a HOST pointer with the shapes of ps_chamfer_fwd / ps_chamfer_bwd.  This is the
 * call for the reference's CPU-allocating wrapper (dist_chamfer_3D.py:33-42 allocates dist/idx on
 * the CPU and copies) and for metric loops whose clouds arrive from the data loader in host memory.
 * The batch is processed in chunks of `chunk` clouds (<= 0: library default) on three internal
 * streams so that upload, kernels and download of consecutive chunks overlap; results are
 * bit-identical to the device entry points for any chunk size (all kernels are per-cloud).
 * The call enqueues and returns: the output buffers are complete once `stream` has passed this
 * point (synchronise it, or an event recorded on it).  Pinned host memory is needed for overlap.
 * graddist1 == graddist2 == NULL => forward only (gradxyz1/2 ignored). */
int ps_chamfer_host(const float* xyz1, const float* xyz2, float* dist1, float* dist2, int* idx1,
                    int* idx2, const float* graddist1, const float* graddist2, float* gradxyz1,
                    float* gradxyz2, int B, int N, int M, int chunk, int dev, void* stream);

/* Training-style step on HOST-resident inputs: the clouds (and, for the backward, the upstream gradients) are
 * uploaded in chunks exactly as in ps_chamfer_host, but only the step's RESULT crosses PCIe on the way back —
 * sums6 (HOST, 6 doubles, the layout of ps_chamfer_sums: what the loss / metric of utils/loss_utils.py:10-31 is
 * made of).  The gradients are written straight into the caller's DEVICE buffers dev_gradxyz1 (B,N,3) /
 * dev_gradxyz2 (B,M,3), where the optimizer consumes them (the reference's Function also returns device tensors,
 * dist_chamfer_3D.py:44-47); dist/idx never leave the staging slots.  graddist1 == graddist2 == NULL => forward +
 * sums only.  Enqueue-only like ps_chamfer_host; sums6 and the gradients are complete once `stream` has passed
 * this point. */
int ps_chamfer_host_step(const float* xyz1, const float* xyz2, const float* graddist1, const float* graddist2,
                         float* dev_gradxyz1, float* dev_gradxyz2, double* sums6, int B, int N, int M, int chunk,
                         int dev, void* stream);

/* ps_chamfer_host_step on a batch shard: sums6 receives the WORLD-WIDE sums (the local sums are exchanged
 * through `comm` by a kernel inside the same graph, after the last chunk). */
int ps_chamfer_host_step_dist(const float* xyz1, const float* xyz2, const float* graddist1, const float* graddist2,
                              float* dev_gradxyz1, float* dev_gradxyz2, double* sums6, ps_comm* comm, int B, int N,
                              int M, int chunk, int dev, void* stream);

/* General host-buffer form: everything ps_chamfer_host downloads (dist, idx, gradients) plus the loss sums
 * (sums6, HOST, may be NULL), world-wide when `comm` is given (may be NULL).  Same pipeline, same graph. */
int ps_chamfer_host_full(const float* xyz1, const float* xyz2, float* dist1, float* dist2, int* idx1, int* idx2,
                         const float* graddist1, const float* graddist2, float* gradxyz1, float* gradxyz2,
                         double* sums6, ps_comm* comm, int B, int N, int M, int chunk, int dev, void* stream);

/* Asynchronous pair for loops that keep several steps in flight (the reference's evaluation loops read one batch
 * from the loader while the previous one is on the GPU, core/eval_pcn.py:44-60): ps_chamfer_host_submit is
 * ps_chamfer_host_full ordered BEHIND the current position of `stream` but not joined back into it — it runs on one
 * of the library's four lanes (own copy streams and staging slots; taken in turn): its uploads and downloads run on the
 * lane's copy streams, its kernels — replayed as one graph — on the one stream that serves all lanes in submission
 * order, so the copies of the neighbouring steps overlap the kernels of step i; up to four steps may be in flight.  *ticket (never 0 for a non-empty call) names the step for
 * ps_chamfer_host_wait: wait_stream != 0 makes `stream` wait for the step's last output byte, block != 0 blocks the
 * calling thread until then.  The buffers of a step must not be reused before it has been waited for.  With a
 * communicator every lane exchanges on its own channel of it, so the steps still overlap; every rank must then
 * submit the same sequence of steps (the i-th submissions of all ranks meet in one exchange). */
int ps_chamfer_host_submit(const float* xyz1, const float* xyz2, float* dist1, float* dist2, int* idx1, int* idx2,
                           const float* graddist1, const float* graddist2, float* gradxyz1, float* gradxyz2,
                           double* sums6, ps_comm* comm, int B, int N, int M, int chunk, int dev, void* stream,
                           long long* ticket);
int ps_chamfer_host_wait(long long ticket, int dev, void* stream, int wait_stream, int block);

/* ---- Furthest point sampling ------------------------------------------------------------
 * Replaces furthest_point_sampling_kernel_wrapper (pointnet2_ops/_ext-src/src/sampling_gpu.cu:175-229,
 * kernel :69-173; pybind `_ext.furthest_point_sampling`, sampling.cpp:66-87).
 *   xyz (B,N,3) f32 -> idx (B,npoint) i32.  No `temp` scratch is needed (the running
 *   min-distance array lives in registers).  Tie-break and origin-skip rule are the reference's.
 */
int ps_fps(const float* xyz, int* idx, int B, int N, int npoint, int dev, void* stream);
/* Same sampling, additionally writing the sampled coordinates new_xyz (B,npoint,3) = xyz[b, idx[b,j]]
 * from inside the FPS kernel (the winner's coordinates are already in registers): the fused form of
 * the call site fps_subsample = FPS + gather + two transposes (models/model_utils.py:489-499).
 * new_xyz may be NULL (then identical to ps_fps). */
int ps_fps_sample(const float* xyz, int* idx, float* new_xyz, int B, int N, int npoint, int dev,
                  void* stream);
/* ps_fps_sample with hints.  PS_FPS_CORUN: another kernel runs next to this one on the same GPU (the sharded losses put
 * the FPS chain on a side stream under a Chamfer term): when the batch's clusters would cover the GPU, the launcher
 * picks the variant that leaves most of each SM's shared memory to the neighbour.  The samples do not depend on the
 * flags. */
#define PS_FPS_CORUN 1
int ps_fps_sample_ex(const float* xyz, int* idx, float* new_xyz, int B, int N, int npoint, int flags, int dev,
                     void* stream);

/* ps_fps_sample on a ragged batch: cloud b is the first n_host[b] points of row b of xyz (B rows of `stride` points,
 * row b at b*stride*3 floats).  n_host (HOST, B ints) is validated (1 <= n <= stride) before any CUDA call and uploaded
 * with one copy.  idx (B,npoint) i32, relative to the row; new_xyz (B,npoint,3) or NULL.  Every cloud's samples are
 * bit-identical to ps_fps_sample on that cloud alone (its own tie-break ranks, origin skip, n < npoint).  One launch
 * whatever B; a cloud padded to more than 8192 ranks (opt_n_threads rounding) returns PS_ERR_UNSUPPORTED. */
int ps_fps_sample_ragged(const float* xyz, const int* n_host, int* idx, float* new_xyz, int B, int stride, int npoint,
                         int dev, void* stream);

/* ---- online cropping (ShapeNet-55/34: utils/helpers.py:62-123 seprate_point_cloud) ------------------------------
 * xyz (B,N,3) f32; centers_host (HOST, B x 3 floats) and num_crop_host (HOST, B ints, each in [0, N]) are validated
 * before any CUDA call and uploaded with one copy.  Per cloud, the points are ordered by the fp32 value of
 * torch.norm(center - p, p=2, dim=-1), ties by index (torch.argsort's stable order on CUDA):
 *   crop row b (crop + b*crop_stride*3): the count nearest points, ascending;
 *   keep row b (keep + b*keep_stride*3): the other N - count points, ascending; with pad_zeros != 0 instead all N
 *     points in their original order, the cropped ones multiplied by 0.
 * Equal counts with strides N-c / c give packed (B,N-c,3) / (B,c,3) tensors; strides N hold ragged rows.  One launch
 * whatever B.  keep / crop may be NULL when all their rows are empty.  N outside 33..16384 returns
 * PS_ERR_UNSUPPORTED. */
int ps_crop_split(const float* xyz, const float* centers_host, const int* num_crop_host, float* keep, float* crop,
                  int B, int N, int keep_stride, int crop_stride, int pad_zeros, int dev, void* stream);

/* ---- gather / group ---------------------------------------------------------------------
 * Replaces gather_points_kernel_wrapper (sampling_gpu.cu:22-30) / _grad_ (:49-57):
 *   out[b,c,j] = features[b,c,idx[b,j]] ; features (B,C,N), idx (B,M) i32, out (B,C,M).
 *   bwd: grad_features (B,C,N) is OVERWRITTEN with the scatter-add of grad_out (B,C,M).
 */
int ps_gather_fwd(const float* features, const int* idx, float* out, int B, int C, int N, int M,
                  int dev, void* stream);
int ps_gather_bwd(const float* grad_out, const int* idx, float* grad_features, int B, int C,
                  int N, int M, int dev, void* stream);
/* Replaces group_points_kernel_wrapper (group_points_gpu.cu:30-39) / _grad_ (:66-75):
 *   out[b,c,s,k] = features[b,c,idx[b,s,k]] ; idx (B,S,K) i32, out (B,C,S,K).
 */
int ps_group_fwd(const float* features, const int* idx, float* out, int B, int C, int N, int S,
                 int K, int dev, void* stream);
int ps_group_bwd(const float* grad_out, const int* idx, float* grad_features, int B, int C, int N,
                 int S, int K, int dev, void* stream);

/* ---- neighbourhood queries --------------------------------------------------------------
 * Replaces query_ball_point_kernel_wrapper (ball_query_gpu.cu:46-54, kernel :9-44; note the
 * argument order of `_ext.ball_query(new_xyz, xyz, radius, nsample)`, ball_query.cpp:8-32).
 *   new_xyz (B,S,3) centres, xyz (B,N,3) -> idx (B,S,nsample) i32: the first nsample indices
 *   (ascending) with d2 < radius*radius, padded with the first hit; all zero when none.
 */
int ps_ball_query(const float* new_xyz, const float* xyz, int* idx, int B, int N, int S,
                  float radius, int nsample, int dev, void* stream);

/* Replaces the torch expression query_knn / square_distance (models/model_utils.py:258-286):
 *   idx (B,S,k) i32 = indices of the k smallest of
 *       dist[s,n] = ((-2*dot(new_xyz_s, xyz_n)) + |new_xyz_s|^2) + |xyz_n|^2   (fp32)
 *   in ascending (dist, index) order, skipping the first `skip` (skip=1 <=> include_self=False).
 *   No (B,S,N) matrix is materialised.
 */
int ps_knn(const float* xyz, const float* new_xyz, int* idx, int B, int N, int S, int k, int skip,
           int dev, void* stream);

/* ---- 3-NN + interpolation (SURVEY 8f rank 1) ---------------------------------------------
 * Replaces three_nn_kernel_wrapper (interpolate_gpu.cu:61-68, kernel :9-59):
 *   unknown (B,n,3), known (B,m,3) -> dist2 (B,n,3) f32 (squared), idx (B,n,3) i32.
 * three_interpolate_kernel_wrapper (:103-112) / _grad_ (:145-154):
 *   out[b,c,j] = sum_t points[b,c,idx[b,j,t]] * weight[b,j,t] ; points (B,C,m), out (B,C,n).
 */
int ps_three_nn(const float* unknown, const float* known, float* dist2, int* idx, int B, int n,
                int m, int dev, void* stream);
int ps_three_interpolate_fwd(const float* points, const int* idx, const float* weight, float* out,
                             int B, int C, int m, int n, int dev, void* stream);
int ps_three_interpolate_bwd(const float* grad_out, const int* idx, const float* weight,
                             float* grad_points, int B, int C, int n, int m, int dev, void* stream);

/* ---- fused call sites and the next ops on the path (SURVEY 8f ranks 2-4) ----------------------
 * Result order of the kNN entry points below. */
#define PS_ORDER_SORT 0 /* ascending (dist, index): torch.argsort, as ps_knn */
#define PS_ORDER_TOPK 1 /* torch.topk(k, largest=False, sorted=True) on CUDA, including its order among
                            equal distances (gather order + 32-slot bitonic network, k <= 32) */

/* query_knn_point (models/model_utils.py:807-810): square_distance + topk(k, largest=False).
 * Same arithmetic as ps_knn, result in torch.topk's order.  idx (B,S,k) i32. */
int ps_knn_point(const float* xyz, const float* new_xyz, int* idx, int B, int N, int S, int k, int dev,
                 void* stream);

/* The kNN + coordinate grouping + centre subtraction of sample_and_group_knn
 * (models/model_utils.py:342-345: query_knn, grouping_operation(xyz, idx), grouped_xyz -= new_xyz) in ONE
 * kernel: idx (B,S,k) i32 as ps_knn, grouped_xyz (B,3,S,k) f32 = xyz[b,idx[b,s,j],c] - new_xyz[b,s,c]. */
int ps_knn_group_xyz(const float* xyz, const float* new_xyz, int* idx, float* grouped_xyz, int B, int N,
                     int S, int k, int dev, void* stream);

/* Feature-space kNN (group_local / EdgeConv neighbourhoods, models/model_utils.py:258-279, 807-826):
 *   xr references, xq queries; channel_major != 0: (B,C,N) / (B,C,S) tensors (EdgeConv's layout), else
 *   (B,N,C) / (B,S,C) (the layout query_knn_point receives).  idx (B,S,k) i32, k <= 32, N <= 6144.
 *   dist = ((-2 * dot) + |q|^2) + |r|^2 with dot an ascending-channel FMA chain (cuBLAS fp32 order) and
 *   |.|^2 in the order of torch.sum(x ** 2, -1) on CUDA; order = PS_ORDER_SORT / PS_ORDER_TOPK.
 *   No (B,S,N) matrix is materialised. */
int ps_knn_feat(const float* xr, const float* xq, int* idx, int B, int C, int N, int S, int k,
                int channel_major, int order, int dev, void* stream);

/* EdgeConv front (models/model_utils.py:869-877 after group_local): x (B,C,N), idx (B,N,K) i32 ->
 *   out (B,2C,N,K): out[b,c,n,k] = x[b,c,n] - x[b,c,idx[b,n,k]], out[b,C+c,n,k] = x[b,c,n].
 * bwd: grad_x (B,C,N) is OVERWRITTEN with the gradient of grad_out (B,2C,N,K). */
int ps_edge_features_fwd(const float* x, const int* idx, float* out, int B, int C, int N, int K, int dev,
                         void* stream);
int ps_edge_features_bwd(const float* grad_out, const int* idx, float* grad_x, int B, int C, int N, int K,
                         int dev, void* stream);

/* index_points (models/model_utils.py:828-845): points (B,N,C), idx (B,M) i32 (trailing index dims
 * flattened) -> out (B,M,C) = points[b, idx[b,m], :].  bwd OVERWRITES grad_points (B,N,C). */
int ps_index_points_fwd(const float* points, const int* idx, float* out, int B, int N, int M, int C,
                        int dev, void* stream);
int ps_index_points_bwd(const float* grad_out, const int* idx, float* grad_points, int B, int N, int M,
                        int C, int dev, void* stream);

/* Evaluation epilogue of one Chamfer call (calc_cd utils/loss_utils.py:98-115, fscore metrics/CD/fscore.py:3-16,
 * calc_dcd utils/loss_utils.py:117-155) in one launch:
 *   out8 (B,8) f32 = { mean sqrt dist1, mean sqrt dist2, mean dist1, mean dist2, precision_1, precision_2,
 *                      fscore, dcd } per cloud; dist1 (B,n1), dist2 (B,n2), idx1 (B,n1) in [0,n2), idx2 (B,n2)
 *   in [0,n1).  idx1 == idx2 == NULL skips the density-aware term (out[7] = 0).  dcd_frac1 / dcd_frac2 are
 *   calc_dcd's frac_21 / frac_12 (the factors applied to the dist1 / dist2 side). */
int ps_chamfer_metrics(const float* dist1, const float* dist2, const int* idx1, const int* idx2, float* out8,
                       int B, int n1, int n2, float fscore_threshold, float dcd_alpha, float dcd_n_lambda,
                       float dcd_frac1, float dcd_frac2, int dev, void* stream);
/* Backward of ps_chamfer_metrics' differentiable outputs (what makes calc_cd / calc_dcd training losses): per-cloud
 * upstream gradients -> per-point gradients of the distances, which ps_chamfer_bwd turns into point gradients.
 * terms: bitmask of the per-cloud upstream gradients present in gcoef5 (B,5) =
 *   bit0 mean sqrt d1, bit1 mean sqrt d2, bit2 mean d1, bit3 mean d2, bit4 dcd; other bits are rejected.
 *   A clear bit contributes nothing (gcoef5 may be NULL when terms == 0); bit4 needs idx1 and idx2.
 * graw1 (B,n1) / graw2 (B,n2): upstream gradients of the raw dist outputs, or NULL.
 * graddist1 (B,n1), graddist2 (B,n2): OVERWRITTEN.  Other arguments as ps_chamfer_metrics.
 *   graddist1[j] = graw1[j] + g0/n1 / (2 sqrt d1[j]) + g2/n1 + g4*0.5/n1 * alpha * exp(-alpha d1[j]) * w1[j]
 *   (w1 = calc_dcd's weight of the hit count of idx1[j], detached); side 2 likewise with bits 1, 3, 4 and dcd_frac2.
 *   torch's formulas, unclamped: a present sqrt term at d = 0 yields inf, as the reference's does. */
int ps_chamfer_metrics_bwd(const float* dist1, const float* dist2, const int* idx1, const int* idx2,
                           const float* gcoef5, unsigned terms, const float* graw1, const float* graw2,
                           float* graddist1, float* graddist2, int B, int n1, int n2, float dcd_alpha,
                           float dcd_n_lambda, float dcd_frac1, float dcd_frac2, int dev, void* stream);

/* ---- scatter-max (PointSea's depth-map renderer) ------------------------------------------
 * torch_scatter.scatter(src, index, dim, out, dim_size, reduce="max") as models_PointSea/mv_utils_zs.py:130 calls it.
 * src (outer, E, inner) f32, index (outer, E, inner) i64 (already broadcast to src's shape), out (outer, D, inner) f32.
 * fresh != 0: out is initialised here and positions that receive nothing become 0 (torch_scatter without `out=`;
 *   as there, a max of exactly -FLT_MAX also reads 0);
 * fresh == 0: out's current values take part in the max (torch_scatter with `out=`), updated in place; a NaN there
 *   is kept (a negative NaN pattern becomes the canonical positive one once a src element reaches it).
 * argmax (outer, D, inner) i64 or NULL: position along E of the lowest-index src element equal to the result (NaN
 *   matching NaN), E if none.
 * Index values outside [0, D) are skipped.  NaN propagates (canonical positive NaN); +0 is larger than -0.  The result
 * does not depend on the order of the updates. */
int ps_scatter_max(const float* src, const long long* index, float* out, long long* argmax, long long outer,
                   long long E, long long inner, long long D, int fresh, int dev, void* stream);

/* ---- measurement helpers (bench.py) ------------------------------------------------------
 * Runs an FFMA2-only kernel on `dev` and returns the best-of-`reps` fp32 TFLOP/s: the live
 * roofline denominator for the Chamfer kernel (MEASURED_PEAKS.json has no fp32 figure).
 */
int ps_measure_fp32_peak(int dev, int reps, double* tflops);
/* Number of kernel launches issued by this library on the calling host thread since the
 * last reset (bench.py reports it as gpu_launches). */
long long ps_launch_count(int reset);

#ifdef __cplusplus
}
#endif
#endif /* POINTSEA_B200_H */
