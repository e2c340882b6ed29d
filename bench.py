#!/usr/bin/env python
"""bench.py — headline measurement of the point-geometry hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scaling weak|strong]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (default, BASELINE.json configs[0], "C1"): Chamfer L2 forward + backward, B=32 clouds per GPU,
partial 2048 points vs ground truth 16384 points, fp32, synthetic `rand - 0.5` clouds.
  step   = ONE launch (ps_chamfer_step, a replayed CUDA graph): key fill, symmetric forward (both directions,
           argmin indices), epilogue (dist/idx + the six loss sums; at N > 1 its last block PUBLISHES the sums
           into every peer's mailbox over NVLink), backward (2 kernels), and at N > 1 a one-warp wait kernel
           that returns the world-wide sums.  The collective is inside the step on every rank, every step.
  value  = 2*B*N*M pair evaluations per step (the reference evaluates both directions) * N_gpus
           / max-over-ranks device time, in Gpair/s, inputs resident in HBM.  The K-step block is repeated
           `--repeats` times (each bracketed by barrier + synchronize, ranks brought into lockstep by 3 untimed
           replayed steps first); the MEDIAN block is reported, all blocks are listed.
  e2e    = the same step through the host-buffer API (chamfer_host_async -> ps_chamfer_host_submit / _wait): clouds
           and upstream gradients come from PINNED HOST buffers (depth + 1 sets in rotation, as a prefetching
           loader would hand them out), and EVERY output goes back to the host — dist, idx, gradients and the loss
           sums (world-wide at N > 1: the peer exchange is one more kernel of the step).  Four steps are in flight
           (--e2e-depth): step i is submitted, then the host joins step i-3 and reads its loss; a step's uploads and
           downloads run on its lane's copy streams, its kernels on the one stream that serves all lanes in order.
           `e2e.per_call` is one call at a time (the latency of a single chamfer_host call); `e2e.loss_readback`
           leaves the gradients on the device and reads back only the loss sums; `e2e.fresh_buffers` hands out a
           NEW address set every step (the cached graph is retargeted in place).
  ops    = the other hot-path ops at their BASELINE configs (C2 FPS+gather, C3 kNN+group, ball query, 3-NN),
           each device-timed, each next to the REFERENCE'S OWN CUDA KERNEL (oracle/_ref, compiled unmodified
           for sm_100a; baseline leg only, never on the product path) timed in the same run: `ref_cuda_ms`,
           `speedup_vs_ref_cuda`.
  roofline = dominant kernel chamfer_sym2_kernel<8,4,2> (+ its fill and epilogue launches): algorithmic 8 flop per
           pair evaluation over the forward's device time against the fp32 FFMA2 peak measured live in this run
           (MEASURED_PEAKS.json carries no fp32 figure); executed_* count each pair once (the kernel evaluates
           it once for both directions).  roofline_hbm = group forward against MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline = pure-PyTorch re-expression on the host cores (oracle/oracle.py), bounded sample.
`--scaling strong` fixes the TOTAL work and splits it over the ranks: `--workload c5` (BASELINE configs[4]:
B=8 clouds of 131072 points, Chamfer fwd+bwd + FPS -> 16384) or `--workload c4loss` (the loss part of configs[3]:
B=32, get_loss = 2 FPS + 3 Chamfer terms + one collective; forward + backward captured once and replayed through
dist.GraphedLoss, the eager autograd call timed beside it as `eager`).
`--impl reference` times the CPU expression alone (the reference has no CPU kernel of its own;
metrics/CD/chamfer_python.py is its pure-torch restatement) on the same config/metric, full B=32 per step.
`--steps K` is the number of timed steps of the headline in all: the `--repeats` blocks share them (default 140 = 7
blocks of 20).  The side measurements size their own loops from K: the forward-only roofline timing max(10, K) launches,
e2e K calls one at a time, 3 blocks of K overlapped steps and K loss-readback calls, fresh buffers max(K, 24) calls,
serial max(3, K // 4) calls.
`--dump-outputs DIR` writes what the timed step returned in its last timed run (rank 0's share) as DIR/<name>.npy,
float32 / float64 (indices as float64, exact); the inputs are seeded, so two builds can be compared output for output.
Inside the tree, `bench_outputs/` is the git-ignored place for them.
"""
import argparse
import importlib.util
import json
import os
import os.path as osp
import statistics
import sys
import threading
import time

ROOT = osp.dirname(osp.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: nothing is written next to the sources

import numpy as np  # noqa: E402
import torch  # noqa: E402

C1 = dict(B=32, N=2048, M=16384)
C2 = dict(B=32, N=16384, npoint=2048)
C3 = dict(B=32, N=2048, S=2048, k=16, C=128)
C5 = dict(B=8, N=131072, M=131072, npoint=16384)
FLOP_PER_PAIR = 8  # 3 sub, 1 mul, 2 fma (SURVEY.md 8d)
WORKLOADS = {
    "c1": "C1 chamfer L2 fwd+bwd B=32/GPU, 2048 vs 16384 pts, fp32 (PCN eval shape)",
    "c1_strong": "C1 chamfer L2 fwd+bwd, B=32 TOTAL split over the ranks, 2048 vs 16384 pts, fp32",
    "c5": "C5 stress: chamfer L2 fwd+bwd, B=8 TOTAL split over the ranks, 131072 vs 131072 pts, fp32",
    "c4loss": "C4 loss part: get_loss (2 FPS + 3 Chamfer terms fwd+bwd + one collective), B=32 TOTAL split over the ranks",
}


def measured_peaks():
    p = osp.join(ROOT, "MEASURED_PEAKS.json")
    if osp.exists(p):
        with open(p) as f:
            return json.load(f), "MEASURED_PEAKS.json"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def make_cloud(g, B, N):
    return (torch.rand(B, N, 3, generator=g) - 0.5).contiguous()


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it is a plain list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = index
            if vis:
                try:
                    phys = int(vis.split(",")[index])
                except Exception:
                    phys = index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=1.0)
        busy = [s for s in self.samples if s > 300] or self.samples
        return {"sm_mhz": statistics.median(busy) if busy else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def timed(fn, iters, warmup, flush):
    """CUDA-event timing of fn() on the current stream: list of ms, L2 flushed between iterations."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(iters):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def timed_pipelined(fn, iters, warmup, flush):
    """Same, but the host never waits inside the loop (events are read after one final synchronize): this is
    how a training loop issues steps, and what lets a host-side cost overlap the previous step's device work."""
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    evs = []
    for i in range(iters):
        flush()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(warmup + i)
        e1.record()
        evs.append((e0, e1))
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in evs]


def dump_outputs(out_dir, arrays):
    """{name: tensor} -> out_dir/<name>.npy, floating point kept as is (float32 / float64), integers as float64."""
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy()
        np.save(osp.join(out_dir, name + ".npy"), a if a.dtype in (np.float32, np.float64) else a.astype(np.float64))


def block_sizes(steps, repeats):
    """`steps` timed steps split into at most `repeats` blocks of near-equal length."""
    n = max(1, min(repeats, steps))
    return [steps // n + (1 if i < steps % n else 0) for i in range(n)]


def max_over_ranks(x, dev, world, dist):
    t = torch.tensor([x], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    import svdformer_pointsea_b200 as ps
    from svdformer_pointsea_b200 import _lib as L
    from svdformer_pointsea_b200 import pointnet2_utils as pu
    from svdformer_pointsea_b200.dist import PeerComm, PipelinedSums

    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_cpus = None
    if world > 1:
        from svdformer_pointsea_b200.dist import bind_to_gpu_numa_node
        numa_cpus = bind_to_gpu_numa_node(local_rank)  # before any pinned allocation (first touch)
        # NCCL writes its version banner / warnings to stdout by default; rank 0 must print ONE JSON line there
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)  # plumbing: barrier, max-over-ranks of the timings, handle exchange
    ps.load_library()
    peaks, peaks_src = measured_peaks()

    # ---- the collective ------------------------------------------------------------------------
    reduce_mode, comm, comm_note = "none (1 GPU)", None, None
    if world > 1:
        reduce_mode = args.reduce
        if reduce_mode == "peer":
            try:
                comm = PeerComm()
            except Exception as e:  # CUDA IPC unavailable in this container: NCCL inside a captured graph instead
                comm_note = f"PeerComm unavailable ({type(e).__name__}: {str(e)[:160]}); fell back to nccl_graph"
                ok = torch.tensor([0.0], device=dev)
            else:
                ok = torch.tensor([1.0], device=dev)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if ok.item() < 1:
                if comm is not None:
                    comm.close()
                comm, reduce_mode = None, "nccl_graph"

    # ---- workload ------------------------------------------------------------------------------
    if args.scaling == "weak":
        wl, B, N, M = "c1", C1["B"], C1["N"], C1["M"]
        Btot = B * world
    else:
        wl = args.workload
        if wl == "c4loss":
            return run_c4loss(args, ps, dist, dev, rank, world, comm, reduce_mode)
        shape = C5 if wl == "c5" else C1
        wl = "c5" if wl == "c5" else "c1_strong"
        Btot, N, M = shape["B"], shape["N"], shape["M"]
        if Btot % world:
            raise SystemExit(f"--scaling strong: {Btot} clouds do not split over {world} ranks")
        B = Btot // world
    g = torch.Generator().manual_seed(1234 + 1 + rank)
    NSETS = 3  # host-buffer sets handed out in rotation by the e2e loops
    h_sets = [tuple(t.pin_memory() for t in (make_cloud(g, B, N), make_cloud(g, B, M), torch.randn(B, N, generator=g),
                                             torch.randn(B, M, generator=g))) for _ in range(NSETS + 1)]
    h_x1, h_x2, h_gd1, h_gd2 = h_sets[0]
    x1, x2, gd1, gd2 = (t.to(dev) for t in (h_x1, h_x2, h_gd1, h_gd2))
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # 256 MB > 126 MB L2

    def flush():
        flush_buf.zero_()

    launches_per_step = [0]
    out_names = ("dist1", "dist2", "idx1", "idx2", "gradxyz1", "gradxyz2", "loss_sums")
    if reduce_mode in ("none (1 GPU)", "peer"):
        stepper = ps.ChamferStep(B, N, M, dev, comm=comm)
        stepper.prepare(x1, x2, gd1, gd2)  # capture + instantiate outside any loop

        def step():
            stepper(x1, x2, gd1, gd2)  # ONE cudaGraphLaunch

        def outputs():
            s = stepper
            return dict(zip(out_names, (s.dist1, s.dist2, s.idx1, s.idx2, s.gradxyz1, s.gradxyz2, s.sums_global)))
    elif reduce_mode == "nccl_graph":
        # the same five kernels + ncclAllReduce captured into one torch CUDA graph
        fwd_out = (torch.empty(B, N, device=dev), torch.empty(B, M, device=dev),
                   torch.empty(B, N, device=dev, dtype=torch.int32), torch.empty(B, M, device=dev, dtype=torch.int32))
        bwd_out = (torch.empty(B, N, 3, device=dev), torch.empty(B, M, 3, device=dev))
        sums = torch.zeros(6, device=dev, dtype=torch.float64)
        gsum = torch.zeros(6, device=dev, dtype=torch.float64)

        def eager():
            d1, d2, i1, i2 = ps.chamfer_forward(x1, x2, out=fwd_out, sums=sums)
            gsum.copy_(sums)
            dist.all_reduce(gsum, op=dist.ReduceOp.SUM)
            ps.chamfer_backward(x1, x2, gd1, gd2, i1, i2, out=bwd_out)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                eager()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        graph = torch.cuda.CUDAGraph()
        L.launch_count(reset=True)
        with torch.cuda.graph(graph, stream=side):
            eager()
        launches_per_step[0] = L.launch_count(reset=True)

        def step():
            graph.replay()

        def outputs():
            return dict(zip(out_names, fwd_out + bwd_out + (gsum,)))
    else:  # "pipelined" / "inline": round 1's eager issue, kept for A/B
        reducer = PipelinedSums()
        fwd_out = (torch.empty(B, N, device=dev), torch.empty(B, M, device=dev),
                   torch.empty(B, N, device=dev, dtype=torch.int32), torch.empty(B, M, device=dev, dtype=torch.int32))
        bwd_out = (torch.empty(B, N, 3, device=dev), torch.empty(B, M, 3, device=dev))
        sum_bufs = [torch.empty(6, device=dev, dtype=torch.float64) for _ in range(2)]
        step_no = [0]

        def step():
            vec = sum_bufs[step_no[0] & 1]
            step_no[0] += 1
            d1, d2, i1, i2 = ps.chamfer_forward(x1, x2, out=fwd_out, sums=vec)
            if reduce_mode == "inline":
                dist.all_reduce(vec, op=dist.ReduceOp.SUM)
            ps.chamfer_backward(x1, x2, gd1, gd2, i1, i2, out=bwd_out)
            if reduce_mode == "pipelined":
                reducer.submit(vec)

        def outputs():
            return dict(zip(out_names, fwd_out + bwd_out + (sum_bufs[(step_no[0] - 1) & 1],)))

    # ---- warm-up, fp32 peak, forward-only timing for the roofline ------------------------------
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    fp32_peak = L.measure_fp32_peak(local_rank, 5)
    fwd_bufs = (torch.empty(B, N, device=dev), torch.empty(B, M, device=dev),
                torch.empty(B, N, device=dev, dtype=torch.int32), torch.empty(B, M, device=dev, dtype=torch.int32))
    fwd_ms = timed(lambda: ps.chamfer_forward(x1, x2, out=fwd_bufs), max(10, args.steps), 3, flush)
    fwd_avg_ms = sum(fwd_ms) / len(fwd_ms)

    # ---- the timed K-step blocks ---------------------------------------------------------------
    # everything with a variable host cost (NVML initialisation of the clock sampler) happens BEFORE the barrier
    sampler = ClockSampler(local_rank)
    sampler.start()
    blocks, host_ms_blocks, launches = [], [], 0
    for nsteps in block_sizes(args.steps, args.repeats):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        for _ in range(3):  # untimed, replayed: the collective inside each step brings the ranks into lockstep
            step()
        torch.cuda.synchronize()
        L.launch_count(reset=True)
        evs = []
        t_host0 = time.perf_counter()
        for _ in range(nsteps):
            flush()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step()
            e1.record()
            evs.append((e0, e1))
        t_issue = time.perf_counter() - t_host0
        torch.cuda.synchronize()
        launches = L.launch_count(reset=True) + launches_per_step[0] * nsteps
        if world > 1:
            dist.barrier()
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        blocks.append(max_over_ranks(total_ms, dev, world, dist) / nsteps)
        host_ms_blocks.append(t_issue * 1e3 / nsteps)
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs())
    ms_per_step = statistics.median(blocks)
    pairs_per_step = 2.0 * B * N * M
    value = pairs_per_step * world / (ms_per_step * 1e-3) / 1e9  # Gpair/s, whole job
    comm_status = comm.status() if comm is not None else None

    # ---- e2e: host buffers in, host buffers out ------------------------------------------------
    def host_outs():
        return [torch.empty(B, N).pin_memory(), torch.empty(B, M).pin_memory(),
                torch.empty(B, N, dtype=torch.int32).pin_memory(), torch.empty(B, M, dtype=torch.int32).pin_memory(),
                torch.empty(B, N, 3).pin_memory(), torch.empty(B, M, 3).pin_memory()]

    h_outs = [host_outs() for _ in range(NSETS)]
    h_sums = [torch.empty(6, dtype=torch.float64).pin_memory() for _ in range(NSETS)]
    bwd_dev = (torch.empty(B, N, 3, device=dev), torch.empty(B, M, 3, device=dev))
    h2d = sum(t.numel() * t.element_size() for t in h_sets[0])
    d2h_full = sum(t.numel() * t.element_size() for t in h_outs[0]) + 48

    def e2e_full(i):
        s = i % NSETS
        a, b, ga, gb = h_sets[s]
        ps.chamfer_host(a, b, ga, gb, out=h_outs[s], chunk=args.e2e_chunk, blocking=False, sums_out=h_sums[s], comm=comm)

    def e2e_loss(i):
        s = i % NSETS
        a, b, ga, gb = h_sets[s]
        ps.chamfer_host_step(a, b, ga, gb, grad_out=bwd_dev, sums_out=h_sums[s], chunk=args.e2e_chunk, blocking=False, comm=comm)

    def e2e_serial(i):
        a, b, ga, gb = (t.to(dev, non_blocking=True) for t in h_sets[i % NSETS])
        d1, d2, i1, i2 = ps.chamfer_forward(a, b)
        g1, g2 = ps.chamfer_backward(a, b, ga, gb, i1, i2)
        for dst, src in zip(h_outs[i % NSETS], (d1, d2, i1, i2, g1, g2)):
            dst.copy_(src, non_blocking=True)

    DEPTH = max(1, min(4, args.e2e_depth))  # steps in flight in the e2e loop
    OSETS = DEPTH + 1                       # buffer sets: DEPTH in flight + the one the host is reading
    while len(h_sets) < OSETS:
        h_sets.append(tuple(t.clone().pin_memory() for t in h_sets[len(h_sets) % NSETS]))
    while len(h_outs) < OSETS:
        h_outs.append(host_outs())
        h_sums.append(torch.empty(6, dtype=torch.float64).pin_memory())

    def e2e_overlapped(nsteps, warm):
        """Loop over chamfer_host_async with DEPTH steps in flight: step i is submitted, then the host joins step
        i-DEPTH+1 (blocks until its last output byte is in host memory) and reads its loss — upload and kernels of
        the younger steps overlap the download of the older ones.  Returns the device time of the whole block (CUDA
        events on the submitting stream: the first recorded before the first submission, the last after a
        stream-side join of the last step), the host's wall clock around the same block (ms) and a checksum."""
        import collections
        cur = torch.cuda.current_stream()

        def submit(i):
            s = i % OSETS
            a, b, ga, gb = h_sets[s]
            return ps.chamfer_host_async(a, b, ga, gb, out=h_outs[s], chunk=args.e2e_chunk, sums_out=h_sums[s], comm=comm)

        pending, seen = collections.deque(), 0.0
        for i in range(warm):
            pending.append(submit(i))
            if len(pending) == DEPTH:
                pending.popleft().synchronize()
        while pending:
            pending.popleft().synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(cur)
        for i in range(warm, warm + nsteps):
            pending.append(submit(i))
            if len(pending) == DEPTH:
                st = pending.popleft()
                st.synchronize()
                seen += float(st.sums[2])  # the step's result, read on the host
        for st in pending:
            st.wait(cur)
        e1.record(cur)
        while pending:
            st = pending.popleft()
            st.synchronize()
            seen += float(st.sums[2])
        wall = (time.perf_counter() - t0) * 1e3
        e1.synchronize()
        return e0.elapsed_time(e1), wall, seen

    if world > 1:
        dist.barrier()
    full_ms = timed_pipelined(e2e_full, args.steps, max(args.warmup, 3), flush)
    call_ms = max_over_ranks(sum(full_ms), dev, world, dist) / args.steps
    ov_blocks, ov_wall = [], []
    for _ in range(3):
        dms, wms, _seen = e2e_overlapped(args.steps, max(args.warmup, 3, 4 * OSETS))  # every (buffer set, lane) pair captured before the timed block
        ov_blocks.append(max_over_ranks(dms, dev, world, dist) / args.steps)
        ov_wall.append(max_over_ranks(wms, dev, world, dist) / args.steps)
    e2e_ms = statistics.median(ov_blocks)
    loss_ms_l = timed_pipelined(e2e_loss, args.steps, max(args.warmup, 3), flush)
    loss_ms = max_over_ranks(sum(loss_ms_l), dev, world, dist) / args.steps
    e2e = {"value": round(pairs_per_step * world / (e2e_ms * 1e-3) / 1e9, 2), "unit": "Gpair/s",
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_full, "ms_per_step": round(e2e_ms, 4),
           "api": "svdformer_pointsea_b200.chamfer_host_async(..., sums_out, comm) -> ps_chamfer_host_submit / ps_chamfer_host_wait: pinned "
                  "host clouds + upstream gradients in; dist, idx, gradients AND the loss sums out (world-wide sums at N > 1: the "
                  "peer-memory exchange is one more kernel of the step); a step = uploads on its lane's copy stream -> its kernels, "
                  "replayed as one CUDA graph on the stream that serves ALL lanes in submission order (one step at a time, each with "
                  "the whole GPU) -> downloads on the lane's copy stream; %d steps in flight: step i is submitted, then the host joins "
                  "step i-%d and reads its loss, so the copy engines work on the neighbouring steps while the SMs work on this one"
                  % (DEPTH, DEPTH - 1),
           "timing": f"median of 3 blocks of {args.steps} steps; a block = CUDA events around all of its steps on the submitting stream "
                     f"(max over ranks); every input byte crosses PCIe inside its own step, {OSETS} rotating pinned buffer sets, nothing "
                     "is reused across steps (no L2 flush needed)",
           "blocks_ms_per_step": [round(b, 4) for b in ov_blocks], "host_wall_ms_per_step": round(statistics.median(ov_wall), 4),
           "per_call": {"value": round(pairs_per_step * world / (call_ms * 1e-3) / 1e9, 2), "ms_per_step": round(call_ms, 4),
                        "note": "one step at a time through chamfer_host(..., blocking=False): CUDA events around each call, L2 flushed "
                                "between calls; the latency of a single call (round-2 headline before the asynchronous pair existed)"},
           "steps_in_flight": DEPTH, "host_buffer_sets": OSETS, "chunk": args.e2e_chunk, "numa_bound_cpus": (len(numa_cpus) if numa_cpus else None),
           "loss_readback": {"value": round(pairs_per_step * world / (loss_ms * 1e-3) / 1e9, 2), "ms_per_step": round(loss_ms, 4),
                             "d2h_bytes_per_step": 48,
                             "note": "chamfer_host_step, ONE CALL AT A TIME (compare with per_call, not with value): gradients stay in device buffers "
                                     "for the optimizer, only the six loss sums are read back"}}
    if world == 1 and not args.quick:
        # a loader that never reuses a buffer: 2*cache-size address sets, every call re-captures and RETARGETS a cached graph
        nfresh = 16
        fresh = [tuple(t.clone().pin_memory() for t in h_sets[0]) for _ in range(nfresh)]
        fresh_out = [host_outs() for _ in range(nfresh)]
        fresh_sums = [torch.empty(6, dtype=torch.float64).pin_memory() for _ in range(nfresh)]
        st0 = L.graph_stats(local_rank, "host")

        def e2e_fresh(i):
            s = i % nfresh
            a, b, ga, gb = fresh[s]
            ps.chamfer_host(a, b, ga, gb, out=fresh_out[s], chunk=args.e2e_chunk, blocking=False, sums_out=fresh_sums[s])

        fr = timed_pipelined(e2e_fresh, max(args.steps, 24), nfresh, flush)
        st1 = L.graph_stats(local_rank, "host")
        e2e["fresh_buffers"] = {"ms_per_step": round(sum(fr) / len(fr), 4), "address_sets": nfresh,
                                "graph_updates": st1["updates"] - st0["updates"], "graph_instantiations": st1["instantiations"] - st0["instantiations"],
                                "note": "a new host-buffer address set every step: the call is re-captured and the cached executable "
                                        "updated in place (cudaGraphExecUpdate); full readback, one call at a time (compare with per_call)"}
        ser = timed_pipelined(e2e_serial, max(3, args.steps // 4), 3, flush)
        e2e["serial_ms_per_step"] = round(sum(ser) / len(ser), 4)
        e2e["serial_note"] = "same work as copy-in, device entry points, copy-out on one stream (no overlap)"

    result = {
        "metric": "chamfer_fwd_bwd_gpair_per_s", "value": round(value, 2), "unit": "Gpair/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 4),
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS[wl], "B_per_gpu": B, "B_total": Btot, "N": N, "M": M,
                   "l2": "256 MB buffer written between timed iterations (L2 flush)",
                   "collective": {"none (1 GPU)": "none (1 GPU)",
                                  "peer": "every step, inside the step's graph: the forward epilogue's last block stores the 6 loss sums into all peers' "
                                          "mailboxes over NVLink (CUDA IPC peer memory), a one-warp kernel after the backward adds them in rank order",
                                  "nccl_graph": "every step: ncclAllReduce of the 6 loss sums captured inside the step's CUDA graph",
                                  "pipelined": "c10d all-reduce issued asynchronously and joined one step later (round-1 path)",
                                  "inline": "c10d all-reduce in line between forward and backward (round-1 A/B path)"}[reduce_mode],
                   "timing": f"{args.steps} timed steps in {len(blocks)} blocks, median block; each block: barrier + synchronize, 3 untimed "
                             "lockstep steps, then its steps timed with CUDA events, max over ranks",
                   "parallelism": f"batch-sharded x{world}"},
        "blocks_ms_per_step": [round(b, 4) for b in blocks],
        "spread": {"min": round(min(blocks), 4), "max": round(max(blocks), 4), "median": round(ms_per_step, 4)},
        "e2e": e2e,
        "gpu_launches": int(launches), "launches_note": "kernels inside the replayed graph(s) of the last timed block; ONE cudaGraphLaunch per step",
        "host_issue_ms_per_step": round(statistics.median(host_ms_blocks), 4), "reduce": reduce_mode,
        "clocks": clocks,
        "roofline": {"kernel": "chamfer_sym2_kernel<8,4,2> (+ key fill and epilogue launches): forward, both directions in one pass", "bound": "fp32",
                     "achieved": round(pairs_per_step * FLOP_PER_PAIR / (fwd_avg_ms * 1e-3) / 1e12, 2),
                     "peak": round(fp32_peak, 2), "unit": "TFLOP/s",
                     "frac": round(pairs_per_step * FLOP_PER_PAIR / (fwd_avg_ms * 1e-3) / 1e12 / fp32_peak, 4),
                     "peak_source": "FFMA2 microkernel measured live in this run (MEASURED_PEAKS.json has no fp32 figure)",
                     "note": "achieved/frac count the ALGORITHMIC 2*B*N*M pair evaluations x 8 flop, as the reference executes them. The kernel "
                             "evaluates each (a,b) pair ONCE for both directions, so what the FP32 pipe EXECUTES is half of that: executed_tflops / "
                             "executed_frac (= what ncu's FMA-pipe utilisation corresponds to; ceiling 8/12 because 8 flop take 6 pipe slots).",
                     "executed_tflops": round(0.5 * pairs_per_step * FLOP_PER_PAIR / (fwd_avg_ms * 1e-3) / 1e12, 2),
                     "executed_frac": round(0.5 * pairs_per_step * FLOP_PER_PAIR / (fwd_avg_ms * 1e-3) / 1e12 / fp32_peak, 4),
                     "executed_frac_of_ceiling": round(0.5 * pairs_per_step * FLOP_PER_PAIR / (fwd_avg_ms * 1e-3) / 1e12 / fp32_peak / (8.0 / 12.0), 4),
                     "unique_gpair_per_s": round(0.5 * pairs_per_step / (fwd_avg_ms * 1e-3) / 1e9, 1),
                     "structural_ceiling_frac": round(8.0 / 12.0, 4),
                     "fwd_ms": round(fwd_avg_ms, 4), "fwd_ms_min": round(min(fwd_ms), 4),
                     "gpair_per_s_fwd": round(pairs_per_step / (fwd_avg_ms * 1e-3) / 1e9, 1),
                     "traffic": 11844000 if wl == "c1" else None, "traffic_unit": "bytes per launch (dram read+write)",
                     "traffic_source": "ncu --set full capture of chamfer_sym2_kernel<8,4,2> at the C1 shape (dram read 11.844 MB, write 0: "
                                       "the results leave through L2 in the epilogue launch): profiles/ncu_full_r2_table.txt"},
    }
    if comm_note:
        result["reduce_note"] = comm_note
    if comm_status is not None:
        result["comm"] = comm_status

    # ---- the other hot-path ops at their own configs (rank-local, device-timed) ---------------
    if args.scaling == "strong" and wl == "c5":
        result["ops"] = bench_c5_fps(ps, dev, flush, B, dist, world)
    elif not args.no_ops and not args.quick:
        result["ops"] = bench_ops(ps, pu, dev, flush, peaks, peaks_src, rank, ref_cuda=(rank == 0 and not args.no_ref_cuda))
        result["roofline_hbm"] = result["ops"]["group_fwd"]["roofline"]
    if rank == 0 and world == 1 and not args.no_cpu and not args.quick and args.scaling == "weak":
        result["cpu_baseline"] = cpu_chamfer_baseline(budget_s=12.0)
        if "ops" in result:
            result["ops"]["cpu"] = cpu_ops_baseline()
    if rank == 0:
        emit(result)
    if world > 1:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()


def bench_c5_fps(ps, dev, flush, B, dist, world):
    """C5's second op: FPS 131072 -> 16384 on this rank's clouds (max over ranks)."""
    g = torch.Generator().manual_seed(1234 + 5)
    xyz = make_cloud(g, max(B, 1), C5["N"]).to(dev)
    ms = timed(lambda: ps.furthest_point_sample(xyz, C5["npoint"]), 3, 1, flush)
    t = max_over_ranks(min(ms), dev, world, dist)
    return {"fps": {"config": f"C5 {B} cloud(s)/GPU, 131072 -> 16384", "ms": round(t, 3),
                    "sampled_pts_per_s_whole_job": round(C5["B"] * C5["npoint"] / (t * 1e-3), 1),
                    "us_per_iteration": round(t * 1e3 / (C5["npoint"] - 1), 4)}}


def run_c4loss(args, ps, dist, dev, rank, world, comm, reduce_mode):
    """Strong scaling of the loss part of C4 (utils/loss_utils.get_loss on SVDFormer's PCN outputs: Pc 512, P1 2048,
    P2 16384 points vs gt 16384): B=32 clouds split over the ranks, forward + backward through autograd, one collective."""
    from svdformer_pointsea_b200.dist import get_loss_sharded
    Btot = 32
    if Btot % world:
        raise SystemExit("c4loss: 32 clouds do not split over this world size")
    B = Btot // world
    g = torch.Generator().manual_seed(1234 + 4 + rank)
    gt = make_cloud(g, B, 16384).to(dev)
    preds = [(make_cloud(g, B, n).to(dev)).requires_grad_(True) for n in (512, 2048, 16384)]
    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step():
        loss, _ = get_loss_sharded(preds, gt, sqrt=True, comm=comm)
        loss.backward()
        for p in preds:
            p.grad = None

    # the same step captured once and replayed (GraphedLoss): what a training loop with fixed shapes calls; the copy of
    # the step's clouds into the graph's static inputs is inside the timed call
    from svdformer_pointsea_b200.dist import GraphedLoss
    graphed = GraphedLoss([p.shape for p in preds], gt.shape, sqrt=True, comm=comm if reduce_mode == "peer" else None)

    def step_graphed():
        graphed(preds, gt)

    def timed_blocks(fn):
        for _ in range(max(args.warmup, 3)):
            fn()
        blocks = []
        for nsteps in block_sizes(args.steps, args.repeats):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            fn()
            torch.cuda.synchronize()
            evs = []
            for _ in range(nsteps):
                flush_buf.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                fn()
                e1.record()
                evs.append((e0, e1))
            torch.cuda.synchronize()
            blocks.append(max_over_ranks(sum(a.elapsed_time(b) for a, b in evs), dev, world, dist) / nsteps)
        return blocks

    eager_blocks = timed_blocks(step)
    blocks = timed_blocks(step_graphed)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"loss": graphed.loss.reshape(1), "loss_terms": torch.stack(graphed.terms),
                                         **{f"grad_pred{i}": g for i, g in enumerate(graphed.grads)}})
    ms, eager_ms = statistics.median(blocks), statistics.median(eager_blocks)
    pairs = 2.0 * Btot * (512 * 512 + 2048 * 2048 + 16384 * 16384)
    if rank == 0:
        emit({"metric": "chamfer_fwd_bwd_gpair_per_s", "value": round(pairs / (ms * 1e-3) / 1e9, 2), "unit": "Gpair/s", "n_gpus": world,
              "steps": args.steps, "warmup": max(args.warmup, 3) + 1, "ms_per_step": round(ms, 4), "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
              "config": {"workload": WORKLOADS["c4loss"], "B_per_gpu": B, "B_total": Btot, "reduce": reduce_mode,
                         "l2": "256 MB buffer written between timed iterations (L2 flush)",
                         "api": "svdformer_pointsea_b200.dist.GraphedLoss (get_loss_sharded forward + backward captured once, replayed per step)"},
              "blocks_ms_per_step": [round(b, 4) for b in blocks],
              "eager": {"ms_per_step": round(eager_ms, 4), "blocks_ms_per_step": [round(b, 4) for b in eager_blocks],
                        "api": "get_loss_sharded(...) + loss.backward(), one launch per op"}})
    if world > 1:
        dist.barrier()
        if comm is not None:
            comm.close()
        dist.destroy_process_group()


# ---- the reference's own CUDA kernels (oracle/_ref), baseline leg only ---------------------------
def load_ref_cuda():
    """oracle/_ref/*.so = the reference's unmodified CUDA sources compiled for sm_100a by oracle/build_ref.py.
    Used ONLY as a timed baseline next to our ops (never on the product path).  None when not built."""
    mods = {}
    for name in ("ref_chamfer_3D", "ref_pointnet2_ext"):
        path = osp.join(ROOT, "oracle", "_ref", name + ".so")
        if not osp.exists(path):
            return None
        try:
            spec = importlib.util.spec_from_file_location(name, path)
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            mods[name] = mod
        except Exception:
            return None
    return mods


def torch_query_knn(k, xyz, new_xyz):
    """models/model_utils.py:258-286 (square_distance + argsort) as the reference runs it on the GPU: the kNN baseline."""
    dist = -2 * torch.matmul(new_xyz, xyz.permute(0, 2, 1))
    dist += torch.sum(new_xyz ** 2, -1).view(new_xyz.shape[0], new_xyz.shape[1], 1)
    dist += torch.sum(xyz ** 2, -1).view(xyz.shape[0], 1, xyz.shape[1])
    return torch.argsort(dist, dim=-1, descending=False)[:, :, 0:k].int()


def bench_ops(ps, pu, dev, flush, peaks, peaks_src, rank, ref_cuda=True):
    ref = load_ref_cuda() if ref_cuda else None
    out = {"ref_cuda": "oracle/_ref (the reference's CUDA sources compiled unmodified for sm_100a), timed in this run" if ref
           else "unavailable (oracle/_ref not built)"}

    def vs_ref(entry, ours_ms, ref_fn, iters=5, warm=2):
        if ref is None:
            return
        ms = timed(ref_fn, iters, warm, flush)
        entry["ref_cuda_ms"] = round(min(ms), 4)
        entry["speedup_vs_ref_cuda"] = round(min(ms) / ours_ms, 2)

    g = torch.Generator().manual_seed(1234 + 2 + rank)
    # C1 Chamfer forward and backward against the reference kernels (chamfer3D.cu:12-195)
    a, b = make_cloud(g, C1["B"], C1["N"]).to(dev), make_cloud(g, C1["B"], C1["M"]).to(dev)
    ga, gb = torch.randn(C1["B"], C1["N"], generator=g).to(dev), torch.randn(C1["B"], C1["M"], generator=g).to(dev)
    holder = {}

    def ch_fwd():
        holder["c"] = ps.chamfer_forward(a, b)

    ms = timed(ch_fwd, 10, 3, flush)
    d1, d2, i1, i2 = holder["c"]
    out["chamfer_fwd"] = {"config": "C1 B=32 2048 vs 16384", "ms": round(min(ms), 4)}
    if ref is not None:
        r = [torch.zeros_like(d1), torch.zeros_like(d2), torch.zeros_like(i1), torch.zeros_like(i2)]
        vs_ref(out["chamfer_fwd"], min(ms), lambda: ref["ref_chamfer_3D"].forward(a, b, *r))
        out["chamfer_fwd"]["bit_identical_to_ref_cuda"] = bool(torch.equal(d1, r[0]) and torch.equal(d2, r[1]) and torch.equal(i1, r[2]) and torch.equal(i2, r[3]))
    ms = timed(lambda: ps.chamfer_backward(a, b, ga, gb, i1, i2), 10, 3, flush)
    out["chamfer_bwd"] = {"config": "C1", "ms": round(min(ms), 4),
                          "gbs": round(C1["B"] * (C1["N"] + C1["M"]) * 32 / (min(ms) * 1e-3) / 1e9, 1)}
    if ref is not None:
        g1, g2 = torch.zeros_like(a), torch.zeros_like(b)

        def ref_bwd():
            g1.zero_(); g2.zero_()  # the reference needs pre-zeroed gradients (dist_chamfer_3D.py:56-60)
            ref["ref_chamfer_3D"].backward(a, b, g1, g2, ga, gb, i1, i2)
        vs_ref(out["chamfer_bwd"], min(ms), ref_bwd)
    del a, b, ga, gb, d1, d2, i1, i2
    # C2: FPS + gather
    xyz = make_cloud(g, C2["B"], C2["N"]).to(dev)
    xyz_t = xyz.transpose(1, 2).contiguous()

    def fps_fn():
        holder["idx"] = ps.furthest_point_sample(xyz, C2["npoint"])

    ms = timed(fps_fn, 5, 2, flush)
    t = min(ms) * 1e-3
    out["fps"] = {"config": "C2 B=32 N=16384 -> 2048", "ms": round(min(ms), 4), "ms_median": round(statistics.median(ms), 4),
                  "sampled_pts_per_s": round(C2["B"] * C2["npoint"] / t, 1),
                  "gpair_per_s": round(C2["B"] * (C2["npoint"] - 1) * C2["N"] / t / 1e9, 2),
                  "us_per_iteration": round(t * 1e6 / (C2["npoint"] - 1), 4),
                  "bound": "latency: a serial chain of npoint-1 cluster-wide argmax rounds (DESIGN.md 4.3)"}
    idx = holder["idx"]
    if ref is not None:
        vs_ref(out["fps"], min(ms), lambda: holder.__setitem__("ridx", ref["ref_pointnet2_ext"].furthest_point_sampling(xyz, C2["npoint"])), iters=3, warm=1)
        out["fps"]["bit_identical_to_ref_cuda"] = bool(torch.equal(idx, holder["ridx"]))
    ms = timed(lambda: ps.gather_operation(xyz_t, idx), 20, 3, flush)
    byts = 4 * (C2["B"] * C2["npoint"] + 2 * C2["B"] * 3 * C2["npoint"])
    out["gather_fwd"] = {"config": "C2 (32,3,16384) -> (32,3,2048)", "ms": round(min(ms), 4),
                         "gbs": round(byts / (min(ms) * 1e-3) / 1e9, 2), "note": "launch-latency bound (1.8 MB)"}
    vs_ref(out["gather_fwd"], min(ms), lambda: ref["ref_pointnet2_ext"].gather_points(xyz_t, idx), iters=10)
    ms = timed(lambda: holder.__setitem__("fs", pu.fps_subsample(xyz, C2["npoint"])), 5, 2, flush)
    out["fps_subsample_fused"] = {"config": "C2 FPS + gather in one kernel (ps_fps_sample; models/model_utils.py:489-499)", "ms": round(min(ms), 4)}
    # C3: kNN + group
    g = torch.Generator().manual_seed(1234 + 3 + rank)
    pts = make_cloud(g, C3["B"], C3["N"]).to(dev)
    feat = torch.randn(C3["B"], C3["C"], C3["N"], generator=g).to(dev)

    def knn_fn():
        holder["knn"] = ps.query_knn(C3["k"], pts, pts)

    ms = timed(knn_fn, 10, 3, flush)
    t = min(ms) * 1e-3
    knn_pairs = C3["B"] * C3["S"] * C3["N"]
    out["knn"] = {"config": "C3 B=32 N=S=2048 k=16", "ms": round(min(ms), 4), "ms_median": round(statistics.median(ms), 4),
                  "query_pts_per_s": round(C3["B"] * C3["S"] / t, 1), "gpair_per_s": round(knn_pairs / t / 1e9, 2),
                  "roofline": {"bound": "fp32 + selection", "pair_evals": knn_pairs, "flop_per_pair": 8,
                               "achieved_tflops": round(knn_pairs * 8 / t / 1e12, 2),
                               "note": "distance arithmetic alone would take pair_evals x 6 FP32-pipe slots; the kernel evaluates every pair "
                                       "TWICE (threshold pass + compaction pass) and is bound by the selection's fixed-latency chain, not by "
                                       "the FP32 pipe (ncu r1: issue 59-74 %, fma pipe ~20 %): ~10 % of fp32 peak by design"}}
    kidx = holder["knn"]
    ms_ref = timed(lambda: torch_query_knn(C3["k"], pts, pts), 5, 2, flush)
    out["knn"]["ref_torch_cuda_ms"] = round(min(ms_ref), 4)
    out["knn"]["speedup_vs_ref_torch_cuda"] = round(min(ms_ref) / min(ms), 2)
    out["knn"]["ref_note"] = "the reference has no kNN kernel: models/model_utils.py:258-286 (matmul + argsort) run by torch on this GPU"

    def grp_fn():
        holder["grp"] = pu.group_raw(feat, kidx)

    ms = timed(grp_fn, 20, 3, flush)
    byts = 4 * (C3["B"] * C3["S"] * C3["k"] + C3["B"] * C3["C"] * C3["N"] + C3["B"] * C3["C"] * C3["S"] * C3["k"])
    t = statistics.median(ms) * 1e-3
    out["group_fwd"] = {"config": "C3 (32,128,2048) x idx (32,2048,16) -> (32,128,2048,16)", "ms": round(min(ms), 4),
                        "ms_median": round(statistics.median(ms), 4),
                        "roofline": {"kernel": "gather_staged_kernel (grouping_operation forward)", "bound": "hbm",
                                     "achieved": round(byts / t / 1e9, 1), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                     "frac": round(byts / t / 1e9 / peaks["hbm_gbs"], 4), "peak_source": peaks_src,
                                     "algorithmic_bytes": byts, "traffic": 515676000,
                                     "traffic_source": "ncu --set full capture (dram read 37.8 MB + write 477.9 MB; the rest of the "
                                                       "output is still in L2 at kernel end): profiles/ncu_full_r1_table.txt"}}
    vs_ref(out["group_fwd"], min(ms), lambda: ref["ref_pointnet2_ext"].group_points(feat, kidx), iters=5)
    go = torch.randn_like(holder["grp"])
    ms = timed(lambda: pu.group_grad_raw(go, kidx, C3["N"]), 20, 3, flush)
    t = statistics.median(ms) * 1e-3
    out["group_bwd"] = {"ms": round(min(ms), 4), "ms_median": round(statistics.median(ms), 4),
                        "gbs": round(byts / t / 1e9, 1), "frac_hbm": round(byts / t / 1e9 / peaks["hbm_gbs"], 4)}
    vs_ref(out["group_bwd"], min(ms), lambda: ref["ref_pointnet2_ext"].group_points_grad(go, kidx, C3["N"]), iters=5)
    del go, holder
    # ball query + 3-NN + interpolation (pointnet2 API surface; ball_query_gpu.cu:9-44, interpolate_gpu.cu:9-154)
    ctr = pts[:, :512].contiguous()
    ms = timed(lambda: ps.ball_query(0.2, 32, pts, ctr), 10, 3, flush)
    out["ball_query"] = {"config": "B=32 N=2048 S=512 r=0.2 nsample=32", "ms": round(min(ms), 4), "bound": "latency (one warp per centre, ballot scan)"}
    vs_ref(out["ball_query"], min(ms), lambda: ref["ref_pointnet2_ext"].ball_query(ctr, pts, 0.2, 32))
    tn = {}
    ms = timed(lambda: tn.__setitem__("r", ps.three_nn(pts, ctr)), 10, 3, flush)
    out["three_nn"] = {"config": "B=32 unknown 2048, known 512", "ms": round(min(ms), 4),
                       "gpair_per_s": round(32 * 2048 * 512 / (min(ms) * 1e-3) / 1e9, 1), "bound": "fp32 + 3-way insertion chain"}
    vs_ref(out["three_nn"], min(ms), lambda: ref["ref_pointnet2_ext"].three_nn(pts, ctr))
    d3, i3 = tn["r"]
    w3 = torch.softmax(-d3, dim=2).contiguous()
    f512 = feat[:, :, :512].contiguous()
    ms = timed(lambda: ps.three_interpolate(f512, i3, w3), 10, 3, flush)
    byts3 = 4 * (32 * 128 * 512 + 32 * 2048 * 3 * 2 + 32 * 128 * 2048)
    out["three_interpolate"] = {"config": "B=32 C=128 512 -> 2048", "ms": round(min(ms), 4), "gbs": round(byts3 / (min(ms) * 1e-3) / 1e9, 1), "bound": "hbm / latency (37 MB)"}
    vs_ref(out["three_interpolate"], min(ms), lambda: ref["ref_pointnet2_ext"].three_interpolate(f512, i3, w3))
    # SURVEY 8(f) rows at the models' shapes (EdgeConv of SVDFormer's local encoder; PCN evaluation)
    from svdformer_pointsea_b200 import model_ops as mo
    g = torch.Generator().manual_seed(1234 + 6 + rank)
    nxt = {}
    for (Cc, Nn, kk) in ((64, 512, 8), (256, 512, 4)):
        x = torch.randn(32, Cc, Nn, generator=g).to(dev)
        eidx = mo.knn_self(x, kk)
        ms = timed(lambda: mo.knn_self(x, kk), 10, 3, flush)
        nxt[f"feature_knn_C{Cc}"] = {"config": f"B=32 C={Cc} N={Nn} k={kk} (torch.topk order)", "ms": round(min(ms), 4),
                                     "gpair_per_s": round(32 * Nn * Nn / (min(ms) * 1e-3) / 1e9, 1),
                                     "tflops": round(2.0 * Cc * 32 * Nn * Nn / (min(ms) * 1e-3) / 1e12, 2)}
        if Cc == 64:
            ms = timed(lambda: mo.edge_features_raw(x, eidx), 20, 3, flush)
            byts = 4 * (32 * Nn * kk + 32 * Cc * Nn + 2 * 32 * Cc * Nn * kk)
            nxt["edge_features_fwd"] = {"config": "B=32 C=64 N=512 k=8 -> (32,128,512,8)", "ms": round(min(ms), 4),
                                        "gbs": round(byts / (statistics.median(ms) * 1e-3) / 1e9, 1)}
    gt = make_cloud(g, 32, 16384).to(dev)
    pred = gt + 0.004 * torch.randn(32, 16384, 3, generator=g).to(dev)
    d1, d2, i1, i2 = ps.chamfer_forward(gt, pred)
    ms = timed(lambda: ps.chamfer_metrics_raw(d1, d2, i1, i2), 20, 3, flush)
    nxt["metrics_epilogue"] = {"config": "calc_cd + fscore + calc_dcd, B=32, 16384 vs 16384", "ms": round(min(ms), 4)}
    out["next"] = nxt
    return out


# ------------------------------------------------------------------------------------------------
def _cpu_chamfer_once(bs, seed=1234 + 1):
    from oracle import oracle as O
    g = torch.Generator().manual_seed(seed)
    a, b = make_cloud(g, bs, C1["N"]), make_cloud(g, bs, C1["M"])
    gd1, gd2 = torch.randn(bs, C1["N"], generator=g), torch.randn(bs, C1["M"], generator=g)
    t0 = time.perf_counter()
    O.torch_chamfer_fwd_bwd(a, b, gd1, gd2)
    return time.perf_counter() - t0


def cpu_chamfer_baseline(budget_s=12.0):
    """Pure-torch direct-form Chamfer fwd+bwd on the host cores, bounded sample of C1."""
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    _cpu_chamfer_once(1)  # warm the allocator / thread pool
    t1 = _cpu_chamfer_once(1)
    bs = int(max(1, min(C1["B"], budget_s / max(t1, 1e-3))))
    t = _cpu_chamfer_once(bs)
    pairs = 2.0 * bs * C1["N"] * C1["M"]
    return {"value": round(pairs / t / 1e9, 4), "unit": "Gpair/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"{bs} of the 32 C1 clouds (2048 vs 16384), pure-torch direct-form fwd+bwd (autograd), {t:.2f} s"}


def cpu_ops_baseline():
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    out = {"cores": torch.get_num_threads()}
    g = torch.Generator().manual_seed(1234 + 2)
    xyz = make_cloud(g, C2["B"], C2["N"])
    npnt = 128  # iterations have uniform cost: time 127 of the 2047 and scale
    t0 = time.perf_counter(); O.torch_fps(xyz, npnt); t = time.perf_counter() - t0
    full = t * (C2["npoint"] - 1) / (npnt - 1)
    out["fps"] = {"sampled_pts_per_s": round(C2["B"] * C2["npoint"] / full, 1),
                  "sample": f"127 of 2047 iterations at B=32 N=16384 ({t:.2f} s), scaled"}
    g = torch.Generator().manual_seed(1234 + 3)
    pts = make_cloud(g, 8, C3["N"])
    t0 = time.perf_counter(); kidx = O.torch_knn(C3["k"], pts, pts); t = time.perf_counter() - t0
    out["knn"] = {"query_pts_per_s": round(8 * C3["S"] / t, 1), "sample": f"8 of 32 clouds ({t:.2f} s)"}
    feat = torch.randn(8, C3["C"], C3["N"], generator=g)
    t0 = time.perf_counter(); O.torch_group(feat, kidx); t = time.perf_counter() - t0
    byts = 4 * (8 * C3["S"] * C3["k"] + 8 * C3["C"] * C3["N"] + 8 * C3["C"] * C3["S"] * C3["k"])
    out["group_fwd"] = {"gbs": round(byts / t / 1e9, 2), "sample": f"8 of 32 clouds ({t:.2f} s)"}
    return out


def run_reference(args):
    """Reference arm: the path's CPU expression (pure torch, all host threads) on C1's metric, the full B=32 step."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    bs = args.ref_clouds if args.ref_clouds > 0 else C1["B"]
    warm = max(args.warmup, 1)
    budget = float(os.environ.get("PS_REF_BUDGET_S", 240))  # whole-run bound: fewer steps, never a smaller batch
    t_first = _cpu_chamfer_once(bs)
    warm_done = 1
    while warm_done < warm and t_first * (warm_done + 2) < budget * 0.3:
        _cpu_chamfer_once(bs)
        warm_done += 1
    steps = max(1, min(args.steps, int((budget - t_first * warm_done) / max(t_first, 1e-3))))
    ts = [_cpu_chamfer_once(bs) for _ in range(steps)]
    pairs = 2.0 * bs * C1["N"] * C1["M"]
    value = pairs * len(ts) / sum(ts) / 1e9
    sample = (f"{bs} of the 32 C1 clouds per step, {len(ts)} timed steps (of {args.steps} asked; bounded to ~{budget:.0f} s of CPU work), "
              f"pure-torch direct-form fwd+bwd on {torch.get_num_threads()} threads")
    emit({
        "impl": "reference", "metric": "chamfer_fwd_bwd_gpair_per_s", "value": round(value, 4), "unit": "Gpair/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", args.gpus)), "steps": len(ts), "warmup": warm_done,
        "ms_per_step": round(sum(ts) / len(ts) * 1e3, 2), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOADS["c1"], "B_per_gpu": bs, "B_per_step": bs, "N": C1["N"], "M": C1["M"]},
        "cpu_baseline": {"value": round(value, 4), "unit": "Gpair/s", "cores": torch.get_num_threads(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": round(value, 4), "unit": "Gpair/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    })


_RESULT_FD = None


def claim_stdout():
    """Keep stdout for the ONE JSON line: libraries that print there (NCCL's version banner does, whatever
    NCCL_DEBUG_FILE says) are pointed at stderr for the whole run; emit() writes to the saved descriptor."""
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=140, help="timed steps of the headline in all")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--repeats", type=int, default=7, help="how many blocks the K timed steps are split into (median block reported)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--workload", default="c5", choices=["c1", "c5", "c4loss"], help="--scaling strong: which fixed-size workload to split")
    ap.add_argument("--e2e-depth", type=int, default=4, help="steps in flight in the e2e loop (1-4; 1 = one call at a time)")
    ap.add_argument("--e2e-chunk", type=int, default=0, help="clouds per pipeline chunk of the host-buffer call (0: library default)")
    ap.add_argument("--reduce", default="peer", choices=["peer", "nccl_graph", "pipelined", "inline"],
                    help="how the per-step reduction of the loss sums runs when N > 1 (A/B); default: peer-memory exchange inside the step's graph")
    ap.add_argument("--no-ops", action="store_true", help="skip the FPS/kNN/gather/group section")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline legs")
    ap.add_argument("--no-ref-cuda", action="store_true", help="skip timing the reference's CUDA kernels (oracle/_ref)")
    ap.add_argument("--quick", action="store_true", help="headline + e2e only")
    ap.add_argument("--ref-clouds", type=int, default=0, help="--impl reference: clouds per step (0 = the full B=32)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's outputs to DIR/<name>.npy (in the tree: bench_outputs/)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the CUDA path's outputs (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
