#!/usr/bin/env python
"""bench.py — headline benchmark of the vector-search hot path (BASELINE.json metric).

Workload (config.workload): IVF-Flat, L2, N = 1M x 768 float32 per GPU, nlist = 1024 per GPU, nprobe = 32,
batch = 1024 queries per GPU, top-10 — BASELINE.json configs[1] at the batch size the metric is quoted on.
A "step" is one batched search (b200vs_search) over synthetic U[0,1) vectors.

  value : QPS with queries / results resident in HBM (b200vs_search_device), CUDA events, max over ranks.
  e2e   : QPS through the host-pointer C-ABI call (b200vs_search; b200vs_shard_search when sharded) with pinned host
          buffers: H2D of the queries and D2H of (dist, id) inside the timed region, one caller thread per batch in flight.
  roofline : the list-scan kernel's algorithmic bytes (SURVEY §8d: rows of the distinct probed lists x (d*4+8))
          / its CUDA-event duration (library profiling mode, separate pass) vs MEASURED_PEAKS.json hbm_gbs.
  cpu_baseline : the CPU oracle (restated reference path, AVX-512 order) on the box's host cores, bounded sample.

Multi-GPU (torchrun, one rank per GPU): ONE logical index sharded BY INVERTED LIST (SURVEY §8e) through the product's
own C ABI (b200vs_shard_*, include/b200vs.h): centroids replicated, rows routed to their list owner at add time, every
rank scans the probed lists it owns for the whole (N x 1024)-query batch, then ONE ncclAllGather of the packed per-shard
top-k + the on-GPU k-way merge.  torch.distributed only carries the 128-byte rendezvous blob and the timing reductions.
Weak scaling: per-GPU database and per-GPU batch are fixed.  Every N > 1 line is verified: a query sample is answered by the
sharded path and by the CPU oracle on every rank's exported shard (merged on rank 0) -> recall_at_10_vs_oracle, ids_bit_exact.

--impl reference : times the reference's CPU implementation of the same path (the oracle port; faiss itself is
not vendored in /root/reference), rank 0 only.  `value` = the reference's deployed execution shape (16 pool threads, one
query per task: conf/index-gflags.conf:5, vector_index.cc:54); the all-host-threads number is reported beside it.

--dump-outputs DIR : writes what the last timed step returned (device-resident and e2e paths) as .npy files, one GPU.
Database, ids and queries come from fixed seeds, and the centroids from the seeded CPU k-means (the GPU k-means sums
with float atomics, so its centroids vary from run to run), so two builds run with the same arguments can be compared
output for output.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "dingo-store_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200vs", choices=["b200vs", "reference"])
    ap.add_argument("--nb", type=int, default=1_000_000, help="database vectors per GPU")
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--nlist", type=int, default=1024, help="inverted lists per GPU")
    ap.add_argument("--nprobe", type=int, default=32)
    ap.add_argument("--batch", type=int, default=1024, help="queries per GPU per step")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--exact-only", action="store_true", help="force the exact FP32 scan path")
    ap.add_argument("--in-flight", type=int, default=0, help="batches in flight (streams / caller threads); 0 = 8 on one GPU, 4 per rank "
                    "when sharded (one NCCL communicator per batch in flight).  The reference serves searches from a 16-thread pool, "
                    "so concurrent batches are the deployed shape (round-1 sweep: 2 -> 1.39 M, 3 -> 1.44 M, 4 -> 1.47 M, 8 -> 1.49 M QPS)")
    ap.add_argument("--verify", type=int, default=256, help="multi-GPU: queries answered by the sharded path AND by the CPU oracle on every rank's shard")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="after the timed steps, write the results of the last timed step as DIR/<name>.npy: distances (float32) "
                         "and ids (float64) of the device-resident path and of the host-pointer (e2e) path; a seeded sample of "
                         "query rows (DIR/query_rows.npy) when all rows exceed 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200vs":
        ap.error("--dump-outputs applies to --impl b200vs")
    return args


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays, nq):
    """Writes {name: [nq, k] array} as out_dir/<name>.npy, float32 / float64 only, at most DUMP_LIMIT bytes in all."""
    arrays = {n: a.astype(np.float64) if a.dtype == np.int64 else a for n, a in arrays.items()}
    row_bytes = sum(a.nbytes // nq for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    if row_bytes * nq > DUMP_LIMIT:  # sampled rows + their float64 indices + one 4 KB allowance for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(nq, (DUMP_LIMIT - 4096) // (row_bytes + 8), replace=False))
        arrays = {n: a[rows] for n, a in arrays.items()}
        arrays["query_rows"] = rows.astype(np.float64)
    for n, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (n, a.dtype)
        np.save(os.path.join(out_dir, n + ".npy"), np.ascontiguousarray(a))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def gen_chunks(torch, n, d, seed, device, chunk=131072):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    for a in range(0, n, chunk):
        m = min(chunk, n - a)
        yield a, torch.rand((m, d), generator=g, device=device, dtype=torch.float32)


# --------------------------------------------------------------------------------------------------
# reference arm: the CPU oracle with every host thread (rank 0 only)
# --------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    if rank != 0:
        return
    import oracle_lib
    o = oracle_lib.load()
    cores = os.cpu_count() or 1
    n, d, nlist = args.nb, args.dim, args.nlist
    rng = np.random.default_rng(1234)
    xb = rng.random((n, d), dtype=np.float32)
    ids = np.arange(1, n + 1, dtype=np.int64)
    t0 = time.time()
    # training sample as faiss would take it (<= 256 points per centroid); fewer when the host is small so the
    # whole arm stays within minutes — the index SHAPE (nlist, list lengths) is what the timed search depends on
    max_pts = 256 if cores >= 32 else 64
    niter = 10 if cores >= 32 else 4
    cent = o.kmeans(oracle_lib.L2, xb[: min(n, nlist * max_pts)], nlist, niter=niter, max_pts=max_pts, nthreads=cores)
    asg = o.assign(oracle_lib.L2, xb, cent, nthreads=cores)
    order = np.argsort(asg, kind="stable")
    off = np.zeros(nlist + 1, np.int64)
    off[1:] = np.cumsum(np.bincount(asg, minlength=nlist))
    lx, lids = o.numa_spread(xb[order], cores), ids[order]
    del xb
    build_s = time.time() - t0
    xq = np.random.default_rng(4321).random((args.batch, d), dtype=np.float32)
    shape_threads = min(16, cores)  # the reference's search pool: 16 workers, one query per task

    def timed(nthreads, sample, steps, warmup):
        for _ in range(warmup):
            o.ivfflat_search(oracle_lib.L2, cent, off, lx, lids, xq[:sample], args.k, args.nprobe, nthreads=nthreads)
        per = []
        for _ in range(steps):
            t = time.time()
            o.ivfflat_search(oracle_lib.L2, cent, off, lx, lids, xq[:sample], args.k, args.nprobe, nthreads=nthreads)
            per.append(time.time() - t)
        return per

    # calibrate a bounded sample: ~1.5 s of CPU work per step
    t = time.time()
    o.ivfflat_search(oracle_lib.L2, cent, off, lx, lids, xq[:shape_threads * 2], args.k, args.nprobe, nthreads=shape_threads)
    per_q = (time.time() - t) / (shape_threads * 2)
    budget = 120.0 / max(1, args.steps + args.warmup)
    sample = int(max(shape_threads, min(args.batch, (min(1.5, budget) / max(per_q, 1e-6)))))
    per = timed(shape_threads, sample, args.steps, args.warmup)
    el = float(np.sum(per))
    qps = sample * args.steps / el
    qps_median = sample / float(np.median(per))
    # the same sample on every host thread (a reported extra: NUMA-remote streaming makes it box-dependent)
    per_all = timed(cores, sample, max(2, min(args.steps, 5)), 1)
    qps_all = sample / float(np.median(per_all))
    line = {"impl": "reference", "metric": "QPS at batch-1024 top-10 dim=768; recall@10 vs ref; % HBM roofline", "value": qps,
            "unit": "queries/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, 1),
            "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": shape_threads, "kind": "port", "median_step_qps": qps_median,
                             "all_host_threads_qps": qps_all, "host_threads": cores,
                             "shape": "reference execution shape: 16 search-pool threads, one query per task, OpenMP 1 thread (conf/index-gflags.conf:4-5, vector_index.cc:54); value = this shape",
                             "sample": f"{sample} of the {args.batch}-query batch per step, {shape_threads} threads, one query per task; "
                                       f"oracle port of the reference path (faiss not vendored); index built on CPU in {build_s:.0f}s "
                                       f"(kmeans niter={niter}, {max_pts} pts/centroid)"},
            "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": f"IVF-Flat L2 {args.nb}x{args.dim} f32 per GPU, nlist={args.nlist} per GPU, nprobe={args.nprobe}, "
                        f"batch={args.batch} per GPU, top-{args.k} (BASELINE configs[1] at the metric's batch 1024)",
            "index": "IVF_FLAT", "metric_type": "L2", "nb_per_gpu": args.nb, "dim": args.dim, "nlist_per_gpu": args.nlist,
            "nprobe": args.nprobe, "batch_per_gpu": args.batch, "topk": args.k, "batches_in_flight": max(1, args.in_flight),
            "parallelism": f"list-sharded x{world} behind b200vs_shard_*: coarse quantiser on the rank's query slice + all-gather of the probe table, tile scan of the owned lists, ONE ncclAllGather of packed (distance,id) top-k + merge kernel" if world > 1 else "single GPU",
            "l2_flush": "inputs larger than L2: every step streams the probed lists (~3.1 GB per GPU >> 126 MB L2)"}


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.in_flight <= 0:
        args.in_flight = 8 if world == 1 else 4
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.dump_outputs and world > 1:
        sys.exit("bench.py: --dump-outputs runs on one GPU (the sharded index trains on the GPUs, not reproducibly)")

    import torch
    import b200vs
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    n, d, nlist_local, k = args.nb, args.dim, args.nlist, args.k
    nlist = nlist_local * world
    nq = args.batch * world
    t_build = time.time()

    # ---- build: synthetic data, train, add (multi-GPU: through the shard API, rows travel to their list owner) ----
    L = max(1, args.in_flight)
    ix = b200vs.Index(b200vs.IVF_FLAT, b200vs.L2, d, nlist=nlist, device=local_rank)
    sh = None
    ntrain = min(n, nlist_local * 256)
    if world == 1:
        chunks = [(a, x.cpu().numpy()) for a, x in gen_chunks(torch, n, d, 1234 + rank, dev)]
        train = np.concatenate([c for _, c in chunks], 0)[:ntrain] if len(chunks) > 1 else chunks[0][1][:ntrain]
        if args.dump_outputs:  # the GPU k-means sums with float atomics; the seeded CPU k-means makes the index reproducible
            import oracle_lib
            cent = oracle_lib.load().kmeans(oracle_lib.L2, train, nlist, nthreads=os.cpu_count() or 1)
            ix.set_trained_state(b200vs.ivf_state_blob(cent, b200vs.L2))
        else:
            ix.train(train)
        for a, x in chunks:
            for b in range(0, x.shape[0], 32768):  # kBuildVectorIndexBatchSize, src/common/constant.h:173
                ix.add(x[b:b + 32768], np.arange(a + b + 1, a + b + 1 + min(32768, x.shape[0] - b), dtype=np.int64))
        del chunks, train
    else:
        idb = torch.from_numpy(b200vs.Shard.unique_id() if rank == 0 else np.zeros(128, np.uint8)).to(dev)
        dist.broadcast(idb, 0)
        sh = b200vs.Shard(ix, rank, world, idb.cpu().numpy(), lanes=L)
        train = torch.cat([x for _, x in gen_chunks(torch, ntrain, d, 1234 + rank, dev)], 0).cpu().numpy()
        sh.train(train)  # distributed: nlist / world centroids per rank, one all-gather
        del train
        for a, x in gen_chunks(torch, n, d, 1234 + rank, dev):
            gid = torch.arange(a + 1, a + 1 + x.shape[0], dtype=torch.int64, device=dev) + rank * n
            torch.cuda.synchronize()
            sh.add_device(x.shape[0], x.data_ptr(), gid.data_ptr())
    build_s = time.time() - t_build

    # ---- query batches (all ranks hold the same global batch) ----
    gq = torch.Generator(device=dev)
    gq.manual_seed(4321)
    nbatches = 4
    q_dev = [torch.rand((nq, d), generator=gq, device=dev, dtype=torch.float32) for _ in range(nbatches)]
    out_d = [torch.empty((nq, k), dtype=torch.float32, device=dev) for _ in range(L)]
    out_i = [torch.empty((nq, k), dtype=torch.int64, device=dev) for _ in range(L)]
    sp, _keep = b200vs.make_search_params(nprobe=args.nprobe, exact_only=args.exact_only)
    main_stream = torch.cuda.Stream(device=dev)  # real (non-NULL) streams: the library launches on them, the events time them
    streams = [torch.cuda.Stream(device=dev) for _ in range(L)]
    torch.cuda.set_stream(main_stream)
    stream = streams[0]
    launches = [0]
    seq = [0]  # batch sequence number of the sharded path: the same on every rank, so batch i uses the same communicator everywhere

    def step_device(i, lanes=L):
        ln = i % lanes
        st = streams[ln]
        q = q_dev[i % nbatches]
        if world > 1:
            sh.search_device(nq, q.data_ptr(), k, out_d[ln].data_ptr(), out_i[ln].data_ptr(), stream=st.cuda_stream, sp=sp, seq=seq[0])
            seq[0] += 1
        else:
            ix.search_device(nq, q.data_ptr(), k, out_d[ln].data_ptr(), out_i[ln].data_ptr(), stream=st.cuda_stream, sp=sp)
        launches[0] += ix.stats()[0]

    def timed_device(steps, lanes):
        """K steps on `lanes` streams; CUDA events on main_stream bracket all of them."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(main_stream)
        for st in streams[:lanes]:
            st.wait_event(e0)
        for i in range(steps):
            step_device(i, lanes)
        for st in streams[:lanes]:
            ev = torch.cuda.Event()
            ev.record(st)
            main_stream.wait_event(ev)
        e1.record(main_stream)
        return e0, e1

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(max(3, args.warmup, 2 * L)):  # every lane at least twice: a lane's first search sizes its scratch arena
        step_device(i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches[0] = 0
    prof = os.environ.get("BENCH_PROFILE") == "1"  # ncu --profile-from-start off: only the timed steps are captured
    if prof:
        torch.cuda.profiler.start()
    e0, e1 = timed_device(args.steps, L)
    barrier()
    if prof:
        torch.cuda.profiler.stop()
    ms = e0.elapsed_time(e1)
    gpu_launches = launches[0]
    last = (args.steps - 1) % L  # lane of the last timed step; later passes overwrite lane 0
    dumped = {"distances": out_d[last].cpu().numpy(), "ids": out_i[last].cpu().numpy()} if args.dump_outputs else {}
    # the same K steps strictly one after another on one stream (per-batch latency view)
    e0, e1 = timed_device(args.steps, 1)
    barrier()
    ms_single = e0.elapsed_time(e1)

    # ---- e2e: host buffers through the public C-ABI call, copies inside the timed region ----
    q_host = [q.cpu().pin_memory() for q in q_dev]
    hd = [torch.empty((nq, k), dtype=torch.float32).pin_memory() for _ in range(L)]
    hi = [torch.empty((nq, k), dtype=torch.int64).pin_memory() for _ in range(L)]

    def step_e2e(i, ln=0, base=0):
        q = q_host[i % nbatches]
        if world == 1:
            ix.search_raw(nq, q.data_ptr(), k, hd[ln].data_ptr(), hi[ln].data_ptr(), sp=sp)  # H2D + search + D2H, synchronous
        else:  # H2D of the rank's slice + NVLink all-gather of the batch + sharded search + D2H, synchronous
            sh.search_raw(nq, q.data_ptr(), k, hd[ln].data_ptr(), hi[ln].data_ptr(), sp=sp, seq=base + i)
        return float(hd[ln][0, 0])

    def run_e2e(steps):
        base = seq[0]
        seq[0] += steps
        if L == 1:
            for i in range(steps):
                step_e2e(i, 0, base)
            return
        def worker(t):  # one caller thread per batch in flight; explicit sequence numbers keep the ranks' collectives aligned
            for i in range(t, steps, L):
                step_e2e(i, t, base)
        ths = [threading.Thread(target=worker, args=(t,)) for t in range(L)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()

    run_e2e(max(3, args.warmup, 2 * L))
    barrier()
    t0 = time.perf_counter()
    run_e2e(args.steps)
    barrier()
    e2e_s = time.perf_counter() - t0
    clocks = sampler.stop()
    if args.dump_outputs:
        last = (args.steps - 1) % L  # caller thread (and buffer) of the last timed step
        dumped.update(e2e_distances=hd[last].numpy().copy(), e2e_ids=hi[last].numpy().copy())
        if rank == 0:
            dump_outputs(args.dump_outputs, dumped, nq)

    # max over ranks
    if world > 1:
        t = torch.tensor([ms, e2e_s * 1e3, ms_single], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, e2e_ms, ms_single = t.tolist()
    else:
        e2e_ms = e2e_s * 1e3
    qps = nq * args.steps / (ms / 1e3)
    e2e_qps = nq * args.steps / (e2e_ms / 1e3)

    # ---- roofline of the dominant kernel (separate, profiled pass; never part of the timed numbers) ----
    ix.set_profiling(True)
    kt, rows = [], 0
    phase_ms = {}
    for i in range(3):
        if world > 1:
            sh.search_device(nq, q_dev[i % nbatches].data_ptr(), k, out_d[0].data_ptr(), out_i[0].data_ptr(), stream=stream.cuda_stream, sp=sp, seq=seq[0])
            seq[0] += 1
        else:
            ix.search_device(nq, q_dev[i % nbatches].data_ptr(), k, out_d[0].data_ptr(), out_i[0].data_ptr(), stream=stream.cuda_stream, sp=sp)
        torch.cuda.synchronize()
        st = ix.stats()
        kt.append(st[3] / 1e9)
        rows = st[4]
        phase_ms = ix.phase_times()
    prof_stats = list(st)
    ix.set_profiling(False)
    peak, how = measured_peaks()
    kern_s = float(np.mean(kt)) if kt and min(kt) > 0 else None
    alg_bytes = rows * (d * 4 + 8)
    # DRAM traffic of the same kernel from the committed ncu --set full capture (only for the workload it was taken on)
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "round2", "ncu_traffic.json")
    if world == 1 and (args.nb, args.dim, args.nlist, args.nprobe, args.batch, args.k) == (1_000_000, 768, 1024, 32, 1024, 10) and os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic, traffic_src = int(tj["dram_bytes_per_launch"]), tj["source"]
        except Exception:
            pass
    roofline = {"bound": "hbm", "achieved": (alg_bytes / kern_s / 1e9) if kern_s else None, "peak": peak, "unit": "GB/s",
                "frac": (alg_bytes / kern_s / 1e9 / peak) if kern_s else None, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "ivf list scan", "kernel_ms": kern_s * 1e3 if kern_s else None,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": how + " (MEASURED_PEAKS.json hbm_gbs)" if how == "measured" else "fallback 6650 GB/s"}

    # ---- cpu_baseline: the oracle on the host cores, bounded sample (rank 0, N = 1 only) ----
    cpu_baseline = None
    recall_vs_oracle = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle_lib
        o = oracle_lib.load()
        cores = os.cpu_count() or 1
        off, lx, _, lids = ix.export_lists(nlist)
        lx = o.numa_spread(lx, cores)
        cent = ix.get_trained_state()[32:].view(np.float32).reshape(nlist, d)
        xq = q_host[0].numpy()
        t = time.time()
        o.ivfflat_search(oracle_lib.L2, cent, off, lx, lids, xq[:cores], k, args.nprobe, nthreads=cores)
        per_q = (time.time() - t) / cores
        sample = args.cpu_sample or int(max(cores, min(nq, 15.0 / max(per_q, 1e-6))))
        t = time.time()
        Do, Io = o.ivfflat_search(oracle_lib.L2, cent, off, lx, lids, xq[:sample], k, args.nprobe, nthreads=cores)
        cpu_s = time.time() - t
        ix.search_raw(nq, q_host[0].data_ptr(), k, hd[0].data_ptr(), hi[0].data_ptr(), sp=sp)
        Ig, Dg = hi[0].numpy()[:sample], hd[0].numpy()[:sample]
        recall_vs_oracle = float(np.mean([len(set(a) & set(b)) / k for a, b in zip(Ig, Io)]))
        ids_exact = bool(np.array_equal(Ig, Io))
        # the reference's own execution shape: 16 pool threads, one query per task (conf/index-gflags.conf:5, vector_index.cc:54)
        s16 = int(min(sample, 64))
        t = time.time()
        o.ivfflat_search(oracle_lib.L2, cent, off, lx, lids, xq[:s16], k, args.nprobe, nthreads=min(16, cores))
        qps16 = s16 / max(time.time() - t, 1e-9)
        cpu_baseline = {"value": sample / cpu_s, "unit": "queries/s", "cores": cores, "kind": "port", "reference_shape_16_threads_qps": qps16,
                        "sample": f"first {sample} queries of the {nq}-query batch on the same trained index, {cores} threads, one query per task",
                        "recall_at_k_gpu_vs_oracle": recall_vs_oracle, "ids_bit_exact": ids_exact,
                        "max_rel_dist_err": float(np.max(np.abs(Dg - Do) / np.maximum(np.abs(Do), 1e-12)))}

    # ---- N > 1: answer a query sample through the sharded product path AND with the CPU oracle on every rank's shard ----
    verify = None
    if world > 1 and args.verify > 0:
        import oracle_lib
        import b200vs.shard as shard_host
        o = oracle_lib.load()
        ns = int(min(args.verify, nq))
        xq = q_host[0].numpy()[:ns].copy()
        Dg, Ig = sh.search(xq, k, seq=seq[0], nprobe=args.nprobe)  # host-pointer collective call, merged result on every rank
        seq[0] += 1
        off, lx, _, lids = ix.export_lists(nlist)  # this rank's rows; lists owned elsewhere are empty
        cent = ix.get_trained_state()[32:].view(np.float32).reshape(nlist, d)
        threads = max(1, (os.cpu_count() or 1) // world)
        t = time.time()
        Do, Io = o.ivfflat_search(oracle_lib.L2, cent, off, lx, lids, xq, k, args.nprobe, nthreads=threads)
        oracle_s = time.time() - t
        gd = [torch.empty((ns, k), dtype=torch.float32, device=dev) for _ in range(world)]
        gi = [torch.empty((ns, k), dtype=torch.int64, device=dev) for _ in range(world)]
        dist.all_gather(gd, torch.from_numpy(Do).to(dev))
        dist.all_gather(gi, torch.from_numpy(Io).to(dev))
        cnt = torch.tensor([ix.get_count()], dtype=torch.int64, device=dev)
        dist.all_reduce(cnt)
        if rank == 0:
            Dm, Im = shard_host.merge_topk(torch.stack(gd).cpu().numpy(), torch.stack(gi).cpu().numpy(), k)  # MergeSearchResults rule
            verify = {"queries": ns, "ids_bit_exact": bool(np.array_equal(Ig, Im)),
                      "dist_bit_exact": bool(np.array_equal(Dg.view(np.uint32), Dm.view(np.uint32))),
                      "recall_at_k_gpu_vs_oracle": float(np.mean([len(set(a) & set(b)) / k for a, b in zip(Ig, Im)])),
                      "max_rel_dist_err": float(np.max(np.abs(Dg - Dm) / np.maximum(np.abs(Dm), 1e-12))),
                      "rows_in_index_all_ranks": int(cnt.item()), "oracle_seconds_per_rank": oracle_s,
                      "how": f"first {ns} queries of the batch: b200vs_shard_search on {world} ranks vs the CPU oracle run on every rank's exported shard "
                             f"(global centroids, {threads} threads per rank), per-rank top-k merged on rank 0 with the MergeSearchResults rule"}
            recall_vs_oracle = verify["recall_at_k_gpu_vs_oracle"]

    if rank == 0:
        line = {"metric": "QPS at batch-1024 top-10 dim=768; recall@10 vs ref; % HBM roofline", "value": qps, "unit": "queries/s",
                "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(args, world),
                "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": nq * d * 4, "d2h_bytes_per_step": nq * k * 12,
                        "ms_per_step": e2e_ms / args.steps},
                "single_stream": {"value": nq * args.steps / (ms_single / 1e3), "unit": "queries/s", "ms_per_step": ms_single / args.steps,
                                  "note": "same K steps strictly back to back on one stream"},
                "gpu_launches": gpu_launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu_baseline,
                "recall_at_10_vs_oracle": recall_vs_oracle, "sharded_verification": verify, "build_seconds": build_s, "search_stats": ix.stats(), "profile_stats": prof_stats, "phase_ms": {a: round(v, 4) for a, v in phase_ms.items()}}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        sh.close()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
