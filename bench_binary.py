"""Binary (Hamming) index benchmark: QPS of BINARY_FLAT and BINARY_IVF_FLAT searches from CUDA events, next to the
byte bound and the POPC work of each workload, with ids and distances checked against the CPU binary oracle.

Workloads (1024-bit rows, k 10):
  flat_b1 / flat_b64 : BINARY_FLAT, 2M rows (256 MB, larger than the 126 MB L2), batch 1 and batch 64
  ivf_b1024          : BINARY_IVF_FLAT, 10M rows, nlist 4096, nprobe 32, batch 1024
The IVF centroids are a seeded sample of the rows (set_trained_state): the benchmark times search, not training.
Prints one JSON line per workload plus one with the GPU name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "dingo-store_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

import b200vs  # noqa: E402
import oracle_binary_lib  # noqa: E402

DIM = 1024
CODE = DIM // 8
HBM_BYTES_PER_S = 7.7e12  # data-sheet HBM3e bandwidth of one B200


def sparse_bits(rng, m):
    """[m, CODE] bytes whose bits are set with probability 1/8 (AND of three uniform bytes)."""
    r = rng.integers(0, 256, (3, m, CODE), dtype=np.uint8)
    return r[0] & r[1] & r[2]


def gpu_info():
    import torch
    info = {"gpu": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception as e:  # the numbers are still reported, with the reason the limit is unknown
        info["power_limit_w"] = f"unavailable: {e}"
    return info


def timed_search(ix, xq_all, k, steps, warmup, nq, nprobe=0):
    """Device-pointer searches of `nq` queries each (CUDA events around `steps` batches); returns seconds per batch."""
    import torch
    q = torch.from_numpy(xq_all).cuda()
    nb = xq_all.shape[0] // nq
    od = torch.zeros((nq, k), dtype=torch.float32, device="cuda")
    oi = torch.zeros((nq, k), dtype=torch.int64, device="cuda")
    sp, _ = b200vs.make_search_params(nprobe=nprobe)
    stream = torch.cuda.current_stream().cuda_stream
    for i in range(warmup):
        ix.search_device(nq, q[(i % nb) * nq:].data_ptr(), k, od.data_ptr(), oi.data_ptr(), stream=stream, sp=sp)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        ix.search_device(nq, q[(i % nb) * nq:].data_ptr(), k, od.data_ptr(), oi.data_ptr(), stream=stream, sp=sp)
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / 1e3 / steps


def check(name, D, I, Do, Io):
    ok = bool(np.array_equal(I, Io) and np.array_equal(D.view(np.uint32), Do.view(np.uint32)))
    if not ok:
        bad = np.argwhere(I != Io)
        print(json.dumps({"workload": name, "oracle_check": "FAILED", "first_mismatch": bad[:3].tolist()}), flush=True)
    return ok


def bench_flat(rng, bo, args):
    n = args.flat_rows
    xb = rng.integers(0, 256, (n, CODE), dtype=np.uint8)
    ids = np.arange(n, dtype=np.int64)
    ix = b200vs.Index(b200vs.BINARY_FLAT, b200vs.HAMMING, DIM)
    for a in range(0, n, 1 << 20):
        ix.add(xb[a:a + (1 << 20)], ids[a:a + (1 << 20)])
    xq = rng.integers(0, 256, (max(256, 64 * 8), CODE), dtype=np.uint8)
    xq[:64] = xb[rng.integers(0, n, 64)] ^ np.uint8(3)  # near duplicates: small distances among the hits
    ok = True
    D, I = ix.search(xq[:256], args.k)
    Do, Io = bo.flat_search(xb, ids, xq[:256], args.k)
    ok &= check("flat", D, I, Do, Io)
    out = []
    for nq in (1, 64):
        t = timed_search(ix, xq, args.k, args.steps, args.warmup, nq)
        out.append({"workload": f"flat_b{nq}", "rows": n, "dim_bits": DIM, "nq": nq, "k": args.k, "qps": nq / t, "ms_per_batch": t * 1e3,
                    "bytes_per_batch": n * CODE, "byte_bound_ms": n * CODE / HBM_BYTES_PER_S * 1e3,
                    "popc32_per_batch": nq * n * (DIM // 32), "oracle_check_256q": "passed" if ok else "FAILED"})
    return out, ok


def bench_ivf(rng, bo, args):
    n, nlist, nprobe, nq = args.ivf_rows, 4096, 32, 1024
    centers = rng.integers(0, 256, (nlist, CODE), dtype=np.uint8)
    ix = b200vs.Index(b200vs.BINARY_IVF_FLAT, b200vs.HAMMING, DIM, nlist=nlist)
    xb = np.empty((n, CODE), np.uint8)
    chunk = 1 << 20
    for a in range(0, n, chunk):  # clustered rows: each row is a centre with 1/8 of its bits flipped on average
        m = min(chunk, n - a)
        xb[a:a + m] = centers[rng.integers(0, nlist, m)] ^ sparse_bits(rng, m)
    cent = xb[np.sort(rng.choice(n, nlist, replace=False))]
    ix.set_trained_state(b200vs.binary_ivf_state_blob(cent))
    ids = np.arange(n, dtype=np.int64)
    for a in range(0, n, chunk):
        ix.add(xb[a:a + chunk], ids[a:a + chunk])
    del xb
    xq = centers[rng.integers(0, nlist, 4 * nq)] ^ sparse_bits(rng, 4 * nq)
    ix.set_profiling(True)  # one search outside the timing: rows of the distinct probed lists (the byte bound)
    ix.search(xq[:nq], args.k, nprobe=nprobe)
    st = ix.stats()
    ix.set_profiling(False)
    D, I = ix.search(xq[:256], args.k, nprobe=nprobe)
    off, _, codes, lids = ix.export_lists(nlist)
    Do, Io = bo.ivf_search(cent, off, codes, lids, xq[:256], args.k, nprobe)
    ok = check("ivf", D, I, Do, Io)
    del codes
    t = timed_search(ix, xq, args.k, args.steps, args.warmup, nq, nprobe=nprobe)
    scanned = float(n) * nprobe / nlist * nq  # expected rows scanned per batch (each query scans its own probed lists)
    return [{"workload": "ivf_b1024", "rows": n, "dim_bits": DIM, "nlist": nlist, "nprobe": nprobe, "nq": nq, "k": args.k,
             "qps": nq / t, "ms_per_batch": t * 1e3, "distinct_probed_lists": int(st[5]), "bytes_per_batch_distinct_lists": int(st[4]) * CODE,
             "byte_bound_ms": int(st[4]) * CODE / HBM_BYTES_PER_S * 1e3, "popc32_per_batch_est": scanned * (DIM // 32),
             "oracle_check_256q": "passed" if ok else "FAILED"}], ok


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--flat-rows", type=int, default=2_000_000)
    ap.add_argument("--ivf-rows", type=int, default=10_000_000)
    ap.add_argument("--only", choices=["flat", "ivf"], default=None)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_binary.py needs a CUDA device")
    print(json.dumps(gpu_info()), flush=True)
    rng = np.random.default_rng(0)
    bo = oracle_binary_lib.load()
    ok = True
    for name, fn in (("flat", bench_flat), ("ivf", bench_ivf)):
        if args.only and args.only != name:
            continue
        rows, good = fn(rng, bo, args)
        ok &= good
        for r in rows:
            print(json.dumps(r), flush=True)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
