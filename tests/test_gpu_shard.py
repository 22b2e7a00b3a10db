"""List-sharded deployment behind the C ABI (b200vs_shard_*, csrc/shard.cu): the reference's analogue is one index per
Raft region merged by VectorIndexWrapper::MergeSearchResults (src/vector/vector_index.cc:1056-1108)."""
import os
import subprocess
import sys

import numpy as np
import pytest

import b200vs
import oracle_lib
from gpu_util import assert_same_results, require_gpu

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _build(oracle, metric, om, n, d, nlist, seed=5):
    rng = np.random.default_rng(seed)
    xb = rng.random((n, d)).astype(np.float32)
    ids = np.arange(1, n + 1, dtype=np.int64)
    xn = oracle.normalize_faiss(xb) if metric == b200vs.COSINE else xb
    cent = oracle.kmeans(om, xn, nlist, nthreads=8)
    return xb, ids, cent


@pytest.mark.parametrize("metric,om", [(b200vs.L2, oracle_lib.L2), (b200vs.COSINE, oracle_lib.COSINE)])
def test_world_of_one_equals_the_plain_index_and_the_oracle(oracle, metric, om):
    """world = 1 needs no NCCL: the shard path (slice coarse, packed records, warp merge) must equal b200vs_search."""
    require_gpu()
    n, d, nlist, nq, k, nprobe = 30000, 128, 64, 150, 10, 12
    xb, ids, cent = _build(oracle, metric, om, n, d, nlist)
    ix = b200vs.Index(b200vs.IVF_FLAT, metric, d, nlist=nlist)
    ix.set_trained_state(b200vs.ivf_state_blob(cent, metric))
    sh = b200vs.Shard(ix, 0, 1, None, lanes=2)
    assert sh.list_range() == (0, nlist)
    sh.add(xb[:17000], ids[:17000])
    sh.add(xb[17000:], ids[17000:])
    xq = np.random.default_rng(9).random((nq, d)).astype(np.float32)
    D, I = sh.search(xq, k, nprobe=nprobe)
    Dp, Ip = ix.search(xq, k, nprobe=nprobe)
    assert_same_results(D, I, Dp, Ip)
    off, lx, _, lids = ix.export_lists(nlist)
    qn = oracle.normalize_faiss(xq) if metric == b200vs.COSINE else xq
    Do, Io = oracle.ivfflat_search(om, cent, off, lx, lids, qn, k, nprobe, nthreads=8)
    assert_same_results(D, I, Do, Io)
    # k wide enough to leave the warp merge (world * k > 256 records)
    D2, I2 = sh.search(xq[:20], 300, nprobe=nprobe)
    Do2, Io2 = oracle.ivfflat_search(om, cent, off, lx, lids, qn[:20], 300, nprobe, nthreads=8)
    assert_same_results(D2, I2, Do2, Io2)
    sh.close()


def test_device_add_assign_and_reserved_lists(oracle):
    """b200vs_add_with_ids_device / b200vs_assign_device / b200vs_reserve_lists: a bulk-built index (lists pre-sized from
    the assignment, rows added from device memory with precomputed lists) answers like the host-built one."""
    require_gpu()
    import torch
    n, d, nlist, nq, k, nprobe = 40000, 64, 32, 64, 10, 8
    xb, ids, cent = _build(oracle, b200vs.L2, oracle_lib.L2, n, d, nlist, seed=3)
    ref = b200vs.Index(b200vs.IVF_FLAT, b200vs.L2, d, nlist=nlist)
    ref.set_trained_state(b200vs.ivf_state_blob(cent, b200vs.L2))
    ref.add(xb, ids)
    ix = b200vs.Index(b200vs.IVF_FLAT, b200vs.L2, d, nlist=nlist)
    ix.set_trained_state(b200vs.ivf_state_blob(cent, b200vs.L2))
    xd, idd = torch.from_numpy(xb).cuda(), torch.from_numpy(ids).cuda()
    lst = torch.empty(n, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ix.assign_device(n, xd.data_ptr(), lst.data_ptr())
    want = oracle.assign(oracle_lib.L2, xb, cent, nthreads=8)
    assert np.array_equal(lst.cpu().numpy(), want.astype(np.int64)), "device assignment differs from the oracle's"
    ix.reserve_lists(np.bincount(want, minlength=nlist))
    mem0 = ix.get_memory_size()
    for a in range(0, n, 9000):  # precomputed lists for one half, library-side assignment for the other
        m = min(9000, n - a)
        ix.add_device(m, xd[a:].data_ptr(), idd[a:].data_ptr(), lst[a:].data_ptr() if (a // 9000) % 2 == 0 else None)
    assert ix.get_memory_size() == mem0, "a reserved index must not re-allocate its arena"
    assert ix.get_count() == n
    xq = np.random.default_rng(4).random((nq, d)).astype(np.float32)
    D, I = ix.search(xq, k, nprobe=nprobe)
    Dr, Ir = ref.search(xq, k, nprobe=nprobe)
    assert_same_results(D, I, Dr, Ir)
    # the usual write path keeps working on a reserved index (upsert, delete)
    ix.upsert(xb[:100] + 0.5, ids[:100])
    ref.upsert(xb[:100] + 0.5, ids[:100])
    assert ix.delete(ids[200:300]) == 100 and ref.delete(ids[200:300]) == 100
    D, I = ix.search(xq, k, nprobe=nprobe)
    Dr, Ir = ref.search(xq, k, nprobe=nprobe)
    assert_same_results(D, I, Dr, Ir)


def test_two_ranks_match_oracle():
    """torchrun --nproc-per-node 2: NCCL rendezvous through the ABI, row routing, sharded search == oracle on the gathered index."""
    require_gpu()
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs: launches one torchrun rank per GPU")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29517", os.path.join(ROOT, "tests", "shard_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=420)
    assert r.returncode == 0 and "SHARD_WORKER OK" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])
