"""Multi-GPU behind the C ABI (vix_comm_* / vix_sharded_*): a single rank on one GPU, and -- when the box has two GPUs --
two ranks from a plain C host (fork + pipes, no Python, no MPI) and from torch.distributed.run, over peer memory and over
the NCCL fallback.  Results must equal a single-GPU index holding all rows (same ids; distances to fp32 rounding, bit for
bit when the rows sit in the same slots)."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _ngpus():
    import torch
    return torch.cuda.device_count()


def test_single_rank_comm_equals_plain_index(oracle):
    from vectorindex_b200 import _lib
    from vectorindex_b200.index import Comm, IVFPQIndex
    import ctypes as C
    rng = np.random.default_rng(3)
    n, d, m, kc, nq, k = 5000, 64, 16, 16, 77, 10
    xb = rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal((nq, d)).astype(np.float32)
    coarse = rng.standard_normal((kc, d)).astype(np.float32)
    cb = (0.4 * rng.standard_normal((m, 256, d // m))).astype(np.float32)
    a, b = (IVFPQIndex(d, "euclidean", nlist=kc, nprobe=4, m=m) for _ in range(2))
    for idx in (a, b):
        idx.set_coarse(coarse)
        idx.set_codebooks(cb)
    ids = np.arange(n, dtype=np.int64) + 5
    a.batch_insert(xb, ids)
    comm = Comm(0, 1, Comm.unique_id())
    L = _lib.lib()
    _lib.check(L.vix_sharded_add(b._h, comm._c, None, _lib.ptr(xb), _lib.ptr(ids), C.c_int64(n)))
    dist, out = np.empty((nq, k), np.float32), np.empty((nq, k), np.int64)
    _lib.check(L.vix_sharded_search(b._h, comm._c, _lib.ptr(q), C.c_int64(nq), C.c_int(k), C.c_int(0), _lib.ptr(dist), _lib.ptr(out)))
    ad, ai = a.batch_search(q, k)
    assert np.array_equal(ai, out) and np.array_equal(ad.view(np.uint32), dist.view(np.uint32))
    first, count = C.c_int64(0), C.c_int64(0)
    _lib.check(L.vix_sharded_query_block(C.c_int64(10001), 7, 8, C.byref(first), C.byref(count)))
    assert first.value == 7 * 1252 and count.value == 10001 - 7 * 1252     # blocks of ceil(nq / world) rounded up to 4 rows
    comm.close()


@pytest.mark.parametrize("no_p2p", [False, True])
def test_two_ranks_from_a_c_host(tmp_path, no_p2p):
    if _ngpus() < 2:
        pytest.skip("needs two GPUs")
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    lib_dir = os.path.join(ROOT, "vectorindex_b200")
    exe = str(tmp_path / "sharded_smoke")
    subprocess.check_call([cc, "-std=c11", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "tests", "c", "sharded_smoke.c"), "-o", exe, "-L", lib_dir, "-lvindex_b200",
                           "-Wl,-rpath," + lib_dir, "-lm"])
    env = dict(os.environ)
    if no_p2p:
        env["VIX_NO_P2P"] = "1"
    out = subprocess.run([exe, "2"], capture_output=True, text=True, timeout=600, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "sharded == single-GPU" in out.stdout and ": yes" in out.stdout
    assert f"peer memory {0 if no_p2p else 1}" in out.stdout


@pytest.mark.parametrize("no_p2p", [False, True])
def test_two_ranks_under_torchrun(no_p2p):
    if _ngpus() < 2:
        pytest.skip("needs two GPUs")
    env = dict(os.environ)
    env.pop("VIX_NO_P2P", None)
    if no_p2p:
        env["VIX_NO_P2P"] = "1"
    world = 2 if _ngpus() < 4 else 3                                       # three ranks when the box has them: ragged blocks
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", "29533", os.path.join(ROOT, "tests", "mp_sharded_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert "ok euclidean" in out.stdout and "ok dotProduct" in out.stdout and "ok padded shard" in out.stdout
