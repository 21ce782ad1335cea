"""One rank of the sharded IVF-PQ edge suite (launched by tests/test_sharded_edges.py under torch.distributed.run, one process
per GPU), over peer memory or, with VIX_NO_P2P=1, over NCCL all-gathers.

The reference of every case is one GPU holding the same rows in the same slots: an IVFPQIndex into which the rows are
inserted as the concatenation, over source ranks 0 .. world - 1, of the rows each rank was handed.  That is the order in
which the owning ranks append them (rows sorted stably by owner, received in order of source rank), and inside a list the
slot of a vector decides the order its table entries are summed in (the rotated code layout), so the answers must agree
bit for bit: ids, distance bits, zero signs and NaN / -1 padding.  A case checks
  - that premise: the id and code sequence of every list the rank owns equals the one-GPU index's, the other lists are empty;
  - the merged answer of vix_sharded_search against the one-GPU index, bit for bit, on every rank;
  - every rank's answer against rank 0's (all-gathered), bit for bit;
  - rank 0's answer against the float64 reference of tests/pq_ref64.py on the one-GPU probes and lists (errors the shards
    and the one-GPU index would share);
  - the scan route the shards took (the VIX_SCAN_DEBUG=1 launch line, vix_scan_tc_launches()) and the exchange in use.
Every check is collective: each rank computes its verdict, the verdicts are all-reduced, and every rank raises together
with the failing ranks' messages, so no rank is left waiting in the next collective.

    python -m torch.distributed.run ... tests/mp_sharded_edges.py [case ...]      (no case: all of them)
"""
import ctypes as C
import hashlib
import os
import re
import sys
import tempfile
import traceback
import zlib
from datetime import timedelta

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

ROUTE = re.compile(r"\[vix scan\] kernel (fast G (\d)|generic)")
MAX_K = 512
ERR_INVALID_PARAM = -5
METRICS = {0: "euclidean", 1: "dotProduct"}
NEG_ZERO = np.uint32(0x80000000)


class CaseFailure(AssertionError):
    pass


class Ranks:
    """rank / world of the launch, the communicator the cases share, and the collective verdict"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        from vectorindex_b200 import _lib
        from vectorindex_b200.index import Comm
        self.rank, self.world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
        local = int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(local)
        _lib.check(_lib.lib().vix_set_device(local))
        self.dev = torch.device("cuda", local)
        dist.init_process_group("nccl", device_id=self.dev, timeout=timedelta(seconds=300))
        self.comm = Comm.from_torch()
        # (one rank: vix_sharded_search is the plain index search and never sets up an exchange)
        self.want_peer = -1 if self.world == 1 else 0 if os.environ.get("VIX_NO_P2P") else 1

    def agree(self, what, msg):
        """every rank calls this with its verdict (None: passed); all raise together when one rank failed"""
        import torch
        import torch.distributed as dist
        flag = torch.tensor([0 if msg is None else 1], dtype=torch.int32, device=self.dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX)
        if int(flag.item()):
            msgs = [None] * self.world
            dist.all_gather_object(msgs, msg)
            raise CaseFailure(f"{what}: " + "; ".join(f"rank {r}: {m}" for r, m in enumerate(msgs) if m))

    def step(self, what, fn):
        """fn() on every rank (local work, or one collective call every rank makes); its exceptions become the verdict"""
        out, msg = None, None
        try:
            out = fn()
        except Exception as e:  # noqa: BLE001 -- any failure is this rank's verdict
            msg = f"{type(e).__name__}: {e}"[:3000] or "failed"
            if not isinstance(e, AssertionError):
                msg += "\n" + traceback.format_exc()[-1500:]
        self.agree(what, msg)
        return out

    def same_everywhere(self, what, arrays):
        """the concatenated bytes of `arrays` on this rank equal rank 0's"""
        import torch
        import torch.distributed as dist
        flat = np.concatenate([np.ascontiguousarray(a).view(np.uint8).ravel() for a in arrays])
        t = torch.from_numpy(flat.copy()).to(self.dev)
        allt = torch.empty((self.world, t.numel()), dtype=torch.uint8, device=self.dev)
        dist.all_gather_into_tensor(allt, t)
        allt = allt.cpu().numpy()
        self.agree(what, None if np.array_equal(allt[self.rank], allt[0]) else "answer differs from rank 0's")

    def log(self, line):
        if self.rank == 0:
            print(line, flush=True)


def np_of(a):
    return a.cpu().numpy() if hasattr(a, "cpu") else np.asarray(a)


def bits(a):
    return np.ascontiguousarray(np_of(a), np.float32).view(np.uint32)


def with_stderr(fn):
    """fn() with file descriptor 2 captured (the library prints its VIX_SCAN_DEBUG lines there) -> (result, text)"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile() as f:
        os.dup2(f.fileno(), 2)
        try:
            out = fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        text = f.read().decode("utf-8", "replace")
    return out, text


class Env:
    """environment variables set for the duration of a block"""

    def __init__(self, **kv):
        self.kv, self.old = kv, {}

    def __enter__(self):
        for k, v in self.kv.items():
            self.old[k] = os.environ.get(k)
            os.environ[k] = v

    def __exit__(self, *exc):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# ------------------------------------------------------------------------------------------------ problems
def hand_out(rng, n, world, skip=()):
    """source rank of every row: ragged shares (rank r weighs r + 1), interleaved, none for the ranks in `skip` (unless the
    launch has one rank)"""
    w = np.array([0.0 if r in skip and world > 1 else r + 1.0 for r in range(world)])
    return rng.choice(world, n, p=w / w.sum())


class Problem:
    """one sharded index (ShardedIVFPQIndex over an IVFPQIndex on this rank's GPU) and the one-GPU IVFPQIndex holding the
    same rows in the same slots; `add` and `remove` keep both in step"""

    def __init__(self, R, coarse, cb, metric, ks=256, bounds=None, comm=None, nprobe=8):
        from vectorindex_b200.index import IVFPQIndex, ShardedIVFPQIndex
        self.R = R
        self.coarse = np.ascontiguousarray(coarse, np.float32)
        self.cb = np.ascontiguousarray(cb, np.float32)
        self.kc, self.d = self.coarse.shape
        self.m = self.cb.shape[0]
        self.ks, self.metric = ks, metric
        mk = lambda: IVFPQIndex(self.d, METRICS[metric], nlist=self.kc, nprobe=nprobe, m=self.m, ks=ks)
        self.full, self.local = mk(), mk()
        for idx in (self.full, self.local):
            idx.set_coarse(self.coarse)
            idx.set_codebooks(self.cb)
        self.sh = ShardedIVFPQIndex.wrap(self.local, self.kc, nprobe)
        self.sh.comm = comm if comm is not None else R.comm
        if bounds is not None:
            self.sh.set_list_bounds(bounds)
        # the partition vix_sharded_add uses (default: equal-count blocks kc * r / world)
        self.bounds = np.asarray(bounds if bounds is not None else [self.kc * r // R.world for r in range(R.world + 1)])
        self._lists = None

    def owned(self):
        return int(self.bounds[self.R.rank]), int(self.bounds[self.R.rank + 1])

    def add(self, what, xb, ids, src, device=False):
        """rank r hands in the rows with src == r (in their order); the one-GPU index inserts them rank by rank"""
        import torch
        order = np.concatenate([np.nonzero(src == r)[0] for r in range(self.R.world)])
        self.full.batch_insert(xb[order], ids[order])
        mine = np.nonzero(src == self.R.rank)[0]
        x, i = np.ascontiguousarray(xb[mine]), np.ascontiguousarray(ids[mine])
        if device:
            x, i = torch.from_numpy(x).to(self.R.dev), torch.from_numpy(i).to(self.R.dev)
        self.R.step(f"{what}: sharded add", lambda: self.sh.add(x, i))
        self._lists = None
        self.check_lists(what)

    def remove(self, what, ids):
        want = self.full.batch_remove(ids)
        got = self.R.step(f"{what}: sharded remove", lambda: self.sh.remove(ids))
        self.R.step(f"{what}: removed count", lambda: self._expect(got == want, f"{got} rows removed, one GPU {want}"))
        self._lists = None
        self.check_lists(what)

    @staticmethod
    def _expect(cond, msg):
        assert cond, msg

    def lists(self):
        if self._lists is None:
            self._lists = self.full.export_lists()
        return self._lists

    def check_lists(self, what):
        """the premise of bit-for-bit parity: every list this rank owns holds the one-GPU index's rows in its order"""
        def run():
            off, codes, ids, _ = self.lists()
            soff, scodes, sids, _ = self.local.export_lists()
            b, e = self.owned()
            lens = np.diff(soff)
            assert (lens[:b] == 0).all() and (lens[e:] == 0).all(), "rows in lists this rank does not own"
            for l in range(b, e):
                f, s = slice(off[l], off[l + 1]), slice(soff[l], soff[l + 1])
                assert np.array_equal(ids[f], sids[s]), f"list {l}: ids {sids[s][:8]} vs one GPU {ids[f][:8]}"
                assert np.array_equal(codes[f], scodes[s]), f"list {l}: codes differ"
        self.R.step(f"{what}: list contents", run)

    def compare(self, what, q, k, nprobe, route=None, device=False, tc=False, ref_rows=64):
        """sharded search == one GPU (bits) on every rank == rank 0's answer; rank 0 against float64; the route taken.
        route: 'fast G<g>' / 'generic' (query-major launch line on every rank); tc: the list-major scan on every rank."""
        import torch
        from pq_ref64 import assert_ref64, ref64
        from vectorindex_b200 import _lib
        L = _lib.lib()
        R = self.R
        env = Env(VIX_TC_SCAN="1" if tc else "0", VIX_SCAN_DEBUG="1")
        with env:
            fd, fi, fp = self.full.batch_search(q, k, nprobe=nprobe, return_probes=True)
            qq = torch.from_numpy(np.ascontiguousarray(q)).to(R.dev) if device else q
            tc0 = int(L.vix_scan_tc_launches())

            def search():
                (sd, si), text = with_stderr(lambda: self.sh.batch_search(qq, k, nprobe=nprobe))
                if device:
                    assert sd.is_cuda and si.is_cuda, "device queries: results must stay on the device"
                    torch.cuda.synchronize()
                return np_of(sd), np_of(si), text
            sd, si, text = R.step(f"{what}: sharded search", search)
            tcn = int(L.vix_scan_tc_launches()) - tc0

        def local():
            assert sd.shape == (len(q), k) and si.shape == (len(q), k), f"shape {sd.shape}"
            bad = np.nonzero((si != fi).any(1) | (bits(sd) != bits(fd)).any(1))[0]
            if bad.size:
                r = int(bad[0])
                j = int(np.nonzero((si[r] != fi[r]) | (bits(sd[r]) != bits(fd[r])))[0][0])
                raise AssertionError(f"{bad.size} rows differ from one GPU; row {r} place {j}: id {si[r, j]} dist "
                                     f"{sd[r, j]!r} ({bits(sd[r, j:j + 1])[0]:#010x}) vs one GPU id {fi[r, j]} dist "
                                     f"{fd[r, j]!r} ({bits(fd[r, j:j + 1])[0]:#010x})")
            kernels = ROUTE.findall(text)
            if tc:
                assert tcn == 1, f"list-major scan launched {tcn} times"
            elif route is not None:
                got = ["generic" if not g[1] else f"fast G{g[1]}" for g in kernels]
                assert got == [route], f"query-major launches {got}, expected [{route}]"
            assert R.comm.uses_peer_memory == R.want_peer or self.sh.comm.uses_peer_memory == R.want_peer, \
                f"peer memory state {self.sh.comm.uses_peer_memory}, expected {R.want_peer}"
        R.step(f"{what}: against one GPU", local)
        R.same_everywhere(f"{what}: every rank's answer", [bits(sd), si])

        def against_ref():
            if R.rank != 0:
                return
            off, codes, lids, _ = self.lists()
            rows = np.arange(len(q)) if len(q) <= ref_rows else np.linspace(0, len(q) - 1, ref_rows).astype(np.intp)
            ref = ref64(q[rows], self.coarse, self.cb, fp[rows], off, codes, lids, k, self.metric)
            assert_ref64(sd[rows], si[rows], ref)
        R.step(f"{what}: float64 reference", against_ref)
        return sd, si, fp


def clustered(rng, coarse, n, home=None, noise=0.3):
    kc, d = coarse.shape
    home = rng.integers(0, kc, n) if home is None else home
    return (coarse[home] + noise * rng.standard_normal((n, d))).astype(np.float32)


def random_problem(R, seed, metric, d, m, kc, n, ks=256, bounds=None, skip=(), comm=None, home=None, device=False,
                   noise=0.3):
    rng = np.random.default_rng(seed)
    coarse = rng.standard_normal((kc, d)).astype(np.float32)
    cb = (0.3 * rng.standard_normal((m, ks, d // m))).astype(np.float32)
    P = Problem(R, coarse, cb, metric, ks=ks, bounds=bounds, comm=comm)
    xb = clustered(rng, coarse, n, home, noise)
    ids = rng.permutation(n).astype(np.int64) * 3 + 7
    P.add(f"seed {seed}", xb, ids, hand_out(rng, n, R.world, skip), device=device)
    P.rng = rng
    return P


def block_sizes(world):
    return sorted({1, max(world - 1, 1), 4 * world - 1, 4 * world + 1, 333})


# ------------------------------------------------------------------------------------------------ cases
def case_blocks(R):
    """nq from 1 to 333 at the edges of the 4-row query blocks (some ranks own an empty block), host and device queries,
    asynchronous mode; the fast kernel at m = 48, L2 and IP; ragged contributions, the last rank (L2) or the first (IP)
    handing in nothing."""
    from vectorindex_b200 import _lib
    for metric in (0, 1):
        P = random_problem(R, 11 + metric, metric, 96, 48, 64, 6000, skip=(R.world - 1,) if metric == 0 else (0,))
        for nq in block_sizes(R.world):
            q = clustered(P.rng, P.coarse, nq)
            P.compare(f"blocks {METRICS[metric]} nq {nq}", q, 10, 9, route="fast G3")
        q = clustered(P.rng, P.coarse, 333)
        P.compare(f"blocks {METRICS[metric]} device queries", q, 10, 9, route="fast G3", device=True)
        _lib.lib().vix_set_async(1)
        try:
            P.compare(f"blocks {METRICS[metric]} device queries, asynchronous", q[:4 * R.world + 1], 16, 9, route="fast G3",
                      device=True)
        finally:
            _lib.lib().vix_set_async(0)
    R.log(f"ok blocks: nq {block_sizes(R.world)}, host and device queries, asynchronous mode, route fast G3, L2 and IP")


def case_k_nprobe(R):
    """k = 1 and VIX_MAX_K (the merge of world x 512 keys), k above the vectors every shard probes (nprobe 1) and above the
    whole index; nprobe 1, kc, one above the lists any single rank owns, and 512 at kc = 600."""
    for metric in (0, 1):
        P = random_problem(R, 21 + metric, metric, 96, 48, 64, 6000)
        q = clustered(P.rng, P.coarse, 4 * R.world + 1)
        most = int(np.diff(P.bounds).max())
        for k, nprobe in ((1, 9), (MAX_K, 9), (MAX_K, 1), (20, 1), (20, P.kc), (20, most + 1)):
            P.compare(f"k {k} nprobe {nprobe} {METRICS[metric]}", q, k, nprobe, route="fast G3")
        tiny = random_problem(R, 23 + metric, metric, 32, 16, 16, 300)
        qt = clustered(tiny.rng, tiny.coarse, 2 * R.world + 3)
        sd, si, _ = tiny.compare(f"k above the index {METRICS[metric]}", qt, MAX_K, 16, route="fast G1")
        R.step("padding", lambda: Problem._expect((si[:, 300:] == -1).all() and np.isnan(sd[:, 300:]).all(),
                                                  "results past the 300 stored rows are not -1 / NaN"))
        wide = random_problem(R, 25 + metric, metric, 32, 16, 600, 6000)
        qw = clustered(wide.rng, wide.coarse, 2 * R.world + 1)
        wide.compare(f"nprobe 512 at kc 600 {METRICS[metric]}", qw, 64, 512, route="fast G1")
    R.log("ok k_nprobe: k 1 / 512 / above every probed shard / above the index, nprobe 1 / kc / above a rank's lists / "
          "512, routes fast G3 and G1, L2 and IP")


def case_partitions(R):
    """set_list_bounds edges: a rank that owns no lists (repeated bound), a rank whose lists are all empty, every row owned
    by one rank; and kc < world with the default equal-count blocks."""
    w = R.world
    for metric in (0, 1):
        kc = 48
        eq = np.array([kc * r // w for r in range(w + 1)])
        none = eq.copy()
        none[1] = 0                                                    # rank 0 owns no list
        P = random_problem(R, 31 + metric, metric, 32, 16, kc, 4000, bounds=none)
        q = clustered(P.rng, P.coarse, 4 * w + 1)
        P.compare(f"rank 0 owns no list {METRICS[metric]}", q, 10, 8, route="fast G1")
        rng = np.random.default_rng(32 + metric)
        home = rng.integers(0, int(eq[w - 1]), 4000)                    # the last rank's lists stay empty
        P = random_problem(R, 33 + metric, metric, 32, 16, kc, 4000, bounds=eq, home=home, noise=0.1)
        R.step("empty lists", lambda: Problem._expect(R.rank != w - 1 or P.local.count == 0, f"{P.local.count} rows"))
        q = clustered(P.rng, P.coarse, 4 * w + 1)
        P.compare(f"last rank's lists empty {METRICS[metric]}", q, 10, P.kc, route="fast G1")
        home = rng.integers(int(eq[1]), int(eq[2]), 4000)                # every row on rank 1
        P = random_problem(R, 35 + metric, metric, 32, 16, kc, 4000, bounds=eq, home=home, device=True, noise=0.1)
        R.step("one owner", lambda: Problem._expect((R.rank == 1) == (P.local.count == 4000), f"{P.local.count} rows"))
        q = clustered(P.rng, P.coarse, 4 * w + 1)
        P.compare(f"every row on rank 1 {METRICS[metric]}", q, 10, 8, route="fast G1")
        P = random_problem(R, 37 + metric, metric, 32, 16, w - 1, 500)  # kc < world, default bounds
        q = clustered(P.rng, P.coarse, 4 * w - 1)
        P.compare(f"kc {w - 1} < world {METRICS[metric]}", q, 10, w - 1, route="fast G1")
    R.log("ok partitions: a rank owning no list, a rank with only empty lists, all rows on one rank, kc < world; L2 and IP")


def case_routes(R):
    """the generic kernel (m = 12, d = 36: dsub 3), ks = 16 (packed nibbles, the generic kernel), the fast kernel at m = 16;
    and the list-major tensor-core scan (L2, dsub = 2) on every rank, which must also give the query-major scan's bits."""
    for metric in (0, 1):
        for name, d, m, ks, route in (("generic", 36, 12, 256, "generic"), ("ks16", 32, 16, 16, "generic"),
                                      ("fast16", 32, 16, 256, "fast G1")):
            P = random_problem(R, zlib.crc32(f"{name}{metric}".encode()) & 0xFFFF, metric, d, m, 24, 3000, ks=ks)
            q = clustered(P.rng, P.coarse, 4 * R.world + 1)
            P.compare(f"{name} {METRICS[metric]}", q, 10, 6, route=route)
            P.compare(f"{name} {METRICS[metric]} k 512", q, MAX_K, 6, route=route)
    P = random_problem(R, 41, 0, 96, 48, 64, 8000)
    q = clustered(P.rng, P.coarse, 333)
    td, ti, _ = P.compare("list-major", q, 10, 9, tc=True)
    qd, qi, _ = P.compare("list-major vs query-major", q, 10, 9, route="fast G3")
    R.step("list-major == query-major", lambda: Problem._expect(np.array_equal(ti, qi) and np.array_equal(bits(td), bits(qd)),
                                                                "the two scans differ"))
    P.compare("list-major, second call", q, 10, 9, tc=True)
    R.log("ok routes: generic (m 12, d 36), ks 16 (generic), fast G1 (m 16), fast G3 (m 48), L2 and IP; list-major "
          "tensor-core scan (L2, m 48) on every rank, twice, equal to the query-major scan")


def case_ties(R):
    """Ties across ranks, on grid-valued data (every sum exact whatever its order): the same codes in lists owned by
    different ranks at the same distance (centroids of equal norm orthogonal to the query) and one id stored in lists of
    two ranks -- the one-GPU answer, ties to the smaller id, the twice-stored id twice.  And a zero query under IP: every
    score is 0, the ids are the k smallest probed ids and every distance is -0 (the sign one GPU returns)."""
    w = R.world
    step = 2.0 ** -5
    g = lambda a: (np.round(np.asarray(a) / step) * step).astype(np.float32)
    kc, m, dsub = 4 * w, 32, 2
    d = m * dsub
    half = d // 2                                                      # centroids in the low half, residuals in the high
    assert kc <= half
    coarse = np.zeros((kc, d), np.float32)
    coarse[np.arange(kc), np.arange(kc)] = 2.0
    rng = np.random.default_rng(51)
    cb = g(0.5 * rng.standard_normal((m, 256, dsub)))
    cb[:, 0] = 0.0                                                     # code 0 encodes a zero residual exactly
    lo_sq = half // dsub                                               # sub-quantisers of the low half
    pick = rng.integers(1, 256, (3, m - lo_sq))                        # three residual patterns in the high half
    pattern = lambda p: np.concatenate([np.zeros(half, np.float32), cb[np.arange(lo_sq, m), pick[p]].ravel()])
    per_list = 40
    home = np.repeat(np.arange(kc), per_list)
    pat = rng.integers(0, 3, home.size)
    xb = np.stack([coarse[h] + pattern(p) for h, p in zip(home, pat)]).astype(np.float32)
    ids = rng.permutation(home.size).astype(np.int64) * 5 + 100
    twin = np.nonzero(pat == 0)[0]
    a = twin[home[twin] < kc // w][0]                                 # a row on rank 0 ...
    b = twin[home[twin] >= kc - kc // w][-1]                          # ... and one on the last rank share an id
    ids[b] = ids[a] = 99                                               # the smallest id: returned first, twice
    P = Problem(R, coarse, cb, 0)
    P.add("ties", xb, ids, hand_out(rng, xb.shape[0], w))
    q = np.tile(pattern(0), (3, 1)).astype(np.float32)
    for k in (10, 64):
        sd, si, _ = P.compare(f"ties k {k}", q, k, kc, route="fast G2")
        want = np.sort(ids[pat == 0])[:k]                             # (fewer than k at one rank: the rest is farther)

        def tied():
            t = want.size
            assert np.array_equal(si[0, :t], want), f"ids {si[0][:12]} vs the {t} smallest tied ids {want[:12]}"
            assert (bits(sd[:, :t]) == bits(sd[:, :1])).all(), "tied rows with different distance bits"
        R.step(f"ties k {k}: smallest ids first", tied)
    R.step("twice-stored id", lambda: Problem._expect((si[0] == ids[a]).sum() == 2, "the id stored on two ranks is not "
                                                                                    "returned twice"))
    for name, d, m, route in (("fast16", 32, 16, "fast G1"), ("generic12", 36, 12, "generic")):
        P = random_problem(R, 53 + m, 1, d, m, 16, 3000)
        z = np.zeros((3, d), np.float32)
        for nprobe in (4, 16):
            sd, si, fp = P.compare(f"zero IP query {name} nprobe {nprobe}", z, 10, nprobe, route=route)

            def zero():
                off, _, lids, _ = P.lists()
                assert (bits(sd) == NEG_ZERO).all(), f"zero distances {sorted(set(hex(v) for v in bits(sd).ravel()))}, " \
                                                     "expected -0 (0x80000000)"
                for r in range(len(z)):
                    want = np.sort(np.concatenate([lids[off[l]:off[l + 1]] for l in fp[r] if l >= 0]))[:10]
                    assert np.array_equal(si[r], want), f"row {r}: ids {si[r]} vs the smallest probed {want}"
            R.step(f"zero IP query {name}: -0 and the smallest ids", zero)
    R.log("ok ties: equal codes on different ranks and one id on two ranks (L2, grid data, k 10 / 64), zero IP query "
          "(fast G1 and generic): -0, smallest probed ids")


def case_zero_ip(R):
    """the zero inner-product query alone: every distance -0 as one GPU returns it"""
    P = random_problem(R, 61, 1, 32, 16, 16, 3000)
    z = np.zeros((2, 32), np.float32)
    sd, _, _ = P.compare("zero IP query", z, 10, 4, route="fast G1")
    R.log(f"ok zero_ip: distance bits {bits(sd)[0, :3]}")


def case_region(R):
    """Exchange-region growth and reuse on one new communicator: nq 10, then 3000 (past the first 1024-row capacity), then k
    and nprobe above every earlier call, then small again; then a second index of another d and metric on the same
    communicator, searches alternating between the two."""
    from vectorindex_b200.index import Comm
    comm = Comm.from_torch()
    try:
        A = random_problem(R, 71, 0, 32, 16, 40, 5000, comm=comm)
        qa = clustered(A.rng, A.coarse, 3000)
        for nq, k, nprobe in ((10, 10, 4), (3000, 10, 4), (50, 200, 40), (7, 5, 2)):
            A.compare(f"region A nq {nq} k {k} nprobe {nprobe}", qa[:nq], k, nprobe, route="fast G1")
        B = random_problem(R, 72, 1, 96, 48, 24, 3000, comm=comm)
        qb = clustered(B.rng, B.coarse, 1500)
        for i, (nq, k, nprobe) in enumerate(((1500, 10, 8), (5, 300, 24), (600, 20, 3))):
            B.compare(f"region B nq {nq} k {k} nprobe {nprobe}", qb[:nq], k, nprobe, route="fast G3")
            A.compare(f"region A again ({i})", qa[:nq], min(k, 100), min(nprobe, 40), route="fast G1")
        R.step("region state", lambda: Problem._expect(comm.uses_peer_memory == R.want_peer, f"{comm.uses_peer_memory}"))
    finally:
        comm.close()
    R.log("ok region: growth in nq, k, nprobe and d on one communicator, two indexes alternating")


def case_mutate(R):
    """Build and removal interleaved with search: a second add whose rows all land on the last rank, after a search; then a
    removal of ids (some stored twice, some never stored) through ShardedIVFPQIndex.remove; search again."""
    w = R.world
    P = random_problem(R, 81, 0, 32, 16, 32, 4000)
    q = clustered(P.rng, P.coarse, 4 * w + 1)
    P.compare("before the second add", q, 20, 8, route="fast G1")
    rng = np.random.default_rng(82)
    last = rng.integers(int(P.bounds[w - 1]), P.kc, 1500)
    xb = clustered(rng, P.coarse, 1500, last, noise=0.1)
    ids = rng.permutation(1500).astype(np.int64) * 3 + 8                 # ids of their own, some equal to earlier ones
    ids[:40] = 7 + 3 * np.arange(40)
    count0 = P.local.count
    P.add("second add", xb, ids, hand_out(rng, 1500, w), device=True)
    R.step("second add on the last rank only", lambda: Problem._expect(
        P.local.count - count0 == (1500 if R.rank == w - 1 else 0), f"{P.local.count - count0} rows arrived"))
    P.compare("after the second add", q, 20, 8, route="fast G1")
    gone = np.concatenate([ids[::7], 7 + 3 * np.arange(0, 4000, 5), [2 ** 32 - 2, 3]]).astype(np.int64)
    P.remove("removal", gone)
    P.compare("after the removal", q, 20, 8, route="fast G1")
    P.compare("after the removal, k 512", q, MAX_K, P.kc, route="fast G1")
    R.log("ok mutate: add after a search (all rows on the last rank), removal through ShardedIVFPQIndex.remove, search")


def case_replicated(R):
    """ReplicatedIVFPQIndex on GPUs: ragged and empty contributions; every replica's lists equal (and the one-GPU index's,
    filled rank by rank); the gathered answer equals the one-GPU index bit for bit for host and device queries, ragged and
    empty query blocks, and gather=False returns this rank's block of it."""
    import torch
    from vectorindex_b200.index import IVFPQIndex, ReplicatedIVFPQIndex
    w = R.world
    for metric in (0, 1):
        rng = np.random.default_rng(91 + metric)
        d, m, kc, n = 96, 48, 32, 5000
        coarse = rng.standard_normal((kc, d)).astype(np.float32)
        cb = (0.3 * rng.standard_normal((m, 256, d // m))).astype(np.float32)
        xb = clustered(rng, coarse, n)
        ids = rng.permutation(n).astype(np.int64) * 2 + 1
        src = hand_out(rng, n, w, skip=(w - 1,) if metric == 0 else (0,))
        rp = ReplicatedIVFPQIndex(d, METRICS[metric], nlist=kc, nprobe=8, m=m)
        rp.set_parameters(coarse, cb)
        full = IVFPQIndex(d, METRICS[metric], nlist=kc, nprobe=8, m=m)
        full.set_coarse(coarse)
        full.set_codebooks(cb)
        order = np.concatenate([np.nonzero(src == r)[0] for r in range(w)])
        full.batch_insert(xb[order], ids[order])
        mine = np.nonzero(src == R.rank)[0]
        R.step("replicated add", lambda: rp.add(xb[mine], ids[mine]))
        exp = rp.local.export_lists()
        fexp = full.export_lists()
        R.step("replica lists", lambda: Problem._expect(all(np.array_equal(a, b) for a, b in zip(exp, fexp)),
                                                        "a replica's lists differ from the one-GPU index's"))
        R.same_everywhere("replica lists on every rank", [np.frombuffer(hashlib.sha256(b"".join(
            np.ascontiguousarray(a).tobytes() for a in exp)).digest(), np.uint8)])
        for nq in block_sizes(w):
            q = clustered(rng, coarse, nq)
            fd, fi = full.batch_search(q, 10)
            for device in (False, True):
                qq = torch.from_numpy(q).to(R.dev) if device else q
                gd, gi = R.step("replicated search", lambda: rp.batch_search(qq, 10))
                bd, bi = R.step("replicated search, gather=False", lambda: rp.batch_search(qq, 10, gather=False))
                lo, cnt, _ = rp.query_block(nq)

                def check():
                    for name, (dd, ii), rows in (("gathered", (gd, gi), slice(0, nq)), ("own block", (bd, bi), slice(lo, lo + cnt))):
                        dd, ii = np_of(dd), np_of(ii)
                        assert ii.shape == (rows.stop - rows.start, 10), f"{name}: shape {ii.shape}"
                        assert np.array_equal(ii, fi[rows]) and np.array_equal(bits(dd), bits(fd[rows])), \
                            f"{name} (nq {nq}, device {device}) differs from one GPU"
                R.step(f"replicated {METRICS[metric]} nq {nq} device {device}", check)
                R.same_everywhere("replicated answer on every rank", [bits(gd), np_of(gi)])
    R.log("ok replicated: ragged / empty contributions, identical replicas, gathered and own-block answers equal one GPU "
          "for host and device queries, L2 and IP")


def case_bad_id(R):
    """Collective validation in vix_sharded_add (called directly, so that one rank takes it too): rank 0 hands in one row
    with id 2^32 - 1 whose list another rank owns.  Every rank must refuse the call, naming rank 0, and every rank's count
    and lists must be as before; a valid add then still works."""
    from vectorindex_b200 import _lib
    from vectorindex_b200._lib import VectorIndexError
    w = R.world
    P = random_problem(R, 101, 0, 32, 16, 16, 2000)
    before = (P.local.count, P.local.export_lists())
    target = int(P.bounds[w - 1])                                      # a list the last rank owns
    rng = np.random.default_rng(102)
    x = clustered(rng, P.coarse, 3 * w, np.full(3 * w, target), noise=0.01)
    ids = 50_000 + np.arange(3 * w, dtype=np.int64)
    mine = slice(3 * R.rank, 3 * R.rank + 3)
    xm, im = x[mine].copy(), ids[mine].copy()
    if R.rank == 0:
        im[1] = 2 ** 32 - 1

    def refused():
        bounds = np.ascontiguousarray(P.bounds, np.int64)
        try:
            _lib.check(_lib.lib().vix_sharded_add(P.local._h, P.sh.comm._c, _lib.ptr(bounds), _lib.ptr(xm), _lib.ptr(im),
                                                  C.c_int64(len(im))))
        except VectorIndexError as e:
            assert e.status == ERR_INVALID_PARAM, f"status {e.status}: {e}"
            assert "rank 0" in str(e), f"the error does not name rank 0: {e}"
            return
        raise AssertionError("vix_sharded_add accepted the rows")
    R.step("id 2^32 - 1 on rank 0", refused)

    def unchanged():
        assert P.local.count == before[0], f"count {before[0]} -> {P.local.count}"
        assert all(np.array_equal(a, b) for a, b in zip(P.local.export_lists(), before[1])), "lists changed"
    R.step("nothing stored", unchanged)
    P.add("valid add after the refusal", x, ids, np.repeat(np.arange(w), 3))
    q = clustered(rng, P.coarse, 4 * w + 1)
    P.compare("after the refusal", q, 10, 8, route="fast G1")
    R.log("ok bad_id: every rank refused the call naming rank 0, nothing stored, a valid add afterwards")


CASES = {"blocks": case_blocks, "k_nprobe": case_k_nprobe, "partitions": case_partitions, "routes": case_routes,
         "ties": case_ties, "zero_ip": case_zero_ip, "region": case_region, "mutate": case_mutate,
         "replicated": case_replicated, "bad_id": case_bad_id}


def main():
    import torch.distributed as dist
    names = sys.argv[1:] or [n for n in CASES if n != "zero_ip"]        # (zero_ip: the zero-query check of `ties` alone)
    R = Ranks()
    failed = []
    try:
        R.agree("peer memory", None)
        for name in names:
            try:
                CASES[name](R)
            except CaseFailure as e:                                   # raised on every rank at the same point
                failed.append(f"{name}: {e}")
                R.log(f"FAILED {name}: {e}")
        R.log(f"edges: world {R.world}, peer memory {R.comm.uses_peer_memory}, {len(names) - len(failed)} of {len(names)} "
              "cases ok")
    finally:
        R.comm.close()
        dist.barrier()
        dist.destroy_process_group()
    if failed:
        sys.exit(1)


if __name__ == "__main__":
    main()
