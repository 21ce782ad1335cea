"""One rank of a W-way sharded C5 index on ONE GPU (kernel work without a multi-GPU box):

    python scripts/shard_emul.py [world=8] [rank=0] [workload=c5]

Trains the workload's coarse quantiser / codebooks, assigns + encodes every database chunk, keeps only the rows whose
inverted list lies in `rank`'s block (what the all-to-all of ShardedIVFPQIndex.add delivers), then times the rank's
share of a sharded search step: probe_range over its centroid block, and search_with_probes with the GLOBAL probe
lists (taken from a full probe selection, which is what all-gather + mergeTopK produce)."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import bench  # noqa: E402
from vectorindex_b200._lib import KMeansCfg, PQTrainCfg  # noqa: E402
from vectorindex_b200.index import IVFPQIndex, list_block  # noqa: E402

world = int(sys.argv[1]) if len(sys.argv) > 1 else 8
rank = int(sys.argv[2]) if len(sys.argv) > 2 else 0
cfg = dict(bench.PRESETS[sys.argv[3] if len(sys.argv) > 3 else "c5"])
dev = torch.device("cuda", 0)
synth = bench.Synth(cfg, dev)
n, d, nlist, m, k, nq, nprobe = cfg["n"], cfg["d"], cfg["nlist"], cfg["m"], cfg["k"], cfg["nq"], cfg["nprobe"]
idx = IVFPQIndex(d, cfg.get("metric", "euclidean"), nlist=nlist, nprobe=nprobe, m=m)
ntrain = min(n, max(32 * nlist, 65536))
xt = torch.cat([synth.rows(b, c) for b, c in bench.chunks_of(ntrain)])
idx.optimize(xt, KMeansCfg(1024, 6, 1e-4, 42, 0, False, 1), PQTrainCfg(0, 8, 1e-4, 1024, 65536, 42, 0, 0, 1))
del xt
begin, count = list_block(nlist, rank, world)
for b, c in bench.chunks_of(n):
    x = synth.rows(b, c)
    asg, codes = idx.encode(x)
    keep = (asg >= begin) & (asg < begin + count)
    ids = torch.arange(b, b + c, dtype=torch.int64, device=dev)[keep]
    idx.add_encoded(asg[keep].contiguous(), codes[keep].contiguous(), ids.contiguous())
    del x
idx.list_sizes()
torch.cuda.synchronize()
print(f"rank {rank}/{world}: {idx.count} vectors in lists [{begin}, {begin + count})", flush=True)

q = synth.queries(nq)
_, _, probes = idx.batch_search(q, k, return_probes=True)          # global probe lists (full selection)
probes = probes.contiguous()
e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
per = (nq + world - 1) // world
qblk = q[rank * per:(rank + 1) * per].contiguous()                  # the rank's query block of the probe stage
for it in range(4):
    if it == 3:
        torch.cuda.profiler.start()                               # ncu --profile-from-start off: one full step
    e[3].record()
    idx.probe_range(qblk, nprobe, 0, nlist)                         # what the sharded search runs: its queries x all centroids
    e[0].record()
    pid, psc = idx.probe_range(q, nprobe, begin, count)              # (first version: all queries x its centroid block)
    e[1].record()
    dd, ii = idx.search_with_probes(q, k, probes)
    e[2].record()
    torch.cuda.synchronize()
    if it == 3:
        torch.cuda.profiler.stop()
    print(f"  iter {it}: probe by query block {e[3].elapsed_time(e[0]):.3f} ms, by centroid block {e[0].elapsed_time(e[1]):.3f} ms, search_with_probes {e[1].elapsed_time(e[2]):.3f} ms", flush=True)
dd, ii, st = idx.search_with_probes(q, k, probes, stats=True)
tot = max(1, st.cycles_prologue + st.cycles_scan + st.cycles_tail)
gbs = st.code_bytes_scanned / (st.ms_scan * 1e-3) / 1e9
print(f"scan stage {st.ms_scan:.3f} ms, {st.code_bytes_scanned / 1e9:.3f} GB of codes = {gbs:.0f} GB/s; per-CTA phase split: "
      f"prologue {st.cycles_prologue / tot:.3f} scan {st.cycles_scan / tot:.3f} tail {st.cycles_tail / tot:.3f}; "
      f"cycles/query/SM {tot / nq:.0f} (prologue {st.cycles_prologue / nq:.0f}, scan {st.cycles_scan / nq:.0f}, "
      f"tail {st.cycles_tail / nq:.0f}); pieces per query: select {st.cycles_select / nq:.0f} probe table "
      f"{st.cycles_probe_table / nq:.0f} lut {st.cycles_lut / nq:.0f}; merge candidates per query "
      f"{st.merge_candidates / nq:.1f}")
