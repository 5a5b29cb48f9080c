"""Edge-shape check of the bank-aligned two-slot kernel (grid tier fast path) against the CPU oracle.
   python tools/grid_check.py [rows] [max_iter]     (small sizes run under compute-sanitizer in a minute)
Shapes: ragged row count (not a multiple of 4 / 24), empty rows, rows dropped by the row filter, long rows that make
oversize (flagged) blocks, a chunk fuller than a stage, and a second plain locus."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("SBQ_DUAL_VERIFY", "1")   # libsbq checks the prepared layout (distinct banks per step, disjoint partner rows)
import oracle  # noqa: E402
from strawberry_b200 import api, synth  # noqa: E402


def edge_locus(R, T, seed):
    rng = np.random.default_rng(seed)
    k = 1 + rng.poisson(40.0, R)
    k[rng.random(R) < 0.01] = 0                       # empty rows
    long_rows = rng.choice(R, max(2, R // 400), replace=False)
    k[long_rows] = rng.integers(150, 400, long_rows.size)   # oversize blocks
    burst = min(R - 30, R // 2)
    k[burst:burst + 24] = 90                          # one chunk above the stage capacity, blocks still sortable? (4*90 > 252: flagged)
    k[burst + 24:burst + 48] = 60                     # 24 rows x 60 = 1440 > 1344: chunk read from global memory in the sorted layout
    k = np.minimum(k, T)
    row_ptr = np.zeros(R + 1, np.int64)
    np.cumsum(k, out=row_ptr[1:])
    col = np.concatenate([np.sort(rng.choice(T, kk, replace=False)) for kk in k]).astype(np.int32) if R else np.zeros(0, np.int32)
    alpha = 10.0 ** rng.uniform(-4.0, -1.5, int(row_ptr[-1]))
    dropped = rng.choice(R, max(1, R // 100), replace=False)
    for i in dropped:
        alpha[row_ptr[i]:row_ptr[i + 1]] = 5e-6           # row filter drops these
    count = rng.integers(0, 4, R).astype(np.int32)
    return dict(loc_row_off=np.array([0, R], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=row_ptr, col=col, alpha=alpha,
                count=count, iso_len=rng.integers(400, 8001, T).astype(np.int32), total_mapped_reads=int(count.sum()), meta={})


rows = int(sys.argv[1]) if len(sys.argv) > 1 else 60001   # > 12 chunks per CTA: the stage refill path runs
max_iter = int(sys.argv[2]) if len(sys.argv) > 2 else 1000
b = synth.concat([edge_locus(rows, 733, 11), synth.giant(n_loci=1, rows_per_locus=rows // 2 + 3, seed=4), edge_locus(rows // 3 + 1, 90, 12)])
q = api.Quantifier(max_iter=max_iter)
q.set_plan(3, 0)
q.submit_flat(b)
q.run(b["total_mapped_reads"])
res = q.results()
st = q.stats()
ora = oracle.quantify_batch(b, b["total_mapped_reads"], max_iter=max_iter) if max_iter != 1000 else oracle.quantify_batch(b, b["total_mapped_reads"])
print("status", res["status"], ora["status"], "iters", res["iters"], ora["iters"], "launches", st["kernel_launches"])
scale = np.maximum(np.abs(ora["theta"]), 1e-9 * max(1.0, float(b["count"].sum())))
worst = float((np.abs(res["theta"] - ora["theta"]) / scale).max())
print("worst rel err", worst)
assert np.array_equal(res["status"], ora["status"]) and np.array_equal(res["iters"], ora["iters"]) and worst < 1e-6
q.solve(b["total_mapped_reads"])
q.finalize_tpm(q.fpkm_sum())
q.download()
again = q.results()
assert np.array_equal(res["theta"], again["theta"]), "second solve of the resident batch differs"
print("grid_check ok")
