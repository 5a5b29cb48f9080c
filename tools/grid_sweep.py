"""Randomised parity sweep of the grid tier (two-slot kernel where it qualifies) against the CPU oracle:
   isoform counts from 17 to 1290, 3 to 55 non-zeros per row on average, ragged row counts, zero counts, dropped rows.
   python tools/grid_sweep.py"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("SBQ_DUAL_VERIFY", "1")
import oracle  # noqa: E402
from strawberry_b200 import api, synth  # noqa: E402


def locus(R, T, kmean, seed):
    rng = np.random.default_rng(seed)
    k = np.minimum(T, np.maximum(0, rng.poisson(kmean, R)))
    k[rng.random(R) < 0.02] = 0
    row_ptr = np.zeros(R + 1, np.int64)
    np.cumsum(k, out=row_ptr[1:])
    col = np.concatenate([np.sort(rng.choice(T, kk, replace=False)) for kk in k] + [np.zeros(0, np.int64)]).astype(np.int32)
    alpha = 10.0 ** rng.uniform(-4.0, -1.5, int(row_ptr[-1]))
    for i in rng.choice(R, max(1, R // 150), replace=False):
        alpha[row_ptr[i]:row_ptr[i + 1]] = 3e-6
    count = rng.integers(0, 6, R).astype(np.int32)
    return dict(loc_row_off=np.array([0, R], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=row_ptr, col=col, alpha=alpha,
                count=count, iso_len=rng.integers(300, 9000, T).astype(np.int32), total_mapped_reads=int(count.sum()), meta={})


cases = [(4999, 17, 3), (7001, 64, 20), (6007, 257, 55), (5003, 1000, 40), (4001, 1290, 30), (9999, 500, 8), (3, 40, 10), (12345, 130, 47)]
worst_all = 0.0
for n, (R, T, km) in enumerate(cases):
    b = synth.concat([locus(R, T, km, 100 + n), locus(max(9, R // 7), max(16, T // 2), km, 200 + n)])
    q = api.Quantifier(max_iter=300)
    q.set_plan(3, 0)
    q.submit_flat(b)
    q.run(b["total_mapped_reads"])
    res = q.results()
    kern = sorted({r["kernel"] for r in q.launch_stats()})
    q.close()
    ora = oracle.quantify_batch(b, b["total_mapped_reads"], max_iter=300)
    scale = np.maximum(np.abs(ora["theta"]), 1e-9 * max(1.0, float(b["count"].sum())))
    worst = float((np.abs(res["theta"] - ora["theta"]) / scale).max())
    ok = np.array_equal(res["status"], ora["status"]) and np.array_equal(res["iters"], ora["iters"]) and worst < 1e-6
    worst_all = max(worst_all, worst)
    print(f"R={R:6d} T={T:5d} k~{km:2d}: {kern} status {res['status'].tolist()} iters {res['iters'].tolist()} worst rel err {worst:.2e} {'ok' if ok else 'MISMATCH'}")
    assert ok
print("grid_sweep ok, worst", worst_all)
