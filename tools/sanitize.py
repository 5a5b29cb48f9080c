"""Small all-tier workload for compute-sanitizer (memcheck / racecheck / synccheck): warp tier, cluster tier with cluster
sizes 1 / 4 / 16 (64-, 128- and 512-thread CTAs; all-to-all and owner exchange), grid tier (two-slot kernel incl. its layout and
packing passes, TMA ring kernel; full grid and the 32-CTA sub-grid of the "small giants" running beside the other tiers), the bias kernels (warp tier and clusters of 1 - 16 CTAs), the on-device generator, the device
class-table builder and the GPU class weights."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from strawberry_b200 import api, builder, synth  # noqa: E402
import locusgen  # noqa: E402

b = synth.concat([synth.human_shaped(n_loci=60, total_fragments=30_000, seed=5, max_rows=400),
                  synth.giant(n_loci=1, rows_per_locus=3000, seed=4)])
from strawberry_b200 import partition  # noqa: E402
# Forced grid tier: the giant locus alone. KNOWN ANOMALY (profiles/README.md): when a few dozen TINY loci (R ~ 10 rows) are forced through
# the giant-locus kernel together in one launch, compute-sanitizer's racecheck aborts the run with "an illegal instruction was
# encountered" and reports 0 hazards; memcheck, synccheck, initcheck and the layout verifier pass on the same input, the results equal
# the oracle (tests/test_gpu_em.py forces all 136 golden loci through this tier), and the planner never produces that shape (the tier
# takes loci of >= 300 k non-zeros). Every production-shaped input - one or several giant loci per launch - is racecheck-clean.
b3, _ = partition.take(b, np.array([60]))
for tier, cs, it in ((0, 0, 30), (2, 1, 10), (2, 4, 10), (2, 16, 10), (3, 0, 6)):
    q = api.Quantifier(max_iter=it)
    q.set_plan(tier, cs)
    q.submit_flat(b3 if tier == 3 else b)
    q.run(b["total_mapped_reads"])
    r = q.results()
    print("tier", tier, "cs", cs, "ok", np.isfinite(r["theta"]).all(), q.stats()["kernel_launches"])
    q.close()
q = api.Quantifier(max_iter=3)                            # planner-chosen tiers with a "small giant": 32-CTA sub-grid on its own stream beside the other tiers
bs = synth.concat([b, synth.giant(n_loci=1, rows_per_locus=7000, seed=6)])
q.submit_flat(bs)
q.run(bs["total_mapped_reads"])
print("sub-grid ok", np.isfinite(q.results()["theta"]).all(), [r["cluster_size"] for r in q.launch_stats() if r["kernel"].startswith("em_grid")])
q.close()
q = api.Quantifier(bias_mode=1, max_out_it=2, max_theta_it=4, max_bias_it=2)     # bias kernels: warp tier + clusters of 1 .. 16 CTAs
bb = synth.concat([b] + [synth.giant(n_loci=1, rows_per_locus=r, seed=4) for r in (200, 600, 1500)])     # + 9.6 k / 29 k / 72 k non-zeros: clusters of 2, 4, 8
q.submit_flat(bb)
q.set_covariates(synth.covariates(bb, seed=3))
q.run(bb["total_mapped_reads"])
print("bias ok", np.isfinite(q.results()["theta"]).all(), q.stats()["kernel_launches"])
q.close()
rng = np.random.default_rng(8)                            # forced grid tier, rows of 60 - 99 non-zeros (the two-slot layout takes <= 56 on average): TMA ring kernel
T, R = 200, 600
k = rng.integers(60, 100, R)
rp = np.concatenate([[0], np.cumsum(k)]).astype(np.int64)
bd = dict(loc_row_off=np.array([0, R], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=rp,
          col=np.concatenate([np.sort(rng.choice(T, kk, replace=False)) for kk in k]).astype(np.int32), alpha=10.0 ** rng.uniform(-4, -1.5, int(rp[-1])),
          count=rng.integers(1, 100, R).astype(np.int32), iso_len=rng.integers(300, 5000, T).astype(np.int32), total_mapped_reads=1_000_000)
q = api.Quantifier(max_iter=4)
q.set_plan(3, 0)
q.submit_flat(bd)
q.run(bd["total_mapped_reads"])
print("tma ring ok", np.isfinite(q.results()["theta"]).all(), [r["kernel"] for r in q.launch_stats() if r["n_loci"]])
q.close()
q = api.Quantifier(max_iter=5)                           # device generator -> two-slot kernel (layout + packing passes)
q.synth_giant([0, 3], 7000)
q.solve(14000)
q.finalize_tpm(q.fpkm_sum())
q.download()
print("synth giant ok", np.isfinite(q.results()["theta"]).all(), q.stats()["loci_grid"])
q.clear()                                                 # device class-table builder + GPU weights
q.set_insert_model(builder.Model.normal(200.0, 40.0), 50)
for seed in (3, 4, 6, 9):
    isoforms, hits, _ = locusgen.random_locus(seed)
    builder.submit_raw(q, [locusgen.transcript_features(ex) for ex in isoforms], [(m, builder.pair_features(l, r)) for m, l, r in hits], read_len=50)
q.run(100000)
print("raw builder ok", np.isfinite(q.results()["theta"]).all(), q.stats()["n_row"])
q.close()
