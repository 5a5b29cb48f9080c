"""Bootstrap replicates on the GPU (sbq_bootstrap): device time per replicate on the headline batch and on a wave of giant loci,
next to the point-estimate solve and the CPU restatement.

  python tools/bootstrap_bench.py --out profiles/r03_bootstrap.json

  headline  configs[1] (synth.human_shaped(), seed 2: 20 000 loci, 10 M fragments): --reps replicates in chunks of --chunk, each
            chunk preceded by --solves point-estimate sbq_solve calls on the same context (alternating, for the spread).
            Per replicate: resample ms, EM ms (EM launches + FPKM sum), E-steps (sum over loci) and fragment-iterations per second.
            Then --fresh replicates alone, each next to a fresh sbq_solve of the resampled batch (its EM time from the stats).
  giant     one wave of --giant-loci device-generated loci of the configs[3] shape (1 M single-fragment rows, 500-800 isoforms,
            ~48 entries per row; sbq_synth_giant): --giant-reps replicates.
  cpu       the oracle (oracle.quantify_batch: the C restatement of the reference EM, n_threads = os.cpu_count()) on --cpu-reps
            resampled headline replicates, as the CPU cost of the same replicates.
The card's name, power limit and clocks are read in the same run. The tool refuses to run without a GPU."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

SEED = 20240611


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, check=True).stdout
    return [dict(zip(q.split(","), (x.strip() for x in line.split(",")))) for line in out.strip().splitlines()]


def per_replicate(q, rep, st, frags):
    n = st["n"]
    em_s = st["em_ms"] / 1e3
    fi = int((rep["iters"].astype(np.int64) * frags[None, :]).sum())
    return dict(first=st["first"], n=n, resample_ms_per_rep=st["resample_ms"] / n, em_ms_per_rep=st["em_ms"] / n,
                total_ms_per_rep=st["total_ms"] / n, resample_share=st["resample_ms"] / st["total_ms"],
                em_iters_per_rep=float(rep["iters"].astype(np.int64).sum(axis=1).mean()),
                frag_iters_per_s=fi / em_s if em_s > 0 else None,
                status_counts={int(k): int(v) for k, v in zip(*np.unique(rep["status"], return_counts=True))})


def headline(args, api, synth):
    b = synth.human_shaped(seed=2)
    frags = np.add.reduceat(b["count"].astype(np.int64), b["loc_row_off"][:-1])
    q = api.Quantifier()
    q.submit_flat(api.pinned_batch(b))
    q.run(b["total_mapped_reads"])
    q.bootstrap(SEED + 1, 2)                     # warm-up: every kernel and allocation of the timed calls
    point_iters = q.results()["iters"]
    chunks, solves, max_iters = [], [], []
    for first in range(0, args.reps, args.chunk):
        for _ in range(args.solves):
            q.solve(b["total_mapped_reads"])
            s = q.stats()
            solves.append(dict(solve_ms=s["solve_ms"], em_ms=s["em_ms"]))
        n = min(args.chunk, args.reps - first)
        rep = q.bootstrap(SEED, n, first)
        max_iters += [int(x) for x in rep["iters"].max(axis=1)]
        chunks.append(per_replicate(q, rep, q.bootstrap_stats(), frags))
    point = q.stats()
    # the same replicates solved as fresh batches: separates the cost of the resampled data (iterations, critical path) from any
    # cost of the bootstrap path itself
    import bootstrap_ref as br
    fresh = []
    for r in range(args.fresh):
        single = q.bootstrap(SEED, 1, r)
        st1 = q.bootstrap_stats()
        rb = br.resampled_batch(b, SEED, r)
        qf = api.Quantifier()
        qf.submit_flat(api.pinned_batch(rb))
        qf.run(b["total_mapped_reads"])
        em_f = []
        for _ in range(args.solves):
            qf.solve(b["total_mapped_reads"])
            em_f.append(qf.stats()["em_ms"])
        qf.close()
        fresh.append(dict(replicate=r, bootstrap_em_ms=st1["em_ms"], fresh_solve_em_ms=em_f, max_locus_iters=int(single["iters"].max()),
                          em_iters_total=int(single["iters"].astype(np.int64).sum())))
    q.close()
    em = np.array([c["em_ms_per_rep"] for c in chunks])
    rs = np.array([c["resample_ms_per_rep"] for c in chunks])
    se = np.array([s["em_ms"] for s in solves])
    return dict(batch=dict(n_loci=int(point["n_loci"]), n_row=int(point["n_row"]), nnz=int(point["nnz"]), fragments=int(frags.sum())),
                replicates=args.reps, chunk=args.chunk, chunks=chunks, point_solves=solves,
                summary=dict(resample_ms_per_rep=dict(median=float(np.median(rs)), min=float(rs.min()), max=float(rs.max())),
                             em_ms_per_rep=dict(median=float(np.median(em)), min=float(em.min()), max=float(em.max())),
                             point_em_ms=dict(median=float(np.median(se)), min=float(se.min()), max=float(se.max())),
                             resample_share_max=float(max(c["resample_share"] for c in chunks))),
                point_estimate=dict(em_iters_total=int(point["em_iters_total"]), frag_iters=int(point["frag_iters"]),
                                    max_locus_iters=int(point_iters.max()), frag_iters_per_s=point["frag_iters"] / (float(np.median(se)) / 1e3)),
                replicate_max_locus_iters=max_iters, fresh_solves_of_replicates=fresh), b


def giant(args, api):
    rows = 1_000_000
    q = api.Quantifier()
    q.synth_giant(list(range(args.giant_loci)), rows)
    q.solve(rows * args.giant_loci)
    q.download()
    point = q.stats()
    frags = np.full(args.giant_loci, rows, np.int64)
    rep = q.bootstrap(SEED, args.giant_reps)
    out = per_replicate(q, rep, q.bootstrap_stats(), frags)
    q.close()
    return dict(loci=args.giant_loci, rows_per_locus=rows, nnz=int(point["nnz"]), point_solve_ms=point["solve_ms"],
                point_em_ms=point["em_ms"], point_em_iters_total=int(point["em_iters_total"]), replicates=out)


def cpu(args, batch):
    import bootstrap_ref as br
    import oracle
    n_threads = os.cpu_count()
    secs = []
    for r in range(args.cpu_reps):
        rb = br.resampled_batch(batch, SEED, r)
        t0 = time.perf_counter()
        oracle.quantify_batch(rb, batch["total_mapped_reads"], n_threads=n_threads)
        secs.append(time.perf_counter() - t0)
    return dict(what="oracle.quantify_batch (C restatement of the reference EmSolver + epilogue), wall time per replicate",
                n_threads=n_threads, replicates=args.cpu_reps, seconds=secs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--chunk", type=int, default=25)
    ap.add_argument("--solves", type=int, default=3)
    ap.add_argument("--giant-loci", type=int, default=25)
    ap.add_argument("--giant-reps", type=int, default=4)
    ap.add_argument("--cpu-reps", type=int, default=2)
    ap.add_argument("--fresh", type=int, default=3, help="replicates also solved as fresh batches")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bootstrap_bench: no CUDA device (the measurement has no CPU fallback)")
    from strawberry_b200 import api, synth
    res = dict(gpu_before=gpu_info(), seed=SEED)
    res["headline"], batch = headline(args, api, synth)
    res["giant"] = giant(args, api)
    res["gpu_after"] = gpu_info()
    res["cpu"] = cpu(args, batch)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(headline=res["headline"]["summary"], giant=res["giant"]["replicates"], cpu=res["cpu"]["seconds"],
                          gpu=res["gpu_before"]), indent=1))


if __name__ == "__main__":
    main()
