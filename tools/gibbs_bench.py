"""Gibbs posterior samples on the GPU (sbq_gibbs): device time per round and per sample on the headline batch and on a wave of
giant loci, with bootstrap replicates of the same resident batches timed alternately in the same run.

  python tools/gibbs_bench.py --out profiles/r03_gibbs.json

  headline  configs[1] (synth.human_shaped(), seed 2: 20 000 loci, 10 M fragments): --rounds alternations of one sbq_bootstrap call
            of --boot-reps replicates and one sbq_gibbs call of --samples samples at thin --thin, burn-in --burn-in.
  giant     one wave of --giant-loci device-generated loci of the configs[3] shape (1 M single-fragment rows, 500-800 isoforms,
            ~48 entries per row; sbq_synth_giant): --giant-rounds alternations of --giant-boot-reps replicates and
            --giant-samples samples.
Per Gibbs call: ms per round (assign + theta), ms per sample (the rounds it costs: thin), and the one-off setup (colsum_ms).
The card's name, power limit and clocks are read in the same run. The tool refuses to run without a GPU."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SEED = 20261022


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True, check=True).stdout
    return [dict(zip(q.split(","), (x.strip() for x in line.split(",")))) for line in out.strip().splitlines()]


def _stats(vals):
    a = np.asarray(vals, np.float64)
    return dict(median=float(np.median(a)), min=float(a.min()), max=float(a.max()))


def alternate(q, n_alt, boot_reps, samples, thin, burn_in):
    q.bootstrap(SEED + 1, 1)                                  # warm-up: every kernel and allocation of the timed calls
    q.gibbs(SEED + 1, 1, thin=1, burn_in=0)
    boots, gibbs = [], []
    for i in range(n_alt):
        q.bootstrap(SEED, boot_reps, i * boot_reps)
        b = q.bootstrap_stats()
        boots.append(dict(n=b["n"], ms_per_rep=b["total_ms"] / b["n"], em_ms_per_rep=b["em_ms"] / b["n"],
                          resample_ms_per_rep=b["resample_ms"] / b["n"]))
        q.gibbs(SEED + i, samples, thin=thin, burn_in=burn_in)
        g = q.gibbs_stats()
        r = g["rounds"]
        gibbs.append(dict(g, assign_ms_per_round=g["assign_ms"] / r, theta_ms_per_round=g["theta_ms"] / r,
                          ms_per_round=(g["assign_ms"] + g["theta_ms"]) / r, ms_per_sample=(g["assign_ms"] + g["theta_ms"]) / r * thin))
    summary = dict(bootstrap_ms_per_replicate=_stats([b["ms_per_rep"] for b in boots]),
                   gibbs_ms_per_round=_stats([g["ms_per_round"] for g in gibbs]),
                   gibbs_assign_ms_per_round=_stats([g["assign_ms_per_round"] for g in gibbs]),
                   gibbs_theta_ms_per_round=_stats([g["theta_ms_per_round"] for g in gibbs]),
                   gibbs_ms_per_sample_at_thin=_stats([g["ms_per_sample"] for g in gibbs]),
                   gibbs_colsum_ms=_stats([g["colsum_ms"] for g in gibbs]), thin=thin)
    return dict(bootstrap_calls=boots, gibbs_calls=gibbs, summary=summary)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--boot-reps", type=int, default=25)
    ap.add_argument("--samples", type=int, default=25)
    ap.add_argument("--thin", type=int, default=16)
    ap.add_argument("--burn-in", type=int, default=16)
    ap.add_argument("--giant-loci", type=int, default=25)
    ap.add_argument("--giant-rounds", type=int, default=2)
    ap.add_argument("--giant-boot-reps", type=int, default=1)
    ap.add_argument("--giant-samples", type=int, default=4)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("gibbs_bench: no CUDA device (the measurement has no CPU fallback)")
    from strawberry_b200 import api, synth
    res = dict(gpu_before=gpu_info(), seed=SEED)
    b = synth.human_shaped(seed=2)
    q = api.Quantifier()
    q.submit_flat(api.pinned_batch(b))
    q.run(b["total_mapped_reads"])
    st = q.stats()
    res["headline"] = dict(batch=dict(n_loci=int(st["n_loci"]), n_row=int(st["n_row"]), nnz=int(st["nnz"]), fragments=int(b["count"].sum())),
                           **alternate(q, args.rounds, args.boot_reps, args.samples, args.thin, args.burn_in))
    q.close()
    rows = 1_000_000
    q = api.Quantifier()
    q.synth_giant(list(range(args.giant_loci)), rows)
    q.solve(rows * args.giant_loci)
    q.download()
    st = q.stats()
    res["giant"] = dict(loci=args.giant_loci, rows_per_locus=rows, nnz=int(st["nnz"]), point_em_ms=st["em_ms"],
                        **alternate(q, args.giant_rounds, args.giant_boot_reps, args.giant_samples, args.thin, args.burn_in))
    q.close()
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(dict(headline=res["headline"]["summary"], giant=res["giant"]["summary"], gpu=res["gpu_before"]), indent=1))


if __name__ == "__main__":
    main()
