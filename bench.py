#!/usr/bin/env python
"""bench.py - the reference's headline metric on B200: fragments*EM-iters/sec (and wall time to
converge) of the per-locus Latent-Class-Model EM on synthetic 10M-fragment, ~20k-locus human-shaped
batches (BASELINE.json configs[1]; generator strawberry_b200.synth.human_shaped, seeds 2, 3, ...).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the timed legs computed in their last step, as a caller of the path receives it, to
DIR/<name>.npy (float64; integer outputs converted exactly): theta / fpkm / frac / tpm / keep per isoform and iters /
status per locus of the headline, the same with a bias_ prefix plus bias_beta / bias_outer of the bias leg, and giant_*
of the giant leg (no TPM there: a wave's TPM uses a placeholder denominator). With N > 1 ranks every rank writes its own
loci as <name>.rank<r>.npy. The inputs are seeded, so two builds run with the same arguments can be compared file by file.

A step = one pass of the hot path (EM to convergence + FPKM/frac/filter epilogue + TPM denominator) over
the job. `value` is timed with the loci resident in HBM (CUDA events inside libsbq on the stream the
kernels run on); `e2e` is the same work through the public host-buffer calls from page-locked host
arrays, H2D and D2H inside the timed region.

N > 1 runs the path north_star describes: ONE job is partitioned over the N ranks by non-zeros (greedy
LPT, strawberry_b200.partition), every rank solves its own loci, and the only collective is the scalar
all-reduce of the TPM denominator (NCCL). Three legs, all through that partition:
  headline (weak scaling)  the job is N human-shaped batches pooled (seeds 2 .. N+1, 20000 N loci):
                           per-GPU work is fixed as N grows; value = fragment-iters of the whole job /
                           max-over-ranks time.
  strong                   ONE seed-2 batch (10 M fragments) split over N ranks, with a bitwise check of
                           every rank's theta / FPKM / frac against the unpartitioned solve.
  giant                    BASELINE configs[3]: 200 loci x 1 M single-fragment rows x ~48 non-zeros
                           (~115 GB of CSR), GENERATED ON THE DEVICE from the seed (sbq_synth_giant),
                           split over N ranks, solved in waves that fit HBM.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before CUDA is initialised: one hardware queue per concurrent launch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "fragments*EM-iters/sec"
UNIT = "fragment-iters/s"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons while the timed region runs."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])), mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def cpu_workload(batch):
    """The whole workload as the CPU sample (the dense reference finishes it in seconds)."""
    import oracle
    ora = oracle.quantify_batch(batch, batch["total_mapped_reads"], n_threads=os.cpu_count() or 1)
    frag_iters = int((np.add.reduceat(batch["count"].astype(np.int64), batch["loc_row_off"][:-1]) * ora["iters"]).sum())
    return oracle, frag_iters


def cpu_baseline_sample(batch):
    """CPU baseline, one thread, on the full 20k-locus workload: the reference's own EmSolver
    (oracle/_ref/libsbref.so, kind "reference") when it was built, else our C port (kind "port")."""
    oracle, frag_iters = cpu_workload(batch)
    if oracle.have_ref():
        secs, kind = oracle.ref_em_batch(batch, n_threads=1)["seconds"], "reference"
    else:
        secs, kind = oracle.quantify_batch(batch, batch["total_mapped_reads"], n_threads=1)["seconds"], "port"
    return dict(value=frag_iters / secs, unit=UNIT, cores=1, kind=kind,
                sample=f"the full workload, one pass: 20000 loci, {frag_iters} fragment-iters, {secs:.2f} s on one core "
                       f"({'reference EmSolver::init/run, dense Eigen' if kind == 'reference' else 'C port of the reference EM'})")


def reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the host cores (all of them)."""
    if rank != 0:
        return
    from strawberry_b200 import synth
    batch = synth.human_shaped(seed=2)
    oracle, frag_iters = cpu_workload(batch)
    cores = os.cpu_count() or 1
    use_ref = oracle.have_ref()
    kind = "reference" if use_ref else "port"

    def step():
        if use_ref:
            return oracle.ref_em_batch(batch, n_threads=cores)["seconds"]
        return oracle.quantify_batch(batch, batch["total_mapped_reads"], n_threads=cores)["seconds"]

    for _ in range(args.warmup):
        step()
    secs = [step() for _ in range(args.steps)]
    ms = 1e3 * float(np.mean(secs))
    value = frag_iters / (ms / 1e3)
    sample = (f"the full workload per step: 20000 loci, {frag_iters} fragment-iters; "
              f"{'reference EmSolver::init/run (dense Eigen, src/estimate.cpp:366-488), one std::thread per core pulling loci largest first (dense cost R x T)' if use_ref else 'C port of the reference EM, pthreads'}")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1]: synthetic 10M-fragment paired-end human-shaped loci (20000 loci), quantification only",
                       "generator": synth.GENERATOR_VERSION, "seed": 2, "l2": "n/a (CPU)"},
            "wall_ms_to_converge": ms,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


_REAL_STDOUT = None


def claim_stdout():
    """stdout must carry exactly one JSON line. Libraries write there behind Python's back (NCCL prints its version banner to
    fd 1 when NCCL_DEBUG is set), so fd 1 is pointed at stderr for the run and the line goes to the saved descriptor."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-giant", action="store_true", help="skip the giant-locus leg (BASELINE configs[3])")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling leg (N > 1)")
    ap.add_argument("--no-bias", action="store_true", help="skip the bias-in-EM leg (BASELINE configs[2]; our own definition, parity unpinned)")
    ap.add_argument("--giant-rows", type=int, default=1_000_000)
    ap.add_argument("--giant-loci", type=int, default=200)
    ap.add_argument("--giant-wave", type=int, default=25, help="giant loci resident at once per GPU (~0.7 GB each)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step of every leg as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from strawberry_b200 import api, partition, synth

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    gsum = torch.zeros(1, dtype=torch.float64, device=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(*vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    def reduce_sum(*vals):
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(x) for x in t]

    def tpm_exchange(q):
        """the path's only exchange step: sum of FPKM over all ranks (src/alignments.cpp:1821-1824)"""
        if world > 1:
            q.fpkm_sum_to_device(gsum.data_ptr())
            dist.all_reduce(gsum)
            q.finalize_tpm(float(gsum.item()))
        else:
            q.finalize_tpm(q.fpkm_sum())

    def timed_legs(q, pinned, total_reads, steps, warmup):
        """resident leg (per-step solve_ms from CUDA events inside libsbq) and end-to-end leg (host buffers, wall clock)."""
        def resident_step():
            flush.fill_(1)               # L2 flush between timed iterations (not timed: events live inside sbq_solve)
            torch.cuda.synchronize()
            q.solve(total_reads)
            tpm_exchange(q)
            return q.stats()["solve_ms"]

        def e2e_step():
            flush.fill_(1)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            q.clear()
            q.submit_flat(pinned)        # page-locked arrays are used in place
            q.upload_begin()             # copies enqueued in the order the solve needs them; launches wait for their own data only
            q.solve(total_reads)
            tpm_exchange(q)
            q.download()
            torch.cuda.synchronize()
            return time.perf_counter() - t0

        q.clear()
        q.submit_flat(pinned)
        q.upload()
        for _ in range(warmup):
            resident_step()
        barrier()
        t0 = time.perf_counter()
        step_ms = [resident_step() for _ in range(steps)]
        barrier()
        wall = time.perf_counter() - t0
        q.download()
        st, launches, res = q.stats(), q.launch_stats(), q.results()
        for _ in range(2):
            e2e_step()
        barrier()
        e2e_s = [e2e_step() for _ in range(steps)]
        barrier()
        return dict(ms=float(np.mean(step_ms)), e2e_s=float(np.mean(e2e_s)), wall=wall, st=st, st_e2e=q.stats(), launches=launches, res=res)

    # ---- the job: N human-shaped batches pooled, LPT-partitioned over the N ranks by non-zeros (weak scaling)
    seeds = list(range(2, 2 + world))
    job = synth.concat([synth.human_shaped(seed=s_) for s_ in seeds]) if world > 1 else synth.human_shaped(seed=2)
    total_reads = job["total_mapped_reads"]
    parts = partition.lpt_partition(partition.locus_cost(job), world)
    mine, _ = partition.take(job, parts[rank]) if world > 1 else (job, None)
    pinned = api.pinned_batch(mine)
    q = api.Quantifier(device=local_rank)

    clk = ClockSampler(local_rank)
    clk.__enter__()                      # sampled over the timed legs of the headline
    t_wall0 = time.perf_counter()
    hd = timed_legs(q, pinned, total_reads, args.steps, args.warmup)
    clk.__exit__(None, None, None)
    st, launches, res = hd["st"], hd["launches"], hd["res"]
    outputs = dict(res)                  # --dump-outputs: the headline's last resident step, then the other legs add theirs
    ms_per_step, e2e_per_step = reduce_max(hd["ms"], hd["e2e_s"])
    total_frag_iters, total_alg, total_launches = reduce_sum(st["frag_iters"], st["alg_bytes"], st["kernel_launches"])
    em_ms_max, = reduce_max(st["em_ms"])
    status_counts = reduce_sum(*[float(x) for x in np.bincount(res["status"], minlength=4)])

    # ---- roofline of the headline step. The EM kernels of a step (one warp-tier launch + one launch per cluster size) run
    # concurrently on separate streams, so the phase is timed as a whole with CUDA events on the context's main stream (em_ms)
    # and every launch also carries its own event pair on its own stream (launches[]). `kernel` names the launch with the most
    # algorithmic bytes on rank 0.
    peak, peak_src = load_peaks()
    dom = max(launches, key=lambda r: r["alg_bytes"])
    achieved = st["alg_bytes"] / (st["em_ms"] * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                "kernel": f"{dom['kernel']} (cluster_size={dom['cluster_size']}) + {len(launches) - 1} concurrent EM launches",
                "kernel_ms": st["em_ms"], "alg_bytes_per_launch": st["alg_bytes"], "peak_source": peak_src, "rank": 0,
                "note": "per GPU (rank 0). The CSR of the rank's loci is read from HBM once and then lives in shared memory (cluster tier) / L1 (warp tier) "
                        "for up to 1000 sequential EM iterations, so this step is bound by per-iteration latency of its longest loci, not by HBM "
                        "(DRAM traffic of the phase is a few tens of MB: traffic is not meaningful here); the HBM-bound kernel of this path is the "
                        "giant-locus one, see `giant.roofline`",
                "launches": [{k: r[k] for k in ("kernel", "cluster_size", "threads", "n_loci", "nnz", "start_ms", "ms", "alg_bytes", "max_iters")} for r in launches]}

    line = {"metric": METRIC, "value": total_frag_iters / (ms_per_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1]: synthetic 10M-fragment paired-end human-shaped loci (20000 loci), quantification only"
                                   + ("" if world == 1 else f"; {world} such batches (seeds {seeds[0]}..{seeds[-1]}) pooled into one job of {20000 * world} loci and "
                                                            f"LPT-partitioned by non-zeros over the {world} GPUs (one scalar NCCL all-reduce per step)"),
                       "generator": synth.GENERATOR_VERSION, "seeds": seeds, "loci_total": int(len(job["loc_row_off"]) - 1),
                       "fragments_total": int(job["count"].sum()), "nnz_total": int(job["row_ptr"][-1]),
                       "loci_rank0": st["n_loci"], "rows_rank0": st["n_row"], "isoforms_rank0": st["n_iso"], "nnz_rank0": st["nnz"],
                       "em_iters_total_rank0": st["em_iters_total"], "max_iter": 1000, "theta_tol": 1e-2,
                       "tiers_rank0": {"warp": st["loci_warp"], "cluster": st["loci_cta"], "grid": st["loci_grid"]},
                       "l2": "flushed between timed iterations (256 MiB fill)", "parallelism": f"loci partitioned x{world} (LPT by nnz)"},
            "wall_ms_to_converge": ms_per_step,
            "e2e": {"value": total_frag_iters / e2e_per_step, "unit": UNIT, "ms_per_step": e2e_per_step * 1e3,
                    "h2d_bytes_per_step": int(reduce_sum(hd["st_e2e"]["h2d_bytes"])[0]), "d2h_bytes_per_step": int(reduce_sum(hd["st_e2e"]["d2h_bytes"])[0]),
                    "stages_ms_rank0": {"upload": hd["st_e2e"]["upload_ms"], "solve": hd["st_e2e"]["solve_ms"], "download": hd["st_e2e"]["download_ms"]}},
            "gpu_launches": int(total_launches * args.steps),
            "timed_region_wall_s": hd["wall"],
            "roofline": roofline,
            "clocks": clk.summary(),
            "statuses": {k: int(v) for k, v in zip(("ok", "iter_cap", "zero_denom", "no_rows"), status_counts)}}

    # ---- strong scaling: ONE seed-2 batch split over the N ranks, bitwise check against the unpartitioned solve
    if world > 1 and not args.no_strong:
        try:
            one = job if world == 1 else synth.human_shaped(seed=2)
            q.clear()
            q.submit_flat(one)
            q.run(one["total_mapped_reads"])
            full = q.results()                                   # the 1-GPU answer, computed on every rank
            sparts = partition.lpt_partition(partition.locus_cost(one), world)
            sub, isos = partition.take(one, sparts[rank])
            sd = timed_legs(q, api.pinned_batch(sub), one["total_mapped_reads"], args.steps, args.warmup)
            r = sd["res"]
            bad = sum(int(not np.array_equal(r[k], full[k][isos], equal_nan=True)) for k in ("theta", "fpkm", "frac", "keep"))
            bad += int(not np.array_equal(r["iters"], full["iters"][sparts[rank]])) + int(not np.array_equal(r["status"], full["status"][sparts[rank]]))
            tpm_dev = float(np.nanmax(np.abs(r["tpm"] - full["tpm"][isos]) / np.maximum(np.abs(full["tpm"][isos]), 1e-300))) if len(isos) else 0.0
            s_ms, s_e2e, tpm_dev = reduce_max(sd["ms"], sd["e2e_s"], tpm_dev)
            s_fi, s_bad = reduce_sum(sd["st"]["frag_iters"], bad)
            nnz_rank = reduce_max(float(sd["st"]["nnz"]))[0]
            big = int(np.argmax(partition.locus_cost(one)))
            line["strong"] = {"scaling": "strong", "workload": "configs[1]: ONE seed-2 batch (20000 loci, 10M fragments) LPT-partitioned over the ranks",
                              "n_gpus": world, "value": s_fi / (s_ms * 1e-3), "unit": UNIT, "ms_per_step": s_ms,
                              "e2e_ms_per_step": s_e2e * 1e3, "e2e_value": s_fi / s_e2e,
                              "partition_invariance": {"arrays_differing_bitwise": int(s_bad), "checked": "theta, fpkm, frac, keep, iters, status of every rank's loci vs the 1-GPU solve",
                                                       "tpm_max_rel_dev": tpm_dev, "tpm_note": "TPM divides by a sum taken in a different order (NCCL all-reduce of per-rank sums)"},
                              "max_nnz_per_rank": int(nnz_rank),
                              "floor_note": f"a locus is never split across GPUs: the largest locus ({int(partition.locus_cost(one)[big])} cost units, "
                                            f"{int(full['iters'][big])} EM iterations) bounds the step from below"}
        except Exception as e:
            line["strong"] = {"error": repr(e)}

    # ---- bias-in-EM leg: BASELINE configs[2] (the same 10M batch with per-row covariates), LPT-partitioned over the ranks
    if not args.no_bias:
        try:
            line["bias"] = bias_leg(args, api, partition, synth, local_rank, rank, world, flush, reduce_max, reduce_sum, barrier, tpm_exchange, outputs)
        except Exception as e:
            line["bias"] = {"error": repr(e)}

    # ---- giant-locus leg: BASELINE configs[3], generated on the device, partitioned over the ranks, solved in waves
    if not args.no_giant:
        try:
            line["giant"] = giant_leg(args, api, partition, synth, local_rank, rank, world, flush, reduce_max, reduce_sum, barrier, dist, peak, peak_src, outputs)
        except Exception as e:   # the headline line must still be printed
            line["giant"] = {"error": repr(e)}
        if line.get("giant", {}).get("roofline_burst"):
            line["roofline_giant"] = line["giant"].pop("roofline_burst")      # the giant-locus kernel timed alone (burst); giant.roofline = over the whole 200-locus job

    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            fname = f"{name}.npy" if world == 1 else f"{name}.rank{rank}.npy"
            np.save(os.path.join(args.dump_outputs, fname), np.asarray(a, dtype=np.float64))

    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline_sample(job)
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# DRAM bytes per non-zero and EM pass of the giant-locus kernel, from `ncu --set full` captures of this kernel on this shape
# (dram__bytes_read.sum + dram__bytes_write.sum of one launch / (passes x non-zeros)); see profiles/ for the capture files.
GIANT_DRAM_BYTES_PER_NNZ_PASS = {"em_grid_dual_kernel": (10.854, "profiles/r02_grid_dual_ncu_summary.txt"),
                                 "em_grid_tma_kernel": (10.34, "profiles/r01_grid_tma_ncu_summary.txt")}


def bias_leg(args, api, partition, synth, local_rank, rank, world, flush, reduce_max, reduce_sum, barrier, tpm_exchange, outputs):
    """BASELINE configs[2]: the seed-2 10M-fragment batch with sequencing-bias correction inside the EM (bias_mode = 1), loci
    LPT-partitioned over the ranks. THE REFERENCE HAS NO BIAS IMPLEMENTATION (src/bias.cpp is commented out): the mode is our
    own definition (DESIGN.md section 7) and its only oracle is our CPU restatement - PARITY UNPINNED; no speed-up is quoted."""
    import torch
    one = synth.human_shaped(seed=2)
    X = synth.covariates(one, seed=3)
    parts = partition.lpt_partition(partition.locus_cost(one), world)
    sub, _ = partition.take(one, parts[rank])
    lro = np.asarray(one["loc_row_off"])
    rows = np.concatenate([np.arange(lro[l], lro[l + 1]) for l in parts[rank]]) if len(parts[rank]) else np.zeros(0, np.int64)
    qb = api.Quantifier(device=local_rank, bias_mode=1)
    qb.submit_flat(sub)
    qb.set_covariates(X[rows])
    qb.upload()
    ms = []
    n_solves = args.warmup + args.steps
    for i in range(n_solves):
        flush.fill_(1)
        torch.cuda.synchronize()
        qb.solve(one["total_mapped_reads"])
        tpm_exchange(qb)
        if i >= args.warmup:
            ms.append(qb.stats()["solve_ms"])
    qb.download()
    st, res = qb.stats(), qb.results()
    beta, outer = qb.bias_results()
    outputs.update({"bias_" + k: v for k, v in res.items()}, bias_beta=beta, bias_outer=outer)
    frag = np.add.reduceat(np.asarray(sub["count"], np.int64), np.asarray(sub["loc_row_off"])[:-1]) if len(parts[rank]) else np.zeros(0, np.int64)
    fi_local = float((frag * res["iters"]).sum())
    qb.close()
    barrier()
    ms_max, = reduce_max(float(np.mean(ms)))
    fi, it_all, outer_all, launches = reduce_sum(fi_local, float(res["iters"].sum()), float(outer.sum()), float(st["kernel_launches"]))
    out = {"scaling": "strong", "n_gpus": world, "parity": "UNPINNED: the reference has no bias-in-EM implementation (src/bias.cpp is commented out); "
                                                           "bias_mode = 1 is our own definition, checked against our CPU restatement only",
           "workload": "configs[2]: the seed-2 batch (20000 loci, 10M fragments) with 5 per-row covariates (gc, gc^2, gc^3, log bin length, mean fragment length; seed 3), "
                       f"bias-corrected EM, LPT over {world} GPU(s)",
           "value": fi / (ms_max * 1e-3), "unit": UNIT, "ms_per_step": ms_max, "theta_iters_total": int(it_all), "outer_rounds_total": int(outer_all),
           "kernel": "em_bias_warp_kernel (small loci: one warp per locus, persistent warps) + em_bias_kernel (one cluster of 1 / 2 / 4 / 8 / 16 CTAs per locus by non-zeros, rows streamed from L2, partial sums exchanged through distributed shared memory)",
           "gpu_launches": int(launches * n_solves)}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import oracle
        rng = np.random.default_rng(7)
        pick = rng.choice(len(frag), 1500, replace=False)
        t0 = time.perf_counter()
        fi_cpu = 0
        for l in pick:
            T, rpl, col, al, cnt, il = synth.locus_slice(one, int(l))
            _, _, _, iters, _ = oracle.em_bias_csr(T, rpl, col, al, cnt, X[lro[l]:lro[l + 1]])
            fi_cpu += int(cnt.sum()) * int(iters)
        secs = time.perf_counter() - t0
        out["cpu_restatement"] = {"value": fi_cpu / secs, "unit": UNIT, "cores": 1, "kind": "port (our own restatement; no reference exists for this mode)",
                                  "sample": f"1500 of the 20000 loci (random, seed 7), {fi_cpu} fragment-iters in {secs:.2f} s on one core"}
    return out


def giant_leg(args, api, partition, synth, local_rank, rank, world, flush, reduce_max, reduce_sum, barrier, dist, peak, peak_src, outputs):
    """BASELINE configs[3]: `giant_loci` loci of `giant_rows` single-fragment rows, k ~ 1 + Poisson(47) isoforms per row,
    T ~ U{500..800}, generated ON THE DEVICE from seed 4 (sbq_synth_giant: a locus is a pure function of (seed, global id), so
    the partition does not change the data). Loci are dealt to the ranks by LPT (equal expected cost: round robin) and solved
    in waves of `giant_wave` resident loci. One pass over all loci = one step, `steps` of them timed (times reported per step);
    EM time from CUDA events inside libsbq."""
    import torch
    n, rows, seed = args.giant_loci, args.giant_rows, 4
    owner = partition.lpt_partition(np.full(n, rows * 48, np.int64), world)
    my_ids = [int(x) for x in owner[rank]]
    qg = api.Quantifier(device=local_rank)
    waves = [my_ids[i:i + args.giant_wave] for i in range(0, len(my_ids), args.giant_wave)]
    # warm-up: a small wave through the same kernels (module load, first allocations)
    qg.synth_giant(my_ids[:1] or [0], min(rows, 100_000), seed=seed)
    qg.solve(rows)
    barrier()
    # ---- burst measurement for the roofline of the giant-locus kernel: two loci, kernel timed alone (1 warm-up + 2 timed solves)
    burst = None
    if my_ids:
        bid = my_ids[:2]
        qg.clear()
        qg.synth_giant(bid, rows, seed=seed)
        b_ms = []
        for i in range(3):
            flush.fill_(1)
            torch.cuda.synchronize()
            qg.solve(rows * n)
            if i:
                b_ms.append(qg.stats()["grid_em_ms"])
        qg.finalize_tpm(1.0)
        qg.download()
        bst = qg.stats()
        burst = dict(ms=float(np.mean(b_ms)), alg=bst["grid_alg_bytes"], nnz=bst["nnz"], iters=bst["em_iters_total"], n=len(bid), frag_iters=bst["frag_iters"],
                     kernel=next((r["kernel"] for r in qg.launch_stats() if r["kernel"].startswith("em_grid")), "em_grid_kernel"))
    barrier()
    em_ms = solve_ms = gen_ms = 0.0                                  # summed over the steps
    kernel = "em_grid_kernel"
    wave_ms_per_pass = []
    # untimed warm-up at FULL wave size: the first full-size solve allocates the layout buffers of the grid tier (packed chunk stream,
    # row records, 16-bit slots: ~ 12 GB for 25 loci) between the timing events - seen to cost up to 1 s on a fresh box
    if waves:
        qg.clear()
        qg.synth_giant(waves[0], rows, seed=seed)
        qg.solve(rows * n)
        barrier()
    clk = ClockSampler(local_rank)
    clk.__enter__()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        frag_iters = alg = iters = nnz = launches = 0                # one pass: every step does the same work
        fpkm_local = 0.0
        step_res = []
        for ids in waves:
            qg.clear()
            qg.synth_giant(ids, rows, seed=seed)
            flush.fill_(1)
            torch.cuda.synchronize()
            qg.solve(rows * n)                       # total_mapped_reads of the whole 200-locus job
            fpkm_local += qg.fpkm_sum()
            qg.finalize_tpm(1.0)                     # placeholder denominator: TPM of a wave needs the all-reduced sum of ALL waves
            qg.download()
            st = qg.stats()
            em_ms += st["grid_em_ms"]
            wave_ms_per_pass.append(round(st["grid_em_ms"] / max(st["em_iters_total"] + len(ids), 1), 5))
            solve_ms += st["solve_ms"]
            gen_ms += st["upload_ms"]
            frag_iters += st["frag_iters"]
            alg += st["grid_alg_bytes"]
            iters += st["em_iters_total"]
            nnz += st["nnz"]
            launches += st["kernel_launches"]
            kernel = next((r["kernel"] for r in qg.launch_stats() if r["kernel"].startswith("em_grid")), kernel)
            if args.dump_outputs:
                step_res.append(qg.results())
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / args.steps
    em_ms, solve_ms, gen_ms = em_ms / args.steps, solve_ms / args.steps, gen_ms / args.steps
    clk.__exit__(None, None, None)
    if step_res:
        outputs.update({"giant_" + k: np.concatenate([r[k] for r in step_res]) for k in ("theta", "fpkm", "frac", "keep", "iters", "status")})
    barrier()
    # the exchange step of this leg: the TPM denominator over all ranks and waves
    g = torch.tensor([fpkm_local], dtype=torch.float64, device=torch.device("cuda", local_rank))
    if world > 1:
        dist.all_reduce(g)
    qg.close()
    em_max, solve_max, wall_max, gen_max = reduce_max(em_ms, solve_ms, wall, gen_ms)
    fi, alg_all, it_all, nnz_all, launch_all = reduce_sum(frag_iters, alg, iters, nnz, launches)
    ach = alg / (em_ms * 1e-3) / 1e9 if em_ms > 0 else 0.0          # this rank's kernel over the whole job: algorithmic bytes / its own EM time
    bpn, src = GIANT_DRAM_BYTES_PER_NNZ_PASS.get(kernel, (None, None))
    passes = iters + len(my_ids)                                     # EM passes + one setup pass per locus
    traffic = bpn * (nnz / max(len(my_ids), 1)) * passes if bpn else None
    roof_burst = None
    if burst:
        b_ach = burst["alg"] / (burst["ms"] * 1e-3) / 1e9
        b_bpn, b_src = GIANT_DRAM_BYTES_PER_NNZ_PASS.get(burst["kernel"], (None, None))
        roof_burst = {"bound": "hbm", "achieved": b_ach, "peak": peak, "unit": "GB/s", "frac": b_ach / peak,
                      "traffic": b_bpn * (burst["nnz"] / burst["n"]) * (burst["iters"] + burst["n"]) if b_bpn else None,
                      "traffic_source": f"{b_bpn} DRAM bytes per non-zero and pass: dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel on this shape under "
                                        f"ncu --set full ({b_src}), x non-zeros per locus x passes of this launch" if b_bpn else None,
                      "real_bytes_frac": (b_bpn / 12.0) * b_ach / peak if b_bpn else None,
                      "kernel": burst["kernel"], "kernel_ms": burst["ms"], "alg_bytes_per_launch": burst["alg"], "peak_source": peak_src + " (burst copy figure)", "rank": rank,
                      "workload": f"configs[3] shape, kernel timed alone: {burst['n']} device-generated loci x {rows} rows ({burst['nnz']} nnz, {burst['iters']} EM iterations); "
                                  f"CSR {burst['nnz'] * 12 / 1e9:.2f} GB > L2; each launch includes its one-off layout pass only on the first solve (not timed)",
                      "value": burst["frag_iters"] / (burst["ms"] * 1e-3), "unit_value": UNIT}
    return {"scaling": "strong", "n_gpus": world, "roofline_burst": roof_burst, "wave_ms_per_pass": wave_ms_per_pass, "clocks": clk.summary(),
            "workload": f"configs[3]: {n} loci x {rows} single-fragment rows, k~1+Poisson(47) isoforms per row, T~U{{500..800}}, seed {seed}, generated on the device "
                        f"({synth.DEVICE_GENERATOR_VERSION}); {int(nnz_all)} non-zeros = {nnz_all * 12 / 1e9:.1f} GB of CSR in total; LPT over {world} GPU(s), waves of <= {args.giant_wave} loci",
            "value": fi / (solve_max * 1e-3), "unit": UNIT, "ms_per_step": solve_max, "em_ms_per_step": em_max, "generate_ms": gen_max,
            "wall_ms_incl_generation": wall_max * 1e3, "em_iters_total": int(it_all), "loci_per_rank": len(my_ids), "gpu_launches": int(launch_all),
            "fpkm_sum_allreduced": float(g.item()),
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                         "traffic_source": f"{bpn} DRAM bytes per non-zero and pass (ncu --set full of this kernel on this shape, {src}) x this rank's non-zeros per locus x passes"
                                           if bpn else None,
                         "real_bytes_frac": (bpn / 12.0) * ach / peak if bpn else None,
                         "kernel": kernel, "kernel_ms": em_ms, "alg_bytes_per_launch": alg, "peak_source": peak_src, "rank": rank,
                         "note": "SUSTAINED figure: kernel_ms sums the giant-locus launches of this rank's waves over the whole job (each includes its one-off layout pass; "
                                 "seconds of back-to-back streaming, see `clocks` of this leg), against the burst copy peak; "
                                 "achieved counts the SURVEY 8d algorithmic bytes (12 B per non-zero); real_bytes_frac rescales to the DRAM bytes ncu measured "
                                 "(u16 slots instead of 4-byte columns)"}}


if __name__ == "__main__":
    main()
