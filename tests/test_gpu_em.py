"""GPU parity: the CUDA path (through the C ABI in include/sbq.h) against the CPU oracle on the same
seeded inputs, against the reference's golden vectors, and - at full BASELINE size - through
size-independent properties."""
import numpy as np
import pytest

import cluster_paths
from strawberry_b200 import synth
from util import assert_matches_oracle, load_golden, theta_close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def q(sbq_lib_path):
    from strawberry_b200 import api
    qq = api.Quantifier()
    yield qq
    qq.close()


def run_gpu(q, batch, tier=0, cluster=0, **cfg):
    from strawberry_b200 import api
    qq = q if not cfg else api.Quantifier(**cfg)
    qq.clear()
    qq.set_plan(tier, cluster)
    qq.submit_flat(batch)
    qq.validate()
    qq.run(batch["total_mapped_reads"])
    res = qq.results()
    res["stats"] = qq.stats()
    if cfg:
        qq.close()
    return res


def test_golden_vectors_from_the_reference(q, oracle_mod):
    """theta against what the UNMODIFIED reference EmSolver returned (tests/golden/em_golden.npz)."""
    b, theta_ref, rc_ref, iters, status = load_golden()
    res = run_gpu(q, b)
    assert np.array_equal(res["status"], status)
    assert np.array_equal(res["iters"], iters)
    ok, worst = theta_close(res["theta"], theta_ref, b)
    assert ok.all(), worst


@pytest.fixture(scope="module")
def golden_capped():
    """The golden batch after 1, 2 and 5 EM steps, restated in long double (tests/cluster_paths.py)."""
    b, *_ = load_golden()
    return {m: cluster_paths.batch_em_longdouble(b, max_iter=m) for m in (1, 2, 5)}


@pytest.mark.parametrize("tier,cluster", [(0, 0), (1, 0), (2, 1), (2, 2), (2, 4), (2, 8), (2, 16), (3, 0)])
def test_every_tier_matches_the_oracle(q, oracle_mod, golden_capped, tier, cluster):
    """Converged, against the oracle at the parity bar; and capped at 1, 2 and 5 EM steps, against the long-double restatement at
    cluster_paths.CAPPED_REL (a bar the converged check is far too loose to replace: see tests/test_gpu_cluster_paths.py)."""
    b, *_ = load_golden()
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"])
    res = run_gpu(q, b, tier, cluster)
    assert_matches_oracle(res, ora, b, f"tier {tier} cluster {cluster}")
    st = res["stats"]
    if tier == 3:
        assert st["loci_grid"] > 0
    if tier == 2:
        assert st["loci_cta"] > 0
    for m, ld in golden_capped.items():
        capped = run_gpu(None, b, tier, cluster, max_iter=m)
        assert np.array_equal(capped["status"], ld["status"]) and np.array_equal(capped["iters"], ld["iters"]), m
        ok, worst = cluster_paths.theta_close_ld(capped["theta"], ld["theta"], b, cluster_paths.CAPPED_REL)
        print(f"capped worst ratio: golden tier {tier} cluster {cluster} max_iter {m}: {worst:.3e}")
        assert ok.all(), (m, worst)


def test_human_shaped_sample_matches_oracle(q, oracle_mod):
    b = synth.human_shaped(n_loci=2500, total_fragments=1_200_000, seed=31)
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=8)
    res = run_gpu(q, b)
    worst = assert_matches_oracle(res, ora, b, "human-shaped 2500 loci")
    assert worst < 1e-6
    assert res["stats"]["loci_warp"] > 0 and res["stats"]["loci_cta"] > 0
    assert res["stats"]["frag_iters"] == int((np.add.reduceat(b["count"], b["loc_row_off"][:-1]).astype(np.int64) * ora["iters"]).sum())


def test_filter_and_effective_length_epilogue(oracle_mod):
    b = synth.human_shaped(n_loci=600, total_fragments=300_000, seed=41, max_rows=300)
    b["iso_len"] = b["iso_len"].copy()
    b["iso_len"][::17] = 150           # shorter than the insert mean -> "NA" branch (src/estimate.cpp:320-323)
    kw = dict(min_iso_frac=0.01, effective_len_norm=1, insert_mean=200.0)
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], min_iso_frac=0.01, effective_len_norm=True, insert_mean=200.0)
    res = run_gpu(None, b, **kw)
    assert_matches_oracle(res, ora, b, "epilogue")
    assert (res["keep"] == 0).any() and (res["keep"] == 1).any()


def test_giant_locus_grid_tier_matches_oracle(q, oracle_mod):
    b = synth.giant(n_loci=2, rows_per_locus=60_000, seed=4)
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=2)
    res = run_gpu(q, b)
    assert res["stats"]["loci_grid"] == 2
    assert_matches_oracle(res, ora, b, "giant grid tier")
    # same loci through the cluster tier must give the same answer within the bar
    res2 = run_gpu(q, b, 2, 16)
    assert_matches_oracle(res2, ora, b, "giant through clusters")


def test_submit_aos_equals_submit_flat(q):
    b, *_ = load_golden()
    flat = run_gpu(q, b)
    q.clear()
    L = len(b["loc_row_off"]) - 1
    q.submit([synth.locus_slice(b, l) for l in range(L)])
    q.run(b["total_mapped_reads"])
    aos = q.results()
    for k in ("theta", "fpkm", "frac", "tpm", "keep", "iters", "status"):
        assert np.array_equal(flat[k], aos[k], equal_nan=True), k


def test_solve_is_rerunnable_and_bit_reproducible(q):
    b = synth.human_shaped(n_loci=1500, total_fragments=700_000, seed=51)
    first = run_gpu(q, b)
    q.solve(b["total_mapped_reads"])
    q.finalize_tpm(q.fpkm_sum())
    q.download()
    again = q.results()
    for k in ("theta", "fpkm", "frac", "tpm", "keep", "iters", "status"):
        assert np.array_equal(first[k], again[k], equal_nan=True), k


def test_em_solver_mirror_keeps_reference_semantics(q, oracle_mod):
    from strawberry_b200 import api
    rng = np.random.default_rng(3)
    model = rng.random((40, 6)) * (rng.random((40, 6)) < 0.4) * 0.01
    count = rng.integers(0, 50, 40)
    em = api.EmSolver(q)
    assert em.init(6, count, model) is True and em.run() is True       # src/estimate.cpp:366-488
    st, th, it = oracle_mod.em_dense(count, model)
    assert st == 0 and em.iters == it
    assert np.allclose(em._theta, th, rtol=1e-9, atol=0)
    em2 = api.EmSolver(q)
    assert em2.init(2, [3, 4], np.full((2, 2), 5e-6)) is False and em2.run() is False   # init() false: no row > 1e-5
    assert em2._theta == [3.5, 3.5]


def test_full_size_config2_matches_oracle(q, oracle_mod):
    """BASELINE configs[1] at FULL size - the exact batch bench.py times (seed 2, 20 000 loci, 10 M fragments,
    4.82 M non-zeros) - against the CPU oracle: equal status and iteration count for every locus,
    theta / FPKM / frac / TPM within 1e-6 relative, equal keep flags. The oracle needs well under a second."""
    b = synth.human_shaped(seed=2)
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=8)
    res = run_gpu(q, b)
    assert res["stats"]["n_loci"] == 20000 and res["stats"]["nnz"] == int(b["row_ptr"][-1])
    worst = assert_matches_oracle(res, ora, b, "configs[1] full size")
    assert worst < 1e-6
    frag = np.add.reduceat(b["count"].astype(np.int64), b["loc_row_off"][:-1])
    assert res["stats"]["frag_iters"] == int((frag * ora["iters"]).sum())
    assert res["stats"]["em_iters_total"] == int(ora["iters"].sum())


def test_config5_shape_matches_oracle(oracle_mod):
    """BASELINE configs[4] shape (SURVEY 8d row 5): the human-shaped generator with 60 000 loci and 100 M fragments,
    min_iso_frac = 0.01 (the assembly-mode default, so the low-fraction erase path runs) against the oracle: status,
    iteration count, theta / FPKM / frac / TPM within 1e-6, keep flags equal."""
    b = synth.human_shaped(n_loci=60000, total_fragments=100_000_000, seed=5)
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=8, min_iso_frac=0.01)
    res = run_gpu(None, b, min_iso_frac=0.01)
    assert res["stats"]["n_loci"] == 60000 and int(b["count"].sum()) == 100_000_000
    worst = assert_matches_oracle(res, ora, b, "configs[4] shape")
    assert worst < 1e-6
    assert (res["keep"] == 0).any()


def test_full_size_config2_properties(q):
    """BASELINE configs[1] at full size: 20k loci / 10M fragments. Oracle-free, size-independent checks."""
    b = synth.human_shaped()
    res = run_gpu(q, b)
    assert res["stats"]["n_loci"] == 20000 and int(b["count"].sum()) == 10_000_000
    lio = b["loc_iso_off"]
    theta_sum = np.add.reduceat(res["theta"], lio[:-1])
    # mass conservation for converged loci that advanced at least once
    kept_row = np.maximum.reduceat((b["alpha"] > 1e-5).astype(np.int8), b["row_ptr"][:-1]) > 0
    kept_cnt = np.add.reduceat(np.where(kept_row, b["count"], 0).astype(np.int64), b["loc_row_off"][:-1])
    sel = (res["status"] == 0) & (res["iters"] > 1)
    assert sel.sum() > 10000
    rel = np.abs(theta_sum[sel] - kept_cnt[sel]) / np.maximum(kept_cnt[sel], 1)
    assert rel.max() < 1e-9, rel.max()
    # zero-denominator loci keep the uniform initial value total / T
    tot = np.add.reduceat(b["count"].astype(np.int64), b["loc_row_off"][:-1])
    for l in np.nonzero(res["status"] == 2)[0][:50]:
        T = lio[l + 1] - lio[l]
        assert np.array_equal(res["theta"][lio[l]:lio[l + 1]], np.full(T, tot[l] / T))
    # per-locus fractions sum to one, TPM sums to 1e6 over the survivors
    live = np.repeat(res["status"] != 3, np.diff(lio))
    fsum = np.add.reduceat(np.where(live, res["frac"], 0.0), lio[:-1])
    ok = (res["status"] != 3) & np.isfinite(fsum)
    assert np.abs(fsum[ok] - 1.0).max() < 1e-9
    assert abs(np.nansum(res["tpm"][res["keep"] != 0]) - 1e6) < 1e-3
    # idempotence: a second solve of the resident batch is bit-identical
    q.solve(b["total_mapped_reads"])
    q.finalize_tpm(q.fpkm_sum())
    q.download()
    again = q.results()
    assert np.array_equal(res["theta"], again["theta"]) and np.array_equal(res["iters"], again["iters"])


def test_full_size_giant_locus_properties(q):
    """BASELINE configs[3] shape at full per-locus size (1 M rows x ~48 non-zeros, T ~ U{500..800}; CSR 0.58 GB > L2)
    through the TMA grid kernel: oracle-free properties, plus agreement with the cluster-tier streaming path."""
    b = synth.giant(n_loci=1, rows_per_locus=1_000_000, seed=4)
    qq = q
    qq.clear()
    qq.set_plan(0, 0)
    qq.submit_flat(b)
    qq.run(b["total_mapped_reads"])
    res = qq.results()
    st = qq.stats()
    assert st["loci_grid"] == 1 and res["status"][0] == 0 and 1 < res["iters"][0] < 1000
    # every row is kept (alpha > 1e-5) so the EM conserves the full mass
    assert abs(res["theta"].sum() - 1_000_000) < 1e-6 * 1_000_000
    assert abs(res["frac"].sum() - 1.0) < 1e-9 and abs(res["tpm"].sum() - 1e6) < 1e-3
    # bit-reproducible: the resident batch solved again gives identical bits (fixed-shape reductions, no atomics)
    qq.solve(b["total_mapped_reads"])
    qq.finalize_tpm(qq.fpkm_sum())
    qq.download()
    again = qq.results()
    assert np.array_equal(res["theta"], again["theta"]) and again["iters"][0] == res["iters"][0]
    # fixed point: theta is the previous iterate of a converged run, so one more EM step moves it by < tol
    T = int(b["loc_iso_off"][1])
    rows = np.repeat(np.arange(1_000_000), np.diff(b["row_ptr"]))
    s = np.bincount(b["col"], weights=b["alpha"], minlength=T)
    th = res["theta"] / s
    d = np.bincount(rows, weights=b["alpha"] * th[b["col"]], minlength=1_000_000)
    nxt = np.bincount(b["col"], weights=b["alpha"] * th[b["col"]] / d[rows], minlength=T)
    assert np.linalg.norm(nxt - res["theta"]) < 1e-2


def test_config5_shape_with_low_fraction_filter(oracle_mod):
    """BASELINE configs[4] shape: 60 k loci, 1e8 fragments, assembly-mode default min_iso_frac = 0.01."""
    b = synth.human_shaped(n_loci=60_000, total_fragments=100_000_000, seed=5)
    res = run_gpu(None, b, min_iso_frac=0.01)
    assert res["stats"]["n_loci"] == 60_000 and int(b["count"].sum()) == 100_000_000
    kept = res["keep"] != 0
    assert (~kept).any() and (res["frac"][kept] >= 0.01).all()
    live = np.repeat(res["status"] != 3, np.diff(b["loc_iso_off"]))
    assert (res["frac"][~kept & live & np.isfinite(res["frac"])] < 0.01).all()
    assert abs(np.nansum(res["tpm"][kept]) - 1e6) < 1e-3
    # spot-check 300 loci against the oracle
    idx = np.arange(0, 60_000, 200)
    from strawberry_b200 import partition
    sub, isos = partition.take(b, idx)
    ora = oracle_mod.quantify_batch(sub, b["total_mapped_reads"], min_iso_frac=0.01)
    assert np.array_equal(res["iters"][idx], ora["iters"]) and np.array_equal(res["status"][idx], ora["status"])
    scale = np.maximum(np.abs(ora["theta"]), 1e-9 * np.repeat(np.add.reduceat(sub["count"].astype(np.float64), sub["loc_row_off"][:-1]), np.diff(sub["loc_iso_off"])))
    assert (np.abs(res["theta"][isos] - ora["theta"]) / np.maximum(scale, 1e-300)).max() < 1e-6
    assert np.array_equal(res["keep"][isos] != 0, ora["keep"] != 0)


def test_grid_tier_dense_rows_take_the_oversize_chunk_path(q, oracle_mod):
    """Rows of ~600 non-zeros: every 32-row chunk exceeds the TMA stage capacity, so the grid kernel's consumers read
    those chunks straight from global memory while the ring is bypassed."""
    rng = np.random.default_rng(8)
    T, R = 900, 2200
    rows, rp = [], [0]
    for i in range(R):
        k = int(rng.integers(450, 750))
        rows.append(np.sort(rng.choice(T, k, replace=False)))
        rp.append(rp[-1] + k)
    col = np.concatenate(rows).astype(np.int32)
    b = dict(loc_row_off=np.array([0, R], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=np.array(rp, np.int64), col=col,
             alpha=10.0 ** rng.uniform(-4, -1.5, len(col)), count=rng.integers(0, 50, R).astype(np.int32),
             iso_len=rng.integers(400, 8000, T).astype(np.int32), total_mapped_reads=1_000_000)
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], max_iter=60)
    from strawberry_b200 import api
    qq = api.Quantifier(max_iter=60)
    qq.submit_flat(b)
    qq.run(b["total_mapped_reads"])
    res = qq.results()
    assert qq.stats()["loci_grid"] == 1
    assert_matches_oracle(res, ora, b, "dense-row giant locus")
    qq.close()


def test_golden_vectors_through_the_two_slot_grid_kernel(q, monkeypatch):
    """The reference's golden vectors (all four locus outcomes) through the grid tier: 135 of the 136 loci qualify for the
    two-slot kernel, the one whose rows average more than 56 non-zeros runs on the TMA ring kernel in the same solve."""
    b, theta_ref, rc_ref, iters, status = load_golden()
    monkeypatch.setenv("SBQ_DUAL_VERIFY", "1")
    res = run_gpu(q, b, 3, 0)
    assert res["stats"]["loci_grid"] == len(status)
    assert any(r["kernel"] == "em_grid_dual_kernel" for r in q.launch_stats())
    assert np.array_equal(res["status"], status) and np.array_equal(res["iters"], iters)
    ok, worst = theta_close(res["theta"], theta_ref, b)
    assert ok.all(), worst


def _two_slot_edge_locus(R, T, seed):
    """A giant-tier locus for the two-slot layout (sbq_grid_dual.cuh): Poisson(40) rows plus empty rows, rows dropped by
    the row filter, rows too long for the sorted layout (walked from global memory), a run of 90-entry rows and a run of
    60-entry rows (chunks fuller than a ring stage), zero counts."""
    rng = np.random.default_rng(seed)
    k = 1 + rng.poisson(40.0, R)
    k[rng.random(R) < 0.01] = 0
    long_rows = rng.choice(R, max(2, R // 400), replace=False)
    k[long_rows] = rng.integers(150, 400, long_rows.size)
    burst = min(R - 50, R // 2)
    k[burst:burst + 24] = 90
    k[burst + 24:burst + 48] = 60
    k = np.minimum(k, T)
    row_ptr = np.zeros(R + 1, np.int64)
    np.cumsum(k, out=row_ptr[1:])
    col = np.concatenate([np.sort(rng.choice(T, kk, replace=False)) for kk in k]).astype(np.int32)
    alpha = 10.0 ** rng.uniform(-4.0, -1.5, int(row_ptr[-1]))
    for i in rng.choice(R, max(1, R // 100), replace=False):
        alpha[row_ptr[i]:row_ptr[i + 1]] = 5e-6
    count = rng.integers(0, 4, R).astype(np.int32)
    return dict(loc_row_off=np.array([0, R], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=row_ptr, col=col, alpha=alpha,
                count=count, iso_len=rng.integers(400, 8001, T).astype(np.int32), total_mapped_reads=int(count.sum()), meta={})


def test_grid_tier_two_slot_layout_edge_shapes(q, oracle_mod, monkeypatch):
    """Grid tier through the bank-aligned two-slot kernel: ragged row counts (not a multiple of the 8-row chunk), empty /
    dropped / over-long rows, over-full chunks, a 90-isoform locus (fewer than 16 banks per row in use), and a plain
    giant-shaped locus; bit-reproducible when the resident batch is solved again."""
    b = synth.concat([_two_slot_edge_locus(40001, 733, 11), synth.giant(n_loci=1, rows_per_locus=4503, seed=4), _two_slot_edge_locus(3001, 90, 12)])   # 40001 rows: > 12 chunks per CTA, the stage refill path runs
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=2)
    monkeypatch.setenv("SBQ_DUAL_VERIFY", "1")   # libsbq checks the prepared layout: distinct banks per step, disjoint slots of rows r, r + 4
    res = run_gpu(q, b, 3, 0)
    assert res["stats"]["loci_grid"] == 3
    assert_matches_oracle(res, ora, b, "two-slot grid kernel")
    q.solve(b["total_mapped_reads"])
    q.finalize_tpm(q.fpkm_sum())
    q.download()
    again = q.results()
    assert np.array_equal(res["theta"], again["theta"]) and np.array_equal(res["iters"], again["iters"])


@pytest.mark.parametrize("T", [1400, 2000])
def test_grid_tier_two_slot_wide_loci(q, oracle_mod, monkeypatch, T):
    """Loci wider than T = 1300 run the two-slot kernel with 6 / 4 warps per CTA (by default since round 2: faster than the
    TMA ring kernel there): same edge-shape locus as above, layout verified, against the oracle."""
    b = _two_slot_edge_locus(9001, T, 31)
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=2)
    monkeypatch.setenv("SBQ_DUAL_VERIFY", "1")
    res = run_gpu(q, b, 3, 0)
    assert [r["kernel"] for r in q.launch_stats() if r["n_loci"]] == ["em_grid_dual_kernel"]
    assert_matches_oracle(res, ora, b, "two-slot grid kernel, T = %d" % T)


def test_small_giants_run_on_a_sub_grid_beside_the_other_tiers(q, oracle_mod, monkeypatch):
    """Grid-tier loci below 1 M non-zeros ("small giants") are solved by the same grid kernels on a 32-CTA sub-grid, on a stream
    of their own, while the cluster and warp tiers use the other SMs. Planner-chosen tiers (nothing forced): a sparse small giant
    (two-slot kernel) and a dense one (TMA ring kernel) inside a human-shaped batch, every locus against the oracle, bit-
    reproducible when solved again, and identical to the full-grid solve of the same loci to the tolerance of the oracle test."""
    rng = np.random.default_rng(11)
    dense = _shape_locus(rng, 200, 2600, 125)
    dense["total_mapped_reads"] = int(dense["count"].sum())
    b = synth.concat([synth.human_shaped(n_loci=300, total_fragments=150_000, seed=9, max_rows=400), synth.giant(n_loci=1, rows_per_locus=8000, seed=5), dense])
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=2)
    monkeypatch.setenv("SBQ_DUAL_VERIFY", "1")
    res = run_gpu(q, b)
    sub = [r for r in q.launch_stats() if r["kernel"].startswith("em_grid")]
    assert len(sub) == 1 and sub[0]["cluster_size"] == 32 and sub[0]["n_loci"] == 2, sub        # both on the sub-grid
    assert res["stats"]["loci_grid"] == 2 and res["stats"]["loci_warp"] > 0 and res["stats"]["loci_cta"] > 0
    assert_matches_oracle(res, ora, b, "small giants on a sub-grid")
    q.solve(b["total_mapped_reads"])
    q.finalize_tpm(q.fpkm_sum())
    q.download()
    again = q.results()
    assert np.array_equal(res["theta"], again["theta"]) and np.array_equal(res["iters"], again["iters"])


def test_grid_tier_two_slot_rows_with_unsorted_columns(q, oracle_mod, monkeypatch):
    """The two-slot layout pairs rows by merging their (ascending) column lists; a row whose columns are not strictly
    ascending (out of contract: sbq_validate rejects it, but validation is optional) must stay in CSR order and be walked
    from global memory - same results."""
    b = _two_slot_edge_locus(3001, 300, 21)
    rng = np.random.default_rng(5)
    rp = b["row_ptr"]
    for i in range(0, 3001, 3):                      # every third row: columns (and their alphas) in random order
        k0, k1 = int(rp[i]), int(rp[i + 1])
        perm = rng.permutation(k1 - k0)
        b["col"][k0:k1] = b["col"][k0:k1][perm]
        b["alpha"][k0:k1] = b["alpha"][k0:k1][perm]
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"])
    monkeypatch.setenv("SBQ_DUAL_VERIFY", "1")
    q.clear()                                        # (sbq_validate rejects such input; callers may skip validation)
    q.set_plan(3, 0)
    q.submit_flat(b)
    q.run(b["total_mapped_reads"])
    res = q.results()
    assert any(r["kernel"] == "em_grid_dual_kernel" for r in q.launch_stats())
    assert_matches_oracle(res, ora, b, "two-slot kernel, unsorted columns")


def test_grid_tier_random_sweep_against_the_oracle():
    """tools/grid_sweep.py: eight randomised giant-tier shapes (17 to 1290 isoforms, 3 to 55 non-zeros per row, 3 to 12 345 rows,
    zero counts, dropped rows) through the grid tier with the prepared layout verified, each against the oracle."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "grid_sweep.py")], capture_output=True, text=True, timeout=900)
    assert out.returncode == 0 and "grid_sweep ok" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]


def _shape_locus(rng, T, R, k_mean, empty_rows=0, dropped_rows=0):
    """One locus with Poisson(k_mean) columns per row (clamped to 1..T), plus rows without entries and rows whose
    alphas are all below the row filter."""
    rows = []
    for i in range(R):
        k = int(min(T, max(1, rng.poisson(k_mean))))
        c = np.sort(rng.choice(T, k, replace=False)).astype(np.int32)
        a = 10.0 ** rng.uniform(-4, -1.5, k)
        rows.append((c, a))
    for _ in range(empty_rows):
        rows.insert(int(rng.integers(0, len(rows) + 1)), (np.zeros(0, np.int32), np.zeros(0)))
    for _ in range(dropped_rows):
        k = int(min(T, 2))
        rows.insert(int(rng.integers(0, len(rows) + 1)), (np.arange(k, dtype=np.int32), np.full(k, 1e-6)))
    rp = np.concatenate([[0], np.cumsum([len(c) for c, _ in rows])]).astype(np.int64)
    n = len(rows)
    return dict(loc_row_off=np.array([0, n], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=rp,
                col=np.concatenate([c for c, _ in rows]).astype(np.int32), alpha=np.concatenate([a for _, a in rows]),
                count=rng.integers(1, 100, n).astype(np.int32), iso_len=rng.integers(300, 5000, T).astype(np.int32),
                total_mapped_reads=1_000_000)


def test_giant_loci_are_solved_the_same_whatever_shares_their_batch(q, oracle_mod):
    """The grid kernel and its warp count are chosen from the locus' own shape: four giant-tier loci that take four different
    launches - TMA ring with 24 warps, TMA ring with 12 warps, register-staged, two-slot - solved in one batch give the same bits as
    each solved alone."""
    rng = np.random.default_rng(29)
    loci = [_shape_locus(rng, 300, 3000, 80),     # dense rows (> 56 non-zeros on average): TMA ring, 24 warps
            _shape_locus(rng, 1200, 3000, 80),    # dense rows: TMA ring, 12 warps
            _shape_locus(rng, 2700, 3000, 30),    # too wide for the two-slot and TMA ring kernels: register-staged
            _shape_locus(rng, 600, 3000, 30)]     # two-slot kernel
    b = synth.concat(loci)
    b["total_mapped_reads"] = 1_000_000
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=2)
    res = run_gpu(q, b, 3, 0)
    assert [r["kernel"] for r in q.launch_stats() if r["n_loci"]] == ["em_grid_dual_kernel"]
    assert_matches_oracle(res, ora, b, "mixed giant-tier batch")
    iso = b["loc_iso_off"]
    for l, one in enumerate(loci):
        alone = run_gpu(q, one, 3, 0)
        sl = slice(iso[l], iso[l + 1])
        assert np.array_equal(res["theta"][sl].view(np.uint64), alone["theta"].view(np.uint64)), l
        assert res["iters"][l] == alone["iters"][0] and res["status"][l] == alone["status"][0], l


@pytest.mark.parametrize("min_iso_frac", [0.01, 0.0])
def test_epilogue_options_through_every_em_kernel(oracle_mod, min_iso_frac):
    """The low-fraction filter and the effective-length "NA" branch (iso_len < insert_mean) through kernels the planner would
    not send such loci to: the four giant-tier launches of the batch above (two-slot, TMA ring at 24 and 12 warps,
    register-staged), and the warp and cluster tiers on the golden batch (all four locus outcomes). Every solve against the
    oracle, keep flags signed: -1 for a kept NA isoform, which only happens without the filter (it has frac 0)."""
    rng = np.random.default_rng(29)
    giant = synth.concat([_shape_locus(rng, 300, 3000, 80), _shape_locus(rng, 1200, 3000, 80), _shape_locus(rng, 2700, 3000, 30),
                          _shape_locus(rng, 600, 3000, 30)])
    giant["total_mapped_reads"] = 1_000_000
    golden, *_ = load_golden()
    kw = dict(min_iso_frac=min_iso_frac, effective_len_norm=1, insert_mean=200.0)
    for b, tier, cluster, counter in ((giant, 3, 0, "loci_grid"), (golden, 1, 0, "loci_warp"), (golden, 2, 2, "loci_cta")):
        b["iso_len"] = b["iso_len"].copy()
        b["iso_len"][::13] = 150
        ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], min_iso_frac=min_iso_frac, effective_len_norm=True, insert_mean=200.0,
                                        n_threads=4)
        res = run_gpu(None, b, tier, cluster, **kw)
        what = f"epilogue options, tier {tier} cluster {cluster}, min_iso_frac {min_iso_frac}"
        assert res["stats"][counter] > 0, what
        assert_matches_oracle(res, ora, b, what)
        na = b["iso_len"] < 200
        assert np.array_equal(res["keep"], np.where(na & (ora["keep"] != 0), -1, ora["keep"])), what
        want = [0, 1] if min_iso_frac > 0 else [-1, 1]
        assert all((res["keep"] == k).any() for k in want), what


@pytest.mark.parametrize("cluster", [1, 2, 16])
def test_cluster_tier_edge_shapes(q, oracle_mod, cluster):
    """Shapes that take the less common branches of the cluster kernel: more isoforms than threads (generic M-step),
    more rows than threads (four-rows-per-thread E-step), a slice too large for shared memory (streaming fallback),
    empty and dropped rows, a single isoform, rows as long as T."""
    rng = np.random.default_rng(77)
    shapes = [dict(T=600, R=400, k_mean=40), dict(T=20, R=3000, k_mean=3), dict(T=100, R=3000, k_mean=30),
              dict(T=5, R=40, k_mean=2, empty_rows=7, dropped_rows=9), dict(T=1, R=10, k_mean=1),
              dict(T=700, R=40, k_mean=650), dict(T=40, R=700, k_mean=12, empty_rows=3), dict(T=33, R=33, k_mean=33)]
    b = synth.concat([_shape_locus(rng, **s) for s in shapes])
    b["total_mapped_reads"] = 1_000_000
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"])
    res = run_gpu(q, b, 2, cluster)
    assert_matches_oracle(res, ora, b, f"edge shapes, cluster {cluster}")
    assert res["stats"]["loci_cta"] == len(shapes)
