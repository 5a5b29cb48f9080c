"""Bias mode (bias_mode = 1) on the GPU against the CPU restatement (oracle.bias_quantify_batch), which is its only oracle: the
reference has no bias implementation, so parity with the reference is unpinned (DESIGN section 7).

(a) the whole benchmark workload (BASELINE configs[2]: 20 000 human-shaped loci, 5 covariates) at 1, 3 and 100 outer rounds;
(b) edge shapes, one batch per covariate count, placed by shape into the warp kernel (fast and general path) and every cluster
    size of em_bias_kernel, with dropped / empty / zero-count rows, NO_ROWS and ZERO_DENOM exits, degenerate and clamped
    covariates, binding caps, the epilogue options and the width limit;
(c) two GPUs in one context against one."""
import numpy as np
import pytest

import util
from strawberry_b200 import synth

pytestmark = pytest.mark.gpu

ROW_EPS = 1e-5
# restated from strawberry_b200/csrc/sbq_bias.cuh and sbq_kernels.cuh (which loci go where; bias mode records no launch stats)
WT_MAX_ISO, WT_MAX_ROWS, WT_MAX_NNZ, BW_REG, BI_W = 32, 64, 256, 8, 8
SMEM_CAP = 220 * 1024          # dynamic shared memory em_bias_kernel may ask for (sbq.cu SMEM_CAP)


def bias_warp_tier(nnz, R, T):
    return T <= WT_MAX_ISO and R <= WT_MAX_ROWS and nnz <= WT_MAX_NNZ


def bias_cluster_size(nnz):
    return 1 if nnz <= 6000 else 2 if nnz <= 16000 else 4 if nnz <= 40000 else 8 if nnz <= 100000 else 16


def bias_smem_bytes(T):
    return (5 * T + 8 + BI_W * T) * 8


BIAS_MAX_ISO = (SMEM_CAP // 8 - 8) // (5 + BI_W)      # 2165: the widest locus em_bias_kernel takes


def placement(batch, l):
    """'warp-fast' / 'warp' (general path of em_bias_warp_kernel) or 'cs<N>' (em_bias_kernel on clusters of N CTAs)."""
    r0, r1 = int(batch["loc_row_off"][l]), int(batch["loc_row_off"][l + 1])
    T = int(batch["loc_iso_off"][l + 1] - batch["loc_iso_off"][l])
    rp = batch["row_ptr"][r0:r1 + 1]
    nnz = int(rp[-1] - rp[0])
    if bias_warp_tier(nnz, r1 - r0, T):
        return "warp-fast" if r1 - r0 <= 32 and (len(rp) < 2 or np.diff(rp).max() <= BW_REG) else "warp"
    return f"cs{bias_cluster_size(nnz)}"


def kept_rows(batch):
    """row filter of the EM: a row counts when one of its alphas exceeds row_eps"""
    big = np.concatenate([[0], np.cumsum(batch["alpha"] > ROW_EPS)])
    return np.diff(big[batch["row_ptr"]]) > 0


def run_gpu(batch, X, n_gpus=1, resolve=False, **cfg):
    from strawberry_b200 import api
    q = api.Quantifier(device=0, bias_mode=1, n_gpus=n_gpus, **cfg)
    try:
        q.submit_flat(batch)
        q.set_covariates(X)
        q.run(batch["total_mapped_reads"])
        res = q.results()
        res["beta"], res["outer"] = q.bias_results()
        res["stats"] = q.stats()
        if resolve:   # a second solve of the resident batch
            q.solve(batch["total_mapped_reads"])
            q.finalize_tpm(q.fpkm_sum())
            q.download()
            again = q.results()
            again["beta"], again["outer"] = q.bias_results()
            res["again"] = again
        return res
    finally:
        q.close()


def oracle_limits(cfg):
    return {k: v for k, v in cfg.items() if k in ("max_out_it", "max_theta_it", "max_bias_it", "theta_tol", "bias_tol")}


def oracle_epilogue_opts(cfg):
    return {k: v for k, v in cfg.items() if k in ("min_iso_frac", "effective_len_norm", "insert_mean")}


def eta_error(res, ora, batch, X, loci_mask):
    """worst |eta_gpu - eta_cpu| / max(1, |eta_cpu|) over the kept rows of the loci in loci_mask, eta_i = x_i . beta"""
    if X.shape[1] == 0:
        return 0.0
    nrow = np.diff(batch["loc_row_off"])
    rows = kept_rows(batch) & np.repeat(loci_mask, nrow)
    bg, bo = np.repeat(res["beta"], nrow, axis=0), np.repeat(ora["beta"], nrow, axis=0)
    eg, eo = (X * bg).sum(1)[rows], (X * bo).sum(1)[rows]
    return float((np.abs(eg - eo) / np.maximum(1.0, np.abs(eo))).max()) if rows.any() else 0.0


# ---------------------------------------------------------------------------------------------------------------- (a) configs[2]
@pytest.fixture(scope="module")
def configs2():
    b = synth.human_shaped(seed=2)
    return b, synth.covariates(b, seed=3)


def _flips(oracle_mod, batch, X, l, limits):
    """does the restatement's own (status, iters, outer) change when both tolerances move by a factor 1 +- 1e-6?"""
    T, rp, col, al, cnt, _ = synth.locus_slice(batch, l)
    x = X[batch["loc_row_off"][l]:batch["loc_row_off"][l + 1]]
    tt, bt = limits.get("theta_tol", 1e-2), limits.get("bias_tol", 1e-2)
    lim = {k: v for k, v in limits.items() if k not in ("theta_tol", "bias_tol")}
    base = oracle_mod.em_bias_csr(T, rp, col, al, cnt, x, theta_tol=tt, bias_tol=bt, **lim)
    for f in (1 + 1e-6, 1 - 1e-6):
        r = oracle_mod.em_bias_csr(T, rp, col, al, cnt, x, theta_tol=tt * f, bias_tol=bt * f, **lim)
        if (r[0], r[3], r[4]) != (base[0], base[3], base[4]):
            return True
    return False


# max_out_it -> (bar on theta / FPKM / frac / TPM, bar on eta, eta compared on converged loci only). After one outer round the
# parity bar holds: theta within 1e-6, eta = X beta within 1e-6 max(1, |eta|) on every kept row. Later rounds solve the Newton
# system again from a beta that is itself ill-determined (gc, gc^2, gc^3 nearly collinear, 5 covariates on 8 - 21 rows), and the
# restatement's own answer moves when X moves by one ulp: perturbing every covariate by a random +-1 ulp changes no
# (status, iters, outer), but moves theta by up to 6.2e-7 / 1.07e-5 (ratio of util.theta_close) and eta by up to 2.4e-4 / 1.0
# after 3 / 100 rounds (1.5e-4 on the 6 338 loci that converge within 100 rounds). The bars are 4x those measurements.
CONFIGS2_BARS = {1: (1e-6, 1e-6, False), 3: (2.5e-6, 1e-3, False), 100: (5e-5, 6e-4, True)}


@pytest.mark.parametrize("max_out_it", [1, 3, 100])
def test_configs2_matches_restatement(oracle_mod, configs2, max_out_it):
    """The benchmark's bias workload, every locus: status / theta iterations / outer rounds equal, theta / FPKM / frac / TPM /
    keep as in every other parity test (bars of CONFIGS2_BARS), eta = X beta on every kept row, the fragment-iteration count of
    the metric, and a second solve bit-identical. beta itself is not compared: it is ill-determined where eta is not.
    A locus whose counts differ is accepted only when the restatement itself flips under tolerances x (1 +- 1e-6); at most 4."""
    rel, eta_bar, eta_converged_only = CONFIGS2_BARS[max_out_it]
    b, X = configs2
    cfg = dict(max_out_it=max_out_it)
    res = run_gpu(b, X, resolve=True, **cfg)
    ora = oracle_mod.bias_quantify_batch(b, X, b["total_mapped_reads"], n_threads=16, **cfg)
    diff = np.nonzero((res["status"] != ora["status"]) | (res["iters"] != ora["iters"]) | (res["outer"] != ora["outer"]))[0]
    marginal = [int(l) for l in diff if _flips(oracle_mod, b, X, int(l), cfg)]
    if len(diff):
        print(f"max_out_it {max_out_it}: counts differ at loci {diff[:20].tolist()}, marginal (restatement flips at tol x (1 +- 1e-6)): {marginal}")
    assert len(marginal) == len(diff), f"counts differ at non-marginal loci {sorted(set(diff.tolist()) - set(marginal))[:10]}"
    assert len(marginal) <= 4, f"{len(marginal)} marginal loci"
    ok_loci = np.ones(len(res["status"]), bool)
    ok_loci[marginal] = False
    ora_m = {k: ora[k].copy() for k in ("theta", "fpkm", "frac", "tpm", "keep", "iters", "status")}
    iso = util.expand_loci(~ok_loci, b)
    for k in ("theta", "fpkm", "frac", "tpm", "keep"):
        ora_m[k][iso] = res[k][iso]          # marginal loci: stopping decision differs, compared above instead
    for k in ("iters", "status"):
        ora_m[k][~ok_loci] = res[k][~ok_loci]
    worst = util.assert_matches_oracle(res, ora_m, b, what=f"configs[2] bias, max_out_it {max_out_it}", rel=rel)
    eta = eta_error(res, ora, b, X, ok_loci & (ora["status"] == 0) if eta_converged_only else ok_loci)
    print(f"max_out_it {max_out_it}: worst theta ratio {worst:.3e}, worst eta error {eta:.3e}, {len(marginal)} marginal loci")
    assert eta <= eta_bar, f"eta = X beta off by {eta:.3e}"
    tot = util.locus_totals(b)
    assert res["stats"]["frag_iters"] == int((tot * res["iters"].astype(np.int64)).sum())
    assert res["stats"]["frag_iters"] == int((tot[ok_loci] * ora["iters"][ok_loci].astype(np.int64)).sum()) + \
        int((tot[~ok_loci] * res["iters"][~ok_loci].astype(np.int64)).sum())
    for k in ("theta", "fpkm", "frac", "tpm", "keep", "iters", "status", "beta", "outer"):
        assert np.array_equal(res["again"][k], res[k], equal_nan=True), f"second solve differs in {k}"


# ---------------------------------------------------------------------------------------------------------------- (b) edge shapes
def _locus(rng, T, R, K, nnz=(1, 8), drop=(), empty=(), zero=(), long_rows=None, zero_denom=False, x=None, set_count=None, faint=(), n_total=20_000):
    """One locus with a planted bias. Row i covers k_i ~ U{nnz} distinct isoforms (long_rows: {row: k} overrides), alphas
    10^U(-3.5, -1.5), counts Poisson from the planted model; then rows in `drop` get every alpha below row_eps (dropped by the
    row filter, count kept), rows in `empty` no entries (and a count), rows in `zero` count 0, set_count: {row: count}, rows in `faint` alphas of 2e-5 (kept). zero_denom: the last isoform is
    covered only by one extra count-0 row, so its theta is 0 after one EM step and that kept row's denominator vanishes."""
    Tr = T - 1 if zero_denom else T
    ks = rng.integers(nnz[0], min(nnz[1], Tr) + 1, R)
    for i, k in (long_rows or {}).items():
        ks[i] = k
    ks[list(empty)] = 0
    col = np.concatenate([np.sort(rng.choice(Tr, k, replace=False)) for k in ks] + [np.zeros(0, np.int64)]).astype(np.int32)
    rp = np.concatenate([[0], np.cumsum(ks)]).astype(np.int64)
    alpha = 10.0 ** rng.uniform(-3.5, -1.5, len(col))
    X = rng.normal(0.0, 0.5, (R, K)) if x is None else x
    w = np.exp(X @ rng.uniform(-0.6, 0.6, K))
    s = np.zeros(T)
    np.add.at(s, col, alpha * np.repeat(w, ks))
    theta = rng.dirichlet(np.ones(T)) * n_total
    p = np.array([w[i] * np.sum(alpha[rp[i]:rp[i + 1]] * theta[col[rp[i]:rp[i + 1]]] / s[col[rp[i]:rp[i + 1]]]) for i in range(R)])
    count = rng.poisson(n_total * p / max(p.sum(), 1e-300)).astype(np.int32)
    for i in drop:
        alpha[rp[i]:rp[i + 1]] = 5e-6
    for i in faint:
        alpha[rp[i]:rp[i + 1]] = 2e-5
    count[list(empty)] = rng.integers(1, 50, len(empty))
    count[list(zero)] = 0
    for i, n in (set_count or {}).items():
        count[i] = n
    if zero_denom:
        col, rp = np.append(col, T - 1).astype(np.int32), np.append(rp, rp[-1] + 1)
        alpha, count, X = np.append(alpha, 1e-2), np.append(count, 0).astype(np.int32), np.vstack([X, rng.normal(0.0, 0.5, (1, K))])
    iso_len = rng.integers(400, 8000, T).astype(np.int32)
    iso_len[rng.choice(T, max(1, T // 8), replace=False)] = 120     # shorter than insert_mean: effective length < 0 (FPKM n/a)
    return dict(loc_row_off=np.array([0, len(count)]), loc_iso_off=np.array([0, T]), row_ptr=rp, col=col, alpha=alpha, count=count,
                iso_len=iso_len, total_mapped_reads=int(count.sum()), X=X)


def edge_loci(K):
    """[(name, intended placement, intended status or None, locus)] of the edge batch with K covariates"""
    rng = np.random.default_rng(1000 + K)
    out = []

    def add(name, where, status=None, **kw):
        out.append((name, where, status, _locus(rng, K=K, **kw)))

    mid = dict(drop=(5, 9), empty=(7,), zero=(3, 12))
    # warp kernel
    add("fast path", "warp-fast", T=6, R=20, nnz=(1, 8), **mid)
    add("rows of 9 - 12", "warp", T=16, R=20, nnz=(9, 12), **mid)
    add("a row of 32", "warp", T=32, R=12, nnz=(1, 6), long_rows={3: 32}, drop=(7,), empty=(1,), zero=(5,))
    add("R = 32", "warp-fast", T=8, R=32, nnz=(1, 6), drop=(30,), empty=(0,), zero=(16,))
    add("R = 33", "warp", T=8, R=33, nnz=(1, 6), drop=(32,), empty=(31,), zero=(1,))
    add("R = 64", "warp", T=4, R=64, nnz=(1, 4), drop=(40, 63), empty=(33,), zero=(10, 50))
    add("T = 32", "warp-fast", T=32, R=30, nnz=(1, 8), **mid)
    add("T = 33", "cs1", T=33, R=40, nnz=(1, 6), **mid)
    add("no kept rows", "warp-fast", 3, T=3, R=6, nnz=(1, 3), drop=range(6))
    add("no rows at all", "warp-fast", 3, T=2, R=0)
    add("zero denominator", "warp-fast", 2, T=5, R=6, nnz=(1, 3), zero_denom=True)
    # em_bias_kernel, every cluster size
    add("cluster 1", "cs1", T=40, R=150, nnz=(1, 30), **mid)
    add("cluster 2", "cs2", T=40, R=500, nnz=(10, 40), **mid)
    add("cluster 4", "cs4", T=50, R=1000, nnz=(15, 45), **mid)
    add("cluster 8", "cs8", T=60, R=2000, nnz=(20, 60), **mid)
    add("cluster 16", "cs16", T=64, R=2600, nnz=(30, 64), drop=(5, 1300, 2599), empty=(7, 1301), zero=(3, 12, 2000))
    add("cluster, no kept rows", "cs1", 3, T=40, R=10, nnz=(1, 5), drop=range(10))
    add("cluster, zero denominator", "cs1", 2, T=40, R=60, nnz=(1, 10), zero_denom=True)
    add("cluster 2, zero denominator", "cs2", 2, T=40, R=500, nnz=(10, 40), zero_denom=True)
    if K:
        # degenerate Newton systems, held up by the ridge only: a constant-zero covariate and (K >= 3) a duplicated one
        x = np.random.default_rng(77).normal(0.0, 0.5, (30, K))
        x[:, 0] = 0.0
        if K >= 3:
            x[:, 2] = x[:, 1]
        add("singular covariates", "warp-fast", T=6, R=30, nnz=(1, 4), x=x)
        x = np.random.default_rng(78).normal(0.0, 0.5, (400, K))
        x[:, 0] = 0.0
        if K >= 3:
            x[:, 2] = x[:, 1]
        add("singular covariates, cluster", "cs1", T=40, R=400, nnz=(1, 12), x=x)
        # a covariate carried by one faint row only, whose count is far above what the unbiased model gives it: the first Newton step
        # moves its eta to about n_i / mu_i - 1, far past the +30 clamp, and later steps walk it back one unit at a time
        for where, T, R, z in (("warp-fast", 5, 24, 20), ("cs1", 40, 200, 7)):
            x = np.random.default_rng(79).normal(0.0, 0.5, (R, K))
            x[:, 0], x[z] = 0.0, 0.0
            x[z, 0] = 1.0
            add("clamp", where, T=T, R=R, nnz=(1, 4), x=x, long_rows={z: T}, set_count={z: 200_000}, faint=(z,))
    return out


def edge_batch(K):
    loci = edge_loci(K)
    b = synth.concat([l for _, _, _, l in loci])
    X = np.concatenate([l["X"] for _, _, _, l in loci])
    return loci, b, X


EDGE_CFGS = {
    "defaults+epilogue": dict(min_iso_frac=0.01, effective_len_norm=1, insert_mean=250.0),
    "caps": dict(max_theta_it=3, max_bias_it=1, max_out_it=2),
}


@pytest.mark.parametrize("cfg_name", list(EDGE_CFGS))
@pytest.mark.parametrize("K", [0, 1, 4, 6])
def test_edge_shapes_match_restatement(oracle_mod, K, cfg_name):
    """Edge-shape batch with K covariates: every locus lands where it is meant to, and status / iterations / outer rounds /
    theta / FPKM / frac / TPM / keep / beta (absolute 1e-7) agree with the restatement locus by locus."""
    cfg = EDGE_CFGS[cfg_name]
    loci, b, X = edge_batch(K)
    where = [placement(b, l) for l in range(len(loci))]
    assert where == [w for _, w, _, _ in loci]
    assert {"warp-fast", "warp", "cs1", "cs2", "cs4", "cs8", "cs16"} <= set(where)
    res = run_gpu(b, X, **cfg)
    ora = oracle_mod.bias_quantify_batch(b, X, b["total_mapped_reads"], n_threads=16, **oracle_limits(cfg), **oracle_epilogue_opts(cfg))
    for l, (name, w, status, _) in enumerate(loci):
        if status is not None:
            assert ora["status"][l] == status, f"{name}: the restatement does not reach status {status}"
        assert (res["status"][l], res["iters"][l], res["outer"][l]) == (ora["status"][l], ora["iters"][l], ora["outer"][l]), \
            f"{name} ({w}): (status, iters, outer) {(res['status'][l], res['iters'][l], res['outer'][l])} vs {(ora['status'][l], ora['iters'][l], ora['outer'][l])}"
        if K:
            err = np.abs(res["beta"][l] - ora["beta"][l]).max()
            assert err < 1e-7, f"{name} ({w}): beta off by {err:.3e}: {res['beta'][l]} vs {ora['beta'][l]}"
    util.assert_matches_oracle(res, ora, b, what=f"edge shapes K={K} {cfg_name}")
    for name, _, _, loc in loci:
        if name == "clamp":   # the clamp cases do reach it: eta beyond 30 after the first outer round of the restatement
            beta1 = oracle_mod.em_bias_csr(int(loc["loc_iso_off"][1]), loc["row_ptr"], loc["col"], loc["alpha"], loc["count"], loc["X"], max_out_it=1)[2]
            assert np.abs(loc["X"] @ beta1).max() > 30.0


def test_width_limit(oracle_mod):
    """T = 2165 is the widest locus whose shared-memory footprint fits em_bias_kernel; T = 2166 is refused with SBQ_ERR_UNSUPPORTED."""
    from strawberry_b200 import api
    assert bias_smem_bytes(BIAS_MAX_ISO) <= SMEM_CAP < bias_smem_bytes(BIAS_MAX_ISO + 1) and BIAS_MAX_ISO == 2165
    rng = np.random.default_rng(5)
    loc = _locus(rng, T=BIAS_MAX_ISO, R=2400, K=2, nnz=(1, 3), drop=(10,), zero=(20,))
    assert placement(loc, 0) == "cs1"
    res = run_gpu(loc, loc["X"])
    ora = oracle_mod.bias_quantify_batch(loc, loc["X"], loc["total_mapped_reads"])
    assert (res["status"][0], res["iters"][0], res["outer"][0]) == (ora["status"][0], ora["iters"][0], ora["outer"][0])
    assert np.abs(res["beta"] - ora["beta"]).max() < 1e-7
    util.assert_matches_oracle(res, ora, loc, what="T = 2165")
    wide = _locus(rng, T=BIAS_MAX_ISO + 1, R=3000, K=2, nnz=(1, 3))
    with pytest.raises(api.SbqError) as e:
        run_gpu(wide, wide["X"])
    assert e.value.code == api.SBQ_ERR_UNSUPPORTED


# ---------------------------------------------------------------------------------------------------------------- (c) N GPUs
@pytest.mark.parametrize("K", [5, 0])
def test_two_gpus_match_one(K):
    """n_gpus = 2 in one context: covariate rows gathered per device, beta / outer scattered back into submit order; every result
    bitwise equal to one GPU, TPM up to the order of one sum."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    b = synth.human_shaped(n_loci=3000, total_fragments=1_500_000, seed=77)
    X = synth.covariates(b, seed=3)[:, :K]
    one, two = run_gpu(b, X), run_gpu(b, X, n_gpus=2)
    for k in ("theta", "fpkm", "frac", "keep", "iters", "status", "beta", "outer"):
        assert np.array_equal(two[k], one[k], equal_nan=True), k
    assert np.allclose(two["tpm"], one["tpm"], rtol=1e-12, atol=0, equal_nan=True)
