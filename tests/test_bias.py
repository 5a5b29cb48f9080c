"""Bias mode (bias_mode = 1). The reference has NO bias implementation (src/bias.cpp is commented out), so parity
here is against OUR CPU restatement (oracle.em_bias_csr) only - "parity unpinned" with respect to the reference.
CPU tests pin the restatement's own properties; the GPU test checks the fused CUDA kernel against it."""
import numpy as np
import pytest

from strawberry_b200 import synth


def biased_locus(seed, T=6, R=120, K=5, beta_true=(0.8, -0.5, 0.3, 0.0, 0.4), n_total=200_000):
    rng = np.random.default_rng(seed)
    rows, rp = [], [0]
    for i in range(R):
        k = int(rng.integers(1, T + 1))
        rows.append(np.sort(rng.choice(T, k, replace=False)))
        rp.append(rp[-1] + k)
    col = np.concatenate(rows).astype(np.int32)
    alpha = 10.0 ** rng.uniform(-3.5, -2.0, len(col))
    gc = rng.beta(8, 8, R)
    X = np.stack([gc, gc ** 2, gc ** 3, np.log(rng.integers(50, 400, R)) / 5.0, rng.normal(0.25, 0.03, R)], axis=1)[:, :K]
    theta_true = rng.dirichlet(np.ones(T)) * n_total
    w = np.exp(X @ np.array(beta_true[:K]))
    rp = np.array(rp, np.int64)
    s = np.zeros(T)
    np.add.at(s, col, alpha * np.repeat(w, np.diff(rp)))
    p = np.array([w[i] * np.sum(alpha[rp[i]:rp[i + 1]] * theta_true[col[rp[i]:rp[i + 1]]] / s[col[rp[i]:rp[i + 1]]]) for i in range(R)])
    count = rng.poisson(n_total * p / p.sum()).astype(np.int32)
    return dict(T=T, row_ptr=rp, col=col, alpha=alpha, count=count, X=X, iso_len=np.full(T, 1500, np.int32))


def test_restatement_without_covariates_is_a_plain_em_fixed_point(oracle_mod):
    L = biased_locus(1, K=0)
    st, th, beta, iters, outer = oracle_mod.em_bias_csr(L["T"], L["row_ptr"], L["col"], L["alpha"], L["count"], L["X"])
    assert st == 0 and outer == 1 and len(beta) == 0
    # one more reference-style EM step from th moves it by less than the tolerance
    st2, th2, it2 = oracle_mod.em_csr(L["T"], L["row_ptr"], L["col"], L["alpha"], L["count"])
    assert np.allclose(th, th2, rtol=5e-3, atol=5e-2)


def test_restatement_recovers_a_planted_bias_direction(oracle_mod):
    L = biased_locus(2)
    st, th, beta, iters, outer = oracle_mod.em_bias_csr(L["T"], L["row_ptr"], L["col"], L["alpha"], L["count"], L["X"])
    assert st in (0, 1) and outer >= 2
    w_fit = L["X"] @ beta
    w_true = L["X"] @ np.array([0.8, -0.5, 0.3, 0.0, 0.4])
    assert np.corrcoef(w_fit, w_true)[0, 1] > 0.9      # the fitted row weights follow the planted ones
    assert abs(th.sum() - L["count"].sum()) < 1e-6 * L["count"].sum()


@pytest.mark.parametrize("opts", [{}, dict(min_iso_frac=0.01, effective_len_norm=True, insert_mean=250.0)])
def test_batch_epilogue_reproduces_quantify_batch(oracle_mod, opts):
    """The FPKM / frac / keep / TPM tail of oracle.bias_quantify_batch, fed quantify_batch's theta and status, gives
    quantify_batch's own answers on the golden batch (pins the helper's arithmetic, TPM summation order included)."""
    import util
    b, *_ = util.load_golden()
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], **opts)
    got = oracle_mod.batch_epilogue(b, ora["theta"], ora["status"], b["total_mapped_reads"], **opts)
    for k in ("fpkm", "frac", "tpm", "keep"):
        assert np.array_equal(got[k], ora[k], equal_nan=True), k


@pytest.mark.gpu
def test_bias_kernel_matches_restatement(oracle_mod, sbq_lib_path):
    from strawberry_b200 import api
    loci = [biased_locus(s, T=int(t), R=int(r), K=k) for s, t, r, k in ((3, 4, 60, 5), (4, 12, 300, 5), (5, 40, 900, 3), (6, 3, 20, 2), (7, 8, 150, 0),
                                                                                # loci large enough for clusters of 2, 8 and 16 CTAs (non-zeros > 6 k / 40 k / 100 k)
                                                                                (8, 30, 700, 3), (9, 60, 2000, 5), (10, 80, 3000, 2))]
    for K in sorted({l["X"].shape[1] for l in loci}):
        group = [l for l in loci if l["X"].shape[1] == K]
        parts = [dict(loc_row_off=np.array([0, len(l["count"])]), loc_iso_off=np.array([0, l["T"]]), row_ptr=l["row_ptr"], col=l["col"],
                      alpha=l["alpha"], count=l["count"], iso_len=l["iso_len"], total_mapped_reads=int(l["count"].sum())) for l in group]
        b = synth.concat(parts)
        q = api.Quantifier(bias_mode=1)
        q.submit_flat(b)
        q.set_covariates(np.concatenate([l["X"] for l in group]) if K else np.zeros((int(b["loc_row_off"][-1]), 0)))
        q.run(b["total_mapped_reads"])
        res = q.results()
        beta, outer = q.bias_results()
        for i, l in enumerate(group):
            st, th, be, iters, out = oracle_mod.em_bias_csr(l["T"], l["row_ptr"], l["col"], l["alpha"], l["count"], l["X"])
            t0 = int(b["loc_iso_off"][i])
            assert res["status"][i] == st
            assert outer[i] == out and res["iters"][i] == iters
            scale = np.maximum(np.abs(th), 1e-9 * l["count"].sum())
            assert (np.abs(res["theta"][t0:t0 + l["T"]] - th) / scale).max() < 1e-6
            assert np.abs(beta[i] - be).max() < 1e-7 if K else True
        q.close()


@pytest.mark.gpu
def test_bias_mode_needs_covariates(sbq_lib_path):
    from strawberry_b200 import api
    b = synth.human_shaped(n_loci=20, total_fragments=5000, seed=3, max_rows=50)
    q = api.Quantifier(bias_mode=1)
    q.submit_flat(b)
    with pytest.raises(api.SbqError) as e:
        q.run(b["total_mapped_reads"])
    assert e.value.code == api.SBQ_ERR_STATE
    q.close()
