"""GPU: bootstrap replicates (sbq_bootstrap, strawberry_b200/csrc/sbq_bootstrap.cuh, DESIGN.md "Bootstrap replicates").

The resampled counts equal the CPU restatement (tests/bootstrap_ref.py) bit for bit; a replicate equals a fresh solve of the batch
with those counts, bitwise, on every tier (which would catch a tier that kept counts from an earlier solve); every forced tier
agrees with the oracle on resampled batches; chunking does not change a replicate; the point estimate is left alone; and the
refusals are the documented ones."""
import numpy as np
import pytest

import bootstrap_ref as br
from strawberry_b200 import synth
from util import load_golden, theta_close

pytestmark = pytest.mark.gpu

SEED = 20240611


@pytest.fixture(scope="module")
def api_mod(sbq_lib_path):
    from strawberry_b200 import api
    return api


@pytest.fixture(scope="module")
def headline():
    return synth.human_shaped(seed=2)


@pytest.fixture(scope="module")
def qh(api_mod, headline):
    """the headline batch (configs[1]) uploaded and solved once"""
    q = api_mod.Quantifier()
    q.submit_flat(headline)
    q.run(headline["total_mapped_reads"])
    yield q
    q.close()


def fresh(api_mod, batch, tier=0, cluster=0, **cfg):
    q = api_mod.Quantifier(**cfg)
    try:
        q.set_plan(tier, cluster)
        q.submit_flat(batch)
        q.run(batch["total_mapped_reads"])
        res = q.results()
        res["launches"] = q.launch_stats()
        return res
    finally:
        q.close()


def boot(api_mod, batch, n, first=0, tier=0, cluster=0, seed=SEED, **cfg):
    q = api_mod.Quantifier(**cfg)
    try:
        q.set_plan(tier, cluster)
        q.submit_flat(batch)
        q.run(batch["total_mapped_reads"])
        return q.bootstrap(seed, n, first)
    finally:
        q.close()


def assert_replicate_is_fresh_solve(rep, j, ref):
    for k in ("theta", "tpm", "iters", "status"):
        assert np.array_equal(rep[k][j], ref[k]), k


def assert_replicate_matches_oracle(rep, j, ora, batch, what):
    assert np.array_equal(rep["status"][j], ora["status"]), what
    assert np.array_equal(rep["iters"][j], ora["iters"]), what
    ok, worst = theta_close(rep["theta"][j], ora["theta"], batch)
    assert ok.all(), (what, worst)
    live = np.repeat(ora["status"], np.diff(batch["loc_iso_off"])) != 3
    a, b = rep["tpm"][j][live], ora["tpm"][live]
    scale = np.maximum(np.abs(b), 1e-9 * max(float(np.abs(b).max()), 1e-300))
    assert (np.abs(a - b) <= 1e-6 * scale).all(), what


def _raw_loci(q, n, seed0):
    """n random loci (tests/locusgen.py) of one read length, submitted raw: the device builds their class tables"""
    import locusgen
    from strawberry_b200 import builder
    s, done, rl0 = seed0, 0, None
    while done < n:
        isoforms, hits, rl = locusgen.random_locus(s)
        s += 1
        if rl0 is None:
            rl0 = rl
            q.set_insert_model(builder.Model.normal(200.0, 40.0), rl)
        if rl != rl0:
            continue
        tfe = [locusgen.transcript_features(ex) for ex in isoforms]
        builder.submit_raw(q, tfe, [(m, builder.pair_features(l, r)) for m, l, r in hits], read_len=rl)
        done += 1


# ---- 1. counts ----------------------------------------------------------------------------------------------------------------

def test_counts_equal_the_restatement_on_the_headline_batch(qh, headline):
    for rep in (0, 1, 1000):
        got = qh.bootstrap_counts(SEED, rep)
        assert np.array_equal(got, br.resample(headline, SEED, rep)), rep
    assert not np.array_equal(qh.bootstrap_counts(SEED, 0), br.resample(headline, SEED + 1, 0))   # negative control


def test_counts_equal_the_restatement_on_a_raw_built_batch(api_mod):
    q = api_mod.Quantifier()
    try:
        _raw_loci(q, 12, 300)
        q.upload()
        b = q.fetch_batch()           # the class counts the device built
        assert b["count"].sum() > 0
        for rep in (0, 5):
            assert np.array_equal(q.bootstrap_counts(SEED, rep), br.resample(b, SEED, rep)), rep
    finally:
        q.close()


def test_counts_equal_the_restatement_on_a_device_generated_giant_locus(api_mod):
    q = api_mod.Quantifier()
    try:
        rows = 1_000_000
        q.synth_giant([3], rows)
        b = dict(count=np.ones(rows, np.int32), loc_row_off=np.array([0, rows], np.int64))   # every generated row is one fragment
        got = q.bootstrap_counts(SEED, 2)
        assert got.sum() == rows
        assert np.array_equal(got, br.resample(b, SEED, 2))
    finally:
        q.close()


# ---- 2. a replicate is a fresh solve of the resampled batch, bitwise -------------------------------------------------------------

def test_headline_replicates_equal_fresh_solves(api_mod, qh, headline):
    rep = qh.bootstrap(SEED, 3)
    for j in range(3):
        assert_replicate_is_fresh_solve(rep, j, fresh(api_mod, br.resampled_batch(headline, SEED, j)))


@pytest.mark.parametrize("rows,variant,sub_grid", [(40_000, 3, False), (10_000, None, True)])
def test_giant_replicates_equal_fresh_solves(api_mod, rows, variant, sub_grid):
    """a giant locus on the full grid's two-slot kernel and a small giant on the sub-grid"""
    b = synth.giant_device([1], rows)
    rep = boot(api_mod, b, 2)
    for j in range(2):
        ref = fresh(api_mod, br.resampled_batch(b, SEED, j))
        (ls,) = [x for x in ref["launches"] if x["kernel"].startswith("em_grid")]
        assert (ls["cluster_size"] > 0) == sub_grid
        if variant == 3:
            assert ls["kernel"] == "em_grid_dual_kernel"
        assert_replicate_is_fresh_solve(rep, j, ref)


# ---- 3. oracle ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("tier,cluster", [(0, 0), (1, 0), (2, 1), (2, 2), (2, 4), (2, 8), (2, 16), (3, 0)])
def test_every_tier_matches_the_oracle_on_resampled_golden_batches(api_mod, oracle_mod, tier, cluster):
    b, *_ = load_golden()
    rep = boot(api_mod, b, 4, tier=tier, cluster=cluster)
    for j in range(4):
        rb = br.resampled_batch(b, SEED, j)
        ora = oracle_mod.quantify_batch(rb, b["total_mapped_reads"])
        assert_replicate_matches_oracle(rep, j, ora, rb, f"tier {tier} cluster {cluster} replicate {j}")


def test_headline_replicate_matches_the_oracle(qh, oracle_mod, headline):
    rep = qh.bootstrap(SEED, 1, first=7)
    rb = br.resampled_batch(headline, SEED, 7)
    ora = oracle_mod.quantify_batch(rb, headline["total_mapped_reads"], n_threads=8)
    assert_replicate_matches_oracle(rep, 0, ora, rb, "configs[1] replicate 7")


def test_filter_and_effective_length_epilogue(api_mod, oracle_mod):
    b = synth.human_shaped(n_loci=600, total_fragments=300_000, seed=41, max_rows=300)
    b["iso_len"] = b["iso_len"].copy()
    b["iso_len"][::17] = 150
    rep = boot(api_mod, b, 2, min_iso_frac=0.01, effective_len_norm=1, insert_mean=200.0)
    for j in range(2):
        rb = br.resampled_batch(b, SEED, j)
        ora = oracle_mod.quantify_batch(rb, b["total_mapped_reads"], min_iso_frac=0.01, effective_len_norm=True, insert_mean=200.0)
        assert_replicate_matches_oracle(rep, j, ora, rb, f"epilogue replicate {j}")
        assert (ora["keep"] == 0).any()


# ---- 4. chunking ------------------------------------------------------------------------------------------------------------------

def test_chunks_do_not_change_a_replicate(api_mod):
    b = synth.human_shaped(n_loci=1500, total_fragments=600_000, seed=5)
    q = api_mod.Quantifier()
    try:
        q.submit_flat(b)
        q.run(b["total_mapped_reads"])
        whole = q.bootstrap(SEED, 6)
        a, c = q.bootstrap(SEED, 3), q.bootstrap(SEED, 3, first=3)
        four = q.bootstrap(SEED, 1, first=4)
        st = q.bootstrap_stats()
    finally:
        q.close()
    for k in ("theta", "tpm", "iters", "status"):
        assert np.array_equal(whole[k], np.concatenate([a[k], c[k]])), k
        assert np.array_equal(whole[k][4], four[k][0]), k
    assert st["first"] == 4 and st["n"] == 1 and 0 < st["resample_ms"] and 0 < st["em_ms"] <= st["total_ms"]


# ---- 5. the point estimate is untouched ----------------------------------------------------------------------------------------

def test_point_estimate_is_untouched(api_mod):
    b = synth.human_shaped(n_loci=1500, total_fragments=600_000, seed=6)
    q = api_mod.Quantifier()
    try:
        q.submit_flat(b)
        q.run(b["total_mapped_reads"])
        before, stats = q.results(), q.stats()
        q.bootstrap(SEED, 3)
        after = q.results()
        assert q.stats() == stats
        q.download()
        again = q.results()
        q.solve(b["total_mapped_reads"])
        q.finalize_tpm(q.fpkm_sum())
        q.download()
        resolved = q.results()
    finally:
        q.close()
    for k in before:
        assert np.array_equal(before[k], after[k]), k
        assert np.array_equal(before[k], again[k]), k
        assert np.array_equal(before[k], resolved[k]), k


# ---- 6. refusals -------------------------------------------------------------------------------------------------------------------

def test_refusals(api_mod):
    b = synth.human_shaped(n_loci=300, total_fragments=100_000, seed=7)
    q = api_mod.Quantifier()
    try:
        with pytest.raises(api_mod.SbqError) as e:
            q.bootstrap(SEED, 1)                       # nothing resident
        assert e.value.code == api_mod.SBQ_ERR_STATE
        q.submit_flat(b)
        q.upload()
        with pytest.raises(api_mod.SbqError) as e:
            q.bootstrap(SEED, 1)                       # resident but not solved
        assert e.value.code == api_mod.SBQ_ERR_STATE
        assert np.array_equal(q.bootstrap_counts(SEED, 0), br.resample(b, SEED, 0))   # counts need the upload only
        q.solve(b["total_mapped_reads"])
        for n, first in ((0, 0), (-1, 0), (1, -1)):
            with pytest.raises(api_mod.SbqError) as e:
                q.bootstrap(SEED, n, first)
            assert e.value.code == api_mod.SBQ_ERR_INVALID
        with pytest.raises(api_mod.SbqError) as e:
            q.bootstrap_counts(SEED, -1)
        assert e.value.code == api_mod.SBQ_ERR_INVALID
        with pytest.raises(api_mod.SbqError) as e:
            q.bootstrap(SEED, 2**31 - 1)               # ~2 PB of replicate matrices: a plain failed allocation
        assert e.value.code == api_mod.SBQ_ERR_NOMEM
        rep = q.bootstrap(SEED, 2)                     # the context stays usable
        ref = fresh(api_mod, br.resampled_batch(b, SEED, 1))
        assert_replicate_is_fresh_solve(rep, 1, ref)
    finally:
        q.close()
    qb = api_mod.Quantifier(bias_mode=1)
    try:
        with pytest.raises(api_mod.SbqError) as e:
            qb.bootstrap(SEED, 1)
        assert e.value.code == api_mod.SBQ_ERR_UNSUPPORTED
    finally:
        qb.close()


# ---- 7. multi-GPU ------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("kind", ["flat", "raw"])
def test_two_gpus_equal_one(api_mod, kind):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = {}
    for n_gpus in (1, 2):
        q = api_mod.Quantifier(device=0, n_gpus=n_gpus)
        try:
            if kind == "flat":
                b = synth.human_shaped(n_loci=2000, total_fragments=800_000, seed=8)
                q.submit_flat(b)
                q.run(b["total_mapped_reads"])
            else:
                _raw_loci(q, 24, 500)
                q.upload()
                q.solve(1_000_000)
            out[n_gpus] = (q.bootstrap_counts(SEED, 3), q.bootstrap(SEED, 3, first=2))
        finally:
            q.close()
    (c1, r1), (c2, r2) = out[1], out[2]
    assert np.array_equal(c1, c2)
    for k in ("theta", "iters", "status"):
        assert np.array_equal(r1[k], r2[k]), k
    assert np.allclose(r1["tpm"], r2["tpm"], rtol=1e-12, atol=0)
