"""GPU: Gibbs posterior samples (sbq_gibbs, strawberry_b200/csrc/sbq_gibbs.cuh, DESIGN.md "Gibbs posterior samples").

Every sample's theta equals the CPU restatement (tests/gibbs_ref.py) bit for bit, its status is the point estimate's, its TPM
agrees to 1e-12; on the golden, headline-shaped, raw-built, heavy-row and giant-tier batches. Also: a locus alone equals the same
locus in a batch, two calls agree, the point estimate and a later bootstrap are untouched, the refusals, two GPUs against one,
and negative controls (seed + 1, one fragment more) that the bitwise check does catch."""
import numpy as np
import pytest

import gibbs_ref as gr
from strawberry_b200 import synth
from util import load_golden

pytestmark = pytest.mark.gpu

SEED = 20261022


@pytest.fixture(scope="module")
def api_mod(sbq_lib_path):
    from strawberry_b200 import api
    return api


def solve(api_mod, batch, **cfg):
    q = api_mod.Quantifier(**cfg)
    q.submit_flat(batch)
    q.run(batch["total_mapped_reads"])
    return q


def gibbs_of(q, n=3, thin=2, burn_in=2, prior=0.01, seed=SEED):
    return q.gibbs(seed, n, thin=thin, burn_in=burn_in, prior=prior)


def reference(batch, point, n=3, thin=2, burn_in=2, prior=0.01, seed=SEED, **epi):
    return gr.samples(batch, point["theta"], point["status"], seed, n, thin, burn_in, prior, batch["total_mapped_reads"], **epi)


def assert_samples_equal(got, ref, what=""):
    assert np.array_equal(got["status"], ref["status"]), what
    bad = got["theta"] != ref["theta"]
    assert not bad.any(), (what, int(bad.sum()), np.argwhere(bad)[:5])
    assert np.allclose(got["tpm"], ref["tpm"], rtol=1e-12, atol=1e-300), what


def check(api_mod, batch, what, **kw):
    q = solve(api_mod, batch)
    try:
        point = q.results()
        got = gibbs_of(q, **kw)
        st = q.gibbs_stats()
    finally:
        q.close()
    assert_samples_equal(got, reference(batch, point, **kw), what)
    return got, st


def _raw_batch(api_mod):
    """12 random loci (tests/locusgen.py) submitted raw: the device builds their class tables"""
    import locusgen
    from strawberry_b200 import builder
    q = api_mod.Quantifier()
    s, done, rl0 = 300, 0, None
    while done < 12:
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
    q.upload()
    b = q.fetch_batch()
    b["total_mapped_reads"] = 1_000_000
    return q, b


def _heavy_batch():
    """a small human-shaped batch plus one locus whose first row holds 150 000 fragments (gibbs_heavy_kernel)"""
    rng = np.random.default_rng(9)
    T, R = 6, 40
    rows = [np.sort(rng.choice(T, size=rng.integers(1, T + 1), replace=False)) for _ in range(R)]
    rp = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    cnt = rng.integers(0, 30, R).astype(np.int32)
    cnt[0], cnt[5] = 150_000, 9
    heavy = dict(loc_row_off=np.array([0, R], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=rp,
                 col=np.concatenate(rows).astype(np.int32), alpha=rng.uniform(1e-4, 1e-2, int(rp[-1])), count=cnt,
                 iso_len=rng.integers(500, 5000, T).astype(np.int32), total_mapped_reads=int(cnt.sum()))
    b = synth.concat([heavy, synth.human_shaped(n_loci=200, total_fragments=100_000, seed=12, max_rows=300)])
    b["total_mapped_reads"] = int(b["count"].sum())
    return b


# ---- bitwise against the restatement ----------------------------------------------------------------------------------------

def test_golden_batch(api_mod):
    b, *_ = load_golden()
    check(api_mod, b, "golden")


def test_human_shaped_batch(api_mod):
    b = synth.human_shaped(n_loci=2000, total_fragments=800_000, seed=8)
    _, st = check(api_mod, b, "human_shaped 2000", n=4, thin=3, burn_in=1)
    assert st["n"] == 4 and st["rounds"] == 13
    assert 0 < st["colsum_ms"] and 0 < st["assign_ms"] and 0 < st["theta_ms"] and st["assign_ms"] + st["theta_ms"] <= st["total_ms"]


def test_raw_built_batch(api_mod):
    q, b = _raw_batch(api_mod)
    try:
        q.solve(b["total_mapped_reads"])
        q.finalize_tpm(q.fpkm_sum())
        q.download()
        point = q.results()
        got = gibbs_of(q)
    finally:
        q.close()
    assert b["count"].sum() > 0
    assert_samples_equal(got, reference(b, point), "raw")


def test_heavy_row(api_mod):
    b = _heavy_batch()
    got, _ = check(api_mod, b, "heavy row", n=2, thin=2, burn_in=1, prior=0.5)
    assert got["theta"][:, :6].sum(1) == pytest.approx(b["count"][:40].sum(), rel=1e-12)


@pytest.mark.parametrize("locus,rows", [(1, 10_000), (3, 40_000)])
def test_giant_locus_on_the_grid_tier(api_mod, locus, rows):
    """a device-generated giant locus (>= 300 k non-zeros): the grid tier's layout pass reorders its rows in place, the
    sampler reads them in submitted order"""
    b = synth.giant_device([locus], rows)
    assert int(b["row_ptr"][-1]) >= 300_000
    q = api_mod.Quantifier()
    try:
        q.synth_giant([locus], rows)
        q.solve(b["total_mapped_reads"])
        q.finalize_tpm(q.fpkm_sum())
        q.download()
        assert any(x["kernel"].startswith("em_grid") for x in q.launch_stats())
        point = q.results()
        got = gibbs_of(q, n=2, thin=2, burn_in=1)
    finally:
        q.close()
    assert_samples_equal(got, reference(b, point, n=2, thin=2, burn_in=1), f"giant {locus}")


def test_effective_length_epilogue(api_mod):
    b = synth.human_shaped(n_loci=400, total_fragments=200_000, seed=41, max_rows=300)
    b["iso_len"] = b["iso_len"].copy()
    b["iso_len"][::17] = 150
    cfg = dict(min_iso_frac=0.01, effective_len_norm=1, insert_mean=200.0)
    q = solve(api_mod, b, **cfg)
    try:
        point = q.results()
        got = gibbs_of(q)
    finally:
        q.close()
    assert_samples_equal(got, reference(b, point, min_iso_frac=0.01, effective_len_norm=1, insert_mean=200.0), "epilogue")


# ---- independence of batch mates, repeatability, the point estimate ---------------------------------------------------------

def test_a_locus_alone_equals_the_locus_in_a_batch(api_mod):
    b = synth.human_shaped(n_loci=600, total_fragments=300_000, seed=13, max_rows=400)
    big = int(np.argmax(np.diff(b["row_ptr"][b["loc_row_off"]])))
    order = [big] + [l for l in range(600) if l != big]          # the locus at submit position 0 in both batches
    parts = [synth.locus_slice(b, l) for l in order]
    q = api_mod.Quantifier()
    try:
        q.submit(parts)
        q.run(b["total_mapped_reads"])
        many = gibbs_of(q)
        q.clear()
        q.submit(parts[:1])
        q.run(b["total_mapped_reads"])
        one = gibbs_of(q)
    finally:
        q.close()
    T = parts[0][0]
    assert np.array_equal(one["theta"], many["theta"][:, :T])
    assert np.array_equal(one["status"][:, 0], many["status"][:, 0])


def test_two_calls_give_the_same_bits_and_the_point_estimate_is_untouched(api_mod):
    b = synth.human_shaped(n_loci=1500, total_fragments=600_000, seed=6)
    q = solve(api_mod, b)
    try:
        before, stats = q.results(), q.stats()
        boot_ref = q.bootstrap(SEED, 2)
        g1 = gibbs_of(q)
        g2 = gibbs_of(q)
        after = q.results()
        assert q.stats() == stats
        boot = q.bootstrap(SEED, 2)
        q.solve(b["total_mapped_reads"])
        q.finalize_tpm(q.fpkm_sum())
        q.download()
        resolved = q.results()
    finally:
        q.close()
    for k in g1:
        assert np.array_equal(g1[k], g2[k]), k
    for k in before:
        assert np.array_equal(before[k], after[k]), k
        assert np.array_equal(before[k], resolved[k]), k
    for k in boot:
        assert np.array_equal(boot[k], boot_ref[k]), k


# ---- refusals -----------------------------------------------------------------------------------------------------------------

def test_refusals(api_mod):
    b = synth.human_shaped(n_loci=300, total_fragments=100_000, seed=7)
    q = api_mod.Quantifier()
    try:
        with pytest.raises(api_mod.SbqError) as e:
            q.gibbs(SEED, 1)                              # nothing resident
        assert e.value.code == api_mod.SBQ_ERR_STATE
        q.submit_flat(b)
        q.upload()
        with pytest.raises(api_mod.SbqError) as e:
            q.gibbs(SEED, 1)                              # resident but not solved
        assert e.value.code == api_mod.SBQ_ERR_STATE
        with pytest.raises(api_mod.SbqError) as e:
            q.gibbs_stats()
        assert e.value.code == api_mod.SBQ_ERR_STATE
        q.solve(b["total_mapped_reads"])
        q.finalize_tpm(q.fpkm_sum())
        q.download()
        point = q.results()
        for kw in (dict(n=0), dict(n=-1), dict(thin=0), dict(burn_in=-1), dict(prior=0.0), dict(prior=-1.0), dict(prior=float("nan")),
                   dict(prior=float("inf"))):
            args = dict(n=1, thin=1, burn_in=0, prior=0.5)
            args.update(kw)
            with pytest.raises(api_mod.SbqError) as e:
                q.gibbs(SEED, args["n"], thin=args["thin"], burn_in=args["burn_in"], prior=args["prior"])
            assert e.value.code == api_mod.SBQ_ERR_INVALID, kw
        with pytest.raises(api_mod.SbqError) as e:
            q.gibbs(SEED, 2**31 - 1, thin=1, burn_in=0)   # ~2 PB of sample matrices: a plain failed allocation
        assert e.value.code == api_mod.SBQ_ERR_NOMEM
        got = gibbs_of(q)                                 # the context stays usable
    finally:
        q.close()
    assert_samples_equal(got, reference(b, point), "after refusals")
    qb = api_mod.Quantifier(bias_mode=1)
    try:
        with pytest.raises(api_mod.SbqError) as e:
            qb.gibbs(SEED, 1)
        assert e.value.code == api_mod.SBQ_ERR_UNSUPPORTED
    finally:
        qb.close()


# ---- negative controls ---------------------------------------------------------------------------------------------------------

def test_negative_controls_fail_the_bitwise_check(api_mod):
    b = synth.human_shaped(n_loci=500, total_fragments=200_000, seed=14, max_rows=300)
    q = solve(api_mod, b)
    try:
        point = q.results()
        got = gibbs_of(q)
    finally:
        q.close()
    with pytest.raises(AssertionError):
        assert_samples_equal(got, reference(b, point, seed=SEED + 1))
    # theta depends on the weights only through the integer class counts, so a last-bit change of one weight rarely moves a draw;
    # one fragment more in the heaviest row changes the draws of every later row of its locus
    more = dict(b)
    more["count"] = b["count"].copy()
    more["count"][int(np.argmax(b["count"]))] += 1
    with pytest.raises(AssertionError):
        assert_samples_equal(got, reference(more, point))


# ---- multi-GPU ------------------------------------------------------------------------------------------------------------------

def test_two_gpus_equal_one(api_mod):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    b = synth.human_shaped(n_loci=2000, total_fragments=800_000, seed=8)
    out = {}
    for n_gpus in (1, 2):
        q = api_mod.Quantifier(device=0, n_gpus=n_gpus)
        try:
            q.submit_flat(b)
            q.run(b["total_mapped_reads"])
            out[n_gpus] = gibbs_of(q)
        finally:
            q.close()
    for k in ("theta", "status"):
        assert np.array_equal(out[1][k], out[2][k]), k
    assert np.allclose(out[1]["tpm"], out[2]["tpm"], rtol=1e-12, atol=0)
