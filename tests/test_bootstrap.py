"""CPU: the restatement of the bootstrap resampler (tests/bootstrap_ref.py) - exactness of its integer arithmetic, the properties
DESIGN.md "Bootstrap replicates" states, and the statistics of a multinomial draw. tests/test_gpu_bootstrap.py holds the device to
this restatement bit for bit."""
import numpy as np

import bootstrap_ref as br
from strawberry_b200 import synth


def _batch(counts_per_locus):
    counts = np.concatenate([np.asarray(c, np.int32) for c in counts_per_locus]) if counts_per_locus else np.zeros(0, np.int32)
    lro = np.concatenate([[0], np.cumsum([len(c) for c in counts_per_locus])]).astype(np.int64)
    return dict(count=counts, loc_row_off=lro)


def _random_loci(seed, n_loci, max_rows=12, max_count=60):
    rng = np.random.default_rng(seed)
    loci = []
    for _ in range(n_loci):
        c = rng.integers(0, max_count, rng.integers(1, max_rows + 1))
        c[rng.random(len(c)) < 0.3] = 0
        loci.append(c)
    return loci


def test_umulhi64_equals_big_int_arithmetic():
    rng = np.random.default_rng(1)
    a = rng.integers(0, 2**64, 20000, dtype=np.uint64)
    b = np.concatenate([rng.integers(0, 2**64, 10000, dtype=np.uint64),            # N >= 2^32 included
                        rng.integers(0, 2**32, 10000, dtype=np.uint64)])
    edge = np.array([0, 1, 2**32 - 1, 2**32, 2**63, 2**64 - 1], np.uint64)
    a = np.concatenate([a, np.repeat(edge, len(edge))])
    b = np.concatenate([b, np.tile(edge, len(edge))])
    got = br.umulhi64(a, b)
    assert all(int(g) == (int(x) * int(y)) >> 64 for g, x, y in zip(got, a, b))


def test_numpy_restatement_equals_scalar_python_ints():
    loci = _random_loci(2, 40)
    b = _batch(loci)
    for seed, rep in ((0, 0), (7, 3), (2**64 - 1, 1000)):
        got = br.resample(b, seed, rep)
        ref = np.concatenate([br.resample_locus_scalar(c, seed, rep, l) for l, c in enumerate(loci)])
        assert np.array_equal(got, ref), (seed, rep)
    # caller-supplied hash positions (multi-GPU children)
    ids = [17, 3, 999]
    got = br.resample(_batch(loci[:3]), 5, 2, locus_ids=ids)
    ref = np.concatenate([br.resample_locus_scalar(loci[i], 5, 2, ids[i]) for i in range(3)])
    assert np.array_equal(got, ref)


def test_totals_kept_and_zero_rows_stay_zero():
    b = synth.human_shaped(n_loci=400, total_fragments=200_000, seed=9)
    lro = b["loc_row_off"]
    tot = np.add.reduceat(b["count"].astype(np.int64), lro[:-1])
    for rep in range(3):
        n = br.resample(b, 11, rep)
        assert np.array_equal(np.add.reduceat(n.astype(np.int64), lro[:-1]), tot)
        assert (n[b["count"] == 0] == 0).all()
        assert n.sum() == b["count"].sum()


def test_deterministic_and_differs_between_seeds_replicates_and_loci():
    b = synth.human_shaped(n_loci=200, total_fragments=100_000, seed=9)
    n0 = br.resample(b, 11, 0)
    assert np.array_equal(n0, br.resample(b, 11, 0))
    assert not np.array_equal(n0, br.resample(b, 12, 0))
    assert not np.array_equal(n0, br.resample(b, 11, 1))
    # the same counts at two positions draw differently
    same = _batch([[50, 30, 20], [50, 30, 20]])
    n = br.resample(same, 3, 0)
    assert not np.array_equal(n[:3], n[3:])
    # a locus depends on its own position only: alone under its id it gives the same counts as inside the batch
    alone = br.resample(_batch([b["count"][b["loc_row_off"][5]:b["loc_row_off"][6]]]), 11, 0, locus_ids=[5])
    assert np.array_equal(alone, n0[b["loc_row_off"][5]:b["loc_row_off"][6]])


def test_multinomial_moments_and_independence_of_consecutive_replicates():
    n_i = np.array([400, 250, 150, 100, 70, 30], np.int32)     # N = 1000
    N, R = int(n_i.sum()), 4000
    b = _batch([n_i])
    draws = np.stack([br.resample(b, 2024, r) for r in range(R)]).astype(np.float64)
    p = n_i / N
    var = N * p * (1 - p)
    mean = draws.mean(axis=0)
    assert (np.abs(mean - n_i) <= 4 * np.sqrt(var / R)).all(), mean - n_i
    assert (np.abs(draws.var(axis=0, ddof=1) / var - 1) < 0.10).all(), draws.var(axis=0, ddof=1) / var
    for i in range(len(n_i)):
        assert abs(np.corrcoef(draws[:-1, i], draws[1:, i])[0, 1]) < 0.05, i
