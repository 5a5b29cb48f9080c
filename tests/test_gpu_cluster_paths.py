"""Every path of em_cluster_kernel against the oracle, at shapes that reach it (tests/cluster_paths.py says which CTA takes which
path; tests/test_cluster_paths.py checks that these shapes reach every listed cell): one batch of the cell loci under the planner's
own cluster sizes, and one batch per forced cluster size for the cells only forcing reaches. Besides parity at convergence: the
launch records match the restated plan, a locus gives the same bits alone as inside its batch and when solved again, and a few
EM steps with the iteration cap binding match a long-double restatement of the oracle far more tightly than the parity bar."""
from collections import Counter

import numpy as np
import pytest

import cluster_paths as cp
from util import assert_matches_oracle

pytestmark = pytest.mark.gpu

CAPPED_ITERS = (1, 2, 5)


@pytest.fixture(scope="module")
def q(sbq_lib_path):
    from strawberry_b200 import api
    qq = api.Quantifier()
    yield qq
    qq.close()


@pytest.fixture(scope="module")
def cells():
    return cp.cell_batches()


def solve(q, b, force, **cfg):
    """All loci through the cluster tier (tier 2 forced), cluster size the planner's (force = 0) or forced."""
    from strawberry_b200 import api
    qq = q if not cfg else api.Quantifier(**cfg)
    try:
        qq.clear()
        qq.set_plan(2, force)
        qq.submit_flat(b)
        qq.validate()
        qq.run(b["total_mapped_reads"])
        res = qq.results()
        res["stats"] = qq.stats()
        res["launches"] = [r for r in qq.launch_stats() if r["kernel"] == "em_cluster_kernel" and r["n_loci"]]
        return res
    finally:
        if cfg:
            qq.close()


def capped_worst(res, b, max_iter):
    """Statuses and iteration counts equal to the long-double restatement's; -> worst theta ratio against it."""
    ld = cp.batch_em_longdouble(b, max_iter=max_iter)
    assert np.array_equal(res["status"], ld["status"]), (max_iter, res["status"], ld["status"])
    assert np.array_equal(res["iters"], ld["iters"]), (max_iter, res["iters"], ld["iters"])
    return cp.theta_close_ld(res["theta"], ld["theta"], b, cp.CAPPED_REL)[1]


@pytest.mark.parametrize("force", [0, 4, 16])
def test_cell_batch_matches_the_oracle_and_the_plan(q, oracle_mod, cells, force):
    b, loci = cells[force]
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=4)
    res = solve(q, b, force)
    assert_matches_oracle(res, ora, b, f"cluster paths, force {force}")
    assert res["stats"]["loci_cta"] == len(loci)
    want = Counter(cp.plan(int(lb["loc_iso_off"][1]), len(lb["count"]), int(lb["row_ptr"][-1]), force) for lb in loci)
    got = Counter()
    for r in res["launches"]:
        got[(r["cluster_size"], r["threads"])] += r["n_loci"]
    assert got == want, (got, want)


@pytest.mark.parametrize("force", [0, 4, 16])
def test_cell_loci_are_bitwise_stable(q, cells, force):
    """Each locus alone gives the bits it gets inside its batch (theta, iterations, status), and the resident batch solved again
    gives the same bits again."""
    b, loci = cells[force]
    res = solve(q, b, force)
    q.solve(b["total_mapped_reads"])
    q.finalize_tpm(q.fpkm_sum())
    q.download()
    again = q.results()
    for k in ("theta", "iters", "status"):
        assert np.array_equal(np.asarray(res[k]).view(np.uint8), np.asarray(again[k]).view(np.uint8)), k
    iso = b["loc_iso_off"]
    for l, one in enumerate(loci):
        alone = solve(q, one, force)
        assert np.array_equal(res["theta"][iso[l]:iso[l + 1]].view(np.uint64), alone["theta"].view(np.uint64)), l
        assert res["iters"][l] == alone["iters"][0] and res["status"][l] == alone["status"][0], l


@pytest.mark.parametrize("force", [0, 4, 16])
def test_capped_solves_match_the_longdouble_restatement(cells, force):
    """max_iter 1, 2 and 5 (the cap binds on almost every locus): theta within cp.CAPPED_REL = 1e-12 of em_csr_longdouble, with the
    parity floor of util.theta_close; statuses and iteration counts equal. Worst ratio measured on a B200 (1000 W): 1.3e-15."""
    b, _ = cells[force]
    for m in CAPPED_ITERS:
        res = solve(None, b, force, max_iter=m)
        worst = capped_worst(res, b, m)
        print(f"capped worst ratio: cells force {force} max_iter {m}: {worst:.3e}")
        assert worst <= cp.CAPPED_REL, (m, worst)


def test_capped_check_catches_a_row_weighted_off_by_1e6(q, oracle_mod, cells):
    """Negative control: one row of the T = 100 locus (20 rows of 3; 64-thread CTA, generic M-pass) has its alpha scaled by
    1 + 1e-6 in the GPU's input only. Scaling a whole row leaves its first-pass responsibilities unchanged, so max_iter 1 cannot see it;
    from the second step on the column sums s_j move, and the capped check must fail. Measured on a B200 (1000 W): worst ratio
    4.2e-16 at max_iter 1, 5.9e-9 at 2 and 5.6e-9 at 5 (the bar is 1e-12); the converged check at the 1e-6 parity bar does NOT
    notice the perturbed row (statuses, iterations and theta all pass it). Which of the two happens is printed."""
    b, loci = cells[0]
    l = [int(lb["loc_iso_off"][1]) for lb in loci].index(100)
    r0 = int(b["loc_row_off"][l])
    k0, k1 = int(b["row_ptr"][r0]), int(b["row_ptr"][r0 + 1])
    bad = dict(b)
    bad["alpha"] = b["alpha"].copy()
    bad["alpha"][k0:k1] *= 1.0 + 1e-6
    caught = []
    for m in CAPPED_ITERS:
        res = solve(None, bad, 0, max_iter=m)
        worst = capped_worst(res, b, m)
        print(f"negative control: max_iter {m}: worst ratio {worst:.3e}")
        caught.append(worst > cp.CAPPED_REL)
    assert caught[1] and caught[2], caught
    ora = oracle_mod.quantify_batch(b, b["total_mapped_reads"], n_threads=4)
    res = solve(q, bad, 0)
    try:
        assert_matches_oracle(res, ora, b, "perturbed row, converged")
        print("negative control: the converged 1e-6 check does NOT notice the perturbed row")
    except AssertionError as e:
        print(f"negative control: the converged 1e-6 check notices the perturbed row: {e}")
