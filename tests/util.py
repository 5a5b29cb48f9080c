"""Shared helpers for the parity tests."""
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FLAT_KEYS = ("loc_row_off", "loc_iso_off", "row_ptr", "col", "alpha", "count", "iso_len")

# Parity bar of BASELINE.json north_star: abundances within 1e-6 relative. theta_j that the EM has
# driven to (numerically) nothing are compared on an absolute floor tied to the locus mass instead:
# |d| <= REL_TOL * max(|ref|, ABS_FLOOR_FRAC * total_count).
REL_TOL = 1e-6
ABS_FLOOR_FRAC = 1e-9


def load_golden():
    z = np.load(os.path.join(GOLDEN_DIR, "em_golden.npz"))
    b = {k: z[k] for k in FLAT_KEYS}
    b["total_mapped_reads"] = int(z["total_mapped_reads"])
    return b, z["theta_ref"], z["rc_ref"], z["iters"], z["status"]


def locus_totals(batch):
    lro = batch["loc_row_off"]
    cs = np.concatenate([[0], np.cumsum(batch["count"], dtype=np.int64)])
    return cs[lro[1:]] - cs[lro[:-1]]


def theta_close(got, ref, batch, rel=REL_TOL):
    """Per-isoform closeness under the parity bar; returns (ok_mask, worst_ratio)."""
    tot = np.repeat(locus_totals(batch).astype(np.float64), np.diff(batch["loc_iso_off"]))
    scale = np.maximum(np.abs(ref), ABS_FLOOR_FRAC * np.maximum(tot, 1.0))
    ratio = np.abs(got - ref) / scale
    return ratio <= rel, float(ratio.max()) if len(ratio) else 0.0


def expand_loci(per_locus, batch):
    return np.repeat(per_locus, np.diff(batch["loc_iso_off"]))


def assert_matches_oracle(res, ora, batch, what="", rel=REL_TOL):
    """CUDA results vs oracle results on the same batch: statuses and iteration counts equal,
    theta / fpkm / frac / tpm within the parity bar (rel), keep flags equal."""
    bad_st = np.nonzero(res["status"] != ora["status"])[0]
    assert len(bad_st) == 0, f"{what}: status differs at loci {bad_st[:10]}: {res['status'][bad_st[:10]]} vs {ora['status'][bad_st[:10]]}"
    bad_it = np.nonzero(res["iters"] != ora["iters"])[0]
    assert len(bad_it) == 0, f"{what}: iteration count differs at loci {bad_it[:10]}: {res['iters'][bad_it[:10]]} vs {ora['iters'][bad_it[:10]]}"
    ok, worst = theta_close(res["theta"], ora["theta"], batch, rel)
    assert ok.all(), f"{what}: theta off at {np.nonzero(~ok)[0][:10]}, worst ratio {worst:.3e}"
    live = expand_loci(ora["status"], batch) != 3
    for k in ("fpkm", "frac", "tpm"):
        a, b = res[k][live], ora[k][live]
        fin = np.isfinite(b)
        assert np.array_equal(np.isfinite(a), fin), f"{what}: {k} finiteness differs"
        scale = np.maximum(np.abs(b[fin]), 1e-9 * max(float(np.nanmax(np.abs(b[fin]))) if fin.any() else 1.0, 1e-300))
        r = np.abs(a[fin] - b[fin]) / scale
        assert (r <= rel).all(), f"{what}: {k} worst ratio {r.max():.3e}"
    assert np.array_equal(res["keep"] != 0, ora["keep"] != 0), f"{what}: keep flags differ"
    return worst
