"""CPU checks of tests/cluster_paths.py: the restatement of the cluster kernel's path choice equals the header's own host-callable
functions (cluster_cta_path included), the shapes of tests/test_gpu_cluster_paths.py reach every path listed below, the kernel is
launched with exactly the planner's thread counts, and the long-double EM restatement agrees with the oracle."""
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

import cluster_paths as cp
from util import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "strawberry_b200", "csrc")

# Every (CS, NT, exchange, slice, E-pass, M-pass) cell the GPU test's shapes must reach: the paths no other test runs. Written out so
# that a threshold or layout change that moves a shape off its cell fails here, by name, instead of silently testing something else.
REQUIRED_CELLS = {
    (1, 64, "single", "csc_smem", "row_slots", "generic"),        # generic M-pass in a 64-thread CTA
    (1, 128, "single", "csc_smem", "row_slots", "generic"),       # ... and in a 128-thread CTA
    (8, 512, "owner", "csc_partial", "rows4", "col_slots"),       # four rows per thread at CS 8, part of the CSC index in L2
    (16, 512, "owner", "csc_smem", "rows4", "col_slots"),         # four rows per thread at CS 16
    (16, 512, "owner", "csc_partial", "rows4", "col_slots"),
    (4, 512, "owner", "csc_partial", "row_slots", "generic"),     # generic M-pass at CS 4 and 8, partial CSC index
    (8, 512, "owner", "csc_partial", "row_slots", "generic"),
    (4, 512, "owner", "stream", "stream", "stream"),              # streaming at CS 4
    (4, 512, "owner", "csc_smem", "row_slots", "col_slots"),      # (the resident half of the mixed cluster below)
    (4, 512, "a2a", "csc_smem", "row_slots", "generic"),          # generic M-pass under all-to-all (forced CS 4)
    (16, 512, "owner", "csc_smem", "row_slots", "col_slots"),     # owner form with CTAs that have no rows (forced CS 16)
}
# Whole-cluster situations: (forced CS, CS, what)
REQUIRED_LOCUS_FEATURES = {
    (0, 4, "mixed slice"),            # one cluster, some CTAs resident and some streaming
    (0, 16, "owner, idle columns"),   # owner form where some CTAs own no column
    (16, 16, "owner, no rows"),       # owner form with CTAs that have no rows
    (0, 1, "CSC index in L2"),        # a resident slice with all or almost all of its CSC index in L2 (n_ent_s < 64) ...
    (0, 2, "CSC index in L2"),        # ... n_ent_s = 0 here
}


def locus_features(paths):
    f = set()
    if len({p["slice"] == "stream" for p in paths}) > 1:
        f.add("mixed slice")
    if paths[0]["exchange"] == "owner" and any(p["owned"] == 0 for p in paths):
        f.add("owner, idle columns")
    if paths[0]["exchange"] == "owner" and any(p["nrows"] == 0 for p in paths):
        f.add("owner, no rows")
    if any(p["slice"] == "csc_partial" and p["n_ent_s"] < 64 for p in paths):
        f.add("CSC index in L2")
    return f


@pytest.fixture(scope="module")
def cell_batches():
    return cp.cell_batches()


def test_shape_set_reaches_every_required_cell(cell_batches):
    cells, feats = set(), set()
    for force, (b, loci) in cell_batches.items():
        cells |= cp.batch_cells(b, force)
        for lb in loci:
            paths = cp.cta_paths(int(lb["loc_iso_off"][1]), lb["row_ptr"], force)
            feats |= {(force, paths[0]["CS"], f) for f in locus_features(paths)}
    assert REQUIRED_CELLS <= cells, sorted(REQUIRED_CELLS - cells)
    assert REQUIRED_LOCUS_FEATURES <= feats, sorted(REQUIRED_LOCUS_FEATURES - feats)


def test_mixed_cluster_split(cell_batches):
    """The locus of 400 rows of 64 and 25 600 rows of 1 at CS 4: the nnz split gives CTAs 0 - 1 the long rows (resident) and CTAs
    2 - 3 12 800 one-entry rows each, whose slice is far beyond the 12 % slack of the estimate (streaming)."""
    b, loci = cell_batches[0]
    lb = next(x for x in loci if int(x["loc_iso_off"][1]) == 64)
    paths = cp.cta_paths(64, lb["row_ptr"])
    assert [p["slice"] for p in paths] == ["csc_smem", "csc_smem", "stream", "stream"]
    assert [p["nrows"] for p in paths] == [200, 200, 12800, 12800]
    assert all(p["G"] > 0 for p in paths[2:])


def test_resident_slices_with_the_csc_index_in_l2(cell_batches):
    """Within a few bytes of the shared-memory cap of the locus, a resident slice keeps (almost) none of its CSC index in shared
    memory: 110 rows of 100 + 8 621 rows of 1 at CS 2 (CTA 1: n_ent_s = 0), 100 rows of 32 + 7 881 rows of 1 at CS 1 (n_ent_s = 1)."""
    _, loci = cell_batches[0]
    two = cp.cta_paths(100, loci[-2]["row_ptr"])
    assert [(q["slice"], q["n_ent_s"]) for q in two] == [("csc_smem", 9900), ("csc_partial", 0)]
    one = cp.cta_paths(32, loci[-1]["row_ptr"])
    assert [(q["slice"], q["n_ent_s"], q["nnz_c"]) for q in one] == [("csc_partial", 1, 11081)]


_SHIM = r"""
#include <cstdio>
#include <cstring>
#include "sbq_kernels.cuh"
using namespace sbq;
int main(int argc, char** argv) {
   if (argc > 1 && !strcmp(argv[1], "path")) {       // cluster_cta_path
      int T, cs, nt, nrows, too_long;
      unsigned nnz_c, smem_launch;
      size_t slice_est;
      while (scanf("%d %d %d %d %u %d %zu %u", &T, &cs, &nt, &nrows, &nnz_c, &too_long, &slice_est, &smem_launch) == 8) {
         const ClusterCtaPath c = cluster_cta_path(T, cs, nt, nrows, nnz_c, too_long != 0, slice_est, smem_launch);
         printf("%d %d %u %d %d %d %d %d\n", (int)c.resident, (int)c.csc_in_smem, c.n_ent_s, c.G, (int)c.row_slots, (int)c.col_slots,
                (int)c.a2a, c.B);
      }
      return 0;
   }
   int T, cs, nt;
   long long R, nnz, smem;
   while (scanf("%d %lld %lld %d %d %lld", &T, &R, &nnz, &cs, &nt, &smem) == 6) {
      const size_t sl = cluster_slice_estimate(nnz, R, T, cs);
      const size_t cls = cluster_class_smem(T, sl, nt, cs);
      printf("%zu %d %zu %zu %d %d %zu %zu\n", sl, (int)cluster_a2a(T, cs, sl), cluster_fixed_doubles(T, cs, sl), cls,
             cluster_stream_groups(T, cls, nt, cs, sl), cluster_stream_groups(T, (size_t)smem, nt, cs, sl),
             cluster_resident_bytes((size_t)(nnz / cs), (size_t)(R / cs), T), cluster_resident_csr_bytes((size_t)(nnz / cs), (size_t)(R / cs), T));
   }
   return 0;
}
"""


def _nvcc():
    n = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    return n if os.path.exists(n) else shutil.which("nvcc")


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    """The header's host-callable functions compiled host-only: run(mode args, input text) -> output lines."""
    nvcc = _nvcc()
    if not nvcc:
        pytest.skip("nvcc not found")
    d = tmp_path_factory.mktemp("shim")
    (d / "shim.cu").write_text(_SHIM)
    exe = str(d / "shim")
    subprocess.check_call([nvcc, "-arch=sm_100a", "-std=c++17", "-O1", "-I", CSRC, "-o", exe, str(d / "shim.cu")])
    return lambda args, inp: [o for o in subprocess.run([exe, *args], input=inp, capture_output=True, text=True, check=True).stdout.split("\n") if o]


def test_restatement_equals_the_header(shim):
    """20 000 random (T, R, nnz, CS, NT) through the header's host-callable functions (compiled host-only) and through the restatement."""
    rng = np.random.default_rng(12345)
    n = 20_000
    T = np.minimum(3600, np.exp(rng.uniform(0, np.log(3600), n)).astype(np.int64))
    R = np.exp(rng.uniform(0, np.log(300_000), n)).astype(np.int64) + 1
    nnz = np.minimum(R * T, (R * np.exp(rng.uniform(0, np.log(200), n))).astype(np.int64))
    cs = rng.choice([1, 2, 4, 8, 16], n)
    nt = rng.choice([64, 128, 256, 512], n)
    smem = rng.integers(0, cp.CL_SMEM_CAP + 1, n)
    inp = "\n".join(f"{a} {b} {c} {d} {e} {f}" for a, b, c, d, e, f in zip(T, R, nnz, cs, nt, smem)) + "\n"
    out = shim([], inp)
    assert len(out) == n
    for i in range(n):
        t, r, z, c, m = int(T[i]), int(R[i]), int(nnz[i]), int(cs[i]), int(nt[i])
        sl = cp.cluster_slice_estimate(z, r, t, c)
        cls = cp.cluster_class_smem(t, sl, m, c)
        want = [sl, int(cp.cluster_a2a(t, c, sl)), cp.cluster_fixed_doubles(t, c, sl), cls, cp.cluster_stream_groups(t, cls, m, c, sl),
                cp.cluster_stream_groups(t, int(smem[i]), m, c, sl), cp.cluster_resident_bytes(z // c, r // c, t),
                cp.cluster_resident_csr_bytes(z // c, r // c, t)]
        assert [int(x) for x in out[i].split()] == want, (t, r, z, c, m, int(smem[i]))


_PATH_FIELDS = ("resident", "csc_in_smem", "n_ent_s", "G", "row_slots", "col_slots", "a2a", "B")


def test_cta_path_equals_the_kernel_function(shim):
    """40 000 random CTAs through cluster_cta_path - the function em_cluster_kernel calls to pick a CTA's path - and through
    cp.cta_path, field by field: every CS and NT, rows and non-zeros of the CTA up to and beyond the 16-bit limit of the resident
    index, too_long both ways, and launch shared memory anywhere from 0 to the cap."""
    rng = np.random.default_rng(2027)
    n = 40_000
    T = np.minimum(3600, np.exp(rng.uniform(0, np.log(3600), n)).astype(np.int64))
    cs = rng.choice([1, 2, 4, 8, 16], n)
    nt = rng.choice([64, 128, 512], n)
    R = np.exp(rng.uniform(0, np.log(400_000), n)).astype(np.int64) + 1
    nnz = np.minimum(R * T, (R * np.exp(rng.uniform(0, np.log(100), n))).astype(np.int64))
    slice_est = [cp.cluster_slice_estimate(int(z), int(r), int(t), int(c)) for z, r, t, c in zip(nnz, R, T, cs)]
    # the CTA's share of the locus, from a tenth to three times an even share (the row split is by non-zeros), some with no rows
    f = np.exp(rng.uniform(np.log(0.1), np.log(3.0), n))
    nrows = np.where(rng.random(n) < 0.02, 0, np.maximum(1, (R / cs * f).astype(np.int64)))
    nnz_c = np.where(nrows == 0, 0, np.maximum(nrows, (nnz / cs * f).astype(np.int64)))
    too_long = rng.random(n) < 0.1
    smem = rng.integers(0, cp.CL_SMEM_CAP + 1, n)
    rows = list(zip(T, cs, nt, nrows, nnz_c, too_long.astype(int), slice_est, smem))
    out = shim(["path"], "\n".join(" ".join(str(int(x)) for x in r) for r in rows) + "\n")
    assert len(out) == n
    seen = set()
    for i, (t, c, m, nr, z, tl, sl, sm) in enumerate(rows):
        want = cp.cta_path(int(t), int(c), int(m), int(nr), int(z), bool(tl), int(sl), int(sm))
        got = [int(x) for x in out[i].split()]
        assert got == [int(want[k]) for k in _PATH_FIELDS], (rows[i], dict(zip(_PATH_FIELDS, got)), want)
        seen.add("stream" if not want["resident"] else "csc_smem" if want["csc_in_smem"] else
                 "csc_partial, clamped" if want["n_ent_s"] < z else "csc_partial")
        seen.add(("row_slots", want["row_slots"]))
        seen.add(("col_slots", want["col_slots"]))
        seen.add(("a2a", want["a2a"]))
        if z + t > 65535 or nr > 65535:
            seen.add("index over 16 bits")
    assert seen >= {"stream", "csc_smem", "csc_partial, clamped", "index over 16 bits", ("row_slots", True), ("row_slots", False),
                    ("col_slots", True), ("col_slots", False), ("a2a", True), ("a2a", False)}, seen


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def test_restated_planner_and_header_constants_match_the_source():
    """cluster_size_for, smem_bucket / BUCKET_NT (sbq.cu) and the header constants are restated by value: a change there fails here."""
    cu, hdr = _src("sbq.cu"), _src("sbq_kernels.cuh")
    m = re.search(r"const int BUCKET_NT\[N_BUCKETS\] = \{([^}]*)\};", cu)
    assert tuple(int(x) for x in m.group(1).split(",")) == cp.BUCKET_NT
    m = re.search(r"int smem_bucket\(size_t bytes\) \{ return ([^;]*);", cu)
    assert tuple(int(a) * int(b) for a, b in re.findall(r"bytes <= (\d+) \* (\d+)", m.group(1))) == cp.SMEM_BUCKET_BOUNDS
    m = re.search(r"int cluster_size_for\(int64_t nnz\) \{(.*?)\n\}", cu, re.S)
    assert re.findall(r"if \(nnz <= (\d+) \* 1024\) return (\d+);", m.group(1)) == \
        [(str(b // 1024), str(c)) for b, c in zip(cp.CLUSTER_NNZ_BOUNDS, (1, 2, 4, 8))]
    assert "return 16;" in m.group(1)
    for name, val in (("CL_NT", cp.CL_NT), ("CL_LPR_STREAM", cp.CL_LPR_STREAM), ("CL_A2A_MAX", cp.CL_A2A_MAX)):
        assert re.search(rf"constexpr int {name} = (\d+);", hdr).group(1) == str(val), name
    assert "constexpr size_t CL_SMEM_CAP = 220 * 1024;" in hdr and cp.CL_SMEM_CAP == 220 * 1024


def test_launch_arms_are_the_bucket_thread_counts():
    """sbq.cu launches em_cluster_kernel through one arm per thread count: exactly the values of BUCKET_NT, each arm taken for the
    thread count it instantiates."""
    cu = _src("sbq.cu")
    m = re.search(r"int rc = (lc\.nt == .*?);\n", cu, re.S)
    arms = re.findall(r"lc\.nt == (\d+) \? launch_cluster_class_nt<(\d+)>\(c, lc, ss\)", m.group(1))
    assert arms and all(a == b for a, b in arms), arms
    last = re.findall(r":\s*launch_cluster_class_nt<(\d+)>\(c, lc, ss\)$", m.group(1))
    assert sorted({int(a) for a, _ in arms} | {int(x) for x in last}) == sorted(set(cp.BUCKET_NT)), m.group(1)
    assert len(re.findall(r"launch_cluster_class_nt<", cu)) == len(set(cp.BUCKET_NT)), "a launch arm outside the dispatch"


def test_streaming_always_has_a_group():
    """A CTA that streams needs at least one accumulator group (G = 0 would skip its rows): for every T up to SBQ_MAX_ISO and
    every cluster size and thread count the class shared memory leaves room for one."""
    for T in range(1, 3601, 7):
        for cs in (1, 2, 4, 8, 16):
            for nt in set(cp.BUCKET_NT):
                for nnz, R in ((T, 1), (1 << 16, 1 << 14), (1 << 20, 1 << 18)):
                    sl = cp.cluster_slice_estimate(nnz, R, T, cs)
                    assert cp.cluster_stream_groups(T, cp.cluster_class_smem(T, sl, nt, cs), nt, cs, sl) >= 1, (T, cs, nt)


def _oracle_batch(oracle_mod, b, **kw):
    lro, lio, rp = b["loc_row_off"], b["loc_iso_off"], b["row_ptr"]
    L = len(lro) - 1
    st, it = np.zeros(L, np.int32), np.zeros(L, np.int32)
    th = np.zeros(int(lio[-1]))
    for l in range(L):
        r0, r1 = int(lro[l]), int(lro[l + 1])
        k0, k1 = int(rp[r0]), int(rp[r1])
        st[l], th[lio[l]:lio[l + 1]], it[l] = oracle_mod.em_csr(int(lio[l + 1] - lio[l]), rp[r0:r1 + 1] - k0, b["col"][k0:k1],
                                                               b["alpha"][k0:k1], b["count"][r0:r1], **kw)
    return dict(status=st, theta=th, iters=it)


@pytest.mark.parametrize("max_iter", [1, 2, 3, 4, 5, 1000])
def test_longdouble_restatement_matches_the_oracle(oracle_mod, cell_batches, max_iter):
    """em_csr_longdouble against orc_em_csr (double) on the golden batch and on every cell locus: equal statuses and iteration
    counts, theta within 1e-12 relative (with the parity floor of 1e-9 x the locus' fragment total)."""
    golden, *_ = load_golden()
    for what, b in [("golden", golden)] + [(f"cells {k}", v[0]) for k, v in cell_batches.items()]:
        ld = cp.batch_em_longdouble(b, max_iter=max_iter)
        ora = _oracle_batch(oracle_mod, b, max_iter=max_iter)
        assert np.array_equal(ld["status"], ora["status"]), what
        assert np.array_equal(ld["iters"], ora["iters"]), what
        ok, worst = cp.theta_close_ld(ora["theta"], ld["theta"], b, 1e-12)
        assert ok.all(), (what, worst)
