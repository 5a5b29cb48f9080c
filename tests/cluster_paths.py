"""Which path every CTA of em_cluster_kernel takes, restated on the host; and a long-double restatement of the oracle's EM.

The cluster kernel (strawberry_b200/csrc/sbq_kernels.cuh, em_cluster_kernel) picks its path per CTA at run time, from the
locus alone and the CTA's share of its rows: whether the slice and its transposed (CSC) index sit in shared memory, how the
E- and M-passes spread over the threads, and how the partial theta' are exchanged inside the cluster. The planner
(strawberry_b200/csrc/sbq.cu, plan) picks the cluster size and the thread count. `cta_paths` restates all of it - the per-CTA
choice is `cta_path`, the restatement of the header's cluster_cta_path - so that the tests can say which paths a batch reaches and
check that a shape still reaches the path it was built for.

`em_csr_longdouble` is orc_em_csr (oracle/sbq_oracle.c:81-135) in np.longdouble: the yardstick for a few capped EM steps,
where a double-precision restatement would be no more exact than the kernel it checks.
"""
import numpy as np

# ---- constants (sbq_kernels.cuh, sbq.cu)
CL_NT = 512
CL_LPR_STREAM = 32
CL_A2A_MAX = 4096
CL_SMEM_CAP = 220 * 1024
BUCKET_NT = (64, 128, 512, 512, 512)                        # sbq.cu: BUCKET_NT
SMEM_BUCKET_BOUNDS = (12 * 1024, 24 * 1024, 56 * 1024, 112 * 1024)   # sbq.cu: smem_bucket
CLUSTER_NNZ_BOUNDS = (16 * 1024, 32 * 1024, 64 * 1024, 150 * 1024)   # sbq.cu: cluster_size_for

# Bar of the capped-solve checks (theta after max_iter = 1, 2, 5 EM steps against em_csr_longdouble, relative, with the parity floor
# of util.theta_close). Worst ratio measured on a B200 (1000 W power limit): 1.9e-15, over every tier on the golden batch and the
# cluster-path batches; the bar leaves a margin of more than 500x. A row of alpha off by 1e-6 relative moves theta by 5.9e-9
# after two steps (tests/test_gpu_cluster_paths.py, negative control).
CAPPED_REL = 1e-12

ORC_OK, ORC_ITER_CAP, ORC_ZERO_DENOM, ORC_NO_ROWS = 0, 1, 2, 3


def _tdiv(a, b):
    """C integer division (truncates toward zero)."""
    q = abs(a) // abs(b)
    return q if (a >= 0) == (b >= 0) else -q


# ---- host-callable functions of the header (sbq_kernels.cuh), one each under the same name
def cluster_a2a_stride(T):
    return (T + 1) & ~1


def cluster_a2a(T, cs, slice_bytes):
    if cs <= 1 or cs * cluster_a2a_stride(T) > CL_A2A_MAX:
        return False
    return (4 * T + cs * cluster_a2a_stride(T) + 64) * 8 + slice_bytes + 256 <= CL_SMEM_CAP


def cluster_fixed_doubles(T, cs, slice_bytes):
    return 4 * T + (cs * cluster_a2a_stride(T) + 64 if cluster_a2a(T, cs, slice_bytes) else 2 * T + 64)


def cluster_stream_groups(T, smem_bytes, nt, cs, slice_bytes):
    budget = smem_bytes // 8 - cluster_fixed_doubles(T, cs, slice_bytes)
    G = _tdiv(budget, T if T > 0 else 1)
    return min(G, nt // CL_LPR_STREAM)


def cluster_diag_slots(T):
    return (T + 7) & ~3


def cluster_resident_csr_bytes(nnz_c, nrows, T):
    npos = nnz_c + T
    return (npos + 1) * 8 + (nrows + 2) * 8 + cluster_diag_slots(T) * 4 + nrows * 4 + (T + 1) * 4 + nrows * 2 + npos * 2 + 64


def cluster_resident_bytes(nnz_c, nrows, T):
    return cluster_resident_csr_bytes(nnz_c, nrows, T) + nnz_c * 4 + 4


def cluster_class_smem(max_iso, slice_bytes, nt, cs):
    fixed = cluster_fixed_doubles(max_iso, cs, slice_bytes) * 8
    stream = (nt // CL_LPR_STREAM) * max_iso * 8
    want = fixed + max(slice_bytes, stream) + 256
    return min(want, CL_SMEM_CAP)


def cluster_slice_estimate(nnz, R, T, cs):                       # the product is a C double, as here
    return int(1.12 * float(cluster_resident_bytes(nnz // cs + 1, R // cs + 1, T))) + 512


def cta_path(T, cs, nt, nrows, nnz_c, too_long, slice_est, smem_launch):
    """cluster_cta_path: the path of one CTA with nrows rows and nnz_c non-zeros (too_long: a row has more than T entries)."""
    smem_bytes = min(smem_launch, cluster_class_smem(T, slice_est, nt, cs))
    used = cluster_fixed_doubles(T, cs, slice_est) * 8
    csr = cluster_resident_csr_bytes(nnz_c, nrows, T)
    small_idx = nnz_c + T <= 65535 and nrows <= 65535 and not too_long
    csc_in_smem = small_idx and used + cluster_resident_bytes(nnz_c, nrows, T) <= smem_bytes
    resident = small_idx and used + csr <= smem_bytes
    n_ent_s = nnz_c if csc_in_smem else min(nnz_c, (smem_bytes - used - csr) // 4) if resident else 0
    a2a = cluster_a2a(T, cs, slice_est)
    return dict(resident=resident, csc_in_smem=csc_in_smem, n_ent_s=n_ent_s,
                G=0 if resident else cluster_stream_groups(T, smem_bytes, nt, cs, slice_est),
                row_slots=resident and nrows <= nt, col_slots=resident and T <= nt, a2a=a2a,
                B=cluster_a2a_stride(T) if a2a else (T + cs - 1) // cs)


# ---- planner (sbq.cu: plan)
def smem_bucket(nbytes):
    for b, bound in enumerate(SMEM_BUCKET_BOUNDS):
        if nbytes <= bound:
            return b
    return len(SMEM_BUCKET_BOUNDS)


def cluster_size_for(nnz):
    for cs, bound in zip((1, 2, 4, 8), CLUSTER_NNZ_BOUNDS):
        if nnz <= bound:
            return cs
    return 16


def plan(T, R, nnz, force_cluster=0):
    """-> (cluster size, threads per CTA) of a cluster-tier locus."""
    cs = force_cluster or cluster_size_for(nnz)
    slice_bytes = cluster_slice_estimate(nnz, R, T, cs)
    bucket = smem_bucket(cluster_fixed_doubles(T, 1, slice_bytes) * 8 + slice_bytes + 256) if cs == 1 else len(BUCKET_NT) - 1
    return cs, BUCKET_NT[bucket]


# ---- per-CTA path (em_cluster_kernel: the row split, the too_long scan, then cluster_cta_path)
def cta_paths(T, row_ptr, force_cluster=0):
    """Paths of every CTA that solves the locus (T isoforms, locus-local row_ptr). -> list of dicts, one per rank."""
    rp = np.asarray(row_ptr, np.int64)
    rp = rp - rp[0]
    R = len(rp) - 1
    nnz = int(rp[R])
    CS, NT = plan(T, R, nnz, force_cluster)
    slice_est = cluster_slice_estimate(nnz, R, T, CS)
    smem_launch = cluster_class_smem(T, slice_est, NT, CS)                    # the launch provides at least this much
    lens = np.diff(rp)
    out = []
    for rank in range(CS):
        bounds = []
        for tid in (0, 1):                                                     # lower_bound on row_ptr
            if rank + tid >= CS:
                bounds.append(R)
            elif rank + tid == 0:
                bounds.append(0)
            else:
                target = (nnz * (rank + tid)) // CS
                bounds.append(int(np.searchsorted(rp[:R], target, side="left")))
        ra, rb = bounds
        nrows = rb - ra
        nnz_c = int(rp[rb] - rp[ra])
        too_long = bool(nrows and lens[ra:rb].max() > T)
        c = cta_path(T, CS, NT, nrows, nnz_c, too_long, slice_est, smem_launch)
        if not c["resident"]:
            slice_state, e_pass, m_pass = "stream", "stream", "stream"
        else:
            slice_state = "csc_smem" if c["csc_in_smem"] else "csc_partial"
            e_pass = "row_slots" if c["row_slots"] else "rows4"
            m_pass = "col_slots" if c["col_slots"] else "generic"
        B = c["B"]
        out.append(dict(CS=CS, NT=NT, exchange="single" if CS == 1 else "a2a" if c["a2a"] else "owner", slice=slice_state,
                        n_ent_s=c["n_ent_s"], nnz_c=nnz_c, E=e_pass, M=m_pass, rows=(ra, rb), nrows=nrows, G=c["G"], B=B,
                        owned=max(0, min(B, T - rank * B)) if CS > 1 and not c["a2a"] else T))
    return out


def cell(p):
    """The (CS, NT, exchange, slice, E-pass, M-pass) cell of one CTA's path."""
    return (p["CS"], p["NT"], p["exchange"], p["slice"], p["E"], p["M"])


def batch_cells(batch, force_cluster=0):
    """Cells reached by the cluster-tier CTAs of a flat batch (every locus taken through the cluster tier)."""
    lro, lio, rp = batch["loc_row_off"], batch["loc_iso_off"], batch["row_ptr"]
    cells = set()
    for l in range(len(lro) - 1):
        T = int(lio[l + 1] - lio[l])
        cells |= {cell(p) for p in cta_paths(T, rp[lro[l]:lro[l + 1] + 1], force_cluster)}
    return cells


# ---- long-double restatement of orc_em_csr (oracle/sbq_oracle.c:81-135)
def em_csr_longdouble(T, row_ptr, col, alpha, count, max_iter=1000, theta_tol=1e-2, row_eps=1e-5):
    """-> (status, theta as np.longdouble, iters), with orc_em_csr's row filter (:90-97), first pass on the raw alpha (:103),
    column normalisation of the kept rows after every pass (:121-125), stopping rule (:126-129; theta is not advanced on the
    step that converges) and statuses (a zero denominator keeps the initial theta, :114)."""
    ld = np.longdouble
    rp = np.asarray(row_ptr, np.int64)
    rp = rp - rp[0]
    col = np.asarray(col, np.int64)
    count = np.asarray(count, np.int64)
    R = len(count)
    total = ld(int(count.sum()))
    theta0 = np.full(T, total / ld(T), dtype=ld)
    lens = np.diff(rp)
    row_of = np.repeat(np.arange(R), lens)
    keep = np.zeros(R, bool)
    np.logical_or.at(keep, row_of, np.asarray(alpha) > row_eps)          # :92-96
    if not keep.any():
        return ORC_NO_ROWS, theta0, 0
    # the entries of the kept rows (each has one at least), in row order; row sums by reduceat over the rows' starts
    sel = np.nonzero(keep[row_of])[0]
    c = col[sel]
    F = np.asarray(alpha, dtype=ld)[sel]
    cnt_e = count[row_of[sel]].astype(ld)
    seg = np.searchsorted(sel, rp[np.nonzero(keep)[0]])
    order = np.argsort(c, kind="stable")                                 # entries by column, for the column sums
    cs_sorted = c[order]
    cstart = np.nonzero(np.r_[True, cs_sorted[1:] != cs_sorted[:-1]])[0] if len(c) else np.zeros(0, np.int64)
    ccols = cs_sorted[cstart]

    def colsum(v):
        out = np.zeros(T, dtype=ld)
        if len(v):
            out[ccols] = np.add.reduceat(v[order], cstart)
        return out

    cur = theta0.copy()
    status, iters = ORC_ITER_CAP, 0
    for it in range(max_iter):
        iters = it + 1
        prod = F * cur[c]
        denom = np.add.reduceat(prod, seg)
        if (denom == 0).any():                                           # :114
            return ORC_ZERO_DENOM, theta0, iters
        d_e = np.repeat(denom, np.diff(np.r_[seg, len(sel)]))
        nxt = colsum(cnt_e * prod / d_e)                                 # :115-118
        s = colsum(F)
        sc = s[c]
        F = np.where(sc != 0, F / np.where(sc != 0, sc, 1), F)           # :121-125
        d2 = ((nxt - cur) ** 2).sum()                                    # :126-128
        if np.sqrt(d2) < theta_tol:
            status = ORC_OK
            break
        cur = nxt
    return status, cur, iters


def batch_em_longdouble(batch, **kw):
    """em_csr_longdouble over every locus of a flat batch. -> dict(theta (longdouble), iters, status)."""
    lro, lio, rp = (np.asarray(batch[k], np.int64) for k in ("loc_row_off", "loc_iso_off", "row_ptr"))
    L = len(lro) - 1
    theta = np.zeros(int(lio[-1]), dtype=np.longdouble)
    iters, status = np.zeros(L, np.int32), np.zeros(L, np.int32)
    for l in range(L):
        r0, r1 = int(lro[l]), int(lro[l + 1])
        k0, k1 = int(rp[r0]), int(rp[r1])
        st, th, it = em_csr_longdouble(int(lio[l + 1] - lio[l]), rp[r0:r1 + 1], batch["col"][k0:k1], batch["alpha"][k0:k1],
                                       batch["count"][r0:r1], **kw)
        theta[lio[l]:lio[l + 1]], iters[l], status[l] = th, it, st
    return dict(theta=theta, iters=iters, status=status)


# ---- loci of fixed row lengths, and the shapes that reach the paths no other test runs
def fixed_rows_locus(rng, T, lengths):
    """One locus of T isoforms whose rows have exactly the given lengths (each <= T): distinct ascending columns, alpha in
    10^U(-4, -1.5), counts in 1..99."""
    lengths = np.asarray(lengths, np.int64)
    R = len(lengths)
    row_ptr = np.zeros(R + 1, np.int64)
    np.cumsum(lengths, out=row_ptr[1:])
    col = np.empty(int(row_ptr[-1]), np.int32)
    for k in np.unique(lengths):
        rows = np.nonzero(lengths == k)[0]
        if k == 0:
            continue
        pick = np.sort(np.argsort(rng.random((len(rows), T)), axis=1)[:, :k], axis=1)   # k distinct columns per row
        col[(row_ptr[rows][:, None] + np.arange(k)).ravel()] = pick.ravel()
    return dict(loc_row_off=np.array([0, R], np.int64), loc_iso_off=np.array([0, T], np.int64), row_ptr=row_ptr, col=col,
                alpha=10.0 ** rng.uniform(-4.0, -1.5, len(col)), count=rng.integers(1, 100, R).astype(np.int32),
                iso_len=rng.integers(300, 5000, T).astype(np.int32), total_mapped_reads=1_000_000)


# (T, [(rows, length), ...]) of the loci each batch holds; the cluster size is the planner's own (0) or forced
CELL_SHAPES = {
    0: [(100, [(20, 3)]),                      # NT 64, T > NT: generic M-pass
        (300, [(12, 3)]),                      # NT 128, T > NT: generic M-pass
        (40, [(40_000, 3)]),                   # CS 8, owner form, part of the CSC index in L2, four rows per thread
        (40, [(60_000, 3)]),                   # CS 16, four rows per thread
        (700, [(1_200, 50)]),                  # CS 4, generic M-pass
        (900, [(2_400, 50)]),                  # CS 8, owner form, partial CSC index, generic M-pass
        (600, [(12_000, 5)]),                  # CS 4, streaming
        (64, [(400, 64), (25_600, 1)]),        # CS 4: two CTAs resident, two streaming (the nnz split gives the short-row CTAs
                                               # far more rows than the 12 % slack of cluster_slice_estimate allows for)
        (5, [(55_000, 5)]),                    # CS 16, owner form with B = 1: ranks 5 - 15 own no column
        (100, [(110, 100), (8_621, 1)]),       # CS 2: CTA 1 resident with none of its CSC index in shared memory (n_ent_s = 0)
        (32, [(100, 32), (7_881, 1)])],        # CS 1: resident with one CSC entry in shared memory, the rest in L2
    4: [(800, [(200, 20)])],                   # forced CS 4, all-to-all, generic M-pass
    16: [(300, [(10, 30)])],                   # forced CS 16: 16 x T is over the all-to-all limit, six CTAs get no rows
}


def cell_batches(seed=2024):
    """{forced cluster size (0 = the planner's): (flat batch, [locus batch, ...])} of CELL_SHAPES, seeded."""
    from strawberry_b200 import synth
    rng = np.random.default_rng(seed)
    out = {}
    for cs, shapes in CELL_SHAPES.items():
        loci = [fixed_rows_locus(rng, T, np.concatenate([np.full(n, k) for n, k in rows])) for T, rows in shapes]
        b = synth.concat(loci)
        b["total_mapped_reads"] = 1_000_000
        out[cs] = (b, loci)
    return out


def theta_close_ld(got, ref, batch, rel):
    """util.theta_close against a long-double reference, the ratio taken in long double. -> (ok mask, worst ratio)."""
    from util import ABS_FLOOR_FRAC, locus_totals
    ld = np.longdouble
    tot = np.repeat(locus_totals(batch).astype(ld), np.diff(batch["loc_iso_off"]))
    scale = np.maximum(np.abs(ref), ld(ABS_FLOOR_FRAC) * np.maximum(tot, ld(1)))
    ratio = np.abs(np.asarray(got, ld) - ref) / scale
    return ratio <= rel, float(ratio.max()) if len(ratio) else 0.0
