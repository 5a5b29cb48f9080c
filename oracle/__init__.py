"""TEST INFRASTRUCTURE ONLY.

ctypes loaders for the CPU checkers:

* ``liboracle.so``      - our plain-C restatement (``sbq_oracle.c``), always buildable (gcc only).
* ``_ref/libsbref.so``  - the unmodified reference compiled from ``/root/reference`` plus our seam
                          harness (``ref_harness/ref_seams.cpp``); only buildable where the reference
                          checkout exists, but the built file travels to the GPU box.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference``
legs may import this package. The product (``strawberry_b200``) never does.
"""
import ctypes
import json
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_SO = os.path.join(_HERE, "liboracle.so")
REF_SO = os.path.join(_HERE, "_ref", "libsbref.so")
REFERENCE_ROOT = os.environ.get("SBQ_REFERENCE_ROOT", "/root/reference")

ORC_OK, ORC_ITER_CAP, ORC_ZERO_DENOM, ORC_NO_ROWS = 0, 1, 2, 3


def build(ref=True, quiet=True):
    """Compile liboracle.so and, when the reference checkout is present, _ref/libsbref.so."""
    out = subprocess.DEVNULL if quiet else None
    subprocess.check_call(["make", "-C", _HERE, "oracle"], stdout=out)
    if ref and os.path.isdir(os.path.join(REFERENCE_ROOT, "src")):
        subprocess.check_call(["make", "-C", _HERE, "-j8", "ref", f"REF={REFERENCE_ROOT}"], stdout=out)


class _EmParams(ctypes.Structure):
    _fields_ = [("max_iter", ctypes.c_int), ("theta_tol", ctypes.c_double), ("row_eps", ctypes.c_double)]


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


_oracle = None
_ref = None


def oracle_lib():
    global _oracle
    if _oracle is None:
        if not os.path.exists(ORACLE_SO):
            build(ref=False)
        _oracle = ctypes.CDLL(ORACLE_SO)
        _oracle.orc_em_dense.restype = ctypes.c_int
        _oracle.orc_em_csr.restype = ctypes.c_int
        _oracle.orc_epilogue.restype = ctypes.c_double
        _oracle.orc_quantify_batch.restype = ctypes.c_double
        _oracle.orc_em_bias_csr.restype = ctypes.c_int
    return _oracle


def have_ref():
    return os.path.exists(REF_SO)


def ref_lib():
    global _ref
    if _ref is None:
        _ref = ctypes.CDLL(REF_SO)
        _ref.ref_em_solve.restype = ctypes.c_int
        _ref.ref_em_solve_batch.restype = ctypes.c_double
        _ref.ref_locus_context.restype = ctypes.c_long
    return _ref


def em_params(max_iter=1000, theta_tol=1e-2, row_eps=1e-5):
    return _EmParams(max_iter, theta_tol, row_eps)


# ---------------------------------------------------------------- restatement (liboracle.so)
def em_dense(count, alpha, **kw):
    """-> (status, theta, iters) for a dense R x T model."""
    alpha = _c(alpha, np.float64)
    R, T = alpha.shape
    count = _c(count, np.int32)
    theta = np.zeros(T)
    iters = ctypes.c_int32(0)
    p = em_params(**kw)
    st = oracle_lib().orc_em_dense(T, R, _p(count), _p(alpha), ctypes.byref(p), _p(theta), ctypes.byref(iters))
    return st, theta, iters.value


def em_csr(T, row_ptr, col, alpha, count, **kw):
    row_ptr = _c(row_ptr, np.int64)
    col = _c(col, np.int32)
    alpha = _c(alpha, np.float64)
    count = _c(count, np.int32)
    R = len(count)
    theta = np.zeros(T)
    iters = ctypes.c_int32(0)
    p = em_params(**kw)
    st = oracle_lib().orc_em_csr(T, R, _p(row_ptr), _p(col), _p(alpha), _p(count), ctypes.byref(p),
                                 _p(theta), ctypes.byref(iters))
    return st, theta, iters.value


def epilogue(theta, iso_len, total_mapped_reads, min_iso_frac=0.0, effective_len_norm=False, insert_mean=0.0):
    theta = _c(theta, np.float64)
    iso_len = _c(iso_len, np.int32)
    T = len(theta)
    fpkm, frac = np.zeros(T), np.zeros(T)
    keep, na = np.zeros(T, np.int32), np.zeros(T, np.int32)
    s = oracle_lib().orc_epilogue(T, _p(theta), _p(iso_len), ctypes.c_int64(total_mapped_reads),
                                  ctypes.c_double(min_iso_frac), int(effective_len_norm),
                                  ctypes.c_double(insert_mean), _p(fpkm), _p(frac), _p(keep), _p(na))
    return dict(fpkm=fpkm, frac=frac, keep=keep, na=na, kept_sum=s)


def quantify_batch(batch, total_mapped_reads, min_iso_frac=0.0, effective_len_norm=False, insert_mean=0.0,
                   n_threads=1, **kw):
    """batch: dict with loc_row_off, loc_iso_off, row_ptr, col, alpha, count, iso_len (flat layout)."""
    lro, lio = _c(batch["loc_row_off"], np.int64), _c(batch["loc_iso_off"], np.int64)
    rp, col = _c(batch["row_ptr"], np.int64), _c(batch["col"], np.int32)
    al, cnt, il = _c(batch["alpha"], np.float64), _c(batch["count"], np.int32), _c(batch["iso_len"], np.int32)
    L, NI = len(lro) - 1, int(lio[-1])
    theta, fpkm, frac, tpm = (np.zeros(NI) for _ in range(4))
    keep = np.zeros(NI, np.int32)
    iters, status = np.zeros(L, np.int32), np.zeros(L, np.int32)
    p = em_params(**kw)
    secs = oracle_lib().orc_quantify_batch(
        ctypes.c_int64(L), _p(lro), _p(lio), _p(rp), _p(col), _p(al), _p(cnt), _p(il),
        ctypes.c_int64(total_mapped_reads), ctypes.byref(p), ctypes.c_double(min_iso_frac),
        int(effective_len_norm), ctypes.c_double(insert_mean), int(n_threads),
        _p(theta), _p(fpkm), _p(frac), _p(tpm), _p(keep), _p(iters), _p(status))
    return dict(theta=theta, fpkm=fpkm, frac=frac, tpm=tpm, keep=keep, iters=iters, status=status, seconds=secs)


class _BiasParams(ctypes.Structure):
    _fields_ = [("max_out_it", ctypes.c_int), ("max_theta_it", ctypes.c_int), ("max_bias_it", ctypes.c_int),
                ("theta_tol", ctypes.c_double), ("bias_tol", ctypes.c_double), ("row_eps", ctypes.c_double)]


def em_bias_csr(T, row_ptr, col, alpha, count, x, max_out_it=100, max_theta_it=5000, max_bias_it=10, theta_tol=1e-2,
                bias_tol=1e-2, row_eps=1e-5):
    """Bias mode restatement (OUR definition; parity unpinned vs the reference). -> (status, theta, beta, iters, outer)"""
    row_ptr, col = _c(row_ptr, np.int64), _c(col, np.int32)
    alpha, count, x = _c(alpha, np.float64), _c(count, np.int32), _c(x, np.float64)
    K = x.shape[1] if x.ndim == 2 else 0
    theta, beta = np.zeros(T), np.zeros(max(K, 1))
    iters, outer = ctypes.c_int32(0), ctypes.c_int32(0)
    p = _BiasParams(max_out_it, max_theta_it, max_bias_it, theta_tol, bias_tol, row_eps)
    L = oracle_lib()
    st = L.orc_em_bias_csr(T, len(count), _p(row_ptr), _p(col), _p(alpha), _p(count), _p(x) if x.size else None, K, ctypes.byref(p),
                           _p(theta), _p(beta), ctypes.byref(iters), ctypes.byref(outer))
    return st, theta, beta[:K], iters.value, outer.value


def batch_epilogue(batch, theta, status, total_mapped_reads, min_iso_frac=0.0, effective_len_norm=False, insert_mean=0.0):
    """FPKM / frac / keep per locus (orc_epilogue; NO_ROWS loci keep nothing) and the batch TPM over the kept isoforms, summed in
    isoform order - the tail of orc_quantify_batch (sbq_oracle.c) applied to a given theta. -> dict(fpkm, frac, tpm, keep)."""
    lio = np.asarray(batch["loc_iso_off"], np.int64)
    il = _c(batch["iso_len"], np.int32)
    NI = int(lio[-1])
    fpkm, frac, tpm = np.zeros(NI), np.zeros(NI), np.zeros(NI)
    keep = np.zeros(NI, np.int32)
    for l in range(len(lio) - 1):
        t0, t1 = int(lio[l]), int(lio[l + 1])
        e = epilogue(theta[t0:t1], il[t0:t1], total_mapped_reads, min_iso_frac, effective_len_norm, insert_mean)
        fpkm[t0:t1], frac[t0:t1] = e["fpkm"], e["frac"]
        keep[t0:t1] = 0 if status[l] == ORC_NO_ROWS else e["keep"]
    kept = np.where(keep != 0, fpkm, 0.0)
    total_fpkm = float(np.cumsum(kept)[-1]) if NI else 0.0     # sequential, in isoform order, like the C loop
    with np.errstate(divide="ignore", invalid="ignore"):
        tpm[:] = 1e6 * fpkm / total_fpkm
    return dict(fpkm=fpkm, frac=frac, tpm=tpm, keep=keep)


def bias_quantify_batch(batch, X, total_mapped_reads, min_iso_frac=0.0, effective_len_norm=False, insert_mean=0.0, n_threads=8,
                        **limits):
    """Bias mode over a flat batch: em_bias_csr per locus on a thread pool (ctypes releases the GIL), then batch_epilogue.
    X: (n_row, K) covariates in row order; limits: em_bias_csr's keywords. -> the keys of quantify_batch plus beta (L x K) and outer."""
    from concurrent.futures import ThreadPoolExecutor
    lro, lio, rp = (np.asarray(batch[k], np.int64) for k in ("loc_row_off", "loc_iso_off", "row_ptr"))
    col, al, cnt = _c(batch["col"], np.int32), _c(batch["alpha"], np.float64), _c(batch["count"], np.int32)
    X = np.asarray(X, np.float64)
    L, K = len(lro) - 1, X.shape[1]
    theta = np.zeros(int(lio[-1]))
    beta = np.zeros((L, K))
    status, iters, outer = np.zeros(L, np.int32), np.zeros(L, np.int32), np.zeros(L, np.int32)

    def one(l):
        r0, r1 = int(lro[l]), int(lro[l + 1])
        k0, k1 = int(rp[r0]), int(rp[r1])
        st, th, be, it, out = em_bias_csr(int(lio[l + 1] - lio[l]), rp[r0:r1 + 1] - k0, col[k0:k1], al[k0:k1], cnt[r0:r1], X[r0:r1], **limits)
        theta[lio[l]:lio[l + 1]], beta[l] = th, be
        status[l], iters[l], outer[l] = st, it, out

    with ThreadPoolExecutor(max(1, int(n_threads))) as ex:
        list(ex.map(one, range(L)))
    out = batch_epilogue(batch, theta, status, total_mapped_reads, min_iso_frac, effective_len_norm, insert_mean)
    out.update(theta=theta, iters=iters, status=status, beta=beta, outer=outer)
    return out


# ---------------------------------------------------------------- compiled reference (_ref/libsbref.so)
def ref_em(count, alpha):
    """EmSolver::init + run of the unmodified reference. -> (rc, theta); rc bit0 init ok, bit1 run ok."""
    alpha = _c(alpha, np.float64)
    R, T = alpha.shape
    count = _c(count, np.int32)
    theta = np.zeros(T)
    rc = ref_lib().ref_em_solve(T, R, _p(count), _p(alpha), _p(theta))
    return rc, theta


def ref_em_batch(batch, n_threads=1):
    lro, lio = _c(batch["loc_row_off"], np.int64), _c(batch["loc_iso_off"], np.int64)
    rp, col = _c(batch["row_ptr"], np.int64), _c(batch["col"], np.int32)
    al, cnt = _c(batch["alpha"], np.float64), _c(batch["count"], np.int32)
    L, NI = len(lro) - 1, int(lio[-1])
    theta = np.zeros(NI)
    rc = np.zeros(L, np.int32)
    secs = ref_lib().ref_em_solve_batch(ctypes.c_long(L), _p(lro), _p(lio), _p(rp), _p(col), _p(al), _p(cnt),
                                        _p(theta), _p(rc), int(n_threads))
    return dict(theta=theta, rc=rc, seconds=secs)


def ref_locus_context(transcripts, hits, *, read_len, mean=0.0, sd=0.0, frag_lens=None, long_read=False,
                      min_iso_frac=0.0, effective_len_norm=False, total_mapped_reads=1000):
    """Wide seam: LocusContext ctor + estimate_abundances of the unmodified reference.

    transcripts: list of feature lists [(code, offset, len), ...] (alternating MATCH=0 / INTRON=1)
    hits: list of (mass, left_mate, right_mate); a mate is None or (pos, [(cigar_op, len), ...])
          with BAM op codes (M=0, I=1, D=2, N=3, S=4).
    Returns the parsed JSON dump.
    """
    ptr, off, ln, code = [0], [], [], []
    for feats in transcripts:
        for c, o, l in feats:
            code.append(c), off.append(o), ln.append(l)
        ptr.append(len(off))
    cp, pos, ct, cl, mass = [0], [], [], [], []
    for m, left, right in hits:
        mass.append(m)
        for mate in (left, right):
            if mate is None:
                pos.append(0)
            else:
                pos.append(mate[0])
                for t, le in mate[1]:
                    ct.append(t), cl.append(le)
            cp.append(len(ct))
    a = [_c(ptr, np.int32), _c(off, np.uint32), _c(ln, np.int32), _c(code, np.int32)]
    h = [_c(mass, np.float64), _c(cp, np.int32), _c(pos, np.uint32), _c(ct, np.int32), _c(cl, np.int32)]
    fl = _c(frag_lens, np.int32) if frag_lens is not None else None
    cap = 1 << 22
    while True:
        buf = ctypes.create_string_buffer(cap)
        n = ref_lib().ref_locus_context(
            int(fl is not None), _p(fl), 0 if fl is None else len(fl), ctypes.c_double(mean), ctypes.c_double(sd),
            int(read_len), int(long_read), ctypes.c_double(min_iso_frac), int(effective_len_norm),
            int(total_mapped_reads), len(transcripts), *[_p(x) for x in a], len(hits), *[_p(x) for x in h],
            buf, ctypes.c_long(cap))
        if n >= 0:
            break
        cap = -n + 16

    def _num(x):
        return float(x)
    return json.loads(buf.value.decode(), parse_constant=_num)
