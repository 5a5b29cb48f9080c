"""Host-side Python mirror of the reference's quantification interface, over the C ABI (include/sbq.h).

Everything numeric runs in libsbq.so on the GPU; this module only marshals arrays. If the CUDA
library is missing or no B200 is visible, the calls raise - there is no CPU path here.

Mirrored reference interfaces (file:line under the ruolin/strawberry checkout):
  EmSolver.init / run / _theta                 include/estimate.hpp:230-257, src/estimate.cpp:366-488
  Quantifier.submit* / run / results           LocusContext::estimate_abundances (src/estimate.cpp:279-364)
                                               + the TPM tail of Sample::procSample (src/alignments.cpp:1821-1829)
"""
import ctypes
import os
import weakref

# a solve runs ~12 kernels concurrently, one stream each: more hardware work queues than the default 8 (no effect once the
# process has created its CUDA context - import this module, or export the variable, before touching CUDA)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SBQ_LIB_PATH", os.path.join(_HERE, "libsbq.so"))   # override: A/B-testing kernel variants

SBQ_SUCCESS, SBQ_ERR_INVALID, SBQ_ERR_NO_DEVICE, SBQ_ERR_CUDA, SBQ_ERR_NOMEM, SBQ_ERR_STATE, SBQ_ERR_UNSUPPORTED = 0, -1, -2, -3, -4, -5, -6
LOCUS_OK, LOCUS_ITER_CAP, LOCUS_ZERO_DENOM, LOCUS_NO_ROWS = 0, 1, 2, 3

# every symbol include/sbq.h declares (tests check that the library exports all of them)
ABI_SYMBOLS = [
    "sbq_abi_version", "sbq_error_string", "sbq_last_error", "sbq_config_default", "sbq_create", "sbq_destroy",
    "sbq_submit", "sbq_submit_flat", "sbq_clear", "sbq_validate", "sbq_host_alloc", "sbq_host_free",
    "sbq_upload", "sbq_upload_begin", "sbq_solve", "sbq_download", "sbq_run", "sbq_fpkm_sum", "sbq_fpkm_sum_to_device",
    "sbq_finalize_tpm", "sbq_results", "sbq_get_stats", "sbq_get_launch_stats", "sbq_em_solve", "sbq_set_plan",
    "sbq_set_covariates", "sbq_bias_results", "sbq_partition_lpt", "sbq_locus_devices", "sbq_synth_giant", "sbq_fetch_batch",
    "sbq_bootstrap", "sbq_bootstrap_results", "sbq_bootstrap_counts", "sbq_bootstrap_stats",
    "sbq_gibbs", "sbq_gibbs_results", "sbq_gibbs_stats",
]


class SbqError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"sbq error {code}: {msg}")
        self.code = code


class Config(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int32), ("max_iter", ctypes.c_int32), ("theta_tol", ctypes.c_double),
                ("row_eps", ctypes.c_double), ("min_iso_frac", ctypes.c_double),
                ("effective_len_norm", ctypes.c_int32), ("insert_mean", ctypes.c_double),
                ("bias_mode", ctypes.c_int32), ("max_out_it", ctypes.c_int32), ("max_theta_it", ctypes.c_int32),
                ("max_bias_it", ctypes.c_int32), ("bias_tol", ctypes.c_double), ("n_gpus", ctypes.c_int32)]


class Locus(ctypes.Structure):
    _fields_ = [("n_iso", ctypes.c_int32), ("n_row", ctypes.c_int32), ("row_ptr", ctypes.c_void_p),
                ("col", ctypes.c_void_p), ("alpha", ctypes.c_void_p), ("count", ctypes.c_void_p),
                ("iso_len", ctypes.c_void_p)]


class SynthGiantSpec(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("n_loci", ctypes.c_int32), ("locus_ids", ctypes.c_void_p), ("rows_per_locus", ctypes.c_int64),
                ("iso_lo", ctypes.c_int32), ("iso_hi", ctypes.c_int32), ("mean_extra", ctypes.c_double)]


class Stats(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int64) for n in ("n_loci", "n_row", "n_iso", "nnz", "loci_warp", "loci_cta", "loci_grid",
                                              "kernel_launches", "h2d_bytes", "d2h_bytes")] + \
               [(n, ctypes.c_double) for n in ("upload_ms", "solve_ms", "download_ms", "em_ms", "grid_em_ms")] + \
               [(n, ctypes.c_int64) for n in ("em_iters_total", "frag_iters", "alg_bytes", "grid_alg_bytes")] + \
               [("weights_ms", ctypes.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class LaunchStat(ctypes.Structure):
    _fields_ = [("kind", ctypes.c_int32), ("cluster_size", ctypes.c_int32), ("lanes_per_row", ctypes.c_int32),
                ("variant", ctypes.c_int32), ("n_loci", ctypes.c_int64), ("nnz", ctypes.c_int64), ("ms", ctypes.c_double),
                ("alg_bytes", ctypes.c_int64), ("frag_iters", ctypes.c_int64), ("max_iters", ctypes.c_int64), ("start_ms", ctypes.c_double)]


class BootstrapStat(ctypes.Structure):
    _fields_ = [("first", ctypes.c_int64), ("n", ctypes.c_int64), ("resample_ms", ctypes.c_double), ("em_ms", ctypes.c_double),
                ("total_ms", ctypes.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class GibbsStat(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int64), ("rounds", ctypes.c_int64), ("colsum_ms", ctypes.c_double), ("assign_ms", ctypes.c_double),
                ("theta_ms", ctypes.c_double), ("total_ms", ctypes.c_double)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


_lib = None


def lib():
    """Load libsbq.so. Fails loudly when it has not been built (python -m strawberry_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build the CUDA extension first "
                               "(python -m strawberry_b200.build or __graft_entry__.build()); there is no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        L.sbq_error_string.restype = ctypes.c_char_p
        L.sbq_last_error.restype = ctypes.c_char_p
        L.sbq_last_error.argtypes = [ctypes.c_void_p]
        L.sbq_host_alloc.restype = ctypes.c_void_p
        L.sbq_host_alloc.argtypes = [ctypes.c_size_t]
        L.sbq_host_free.argtypes = [ctypes.c_void_p]
        L.sbq_config_default.argtypes = [ctypes.POINTER(Config)]
        L.sbq_create.argtypes = [ctypes.POINTER(Config), ctypes.POINTER(ctypes.c_void_p)]
        L.sbq_destroy.argtypes = [ctypes.c_void_p]
        for name in ("sbq_clear", "sbq_validate", "sbq_upload", "sbq_upload_begin", "sbq_download"):
            getattr(L, name).argtypes = [ctypes.c_void_p]
        L.sbq_submit.argtypes = [ctypes.c_void_p, ctypes.POINTER(Locus), ctypes.c_int64]
        L.sbq_submit_flat.argtypes = [ctypes.c_void_p, ctypes.c_int64] + [ctypes.c_void_p] * 7
        L.sbq_solve.argtypes = [ctypes.c_void_p, ctypes.c_int64]
        L.sbq_run.argtypes = [ctypes.c_void_p, ctypes.c_int64]
        L.sbq_fpkm_sum.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]
        L.sbq_fpkm_sum_to_device.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.sbq_finalize_tpm.argtypes = [ctypes.c_void_p, ctypes.c_double]
        L.sbq_results.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 7
        L.sbq_get_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(Stats)]
        L.sbq_get_launch_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(LaunchStat), ctypes.c_int]
        L.sbq_em_solve.argtypes = [ctypes.c_void_p, ctypes.POINTER(Locus), ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32)]
        L.sbq_set_plan.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
        L.sbq_set_covariates.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32]
        L.sbq_bias_results.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
        L.sbq_partition_lpt.argtypes = [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_void_p]
        L.sbq_locus_devices.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.sbq_synth_giant.argtypes = [ctypes.c_void_p, ctypes.POINTER(SynthGiantSpec)]
        L.sbq_fetch_batch.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 7
        L.sbq_bootstrap.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_int32]
        L.sbq_bootstrap_results.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 4
        L.sbq_bootstrap_counts.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int64, ctypes.c_void_p]
        L.sbq_bootstrap_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(BootstrapStat)]
        L.sbq_gibbs.argtypes = [ctypes.c_void_p, ctypes.c_uint64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32, ctypes.c_double]
        L.sbq_gibbs_results.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 3
        L.sbq_gibbs_stats.argtypes = [ctypes.c_void_p, ctypes.POINTER(GibbsStat)]
        _lib = L
    return _lib


def default_config(**overrides):
    cfg = Config()
    lib().sbq_config_default(ctypes.byref(cfg))
    for k, v in overrides.items():
        if not hasattr(cfg, k):
            raise TypeError(f"unknown sbq_config field {k!r}")
        setattr(cfg, k, v)
    return cfg


def _ptr(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def pinned_empty(n, dtype):
    """numpy array over page-locked memory from sbq_host_alloc (freed when the array is collected)."""
    dtype = np.dtype(dtype)
    nbytes = max(int(n) * dtype.itemsize, 1)
    p = lib().sbq_host_alloc(nbytes)
    if not p:
        raise SbqError(SBQ_ERR_NOMEM, "sbq_host_alloc failed (no CUDA device?)")
    buf = (ctypes.c_char * nbytes).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype, count=int(n))
    weakref.finalize(buf, lib().sbq_host_free, p)
    return arr


def pinned_batch(batch):
    """Copy a flat batch (strawberry_b200.synth layout) into page-locked arrays."""
    spec = dict(loc_row_off=np.int64, loc_iso_off=np.int64, row_ptr=np.int64, col=np.int32, alpha=np.float64,
                count=np.int32, iso_len=np.int32)
    out = dict(batch)
    for k, dt in spec.items():
        a = pinned_empty(len(batch[k]), dt)
        a[...] = batch[k]
        out[k] = a
    return out


def partition_lpt(cost, n_parts):
    """sbq_partition_lpt: owner[l] of the greedy LPT partition the multi-GPU context uses (host-only, no device needed)."""
    cost = _c(cost, np.int64)
    owner = np.empty(len(cost), np.int32)
    rc = lib().sbq_partition_lpt(_ptr(cost), len(cost), int(n_parts), _ptr(owner))
    if rc:
        raise SbqError(rc, lib().sbq_error_string(rc).decode())
    return owner


class Quantifier:
    """One GPU context: queue loci, run the EM + FPKM/frac/TPM epilogue, read results back."""

    def __init__(self, **config):
        self._L = lib()
        self.cfg = default_config(**config)
        h = ctypes.c_void_p()
        rc = self._L.sbq_create(ctypes.byref(self.cfg), ctypes.byref(h))
        if rc != SBQ_SUCCESS:
            raise SbqError(rc, self._L.sbq_error_string(rc).decode())
        self._h = h
        self._keepalive = []
        self._fin = weakref.finalize(self, self._L.sbq_destroy, h)

    def close(self):
        self._fin()
        self._h = None          # a call on a closed Quantifier raises (ctypes passes NULL -> SBQ_ERR_INVALID) instead of touching freed memory

    def _chk(self, rc):
        if rc < 0:
            msg = self._L.sbq_last_error(self._h).decode() or self._L.sbq_error_string(rc).decode()
            raise SbqError(rc, msg)
        return rc

    def clear(self):
        self._keepalive = []
        self._chk(self._L.sbq_clear(self._h))

    def set_plan(self, force_tier=0, force_cluster=0):
        self._chk(self._L.sbq_set_plan(self._h, int(force_tier), int(force_cluster)))

    def submit_flat(self, batch):
        a = [_c(batch["loc_row_off"], np.int64), _c(batch["loc_iso_off"], np.int64), _c(batch["row_ptr"], np.int64),
             _c(batch["col"], np.int32), _c(batch["alpha"], np.float64), _c(batch["count"], np.int32),
             _c(batch["iso_len"], np.int32)]
        self._keepalive.append(a)   # borrowed in place when page-locked
        self._chk(self._L.sbq_submit_flat(self._h, len(a[0]) - 1, *[_ptr(x) for x in a]))

    def submit(self, loci):
        """loci: iterable of (n_iso, row_ptr, col, alpha, count, iso_len)."""
        arr, keep = [], []
        for n_iso, row_ptr, col, alpha, count, iso_len in loci:
            rp, c, a = _c(row_ptr, np.int64), _c(col, np.int32), _c(alpha, np.float64)
            n, il = _c(count, np.int32), _c(iso_len, np.int32)
            keep.append((rp, c, a, n, il))
            arr.append(Locus(int(n_iso), len(n), rp.ctypes.data, c.ctypes.data, a.ctypes.data, n.ctypes.data, il.ctypes.data))
        buf = (Locus * len(arr))(*arr)
        self._chk(self._L.sbq_submit(self._h, buf, len(arr)))

    def set_covariates(self, x):
        """bias mode: per-row covariates, shape (n_row, n_cov), rows in submit order"""
        x = _c(x, np.float64)
        self._n_cov = x.shape[1] if x.ndim == 2 else 0
        self._chk(self._L.sbq_set_covariates(self._h, _ptr(x) if x.size else None, x.shape[0], self._n_cov))

    def bias_results(self):
        nl = self.stats()["n_loci"]
        beta = np.zeros((nl, max(self._n_cov, 1)))
        outer = np.zeros(nl, np.int32)
        self._chk(self._L.sbq_bias_results(self._h, _ptr(beta), _ptr(outer)))
        return beta[:, :self._n_cov], outer

    def set_insert_model(self, model, read_len):
        """deferred (GPU) weights: the context's insert-size model (builder.Model) and read length"""
        from . import builder
        builder._lib()
        self._model = model
        self._chk(self._L.sbq_set_insert_model(self._h, ctypes.byref(model.struct), int(read_len)))

    def submit_deferred(self, tables):
        """tables: builder.TableHandle objects built with defer_weights=True"""
        from . import builder
        builder._lib()
        arr = (ctypes.c_void_p * len(tables))(*[t.handle for t in tables])
        self._keepalive.append(tables)
        self._chk(self._L.sbq_submit_deferred(self._h, arr, len(tables)))

    def fetch_alpha(self):
        out = np.empty(self.stats()["nnz"])
        self._chk(self._L.sbq_fetch_alpha(self._h, _ptr(out)))
        return out

    def validate(self):
        self._chk(self._L.sbq_validate(self._h))

    def upload(self):
        self._chk(self._L.sbq_upload(self._h))

    def upload_begin(self):
        """asynchronous upload: the next solve() overlaps the tail of the copies (arrays must stay alive until it returns)"""
        self._chk(self._L.sbq_upload_begin(self._h))

    def solve(self, total_mapped_reads):
        self._chk(self._L.sbq_solve(self._h, int(total_mapped_reads)))

    def download(self):
        self._chk(self._L.sbq_download(self._h))

    def run(self, total_mapped_reads):
        self._chk(self._L.sbq_run(self._h, int(total_mapped_reads)))

    def fpkm_sum(self):
        s = ctypes.c_double(0)
        self._chk(self._L.sbq_fpkm_sum(self._h, ctypes.byref(s)))
        return s.value

    def fpkm_sum_to_device(self, dev_ptr):
        self._chk(self._L.sbq_fpkm_sum_to_device(self._h, ctypes.c_void_p(dev_ptr)))

    def finalize_tpm(self, global_fpkm_sum):
        self._chk(self._L.sbq_finalize_tpm(self._h, float(global_fpkm_sum)))

    def stats(self):
        s = Stats()
        self._chk(self._L.sbq_get_stats(self._h, ctypes.byref(s)))
        return s.as_dict()

    def launch_stats(self):
        cap = 32 * max(1, int(self.cfg.n_gpus))
        buf = (LaunchStat * cap)()
        n = self._chk(self._L.sbq_get_launch_stats(self._h, buf, cap))
        names = {1: "em_warp_kernel", 2: "em_cluster_kernel", 3: "em_grid_kernel"}
        grid = {1: "em_grid_kernel", 2: "em_grid_tma_kernel", 3: "em_grid_dual_kernel"}
        return [dict(kernel=grid.get(buf[i].variant, names[buf[i].kind]) if buf[i].kind == 3 else names[buf[i].kind], cluster_size=buf[i].cluster_size, lanes_per_row=buf[i].lanes_per_row,
                     n_loci=buf[i].n_loci, nnz=buf[i].nnz, ms=buf[i].ms, alg_bytes=buf[i].alg_bytes,
                     frag_iters=buf[i].frag_iters, max_iters=buf[i].max_iters, start_ms=buf[i].start_ms, threads=buf[i].lanes_per_row) for i in range(min(n, cap))]

    def synth_giant(self, locus_ids, rows_per_locus, seed=4, iso_lo=500, iso_hi=800, mean_extra=47.0):
        """Generate giant loci ON THE DEVICE (sbq_synth_giant): replaces submit + upload, the batch lives in HBM only."""
        ids = _c(locus_ids, np.int32)
        spec = SynthGiantSpec(int(seed), len(ids), ids.ctypes.data, int(rows_per_locus), int(iso_lo), int(iso_hi), float(mean_extra))
        self._keepalive = []
        self._chk(self._L.sbq_synth_giant(self._h, ctypes.byref(spec)))

    def fetch_batch(self):
        """Device -> host copy of the resident batch (flat layout of include/sbq.h); for tests of device-generated input."""
        st = self.stats()
        out = dict(loc_row_off=np.empty(st["n_loci"] + 1, np.int64), loc_iso_off=np.empty(st["n_loci"] + 1, np.int64),
                   row_ptr=np.empty(st["n_row"] + 1, np.int64), col=np.empty(st["nnz"], np.int32), alpha=np.empty(st["nnz"]),
                   count=np.empty(st["n_row"], np.int32), iso_len=np.empty(st["n_iso"], np.int32))
        self._chk(self._L.sbq_fetch_batch(self._h, *[_ptr(out[k]) for k in ("loc_row_off", "loc_iso_off", "row_ptr", "col", "alpha", "count", "iso_len")]))
        out["total_mapped_reads"] = int(out["count"].sum())
        return out

    def locus_devices(self):
        """device ordinal that solved each queued locus (multi-GPU contexts partition loci by non-zeros)"""
        out = np.empty(self.stats()["n_loci"], np.int32)
        self._chk(self._L.sbq_locus_devices(self._h, _ptr(out)))
        return out

    def results(self):
        st = self.stats()
        ni, nl = st["n_iso"], st["n_loci"]
        out = dict(theta=np.empty(ni), fpkm=np.empty(ni), frac=np.empty(ni), tpm=np.empty(ni),
                   keep=np.empty(ni, np.int32), iters=np.empty(nl, np.int32), status=np.empty(nl, np.int32))
        self._chk(self._L.sbq_results(self._h, *[_ptr(out[k]) for k in ("theta", "fpkm", "frac", "tpm", "keep", "iters", "status")]))
        return out

    def bootstrap(self, seed, n, first=0):
        """Bootstrap replicates first .. first + n - 1 of the solved, resident batch (DESIGN.md "Bootstrap replicates"): theta and
        tpm shaped (n, n_iso), iters and status shaped (n, n_loci), submit order. The point estimate (results()) is unchanged."""
        self._chk(self._L.sbq_bootstrap(self._h, int(seed) & (2**64 - 1), int(first), int(n)))
        st = self.stats()
        ni, nl = st["n_iso"], st["n_loci"]
        out = dict(theta=np.empty((n, ni)), tpm=np.empty((n, ni)), iters=np.empty((n, nl), np.int32), status=np.empty((n, nl), np.int32))
        self._chk(self._L.sbq_bootstrap_results(self._h, *[_ptr(out[k]) for k in ("theta", "tpm", "iters", "status")]))
        return out

    def bootstrap_counts(self, seed, replicate):
        """The resampled class counts of one replicate, per row in submit order (needs a resident batch only)."""
        out = np.empty(self.stats()["n_row"], np.int32)
        self._chk(self._L.sbq_bootstrap_counts(self._h, int(seed) & (2**64 - 1), int(replicate), _ptr(out) if out.size else ctypes.c_void_p(1)))
        return out

    def bootstrap_stats(self):
        """Device time of the last bootstrap(): resample_ms, em_ms (EM + FPKM sum, all replicates) and total_ms."""
        s = BootstrapStat()
        self._chk(self._L.sbq_bootstrap_stats(self._h, ctypes.byref(s)))
        return s.as_dict()

    def gibbs(self, seed, n, thin=16, burn_in=16, prior=0.01):
        """n Gibbs posterior samples of the solved, resident batch (DESIGN.md "Gibbs posterior samples"): sample s is the chain's
        state after round burn_in + (s + 1) * thin, every chain started from the point estimate. theta and tpm shaped (n, n_iso),
        status (the point estimate's) shaped (n, n_loci), submit order. The point estimate (results()) is unchanged.
        The defaults (thin 16, burn_in 16, a symmetric Dirichlet(0.01) prior) are this project's choice, not the reference's."""
        self._chk(self._L.sbq_gibbs(self._h, int(seed) & (2**64 - 1), int(n), int(thin), int(burn_in), float(prior)))
        st = self.stats()
        ni, nl = st["n_iso"], st["n_loci"]
        out = dict(theta=np.empty((n, ni)), tpm=np.empty((n, ni)), status=np.empty((n, nl), np.int32))
        self._chk(self._L.sbq_gibbs_results(self._h, *[_ptr(out[k]) for k in ("theta", "tpm", "status")]))
        return out

    def gibbs_stats(self):
        """Device time of the last gibbs(): n, rounds, colsum_ms (one-off setup), assign_ms and theta_ms (all rounds), total_ms."""
        s = GibbsStat()
        self._chk(self._L.sbq_gibbs_stats(self._h, ctypes.byref(s)))
        return s.as_dict()

    def em_solve(self, n_iso, row_ptr, col, alpha, count):
        rp, c, a, n = _c(row_ptr, np.int64), _c(col, np.int32), _c(alpha, np.float64), _c(count, np.int32)
        il = np.full(n_iso, 1000, np.int32)
        loc = Locus(int(n_iso), len(n), rp.ctypes.data, c.ctypes.data, a.ctypes.data, n.ctypes.data, il.ctypes.data)
        theta = np.empty(n_iso)
        iters = ctypes.c_int32(0)
        st = self._chk(self._L.sbq_em_solve(self._h, ctypes.byref(loc), _ptr(theta), ctypes.byref(iters)))
        return st, theta, iters.value


class EmSolver:
    """Drop-in for the reference's EmSolver (include/estimate.hpp:230-257).

    init(num_iso, count, model) -> bool and run() -> bool keep the reference's meaning
    (src/estimate.cpp:366-409, :411-488); `_theta` holds the abundances. The solve itself is
    sbq_em_solve on the GPU; init() only reshapes the dense model into CSR rows.
    """

    def __init__(self, quantifier=None):
        self._q = quantifier or Quantifier()
        self._theta = []
        self._status = None
        self.iters = 0

    def init(self, num_iso, count, model):
        model = np.asarray(model, dtype=np.float64).reshape(len(count), num_iso)
        rows, cols = np.nonzero(model)
        row_ptr = np.zeros(len(count) + 1, np.int64)
        np.cumsum(np.bincount(rows, minlength=len(count)), out=row_ptr[1:])
        st, theta, it = self._q.em_solve(num_iso, row_ptr, cols.astype(np.int32), model[rows, cols], count)
        self._status, self._theta, self.iters = st, list(theta), it
        return st != LOCUS_NO_ROWS

    def run(self):
        if self._status is None or self._status == LOCUS_NO_ROWS:
            return False
        return self._status != LOCUS_ZERO_DENOM
