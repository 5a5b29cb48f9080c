"""Python binding of the host class-table builder (include/sbq_builder.h, strawberry_b200/csrc/sbq_builder.cpp).

Mirrors the inputs of the reference's LocusContext constructor (include/estimate.hpp:61-109): the
locus' transcripts and its collapsed fragments, plus the insert-size model and read length that the
reference reads from Sample. Returns the class table and the CSR locus sbq_submit() takes.
"""
import ctypes

import numpy as np

from . import api

MATCH, INTRON, GAP = 0, 1, 2
CIG_M, CIG_I, CIG_D, CIG_N, CIG_S = 0, 1, 2, 3, 4

BUILDER_SYMBOLS = ["sbq_build_locus", "sbq_table_free", "sbq_table_locus", "sbq_table_get_dims", "sbq_table_segments",
                   "sbq_table_iso_segments", "sbq_table_classes", "sbq_table_hit_classes", "sbq_table_weight_desc",
                   "sbq_set_insert_model", "sbq_submit_deferred", "sbq_fetch_alpha", "sbq_pair_features", "sbq_effective_len", "sbq_insert_pdf",
                   "sbq_submit_raw", "sbq_fetch_raw_classes", "sbq_fetch_raw_coords", "sbq_set_raw_mass_mode"]
RAW_MASS_HALVES, RAW_MASS_ANY = 0, 1


class InsertModel(ctypes.Structure):
    _fields_ = [("use_emp", ctypes.c_int32), ("start_offset", ctypes.c_int32), ("end_offset", ctypes.c_int32),
                ("emp_dist", ctypes.c_void_p), ("total_reads", ctypes.c_int32), ("mean", ctypes.c_double), ("sd", ctypes.c_double)]


class LocusInput(ctypes.Structure):
    _fields_ = [("n_iso", ctypes.c_int32), ("iso_feat_ptr", ctypes.c_void_p), ("iso_feat_off", ctypes.c_void_p),
                ("iso_feat_len", ctypes.c_void_p), ("iso_feat_code", ctypes.c_void_p), ("n_hit", ctypes.c_int32),
                ("hit_feat_ptr", ctypes.c_void_p), ("hit_feat_off", ctypes.c_void_p), ("hit_feat_len", ctypes.c_void_p),
                ("hit_feat_code", ctypes.c_void_p), ("hit_mass", ctypes.c_void_p), ("hit_ref_id", ctypes.c_void_p),
                ("read_len", ctypes.c_int32), ("long_read", ctypes.c_int32), ("defer_weights", ctypes.c_int32)]


class TableDims(ctypes.Structure):
    _fields_ = [("n_seg", ctypes.c_int32), ("n_class", ctypes.c_int32), ("n_iso", ctypes.c_int32), ("nnz", ctypes.c_int64),
                ("n_coord", ctypes.c_int64), ("n_dropped_hits", ctypes.c_int32)]


def _lib():
    L = api.lib()
    if not getattr(L, "_builder_ready", False):
        L.sbq_build_locus.argtypes = [ctypes.POINTER(LocusInput), ctypes.POINTER(InsertModel), ctypes.POINTER(ctypes.c_void_p)]
        L.sbq_table_free.argtypes = [ctypes.c_void_p]
        L.sbq_table_locus.argtypes = [ctypes.c_void_p, ctypes.POINTER(api.Locus)]
        L.sbq_table_get_dims.argtypes = [ctypes.c_void_p, ctypes.POINTER(TableDims)]
        L.sbq_table_segments.argtypes = [ctypes.c_void_p] * 3
        L.sbq_table_iso_segments.argtypes = [ctypes.c_void_p] * 3
        L.sbq_table_classes.argtypes = [ctypes.c_void_p] * 6
        L.sbq_table_hit_classes.argtypes = [ctypes.c_void_p] * 2
        L.sbq_set_insert_model.argtypes = [ctypes.c_void_p, ctypes.POINTER(InsertModel), ctypes.c_int32]
        L.sbq_submit_deferred.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64]
        L.sbq_fetch_alpha.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.sbq_pair_features.argtypes = [ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                        ctypes.c_uint32, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32,
                                        ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int32]
        L.sbq_submit_raw.argtypes = [ctypes.c_void_p, ctypes.POINTER(LocusInput), ctypes.c_void_p]
        L.sbq_fetch_raw_classes.argtypes = [ctypes.c_void_p] * 7
        L.sbq_fetch_raw_coords.argtypes = [ctypes.c_void_p] * 3
        L.sbq_set_raw_mass_mode.argtypes = [ctypes.c_void_p, ctypes.c_int32]
        L.sbq_effective_len.restype = ctypes.c_int32
        L.sbq_effective_len.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]
        L.sbq_insert_pdf.restype = ctypes.c_double
        L.sbq_insert_pdf.argtypes = [ctypes.POINTER(InsertModel), ctypes.c_uint32]
        L._builder_ready = True
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None and a.size else None


class Model:
    """InsertSize (include/read.hpp:176-192): Model.normal(mean, sd) or Model.empirical(frag_lens)."""

    def __init__(self, struct, keep):
        self.struct, self._keep = struct, keep

    @classmethod
    def normal(cls, mean, sd):
        return cls(InsertModel(0, 0, 0, None, 0, float(mean), float(sd)), None)

    @classmethod
    def empirical(cls, frag_lens):
        """InsertSize(vector<int>) (src/read.cpp:236-267): histogram + mean/sd of the observed lengths."""
        fl = np.asarray(frag_lens, dtype=np.int64)
        lo, hi = int(fl.min()), int(fl.max())
        dist = np.bincount(fl - lo, minlength=hi - lo + 1).astype(np.float64)
        s = float(fl.sum())
        mean = s / len(fl)
        sd = float(np.sqrt(float((fl * fl).sum()) / len(fl) - mean * mean))
        return cls(InsertModel(1, lo, hi, dist.ctypes.data, len(fl), mean, sd), dist)

    def pdf(self, x):
        return _lib().sbq_insert_pdf(ctypes.byref(self.struct), int(x))


def _flatten(lists):
    ptr, off, ln, code = [0], [], [], []
    for feats in lists:
        for c, o, l in feats:
            code.append(c), off.append(o), ln.append(l)
        ptr.append(len(off))
    return (np.asarray(ptr, np.int32), np.asarray(off, np.uint32), np.asarray(ln, np.uint32), np.asarray(code, np.uint8))


def pair_features(left, right):
    """Contig(PairedHit) feature list (src/contig.cpp:216-267). A mate is None or (pos, [(cigar_op, len), ...])."""
    def mate(m):
        if m is None:
            return 0, np.zeros(0, np.uint8), np.zeros(0, np.uint32)
        return int(m[0]), np.asarray([o for o, _ in m[1]], np.uint8), np.asarray([l for _, l in m[1]], np.uint32)
    lp, lo, ll = mate(left)
    rp, ro, rl = mate(right)
    cap = 2 * (len(lo) + len(ro)) + 4
    off, ln, code = np.zeros(cap, np.uint32), np.zeros(cap, np.uint32), np.zeros(cap, np.uint8)
    n = _lib().sbq_pair_features(lp, _p(lo), _p(ll), len(lo), rp, _p(ro), _p(rl), len(ro), _p(off), _p(ln), _p(code), cap)
    if n < 0:
        raise api.SbqError(n, "sbq_pair_features")
    return [(int(code[k]), int(off[k]), int(ln[k])) for k in range(n)]


def effective_len(seg_lens, implicit_idx, fl, rl):
    s, im = np.asarray(seg_lens, np.uint32), np.asarray(implicit_idx, np.uint32)
    return _lib().sbq_effective_len(_p(s), len(s), _p(im), len(im), int(fl), int(rl))


class TableHandle:
    """Owns an sbq_table (freed on collection); passed to Quantifier.submit_deferred."""

    def __init__(self, handle):
        self.handle = handle

    def __del__(self):
        if self.handle:
            _lib().sbq_table_free(self.handle)
            self.handle = None


def build_locus(transcripts, hits, *, read_len, model=None, long_read=False, ref_ids=None, defer_weights=False):
    """transcripts: list of feature lists [(code, offset, len), ...]; hits: list of (mass, feature list).

    Returns a dict: segs [(l, r)], iso_segs [[seg idx]], iso_len, classes [{coords, count, mass, nfrag}],
    row_ptr / col / alpha / count (the CSR locus), n_dropped.
    """
    L = _lib()
    ip, io, il, ic = _flatten(transcripts)
    hp, ho, hl, hc = _flatten([f for _, f in hits])
    mass = np.asarray([m for m, _ in hits], np.float64)
    rid = np.asarray(ref_ids, np.int32) if ref_ids is not None else None
    inp = LocusInput(len(transcripts), _p(ip), _p(io), _p(il), _p(ic), len(hits), hp.ctypes.data, _p(ho), _p(hl), _p(hc),
                     _p(mass), _p(rid) if rid is not None else None, int(read_len), int(long_read), int(defer_weights))
    h = ctypes.c_void_p()
    rc = L.sbq_build_locus(ctypes.byref(inp), ctypes.byref(model.struct) if model is not None else None, ctypes.byref(h))
    if rc != 0:
        raise api.SbqError(rc, L.sbq_error_string(rc).decode())
    try:
        d = TableDims()
        L.sbq_table_get_dims(h, ctypes.byref(d))
        sl, sr = np.zeros(d.n_seg, np.uint32), np.zeros(d.n_seg, np.uint32)
        L.sbq_table_segments(h, _p(sl), _p(sr))
        isp, isg = np.zeros(d.n_iso + 1, np.int32), np.zeros(max(1, d.n_seg * d.n_iso), np.int32)
        L.sbq_table_iso_segments(h, isp.ctypes.data, isg.ctypes.data)
        cp, cc = np.zeros(d.n_class + 1, np.int32), np.zeros(max(1, d.n_coord), np.int32)
        cnt, cm, nf = np.zeros(max(1, d.n_class), np.int32), np.zeros(max(1, d.n_class), np.float32), np.zeros(max(1, d.n_class), np.int32)
        L.sbq_table_classes(h, cp.ctypes.data, cc.ctypes.data, cnt.ctypes.data, cm.ctypes.data, nf.ctypes.data)
        hcl = np.full(max(1, len(hits)), -1, np.int32)
        L.sbq_table_hit_classes(h, hcl.ctypes.data)
        loc = api.Locus()
        L.sbq_table_locus(h, ctypes.byref(loc))

        def view(ptr, n, dt):
            if n == 0 or not ptr:
                return np.zeros(0, dt)
            return np.ctypeslib.as_array(ctypes.cast(ptr, ctypes.POINTER(np.ctypeslib.as_ctypes_type(dt))), shape=(n,)).copy()
        row_ptr = view(loc.row_ptr, d.n_class + 1, np.int64)
        out = dict(
            segs=[(int(a), int(b)) for a, b in zip(sl, sr)],
            iso_segs=[[int(x) for x in isg[isp[t]:isp[t + 1]]] for t in range(d.n_iso)],
            iso_len=view(loc.iso_len, d.n_iso, np.int32),
            classes=[dict(coords=[int(x) for x in cc[cp[c]:cp[c + 1]]], count=int(cnt[c]), mass=float(cm[c]), nfrag=int(nf[c]))
                     for c in range(d.n_class)],
            row_ptr=row_ptr, col=view(loc.col, d.nnz, np.int32), alpha=view(loc.alpha, d.nnz, np.float64),
            count=cnt[:d.n_class].copy(), n_dropped=d.n_dropped_hits, n_iso=d.n_iso, hit_class=hcl[:len(hits)].copy())
    except BaseException:
        L.sbq_table_free(h)
        raise
    if defer_weights:
        out["table"] = TableHandle(h)      # alpha in `out` is a placeholder (zeros) until the GPU fills it
    else:
        L.sbq_table_free(h)
    return out


def submit_raw(q, transcripts, hits, *, read_len, long_read=False, ref_ids=None):
    """Queue one locus for class assignment ON THE DEVICE (sbq_submit_raw): same inputs as build_locus; the insert model and
    read length come from q.set_insert_model(). The whole class table of the batch is built by q.upload()."""
    L = _lib()
    ip, io, il, ic = _flatten(transcripts)
    hp, ho, hl, hc = _flatten([f for _, f in hits])
    mass = np.asarray([m for m, _ in hits], np.float64)
    rid = np.asarray(ref_ids, np.int32) if ref_ids is not None else None
    inp = LocusInput(len(transcripts), _p(ip), _p(io), _p(il), _p(ic), len(hits), hp.ctypes.data, _p(ho), _p(hl), _p(hc),
                     _p(mass), _p(rid) if rid is not None else None, int(read_len), int(long_read), 1)
    q._chk(L.sbq_submit_raw(q._h, ctypes.byref(inp), None))


def set_raw_mass_mode(q, mode):
    """How q.upload() adds the class masses of raw loci (sbq_set_raw_mass_mode): RAW_MASS_HALVES (default; masses must be
    multiples of 1/2, the atomic sum is exact) or RAW_MASS_ANY (any finite non-negative mass, e.g. the 1/NH fractions of
    multimapped hits, added in the reference's std::set order)."""
    q._chk(_lib().sbq_set_raw_mass_mode(q._h, int(mode)))


def fetch_raw_classes(q, n_hit):
    """Device-built class table of the last raw upload (tests): per hit class id / touched segments (the first 16; ncoord
    saturates at 255, fetch_raw_coords has the full lists), per class representative hit, float mass and member count."""
    L = _lib()
    st = q.stats()
    R = st["n_row"]
    hit_class, ncoord = np.full(max(n_hit, 1), -1, np.int32), np.zeros(max(n_hit, 1), np.uint8)
    coords = np.zeros((max(n_hit, 1), 16), np.uint16)
    rep, mass, nfrag = np.zeros(max(R, 1), np.int64), np.zeros(max(R, 1), np.float32), np.zeros(max(R, 1), np.int32)
    q._chk(L.sbq_fetch_raw_classes(q._h, hit_class.ctypes.data, ncoord.ctypes.data, coords.ctypes.data, rep.ctypes.data, mass.ctypes.data, nfrag.ctypes.data))
    return dict(hit_class=hit_class[:n_hit], ncoord=ncoord[:n_hit], coords=coords[:n_hit], class_rep=rep[:R], class_mass=mass[:R], class_nfrag=nfrag[:R])


def fetch_raw_coords(q, n_hit):
    """Full coordinate lists of the last raw upload (tests): list h of the result is the segments hit h touches."""
    L = _lib()
    off = np.zeros(n_hit + 1, np.int64)
    q._chk(L.sbq_fetch_raw_coords(q._h, off.ctypes.data, None))
    pool = np.zeros(max(int(off[-1]), 1), np.uint16)
    q._chk(L.sbq_fetch_raw_coords(q._h, None, pool.ctypes.data))
    return [pool[off[h]:off[h + 1]] for h in range(n_hit)]
