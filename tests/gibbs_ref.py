"""CPU restatement of the Gibbs sampler (strawberry_b200/csrc/sbq_gibbs.cuh, DESIGN.md "Gibbs posterior samples"), bit for bit.

Every floating-point operation below is one numpy float64 operation on arrays (correctly rounded, never fused), in the order the
device performs it. What is vectorised:
  * running sums of a row are sequential: one step per entry position over every row that is long enough (np.cumsum over the
    flat array would give other bits);
  * column sums use np.add.at, which adds repeated indices in index order, i.e. in ascending row order;
  * a draw's entry is found by a vectorised binary search for the first running sum above the threshold (the device's light rows
    walk the row instead: the sums are non-decreasing, so both pick the same entry);
  * gamma draws run their rejection loops on the set of still-pending isoforms;
  * block_sum<256> is emulated: strided per-thread partials, a 32-lane xor butterfly, then the 8 warp totals in order.
The sample's theta comes out bit for bit; FPKM / TPM are restated with ordinary numpy sums (they are checked to 1e-12).
sm64 is strawberry_b200.synth._sm64, the restatement of sbq_synth.cuh::sm64."""
import numpy as np

from strawberry_b200.synth import _sm64

GIBBS_SALT = 0x9FB21C651E98DF25
GAMMA_SALT = 0xC2B2AE3D27D4EB4F
GIBBS_NT = 256
_M64 = (1 << 64) - 1
LOCUS_ZERO_DENOM, LOCUS_NO_ROWS = 2, 3

LG = (6.666666666666735130e-01, 3.999999999940941908e-01, 2.857142874366239149e-01, 2.222219843214978396e-01,
      1.818357216161805012e-01, 1.531383769920937332e-01, 1.479819860511658591e-01)
LN2_HI, LN2_LO, INV_LN2 = 6.93147180369123816490e-01, 1.90821492927058770002e-10, 1.44269504088896338700e+00
EP = (1.66666666666666019037e-01, -2.77777777770155933842e-03, 6.61375632143793436117e-05, -1.65339022054652515390e-06,
      4.13813679705723846039e-08)


def u64(x):
    return np.asarray(x, np.uint64) if not isinstance(x, int) else np.uint64(x & _M64)


def g_u(h):
    """uniform in (0, 1) from a hash: (2 (h >> 12) + 1) 2^-53, exact"""
    h = np.asarray(h, np.uint64)
    return (((h >> np.uint64(12)) << np.uint64(1)) | np.uint64(1)).astype(np.float64) * 2.0 ** -53


def g_log(x):
    """log of finite x > 0 (sbq_gibbs.cuh::g_log)"""
    x = np.asarray(x, np.float64)
    m, e = np.frexp(x)
    lo = m < 0.70710678118654752440
    m = np.where(lo, m * 2.0, m)
    e = np.where(lo, e - 1, e)
    f = m - 1.0
    s = f / (2.0 + f)
    dk = e.astype(np.float64)
    z = s * s
    w = z * z
    t1 = w * (LG[1] + w * (LG[3] + w * LG[5]))
    t2 = z * (LG[0] + w * (LG[2] + w * (LG[4] + w * LG[6])))
    R = t2 + t1
    hfsq = (0.5 * f) * f
    return dk * LN2_HI - ((hfsq - (s * (hfsq + R) + dk * LN2_LO)) - f)


def _pow2(n):
    return ((np.asarray(n, np.int64) + 1023).astype(np.uint64) << np.uint64(52)).view(np.float64)


def g_exp(x):
    """e^x (sbq_gibbs.cuh::g_exp)"""
    x = np.atleast_1d(np.asarray(x, np.float64))
    over, under = x > 709.782712893383973096, x < -745.133219101941108420
    xs = np.where(over | under, 0.0, x)
    kd = np.floor(xs * INV_LN2 + 0.5)
    k = kd.astype(np.int64)
    hi = xs - kd * LN2_HI
    lo = kd * LN2_LO
    r = hi - lo
    t = r * r
    c = r - t * (EP[0] + t * (EP[1] + t * (EP[2] + t * (EP[3] + t * EP[4]))))
    y = 1.0 - ((lo - (r * c) / (2.0 - c)) - hi)
    big, small = k > 1000, k < -1000
    with np.errstate(over="ignore", under="ignore"):
        out = np.where(big, (y * _pow2(np.where(big, k - 1000, 0))) * _pow2(1000),
                       np.where(small, (y * _pow2(np.where(small, k + 1000, 0))) * _pow2(-1000), y * _pow2(np.clip(k, -1000, 1000))))
    return np.where(over, np.inf, np.where(under, 0.0, out))


class _Streams:
    """the uniform streams of a set of gamma draws: uniform t of draw i is g_u(sm64(key_i + t))"""

    def __init__(self, keys):
        self.key = np.asarray(keys, np.uint64)
        self.t = np.zeros(len(self.key), np.uint64)

    def next(self, idx):
        with np.errstate(over="ignore"):
            h = _sm64(self.key[idx] + self.t[idx])
        self.t[idx] += np.uint64(1)
        return g_u(h)


def _normal(S, idx):
    out = np.empty(len(idx))
    todo = np.arange(len(idx))
    while todo.size:
        ii = idx[todo]
        x = 2.0 * S.next(ii) - 1.0
        y = 2.0 * S.next(ii) - 1.0
        q = x * x + y * y
        ok = (q < 1.0) & (q > 0.0)
        qo = q[ok]
        out[todo[ok]] = x[ok] * np.sqrt((-2.0 * g_log(qo)) / qo)
        todo = todo[~ok]
    return out


def _gamma_ge1(a, S, idx):
    d = a - 1.0 / 3.0
    c = 1.0 / np.sqrt(9.0 * d)
    out = np.empty(len(idx))
    todo = np.arange(len(idx))
    while todo.size:
        ii = idx[todo]
        x, v = np.empty(len(todo)), np.empty(len(todo))
        need = np.arange(len(todo))
        while need.size:
            xx = _normal(S, ii[need])
            vv = 1.0 + c[todo[need]] * xx
            ok = vv > 0.0
            x[need[ok]], v[need[ok]] = xx[ok], vv[ok]
            need = need[~ok]
        v = (v * v) * v
        u = S.next(ii)
        x2 = x * x
        dt = d[todo]
        acc = u < 1.0 - 0.0331 * (x2 * x2)
        rest = ~acc
        acc[rest] = g_log(u[rest]) < 0.5 * x2[rest] + dt[rest] * ((1.0 - v[rest]) + g_log(v[rest]))
        out[todo[acc]] = dt[acc] * v[acc]
        todo = todo[~acc]
    return out


def gamma(a, keys):
    """Gamma(a_i, 1) draws, one per key (sbq_gibbs.cuh::gibbs_gamma)"""
    a = np.atleast_1d(np.asarray(a, np.float64))
    S = _Streams(np.atleast_1d(keys))
    small = a < 1.0
    g = _gamma_ge1(np.where(small, a + 1.0, a), S, np.arange(len(a)))
    si = np.nonzero(small)[0]
    if si.size:
        U = S.next(si)
        g[si] = g[si] * g_exp(g_log(U) / a[si])
    return g


def block_sum(vals, seg_off, nt=GIBBS_NT):
    """block_sum<nt> of every segment [seg_off[l], seg_off[l + 1]) of vals, thread t holding entries t, t + nt, ... in order"""
    L = len(seg_off) - 1
    T = np.diff(seg_off)
    part = np.zeros((L, nt))
    for ch in range(int(-(-T.max() // nt)) if L and T.max() > 0 else 0):
        j = ch * nt + np.arange(nt)
        ok = j[None, :] < T[:, None]
        idx = np.where(ok, seg_off[:-1, None] + j[None, :], 0)
        part = part + np.where(ok, vals[idx], 0.0)
    v = part.reshape(L, nt // 32, 32)
    lane = np.arange(32)
    for o in (16, 8, 4, 2, 1):
        v = v + v[:, :, lane ^ o]
    t = np.zeros(L)
    for w in range(nt // 32):
        t = t + v[:, w, 0]
    return t


def round_key(seed, r):
    with np.errstate(over="ignore"):
        return _sm64(_sm64(np.uint64(int(seed) & _M64) ^ np.uint64(GIBBS_SALT)) + np.uint64(r))


class Chain:
    """The sampler's state for one batch: call rounds() / sample as the device does."""

    def __init__(self, batch, theta_hat, status, seed, prior, row_eps=1e-5, locus_ids=None):
        self.b = b = batch
        lro, lio = np.asarray(b["loc_row_off"], np.int64), np.asarray(b["loc_iso_off"], np.int64)
        rp = np.asarray(b["row_ptr"], np.int64)
        self.col, self.alpha = np.asarray(b["col"], np.int64), np.asarray(b["alpha"], np.float64)
        cnt = np.asarray(b["count"], np.int64)
        L, R = len(lro) - 1, len(rp) - 1
        self.lro, self.lio, self.rp = lro, lio, rp
        self.T = np.diff(lio)
        self.row_locus = np.repeat(np.arange(L), np.diff(lro))
        self.status = np.asarray(status)
        self.sampled = (self.status != LOCUS_NO_ROWS) & (self.status != LOCUS_ZERO_DENOM)
        rlen = np.diff(rp)
        big = np.maximum.reduceat(self.alpha, rp[:-1][rlen > 0]) > row_eps if R else np.zeros(0, bool)
        keep = np.zeros(R, bool)
        keep[rlen > 0] = big
        self.keep = keep & self.sampled[self.row_locus]
        self.n = np.where(self.keep, cnt, 0)
        self.ids = np.arange(L) if locus_ids is None else np.asarray(locus_ids, np.int64)
        C = np.zeros(R + 1, np.int64)
        np.cumsum(cnt, out=C[1:])
        self.dbase = C[:-1] - C[lro[self.row_locus]]          # first draw of every row, counted from its locus' first
        self.nkept = np.bincount(self.row_locus, weights=self.n, minlength=L).astype(np.float64)
        self.ent_row = np.repeat(np.arange(R), rlen)
        self.ent_iso = lio[self.row_locus[self.ent_row]] + self.col
        n_iso = int(lio[-1])
        s = np.zeros(n_iso)
        ke = self.keep[self.ent_row]
        np.add.at(s, self.ent_iso[ke], self.alpha[ke])
        self.s = s
        th = np.asarray(theta_hat, np.float64)
        with np.errstate(divide="ignore", invalid="ignore"):
            self.phi = np.where(s != 0.0, th / np.where(s != 0, s, 1.0), 0.0)
        self.seed, self.prior, self.r = seed, float(prior), 0
        self.theta_hat = th

    def _cum(self):
        w = self.alpha * self.phi[self.ent_iso]
        cum = w.copy()
        rp, rlen = self.rp, np.diff(self.rp)
        for p in range(1, int(rlen.max()) if len(rlen) else 0):
            idx = rp[:-1][rlen > p] + p
            cum[idx] = cum[idx - 1] + w[idx]
        return cum

    def step(self):
        """one round; returns pi"""
        self.r += 1
        rkey = round_key(self.seed, self.r)
        with np.errstate(over="ignore"):
            gk = _sm64(rkey + self.ids.astype(np.uint64))
        cum = self._cum()
        rows = np.nonzero(self.n > 0)[0]
        nd = self.n[rows]
        drow = np.repeat(rows, nd)
        m = np.arange(len(drow)) - np.repeat(np.cumsum(nd) - nd, nd)
        d = (self.dbase[drow] + m).astype(np.uint64)
        with np.errstate(over="ignore"):
            u = g_u(_sm64(gk[self.row_locus[drow]] + d))
        lo, hi = self.rp[drow].copy(), self.rp[drow + 1] - 1
        thr = u * cum[hi]
        while True:
            act = lo < hi
            if not act.any():
                break
            mid = lo + ((hi - lo) >> 1)
            gt = cum[mid] > thr
            hi = np.where(act & gt, mid, hi)
            lo = np.where(act & ~gt, mid + 1, lo)
        c = np.bincount(self.ent_iso[lo], minlength=len(self.s))
        # Dirichlet
        L = len(self.T)
        iso_loc = np.repeat(np.arange(L), self.T)
        j = np.arange(len(self.s)) - self.lio[iso_loc]
        with np.errstate(over="ignore"):
            gkey = _sm64(gk ^ np.uint64(GAMMA_SALT))
            keys = _sm64(gkey[iso_loc] + j.astype(np.uint64))
        live = self.sampled[iso_loc]
        g = np.zeros(len(self.s))
        g[live] = gamma(c[live] + self.prior, keys[live])
        G = block_sum(g, self.lio)
        Gi = G[iso_loc]
        pi = np.where(Gi != 0.0, g / np.where(Gi != 0, Gi, 1.0), 1.0 / self.T[iso_loc])
        with np.errstate(divide="ignore", invalid="ignore"):
            self.phi = np.where(live, np.where(self.s != 0.0, pi / np.where(self.s != 0, self.s, 1.0), 0.0), self.phi)
        self.pi = pi
        return pi

    def theta(self):
        L = len(self.T)
        iso_loc = np.repeat(np.arange(L), self.T)
        return np.where(self.sampled[iso_loc], self.nkept[iso_loc] * self.pi, self.theta_hat)


def epilogue(batch, theta, status, total_mapped_reads, min_iso_frac=0.0, effective_len_norm=0, insert_mean=200.0):
    """FPKM, frac, keep and the TPM of one sample (sbq_kernels.cuh::locus_epilogue_block + fpkm_sum + TPM), to rounding"""
    lio = np.asarray(batch["loc_iso_off"], np.int64)
    T = np.diff(lio)
    iso_loc = np.repeat(np.arange(len(T)), T)
    ln = np.asarray(batch["iso_len"], np.float64)
    rpm = 1e6 / total_mapped_reads
    if effective_len_norm:
        kb = ln - insert_mean
        na = kb < 0
        kb = np.where(na, 1.0, 1e3 / np.where(na, 1.0, kb))
    else:
        na = np.zeros(len(ln), bool)
        kb = 1e3 / ln
    nr = status[iso_loc] == LOCUS_NO_ROWS
    f = np.where(na | nr, 0.0, (theta * rpm) * kb)
    fs = np.bincount(iso_loc, weights=f, minlength=len(T))[iso_loc]
    with np.errstate(divide="ignore", invalid="ignore"):
        fr = np.where(na | nr, 0.0, f / fs)
    kp = np.where(nr, 0, np.where(~(fr < min_iso_frac), np.where(na, -1, 1), 0))
    total = f[kp != 0].sum()
    return dict(fpkm=f, frac=fr, keep=kp, tpm=1e6 * f / total)


def samples(batch, theta_hat, status, seed, n, thin, burn_in, prior, total_mapped_reads, row_eps=1e-5, locus_ids=None, **epi):
    """The n samples of sbq_gibbs: theta [n, n_iso] bit for bit, tpm [n, n_iso] to rounding, status [n, n_loci]"""
    ch = Chain(batch, theta_hat, status, seed, prior, row_eps, locus_ids)
    th, tp = [], []
    for s in range(n):
        target = burn_in + (s + 1) * thin
        while ch.r < target:
            ch.step()
        t = ch.theta()
        th.append(t)
        tp.append(epilogue(batch, t, np.asarray(status), total_mapped_reads, **epi)["tpm"])
    return dict(theta=np.array(th), tpm=np.array(tp), status=np.repeat(np.asarray(status)[None, :], n, 0))
