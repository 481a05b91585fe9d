"""Agreement rules between an implementation of the small dense routines (the host build or the device
harness, both batched: inputs [N][...]) and the 50-digit reference (tests/smallref.py).

Discrete outcomes must equal the reference's wherever the margin exceeds its rounding bound; inside
the band either outcome is accepted, provided the implementation agrees with the other build or with
numpy (the oracle).  Each check returns a report (problems, band count, worst error over its bound)
and a list of violations."""
import ctypes as C
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, os.path.join(ROOT, "arboris-python_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import smallref as ref  # noqa: E402

EPS = ref.EPS
ST_NOROOT, ST_NOCONV = ref.ST_EIG_NOROOT, ref.ST_EIG_NOCONV
BAND_IMAG = 1e-6     # |Im| / ||B|| of a pair: a float solver may see it on the axis (a double root splits by sqrt(eps))
BAND_ZERO = 1e-10    # |lambda| / ||B|| of the real eigenvalue nearest 0, against the s <= 0 inclusion
BAND_GAP = 1e-6      # relative separation of s below which s is not "well separated"
BAND_CLAMP = 1e-10   # |s + 1e10| / 1e10


class Report(object):
    def __init__(self, name):
        self.name, self.n, self.band, self.worst, self.bad = name, 0, 0, 0., []
        self.illcond = 0     # determined outcome, but a value (s) too ill-conditioned to compare
        self.band_idx = []   # the problems counted in the band (check_contact)

    def ratio(self, err, bound, what, k):
        r = err / bound if bound > 0 else (0. if err == 0 else np.inf)
        self.worst = max(self.worst, r)
        if not r <= 1.:
            self.bad.append((k, what, err, bound))

    def fail(self, k, what, *info):
        self.bad.append((k, what) + info)

    def __str__(self):
        return "%-22s problems %4d  band %3d  ill-conditioned %3d  worst err/bound %.3g  violations %d" % (
            self.name, self.n, self.band, self.illcond, self.worst, len(self.bad))


# ---------------------------------------------------------------------------------------------------
# host build, batched like the device harness
# ---------------------------------------------------------------------------------------------------
class HostLib(object):
    def __init__(self):
        sys.path.insert(0, os.path.join(HERE, "hosttest"))
        import harness
        self.L = L = harness.lib()
        dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
        L.ht_softfinger_solve.argtypes = [dp, dp, dp, C.c_double, C.c_double, dp, C.c_double, dp, dp, ip]
        L.ht_softfinger_solve.restype = C.c_int
        L.ht_sliding_root.argtypes = [dp, dp, C.c_double, dp, ip]
        L.ht_poly6_fast.argtypes = [dp, dp]
        L.ht_poly6_slow.argtypes = [dp, dp]
        L.ht_poly6_positive.argtypes = [dp]
        L.ht_certify.argtypes = [dp, C.c_double]
        L.ht_eig6.argtypes = [dp, dp, dp]
        L.ht_pinv.argtypes = [C.c_int, dp, dp]
        L.ht_inv_cond4.argtypes = [dp, dp]
        L.ht_inv_cond4.restype = C.c_double
        L.ht_solve4.argtypes = [dp, dp, dp]
        L.ht_exp.argtypes = [dp, dp]
        L.ht_zaligned.argtypes = [dp, dp, ip]
        L.ht_collide.argtypes = [C.c_int, dp, dp, dp, dp, dp, ip]
        L.ht_collide.restype = C.c_double
        L.ht_fastroot_fail.restype = C.c_long
        L.ht_fastroot_hits.restype = C.c_long
        self.dp, self.ip = dp, ip

    def _d(self, a):
        return np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(self.dp)

    def softfinger_solve(self, v, A, P, sdist, mu, eps, dt, f0):
        n = len(v)
        F, DF, BR, ST = np.array(f0, np.float64).copy(), np.zeros((n, 4)), np.zeros(n, np.int32), np.zeros(n, np.int32)
        for k in range(n):
            f = np.ascontiguousarray(F[k]); df = np.zeros(4); st = C.c_int(0)
            BR[k] = self.L.ht_softfinger_solve(self._d(v[k]), self._d(A[k]), self._d(P[k]), float(sdist[k]), float(mu[k]),
                                               self._d(eps[k]), float(dt), f.ctypes.data_as(self.dp),
                                               df.ctypes.data_as(self.dp), C.byref(st))
            F[k], DF[k], ST[k] = f, df, st.value
        return F, DF, BR, ST

    def sliding_root(self, A, alpha, mu, coop=0):
        n = len(A)
        S, FO, OK = np.zeros(n), np.zeros(n, np.int32), np.zeros(n, np.int32)
        for k in range(n):
            s, fo = C.c_double(0.), C.c_int(0)
            OK[k] = self.L.ht_sliding_root(self._d(A[k]), self._d(alpha[k]), float(mu[k]), C.byref(s), C.byref(fo))
            S[k], FO[k] = s.value, fo.value
        return S, FO, OK

    def poly6(self, p, x):
        n = len(p)
        out = [np.zeros(n, np.int32), np.zeros(n), np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n),
               np.zeros(n, np.int32)]
        self.recovered = np.zeros(n, bool)
        for k in range(n):
            pk = np.ascontiguousarray(p[k], np.float64)
            r = C.c_double(0.)
            before = self.L.ht_fastroot_fail(5)
            out[0][k] = self.L.ht_poly6_fast(pk.ctypes.data_as(self.dp), C.byref(r))
            self.recovered[k] = self.L.ht_fastroot_fail(5) > before
            out[1][k] = r.value
            out[2][k] = self.L.ht_poly6_positive(pk.ctypes.data_as(self.dp))
            r2 = C.c_double(0.)
            out[3][k] = self.L.ht_poly6_slow(pk.ctypes.data_as(self.dp), C.byref(r2))
            out[4][k] = r2.value if out[3][k] else 0.
            out[5][k] = self.L.ht_certify(pk.ctypes.data_as(self.dp), float(x[k]))
        return tuple(out)

    def eig6(self, A):
        n = len(A)
        WR, WI, OK = np.zeros((n, 6)), np.zeros((n, 6)), np.zeros(n, np.int32)
        for k in range(n):
            wr, wi = np.zeros(6), np.zeros(6)
            OK[k] = self.L.ht_eig6(self._d(A[k]), wr.ctypes.data_as(self.dp), wi.ctypes.data_as(self.dp))
            WR[k], WI[k] = wr, wi
        return WR, WI, OK

    def pinv(self, A):
        A = np.asarray(A)
        m = A.shape[1]
        out = np.zeros(A.shape)
        for k in range(len(A)):
            o = np.zeros((m, m))
            self.L.ht_pinv(m, self._d(A[k]), o.ctypes.data_as(self.dp))
            out[k] = o
        return out

    def inv_cond4(self, A):
        out, cond = np.zeros((len(A), 4, 4)), np.zeros(len(A))
        for k in range(len(A)):
            o = np.zeros((4, 4))
            cond[k] = self.L.ht_inv_cond4(self._d(A[k]), o.ctypes.data_as(self.dp))
            out[k] = o
        return out, cond

    def solve4(self, A, b):
        X, OK = np.zeros((len(A), 4)), np.zeros(len(A), np.int32)
        for k in range(len(A)):
            x = np.zeros(4)
            OK[k] = self.L.ht_solve4(self._d(A[k]), self._d(b[k]), x.ctypes.data_as(self.dp))
            X[k] = x
        return X, OK

    def se3_exp(self, tw):
        out = np.zeros((len(tw), 12))
        for k in range(len(tw)):
            o = np.zeros(12)
            self.L.ht_exp(self._d(tw[k]), o.ctypes.data_as(self.dp))
            out[k] = o
        return out

    def zaligned(self, z):
        R, I = np.zeros((len(z), 3, 3)), np.zeros((len(z), 3), np.int32)
        for k in range(len(z)):
            r, i = np.zeros(9), np.zeros(3, np.int32)
            self.L.ht_zaligned(self._d(z[k]), r.ctypes.data_as(self.dp), i.ctypes.data_as(self.ip))
            R[k], I[k] = r.reshape(3, 3), i
        return R, I

    def collide(self, pair, cd, H0, H1):
        n = len(pair)
        SD, C0, C1, ZI = np.zeros(n), np.zeros((n, 12)), np.zeros((n, 12)), np.zeros((n, 3), np.int32)
        for k in range(n):
            c0, c1, zi = np.zeros(12), np.zeros(12), np.zeros(3, np.int32)
            SD[k] = self.L.ht_collide(int(pair[k]), self._d(cd[k]), self._d(H0[k]), self._d(H1[k]),
                                      c0.ctypes.data_as(self.dp), c1.ctypes.data_as(self.dp), zi.ctypes.data_as(self.ip))
            C0[k], C1[k], ZI[k] = c0, c1, zi
        return SD, C0, C1, ZI


# ---------------------------------------------------------------------------------------------------
# references (computed once per family and process)
# ---------------------------------------------------------------------------------------------------
_cache = {}


def cached(key, fn):
    if key not in _cache:
        _cache[key] = fn()
    return _cache[key]


def contact_refs(fam):
    return [ref.softfinger(fam["v"][k], fam["A"][k], fam["P"][k], fam["sdist"][k], fam["mu"][k], fam["eps"][k],
                           fam["dt"], fam["f0"][k]) for k in range(len(fam["v"]))]


def oracle_softfinger(fam):
    """the numpy oracle's SoftFingerContact.solve on every problem: (branch, force, increment, slide);
    None for a family whose P is not pinv(A) (the oracle computes pinv(A) itself)"""
    if not fam.get("P_is_pinv", True):
        return None
    from oracle.arboris_oracle import softfinger_solve
    out = []
    for k in range(len(fam["v"])):
        vel = fam["v"][k]
        out.append(softfinger_solve(vel, fam["A"][k], fam["f0"][k].copy(), fam["sdist"][k], fam["mu"][k],
                                    fam["eps"][k], fam["dt"]))
    return out


def _slide_decided(sl):
    """True when found / not found and the clamp are determined outside the rounding band: either a real
    eigenvalue lies below -BAND_ZERO with no real neighbour within BAND_IMAG (a root no rounding removes),
    or no eigenvalue can become admissible (none within BAND_ZERO of 0 -- unless the problem is exact --,
    no pair within BAND_IMAG of the axis, no admissible one in a near-double pair).  Relative to the
    spectral radius."""
    if abs(sl.get("clamp", 1.)) <= BAND_CLAMP:
        return False
    eg = sl["eigs"]
    real = [r for r, i in eg if i == 0.]
    exact = sl.get("exact", False)

    def single(r):
        return all(abs(r - q) > BAND_IMAG for q in real if q is not r) and sum(q == r for q in real) == 1

    if any(r < -BAND_ZERO and single(r) for r in real):
        return True
    if any(abs(r) <= BAND_ZERO for r in real) and not exact:
        return False
    if any(i != 0. and abs(i) <= BAND_IMAG and r <= BAND_ZERO for r, i in eg):
        return False
    return all(single(r) for r in real if r <= 0.)


def check_contact(name, fam, res, refs, alt=()):
    """res = (f, df, br, status) of one implementation; alt: (br, f) pairs of other implementations
    (the other build, the oracle) for the band rule."""
    F, DF, BR, ST = res
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        decided = True
        if not (abs(r["rel"]) > r["rel_bound"] or r["rel_bound"] == 0.):
            decided = False
        elif r["br"] != 1 and "stat" in r and not (abs(r["stat"]) > r["stat_bound"] or r["stat_bound"] == 0.):
            decided = False
        elif r["br"] == 3 and not _slide_decided(r["slide"]):
            decided = False
        if ST[k] & ST_NOCONV:
            rep.fail(k, "EIG_NOCONV")
        if not decided:
            rep.band += 1
            rep.band_idx.append(k)
            if not any(int(BR[k]) == int(b[k]) for b, f in alt) and int(BR[k]) != r["br"]:
                rep.fail(k, "band branch agrees with nothing", int(BR[k]), r["br"], [int(b[k]) for b, f in alt])
            continue
        if int(BR[k]) != r["br"]:
            rep.fail(k, "branch", int(BR[k]), r["br"], r["rel"], r.get("stat"))
            continue
        f0 = fam["f0"][k]
        if not np.array_equal(F[k] - f0, DF[k]) and not np.allclose(F[k] - f0, DF[k], rtol=4 * EPS, atol=0):
            rep.fail(k, "df != f - f0")
        if r["br"] == 1:
            if F[k].any():
                rep.fail(k, "release force not zero")
            continue
        fr = r["f"]
        if r["br"] == 2:
            P = fam["P"][k]
            rhs = np.abs(fam["v"][k]) + np.array([0, 0, 0, abs(fam["sdist"][k] / fam["dt"])])
            scale = np.abs(f0) + np.abs(P).dot(rhs)
            rep.ratio(float(np.max(np.abs(F[k] - fr) / np.maximum(scale, 1e-300))), 16 * EPS, "static force", k)
            continue
        sl = r["slide"]
        if "alt" in sl and not (sl["s_used"] <= -ref.CLAMP and sl["alt"]["s_used"] <= -ref.CLAMP and
                                not sl["alt"]["noroot"]):
            # s sits in a near-double real pair: the solve may take the next admissible eigenvalue instead;
            # either solve, with its status, is accepted (the clamp, when both are beyond it, is decided)
            rep.band += 1
            rep.band_idx.append(k)
            ok = []
            for fc, c2, noroot in ((r["f"], sl["cond2"], False), (sl["alt"]["f"], sl["alt"]["cond2"], sl["alt"]["noroot"])):
                e = np.abs(F[k] - fc).max() / max(np.abs(fc).max(), 1e-300)
                ok.append(bool(ST[k] & ST_NOROOT) == noroot and e <= c2 * 1e-6)
            if not any(ok):
                rep.fail(k, "pair: force agrees with neither admissible minimum")
            continue
        if bool(ST[k] & ST_NOROOT) != (not sl["found"]):
            rep.fail(k, "EIG_NOROOT", int(ST[k]), sl["found"])
        if sl["found"] and sl["gap"] <= BAND_GAP and sl["s_used"] > -ref.CLAMP:
            rep.illcond += 1       # s itself is ill-conditioned: the force is not compared
            continue
        # the solve alone is within 100 eps cond; s carries the error the s rule allows, which enters
        # through the matrix (A - s diag(eps^-2)): cond * |ds| / ||M|| more
        Anorm = np.abs(fam["A"][k]).sum(axis=0).max()
        s = sl["s_used"]
        ds = 1e-12 * abs(s) + 1e-14 * Anorm if sl["found"] and s > -ref.CLAMP else 0.
        Mn = np.abs(fam["A"][k] - np.diag(np.r_[s / fam["eps"][k]**2, 0.])).sum(axis=0).max()
        bound = sl["cond2"] * (100 * EPS + ds / Mn)
        rep.ratio(float(np.abs(F[k] - fr).max() / max(np.abs(fr).max(), 1e-300)), bound, "sliding force", k)
    return rep


def slide_refs(fam):
    out = []
    for k in range(len(fam["A"])):
        sl = ref.sliding_root(fam["A"][k], fam["alpha"][k], fam["mu"][k])
        sl["exact"] = _exact_triangular(fam["A"][k], fam["alpha"][k], fam["mu"][k])
        if sl["found"]:
            sl["clamp"] = float((sl["s"] + ref.CLAMP) / ref.CLAMP)
        out.append(sl)
    return out


def _exact_triangular(A, alpha, mu=None):
    """Y_c = 0, beta along e0, a diagonal Y_t of short dyadics, y_n, mu, alpha_n powers of two and the
    scale sigma = |beta_0 / a| + sum |y_i| a power of two: every coefficient of the structured sextic
    is then exact, and a zero eigenvalue is zero in float64 too."""
    A, alpha = np.asarray(A), np.asarray(alpha)
    off = A - np.diag(np.diag(A))
    if off.any() or alpha[1] or alpha[2]:
        return False

    def p2(x):
        return x != 0 and np.frexp(abs(x))[0] == 0.5

    def short(x):
        return float(x * 2.0**40) == int(x * 2.0**40)

    d = np.diag(A)
    if not (p2(d[3]) and p2(alpha[3]) and (mu is None or p2(mu)) and all(short(x) for x in d[:3]) and short(alpha[0])):
        return False
    a = (mu if mu is not None else 1.) / d[3] * alpha[3]
    return p2(abs(alpha[0] / a) + np.abs(d[:3]).sum()) or not alpha[0]


def check_sliding_root(name, fam, res, refs, alt=()):
    S, FO, OK = res
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        if not OK[k]:
            rep.fail(k, "structured path refused a finite eps = 1 problem")
            continue
        if not _slide_decided(r):
            rep.band += 1
            if bool(FO[k]) != r["found"] and not any(bool(a[1][k]) == bool(FO[k]) for a in alt):
                rep.fail(k, "band found agrees with nothing")
            continue
        if bool(FO[k]) != r["found"]:
            rep.fail(k, "found", int(FO[k]), r["found"], r["zero"], r["imag"])
            continue
        if not r["found"]:
            continue
        sm = float(r["s"])
        if sm < -ref.CLAMP * (1. + 1e-6):       # what the solve uses is the clamp
            if not S[k] < -ref.CLAMP:
                rep.fail(k, "beyond the clamp", S[k], sm)
            continue
        if r["gap"] <= BAND_GAP:
            rep.illcond += 1
            continue
        Anorm = np.abs(fam["A"][k]).max()
        rep.ratio(abs(S[k] - sm), 1e-12 * abs(sm) + 1e-14 * Anorm, "s", k)
    return rep


def poly_refs(fam):
    import mpmath as mp
    out = []
    with mp.workdps(ref.DPS):
        for p in fam["p"]:
            c = [mp.mpf(1)] + [mp.mpf(float(x)) for x in p[::-1]]
            rts = mp.polyroots(c, maxsteps=200, extraprec=200)
            real = sorted(float(mp.re(r)) for r in rts if abs(mp.im(r)) < mp.mpf(10)**-30)
            imag = min([abs(float(mp.im(r))) for r in rts if abs(mp.im(r)) >= mp.mpf(10)**-30] or [np.inf])
            out.append(dict(real=real, imag=imag, largest=real[-1] if real else None,
                            nonneg=[t for t in real if t >= 0]))
    return out


def check_poly(name, fam, res, refs):
    fast_ok, fast_root, positive, slow_n, slow_root, certify = res
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        if fast_ok[k]:
            if r["largest"] is None:
                rep.fail(k, "fast root for a polynomial without real roots")
            else:
                rep.ratio(abs(fast_root[k] - r["largest"]), 1e-10 * max(1., abs(r["largest"])), "fast root", k)
        if positive[k] and r["nonneg"]:
            rep.fail(k, "positivity proven with a root t >= 0", r["nonneg"])
        if slow_n[k]:
            if not r["nonneg"]:
                rep.fail(k, "slow isolation found a root t >= 0 that does not exist")
            else:
                rep.ratio(abs(slow_root[k] - r["nonneg"][-1]), 1e-7 * max(1., r["nonneg"][-1]), "slow root", k)
        elif r["nonneg"] and r["nonneg"][-1] > 1e-6 and r["imag"] > 1e-6:
            rep.fail(k, "slow isolation missed a root", r["nonneg"])
    return rep


def pinv_refs(fam):
    return [ref.pinv(a) for a in fam["A"]]


def check_pinv(name, fam, out, refs, alt=()):
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        fr = r["pinv"]
        sc = max(np.abs(fr).max(), 1e-300)
        err = np.abs(out[k] - fr).max() / sc
        bound = 100 * EPS * r["cond"]
        if r["cut_margin"] <= 16 * EPS:
            rep.band += 1
            ok = err <= bound or any(np.abs(out[k] - a[k]).max() <= 100 * EPS * max(np.abs(a[k]).max(), 1e-300) *
                                     r["cond"] for a in alt)
            if not ok:
                rep.fail(k, "band pinv agrees with nothing", err)
            continue
        if not fr.any():
            if out[k].any():
                rep.fail(k, "pinv of zero not zero")
            continue
        rep.ratio(err, bound, "pinv", k)
    return rep


def check_cond(name, fam, cond, refs_cond):
    rep = Report(name)
    for k, c in enumerate(refs_cond):
        rep.n += 1
        if abs(c / 1e12 - 1.) <= 64 * EPS * c:
            rep.band += 1
            continue
        if (cond[k] < 1e12) != (c < 1e12):
            rep.fail(k, "cond_1 < 1e12 decision", cond[k], c)
    return rep


def check_solve(name, fam, res, refs, singular=False):
    X, OK = res
    rep = Report(name)
    for k, (x, c) in enumerate(refs):
        rep.n += 1
        if singular:
            if OK[k]:
                rep.fail(k, "solve_small returned true on an exact zero pivot")
            continue
        if not OK[k]:
            rep.fail(k, "solve_small returned false")
            continue
        rep.ratio(np.abs(X[k] - x).max() / np.abs(x).max(), 100 * EPS * c, "solve", k)
    return rep


def eig_ref(A):
    r = ref.eig6(A)
    kc = ref.eig_cond(A)
    # condition number of each sorted reference eigenvalue (nearest match)
    r["kappa"] = [min(kc, key=lambda e: abs(e[0] - v))[1] for v in r["vals"]]
    r["norm"] = float(np.linalg.norm(A, 2))
    return r


def check_eig(name, fam, res, refs):
    """sorted eigenvalues within 1e-8 max(1, |lambda|max) -- corrected for ill-conditioned eigenvalues: a
    backward-stable solver moves an eigenvalue by up to its condition number times eps ||A|| (clustered
    roots of a companion matrix have condition numbers of 1e8 and more), so the tolerance is at least
    100 eps kappa ||A||_2; and for multiple eigenvalues: a cluster of
    m eigenvalues of a defective matrix is only determined to (eps ||A||^m)^(1/m) (its mean is well
    conditioned, its members are not), so their tolerance is 30 eps^(1/m) times the scale; the count of real
    eigenvalues must match outside the band (a pair within BAND_IMAG of the axis, or two real ones within
    BAND_IMAG of each other)."""
    WR, WI, OK = res
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        if not OK[k]:
            rep.fail(k, "EIG_NOCONV")
            continue
        got = WR[k] + 1j * WI[k]
        want = r["vals"]
        lam = max(1., np.abs(want).max())
        kap = r.get("kappa")
        used = np.zeros(6, bool)
        worst = 0.
        for g in sorted(got, key=lambda z: (z.real, z.imag)):
            d = np.abs(want - g)
            d[used] = np.inf
            j = int(np.argmin(d))
            used[j] = True
            m = int((np.abs(want - want[j]) <= 1e-5 * lam).sum())
            tol = max(1e-8, 30 * EPS**(1. / m)) * lam if m > 1 else 1e-8 * lam
            if kap is not None and np.isfinite(kap[j]):
                tol = max(tol, 100 * EPS * kap[j] * r["norm"])
            worst = max(worst, d[j] / tol)
        rep.worst = max(rep.worst, worst)
        if worst > 1.:
            rep.fail(k, "eigenvalues", worst)
        if r["imag_margin"] <= BAND_IMAG or r["real_gap"] <= BAND_IMAG:
            rep.band += 1
        elif int((WI[k] == 0).sum()) != r["nreal"]:
            rep.fail(k, "real count", int((WI[k] == 0).sum()), r["nreal"])
    return rep


def check_se3(name, fam, out, refs):
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        H = r["H"]
        # R within 4 ulp of its terms: I + sc w^ + cc w^2 sums terms of magnitude 1 + |sc| t + |cc| t^2, not 1
        # (the rule "4 ulp" holds as stated only for |w| <~ 1; at |w| = 50 the terms are O(1) each, but rounded
        # at the magnitude of w^ and w^2 before they cancel)
        t = np.linalg.norm(fam["tw"][k][:3])
        # (plus an ulp of 1 for sin, cos and 1 - cos, each rounded at the magnitude of 1)
        mag = 2. + abs(np.sin(t)) + t * t * (0.5 if t < 1e-3 else (1. - np.cos(t)) / t**2)
        rep.ratio(np.abs(out[k][:9] - H[:9]).max(), 4 * EPS * mag, "R", k)
        rep.ratio(np.abs(out[k][9:] - H[9:]).max(), 1e-13 * max(1., np.abs(H[9:]).max()), "p", k)
    return rep


def check_zaligned(name, fam, res, refs):
    R, I = res
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        if list(I[k]) != list(r["idx"]):
            rep.fail(k, "argsort", list(I[k]), list(r["idx"]))
        rep.ratio(np.abs(R[k] - r["R"]).max(), 4 * EPS, "R", k)
    return rep


def check_collide(name, fam, res, refs):
    SD, C0, C1, ZI = res
    rep = Report(name)
    for k, r in enumerate(refs):
        rep.n += 1
        if list(ZI[k]) != list(r["idx"]):
            rep.fail(k, "zaligned argsort", list(ZI[k]), list(r["idx"]))
        scale = np.abs(fam["H0"][k][9:]).max() + np.abs(fam["H1"][k][9:]).max() + fam["cd"][k][41] + fam["cd"][k][42]
        rep.ratio(abs(SD[k] - r["sdist"]), 4 * EPS * scale, "sdist", k)
        rep.ratio(np.abs(C0[k][:9] - r["Hc0"][:9]).max(), 4 * EPS, "R", k)
        for c, h in ((C0[k], r["Hc0"]), (C1[k], r["Hc1"])):
            rep.ratio(np.abs(c[9:] - h[9:]).max(), 1e-13 * max(1., np.abs(h[9:]).max(), scale), "position", k)
    return rep
