"""High-precision reference (mpmath, 50 digits) of the small dense routines and of the soft-finger
contact solve that the Gauss-Seidel kernels run per contact visit.

Every float64 input is taken exactly.  Every discrete decision returns its MARGIN -- the signed
distance to the decision boundary, positive on the side the code takes when the test is true -- and
a rounding BOUND: the float64 evaluation of the margin cannot be off by more than the bound, so an
outcome with |margin| > bound is determined and must be reproduced bit-for-bit by any correct
float64 implementation (host, device, with or without FMA contraction).  Within the bound either
outcome is acceptable; the tests count such problems per family.

The knobs RCOND, SERIES_SWITCH and INCLUSIVE_ZERO are module constants so that a test can move
them and show that the families targeting each boundary detect the change."""
import math

import mpmath as mp
import numpy as np

DPS = 50
EPS = 2.0**-52
RCOND = 1e-15              # numpy.linalg.pinv's default cut, sigma_j > RCOND sigma_max
SERIES_SWITCH = 1e-3       # twist_exp: Rodrigues for |w| >= SERIES_SWITCH, series below
INCLUSIVE_ZERO = True      # SoftFingerContact.solve keeps real eigenvalues s <= 0 (False: s < 0)
CLAMP = 1e10
PAIR_BAND = 1e-6           # real eigenvalues closer than this (over the spectral radius) may merge into a pair

ST_EIG_NOROOT = 4
ST_EIG_NOCONV = 8


def _m(x):
    return mp.mpf(float(x))


def _mat(a):
    a = np.asarray(a, dtype=np.float64)
    return mp.matrix([[mp.mpf(float(x)) for x in row] for row in a])


def _f(x):
    return float(mp.re(x)) if isinstance(x, mp.mpc) else float(x)


def _representable(x):
    return mp.mpf(float(x)) == x


# -------------------------------------------------------------------------------------------------
# eigenvalues
# -------------------------------------------------------------------------------------------------
def eigvals(B):
    """eigenvalues of a real matrix at DPS digits, with the real ones identified (|Im| below
    1e-25 of the spectral radius: exact real eigenvalues come out with |Im| of 1e-48 .. 1e-29)."""
    a = np.abs(np.asarray(B, np.float64))
    nz = a[a > 0]
    # a badly balanced matrix needs the digits of its dynamic range on top (mp.eig does not balance)
    dps = DPS + (int(np.log10(nz.max() / nz.min())) if nz.size else 0)
    with mp.workdps(dps):
        M = _mat(B)
        ev = mp.eig(M, left=False, right=False)
        ev = ev[0] if isinstance(ev, tuple) else ev
        # (relative to the spectral radius, not ||B||: of a badly balanced matrix ||B|| is many orders larger)
        scale = max(max(abs(mp.mpc(e)) for e in ev), mp.mpf(1e-300))
        out = []
        for e in ev:
            e = mp.mpc(e)
            out.append((mp.re(e), mp.im(e) if abs(mp.im(e)) > mp.mpf(1e-25) * scale else mp.mpf(0)))
        return out, scale


def eig_cond(B):
    """condition numbers 1 / |y^H x| (unit left and right eigenvectors) of the eigenvalues, in the order
    of mp.eig, with the eigenvalues; inf for a (numerically) defective one."""
    with mp.workdps(DPS):
        E, EL, ER = mp.eig(_mat(B), left=True, right=True)
        out = []
        for k in range(len(E)):
            x = ER[:, k]; y = EL[k, :]
            d = abs(sum(y[j] * x[j] for j in range(len(E)))) / (mp.norm(x) * mp.norm(y))
            out.append((complex(E[k]), float(1 / d) if d > mp.mpf(10)**-40 else float("inf")))
        return out


def eig6(B):
    """eigenvalues of a 6x6 as a sorted complex numpy array, the number of real ones, and the
    margin of that count: the smallest |Im| of a complex pair and the smallest gap between two real
    eigenvalues (either small means a float64 solver may legitimately count differently)."""
    ev, scale = eigvals(B)
    with mp.workdps(DPS):
        scale = max(max(abs(mp.mpc(r, i)) for r, i in ev), mp.mpf(1e-300))
        vals = np.array([complex(float(r), float(i)) for r, i in ev])
        real = [r for r, i in ev if i == 0]
        imag_margin = min([abs(i) for r, i in ev if i != 0] or [mp.inf]) / scale
        rs = sorted(real)
        gap = min([rs[k + 1] - rs[k] for k in range(len(rs) - 1)] or [mp.inf]) / scale
        return dict(vals=np.sort_complex(vals), nreal=len(real), imag_margin=float(imag_margin),
                    real_gap=float(gap), scale=float(scale))


# -------------------------------------------------------------------------------------------------
# SoftFingerContact.solve (constraints.py:780-836)
# -------------------------------------------------------------------------------------------------
def sliding_matrix(A, alpha, mu, eps):
    """B of constraints.py:807-821, with the reference's scalar inner products (Y_c, beta, b are
    1-D: every dot(x, y.T) is a scalar that broadcasts over a 3x3 block).  mp matrix."""
    A = [[_m(x) for x in row] for row in np.asarray(A)]
    al = [a if isinstance(a, mp.mpf) else _m(a) for a in alpha]
    mu, e2 = _m(mu), [_m(e)**2 for e in eps]
    Yc = [A[0][3], A[1][3], A[2][3]]
    yn = A[3][3]
    beta = [al[i] - al[3] / yn * Yc[i] for i in range(3)]
    a = mu / yn * al[3]
    b = [mu / yn * Yc[i] for i in range(3)]
    ycyc = sum(y * y for y in Yc)
    betab = sum(beta[i] * b[i] for i in range(3))
    bb = sum(beta[i] * beta[i] for i in range(3))
    bdotb = sum(x * x for x in b)
    B = mp.zeros(6, 6)
    for i in range(3):
        for j in range(3):
            yhat = A[i][j] - ycyc / yn
            B[3 + i, 3 + j] = e2[i] * yhat
            B[i, j] = e2[i] * (yhat + 2 / a * betab)
        B[i, 3 + i] = -(e2[i] * (bb / a**2))
        B[3 + i, i] = e2[i] * bdotb - 1
    return B


def sliding_root(A, alpha, mu, eps=(1., 1., 1.)):
    """The admissible root of the sliding branch: s = min real eigenvalue <= 0 of B (constraints.py:
    825-830), or none.  Margins: 'imag' -- smallest |Im| of a complex pair over ||B|| (a pair that
    close to the axis may come out real from a float solver); 'zero' -- smallest |lambda| over ||B||
    among the real eigenvalues (the s <= 0 inclusion); 'gap' -- distance from s to the nearest other
    eigenvalue over max(|s|, 1e-300) (relative separation of the chosen root); 'clamp' -- (s + 1e10)/1e10.
    ||B|| here is the spectral radius."""
    with mp.workdps(DPS):
        B = sliding_matrix(A, alpha, mu, eps)
        ev = mp.eig(B, left=False, right=False)
        ev = ev[0] if isinstance(ev, tuple) else ev
        pairs = [(mp.re(mp.mpc(e)), mp.im(mp.mpc(e))) for e in ev]
        # margins relative to the spectral radius: the structured path works on the sextic scaled by it
        scale = max(max(abs(mp.mpc(r, i)) for r, i in pairs), mp.mpf(1e-300))
        real = [r for r, i in pairs if abs(i) <= mp.mpf(1e-25) * scale]
        cplx = [(r, i) for r, i in pairs if abs(i) > mp.mpf(1e-25) * scale]
        adm = [r for r in real if (r <= 0 if INCLUSIVE_ZERO else r < 0)]
        found = len(adm) > 0
        s = min(adm) if found else None
        imag = min([abs(i) for r, i in cplx] or [mp.inf]) / scale
        zero = min([abs(r) for r in real] or [mp.inf]) / scale
        gap = mp.inf
        if found:
            others = [abs(mp.mpc(r, i) - s) for r, i in pairs]
            others.remove(min(others))
            gap = min(others) / max(abs(s), mp.mpf(1e-300))
        return dict(found=found, s=s, imag=float(imag), zero=float(zero), gap=float(gap),
                    scale=float(scale), nreal=len(real),
                    eigs=[(float(r / scale), float(i / scale) if abs(i) > mp.mpf(1e-25) * scale else 0.)
                          for r, i in pairs])


def _rel_bound_release(v, A, sdist, dt, f0):
    """rounding bound of sdist + dt (v3 - A[3,:] f0): 0 when f0 = 0 and dt is a power of two (then
    dt v3 is exact and the one rounded sum keeps its sign, fused or not); else 16 eps times the
    magnitudes of the terms."""
    if not np.any(f0) and math.frexp(dt)[0] == 0.5:
        return 0.
    return 16 * EPS * (abs(sdist) + dt * abs(v[3]) + dt * float(np.abs(A[3] * f0).sum()))


def softfinger(v, A, P, sdist, mu, eps, dt, f0):
    """SoftFingerContact.solve with P = pinv(A) given (as the kernels receive it).  Returns the
    branch (1 separating, 2 static, 3 sliding), the new force, the status bits and the margins:
      release: sdist + dt vnf3 (> 0: separating) and its bound;
      static:  rr^2 - lhs (>= 0: static) and its bound;
      the sliding_root() record and 'clamp' for branch 3."""
    v, A, P, eps, f0 = (np.asarray(x, np.float64) for x in (v, A, P, eps, f0))
    with mp.workdps(DPS):
        Am = [[_m(x) for x in row] for row in A]
        Pm = [[_m(x) for x in row] for row in P]
        fm = [_m(x) for x in f0]
        vm = [_m(x) for x in v]
        sd, dtm, mum = _m(sdist), _m(dt), _m(mu)
        vnf = [vm[i] - sum(Am[i][j] * fm[j] for j in range(4)) for i in range(4)]
        rel = sd + dtm * vnf[3]
        out = dict(rel=float(rel), rel_bound=_rel_bound_release(v, A, sdist, dt, f0), status=0)
        if rel > 0:
            out.update(br=1, f=np.zeros(4), stat=None)
            return out
        sdt = float(sdist / dt)          # the kernels take sdist / dt rounded (computed once per step)
        rhs = [vm[0], vm[1], vm[2], vm[3] + _m(sdt)]
        terms = [[-Pm[i][j] * rhs[j] for j in range(4)] for i in range(4)]
        nf = [fm[i] + sum(terms[i]) for i in range(4)]
        em = [_m(e) for e in eps]
        lhs = sum((nf[i] / em[i])**2 for i in range(3))
        rr = nf[3] * mum
        out["stat"] = float(rr * rr - lhs)
        # bound: exact evaluation when every product, partial sum, force and square is a float64 (the
        # boundary families are built so) and fl(rr rr) is rr^2 or not lhs itself; else 16 eps times magnitudes
        exact = (all(_representable(t) for row in terms for t in row) and all(_representable(x) for x in nf)
                 and all(e == 1 for e in eps) and all(_representable(nf[i]**2) for i in range(3))
                 and _representable(nf[0]**2 + nf[1]**2) and _representable(lhs) and _representable(rr)
                 and (_representable(rr * rr) or float(rr) * float(rr) != float(lhs)))
        if exact:
            out["stat_bound"] = 0.
        else:
            g = [abs(fm[i]) + sum(abs(t) for t in terms[i]) for i in range(4)]
            out["stat_bound"] = float(16 * EPS * (sum(((abs(nf[i]) + g[i]) / em[i])**2 for i in range(3))
                                                  + (mum * (abs(nf[3]) + g[3]))**2))
        if rr * rr >= lhs:
            out.update(br=2, f=np.array([float(x) for x in nf]))
            return out
        alpha = [vnf[0], vnf[1], vnf[2], vnf[3] + _m(sdt)]
        sl = sliding_root(A, alpha, mu, eps)
        s = sl["s"] if sl["found"] else mp.mpf(-CLAMP)
        if not sl["found"]:
            out["status"] |= ST_EIG_NOROOT
        if sl["found"]:        # (no root: the clamp is the outcome itself, not a margin against it)
            sl["clamp"] = float((s + CLAMP) / CLAMP)
        if s < -CLAMP:
            s = mp.mpf(-CLAMP)
        M = mp.matrix(Am)
        for i in range(3):
            M[i, i] -= s / em[i]**2
        newf = mp.lu_solve(M, mp.matrix([-x for x in alpha]))
        sl["cond2"] = float(mp.cond(M, lambda X: mp.mnorm(X, 1)))     # cond_1, within 4x of cond_2 for 4x4
        sl["s_used"] = float(s)
        # s in a near-double real pair: rounding may turn the pair complex, and the admissible minimum is then
        # the next admissible eigenvalue outside the pair (or none: the clamp).  The force of that solve too.
        if sl["found"]:
            sc = sl["scale"]
            pair = [r * sc for r, i in sl["eigs"] if i == 0. and abs(r * sc - float(sl["s"])) <= PAIR_BAND * sc]
            if len(pair) > 1:
                rest = [r * sc for r, i in sl["eigs"] if i == 0. and r <= 0. and
                        abs(r * sc - float(sl["s"])) > PAIR_BAND * sc]
                s2 = max(mp.mpf(min(rest)), mp.mpf(-CLAMP)) if rest else mp.mpf(-CLAMP)
                M2 = mp.matrix(Am)
                for i in range(3):
                    M2[i, i] -= s2 / em[i]**2
                sl["alt"] = dict(f=np.array([float(x) for x in mp.lu_solve(M2, mp.matrix([-x for x in alpha]))]),
                                 s_used=float(s2), noroot=not rest,
                                 cond2=float(mp.cond(M2, lambda X: mp.mnorm(X, 1))))
        out.update(br=3, f=np.array([float(x) for x in newf]), slide=sl)
        return out


# -------------------------------------------------------------------------------------------------
# pinv / solve / inv_small_cond
# -------------------------------------------------------------------------------------------------
def pinv(a):
    """numpy.linalg.pinv semantics (sigma_j > RCOND sigma_max kept) at DPS digits.  Returns the
    pseudo-inverse, the rank kept, the 2-norm condition number of the part inverted, and the margin
    min_j |sigma_j / sigma_max - RCOND| of the cut."""
    a = np.atleast_2d(np.asarray(a, np.float64))
    n = a.shape[0]
    with mp.workdps(DPS):
        M = _mat(a)
        if n == 1:
            x = M[0, 0]
            return dict(pinv=np.array([[float(1 / x) if x != 0 else 0.]]), rank=int(x != 0), cond=1.,
                        cut_margin=float("inf"))
        U, S, V = mp.svd_r(M)
        smax = max(S) if len(S) else mp.mpf(0)
        if smax == 0:
            return dict(pinv=np.zeros((n, n)), rank=0, cond=1., cut_margin=float("inf"))
        keep = [j for j in range(n) if S[j] > RCOND * smax]
        out = mp.zeros(n, n)
        for j in keep:
            for r in range(n):
                for c in range(n):
                    out[r, c] += V[j, r] * U[c, j] / S[j]
        margin = min(abs(S[j] / smax - RCOND) for j in range(n))
        cond = smax / min(S[j] for j in keep)
        return dict(pinv=np.array([[float(out[r, c]) for c in range(n)] for r in range(n)]), rank=len(keep),
                    cond=float(cond), cut_margin=float(margin))


def cond1(a):
    """||A||_1 ||A^-1||_1 (inf for a singular matrix), the quantity of inv_small_cond."""
    with mp.workdps(DPS):
        M = _mat(a)
        try:
            Mi = mp.inverse(M)
        except ZeroDivisionError:
            return float("inf")
        return float(mp.mnorm(M, 1) * mp.mnorm(Mi, 1))


def solve(a, b):
    """x = A^-1 b and cond_2(A) (None, inf for a singular A)."""
    with mp.workdps(DPS):
        M = _mat(a)
        if mp.det(M) == 0:
            return None, float("inf")
        x = mp.lu_solve(M, mp.matrix([_m(t) for t in b]))
        U, S, V = mp.svd_r(M)
        return np.array([float(t) for t in x]), float(max(S) / min(S))


# -------------------------------------------------------------------------------------------------
# SE(3) exponential, zaligned, collisions
# -------------------------------------------------------------------------------------------------
def twist_exp(tw):
    """twistvector.py:35-70 at DPS digits: 12 doubles (R row-major, p), the series side (True:
    Rodrigues) and the margin |w| - SERIES_SWITCH."""
    with mp.workdps(DPS):
        w = [_m(x) for x in tw[:3]]
        v = [_m(x) for x in tw[3:]]
        t = mp.sqrt(sum(x * x for x in w))
        rod = t >= SERIES_SWITCH
        if rod:
            cc, sc, dsc = (1 - mp.cos(t)) / t**2, mp.sin(t) / t, (t - mp.sin(t)) / t**3
        else:
            cc, sc, dsc = mp.mpf(1) / 2, 1 - t**2 / 6, mp.mpf(1) / 6
        wx = mp.matrix([[0, -w[2], w[1]], [w[2], 0, -w[0]], [-w[1], w[0], 0]])
        R = mp.eye(3) + sc * wx + cc * wx * wx
        wv = sum(w[i] * v[i] for i in range(3))
        c3 = [w[1] * v[2] - w[2] * v[1], w[2] * v[0] - w[0] * v[2], w[0] * v[1] - w[1] * v[0]]
        p = [sc * v[i] + cc * c3[i] + dsc * w[i] * wv for i in range(3)]
        out = np.array([float(R[i, j]) for i in range(3) for j in range(3)] + [float(x) for x in p])
        return dict(H=out, rodrigues=bool(rod), margin=float(t - SERIES_SWITCH))


def zaligned(z):
    """homogeneousmatrix.py:201-232: numpy's stable argsort of |z| and the frame built from it.
    Returns R (3x3), idx and the tie margin (smallest gap between two |z_i|; 0 = a tie, where the
    order is the stable one)."""
    z = np.asarray(z, np.float64)
    idx = np.argsort(np.abs(z), kind="stable")
    with mp.workdps(DPS):
        zm = [_m(t) for t in z]
        x = [mp.mpf(0)] * 3
        x[idx[1]] = zm[idx[2]]
        x[idx[2]] = -zm[idx[1]]
        nx = mp.sqrt(sum(t * t for t in x))
        x = [t / nx for t in x]
        y = [zm[1] * x[2] - zm[2] * x[1], zm[2] * x[0] - zm[0] * x[2], zm[0] * x[1] - zm[1] * x[0]]
        R = np.array([[float(x[i]), float(y[i]), float(zm[i])] for i in range(3)])
    a = np.sort(np.abs(z))
    return dict(R=R, idx=idx, margin=float(min(a[1] - a[0], a[2] - a[1])))


def _hinv_apply(H, p):
    R = [[_m(H[3 * i + j]) for j in range(3)] for i in range(3)]
    t = [_m(H[9 + i]) for i in range(3)]
    return [sum(R[j][i] * (p[j] - t[j]) for j in range(3)) for i in range(3)]


def collide(pair, cd, H0, H1):
    """collisions.py pairs (0 plane/sphere-point, 1 sphere/sphere, 2 box/sphere) as the oracle
    composes them, frames given as 12 doubles.  Returns sdist, Hc0 and Hc1 (12 doubles each), the
    zaligned indices and the margins of the discrete decisions: 'inside' (box: min_i he_i - |p_i|,
    >= 0 inside), 'face' (box inside: gap between the two smallest face distances, 0 = a tie resolved
    by numpy.argmin's first minimum), 'sign' (plane: sdist itself, numpy.sign)."""
    cd = np.asarray(cd, np.float64)
    r0, r1 = cd[41], cd[42]
    with mp.workdps(DPS):
        g0 = [_m(H0[9 + i]) for i in range(3)]
        g1 = [_m(H1[9 + i]) for i in range(3)]
        R0 = [[_m(H0[3 * i + j]) for j in range(3)] for i in range(3)]
        marg = {}
        if pair == 1:
            vec = [g1[i] - g0[i] for i in range(3)]
            nrm = mp.sqrt(sum(x * x for x in vec))
            sdist = nrm - _m(r0) - _m(r1)
            normal = [x / nrm for x in vec]
            nf = np.array([float(x) for x in normal])
            za = zaligned(nf)
            # (the frame follows zaligned of the float normal, as every implementation builds it)
            z = [_m(x) for x in nf]
            p0 = [g0[i] + _m(r0) * z[i] for i in range(3)]
            p1 = [p0[i] + sdist * z[i] for i in range(3)]
        elif pair == 2:
            he = [_m(x) for x in cd[32:35]]
            p01 = _hinv_apply(H0, g1)
            ins = min(he[i] - abs(p01[i]) for i in range(3))
            marg["inside"] = float(ins)
            normal = [mp.mpf(0)] * 3
            if ins >= 0:
                d = [he[i] - p01[i] for i in range(3)] + [he[i] + p01[i] for i in range(3)]
                im = min(range(6), key=lambda k: (d[k], k))
                ds = sorted(d)
                marg["face"] = float(ds[1] - ds[0])
                marg["face_index"] = im
                f0 = list(p01)
                if im < 3:
                    f0[im] = he[im]
                    normal[im] = mp.mpf(1)
                else:
                    f0[im - 3] = -he[im - 3]
                    normal[im - 3] = mp.mpf(-1)
                fg = [sum(R0[i][j] * f0[j] for j in range(3)) + g0[i] for i in range(3)]
                sdist = -mp.sqrt(sum((fg[i] - g1[i])**2 for i in range(3))) - _m(r1)
            else:
                f0 = [max(min(he[i], p01[i]), -he[i]) for i in range(3)]
                fg = [sum(R0[i][j] * f0[j] for j in range(3)) + g0[i] for i in range(3)]
                vec = [g1[i] - fg[i] for i in range(3)]
                nrm = mp.sqrt(sum(x * x for x in vec))
                normal = [x / nrm for x in vec]
                sdist = nrm - _m(r1)
            nf = np.array([float(x) for x in normal])
            za = zaligned(nf)
            p0 = fg
            p1 = [g1[i] - _m(r1) * _m(nf[i]) for i in range(3)]
        else:
            coef = [_m(x) for x in cd[32:36]]
            p01 = _hinv_apply(H0, g1)
            csdist = sum(coef[i] * p01[i] for i in range(3)) - coef[3]
            sdist = csdist - _m(r1)
            marg["sign"] = float(sdist)
            za = zaligned(cd[32:35])
            sg = 1 if sdist > 0 else (-1 if sdist < 0 else 0)
            p0 = [p01[i] - csdist * coef[i] for i in range(3)]
            p1 = [p01[i] - sg * _m(r1) * coef[i] for i in range(3)]
        R = za["R"].reshape(-1)
        return dict(sdist=float(sdist), Hc0=np.concatenate([R, [float(x) for x in p0]]),
                    Hc1=np.concatenate([R, [float(x) for x in p1]]), idx=za["idx"], zmargin=za["margin"],
                    **marg)
