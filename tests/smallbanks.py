"""Seeded input banks for the small dense routines and the soft-finger contact solve: families of
problems placed on purpose at the decision boundaries of the code (see tests/smallref.py for the
margins).  Each family is a dict of numpy arrays, problem-major ([N][...]); the tests check that
each family lands where it claims.

Nothing here holds a non-finite input; every problem completes on the host build."""
import numpy as np

DT = 2.0**-10            # a power of two near the 1 ms step: dt v3 and sdist / dt stay exact where a family needs it


def _ulps(x, k):
    """x moved by k ulps (k may be negative)."""
    x = np.float64(x)
    for _ in range(abs(k)):
        x = np.nextafter(x, np.inf if k > 0 else -np.inf)
    return float(x)


def _spd4(rng, cond=None, nterm=True):
    """admittance-like 4x4 block: SPD (like J Y J^T) with condition number `cond` (random when None),
    plus the non-symmetric N-term perturbation of test_hostmath.py."""
    Q, _ = np.linalg.qr(rng.normal(size=(4, 4)))
    if cond is None:
        cond = 10.**rng.uniform(0, 4)
    sv = np.geomspace(1., 1./cond, 4)
    A = (Q * sv).dot(Q.T) * 10.**rng.uniform(-3, 1)
    if nterm:
        A = A + rng.normal(size=(4, 4)) * 1e-2 * np.abs(A).min()
    return A


def _contact(rng, n, conds=None, mus=(0.1, 1.5), warm=0.5):
    v, A, P, sd, mu, eps, f0 = [], [], [], [], [], [], []
    for k in range(n):
        a = _spd4(rng, None if conds is None else conds[k % len(conds)])
        v.append(rng.normal(size=4) * 10.**rng.uniform(-3, 0))
        A.append(a)
        P.append(np.linalg.pinv(a))
        sd.append(-abs(rng.normal()) * 1e-3)
        mu.append(rng.uniform(*mus))
        eps.append(np.ones(3))
        f0.append(rng.normal(size=4) * 1e-2 * (rng.uniform() < warm))
    return _pack(v, A, P, sd, mu, eps, f0)


def _pack(v, A, P, sd, mu, eps, f0):
    return dict(v=np.array(v), A=np.array(A), P=np.array(P), sdist=np.array(sd, np.float64),
                mu=np.array(mu, np.float64), eps=np.array(eps), f0=np.array(f0), dt=DT)


def contact_families(seed=0):
    """SoftFingerContact.solve problems (v, A, P = pinv(A), sdist, mu, eps, dt, f0)."""
    rng = np.random.default_rng(seed)
    fam = {}
    # control: generic SPD blocks from cond 1 to 1e12, cold and warm starts, all three branches
    fam["contact_generic"] = _contact(rng, 160, conds=[1., 1e2, 1e4, 1e6, 1e9, 1e12])
    # release boundary: sdist + dt v3 = 0 and +-1..4 ulp (f0 = 0, dt a power of two: exactly representable).
    # The normal row is decoupled and v_t = 0, so a contact that is not released holds statically: at the
    # boundary alpha_n = v3 + sdist / dt vanishes and the sliding matrix of the reference divides by it
    v, A, P, sd, mu, eps, f0 = [], [], [], [], [], [], []
    for k in range(36):
        a = _spd4(rng)
        a[:3, 3] = a[3, :3] = 0.
        vv = np.zeros(4)
        vv[3] = rng.normal() * 1e-2
        off = (k % 9) - 4
        v.append(vv); A.append(a); P.append(np.linalg.pinv(a))
        sd.append(_ulps(-DT * vv[3], off)); mu.append(rng.uniform(0.1, 1.5)); eps.append(np.ones(3))
        f0.append(np.zeros(4))
    fam["contact_release_edge"] = _pack(v, A, P, sd, mu, eps, f0)
    # static boundary: lhs - rr^2 = 0 and +-1..4 ulp with exact arithmetic (P diagonal of powers of two,
    # forces small dyadics, rr = nf3 mu): nf = s (0.75, 1, 0, 1), mu = 1.25 moved by k ulps; mu = 0 with a
    # zero tangential force (0 <= 0: static) and mu = 2
    v, A, P, sd, mu, eps, f0 = [], [], [], [], [], [], []
    for k in range(40):
        a = _spd4(rng)
        s = 2.0**int(rng.integers(-6, 3))
        p = 2.0**rng.integers(-3, 4, size=4).astype(float)
        p[3] = abs(p[3])
        if k < 27:
            nf, m = s * np.array([0.75, 1., 0., 1.]), _ulps(1.25, (k % 9) - 4)
        elif k < 33:
            nf, m = s * np.array([0., 0., 0., 1.]), 0.
        else:
            nf, m = s * np.array([1.5, 1., 0.5, 1.]), 2.
        c = 2.0**int(rng.integers(-4, 2))                # sdist / dt = -c: exact
        rhs = -nf / p
        vv = rhs.copy()
        vv[3] = rhs[3] + c
        v.append(vv); A.append(a); P.append(np.diag(p)); sd.append(-c * DT); mu.append(m)
        eps.append(np.ones(3)); f0.append(np.zeros(4))
    fam["contact_static_edge"] = _pack(v, A, P, sd, mu, eps, f0)
    fam["contact_static_edge"]["P_is_pinv"] = False
    # y_n tiny against Y_t: the normal row of G scaled down
    v, A, P, sd, mu, eps, f0 = [], [], [], [], [], [], []
    for k in range(24):
        G = rng.normal(size=(4, 6))
        G[3] *= 10.**rng.uniform(-5, -3)
        a = G.dot(G.T)
        v.append(rng.normal(size=4) * 1e-3); A.append(a); P.append(np.linalg.pinv(a))
        sd.append(-1e-6 * rng.uniform()); mu.append(rng.uniform(0.01, 0.1)); eps.append(np.ones(3))
        f0.append(np.zeros(4) if k % 2 else rng.normal(size=4) * 1e-6)
    fam["contact_yn_tiny"] = _pack(v, A, P, sd, mu, eps, f0)
    # eps != 1: the general eigenvalue path (eig_real_general6) for the sliding root
    d = _contact(rng, 48, mus=(0.3, 1.5), warm=0.)
    d["eps"][:] = np.array([0.5, 1., 2.])
    fam["contact_eps"] = d
    # sliding problems with no admissible root (s = -1e10 and EIG_NOROOT) and with a root beyond the clamp
    # (tiny alpha_n): f0 = 0 and v = alpha - (0, 0, 0, sdist / dt), alpha_n < 0 (the contact stays), kept when
    # the static test fails and numpy's eigvals of B puts the family where it belongs
    v, A, P, sd, mu, eps, f0 = [], [], [], [], [], [], []
    nroot = nclamp = 0
    while nroot < 16 or nclamp < 16:
        a = _spd4(rng)
        x = rng.normal(size=4) * 10.**rng.uniform(-3, 0)
        m = rng.uniform(0.1, 1.5)
        x[3] = -abs(x[3])
        beyond = nroot >= 16 or (nclamp < 16 and rng.uniform() < 0.5)
        if beyond:
            x[3] = -1e-12
        S = np.linalg.eigvals(_np_sliding_matrix(a, x, m))
        S = S[(S.imag == 0) & (S.real <= 0)]
        want = (len(S) and S.real.min() < -2e10) if beyond else len(S) == 0
        pa = np.linalg.pinv(a)
        nf = -pa.dot(x)
        if not want or (nf[:3]**2).sum() <= (nf[3] * m)**2 * 1.01:
            continue
        sdist = -2.0**int(rng.integers(-14, -8))
        vv = x.copy()
        vv[3] = x[3] - sdist / DT
        v.append(vv); A.append(a); P.append(pa); sd.append(sdist); mu.append(m); eps.append(np.ones(3))
        f0.append(np.zeros(4))
        nclamp += beyond
        nroot += not beyond
    fam["contact_clamp"] = _pack(v, A, P, sd, mu, eps, f0)
    return fam


def _sliding_from(A, alpha, mu):
    return dict(A=np.array(A), alpha=np.array(alpha), mu=np.array(mu, np.float64))


def sliding_families(seed=1):
    """sliding_root_structured problems (A, alpha, mu), eps = 1."""
    rng = np.random.default_rng(seed)
    fam = {}
    A, al, mu = [], [], []
    for _ in range(96):
        a = _spd4(rng)
        A.append(a); al.append(rng.normal(size=4) * 10.**rng.uniform(-3, 1)); mu.append(rng.uniform(0.1, 1.5))
    fam["slide_generic"] = _sliding_from(A, al, mu)
    # Y_c = 0, Y_t = diag(y) and beta = (beta_0, 0, 0): B splits into the 2x2 blocks [[y_i, -r^2], [-1, y_i]],
    # r = |beta_0 / a|, with the simple eigenvalues y_i +- r.  With y = (1.25, 0.5, 1/8 + d) and r = 1/8 the
    # smallest is d; at d = 0 every coefficient of the structured sextic is exact (the scale is 2), so the
    # zero eigenvalue is zero in float64 too: the s <= 0 inclusion.  d = +-2^-30, +-2^-20 beside it
    A, al, mu = [], [], []
    for k in range(30):
        d = [0., 2.0**-30, -2.0**-30, 2.0**-20, -2.0**-20, 0.][k % 6]
        s = 2.0**int(rng.integers(-3, 3))             # overall scale: a power of two keeps everything exact
        yn, m, a3 = 2.0**int(rng.integers(-3, 1)), 2.0**int(rng.integers(-2, 1)), 2.0**int(rng.integers(-4, 2))
        a = m / yn * a3
        A.append(np.diag([1.25 * s, 0.5 * s, (0.125 + d) * s, yn]))
        al.append([0.125 * s * a * (1. if k % 2 else -1.), 0., 0., a3]); mu.append(m)
    fam["slide_zero_root"] = _sliding_from(A, al, mu)
    # a complex pair next to the real axis and two real eigenvalues that nearly meet (tangent): bisection
    # on mu of a generic problem for the point where the count of real eigenvalues of B changes, the
    # problems taken on both sides of it at relative distances 1e-4 .. 1e-9
    A, al, mu = [], [], []
    while len(A) < 40:
        a = _spd4(rng)
        x = rng.normal(size=4) * 10.**rng.uniform(-2, 0)
        grid = np.linspace(0.1, 2., 40)
        cnt = [int((np.linalg.eigvals(_np_sliding_matrix(a, x, m)).imag == 0).sum()) for m in grid]
        ch = [i for i in range(len(grid) - 1) if cnt[i] != cnt[i + 1]]
        if not ch:
            continue
        lo, hi = grid[ch[0]], grid[ch[0] + 1]
        clo = cnt[ch[0]]
        for _ in range(60):
            mid = 0.5 * (lo + hi)
            if int((np.linalg.eigvals(_np_sliding_matrix(a, x, mid)).imag == 0).sum()) == clo:
                lo = mid
            else:
                hi = mid
        m0 = 0.5 * (lo + hi)
        for d in (1e-4, 1e-6, 1e-9):
            for sg in (-1., 1.):
                A.append(a); al.append(x); mu.append(m0 * (1. + sg * d))
    fam["slide_tangent"] = _sliding_from(A, al, mu)
    # no admissible root, and roots beyond the -1e10 clamp (tiny alpha_n: a ~ 1e-12)
    A, al, mu, B2, al2, mu2 = [], [], [], [], [], []
    while len(A) < 24 or len(B2) < 24:
        a = _spd4(rng)
        x = rng.normal(size=4) * 10.**rng.uniform(-3, 1)
        m = rng.uniform(0.1, 1.5)
        S = np.linalg.eigvals(_np_sliding_matrix(a, x, m))
        S = S[(S.imag == 0) & (S.real <= 0)]
        if len(S) == 0 and len(A) < 24:
            A.append(a); al.append(x); mu.append(m)
        x = x.copy(); x[3] = 1e-13 * np.sign(x[3])
        S = np.linalg.eigvals(_np_sliding_matrix(a, x, m))
        S = S[(S.imag == 0) & (S.real <= 0)]
        if len(S) and S.real.min() < -1e11 and len(B2) < 24:
            B2.append(a); al2.append(x); mu2.append(m)
    fam["slide_no_root"] = _sliding_from(A, al, mu)
    # y_n tiny against Y_t (the reciprocal of y_n in the structured path)
    A, al, mu = [], [], []
    for _ in range(24):
        G = rng.normal(size=(4, 6))
        G[3] *= 10.**rng.uniform(-5, -3)
        A.append(G.dot(G.T)); al.append(rng.normal(size=4) * 1e-3); mu.append(rng.uniform(0.1, 1.5))
    fam["slide_yn_tiny"] = _sliding_from(A, al, mu)
    fam["slide_beyond_clamp"] = _sliding_from(B2, al2, mu2)
    return fam


def bad_sliding_family(seed=8):
    """sliding problems on which the structured path is `bad` (its scale sigma is 0: Y_t = (|Y_c|^2 / y_n) J and
    beta = 0 make Q, c and delta vanish): sliding_root_structured must refuse them, and the solve falls back to
    eig_real_general6 on B = [[0, 0], [(|b|^2 - 1) I, 0]] (eigenvalue 0, six-fold)."""
    rng = np.random.default_rng(seed)
    A, al, mu, Bs = [], [], [], []
    for k in range(12):
        yc = np.zeros(3)
        yc[k % 3] = 2.0**int(rng.integers(-2, 2))
        yn = 2.0**int(rng.integers(-2, 2))
        a = np.zeros((4, 4))
        a[:3, :3] = (yc.dot(yc) / yn) * np.ones((3, 3))
        a[:3, 3] = a[3, :3] = yc
        a[3, 3] = yn
        an = 2.0**int(rng.integers(-3, 1))
        x = np.r_[an / yn * yc, an]
        m = 2.0**int(rng.integers(-2, 1))
        A.append(a); al.append(x); mu.append(m); Bs.append(_np_sliding_matrix(a, x, m))
    return dict(A=np.array(A), alpha=np.array(al), mu=np.array(mu, np.float64), B=np.array(Bs))


def _np_sliding_matrix(A, alpha, mu):
    Y_c, y_n, Y_t = A[0:3, 3], A[3, 3], A[0:3, 0:3]
    beta = alpha[0:3] - alpha[3]/y_n*Y_c
    a = mu/y_n*alpha[3]
    b = mu/y_n*Y_c
    B = np.zeros((6, 6))
    Y_that = Y_t - np.dot(Y_c, Y_c)/y_n
    B[3:6, 3:6] = Y_that
    B[0:3, 0:3] = Y_that + 2/a*np.dot(beta, b)
    B[0:3, 3:6] = -np.eye(3)*np.dot(beta, beta)/a**2
    B[3:6, 0:3] = np.eye(3)*np.dot(b, b) - np.eye(3)
    return B


def _sextic(roots):
    c = np.real(np.poly(roots))
    return np.ascontiguousarray(c[::-1][:6])


def poly_families(seed=2):
    """monic sextics p[0..5] aimed at the exits of the fast path."""
    rng = np.random.default_rng(seed)
    fam = {}
    # left of a root from the start bound (bracket recovery): real roots with a complex pair that pulls the
    # Samuelson bound left of the largest root
    # (kept: the bound mean + sqrt(5) std of the coefficients lies left of the largest real root)
    P = []
    while len(P) < 60:
        r = list(rng.uniform(-1., 1., size=3)) + [rng.uniform(1.5, 2.5)]
        re = rng.uniform(-3., -1.)
        im = rng.uniform(1.5, 3.)
        p = _sextic(r + [complex(re, im), complex(re, -im)])
        mean = -p[5] / 6.
        var = (p[5]**2 - 2. * p[4]) / 6. - mean**2
        if var >= 0. and mean + np.sqrt(5. * var) < max(r):
            P.append(p)
    fam["poly_recover"] = dict(p=np.array(P))
    # no root t >= 0 but not all coefficients positive: the positivity march
    P = []
    for _ in range(60):
        re1, re2 = rng.uniform(0.2, 2.), rng.uniform(-2., 2.)
        im1, im2 = rng.uniform(1., 3.), rng.uniform(0.5, 2.)
        P.append(_sextic([complex(re1, im1), complex(re1, -im1), complex(re2, im2), complex(re2, -im2),
                          rng.uniform(-3., -0.5), rng.uniform(-3., -0.5)]))
    fam["poly_positive"] = dict(p=np.array(P))
    # a positive root the fast path cannot start on: the rigorous isolation (poly6_roots_slow) decides
    P = []
    while len(P) < 60:
        # two complex pairs far from the axis make the variance of the roots negative: no start bound, and
        # the positive root keeps the positivity march from proving anything
        r = rng.uniform(0.2, 1.)
        i1, i2 = rng.uniform(2., 4.), rng.uniform(2., 4.)
        re1, re2 = rng.uniform(-0.5, 0.5), rng.uniform(-0.5, 0.5)
        p = _sextic([r, rng.uniform(-2., -0.5), complex(re1, i1), complex(re1, -i1), complex(re2, i2), complex(re2, -i2)])
        if (p[5]**2 - 2. * p[4]) / 6. - (p[5] / 6.)**2 < 0.:
            P.append(p)
    fam["poly_slow"] = dict(p=np.array(P))
    return fam


def _orth(rng):
    Q, R = np.linalg.qr(rng.normal(size=(4, 4)))
    return Q * np.sign(np.diag(R))


def pinv_families(seed=3):
    rng = np.random.default_rng(seed)
    fam = {}
    # singular values straddling 1e-15 sigma_max, outside the rounding band (16 eps sigma_max) on both sides
    M = []
    for k in range(48):
        rel = [5.5e-15, 8e-15, 2e-14, 1e-13, 1e-16, 1e-18][k % 6]
        U, V = _orth(rng), _orth(rng)
        M.append((U * np.array([1., 0.5, 0.25, rel])).dot(V.T))
    fam["pinv_straddle"] = dict(A=np.array(M))
    # cond_1 on both sides of the 1e12 shortcut
    M = []
    for k in range(48):
        c = [1e11, 4e11, 3e12, 1e13][k % 4]
        U, V = _orth(rng), _orth(rng)
        M.append((U * np.geomspace(1., 1. / c, 4)).dot(V.T))
    fam["pinv_cond"] = dict(A=np.array(M))
    # exact rank 1..3 (integer matrices), the zero matrix
    M = []
    for k in range(36):
        r = 1 + k % 3
        X = rng.integers(-4, 5, size=(4, r)).astype(float)
        Y = rng.integers(-4, 5, size=(r, 4)).astype(float)
        M.append(X.dot(Y))
    M.append(np.zeros((4, 4)))
    fam["pinv_rank"] = dict(A=np.array(M))
    return fam


def solve_families(seed=4):
    rng = np.random.default_rng(seed)
    A, b = [], []
    for k in range(24):          # pivot ties: equal magnitudes in a column
        a = rng.integers(-3, 4, size=(4, 4)).astype(float)
        a[:, 0] = [2., -2., 2., 1.]
        a[:, 1] += 1e-3 * rng.normal(size=4)
        A.append(a); b.append(rng.normal(size=4))
    gen = dict(A=np.array(A), b=np.array(b))
    A, b = [], []
    for k in range(12):          # an exact zero pivot: a zero column or a zero row
        a = rng.normal(size=(4, 4))
        if k % 2:
            a[:, k % 4] = 0.
        else:
            a[k % 4] = 0.
        A.append(a); b.append(rng.normal(size=4))
    return dict(solve_ties=gen, solve_singular=dict(A=np.array(A), b=np.array(b)))


def eig_families(seed=5):
    rng = np.random.default_rng(seed)
    fam = {}
    M = []
    for k in range(24):          # defective: Jordan blocks under an integer similarity
        J = np.diag(rng.integers(-3, 4, size=6).astype(float))
        lam = float(rng.integers(-2, 3))
        J[0, 0] = J[1, 1] = lam
        J[0, 1] = 1.
        if k % 2:
            J[2, 2] = lam; J[1, 2] = 1.
        # S = L U with unit triangular integer factors: det 1, an integer inverse, and S J S^-1 is exact in
        # float64 and full (not triangular: the QR iteration has to find the clusters)
        L = np.eye(6) + np.tril(rng.integers(-1, 2, size=(6, 6)), -1).astype(float)
        U = np.eye(6) + np.triu(rng.integers(-1, 2, size=(6, 6)), 1).astype(float)
        S = L.dot(U)
        Si = np.round(np.linalg.inv(U)).dot(np.round(np.linalg.inv(L)))
        assert np.array_equal(S.dot(Si), np.eye(6))
        M.append(S.dot(J).dot(Si))
    fam["eig_defective"] = dict(A=np.array(M))
    M = []
    for k in range(24):          # companion matrices with clustered roots
        r = 1. + 1e-3 * rng.normal(size=3)
        roots = list(r) + list(rng.uniform(-2., 2., size=3))
        c = np.poly(roots)
        C = np.zeros((6, 6)); C[1:, :5] = np.eye(5); C[:, 5] = -c[:0:-1]
        M.append(C)
    fam["eig_companion"] = dict(A=np.array(M))
    M = []
    for k in range(24):          # badly balanced: D X D^-1 with D across 2^(+-250) ~ 1e(+-75)
        X = rng.normal(size=(6, 6))
        d = 2.0**np.array([-250, -120, 0, 60, 130, 250])[rng.permutation(6)]
        M.append(X * d[:, None] / d[None, :])
    fam["eig_balance"] = dict(A=np.array(M))
    M = []
    for k in range(6):           # the cyclic shift: Francis steps stall without the exceptional shift
        C = np.roll(np.eye(6), 1, axis=0) * (1. + k)
        M.append(C)
    fam["eig_exceptional"] = dict(A=np.array(M))
    return fam


def se3_families(seed=6):
    rng = np.random.default_rng(seed)
    tw = []
    for k in range(-4, 5):       # |w| at the series switch, one nonzero component (sqrt(w^2) is exact)
        for ax in range(3):
            w = np.zeros(3); w[ax] = _ulps(1e-3, k) * (-1. if k % 2 else 1.)
            tw.append(np.concatenate([w, rng.normal(size=3)]))
    for t in (0., 1.5e-3, 1.9e-3, 5e-4, np.pi, 50.):
        for _ in range(3):
            u = rng.normal(size=3); u /= np.linalg.norm(u)
            tw.append(np.concatenate([u * t, rng.normal(size=3)]))
    return dict(se3_switch=dict(tw=np.array(tw)))


def frame_families(seed=7):
    rng = np.random.default_rng(seed)
    Z = []
    for ax in range(3):
        for sg in (1., -1.):
            z = np.zeros(3); z[ax] = sg; Z.append(z)
    h = np.sqrt(0.5)
    t = np.sqrt(1. / 3.)
    for s in ((h, h, 0.), (h, 0., -h), (0., -h, h), (t, t, t), (-t, t, -t), (0.6, 0.6, np.sqrt(1 - 0.72)),
              (0.8, 0.36, 0.48), (0.48, 0.8, -0.36)):
        Z.append(np.array(s))
    for _ in range(16):
        z = rng.normal(size=3); Z.append(z / np.linalg.norm(z))
    fam = dict(zaligned_ties=dict(z=np.array(Z)))
    # collisions: identity frames (exact p01) for the boundary cases, rotated frames for the rest
    I12 = np.concatenate([np.eye(3).reshape(-1), np.zeros(3)])
    pair, cd, H0, H1 = [], [], [], []

    def add(pr, c, h0, h1):
        pair.append(pr); cd.append(c); H0.append(h0); H1.append(h1)

    def cdv(coef=(0., 0., 1., 0.), r0=0., r1=0.):
        c = np.zeros(48); c[32:36] = coef; c[41] = r0; c[42] = r1
        return c

    he = np.array([0.25, 0.25, 0.25])
    for pos in ([0., 0., 0.], [0.25, 0., 0.], [0., -0.25, 0.1], [0.25, 0.25, 0.], [0.25, -0.25, 0.25],
                [0.125, 0.0625, 0.], [0.5, 0., 0.], [0.25, 0.5, 0.]):
        add(2, cdv(tuple(he) + (0.,), 0., 0.0625), I12, np.concatenate([np.eye(3).reshape(-1), pos]))
    he2 = np.array([0.5, 0.25, 0.125])
    for pos in ([0., 0., 0.], [0.5, 0.25, 0.125], [-0.5, 0., 0.]):
        add(2, cdv(tuple(he2) + (0.,), 0., 0.), I12, np.concatenate([np.eye(3).reshape(-1), pos]))
    for coef, pos in (((0., 0., 1., 0.), [0.3, 0.2, 0.]), ((1., 0., 0., 0.5), [0.5, 0.1, 0.2]),
                      ((0., -1., 0., 0.), [0.1, 0., 0.2])):
        for r1 in (0., 0.0625):
            add(0, cdv(coef, 0., r1), I12, np.concatenate([np.eye(3).reshape(-1), pos]))
    for _ in range(12):
        Q = _orth(rng)[:3, :3]
        if np.linalg.det(Q) < 0:
            Q[:, 0] *= -1.
        h0 = np.concatenate([Q.reshape(-1), rng.normal(size=3)])
        h1 = np.concatenate([np.eye(3).reshape(-1), rng.normal(size=3)])
        k = len(pair) % 3
        if k == 0:
            z = rng.normal(size=3); z /= np.linalg.norm(z)
            add(0, cdv(tuple(z) + (rng.normal(),), 0., 0.05), h0, h1)
        elif k == 1:
            add(1, cdv(r0=0.1, r1=0.2), h0, h1)
        else:
            add(2, cdv(tuple(rng.uniform(0.2, 1., 3)) + (0.,), 0., 0.1), h0, h1)
    fam["collide"] = dict(pair=np.array(pair, np.int32), cd=np.array(cd), H0=np.array(H0), H1=np.array(H1))
    return fam
