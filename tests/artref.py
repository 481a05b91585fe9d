"""High-precision reference (mpmath, 50 digits) of the impedance solve that the fused prepare and
finish stages hand over between them (arb_fused.cuh, world_fused_prepare / world_fused_finish).

For ONE world of a flattened model (the dict FlatModel.to_dict() gives; per-world body inertia,
gravity and PD gains are baked into it, see bodyparams.world_model) and its float64 state, every
float64 input is taken exactly and this module restates, at 50 digits:

  * OracleWorld.update_dynamic (core.py:682-734, Body.update_dynamic core.py:1272-1315): body
    poses, twists, J_b, dJ_b, and M, N, B;
  * OracleWorld.update_controllers (core.py:811-818): WeightController (controllers.py:43-60),
    ProportionalDerivativeController (controllers.py:141-159) and the applied forces of
    arb_batch_bind_applied_forces; Z = M/dt + B + N + (dt kp + kd);
  * q_free = Z^-1 (M q'/dt + gforce);
  * G: per generator body its J_b, rotated by blockdiag(R_e, R_e) when contact-aligned (R_e =
    R_c^T R_body, R_c from zaligned(normal), homogeneousmatrix.py:201-232), per joint-limit row a unit
    row; v0 = G q_free and Lambda = G Z^-1 G^T;
  * A_cc = J_c Z^-1 J_c^T of an active constraint from its Jacobian J_c formed the reference's way
    (constraints.py:65-71, :164-191, PointContact.update :277-295 with the collision solvers), NOT
    through generator space (core.py:925-927);
  * the finish: q'+ = q_free + Z^-1 G^T y for a given y, and the joint integration (core.py:974-980,
    joints.py:54-57 with twist_exp's series switch, twistvector.py:35-70).

Linear algebra runs on the ancestor-column sparsity of J_b (as the phase kernels do) and a dense LU
with partial pivoting at 50 digits, whose pivots |d_k| are reported too.

TOLERANCE RULE (fixed before any device result was looked at).  A float64 evaluation of these
quantities by any backward-stable order of operations satisfies, componentwise,

    |x^ - x| <= C u E(x),   u = 2^-53,

where E(x) is the first-order error magnitude of the computation: the forming errors of Z and of the
right-hand side are bounded by the sums of ABSOLUTE values of their terms (Zabs = sum_b |J_b|^T
(|M_b|/dt + |B_b| + |M_b||dJ_b| + |N_b||J_b|) ... + |PD|, babs likewise), so

    E(q_free) = |Z^-1| (Zabs |q_free| + babs)
    E(Lambda) = Ga |Z^-1| (Zabs |X| + Ga^T) + Ga |X|,          X = Z^-1 G^T,  Ga = magnitude of G
    E(A_cc)   = Ja |Z^-1| (Zabs |Xc| + Ja^T) + (1 + o/u) Ja |Xc| + sum_st |T_s| E(Lambda)_st |T_t|^T
                Ja = |T||G| + s |G_angular| on the linear rows (s = distance of the constraint frames
                from the ground origin: the lever arms of T are differences of positions in ground
                axes); the last term is Lambda's own error, which the float64 code carries into
                A_cc = T Lambda T^T; o = max |R_b^T R_b - I| over the bodies: a FreeJoint's rotation
                is float64 state, orthogonal only to rounding, and hinv() takes R^T for R^-1, so the
                two exact forms J_c Z^-1 J_c^T and T Lambda T^T differ by that much (1.5e-12 relative
                on A_cc of the mass-ratio world at cond(Z) = 2e16, 1.4x the bound without this term)
    E(q'+)    = E(q_free) + |Z^-1| (Zabs |Z^-1 G^T y| + Ga^T |y|)

and the bound's constant is C = 64 * (depth of the tree + 6): rounding compounds along the root path
in the elimination and the kinematic chain products.  The componentwise condition number is
E(x)_i / |x_i|.

For the matrices (Lambda, K, A_cc) E is floored, row by row, at the row maximum of the matrix's
magnitude: E_ij >= max_k |Lambda_ik|.  Entries that vanish exactly (the coupling of the angular and
linear rows of a free ball at its centre of mass) have E_ij = 0 by the magnitude rule, while the
articulated elimination forms them in other frames as sums that cancel to rounding of the row's size
(1e-21 against 1e-3 in the host build); the floor makes such entries harmless without loosening the
others.  A test that needs a looser bound writes the cause next to it.

HEADROOM.  The bound is a worst-case first-order sum: the host build and the device stay 10 to 1000
times below it on the families of artbanks.py (worst err / (C u E) per family is printed by the
tests).  It resolves dropped or misplaced terms (artref.MUTATIONS), not errors of a few ulps."""
import hashlib
import math
import os
import pickle

import mpmath as mp
import numpy as np

DPS = 50
U = 2.0**-53
FREE, RZRYRX, RZRY, RZRX, RYRX, RZ, RY, RX, TXTYTZ = range(9)
JOINT_NDOF = (6, 3, 2, 2, 2, 1, 1, 1, 3)
JOINT_NGPOS = (16, 3, 2, 2, 2, 1, 1, 1, 3)
LIM, BALL, CONTACT = 0, 1, 2
CACHE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_build", "artref")
# the mutations a test may apply to the reference, to show that the comparisons bite
MUTATIONS = ("drop_N", "drop_PD", "drop_B", "flip_wrench", "unrotated", "lambda_T", "free_half_dt")

_ZERO = None


def mpf(x):
    return mp.mpf(float(x))


def M(a):
    """object array of mpf from float64, exactly"""
    a = np.asarray(a, dtype=np.float64)
    return np.vectorize(lambda x: mp.mpf(float(x)), otypes=[object])(a) if a.size else a.astype(object)


def zeros(*shape):
    z = np.empty(shape, dtype=object)
    z.fill(mp.mpf(0))
    return z


def eye(n):
    z = zeros(n, n)
    for i in range(n):
        z[i, i] = mp.mpf(1)
    return z


def mabs(a):
    return np.vectorize(abs, otypes=[object])(a)


def tofloat(a):
    return np.vectorize(float, otypes=[float])(a)


# -------------------------------------------------------------------------------------------
# rigid-motion math (arboris/homogeneousmatrix.py, twistvector.py), as the oracle states it
# -------------------------------------------------------------------------------------------
def hinv(H):
    R = H[0:3, 0:3]
    out = eye(4)
    out[0:3, 0:3] = R.T
    out[0:3, 3] = -R.T.dot(H[0:3, 3])
    return out


def skew(p):
    z = mp.mpf(0)
    return np.array([[z, -p[2], p[1]], [p[2], z, -p[0]], [-p[1], p[0], z]], dtype=object)


def adjoint(H):
    R = H[0:3, 0:3]
    Ad = zeros(6, 6)
    Ad[0:3, 0:3] = R
    Ad[3:6, 3:6] = R
    Ad[3:6, 0:3] = skew(H[0:3, 3]).dot(R)
    return Ad


def iadjoint(H):
    return adjoint(hinv(H))


def adjacency(tw):
    ad = zeros(6, 6)
    ad[0:3, 0:3] = skew(tw[0:3])
    ad[3:6, 3:6] = skew(tw[0:3])
    ad[3:6, 0:3] = skew(tw[3:6])
    return ad


def norm(v):
    return mp.sqrt(sum(x*x for x in v))


def twist_exp(tw):
    """twistvector.py:35-70 with its series switch at |w| < 1e-3"""
    w, v = tw[0:3], tw[3:6]
    wx = skew(w)
    t = norm(w)
    if t >= mpf(0.001):
        cc, sc, dsc = (1 - mp.cos(t))/t**2, mp.sin(t)/t, (t - mp.sin(t))/t**3
    else:
        cc, sc, dsc = mp.mpf(1)/2, 1 - t**2/6, mp.mpf(1)/6
    R = eye(3) + sc*wx + cc*wx.dot(wx)
    w31 = w.reshape(3, 1)
    p = (sc*eye(3) + cc*wx + dsc*w31.dot(w31.T)).dot(v)
    H = eye(4)
    H[0:3, 0:3] = R
    H[0:3, 3] = p
    return H


def zaligned(vec):
    """homogeneousmatrix.py:201-232; the argsort of |z| on the float64 values (index work)"""
    z = np.array([mpf(x) for x in vec], dtype=object)
    idx = np.argsort(np.abs(np.asarray(vec, dtype=float)), kind="stable")
    x = zeros(3)
    x[idx[1]] = z[idx[2]]
    x[idx[2]] = -z[idx[1]]
    x = x/norm(x)
    H = eye(4)
    H[0:3, 0] = x
    H[0:3, 1] = np.array([z[1]*x[2] - z[2]*x[1], z[2]*x[0] - z[0]*x[2], z[0]*x[1] - z[1]*x[0]], dtype=object)
    H[0:3, 2] = z
    return H


def rot_h(R):
    H = eye(4)
    H[0:3, 0:3] = np.array(R, dtype=object)
    return H


def joint_pose(t, q):
    """joints.py pose of each joint type (oracle joint_pose)"""
    s, c = mp.sin, mp.cos
    if t == FREE:
        return q.reshape(4, 4).copy()
    if t == RZRYRX:
        sz, cz, sy, cy, sx, cx = s(q[0]), c(q[0]), s(q[1]), c(q[1]), s(q[2]), c(q[2])
        return rot_h([[cz*cy, cz*sy*sx - sz*cx, cz*sy*cx + sz*sx], [sz*cy, sz*sy*sx + cz*cx, sz*sy*cx - cz*sx],
                      [-sy, cy*sx, cy*cx]])
    if t == RZRY:
        sz, cz, sy, cy = s(q[0]), c(q[0]), s(q[1]), c(q[1])
        return rot_h([[cz*cy, -sz, cz*sy], [sz*cy, cz, sz*sy], [-sy, 0, cy]])
    if t == RZRX:
        sz, cz, sx, cx = s(q[0]), c(q[0]), s(q[1]), c(q[1])
        return rot_h([[cz, -sz*cx, sz*sx], [sz, cz*cx, -cz*sx], [0, sx, cx]])
    if t == RYRX:
        sy, cy, sx, cx = s(q[0]), c(q[0]), s(q[1]), c(q[1])
        return rot_h([[cy, sy*sx, sy*cx], [0, cx, -sx], [-sy, cy*sx, cy*cx]])
    if t == RZ:
        cc, ss = c(q[0]), s(q[0])
        return rot_h([[cc, -ss, 0], [ss, cc, 0], [0, 0, 1]])
    if t == RY:
        cc, ss = c(q[0]), s(q[0])
        return rot_h([[cc, 0, ss], [0, 1, 0], [-ss, 0, cc]])
    if t == RX:
        cc, ss = c(q[0]), s(q[0])
        return rot_h([[1, 0, 0], [0, cc, -ss], [0, ss, cc]])
    H = eye(4)
    H[0:3, 3] = q[0:3]
    return H


def joint_jacobian(t, q):
    if t == FREE:
        return eye(6)
    J = zeros(6, JOINT_NDOF[t])
    one, z = mp.mpf(1), mp.mpf(0)
    if t == RZRYRX:
        sx, cx, sy, cy = mp.sin(q[2]), mp.cos(q[2]), mp.sin(q[1]), mp.cos(q[1])
        J[0:3, :] = np.array([[-sy, z, one], [sx*cy, cx, z], [cx*cy, -sx, z]], dtype=object)
    elif t == RZRY:
        sy, cy = mp.sin(q[1]), mp.cos(q[1])
        J[0:3, :] = np.array([[-sy, z], [z, one], [cy, z]], dtype=object)
    elif t == RZRX:
        sx, cx = mp.sin(q[1]), mp.cos(q[1])
        J[0:3, :] = np.array([[z, one], [sx, z], [cx, z]], dtype=object)
    elif t == RYRX:
        sx, cx = mp.sin(q[1]), mp.cos(q[1])
        J[0:3, :] = np.array([[z, one], [cx, z], [-sx, z]], dtype=object)
    elif t == RZ:
        J[2, 0] = one
    elif t == RY:
        J[1, 0] = one
    elif t == RX:
        J[0, 0] = one
    else:
        J[3:6, :] = eye(3)
    return J


def joint_djacobian(t, q, dq):
    dJ = zeros(6, JOINT_NDOF[t])
    z = mp.mpf(0)
    if t == RZRYRX:
        sx, cx, sy, cy = mp.sin(q[2]), mp.cos(q[2]), mp.sin(q[1]), mp.cos(q[1])
        dx, dy = dq[2], dq[1]
        dJ[0:3, :] = np.array([[-dy*cy, z, z], [dx*cx*cy - dy*sx*sy, -dx*sx, z],
                               [-dx*sx*cy - dy*cx*sy, -dx*cx, z]], dtype=object)
    elif t == RZRY:
        sy, cy, dy = mp.sin(q[1]), mp.cos(q[1]), dq[1]
        dJ[0:3, :] = np.array([[-dy*cy, z], [z, z], [-dy*sy, z]], dtype=object)
    elif t == RZRX:
        sx, cx, dx = mp.sin(q[1]), mp.cos(q[1]), dq[1]
        dJ[0:3, :] = np.array([[z, z], [dx*cx, z], [-dx*sx, z]], dtype=object)
    elif t == RYRX:
        sx, cx, dx = mp.sin(q[1]), mp.cos(q[1]), dq[1]
        dJ[0:3, :] = np.array([[z, z], [-dx*sx, z], [-dx*cx, z]], dtype=object)
    return dJ


# -------------------------------------------------------------------------------------------
# dense LU with partial pivoting at DPS digits
# -------------------------------------------------------------------------------------------
class LU(object):
    def __init__(self, A):
        n = A.shape[0]
        a = [list(A[i]) for i in range(n)]
        perm = list(range(n))
        self.pivots = []
        for k in range(n):
            p = max(range(k, n), key=lambda i: abs(a[i][k]))
            if a[p][k] == 0:
                raise ZeroDivisionError("singular")
            a[k], a[p] = a[p], a[k]
            perm[k], perm[p] = perm[p], perm[k]
            piv = a[k][k]
            self.pivots.append(piv)
            rk = a[k]
            for i in range(k + 1, n):
                ri = a[i]
                f = ri[k]/piv
                if f != 0:
                    ri[k] = f
                    for j in range(k + 1, n):
                        ri[j] -= f*rk[j]
                else:
                    ri[k] = f
        self.a, self.perm, self.n = a, perm, n

    def solve(self, b):
        a, n = self.a, self.n
        y = [b[p] for p in self.perm]
        for i in range(n):
            ri = a[i]
            s = y[i]
            for j in range(i):
                s -= ri[j]*y[j]
            y[i] = s
        for i in range(n - 1, -1, -1):
            ri = a[i]
            s = y[i]
            for j in range(i + 1, n):
                s -= ri[j]*y[j]
            y[i] = s/ri[i]
        return np.array(y, dtype=object)

    def solve_cols(self, B):
        return np.stack([self.solve(B[:, j]) for j in range(B.shape[1])], axis=1) if B.shape[1] else zeros(self.n, 0)


# -------------------------------------------------------------------------------------------
# the world
# -------------------------------------------------------------------------------------------
class ArtRef(object):
    """One world at DPS digits.  model: dict of a FlatModel (body inertia, gravity and the PD gains of
    this world baked in); gpos, gvel: float64 state; cforce: warm-start forces (ball-and-socket rows);
    tau (ndof) and wrench {body: [torque; force] in ground axes at the body origin}: applied forces;
    gens: the library's generator layout (BatchedWorld.generators(): body, aligned, c0, limdof);
    mutate: names from MUTATIONS, applied to the reference itself."""

    def __init__(self, model, gpos, gvel, dt, gens, cforce=None, tau=None, wrench=None, mutate=()):
        for k in mutate:
            assert k in MUTATIONS, k
        self.mutate = set(mutate)
        with mp.workdps(DPS):
            self._build(model, gpos, gvel, dt, gens, cforce, tau, wrench)

    # -- update_dynamic (core.py:682-734, 1272-1315) -------------------------------------------
    def _build(self, m, gpos, gvel, dt, gens, cforce, tau, wrench):
        self.m = m
        n = self.n = int(m["ndof"])
        self.nj = nj = len(m["joint_type"])
        jt = [int(t) for t in m["joint_type"]]
        jp = [int(p) for p in m["joint_parent"]]
        jd = [int(d) for d in m["joint_dof"]]
        jg = [int(g) for g in m["joint_gpos"]]
        self.jt, self.jd, self.jg = jt, jd, jg
        Hpr = np.asarray(m["joint_Hpr"], dtype=float).reshape(nj, 4, 4)
        Hcn = np.asarray(m["joint_Hcn"], dtype=float).reshape(nj, 4, 4)
        bmass = np.asarray(m["body_mass"], dtype=float).reshape(nj, 6, 6)
        bvisc = np.asarray(m["body_visc"], dtype=float).reshape(nj, 6, 6)
        self.dt = mpf(dt)
        self.gpos_f, self.gvel_f = np.asarray(gpos, float), np.asarray(gvel, float)
        gp, gv = M(gpos), M(gvel)
        nb = nj + 1
        pose, jac, djac, twist, cols, nle = [None]*nb, [None]*nb, [None]*nb, [None]*nb, [None]*nb, [None]*nb
        depth = [0]*nb
        pose[0], jac[0], djac[0], twist[0], cols[0] = eye(4), zeros(6, n), zeros(6, n), zeros(6), []
        Mb = [None] + [M(bmass[j]) for j in range(nj)]
        Bb = [None] + [M(bvisc[j]) for j in range(nj)]
        for j in range(nj):               # depth-first order: parents first
            b, p, t = j + 1, jp[j], jt[j]
            q = gp[jg[j]:jg[j] + JOINT_NGPOS[t]]
            dq = gv[jd[j]:jd[j] + JOINT_NDOF[t]]
            H_cn, H_pr = M(Hcn[j]), M(Hpr[j])
            H_rn = joint_pose(t, q)
            H_pc = H_pr.dot(H_rn.dot(hinv(H_cn)))
            pose[b] = pose[p].dot(H_pc)
            Ad_cp, Ad_cn, Ad_rp = iadjoint(H_pc), adjoint(H_cn), adjoint(hinv(H_pr))
            J_nr, dJ_nr = joint_jacobian(t, q), joint_djacobian(t, q, dq)
            T_nr = dq.copy() if t == FREE else J_nr.dot(dq)
            iAd = adjoint(joint_pose(t, -q) if t in (RZ, RY, RX) else hinv(H_rn))
            dAd_nr = iAd.dot(adjacency(-iAd.dot(T_nr)))
            dAd_cp = Ad_cn.dot(dAd_nr.dot(Ad_rp))
            twist[b] = Ad_cp.dot(twist[p]) + Ad_cn.dot(T_nr)
            own = list(range(jd[j], jd[j] + JOINT_NDOF[t]))
            pc = cols[p]
            cols[b] = pc + own
            J, dJ = zeros(6, n), zeros(6, n)
            if pc:
                J[:, pc] = Ad_cp.dot(jac[p][:, pc])
                dJ[:, pc] = dAd_cp.dot(jac[p][:, pc]) + Ad_cp.dot(djac[p][:, pc])
            J[:, own] = J[:, own] + Ad_cn.dot(J_nr)
            dJ[:, own] = dJ[:, own] + Ad_cn.dot(dJ_nr)
            jac[b], djac[b] = J, dJ
            depth[b] = depth[p] + 1
        self.pose, self.jac, self.djac, self.twist, self.cols = pose, jac, djac, twist, cols
        # departure of the body rotations from orthogonality (a FreeJoint's rotation is float64 state):
        # hinv() takes R^T for R^-1, as the reference does
        self.orth = max([max(abs(x) for x in (pose[b][0:3, 0:3].T.dot(pose[b][0:3, 0:3]) - eye(3)).reshape(-1))
                         for b in range(1, nb)] or [mp.mpf(0)])
        self.depth = max(depth)
        # M, N, B and their absolute-value magnitudes (core.py:722-734)
        Mm, Nm, Bm = zeros(n, n), zeros(n, n), zeros(n, n)
        Za = zeros(n, n)
        for b in range(1, nb):
            c = cols[b]
            J, dJ, Mbb = jac[b][:, c], djac[b][:, c], Mb[b]
            wx = skew(twist[b][0:3])
            if Mbb[3, 3] <= mpf(1e-10):
                rx = zeros(3, 3)
            else:
                rx = Mbb[0:3, 3:6]/Mbb[3, 3]
            Om = zeros(6, 6)
            Om[0:3, 0:3] = wx
            Om[3:6, 3:6] = wx
            Om[0:3, 3:6] = rx.dot(wx) - wx.dot(rx)
            nle[b] = Om.dot(Mbb)
            ix = np.ix_(c, c)
            Mm[ix] += J.T.dot(Mbb.dot(J))
            Bm[ix] += J.T.dot(Bb[b].dot(J))
            Nm[ix] += J.T.dot(Mbb.dot(dJ) + nle[b].dot(J))
            aJ = mabs(J)
            Za[ix] += aJ.T.dot((mabs(Mbb)/self.dt + mabs(Bb[b])).dot(aJ) + mabs(Mbb).dot(mabs(dJ))
                               + (mabs(Om).dot(mabs(Mbb))).dot(aJ))
        self.M, self.N, self.B = Mm, Nm, Bm
        # update_controllers (core.py:811-818)
        g = zeros(n)
        ga = zeros(n)
        Zpd = zeros(n, n)
        up = M(m["up"])
        for k, t in enumerate(m["ctrl_type"]):
            if int(t) == 0:     # WeightController, controllers.py:43-60
                gd = zeros(6)
                gd[3:6] = mpf(np.asarray(m["ctrl_dbl"], dtype=float).reshape(-1, 4)[k][0])*up
                for b in range(1, nb):
                    if not (bmass[b - 1] > 0.).any():
                        continue
                    c = cols[b]
                    gb = iadjoint(pose[b]).dot(gd)
                    g[c] += jac[b][:, c].T.dot(Mb[b].dot(gb))
                    ga[c] += mabs(jac[b][:, c]).T.dot(mabs(Mb[b]).dot(mabs(iadjoint(pose[b])).dot(mabs(gd))))
            else:               # ProportionalDerivativeController, controllers.py:141-159
                ci = np.asarray(m["ctrl_int"]).reshape(-1, 4)[k]
                mm, off = int(ci[0]), int(ci[1])
                blob = np.asarray(m["ctrl_blob"], dtype=float)
                dofs = blob[off:off + mm].astype(int); off += mm
                gmap = blob[off:off + mm].astype(int); off += mm
                kp = M(blob[off:off + mm*mm].reshape(mm, mm)); off += mm*mm
                kd = M(blob[off:off + mm*mm].reshape(mm, mm)); off += mm*mm
                qd = M(blob[off:off + mm]); off += mm
                dqd = M(blob[off:off + mm])
                if "drop_PD" in self.mutate:
                    continue
                g[dofs] += kp.dot(qd - gp[gmap]) + kd.dot(dqd)
                ga[dofs] += mabs(kp).dot(mabs(qd) + mabs(gp[gmap])) + mabs(kd).dot(mabs(dqd))
                Zpd[np.ix_(dofs, dofs)] += self.dt*kp + kd
        if tau is not None:
            g += M(tau)
            ga += mabs(M(tau))
        for b, wv in (wrench or {}).items():
            wv = M(wv)
            R = pose[b][0:3, 0:3]
            loc = np.concatenate([R.T.dot(wv[0:3]), R.T.dot(wv[3:6])])
            if "flip_wrench" in self.mutate:
                loc = -loc
            c = cols[b]
            g[c] += jac[b][:, c].T.dot(loc)
            ga[c] += mabs(jac[b][:, c]).T.dot(np.concatenate([mabs(R.T).dot(mabs(wv[0:3])), mabs(R.T).dot(mabs(wv[3:6]))]))
        self.gforce = g
        Z = Mm/self.dt + Zpd
        if "drop_B" not in self.mutate:
            Z = Z + Bm
        if "drop_N" not in self.mutate:
            Z = Z + Nm
        self.Z = Z
        self.Zabs = Za + mabs(Zpd)
        self.lu = LU(Z)
        Zi = self.lu.solve_cols(eye(n))
        self.Zinv, self.aZinv = Zi, mabs(Zi)
        rhs = Mm.dot(gv)/self.dt + g
        self.rhs = rhs
        self.rhs_abs = (mabs(Mm)/self.dt).dot(mabs(gv)) + ga
        self.qfree = self.lu.solve(rhs)
        self.E_qfree = self.aZinv.dot(self.Zabs.dot(mabs(self.qfree)) + self.rhs_abs)
        # generators (arb_model_host.h layout, from the library)
        cd = np.asarray(m["cons_dbl"], dtype=float).reshape(-1, 48)
        self.gens = gens
        rows, arows, self.Re = [], [], []
        for gi, b in enumerate(gens["body"]):
            Jb = jac[b]
            if gens["aligned"][gi]:
                Rc = zaligned(cd[gens["c0"][gi]][32:35])[0:3, 0:3]
                Re = Rc.T.dot(pose[b][0:3, 0:3])
                self.Re.append(Re)
                if "unrotated" not in self.mutate or gi > 0:
                    Jb = np.concatenate([Re.dot(Jb[0:3]), Re.dot(Jb[3:6])])
                    # magnitude: the rotation is applied in float64 to the float64 rows
                    aJ = np.concatenate([mabs(Re).dot(mabs(jac[b][0:3])), mabs(Re).dot(mabs(jac[b][3:6]))])
                else:
                    aJ = mabs(Jb)
            else:
                self.Re.append(eye(3))
                aJ = mabs(Jb)
            rows.append(Jb)
            arows.append(aJ)
        for d in gens["limdof"]:
            e = zeros(1, n)
            e[0, d] = mp.mpf(1)
            rows.append(e)
            arows.append(e.copy())
        self.G = np.concatenate(rows) if rows else zeros(0, n)
        self.Ga = np.concatenate(arows) if arows else zeros(0, n)
        self.NG = self.G.shape[0]
        self.X = self.lu.solve_cols(self.G.T.copy())          # K = Z^-1 G^T
        self.v0 = self.G.dot(self.qfree)
        self.E_v0 = self.Ga.dot(self.E_qfree) + self.Ga.dot(mabs(self.qfree))
        L = self.G.dot(self.X)
        self.Lam = L.T.copy() if "lambda_T" in self.mutate else L
        aX = mabs(self.X)
        self.E_K = self.aZinv.dot(self.Zabs.dot(aX) + self.Ga.T)
        self.E_Lam = _row_floor(self.Ga.dot(self.E_K) + self.Ga.dot(aX), self.Lam)
        self.E_K = _row_floor(self.E_K, self.X)

    # -- A_cc from the constraint Jacobians (core.py:925-927) ----------------------------------
    def _frame(self, b, bpose):
        iAd = iadjoint(bpose)
        if b == 0:
            return bpose.copy(), zeros(self.n), zeros(6, self.n)
        return self.pose[b].dot(bpose), None, iAd.dot(self.jac[b])

    def constraint_jacobian(self, c):
        """(J_c, Ja, sides): the rows of constraint c formed the reference's way, the magnitude of their
        generator-space reduction |T1||J_b1| + |T0||J_b0| (the float64 code forms T G), and per body
        with generator rows (first row, T in the frame of those rows)"""
        with mp.workdps(DPS):
            m, n = self.m, self.n
            t = int(np.asarray(m["cons_type"]).reshape(-1)[c])
            ci = np.asarray(m["cons_int"]).reshape(-1, 4)[c]
            d = np.asarray(m["cons_dbl"], dtype=float).reshape(-1, 48)[c]
            if t == LIM:
                J = zeros(1, n)
                J[0, int(ci[1])] = mp.mpf(1)
                types = np.asarray(m["cons_type"]).reshape(-1)
                g = 6*len(self.gens["body"]) + int((types[:c] == LIM).sum())
                return J, J.copy(), [(g, eye(1))]
            b0, b1 = int(ci[0]), int(ci[1])
            if t == BALL:       # constraints.py:164-191
                cb0, cb1 = M(d[0:16].reshape(4, 4)), M(d[16:32].reshape(4, 4))
                r0 = 3
            else:
                cb0, cb1 = self._contact_frames(b0, b1, int(ci[2]), d)
                r0 = 2
            p0, _, J0 = self._frame(b0, cb0)
            p1, _, J1 = self._frame(b1, cb1)
            Ad01 = adjoint(hinv(p0).dot(p1))
            J = Ad01[r0:6].dot(J1) - J0[r0:6]
            T1 = Ad01[r0:6].dot(iadjoint(cb1))
            T0 = iadjoint(cb0)[r0:6]
            Ja = zeros(6 - r0, n)
            # the lever arms of T are formed in float64 from positions in ground axes: their rounding is
            # relative to those positions, not to the (possibly short) arm
            s = max(norm(p0[0:3, 3]), norm(p1[0:3, 3]), mp.mpf(1))
            sides = []
            for b, T in ((b1, T1), (b0, T0)):
                if b:
                    Ja = Ja + mabs(T).dot(mabs(self.jac[b]))
                    ang = mabs(self.jac[b][0:3]).sum(axis=0)
                    for r in range(max(0, 3 - r0), 6 - r0):
                        Ja[r] = Ja[r] + s*ang
                    gi = self.gens["body"].index(b)
                    Tg = T
                    if self.gens["aligned"][gi]:      # the rows of G are blockdiag(R_e, R_e) J_b
                        Re = self.Re[gi]
                        Tg = np.concatenate([T[:, 0:3].dot(Re.T), T[:, 3:6].dot(Re.T)], axis=1)
                    sides.append((6*gi, Tg))
            return J, Ja, sides

    def _contact_frames(self, b0, b1, pair, d):
        """contact frames on the two bodies (PointContact.update constraints.py:277-295 with
        collisions.py:67-111, as the oracle's _contact_update)"""
        bp0, bp1 = M(d[0:16].reshape(4, 4)), M(d[16:32].reshape(4, 4))
        H_g0 = self.pose[b0].dot(bp0)
        H_gp = self.pose[b1].dot(bp1)
        p_g1 = H_gp[0:3, 3]
        r0, r1 = mpf(d[41]), mpf(d[42])
        if pair == 1:
            p_g0 = H_g0[0:3, 3]
            vec = p_g1 - p_g0
            sdist = norm(vec) - r0 - r1
            normal = vec/norm(vec)
            H_gc0 = eye(4)
            H_gc0[0:3, 0:3] = _zaligned_mp(normal, tofloat(normal))
            H_gc0[0:3, 3] = p_g0 + r0*normal
            H_gc1 = H_gc0.copy()
            H_gc1[0:3, 3] = H_gc1[0:3, 3] + sdist*normal
        elif pair == 2:
            half = M(d[32:35])
            Hi = hinv(H_g0)
            p_01 = Hi[0:3, 0:3].dot(p_g1) + Hi[0:3, 3]
            if all(abs(p_01[i]) <= half[i] for i in range(3)):
                cand = [half[i] - p_01[i] for i in range(3)] + [half[i] + p_01[i] for i in range(3)]
                i = min(range(6), key=lambda k: cand[k])
                f_0 = p_01.copy()
                normal = zeros(3)
                if i < 3:
                    f_0[i], normal[i] = half[i], mp.mpf(1)
                else:
                    f_0[i - 3], normal[i - 3] = -half[i - 3], mp.mpf(-1)
                f_g = H_g0[0:3, 0:3].dot(f_0) + H_g0[0:3, 3]
            else:
                f_0 = np.array([max(min(half[i], p_01[i]), -half[i]) for i in range(3)], dtype=object)
                f_g = H_g0[0:3, 0:3].dot(f_0) + H_g0[0:3, 3]
                vec = p_g1 - f_g
                normal = vec/norm(vec)
            H_gc0 = eye(4)
            H_gc0[0:3, 0:3] = _zaligned_mp(normal, tofloat(normal))
            H_gc1 = H_gc0.copy()
            H_gc0[0:3, 3] = f_g
            H_gc1[0:3, 3] = p_g1 - r1*normal
        else:
            coeffs = M(d[32:36])
            normal = coeffs[0:3]
            Hi = hinv(H_g0)
            p_01 = Hi[0:3, 0:3].dot(p_g1) + Hi[0:3, 3]
            csdist = normal.dot(p_01) - coeffs[3]
            sdist = csdist - r1
            H_gc0 = zaligned(d[32:35])
            H_gc0[0:3, 3] = p_01 - csdist*normal
            H_gc1 = H_gc0.copy()
            H_gc1[0:3, 3] = p_01 - mp.sign(sdist)*r1*normal
        return hinv(self.pose[b0]).dot(H_gc0), hinv(self.pose[b1]).dot(H_gc1)

    def delassus(self, c):
        """(A_cc, E(A_cc)) of constraint c"""
        with mp.workdps(DPS):
            J, Ja, sides = self.constraint_jacobian(c)
            Xc = self.lu.solve_cols(J.T.copy())
            A = J.dot(Xc)
            aX = self.aZinv.dot(Ja.T)
            E = Ja.dot(self.aZinv.dot(self.Zabs.dot(aX) + Ja.T)) + Ja.dot(aX)
            # J_c goes through hinv(pose) pose, the identity only up to the rotations' departure from
            # orthogonality: the two exact forms J_c Z^-1 J_c^T and T Lambda T^T differ by that much
            E = E + (self.orth/U)*Ja.dot(aX)
            # the float64 code forms A_cc = T Lambda T^T from its own Lambda: Lambda's error, floor
            # included, reaches A_cc through |T|
            for gs, Ts in sides:
                for gt, Tt in sides:
                    ns, nt = Ts.shape[1], Tt.shape[1]
                    E = E + mabs(Ts).dot(self.E_Lam[gs:gs + ns, gt:gt + nt]).dot(mabs(Tt).T)
            return A, _row_floor(E, A)

    # -- the finish stage -------------------------------------------------------------------
    def finish(self, y):
        """(q'+, E(q'+), gpos+, E(gpos+)) for the generator-space wrench y (float64)"""
        with mp.workdps(DPS):
            yv = M(y)
            x = self.lu.solve(self.G.T.dot(yv))
            qn = self.qfree + x
            E = self.E_qfree + self.aZinv.dot(self.Zabs.dot(mabs(x)) + self.Ga.T.dot(mabs(yv)))
            gp = M(self.gpos_f)
            Eg = zeros(len(gp))
            for j in range(self.nj):
                t, g0, d0 = self.jt[j], self.jg[j], self.jd[j]
                nv = qn[d0:d0 + JOINT_NDOF[t]]
                if t == FREE:
                    h = self.dt/2 if "free_half_dt" in self.mutate else self.dt
                    H = gp[g0:g0 + 16].reshape(4, 4).dot(twist_exp(h*nv))
                    gp[g0:g0 + 16] = H.reshape(-1)
                    # rounding of the exponential and the 4x4 product, relative to the pose's size, and
                    # the velocity's own error carried through dt (both in units of C u)
                    hmax = max(abs(v) for v in H.reshape(-1))
                    s = 1 + hmax + self.dt*max(abs(v) for v in nv)
                    eb = self.dt*max(E[d0:d0 + 6])*(1 + hmax)
                    for i in range(16):
                        Eg[g0 + i] = 16*s + eb
                else:
                    for i in range(len(nv)):
                        gp[g0 + i] = gp[g0 + i] + self.dt*nv[i]
                        Eg[g0 + i] = abs(gp[g0 + i]) + self.dt*abs(nv[i]) + self.dt*E[d0 + i]
            return qn, E, gp, Eg

    # -- what the elimination sees ----------------------------------------------------------
    def sym_min_eig(self):
        """smallest eigenvalue of (Z + Z^T)/2"""
        with mp.workdps(DPS):
            S = tofloat((self.Z + self.Z.T)/2)
            return float(np.linalg.eigvalsh(S).min())

    def pivot_ratio(self):
        """min_k |d_k| / max |Z| of an UNPIVOTED elimination of Z in dof order (what the articulated
        elimination does, one scalar dof at a time)"""
        with mp.workdps(DPS):
            n = self.n
            a = [list(self.Z[i]) for i in range(n)]
            zmax = max(abs(x) for r in a for x in r)
            dmin = None
            for k in range(n - 1, -1, -1):            # leaf-to-root: highest dof first
                piv = a[k][k]
                dmin = abs(piv) if dmin is None else min(dmin, abs(piv))
                if piv == 0:
                    return 0.
                for i in range(k):
                    f = a[i][k]/piv
                    if f != 0:
                        for j in range(k):
                            a[i][j] -= f*a[k][j]
            return float(dmin/zmax)

    def cond_Z(self):
        with mp.workdps(DPS):
            return float(_norm1(self.Z)*_norm1(self.Zinv))


def _row_floor(E, A):
    """E_ij >= max_k |A_ik| (the module docstring)"""
    E = E.copy()
    for i in range(E.shape[0]):
        f = max([abs(x) for x in A[i]] or [mp.mpf(0)])
        for j in range(E.shape[1]):
            if E[i, j] < f:
                E[i, j] = f
    return E


def _norm1(A):
    return max(sum(abs(A[i, j]) for i in range(A.shape[0])) for j in range(A.shape[1]))


def _zaligned_mp(normal, normal_f):
    """zaligned() of a normal formed at DPS digits, the argsort on its float64 image"""
    z = normal
    idx = np.argsort(np.abs(normal_f), kind="stable")
    x = zeros(3)
    x[idx[1]] = z[idx[2]]
    x[idx[2]] = -z[idx[1]]
    x = x/norm(x)
    R = zeros(3, 3)
    R[:, 0] = x
    R[:, 1] = np.array([z[1]*x[2] - z[2]*x[1], z[2]*x[0] - z[0]*x[2], z[0]*x[1] - z[1]*x[0]], dtype=object)
    R[:, 2] = z
    return R


def bound_constant(ref):
    """C of the tolerance rule (module docstring)"""
    return 64.*(ref.depth + 6)


# -------------------------------------------------------------------------------------------
# float64 summary of one world, cached and computed in a process pool
# -------------------------------------------------------------------------------------------
def summary(job):
    """job = dict(model, gpos, gvel, dt, gens, cforce, tau, wrench, active, y, mutate); returns float64
    arrays: qfree, E_qfree, v0, E_v0, Lam, E_Lam, K, E_K, Re, acc {c: (A, E)}, finish (if y), cond_Z,
    sym_min_eig, pivot_ratio, C"""
    key = hashlib.sha256(pickle.dumps(_canon(job), protocol=4)).hexdigest()
    path = os.path.join(CACHE, key + ".pkl")
    if os.path.isfile(path):
        with open(path, "rb") as f:
            return pickle.load(f)
    r = ArtRef(job["model"], job["gpos"], job["gvel"], job["dt"], job["gens"], job.get("cforce"),
               job.get("tau"), job.get("wrench"), job.get("mutate", ()))
    with mp.workdps(DPS):
        out = {"qfree": tofloat(r.qfree), "E_qfree": tofloat(r.E_qfree), "v0": tofloat(r.v0),
               "E_v0": tofloat(r.E_v0), "Lam": tofloat(r.Lam).reshape(r.NG, r.NG),
               "E_Lam": tofloat(r.E_Lam).reshape(r.NG, r.NG), "K": tofloat(r.X).reshape(r.n, r.NG),
               "E_K": tofloat(r.E_K).reshape(r.n, r.NG), "Re": [tofloat(R) for R in r.Re],
               "cond_Z": r.cond_Z(), "sym_min_eig": r.sym_min_eig(), "pivot_ratio": r.pivot_ratio(),
               "C": bound_constant(r), "acc": {}}
        for c in job.get("active", ()):
            A, E = r.delassus(c)
            out["acc"][c] = (tofloat(A), tofloat(E))
        if job.get("y") is not None:
            qn, E, gp, Eg = r.finish(job["y"])
            out["finish"] = (tofloat(qn), tofloat(E), tofloat(gp), tofloat(Eg))
        for k in ("M", "N", "B", "Z", "gforce"):
            out[k] = tofloat(getattr(r, k))
    os.makedirs(CACHE, exist_ok=True)
    tmp = path + ".%d" % os.getpid()
    with open(tmp, "wb") as f:
        pickle.dump(out, f)
    os.replace(tmp, path)
    return out


def _canon(job):
    out = {}
    for k, v in sorted(job.items()):
        if k == "model":
            v = {kk: np.asarray(vv).tolist() for kk, vv in sorted(v.items()) if kk not in ("body_names", "joint_names")}
        elif isinstance(v, np.ndarray):
            v = v.tolist()
        out[k] = v
    return repr(out)


def run(jobs, processes=None):
    """summary() of every job, in a process pool"""
    import multiprocessing as mpr
    todo = [j for j in jobs]
    if len(todo) <= 1:
        return [summary(j) for j in todo]
    n = processes or min(len(todo), os.cpu_count() or 1)
    ctx = mpr.get_context("fork")
    with ctx.Pool(n) as pool:
        return pool.map(summary, todo, chunksize=1)


def err_ratio(x, ref, E, C):
    """worst |x - ref| / (C u E), NaN-aware (a NaN in x is an infinite ratio)"""
    x, ref, E = np.asarray(x, float), np.asarray(ref, float), np.asarray(E, float)
    d = np.abs(x - ref)
    d = np.where(np.isnan(d), np.inf, d)
    den = C*U*E + 1e-300
    return float((d/den).max()) if d.size else 0.
