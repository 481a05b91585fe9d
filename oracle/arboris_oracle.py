"""TEST INFRASTRUCTURE ONLY -- CPU restatement ("port") of the reference step.

This file restates, in plain numpy and one world at a time, the algorithm of
``sbarthelemy/arboris-python`` for the hot path of SURVEY.md section 8(a):
``update_dynamic -> update_controllers -> update_constraints -> integrate``.
It works on the *flattened* model (the dict ``FlatModel.to_dict()`` produces, or
an ``.npz`` fixture) so that it can run on the GPU box where ``/root/reference``
does not exist.  Only ``tests/``, ``__graft_entry__.smoke()`` and the
``cpu_baseline`` / ``--impl reference`` legs of ``bench.py`` may import it; the
product (``arboris-python_b200/``) never does.

PARITY PINNING: the restatement is checked by ``tests/test_oracle.py`` against
(1) the reference's own known-answer vectors -- ``tests/test_update_dynamic.py``
numbers, ``tests/test_human36.rst`` mass diagonals, the ``core.py:754-761``
impedance/admittance doctest, ``tests/test_constraints.py:53`` ball-and-socket
force, ``tests/simplearm_flat.h5`` (99-step trajectory), doctests of
``twistvector.exp``, ``zaligned`` and ``_plane_sphere_collision`` -- and (2)
fixtures in ``tests/golden/`` produced by running the *real* reference in the
build container (``oracle/make_goldens.py`` + ``oracle/ref_loader.py``), which
cover what the reference's tests leave unpinned (soft-finger static/sliding,
joint limits, the 42-dof model under contact).

Every function names the reference lines it follows.  The operation order of
the reference is kept wherever a comparison or branch depends on the result.
Conventions: twists are [angular; linear]; ``H_ab`` maps b-coordinates to a;
body Jacobians are expressed in the body frame; 4x4 matrices are row-major.
"""
import numpy as np
from numpy import array, zeros, eye, dot, sin, cos, hstack, diag
from numpy.linalg import norm, pinv, eigvals, solve, inv as _matinv

JOINT_NDOF = (6, 3, 2, 2, 2, 1, 1, 1, 3)
JOINT_NGPOS = (16, 3, 2, 2, 2, 1, 1, 1, 3)
FREE, RZRYRX, RZRY, RZRX, RYRX, RZ, RY, RX, TXTYTZ = range(9)
CONS_JOINT_LIMITS, CONS_BALL_SOCKET, CONS_SOFT_FINGER = 0, 1, 2
CONS_NDOL = (1, 3, 4)
CTRL_WEIGHT, CTRL_PD = 0, 1
# branch ids reported for SoftFingerContact.solve / JointLimits.solve
BR_NONE, BR_SEPARATING, BR_STATIC, BR_SLIDING = 0, 1, 2, 3
BR_JL_FREE, BR_JL_MIN, BR_JL_MAX = 1, 2, 3


# --------------------------------------------------------------------------
# rigid-motion math   (arboris/homogeneousmatrix.py, twistvector.py)
# --------------------------------------------------------------------------
def hinv(H):
    """homogeneousmatrix.py:254-275  inv(H) = [[R^T, -R^T p],[0,1]]"""
    R = H[0:3, 0:3]
    out = eye(4)
    out[0:3, 0:3] = R.T
    out[0:3, 3] = -dot(R.T, H[0:3, 3])
    return out


def skew(p):
    return array([[0., -p[2], p[1]], [p[2], 0., -p[0]], [-p[1], p[0], 0.]])


def adjoint(H):
    """homogeneousmatrix.py:277-319  Ad = [[R,0],[p^ R, R]]"""
    R = H[0:3, 0:3]
    Ad = zeros((6, 6))
    Ad[0:3, 0:3] = R
    Ad[3:6, 3:6] = R
    Ad[3:6, 0:3] = dot(skew(H[0:3, 3]), R)
    return Ad


def iadjoint(H):
    """homogeneousmatrix.py:321-325"""
    return adjoint(hinv(H))


def adjacency(tw):
    """twistvector.py:10-33"""
    ad = zeros((6, 6))
    ad[0:3, 0:3] = skew(tw[0:3])
    ad[3:6, 3:6] = skew(tw[0:3])
    ad[3:6, 0:3] = skew(tw[3:6])
    return ad


def twist_exp(tw):
    """twistvector.py:35-70  SE(3) exponential, series switch at |w| < 1e-3."""
    w = tw[0:3]
    v = tw[3:6]
    wx = skew(w)
    t = norm(w)
    if t >= 0.001:
        cc = (1 - cos(t))/t**2
        sc = sin(t)/t
        dsc = (t - sin(t))/t**3
    else:
        cc = 1./2.
        sc = 1. - t**2/6.
        dsc = 1./6.
    R = eye(3) + sc*wx + cc*dot(wx, wx)
    w31 = w.reshape(3, 1)
    p = dot(sc*eye(3) + cc*wx + dsc*dot(w31, w31.T), v)
    H = eye(4)
    H[0:3, 0:3] = R
    H[0:3, 3] = p
    return H


def rot_h(R):
    H = eye(4)
    H[0:3, 0:3] = R
    return H


def zaligned(vec):
    """homogeneousmatrix.py:201-232 (integer index work: argsort of |z|)."""
    H = eye(4)
    z = array(vec, dtype=float)
    idx = np.argsort(np.absolute(z), kind="stable")
    x = zeros(3)
    x[idx[0]] = 0
    x[idx[1]] = z[idx[2]]
    x[idx[2]] = -z[idx[1]]
    x /= norm(x)
    H[0:3, 0] = x
    H[0:3, 1] = np.cross(z, x)
    H[0:3, 2] = z
    return H, idx


# --------------------------------------------------------------------------
# joints   (arboris/joints.py)
# --------------------------------------------------------------------------
def joint_pose(t, q):
    """pose of each joint type: joints.py:38-40 (Free), :70-73, :118-120,
    :160-162, :199-201, :244-263, :313-315, :336-338, :362-365 with the closed
    forms of homogeneousmatrix.py:32-199."""
    if t == FREE:
        return q.reshape(4, 4).copy()
    if t == RZRYRX:
        sz, cz, sy, cy, sx, cx = sin(q[0]), cos(q[0]), sin(q[1]), cos(q[1]), sin(q[2]), cos(q[2])
        return rot_h(array([[cz*cy, cz*sy*sx - sz*cx, cz*sy*cx + sz*sx],
                            [sz*cy, sz*sy*sx + cz*cx, sz*sy*cx - cz*sx],
                            [-sy, cy*sx, cy*cx]]))
    if t == RZRY:
        sz, cz, sy, cy = sin(q[0]), cos(q[0]), sin(q[1]), cos(q[1])
        return rot_h(array([[cz*cy, -sz, cz*sy], [sz*cy, cz, sz*sy], [-sy, 0., cy]]))
    if t == RZRX:
        sz, cz, sx, cx = sin(q[0]), cos(q[0]), sin(q[1]), cos(q[1])
        return rot_h(array([[cz, -sz*cx, sz*sx], [sz, cz*cx, -cz*sx], [0., sx, cx]]))
    if t == RYRX:
        sy, cy, sx, cx = sin(q[0]), cos(q[0]), sin(q[1]), cos(q[1])
        return rot_h(array([[cy, sy*sx, sy*cx], [0., cx, -sx], [-sy, cy*sx, cy*cx]]))
    if t == RZ:
        c, s = cos(q[0]), sin(q[0])
        return rot_h(array([[c, -s, 0.], [s, c, 0.], [0., 0., 1.]]))
    if t == RY:
        c, s = cos(q[0]), sin(q[0])
        return rot_h(array([[c, 0., s], [0., 1., 0.], [-s, 0., c]]))
    if t == RX:
        c, s = cos(q[0]), sin(q[0])
        return rot_h(array([[1., 0., 0.], [0., c, -s], [0., s, c]]))
    if t == TXTYTZ:
        H = eye(4)
        H[0:3, 3] = q[0:3]
        return H
    raise ValueError(t)


def joint_ipose(t, q, pose):
    """rigidmotion.py:36-40 (inv of pose); Rz/Ry/Rx override it with rot(-q),
    joints.py:265-279, :317-319, :340-342."""
    if t in (RZ, RY, RX):
        return joint_pose(t, -q)
    return hinv(pose)


def joint_jacobian(t, q):
    """joints.py:46-48, :75-91, :122-135, :164-174, :203-213, :281-293, :321-323,
    :344-346, :367-375"""
    J = zeros((6, JOINT_NDOF[t]))
    if t == FREE:
        return eye(6)
    if t == RZRYRX:
        sx, cx, sy, cy = sin(q[2]), cos(q[2]), sin(q[1]), cos(q[1])
        J[0:3, :] = [[-sy, 0., 1.], [sx*cy, cx, 0.], [cx*cy, -sx, 0.]]
    elif t == RZRY:
        sy, cy = sin(q[1]), cos(q[1])
        J[0:3, :] = [[-sy, 0.], [0., 1.], [cy, 0.]]
    elif t == RZRX:
        sx, cx = sin(q[1]), cos(q[1])
        J[0:3, :] = [[0., 1.], [sx, 0.], [cx, 0.]]
    elif t == RYRX:
        sx, cx = sin(q[1]), cos(q[1])
        J[0:3, :] = [[0., 1.], [cx, 0.], [-sx, 0.]]
    elif t == RZ:
        J[2, 0] = 1.
    elif t == RY:
        J[1, 0] = 1.
    elif t == RX:
        J[0, 0] = 1.
    elif t == TXTYTZ:
        J[3:6, :] = eye(3)
    return J


def joint_djacobian(t, q, dq):
    """joints.py:50-52, :93-104, :137-146, :176-185, :215-224; zero for Rz/Ry/Rx
    (:295-303) and TxTyTz (:377-384)."""
    dJ = zeros((6, JOINT_NDOF[t]))
    if t == RZRYRX:
        sx, cx, sy, cy = sin(q[2]), cos(q[2]), sin(q[1]), cos(q[1])
        dx, dy = dq[2], dq[1]
        dJ[0:3, :] = [[-dy*cy, 0., 0.],
                      [dx*cx*cy - dy*sx*sy, -dx*sx, 0.],
                      [-dx*sx*cy - dy*cx*sy, -dx*cx, 0.]]
    elif t == RZRY:
        sy, cy, dy = sin(q[1]), cos(q[1]), dq[1]
        dJ[0:3, :] = [[-dy*cy, 0.], [0., 0.], [-dy*sy, 0.]]
    elif t == RZRX:
        sx, cx, dx = sin(q[1]), cos(q[1]), dq[1]
        dJ[0:3, :] = [[0., 0.], [dx*cx, 0.], [-dx*sx, 0.]]
    elif t == RYRX:
        sx, cx, dx = sin(q[1]), cos(q[1]), dq[1]
        dJ[0:3, :] = [[0., 0.], [-dx*sx, 0.], [-dx*cx, 0.]]
    return dJ


def softfinger_solve(v, A, f0, sdist, mu, eps, dt):
    """SoftFingerContact.solve constraints.py:780-836 for one contact: constraint velocity v (4),
    admittance block A (4x4), force f0 (4), signed distance, friction mu, eps (3), time step.  Keeps the
    reference's scalar inner-product quirk: Y_c, beta and b are 1-D, so every dot(x, y.T) below is a
    scalar that broadcasts over the 3x3 blocks.  Returns (branch, new force, force increment, (B, s) of a
    sliding solve or None)."""
    adm, vel, force0 = A, v, np.array(f0, dtype=float)
    vel_no_force = vel - dot(adm, force0)
    if sdist + dt*vel_no_force[3] > 0:
        return BR_SEPARATING, zeros(4), -force0, None
    dforce = dot(-pinv(adm), hstack((vel[0:3], vel[3] + sdist/dt)))
    force = force0 + dforce
    if sum((force[0:3]/eps)**2) <= (force[3]*mu)**2:
        return BR_STATIC, force, dforce, None
    alpha = vel - dot(adm, force0)
    alpha[3] += sdist/dt
    Y_c = adm[0:3, 3]
    y_n = adm[3, 3]
    Y_t = adm[0:3, 0:3]
    beta = alpha[0:3] - alpha[3]/y_n*Y_c
    a = mu/y_n*alpha[3]
    b = mu/y_n*Y_c
    B = zeros((6, 6))
    E = diag(eps**2)
    Y_that = Y_t - dot(Y_c, Y_c.T)/y_n
    B[3:6, 3:6] = dot(E, Y_that)
    B[0:3, 0:3] = dot(E, Y_that + 2/a*dot(beta, b.T))
    B[0:3, 3:6] = -dot(E, dot(beta, beta.T)/(a**2))
    B[3:6, 0:3] = dot(E, dot(b, b.T)) - eye(3)
    S = eigvals(B)
    S = S[np.logical_and(S.imag == 0, S.real <= 0)]
    if len(S) == 0:
        s = -1e10
    else:
        s = max(min(S.real), -1e10)
    A2 = adm.copy()
    A2[0:3, 0:3] -= s*diag(eps**-2)
    newf = solve(A2, -alpha)
    return BR_SLIDING, newf, newf - force0, (B.copy(), s)


# --------------------------------------------------------------------------
# the world
# --------------------------------------------------------------------------
class OracleWorld(object):
    """One world stepped with the reference's algorithm on a flat model.

    ``model`` is a mapping with the fields of ``FlatModel`` (numpy arrays).
    State: ``gpos`` (ngpos,), ``gvel`` (ndof,), ``cforce`` (nrows,) -- the
    per-constraint ``_force`` vectors stacked in registration order.
    After each phase the intermediate results are attributes (``mass``,
    ``nleffects``, ``viscosity``, ``impedance``, ``admittance``, ``gforce``,
    ``pose[b]``, ``jac[b]``, ``djac[b]``, ``twist[b]``, ``body_nle[b]``,
    ``active``, ``branch``, ``sdist`` ...), body index 0 being the ground.
    """

    def __init__(self, model):
        m = model
        self.m = m
        self.n = int(m["ndof"])
        self.nj = len(m["joint_type"])
        self.jt = [int(t) for t in m["joint_type"]]
        self.jp = [int(p) for p in m["joint_parent"]]
        self.jd = [int(d) for d in m["joint_dof"]]
        self.jg = [int(g) for g in m["joint_gpos"]]
        self.Hpr = np.asarray(m["joint_Hpr"], dtype=float)
        self.Hcn = np.asarray(m["joint_Hcn"], dtype=float)
        self.bmass = np.asarray(m["body_mass"], dtype=float)
        self.bvisc = np.asarray(m["body_visc"], dtype=float)
        self.children = [[] for _ in range(self.nj + 1)]
        for j in range(self.nj):
            self.children[self.jp[j]].append(j)
        self.nc = len(m["cons_type"])
        self.ct = [int(t) for t in m["cons_type"]]
        self.ci = np.asarray(m["cons_int"])
        self.cd = np.asarray(m["cons_dbl"], dtype=float)
        self.crow = [int(r) for r in m["cons_row"]]
        self.up = np.asarray(m["up"], dtype=float)
        self.gpos = np.array(m["gpos0"], dtype=float)
        self.gvel = np.array(m["gvel0"], dtype=float)
        self.cforce = np.array(m["cforce0"], dtype=float)
        self.time = 0.
        n = self.n
        self.mass = zeros((n, n))
        self.viscosity = zeros((n, n))
        self.nleffects = zeros((n, n))
        self.gforce = zeros(n)
        # WeightController.init, controllers.py:35-41 (norm(x.mass>0.) is truthy
        # when any entry of the body mass matrix is positive)
        self.massive = [b for b in range(1, self.nj + 1)
                        if norm(self.bmass[b - 1] > 0.)]

    # -- helpers ------------------------------------------------------------
    def _q(self, j):
        t = self.jt[j]
        return self.gpos[self.jg[j]:self.jg[j] + JOINT_NGPOS[t]]

    def _dq(self, j):
        t = self.jt[j]
        return self.gvel[self.jd[j]:self.jd[j] + JOINT_NDOF[t]]

    # -- update_dynamic  (core.py:682-734, 1272-1315) ---------------------------
    def update_dynamic(self):
        n, nb = self.n, self.nj + 1
        self.pose = [None]*nb
        self.jac = [None]*nb
        self.djac = [None]*nb
        self.twist = [None]*nb
        self.body_nle = [None]*nb
        # core.py:716-720
        self._body_update(0, eye(4), zeros((6, n)), zeros((6, n)), zeros(6))
        # core.py:722-734 (descendant bodies in depth-first order = index order)
        self.mass[:] = 0.
        self.viscosity[:] = 0.
        self.nleffects[:] = 0.
        for b in range(1, nb):
            J, dJ, Mb = self.jac[b], self.djac[b], self.bmass[b - 1]
            self.mass += dot(dot(J.T, Mb), J)
            self.viscosity += dot(dot(J.T, self.bvisc[b - 1]), J)
            self.nleffects += dot(J.T, dot(Mb, dJ) + dot(self.body_nle[b], J))

    def _body_update(self, b, pose, jac, djac, twist):
        self.pose[b], self.jac[b], self.djac[b], self.twist[b] = pose, jac, djac, twist
        mass = self.bmass[b - 1] if b > 0 else zeros((6, 6))
        # core.py:1276-1288
        wx = skew(twist[0:3])
        if mass[3, 3] <= 1e-10:
            rx = zeros((3, 3))
        else:
            rx = mass[0:3, 3:6]/mass[3, 3]
        nle = zeros((6, 6))
        nle[0:3, 0:3] = wx
        nle[3:6, 3:6] = wx
        nle[0:3, 3:6] = dot(rx, wx) - dot(wx, rx)
        self.body_nle[b] = dot(nle, mass)
        # core.py:1294-1315
        for j in self.children[b]:
            t = self.jt[j]
            q, dq = self._q(j), self._dq(j)
            H_cn, H_pr = self.Hcn[j], self.Hpr[j]
            H_rn = joint_pose(t, q)
            H_pc = dot(H_pr, dot(H_rn, hinv(H_cn)))
            child_pose = dot(pose, H_pc)
            Ad_cp = iadjoint(H_pc)
            Ad_cn = adjoint(H_cn)
            Ad_rp = adjoint(hinv(H_pr))
            J_nr = joint_jacobian(t, q)
            dJ_nr = joint_djacobian(t, q, dq)
            # Joint.twist core.py:197-201; FreeJoint.twist joints.py:42-44
            T_nr = dq.copy() if t == FREE else dot(J_nr, dq)
            # rigidmotion.py:36-75: idadjoint = iadjoint . adjacency(itwist)
            iAd = adjoint(joint_ipose(t, q, H_rn))
            itwist = -dot(iAd, T_nr)
            dAd_nr = dot(iAd, adjacency(itwist))
            dAd_cp = dot(Ad_cn, dot(dAd_nr, Ad_rp))
            child_twist = dot(Ad_cp, twist) + dot(Ad_cn, T_nr)
            sl = slice(self.jd[j], self.jd[j] + JOINT_NDOF[t])
            child_jac = dot(Ad_cp, jac)
            child_jac[:, sl] += dot(Ad_cn, J_nr)
            child_djac = dot(dAd_cp, jac) + dot(Ad_cp, djac)
            child_djac[:, sl] += dot(Ad_cn, dJ_nr)
            self._body_update(j + 1, child_pose, child_jac, child_djac, child_twist)

    # -- update_controllers  (core.py:811-818) ---------------------------------
    def update_controllers(self, dt):
        assert dt > 0
        n = self.n
        self.gforce[:] = 0.
        self.impedance = self.mass/dt + self.viscosity + self.nleffects
        m = self.m
        for k, t in enumerate(m["ctrl_type"]):
            if int(t) == CTRL_WEIGHT:
                g, Za = self._weight_controller(float(m["ctrl_dbl"][k][0]))
            else:
                g, Za = self._pd_controller(k, dt)
            self.gforce += g
            self.impedance -= Za
        self.admittance = _matinv(self.impedance)

    def _weight_controller(self, gravity):
        """controllers.py:43-60 (the principalframe() call there is dead work)."""
        n = self.n
        gravity_dtwist = zeros(6)
        gravity_dtwist[3:6] = float(gravity)*self.up
        gforce = zeros(n)
        for b in self.massive:
            g = dot(iadjoint(self.pose[b]), gravity_dtwist)
            gforce += dot(self.jac[b].T, dot(self.bmass[b - 1], g))
        return gforce, zeros((n, n))

    def _pd_controller(self, k, dt):
        """controllers.py:141-159"""
        n = self.n
        mm, off = int(self.m["ctrl_int"][k][0]), int(self.m["ctrl_int"][k][1])
        blob = np.asarray(self.m["ctrl_blob"], dtype=float)
        dofs = blob[off:off + mm].astype(int); off += mm
        gmap = blob[off:off + mm].astype(int); off += mm
        kp = blob[off:off + mm*mm].reshape(mm, mm); off += mm*mm
        kd = blob[off:off + mm*mm].reshape(mm, mm); off += mm*mm
        q_des = blob[off:off + mm]; off += mm
        dq_des = blob[off:off + mm]
        gforce = zeros(n)
        impedance = zeros((n, n))
        gforce[dofs] = dot(kp, q_des - self.gpos[gmap]) + dot(kd, dq_des)
        impedance[np.ix_(dofs, dofs)] = -(dt*kp + kd)
        return gforce, impedance

    # -- frames attached to bodies (core.py:1017-1032) ---------------------------
    def _frame(self, b, bpose):
        iAd = iadjoint(bpose)
        n = self.n
        if b == 0:
            return bpose.copy(), zeros(6), zeros((6, n))
        return (dot(self.pose[b], bpose), dot(iAd, self.twist[b]),
                dot(iAd, self.jac[b]))

    # -- update_constraints  (core.py:910-937) -----------------------------------
    def update_constraints(self, dt):
        assert dt > 0
        n = self.n
        nc = self.nc
        self.active = [False]*nc
        self.sdist = [0.]*nc
        self.branch = [BR_NONE]*nc     # branch of the LAST Gauss-Seidel sweep
        self.zidx = [None]*nc
        cjac = [None]*nc
        aux = [None]*nc
        act = []
        dol = {}
        ndol = 0
        f = self.cforce
        for c in range(nc):
            t = self.ct[c]
            if not int(self.ci[c][3]):       # is_enabled
                continue
            r0 = self.crow[c]
            rows = slice(r0, r0 + CONS_NDOL[t])
            if t == CONS_JOINT_LIMITS:
                # constraints.py:65-71
                q = self.gpos[int(self.ci[c][2])]
                f[rows] = 0.
                mn, mx, prox = self.cd[c][0:3]
                self.active[c] = bool((q - mn < prox) or (mx - q < prox))
                J = zeros((1, n))
                J[0, int(self.ci[c][1])] = 1
                cjac[c] = J
                aux[c] = q
            elif t == CONS_BALL_SOCKET:
                # constraints.py:164-191 (force is NOT reset: warm start)
                p0, _, J0 = self._frame(int(self.ci[c][0]), self.cd[c][0:16].reshape(4, 4))
                p1, _, J1 = self._frame(int(self.ci[c][1]), self.cd[c][16:32].reshape(4, 4))
                H_01 = dot(hinv(p0), p1)
                aux[c] = H_01[0:3, 3].copy()
                self.active[c] = True
                cjac[c] = dot(adjoint(H_01)[3:6, :], J1) - J0[3:6, :]
            else:
                cjac[c], aux[c] = self._contact_update(c, dt)
                f[rows] = 0.
            if self.active[c]:
                dol[c] = slice(ndol, ndol + CONS_NDOL[t])
                ndol += CONS_NDOL[t]
                act.append(c)
        # core.py:920-927
        jac = zeros((ndol, n))
        gforce = self.gforce.copy()
        for c in act:
            jac[dol[c], :] = cjac[c]
            r0 = self.crow[c]
            gforce += dot(cjac[c].T, f[r0:r0 + CONS_NDOL[self.ct[c]]])
        vel = dot(jac, dot(self.admittance, dot(self.mass, self.gvel/dt) + gforce))
        adm = dot(jac, dot(self.admittance, jac.T))
        self.cons_jac, self.cons_vel0, self.cons_adm = jac, vel.copy(), adm
        self.cons_dol = dol
        # core.py:929-935: 20 sweeps, no convergence test
        for _ in range(20):
            for c in act:
                r0 = self.crow[c]
                t = self.ct[c]
                rows = slice(r0, r0 + CONS_NDOL[t])
                v = vel[dol[c]]
                A = adm[dol[c], dol[c]]
                if t == CONS_JOINT_LIMITS:
                    df = self._solve_limits(c, v, A, dt, aux[c], rows)
                elif t == CONS_BALL_SOCKET:
                    # constraints.py:235-237
                    df = -dot(pinv(A), v + aux[c]/dt)
                    f[rows] += df
                else:
                    df = self._solve_softfinger(c, v, A, dt, rows)
                vel += dot(adm[:, dol[c]], df)
        self.cons_vel = vel
        # core.py:936-937
        for c in act:
            r0 = self.crow[c]
            self.gforce += dot(cjac[c].T, f[r0:r0 + CONS_NDOL[self.ct[c]]])

    def _contact_update(self, c, dt):
        """PointContact.update constraints.py:277-295 with the collision solvers
        collisions.py:67-111 (shape pair ordered by choose_solver :14-65) and
        SoftFingerContact.jacobian constraints.py:429-433."""
        b0, b1, pair = int(self.ci[c][0]), int(self.ci[c][1]), int(self.ci[c][2])
        d = self.cd[c]
        bp0 = d[0:16].reshape(4, 4)     # shape 0 frame on body b0
        bp1 = d[16:32].reshape(4, 4)    # shape 1 frame on body b1
        prox = d[40]
        radius0, radius1 = d[41], d[42]
        H_g0, _, _ = self._frame(b0, bp0)
        H_gp, _, _ = self._frame(b1, bp1)
        p_g1 = H_gp[0:3, 3]
        if pair == 1:
            # _sphere_sphere_collision collisions.py:150-159
            p_g0 = H_g0[0:3, 3]
            vec = p_g1 - p_g0
            sdist = norm(vec) - radius0 - radius1
            normal = vec/norm(vec)
            H_gc0, idx = zaligned(normal)
            z = H_gc0[0:3, 2]
            H_gc0[0:3, 3] = p_g0 + radius0*z
            H_gc1 = H_gc0.copy()
            H_gc1[0:3, 3] += sdist*z
        elif pair == 2:
            # _box_sphere_collision collisions.py:268-299
            half = d[32:35]
            Hi = hinv(H_g0)
            p_01 = dot(Hi[0:3, 0:3], p_g1) + Hi[0:3, 3]
            if (abs(p_01) <= half).all():
                i = int(np.argmin(np.hstack((half - p_01, half + p_01))))
                f_0 = p_01.copy()
                normal = zeros(3)
                if i < 3:
                    f_0[i] = half[i]
                    normal[i] = 1
                else:
                    f_0[i - 3] = -half[i - 3]
                    normal[i - 3] = -1
                f_g = dot(H_g0[0:3, 0:3], f_0) + H_g0[0:3, 3]
                sdist = -norm(f_g - p_g1) - radius1
            else:
                f_0 = np.maximum(np.minimum(half, p_01), -half)
                f_g = dot(H_g0[0:3, 0:3], f_0) + H_g0[0:3, 3]
                vec = p_g1 - f_g
                normal = vec/norm(vec)
                sdist = norm(vec) - radius1
            H_gc0, idx = zaligned(normal)
            H_gc1 = H_gc0.copy()
            H_gc0[0:3, 3] = f_g
            H_gc1[0:3, 3] = p_g1 - radius1*normal
        else:
            # _plane_sphere_collision collisions.py:193-205 (a Point has radius 0)
            coeffs = d[32:36]
            normal = coeffs[0:3]
            Hi = hinv(H_g0)
            p_01 = dot(Hi[0:3, 0:3], p_g1) + Hi[0:3, 3]
            csdist = dot(normal, p_01) - coeffs[3]
            sdist = csdist - radius1
            H_gc0, idx = zaligned(normal)
            H_gc0[0:3, 3] = p_01 - csdist*normal
            H_gc1 = H_gc0.copy()
            H_gc1[0:3, 3] = p_01 - np.sign(sdist)*radius1*normal
        # PointContact.update: contact frames become moving subframes of the bodies
        pose_b0 = self.pose[b0] if b0 > 0 else eye(4)
        pose_b1 = self.pose[b1] if b1 > 0 else eye(4)
        bpose0 = dot(hinv(pose_b0), H_gc0)
        bpose1 = dot(hinv(pose_b1), H_gc1)
        f0_pose, f0_twist, f0_jac = self._frame(b0, bpose0)
        f1_pose, f1_twist, f1_jac = self._frame(b1, bpose1)
        H_c0c1 = dot(hinv(H_gc0), H_gc1)
        dsdist = dot(adjoint(H_c0c1)[5, :], f1_twist) - f0_twist[5]
        self.active[c] = bool(sdist + dsdist*dt < prox)
        self.sdist[c] = sdist
        self.zidx[c] = idx
        H_01 = dot(hinv(f0_pose), f1_pose)
        J = dot(adjoint(H_01)[2:6, :], f1_jac) - f0_jac[2:6, :]
        return J, sdist

    def _solve_limits(self, c, vel, adm, dt, pos0, rows):
        """JointLimits.solve constraints.py:73-90"""
        f = self.cforce
        mn, mx = self.cd[c][0:2]
        pred = pos0 + dt*(vel - dot(adm, f[rows]))
        prev = f[rows].copy()
        if pred <= mn:
            f[rows] = dot(pinv(adm), (mn - pred)/dt)
            self.branch[c] = BR_JL_MIN
            return f[rows] - prev
        elif mx <= pred:
            f[rows] = dot(pinv(adm), (mx - pred)/dt)
            self.branch[c] = BR_JL_MAX
            return f[rows] - prev
        else:
            df = -f[rows]
            f[rows] = 0.
            self.branch[c] = BR_JL_FREE
            return df

    def _solve_softfinger(self, c, vel, adm, dt, rows):
        """SoftFingerContact.solve constraints.py:780-836 (softfinger_solve below)."""
        f = self.cforce
        force0 = f[rows].copy()
        br, newf, df, slide = softfinger_solve(vel, adm, force0, self.sdist[c], self.cd[c][36], self.cd[c][37:40], dt)
        f[rows] = newf
        self.branch[c] = br
        if slide is not None:
            self.last_slide = slide
        return df

    # -- integrate  (core.py:974-980) ----------------------------------------------
    def integrate(self, dt):
        assert dt > 0
        self.gvel[:] = dot(self.admittance,
                           dot(self.mass, self.gvel/dt) + self.gforce)
        for j in range(self.nj):
            t = self.jt[j]
            q, dq = self._q(j), self._dq(j)
            if t == FREE:
                # joints.py:54-57
                q[:] = dot(q.reshape(4, 4), twist_exp(dt*dq)).reshape(-1)
            else:
                # core.py:238-240
                q += dt*dq
        self.time += dt

    def step(self, dt):
        """One iteration of the simulate() loop, core.py:1356-1363."""
        self.update_dynamic()
        self.update_controllers(dt)
        self.update_constraints(dt)
        self.integrate(dt)
