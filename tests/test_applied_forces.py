"""Per-world applied forces (arb_batch_bind_applied_forces) in the CPU build of the device routines:
generalized forces and body wrenches on both the phase routines and the fused step, against the
oracle extended with the controller they stand for."""
import os
import sys

import numpy as np
import pytest

HOSTTEST = os.path.join(os.path.dirname(__file__), "hosttest")
sys.path.insert(0, HOSTTEST)
import harness  # noqa: E402

from conftest import GOLDEN  # noqa: E402

APPLIED_SRC = os.path.join(HOSTTEST, "arb_hosttest_applied.cpp")
APPLIED_OUT = os.path.join(HOSTTEST, "_build", "libarb_hosttest_applied.so")
_applied_lib = None


def applied_lib():
    """the host build with the applied-force exports (arb_hosttest_applied.cpp), built as harness.build()
    builds arb_hosttest.cpp"""
    global _applied_lib
    if _applied_lib is not None:
        return _applied_lib
    import ctypes as C
    import subprocess
    deps = [APPLIED_SRC, harness.SRC] + [os.path.join(harness.CSRC, f) for f in os.listdir(harness.CSRC)]
    if not (os.path.isfile(APPLIED_OUT) and all(os.path.getmtime(APPLIED_OUT) >= os.path.getmtime(d) for d in deps)):
        os.makedirs(os.path.dirname(APPLIED_OUT), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", APPLIED_OUT, APPLIED_SRC])
    L = C.CDLL(APPLIED_OUT)
    base = harness.lib()          # the prototypes harness sets, for the same exports of this library
    for name in ("ht_create", "ht_destroy", "ht_bind", "ht_update_dynamic", "ht_update_controllers",
                 "ht_update_constraints", "ht_integrate", "ht_fused_step", "ht_array", "ht_iarray", "ht_fused_ints"):
        getattr(L, name).restype = getattr(base, name).restype
        getattr(L, name).argtypes = getattr(base, name).argtypes
    L.ht_bind_applied.restype = C.c_int
    L.ht_bind_applied.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
    L.ht_release_applied.argtypes = [C.c_void_p]
    L.ht_applied_update_controllers.argtypes = [C.c_void_p, C.c_double]
    L.ht_applied_fused_step.argtypes = [C.c_void_p, C.c_double]
    _applied_lib = L
    return L


class AppliedHostBatch(harness.HostBatch):
    """harness.HostBatch on the library with the applied forces: update_controllers and fused_step add
    what bind_applied bound (nothing until then)."""

    def __init__(self, model, W):
        import ctypes as C
        self.L = applied_lib()
        self.model, self.W = model, W
        self.desc, self._keep = harness._capi.make_desc(model)
        err = C.create_string_buffer(256)
        self.h = self.L.ht_create(C.byref(self.desc), W, err, 256)
        if not self.h:
            raise RuntimeError(err.value.decode())
        self.gpos = np.zeros((model.ngpos, W))
        self.gvel = np.zeros((model.ndof, W))
        self.cforce = np.zeros((max(model.nrows, 1), W))
        self.L.ht_bind(self.h, self.gpos.ctypes.data, self.gvel.ctypes.data, self.cforce.ctypes.data)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ht_release_applied(self.h)
        harness.HostBatch.__del__(self)

    def bind_applied(self, tau=None, wrench=None, bodies=()):
        """tau (ndof, W), wrench (len(bodies), 6, W), ``None`` for none (kept alive here); raises
        ValueError with the library's message for bad bodies"""
        import ctypes as C
        self._applied = [None if a is None else np.ascontiguousarray(a, dtype=np.float64) for a in (tau, wrench)]
        self._applied_bodies = np.ascontiguousarray(bodies, dtype=np.int32).reshape(-1)
        err = C.create_string_buffer(256)
        ptr = [None if a is None else a.ctypes.data for a in self._applied]
        rc = self.L.ht_bind_applied(self.h, ptr[0], len(self._applied_bodies),
                                    self._applied_bodies.ctypes.data if len(self._applied_bodies) else None,
                                    ptr[1], err, 256)
        if rc:
            raise ValueError(err.value.decode())

    def update_controllers(self, dt):
        self.L.ht_applied_update_controllers(self.h, dt)

    def fused_step(self, dt):
        self.L.ht_applied_fused_step(self.h, dt)

DT = 1e-3
S0 = 40            # first state: the reference's step 40 of the 64 falling humanoids, most of them in contact
NSTEPS = 8
NW = 32
# pelvis, both feet (they carry the contacts) and the left scapula (no mass)
BODIES = (1, 4, 7, 9)


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max()/max(np.abs(b).max(), 1e-300)


def _contact64():
    from arboris_b200.flatten import FlatModel
    model = FlatModel.load(os.path.join(GOLDEN, "model_human36_contact.npz"))
    with np.load(os.path.join(GOLDEN, "traj_human36_contact64.npz")) as z:
        tr = {k: z[k] for k in z.files}
    return model, tr


def applied_forces(model, W, seed=0):
    """Random per-world forces large enough to move the contacts: tau (ndof, W), wrench (nsel, 6, W)."""
    rng = np.random.default_rng(seed)
    tau = rng.normal(scale=5., size=(model.ndof, W))
    wrench = np.concatenate((rng.normal(scale=20., size=(len(BODIES), 3, W)),
                             rng.normal(scale=300., size=(len(BODIES), 3, W))), axis=1)
    return tau, wrench


def applied_oracle(model, tau, wrench, bodies):
    """OracleWorld with one more controller after the model's: tau + sum_b J_b^T [R_b^T t; R_b^T f]."""
    from oracle.arboris_oracle import OracleWorld

    class AppliedOracle(OracleWorld):
        def update_controllers(self, dt):
            OracleWorld.update_controllers(self, dt)
            g = tau.copy()
            for b, w in zip(bodies, wrench):
                R = self.pose[b][0:3, 0:3]
                g += np.dot(self.jac[b].T, np.concatenate((np.dot(R.T, w[0:3]), np.dot(R.T, w[3:6]))))
            self.gforce += g

    return AppliedOracle(model.to_dict())


def test_human36_massless_and_contact_bodies():
    """the body list exercises a massless body and the two contact-carrying feet"""
    model, _ = _contact64()
    bm = np.asarray(model.body_mass)
    assert not (bm[9 - 1] > 0).any()
    cbodies = {int(c[1]) for t, c in zip(model.cons_type, model.cons_int) if int(t) == 2}
    assert cbodies == {4, 7} and cbodies <= set(BODIES)


@pytest.mark.parametrize("path", ["phases", "fused"])
def test_applied_forces_vs_oracle(path):
    """Teacher-forced from the oracle's own states: velocities within 1e-10 relative, active sets and
    branches identical; on the phases, World._gforce after update_controllers as well."""
    model, tr = _contact64()
    W = NW
    tau, wrench = applied_forces(model, W)
    hb = AppliedHostBatch(model, W)
    hb.set_coop(0)
    hb.bind_applied(tau, wrench, BODIES)
    oracles = []
    for w in range(W):
        o = applied_oracle(model, tau[:, w], wrench[:, :, w], BODIES)
        o.gpos[:], o.gvel[:], o.cforce[:] = tr["gpos"][w, S0], tr["gvel"][w, S0], tr["cforce"][w, S0]
        oracles.append(o)
    worst, flips, moved, nact = {}, 0, 0, 0
    for s in range(NSTEPS):
        hb.gpos[:] = np.stack([o.gpos for o in oracles], 1)
        hb.gvel[:] = np.stack([o.gvel for o in oracles], 1)
        hb.cforce[:] = np.stack([o.cforce for o in oracles], 1)
        if path == "phases":
            hb.update_dynamic()
            hb.update_controllers(DT)
            gf = hb.arr("gforce", model.ndof).copy()
            hb.update_constraints(DT)
            hb.integrate(DT)
            act, br = hb.iarr("cactive", model.nc).T, hb.iarr("cbranch", model.nc).T
        else:
            hb.fused_step(DT)
            act, br = hb.iarr("factive", model.nc).T, hb.iarr("fbranch", model.nc).T
        for w, o in enumerate(oracles):
            o.update_dynamic()
            o.update_controllers(DT)
            if path == "phases":
                worst["gforce"] = max(worst.get("gforce", 0.), rel(gf[:, w], o.gforce))
            o.update_constraints(DT)
            o.integrate(DT)
            a = np.array(o.active, dtype=int)
            flips += int((act[w] != a).sum()) + int((br[w]*act[w] != np.array(o.branch)*a).sum())
            nact += int(a.sum())
            worst["gvel"] = max(worst.get("gvel", 0.), rel(hb.gvel[:, w], o.gvel))
            worst["gpos"] = max(worst.get("gpos", 0.), rel(hb.gpos[:, w], o.gpos))
            worst["cforce"] = max(worst.get("cforce", 0.), rel(hb.cforce[:model.nrows, w], o.cforce))
            if s == 0:     # the same state without the forces: the reference's own step S0 + 1
                moved += int((a != tr["active"][w, S0 + 1]).sum()) + \
                    int((np.array(o.branch)*a != tr["branch"][w, S0 + 1]).sum())
    assert nact > 100, "the states must be in contact"
    assert moved > 0, "the forces must change some contact branches"
    assert flips == 0, "active set / branch flips: %d" % flips
    assert not (hb.iarr("status") & 3).any()     # (NONFINITE, SINGULAR; EIG_NOROOT is the reference's clamp)
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


def _run(model, tr, path, bind):
    W = NW
    hb = AppliedHostBatch(model, W)
    hb.set_coop(0)
    if bind:
        hb.bind_applied(np.zeros((model.ndof, W)), np.zeros((len(BODIES), 6, W)), BODIES)
    hb.gpos[:], hb.gvel[:] = tr["gpos"][:W, S0].T, tr["gvel"][:W, S0].T
    hb.cforce[:] = tr["cforce"][:W, S0].T
    for _ in range(NSTEPS):
        if path == "phases":
            hb.update_dynamic(); hb.update_controllers(DT); hb.update_constraints(DT); hb.integrate(DT)
        else:
            hb.fused_step(DT)
    return hb.gpos.copy(), hb.gvel.copy(), hb.cforce.copy()


@pytest.mark.parametrize("path", ["phases", "fused"])
def test_zero_applied_forces_change_nothing(path):
    """bound arrays of zeros give the results of nothing bound, bit for bit"""
    model, tr = _contact64()
    ref = _run(model, tr, path, False)
    got = _run(model, tr, path, True)
    for a, b in zip(ref, got):
        assert a.tobytes() == b.tobytes()


def test_bad_wrench_bodies_are_refused():
    model, _ = _contact64()
    hb = AppliedHostBatch(model, 2)
    w1 = np.zeros((1, 6, 2))
    for bodies, msg in (((0,), "ground"), ((len(model.joint_type) + 1,), "out of range"), ((-1,), "out of range")):
        with pytest.raises(ValueError, match=msg):
            hb.bind_applied(None, w1, bodies)
    with pytest.raises(ValueError, match="twice"):
        hb.bind_applied(None, np.zeros((2, 6, 2)), (3, 3))
    with pytest.raises(ValueError, match="needs its bodies"):
        hb.bind_applied(None, w1, ())
    hb.bind_applied(np.zeros((model.ndof, 2)), None, ())      # generalized forces alone
