"""Per-world contact friction (arb_batch_bind_contact_friction) in the CPU build of the device routines:
the phase routine and the fused step (per-lane and block-cooperative Gauss-Seidel, and the group
prepare stage) against the oracle on each world's own model, bit-identity with a batch built from that
model and with the unbound step, a binding that is read (sliding contacts that stick at mu = 5), and
the refusals."""
import os
import sys

import numpy as np
import pytest

HOSTTEST = os.path.join(os.path.dirname(__file__), "hosttest")
sys.path.insert(0, HOSTTEST)
sys.path.insert(0, os.path.dirname(__file__))
import harness  # noqa: E402

import contactfriction as cf  # noqa: E402

SRC = os.path.join(HOSTTEST, "arb_hosttest_friction.cpp")
OUT = os.path.join(HOSTTEST, "_build", "libarb_hosttest_friction.so")
_lib = None
FIXTURES = sorted(cf.FIXTURES)
PATHS = ["phases", "lane", "coop"]


def fr_lib():
    """the host build with the friction exports (arb_hosttest_friction.cpp), built as harness.build()
    builds arb_hosttest.cpp"""
    global _lib
    if _lib is not None:
        return _lib
    import ctypes as C
    import subprocess
    deps = [SRC, harness.SRC] + [os.path.join(harness.CSRC, f) for f in os.listdir(harness.CSRC)]
    if not (os.path.isfile(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in deps)):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-ffp-contract=off",
                               "-Wno-unknown-pragmas", "-o", OUT, SRC])
    L = C.CDLL(OUT)
    base = harness.lib()
    for name in ("ht_create", "ht_destroy", "ht_bind", "ht_update_dynamic", "ht_update_controllers",
                 "ht_update_constraints", "ht_integrate", "ht_fused_step", "ht_array", "ht_iarray", "ht_fused_ints"):
        getattr(L, name).restype = getattr(base, name).restype
        getattr(L, name).argtypes = getattr(base, name).argtypes
    L.ht_set_coop.argtypes = [C.c_void_p, C.c_int]
    L.ht_bind_friction.restype = C.c_int
    L.ht_bind_friction.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
    L.ht_release_friction.argtypes = [C.c_void_p]
    L.ht_fr_update_constraints.argtypes = [C.c_void_p, C.c_double]
    L.ht_fr_fused_step.argtypes = [C.c_void_p, C.c_double, C.c_int]
    _lib = L
    return L


class FrictionHostBatch(harness.HostBatch):
    """harness.HostBatch on the library with the friction exports: update_constraints and the fused
    step read what bind_friction bound (nothing until then)"""

    def __init__(self, model, W):
        import ctypes as C
        self.L = fr_lib()
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
            self.L.ht_release_friction(self.h)
        harness.HostBatch.__del__(self)

    def bind_friction(self, constraints=(), mu=None):
        """mu (len(constraints), W) or None (kept alive here); raises ValueError with the library's message"""
        import ctypes as C
        m = None if mu is None else np.ascontiguousarray(mu, dtype=np.float64)
        ids = np.ascontiguousarray(constraints, dtype=np.int32).reshape(-1)
        err = C.create_string_buffer(256)
        rc = self.L.ht_bind_friction(self.h, len(ids), ids.ctypes.data if len(ids) else None,
                                     None if m is None else m.ctypes.data, err, 256)
        if rc:
            raise ValueError(err.value.decode())
        self._fr = (m, ids)

    def set_state(self, st):
        self.gpos[:], self.gvel[:] = st[0], st[1]
        self.cforce[:st[2].shape[0]] = st[2]

    def step(self, path, dt=cf.DT):
        if path == "phases":
            self.update_dynamic()
            self.update_controllers(dt)
            self.L.ht_fr_update_constraints(self.h, dt)
            self.integrate(dt)
        else:
            self.set_coop(1 if path == "coop" else 0)
            self.L.ht_fr_fused_step(self.h, dt, 1 if path == "group" else 0)

    def flags(self, path):
        """(active, branch) of the last step, (W, nc)"""
        nc = len(self.model.cons_type)
        if path == "phases":
            return self.iarr("cactive", nc).T.copy(), self.iarr("cbranch", nc).T.copy()
        import ctypes as C
        out = []
        for k in ("factive", "fbranch"):
            a = np.zeros((nc, self.W), dtype=np.int32)
            self.L.ht_fused_ints(self.h, k.encode(), nc, a.ctypes.data_as(C.POINTER(C.c_int)))
            out.append(a.T.copy())
        return out

    def state(self):
        return self.gpos.copy(), self.gvel.copy(), self.cforce.copy()


NW = 6


def _vs_oracle(model, st, cons, mu, full, path, W, nsteps=cf.NSTEPS):
    """teacher-forced from the oracle's states: worst relative errors and active-set / branch flips"""
    hb = FrictionHostBatch(model, W)
    hb.bind_friction(cons, mu)
    oracles = [cf.oracle(model, full[:, w], [a[:, w] for a in st]) for w in range(W)]
    nr = model.nrows
    worst, flips, slid = {}, 0, 0
    for s in range(nsteps):
        hb.gpos[:] = np.stack([o.gpos for o in oracles], 1)
        hb.gvel[:] = np.stack([o.gvel for o in oracles], 1)
        hb.cforce[:nr] = np.stack([o.cforce for o in oracles], 1).reshape(nr, W)
        hb.step(path)
        act, br = hb.flags(path)
        for w, o in enumerate(oracles):
            o.step(cf.DT)
            a = np.array(o.active, dtype=int)
            flips += int((act[w] != a).sum()) + int((br[w]*act[w] != np.array(o.branch)*a).sum())
            slid += int((np.array(o.branch)*a == 3).sum())
            worst["gvel"] = max(worst.get("gvel", 0.), cf.rel(hb.gvel[:, w], o.gvel))
            worst["gpos"] = max(worst.get("gpos", 0.), cf.rel(hb.gpos[:, w], o.gpos))
            worst["cforce"] = max(worst.get("cforce", 0.), cf.rel(hb.cforce[:nr, w], o.cforce))
    assert not (hb.iarr("status") & 3).any()
    return worst, flips, slid


@pytest.mark.parametrize("path", PATHS + ["group"])
@pytest.mark.parametrize("name", FIXTURES)
def test_friction_vs_oracle(name, path):
    """mu in [0.2, 1.5] on a random half of the contacts of every world: within 1e-10 relative of the
    oracle on each world's own model, no active-set or branch flip"""
    model, st = cf.load(name, NW)
    cons, mu, full = cf.perturbed(model, NW, seed=1)
    worst, flips, slid = _vs_oracle(model, st, cons, mu, full, path, NW)
    assert flips == 0
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


def _free_run(model, st, path, W, nsteps, bind=None):
    hb = FrictionHostBatch(model, W)
    if bind is not None:
        hb.bind_friction(*bind)
    hb.set_state(st)
    for _ in range(nsteps):
        hb.step(path)
    return hb.state(), hb.iarr("status").copy(), hb.flags(path)


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", FIXTURES)
def test_bound_friction_equals_own_model(name, path):
    """world w of a bound batch is bit for bit a batch built from world w's own model (_mu edited)"""
    W = 4
    model, st = cf.load(name, W)
    cons, mu, full = cf.perturbed(model, W, seed=2)
    got, _, _ = _free_run(model, st, path, W, cf.NSTEPS, (cons, mu))
    for w in range(W):
        ref, _, _ = _free_run(cf.world_model(model, full[:, w]), [a[:, w:w + 1] for a in st], path, 1, cf.NSTEPS)
        for a, b in zip(got, ref):
            assert a[:, w].tobytes() == b[:, 0].tobytes()


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("name", FIXTURES)
def test_model_mu_bound_equals_unbound(name, path):
    """every contact bound to the model's own mu: the unbound step's bits"""
    W = 4
    model, st = cf.load(name, W)
    cs = cf.contacts(model)
    ref, _, _ = _free_run(model, st, path, W, cf.NSTEPS)
    got, _, _ = _free_run(model, st, path, W, cf.NSTEPS, (cs, np.repeat(cf.model_mu(model)[:, None], W, 1)))
    for a, b in zip(got, ref):
        assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("path", PATHS)
def test_binding_is_read(path):
    """Step 40 of traj_human36_contact64: 13 of the 64 worlds have a sliding contact at mu = 0.6.  With
    mu = 5 in those worlds some of those contacts stick, their states change, and the other worlds'
    bits do not."""
    W = 64
    model, st = cf.load("human36_contact", W)
    cs = cf.contacts(model)
    with np.load(os.path.join(cf.GOLDEN, "traj_human36_contact64.npz")) as z:
        hot = np.nonzero(((z["branch"][:, 40, cs] == 3) & (z["active"][:, 40, cs] == 1)).any(1))[0]
    assert len(hot) == 13
    (g0, v0, f0), _, (act0, br0) = _free_run(model, st, path, W, 1)
    sl = (br0[:, cs] == 3) & (act0[:, cs] == 1)
    sl[np.setdiff1d(np.arange(W), hot)] = False
    assert sl.any()
    mu = np.full((len(cs), W), 0.6)
    mu[:, hot] = 5.
    (g1, v1, f1), status, (act1, br1) = _free_run(model, st, path, W, 1, (cs, mu))
    assert not (status & 3).any()
    assert (br1[:, cs][sl] == 2).any()
    cold = np.setdiff1d(np.arange(W), hot)
    for a, b in ((g0, g1), (v0, v1), (f0, f1)):
        assert a[:, cold].tobytes() == b[:, cold].tobytes()
    for w in hot:
        assert v0[:, w].tobytes() != v1[:, w].tobytes()


@pytest.mark.parametrize("path", PATHS)
def test_unbinding_restores_the_model(path):
    """bound, then unbound: the results of a batch that never bound anything, bit for bit"""
    model, st = cf.load("human36_contact", 4)
    cons, mu, _ = cf.perturbed(model, 4)
    ref, _, _ = _free_run(model, st, path, 4, 3)
    hb = FrictionHostBatch(model, 4)
    hb.bind_friction(cons, mu)
    hb.bind_friction((), None)
    hb.set_state(st)
    for _ in range(3):
        hb.step(path)
    for a, b in zip(hb.state(), ref):
        assert a.tobytes() == b.tobytes()


def test_bad_constraints_are_refused_and_the_binding_kept():
    """out of range, not a contact, a duplicate, mu without constraints: -1 naming mu, and the steps
    after a refusal still read the previous binding"""
    W = 4
    model, st = cf.load("human36_contact", W)
    cons, mu, _ = cf.perturbed(model, W, seed=3)
    ref, _, _ = _free_run(model, st, "lane", W, 2, (cons, mu))
    hb = FrictionHostBatch(model, W)
    hb.bind_friction(cons, mu)
    m1 = np.ones((1, W))
    nc = len(model.cons_type)
    limit = [c for c, t in enumerate(model.cons_type) if int(t) == 0][0]
    for ids, m, msg in (((nc,), m1, "mu constraint %d out of range" % nc), ((-1,), m1, "out of range"),
                        ((limit,), m1, "mu constraint %d is not a contact" % limit),
                        ((3, 3), np.ones((2, W)), "mu constraint 3 listed twice"),
                        ((), m1, "a mu array needs its constraints")):
        with pytest.raises(ValueError, match=msg):
            hb.bind_friction(ids, m)
    hb.set_state(st)
    for _ in range(2):
        hb.step("lane")
    for a, b in zip(hb.state(), ref):
        assert a.tobytes() == b.tobytes()


@pytest.mark.parametrize("path", PATHS)
def test_nan_mu_stays_in_its_world(path):
    """a NaN mu in world 3 (sliding contacts): that world's status bits are set, its neighbours' status
    stays clear and their bits unchanged"""
    W = 4
    model, st = cf.load("human36_contact", W)
    cs = cf.contacts(model)
    mu = np.full((len(cs), W), 0.6)
    ref, _, _ = _free_run(model, st, path, W, 2, (cs, mu))
    mu[:, 3] = np.nan
    got, status, _ = _free_run(model, st, path, W, 2, (cs, mu))
    assert status[3] != 0 and not status[:3].any()
    for a, b in zip(got, ref):
        assert a[:, :3].tobytes() == b[:, :3].tobytes()
