"""Per-world body inertia and gravity (arb_batch_bind_body_inertia, arb_batch_bind_gravity) in the CPU
build of the device routines: the phase routines and the fused step against the oracle on each world's
own model, bit-identity with a batch built from that model, mass-scaling invariance, bodies that gain
or lose their mass in one world, and the refusals."""
import os
import sys

import numpy as np
import pytest

HOSTTEST = os.path.join(os.path.dirname(__file__), "hosttest")
sys.path.insert(0, HOSTTEST)
import harness  # noqa: E402

import bodyparams as bp  # noqa: E402

SRC = os.path.join(HOSTTEST, "arb_hosttest_body_params.cpp")
OUT = os.path.join(HOSTTEST, "_build", "libarb_hosttest_body_params.so")
_lib = None


def bp_lib():
    """the host build with the body-parameter exports (arb_hosttest_body_params.cpp), built as
    harness.build() builds arb_hosttest.cpp"""
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
                 "ht_update_constraints", "ht_integrate", "ht_fused_step", "ht_array", "ht_iarray"):
        getattr(L, name).restype = getattr(base, name).restype
        getattr(L, name).argtypes = getattr(base, name).argtypes
    L.ht_bind_body_params.restype = C.c_int
    L.ht_bind_body_params.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_char_p, C.c_int]
    L.ht_release_body_params.argtypes = [C.c_void_p]
    L.ht_bp_update_dynamic.argtypes = [C.c_void_p]
    L.ht_bp_update_controllers.argtypes = [C.c_void_p, C.c_double]
    L.ht_bp_fused_step.argtypes = [C.c_void_p, C.c_double]
    _lib = L
    return L


class ParamsHostBatch(harness.HostBatch):
    """harness.HostBatch on the library with the body parameters: update_dynamic, update_controllers
    and fused_step read what bind_params bound (nothing until then)."""

    def __init__(self, model, W):
        import ctypes as C
        self.L = bp_lib()
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
            self.L.ht_release_body_params(self.h)
        harness.HostBatch.__del__(self)

    def bind_body_params(self, bodies=(), inertia=None, gravity=None):
        """inertia (len(bodies), 10, W), gravity (3, W), ``None`` for none (kept alive here); raises
        ValueError with the library's message"""
        import ctypes as C
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float64) for a in (inertia, gravity)]
        ids = np.ascontiguousarray(bodies, dtype=np.int32).reshape(-1)
        err = C.create_string_buffer(256)
        rc = self.L.ht_bind_body_params(self.h, len(ids), ids.ctypes.data if len(ids) else None,
                                        None if arrs[0] is None else arrs[0].ctypes.data,
                                        None if arrs[1] is None else arrs[1].ctypes.data, err, 256)
        if rc:
            raise ValueError(err.value.decode())
        self._bp = (arrs, ids)

    def set_state(self, st):
        self.gpos[:], self.gvel[:] = st[0], st[1]
        self.cforce[:st[2].shape[0]] = st[2]

    def update_dynamic(self):
        self.L.ht_bp_update_dynamic(self.h)

    def update_controllers(self, dt):
        self.L.ht_bp_update_controllers(self.h, dt)

    def fused_step(self, dt):
        self.L.ht_bp_fused_step(self.h, dt)

    def step(self, path, dt=bp.DT):
        if path == "phases":
            self.update_dynamic()
            self.update_controllers(dt)
            self.update_constraints(dt)
            self.integrate(dt)
        else:
            self.fused_step(dt)

    def state(self):
        return self.gpos.copy(), self.gvel.copy(), self.cforce.copy()


NW = 8


def _vs_oracle(model, st, bodies, P, G, path, W, nsteps=bp.NSTEPS):
    """teacher-forced from the oracle's states: worst relative errors and active-set / branch flips"""
    hb = ParamsHostBatch(model, W)
    hb.set_coop(0)
    hb.bind_body_params(bodies, P, G)
    oracles = [bp.oracle(model, bodies, P[:, :, w], None if G is None else G[:, w], [a[:, w] for a in st])
               for w in range(W)]
    n, nc, nr = model.ndof, len(model.cons_type), model.nrows
    worst, flips = {}, 0
    for s in range(nsteps):
        hb.gpos[:] = np.stack([o.gpos for o in oracles], 1)
        hb.gvel[:] = np.stack([o.gvel for o in oracles], 1)
        hb.cforce[:nr] = np.stack([o.cforce for o in oracles], 1).reshape(nr, W)
        if path == "phases":
            hb.update_dynamic()
            hb.update_controllers(bp.DT)
            M, N = hb.arr("M", n, n).copy(), hb.arr("N", n, n).copy()
            gf = hb.arr("gforce", n).copy()
            hb.update_constraints(bp.DT)
            hb.integrate(bp.DT)
            act, br = hb.iarr("cactive", nc).T, hb.iarr("cbranch", nc).T
        else:
            hb.fused_step(bp.DT)
            act, br = hb.iarr("factive", nc).T, hb.iarr("fbranch", nc).T
        for w, o in enumerate(oracles):
            Mo, No, gfo = bp.oracle_step(o)
            if path == "phases":
                for k, a, b in (("M", M[..., w], Mo), ("N", N[..., w], No), ("gforce", gf[:, w], gfo)):
                    worst[k] = max(worst.get(k, 0.), bp.rel(a, b))
            if nc:
                a = np.array(o.active, dtype=int)
                flips += int((act[w] != a).sum()) + int((br[w]*act[w] != np.array(o.branch)*a).sum())
            worst["gvel"] = max(worst.get("gvel", 0.), bp.rel(hb.gvel[:, w], o.gvel))
            worst["gpos"] = max(worst.get("gpos", 0.), bp.rel(hb.gpos[:, w], o.gpos))
            if nr:
                worst["cforce"] = max(worst.get("cforce", 0.), bp.rel(hb.cforce[:nr, w], o.cforce))
    assert not (hb.iarr("status") & 3).any()
    return worst, flips


@pytest.mark.parametrize("path", ["phases", "fused"])
@pytest.mark.parametrize("name", ["human36_contact", "zoo", "snake_loop"])
def test_body_params_vs_oracle(name, path):
    """perturbed inertia on a different half of the bodies in every world and a per-world gravity:
    within 1e-10 relative of the oracle on each world's own model, no active-set or branch flip"""
    model, st = bp.load(name, NW)
    bodies, P, G = bp.perturbed(model, NW, seed=1)
    worst, flips = _vs_oracle(model, st, bodies, P, G, path, NW)
    assert flips == 0
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


def _free_run(model, st, path, W, nsteps, bind=None):
    hb = ParamsHostBatch(model, W)
    hb.set_coop(0)
    if bind is not None:
        hb.bind_body_params(*bind)
    hb.set_state(st)
    for _ in range(nsteps):
        hb.step(path)
    return hb.state(), hb.iarr("status").copy()


@pytest.mark.parametrize("path", ["phases", "fused"])
@pytest.mark.parametrize("name", ["human36_contact", "zoo", "snake_loop"])
def test_bound_params_equal_own_model(name, path):
    """world w of a bound batch is bit for bit a batch built from world w's own model (body_mass =
    from_params(p_w), up = g_w with gravity 1)"""
    W = 4
    model, st = bp.load(name, W)
    bodies, P, G = bp.perturbed(model, W, seed=2)
    got, _ = _free_run(model, st, path, W, bp.NSTEPS, (bodies, P, G))
    for w in range(W):
        ref, _ = _free_run(bp.world_model(model, bodies, P[:, :, w], G[:, w]), [a[:, w:w + 1] for a in st],
                           path, 1, bp.NSTEPS)
        for a, b in zip(got, ref):
            assert a[:, w].tobytes() == b[:, 0].tobytes()


@pytest.mark.parametrize("path", ["phases", "fused"])
def test_mass_scaling_invariance(path):
    """human36_free (gravity only): every body's 10 numbers scaled by k = 0.5, 2, 4 in worlds 0, 2, 3
    give world 1's (k = 1) trajectory bit for bit after 20 steps; a term still reading the model's
    mass breaks this at the first step"""
    from arboris_b200 import massmatrix
    model, st = bp.load("human36_free", 4)
    st = [np.repeat(a[:, :1], 4, 1) for a in st]
    p0 = massmatrix.to_params(bp.body_masses(model))
    P = p0[:, :, None]*np.array([0.5, 1., 2., 4.])
    bodies = tuple(range(1, p0.shape[0] + 1))
    (g, v, _), status = _free_run(model, st, path, 4, 20, (bodies, P, None))
    assert not status.any()
    assert np.abs(v[:, 1]).max() > 0.1
    for w in (0, 2, 3):
        assert g[:, w].tobytes() == g[:, 1].tobytes() and v[:, w].tobytes() == v[:, 1].tobytes()


def _chain_body(model):
    """a massive body without contacts whose child is massive (zeroing it leaves Z regular)"""
    bm = bp.body_masses(model)
    cb = {int(c[0]) for c in model.cons_int} | {int(c[1]) for c in model.cons_int}
    par = [int(p) for p in model.joint_parent]
    for b in range(2, len(par) + 1):
        kids = [j + 1 for j, p in enumerate(par) if p == b]
        if (bm[b - 1] > 0).any() and b not in cb and kids and all((bm[k - 1] > 0).any() for k in kids):
            return b
    raise AssertionError("no such body")


@pytest.mark.parametrize("path", ["phases", "fused"])
def test_mass_gained_and_lost(path):
    """the model's massless scapula bound with a body's inertia becomes massive (gravity acts on it),
    a massive body bound with zeros becomes massless (gravity does not act on it); against the oracle"""
    from arboris_b200 import massmatrix
    model, st = bp.load("human36_contact", NW)
    bm = bp.body_masses(model)
    lost = _chain_body(model)
    gained = 9
    assert not (bm[gained - 1] != 0).any()
    P = np.zeros((2, 10, NW))
    P[0] = (massmatrix.to_params(bm[8 - 1])*0.5)[:, None]
    bodies = (gained, lost)
    o = bp.oracle(model, bodies, P[:, :, 0], None, [a[:, 0] for a in st])
    assert gained in o.massive and lost not in o.massive
    worst, flips = _vs_oracle(model, st, bodies, P, None, path, NW)
    assert flips == 0
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


@pytest.mark.parametrize("path", ["phases", "fused"])
def test_unbinding_restores_the_model(path):
    """bound, then unbound: the results of a batch that never bound anything, bit for bit"""
    model, st = bp.load("human36_contact", 4)
    bodies, P, G = bp.perturbed(model, 4)
    ref, _ = _free_run(model, st, path, 4, 3)
    hb = ParamsHostBatch(model, 4)
    hb.set_coop(0)
    hb.bind_body_params(bodies, P, G)
    hb.bind_body_params((), None, None)
    hb.set_state(st)
    for _ in range(3):
        hb.step(path)
    for a, b in zip(hb.state(), ref):
        assert a.tobytes() == b.tobytes()


def test_bad_bodies_and_gravity_are_refused():
    model, _ = bp.load("human36_contact", 2)
    hb = ParamsHostBatch(model, 2)
    p1 = np.zeros((1, 10, 2))
    for bodies, msg in (((0,), "ground"), ((len(model.joint_type) + 1,), "out of range"), ((-1,), "out of range")):
        with pytest.raises(ValueError, match=msg):
            hb.bind_body_params(bodies, p1)
    with pytest.raises(ValueError, match="twice"):
        hb.bind_body_params((3, 3), np.zeros((2, 10, 2)))
    with pytest.raises(ValueError, match="needs its bodies"):
        hb.bind_body_params((), p1)
    hb.bind_body_params((), None, np.zeros((3, 2)))            # gravity alone
    d = model.to_dict()
    for k in ("ctrl_type", "ctrl_int", "ctrl_dbl"):
        d[k] = d[k][:0]
    from arboris_b200.flatten import FlatModel
    hb2 = ParamsHostBatch(FlatModel.from_dict(d), 2)
    with pytest.raises(ValueError, match="no WeightController"):
        hb2.bind_body_params((), None, np.zeros((3, 2)))
    hb2.bind_body_params((1,), p1)                             # inertia needs no WeightController


def test_params_round_trip():
    """from_params(to_params(M)) == M for rigid-body matrices; human36's own matrices are within 3e-17"""
    from arboris_b200 import massmatrix
    rng = np.random.default_rng(0)
    p = rng.normal(size=(5, 3, 10))
    M = massmatrix.from_params(p)
    assert M.shape == (5, 3, 6, 6)
    assert (massmatrix.to_params(M) == p).all() and (massmatrix.from_params(massmatrix.to_params(M)) == M).all()
    assert (M == np.swapaxes(M, -1, -2)).all()
    assert (M[..., 3:, 3:] == p[..., 0, None, None]*np.eye(3)).all()
    model, _ = bp.load("human36_contact", 1)
    bm = bp.body_masses(model)
    assert np.abs(massmatrix.from_params(massmatrix.to_params(bm)) - bm).max() < 3e-17
