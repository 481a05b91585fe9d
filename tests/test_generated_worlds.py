"""The CPU build of the device routines on generated worlds (tests/genworlds.py): model shapes the eight
fixed fixtures never have -- more than 32 constraints, general Gauss-Seidel visits, contact-aligned
runs broken by limits and a second plane, wide trees with many generator bodies -- taught by the
oracle step by step, with the tolerances of test_hostmath.py."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "hosttest"))
sys.path.insert(0, os.path.dirname(__file__))
import genworlds as G  # noqa: E402
import harness  # noqa: E402

NSTEPS = 6
W = 2


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max()/max(np.abs(b).max(), 1e-300)


WORLDS = sorted(G.CATALOGUE) + ["free%d" % s for s in G.FREE_SEEDS]


def spec_of(name):
    return G.free_spec(int(name[4:])) if name.startswith("free") else G.CATALOGUE[name]


@pytest.fixture(scope="module", params=WORLDS)
def world(request):
    name = request.param
    spec = spec_of(name)
    model = G.build(spec, 0)
    gp, gv, _ = G.states(model, spec, 0, W, steps=NSTEPS)
    return name, model, gp, gv


def test_catalogue_reaches_its_branch(world):
    name, model, _, _ = world
    if name.startswith("free"):
        return
    G.expect(name, model)
    g, c = harness.HostBatch(model, 1).aligned()
    if name == "nc_over_32":
        assert g.all() and c.all()
    elif name == "general_visits":
        # every constraint except the root's plane contacts takes a general visit
        ci = np.asarray(model.cons_int)
        ground_plane = (np.asarray(model.cons_type) == G.CONS_CONTACT) & (ci[:, 0] == 0) & (ci[:, 2] == 0)
        assert not g[1:].any() and not c[~ground_plane].any()
    elif name == "aligned_mixed":
        # only the root (plane contacts of one normal) is aligned; the body on two planes and the body
        # with a ball-and-socket are not, and the limits inside its runs are not contacts
        assert g.tolist() == [1] + [0]*(len(g) - 1)
        ci = np.asarray(model.cons_int)
        on_root = (np.asarray(model.cons_type) == G.CONS_CONTACT) & (ci[:, 1] == 1) & (ci[:, 0] == 0)
        assert (c.astype(bool) == on_root).all()
    elif name == "wide_tree":
        assert len(g) >= 6 and g.all()


def test_expect_refuses_an_entry_without_assertion():
    with pytest.raises(KeyError):
        G.expect("no_such_entry", G.build(G.CATALOGUE["aligned_mixed"], 0))


def _cut(model, keep, body_from=None, body=None):
    """the model with its first `keep` constraints; constraints from index `body_from` on moved to `body`"""
    from arboris_b200.flatten import FlatModel
    d = model.to_dict()
    for k in ("cons_type", "cons_int", "cons_dbl", "cons_row"):
        d[k] = np.array(d[k])[:keep]
    if body_from is not None:
        d["cons_int"][body_from:, 1] = body
    d["nrows"] = int(d["cons_row"][-1]) + (1, 3, 4)[int(d["cons_type"][-1])]
    d["cforce0"] = np.asarray(d["cforce0"])[:d["nrows"]]
    return FlatModel.from_dict(d)


def test_catalogue_trigger_removed_fails():
    """the branch assertions are live: nc_over_32 cut to 32 constraints fails them, and so does the model
    cut to 33 constraints whose run of one body ends at index 31 (constraint 32 on another body)"""
    model = G.build(G.CATALOGUE["nc_over_32"], 0)
    G.expect("nc_over_32", _cut(model, 33))
    with pytest.raises(AssertionError):
        G.expect("nc_over_32", _cut(model, 32))
    other = 1 + int(np.asarray(model.cons_int)[31, 1]) % len(model.joint_type)
    with pytest.raises(AssertionError, match="crosses index 32"):
        G.expect("nc_over_32", _cut(model, 33, 32, other))
    with pytest.raises(AssertionError):
        G.expect("group_fallback", G.build(G.CATALOGUE["wide_tree"], 0))


def _teach(model, gp, gv, run):
    """run(hb) from each oracle state for NSTEPS steps; returns (worst, flips, nact, nslide)"""
    from oracle.arboris_oracle import OracleWorld
    hb = harness.HostBatch(model, W)
    oracles = []
    for w in range(W):
        o = OracleWorld(model.to_dict())
        o.gpos[:], o.gvel[:] = gp[:, w], gv[:, w]
        oracles.append(o)
    worst, flips, nact, nslide = {}, 0, 0, 0
    for s in range(NSTEPS):
        hb.gpos[:] = np.stack([o.gpos for o in oracles], 1)
        hb.gvel[:] = np.stack([o.gvel for o in oracles], 1)
        hb.cforce[:model.nrows] = np.stack([o.cforce for o in oracles], 1)
        got = run(hb)
        act, br = got["active"], got["branch"]
        for w, o in enumerate(oracles):
            o.update_dynamic()
            o.update_controllers(G.DT)
            for k, ref in (("M", o.mass), ("N", o.nleffects), ("Z", o.impedance), ("Y", o.admittance)):
                if k in got:
                    worst[k] = max(worst.get(k, 0.), rel(got[k][..., w], ref))
            o.update_constraints(G.DT)
            o.integrate(G.DT)
            a = np.array(o.active, dtype=int)
            flips += int((act[w] != a).sum()) + int((br[w]*act[w] != np.array(o.branch)*a).sum())
            nact += int(a.sum())
            nslide += int(((np.array(o.branch) == 3) & (a == 1)).sum())
            worst["gvel"] = max(worst.get("gvel", 0.), rel(hb.gvel[:, w], o.gvel))
            worst["gpos"] = max(worst.get("gpos", 0.), rel(hb.gpos[:, w], o.gpos))
            if model.nrows:
                worst["cforce"] = max(worst.get("cforce", 0.), rel(hb.cforce[:model.nrows, w], o.cforce))
    assert not (hb.iarr("status") & 3).any()     # (NONFINITE, SINGULAR; EIG_NOROOT is the reference's clamp)
    return worst, flips, nact, nslide


def _check(worst, flips, nact):
    assert nact > 0
    assert flips == 0, flips
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


def test_phase_routines_vs_oracle(world):
    name, model, gp, gv = world
    n, nc = model.ndof, len(model.cons_type)

    def run(hb):
        hb.update_dynamic()
        hb.update_controllers(G.DT)
        got = {k: hb.arr(k, n, n).copy() for k in ("M", "N", "Z", "Y")}
        hb.update_constraints(G.DT)
        hb.integrate(G.DT)
        got["active"], got["branch"] = hb.iarr("cactive", nc).T.copy(), hb.iarr("cbranch", nc).T.copy()
        return got
    _check(*_teach(model, gp, gv, run)[:3])


@pytest.mark.parametrize("coop", [0, 1])
def test_fused_step_vs_oracle(world, coop):
    name, model, gp, gv = world
    nc = len(model.cons_type)

    def run(hb):
        hb.set_coop(coop)
        hb.fused_step(G.DT)
        return {"active": hb.iarr("factive", nc).T.copy(), "branch": hb.iarr("fbranch", nc).T.copy()}
    worst, flips, nact, nslide = _teach(model, gp, gv, run)
    _check(worst, flips, nact)
    print(name, "coop", coop, {k: "%.1e" % v for k, v in worst.items()}, "active", nact, "sliding", nslide)


def test_fused_step_group_vs_oracle(world):
    name, model, gp, gv = world
    nc = len(model.cons_type)

    def run(hb):
        hb.fused_step_group(G.DT)
        return {"active": hb.iarr("factive", nc).T.copy(), "branch": hb.iarr("fbranch", nc).T.copy()}
    _check(*_teach(model, gp, gv, run)[:3])


def _massless_contact_world():
    """11 bodies, the first child (b0) massless and carrying contact spheres, a ball-and-socket between
    b0 and its child b1, 3 hinge limits: the world whose step 3 (from random velocities, seed 0) made
    the host build and the oracle differ by 1e13 relative"""
    from arboris_b200 import constraints as Cn, controllers as Ct, core, homogeneousmatrix as Hg
    from arboris_b200 import joints as J, massmatrix as mm, shapes
    from arboris_b200.flatten import flatten
    from arboris_b200.robots import simpleshapes
    rng = np.random.default_rng(1)
    w = core.World()
    simpleshapes.add_groundplane(w)
    plane = list(w.itershapes())[0]
    root = core.Body(name="root", mass=mm.box((.3, .2, .4), 5.))
    fj = J.FreeJoint(name="rootj")
    w.add_link(w.ground, fj, root)
    fj.gpos[:] = Hg.transl(0, .08, 0)
    bodies, hinges = [root], []
    kinds = [J.RzJoint, J.RxJoint, J.RyJoint, J.RzRyRxJoint, J.RzRxJoint, J.TxTyTzJoint]
    for i in range(10):
        par = bodies[1] if i == 1 else bodies[rng.integers(len(bodies))]
        cls = kinds[rng.integers(len(kinds))]
        m = mm.box((.05, .1, .05), .3 + rng.random()) if i != 0 else None
        b = core.Body(name="b%d" % i, mass=m)
        f0 = core.SubFrame(par, np.dot(Hg.transl(*rng.uniform(-.1, .1, 3)), Hg.rotzyx(*rng.uniform(-.3, .3, 3))), "f%d" % i)
        j = cls(name="j%d" % i)
        w.add_link(f0, j, b)
        bodies.append(b)
        if cls in (J.RzJoint, J.RxJoint, J.RyJoint):
            hinges.append(j)
    sph = []
    for i, b in enumerate(bodies[:7]):
        for k in range(rng.integers(3, 9)):
            s = shapes.Sphere(core.SubFrame(b, Hg.transl(*rng.uniform(-.1, .1, 3)), "s%d_%d" % (i, k)),
                              .03 + .02*rng.random(), "sh%d_%d" % (i, k))
            w.register(s)
            sph.append(s)
    w.register(Ct.WeightController())
    for s in sph:
        w.register(Cn.SoftFingerContact((plane, s), .6))
    w.register(Cn.BallAndSocketConstraint((core.SubFrame(bodies[1], Hg.transl(0, .05, 0), "bsA"),
                                           core.SubFrame(bodies[2], Hg.transl(0, -.05, 0), "bsB"))))
    for j in hinges[:3]:
        w.register(Cn.JointLimits(j, -.2, .2))
    w.init()
    return flatten(w)


def test_massless_contact_body_is_rejected_and_sliding_roots_agree():
    """Regression case of the generator's rules.  Contacts on a massless body: at step 3 the contact
    blocks have condition numbers of 1e24 and more and the reference's own Gauss-Seidel diverges, so
    COND_MAX rejects the state; the structured sliding root still matches numpy's eigvals on every
    sliding solve of that step (no routine of the host build is at fault)."""
    import ctypes as C
    from oracle.arboris_oracle import OracleWorld
    from test_hostmath import _sliding_matrix
    model = _massless_contact_world()
    o = OracleWorld(model.to_dict())
    o.gvel[:] = np.random.default_rng(0).normal(scale=.3, size=(model.ndof, 2))[:, 0]
    for _ in range(3):
        o.step(G.DT)
    spec = G.Spec(min_active=0, sliding=False)
    assert not G.accept(model, spec, o.gpos.copy(), o.gvel.copy(), 1)
    L = harness.lib()
    dp = C.POINTER(C.c_double)
    L.ht_sliding_root.argtypes = [dp, dp, C.c_double, dp, C.POINTER(C.c_int)]
    calls = []
    orig = OracleWorld._solve_softfinger

    def record(self, c, vel, adm, dt, rows):
        f0 = self.cforce[rows].copy()
        df = orig(self, c, vel, adm, dt, rows)
        if self.branch[c] == 3:
            alpha = vel - adm.dot(f0)
            alpha[3] += self.sdist[c]/dt
            calls.append((adm.copy(), alpha, self.cd[c][36]))
        return df
    o._solve_softfinger = record.__get__(o)
    o.step(G.DT)
    assert len(calls) >= 5
    for A, alpha, mu in calls:
        S = np.linalg.eigvals(_sliding_matrix(A, alpha, mu))
        S = S[np.logical_and(S.imag == 0, S.real <= 0)]
        s, found = C.c_double(0.), C.c_int(0)
        assert L.ht_sliding_root(np.ascontiguousarray(A).ctypes.data_as(dp), alpha.ctypes.data_as(dp), mu,
                                 C.byref(s), C.byref(found))
        assert bool(found.value) == (len(S) > 0)
        if len(S):
            ref = float(min(S).real)
            assert abs(s.value - ref) <= 1e-9*abs(ref), (s.value, ref)
