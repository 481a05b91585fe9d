"""Seeded families of worlds for the checks of the fused prepare and finish stages against the
50-digit reference (artref.py): tests/test_prepare_reference.py (host build of the device routines)
and tests/test_gpu_prepare_reference.py (the device, through arb_get_fused).

A family is a list of worlds; a world is a dict: model (FlatModel, with this world's body inertia,
gravity and PD gains baked in -- what the reference reads), gpos, gvel, cforce, dt, and a tag.
expect() checks what a family claims about itself on the reference's own numbers; an unknown family
raises."""
import os

import numpy as np

from conftest import GOLDEN, load_golden

FAMILIES = ("fixtures", "mass_ratio", "instantiations")


def _load(model_name, traj_name):
    from arboris_b200.flatten import FlatModel
    model = FlatModel.load(os.path.join(GOLDEN, "model_%s.npz" % model_name))
    with np.load(os.path.join(GOLDEN, "traj_%s.npz" % traj_name)) as z:
        return model, {k: z[k] for k in z.files}


def _state(tr, w, s):
    if s == 0:
        return tr["gpos_in"][w].copy(), tr["gvel_in"][w].copy()
    return tr["gpos"][w, s - 1].copy(), tr["gvel"][w, s - 1].copy()


def _world(model, gpos, gvel, dt, cforce=None, **kw):
    d = dict(model=model, gpos=np.asarray(gpos, float), gvel=np.asarray(gvel, float), dt=float(dt),
             cforce=np.zeros(max(int(model.nrows), 1)) if cforce is None else np.asarray(cforce, float))
    d.update(kw)
    return d


def fixtures(n=16):
    """teacher-forced states of the reference's trajectories"""
    out = []
    model, tr = _load("human36_contact", "human36_contact64")
    rng = np.random.default_rng(1)
    for k in range(n//2):
        w, s = int(rng.integers(64)), int(rng.integers(20, 120))
        g, v = _state(tr, w, s)
        out.append(_world(model, g, v, tr["dt"], tag="human36_contact64"))
    for name, (w, s) in (("zoo", (0, 100)), ("zoo", (2, 150)), ("snake_loop", (0, 100)), ("snake_loop", (1, 20)),
                         ("balls", (0, 200)), ("simplearm_limits", (0, 150)), ("simplearm_limits", (1, 0)),
                         ("ball_socket", (0, 10))):
        model, tr = load_golden(name)
        act = tr["active"][w].any(axis=1)
        s = s + int(np.argmax(np.roll(act, -s)))         # the first step from s on with an active constraint
        g, v = _state(tr, w, s)
        cf = tr["cforce"][w, s - 1] if "cforce" in tr and s > 0 else None
        out.append(_world(model, g, v, tr["dt"], cforce=cf, tag=name))
    return out


def _human36_in_contact(n, seed):
    model, tr = _load("human36_contact", "human36_contact64")
    rng = np.random.default_rng(seed)
    sel = []
    while len(sel) < n:
        w, s = int(rng.integers(64)), int(rng.integers(40, 120))
        if tr["active"][w, s].any():
            sel.append((w, s))
    return model, tr, sel


def mass_ratio(n=8):
    """human36_contact with the leaf bodies lightened by 1e-3 ... 1e-9 and the pelvis made 1e3 heavier"""
    from arboris_b200 import massmatrix
    import bodyparams
    model, tr, sel = _human36_in_contact(n, 2)
    p0 = massmatrix.to_params(bodyparams.body_masses(model))
    nj = p0.shape[0]
    parents = set(np.asarray(model.joint_parent).tolist())
    leaves = [j + 1 for j in range(nj) if (j + 1) not in parents]
    bodies = tuple(range(1, nj + 1))
    out = []
    for k, (w, s) in enumerate(sel):
        f = 10.0**-(3 + 6*k/max(n - 1, 1))
        p = p0.copy()
        for b in leaves:
            p[b - 1] *= f
        p[0] *= 1e3
        g, v = _state(tr, w, s)
        out.append(_world(bodyparams.world_model(model, bodies, p), g, v, tr["dt"], inertia=(bodies, p),
                          tag="mass x%.0e" % f))
    return out


def instantiations(n=6):
    """human36 states with nothing bound, with applied forces bound, with inertia and gravity bound: the
    prepare stage's instantiations artic_factor<false,false>, <true,false> and <true,true>"""
    from arboris_b200 import massmatrix
    import bodyparams
    model, tr, sel = _human36_in_contact(n, 4)
    rng = np.random.default_rng(5)
    nj = len(model.joint_type)
    p0 = massmatrix.to_params(bodyparams.body_masses(model))
    bodies = tuple(range(1, nj + 1))
    out = []
    for k, (w, s) in enumerate(sel):
        g, v = _state(tr, w, s)
        kind = ("plain", "applied", "params")[k % 3]
        if kind == "plain":
            out.append(_world(model, g, v, tr["dt"], tag=kind))
        elif kind == "applied":
            tau = rng.normal(scale=5., size=int(model.ndof))
            wr = {b: rng.normal(scale=20., size=6) for b in (3, 9, 15)}
            out.append(_world(model, g, v, tr["dt"], tau=tau, wrench=wr, tag=kind))
        else:
            p = p0*rng.uniform(0.7, 1.4, size=(nj, 1))
            grav = np.array([0., 0., -9.81]) + rng.normal(scale=2., size=3)
            out.append(_world(bodyparams.world_model(model, bodies, p, grav), g, v, tr["dt"],
                              inertia=(bodies, p), gravity=grav, tag=kind))
    return out


def family(name):
    if name not in FAMILIES:
        raise KeyError("unknown family %r" % name)
    return globals()[name]()


def job(world, gens, active=(), y=None, mutate=()):
    """the artref.summary() job of one world"""
    d = world["model"].to_dict()
    return dict(model=d, gpos=world["gpos"], gvel=world["gvel"], dt=world["dt"], gens=gens,
                cforce=world["cforce"], tau=world.get("tau"), wrench=world.get("wrench"),
                active=tuple(int(c) for c in active), y=None if y is None else np.asarray(y, float),
                mutate=tuple(mutate))


def _active_generators(world, gens, active):
    """generator rows (first row of each block) that an active constraint of the world reaches"""
    m = world["model"]
    types = np.asarray(m.cons_type).reshape(-1)
    ci = np.asarray(m.cons_int).reshape(-1, 4)
    out = set()
    for c in np.flatnonzero(active):
        if types[c] == 0:
            out.add(6*len(gens["body"]) + int((types[:c] == 0).sum()))
        else:
            out |= {6*gens["body"].index(int(b)) for b in ci[c][:2] if int(b) in gens["body"]}
    return out


def expect(name, worlds, refs, active, gens):
    """the family's claim about itself, on the reference's numbers; active: (W, nc) flags, gens: the
    generator layout of each world.  Returns cond(Z) of every world."""
    assert len(worlds) == len(refs) == len(active) == len(gens)
    if name not in FAMILIES:
        raise KeyError("unknown family %r" % name)
    for a, w in zip(active, worlds):
        assert np.asarray(a).any(), "a world of %s has no active constraint (%s)" % (name, w.get("tag"))
    kz = [r["cond_Z"] for r in refs]
    assert all(np.isfinite(kz))
    if name == "fixtures":
        # every model of the fixtures, and every generator block of each active somewhere in the family
        tags = set(w["tag"] for w in worlds)
        assert {"human36_contact64", "zoo", "snake_loop", "balls", "simplearm_limits", "ball_socket"} <= tags
        for tag in tags:
            ix = [i for i, w in enumerate(worlds) if w["tag"] == tag]
            g = gens[ix[0]]
            every = {6*i for i in range(len(g["body"]))} | set(range(6*len(g["body"]), g["ng"]))
            seen = set().union(*[_active_generators(worlds[i], gens[i], active[i]) for i in ix])
            assert every <= seen, (tag, sorted(every - seen))
    elif name == "mass_ratio":
        # six decades of cond(Z), up to 1e12 and beyond
        assert max(kz) >= 1e6*min(kz) and max(kz) >= 1e12, "cond(Z) %.1e .. %.1e" % (min(kz), max(kz))
    elif name == "instantiations":
        assert {"plain", "applied", "params"} <= set(w["tag"] for w in worlds)
    return kz
