"""Shared by the tests of per-world contact friction (test_contact_friction.py,
test_gpu_contact_friction.py): fixtures, per-world friction and the per-world reference models."""
import os

import numpy as np

from conftest import GOLDEN

DT = 1e-3
NSTEPS = 6
MU_COL = 36         # SoftFingerContact._mu in cons_dbl (flatten.py)
# fixture -> (trajectory, first state).  human36_contact: 8 plane contacts, the plain staged Gauss-Seidel;
# balls: plane/sphere, box/sphere and two-body sphere contacts, the general instantiation and
# gs_visit_two_body (step 200: a two-body contact slides); nc_over_32: a generated world of more than
# 32 constraints, the unstaged kernel
FIXTURES = {"human36_contact": ("human36_contact64", 40), "balls": ("balls", 200), "nc_over_32": None}


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max()/max(np.abs(b).max(), 1e-300)


def contacts(model):
    from arboris_b200.flatten import CONS_SOFT_FINGER
    return [c for c, t in enumerate(np.asarray(model.cons_type).reshape(-1)) if int(t) == CONS_SOFT_FINGER]


def model_mu(model):
    return np.array([float(model.cons_dbl[c][MU_COL]) for c in contacts(model)])


def load(name, W):
    """model and W initial states (gpos, gvel, cforce) of the fixture, the trajectory's worlds in turn
    (nc_over_32: genworlds' accepted states)"""
    from arboris_b200.flatten import FlatModel
    if FIXTURES[name] is None:
        import genworlds as G
        spec = G.CATALOGUE[name]
        model = G.build(spec, 0)
        n = min(W, 4)
        gp, gv, _ = G.states(model, spec, 0, n, steps=NSTEPS)
        ids = np.arange(W) % n
        return model, [gp[:, ids].copy(), gv[:, ids].copy(), np.zeros((max(model.nrows, 1), W))]
    model = FlatModel.load(os.path.join(GOLDEN, "model_%s.npz" % name))
    traj, s0 = FIXTURES[name]
    with np.load(os.path.join(GOLDEN, "traj_%s.npz" % traj)) as z:
        ids = np.arange(W) % z["gpos"].shape[0]
        st = [z[k][ids, s0].T.copy() for k in ("gpos", "gvel", "cforce")]
    return model, st


def perturbed(model, W, seed=0):
    """Every contact but the last bound, in a shuffled order (the last keeps the model's mu through the
    row -1 of the table); in each world a random half of the contacts gets mu in [0.2, 1.5], the
    others the model's.  Returns constraints, (len(constraints), W) and the full (ncontacts, W) mu."""
    rng = np.random.default_rng(seed)
    cs = contacts(model)
    full = np.repeat(model_mu(model)[:, None], W, 1)
    for w in range(W):
        sel = rng.permutation(len(cs) - 1)[:max(1, len(cs)//2)]
        full[sel, w] = rng.uniform(0.2, 1.5, size=len(sel))
    order = rng.permutation(len(cs) - 1)
    return tuple(cs[i] for i in order), full[order].copy(), full


def world_model(model, mu):
    """FlatModel of one world: _mu of contact k (contacts(model)[k]) = mu[k]"""
    from arboris_b200.flatten import FlatModel
    d = model.to_dict()
    cd = np.array(d["cons_dbl"], dtype=float)
    for k, c in enumerate(contacts(model)):
        cd[c][MU_COL] = mu[k]
    d["cons_dbl"] = cd
    return FlatModel.from_dict(d)


def oracle(model, mu, state):
    from oracle.arboris_oracle import OracleWorld
    o = OracleWorld(world_model(model, mu).to_dict())
    o.gpos[:], o.gvel[:], o.cforce[:] = state[0], state[1], state[2][:len(o.cforce)]
    return o
