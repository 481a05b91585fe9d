"""Shared by the tests of per-world body inertia and gravity (test_body_params.py,
test_gpu_body_params.py): fixtures, perturbed parameters and the per-world reference models."""
import os

import numpy as np

from conftest import GOLDEN

DT = 1e-3
NSTEPS = 6
# fixture -> (trajectory, first state); human36_contact: the reference's step 40 of the 64 falling
# humanoids, most of them in contact
FIXTURES = {"human36_contact": ("human36_contact64", 40), "zoo": ("zoo", 100), "snake_loop": ("snake_loop", 100),
            "human36_free": ("human36_free", 50)}


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max()/max(np.abs(b).max(), 1e-300)


def load(name, W):
    """model and W initial states (gpos, gvel, cforce) of the fixture, the trajectory's worlds in turn"""
    from arboris_b200.flatten import FlatModel
    model = FlatModel.load(os.path.join(GOLDEN, "model_%s.npz" % name))
    traj, s0 = FIXTURES[name]
    with np.load(os.path.join(GOLDEN, "traj_%s.npz" % traj)) as z:
        ids = np.arange(W) % z["gpos"].shape[0]
        st = [z[k][ids, s0].T.copy() for k in ("gpos", "gvel", "cforce")]
    return model, st


def body_masses(model):
    return np.asarray(model.body_mass, dtype=float).reshape(-1, 6, 6)


def perturbed(model, W, seed=0):
    """Every body bound; in each world a random half of them gets a perturbed inertia (the mass and
    m c scaled by a, the rotational inertia by b >= a, so that M_b stays positive definite), the others
    the model's own (to_params).  Gravity: the model's scaled and tilted.  Returns bodies, (nb, 10, W),
    (3, W)."""
    from arboris_b200 import massmatrix
    rng = np.random.default_rng(seed)
    p0 = massmatrix.to_params(body_masses(model))                 # (nj, 10)
    nj = p0.shape[0]
    P = np.repeat(p0[:, :, None], W, 2)
    for w in range(W):
        sel = rng.permutation(nj)[:max(1, nj//2)]
        a = rng.uniform(0.7, 1.4, size=len(sel))
        b = a*rng.uniform(1., 1.3, size=len(sel))
        P[sel, 0:4, w] *= a[:, None]
        P[sel, 4:10, w] *= b[:, None]
    g = np.array([0., -9.81, 0.])[:, None]*rng.uniform(0.5, 1.5, size=W) + rng.normal(scale=2., size=(3, W))
    return tuple(range(1, nj + 1)), P, g


def world_model(model, bodies, p, g=None):
    """FlatModel of one world: body_mass of `bodies` = from_params(p[i]) and, with g, up = g and the
    (single) WeightController's gravity 1, so that gravity * up = g exactly"""
    from arboris_b200 import massmatrix
    from arboris_b200.flatten import FlatModel
    d = model.to_dict()
    bm = body_masses(model).copy()
    for i, b in enumerate(bodies):
        bm[b - 1] = massmatrix.from_params(p[i])
    d["body_mass"] = bm.reshape(np.asarray(model.body_mass).shape)
    if g is not None:
        weight = [k for k, t in enumerate(d["ctrl_type"]) if int(t) == 0]
        assert len(weight) == 1
        d["up"] = np.array(g, dtype=float)
        cd = np.array(d["ctrl_dbl"], dtype=float)
        cd[weight[0]][0] = 1.
        d["ctrl_dbl"] = cd
    return FlatModel.from_dict(d)


def oracle(model, bodies, p, g, state):
    from oracle.arboris_oracle import OracleWorld
    o = OracleWorld(world_model(model, bodies, p, g).to_dict())
    o.gpos[:], o.gvel[:], o.cforce[:] = state[0], state[1], state[2][:len(o.cforce)]
    return o


def oracle_step(o, dt=DT):
    o.update_dynamic()
    o.update_controllers(dt)
    gf = o.gforce.copy()
    M, N = o.mass.copy(), o.nleffects.copy()
    o.update_constraints(dt)
    o.integrate(dt)
    return M, N, gf
