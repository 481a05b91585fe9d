"""The 50-digit reference of the impedance solve (artref.py) itself: its M, N, B, Z and controller
forces match the real reference's float64 values (tests/golden/traj_*.npz) to the rounding of forward
products, its admittance to within cond(Z) u, and it is stable in its working precision."""
import numpy as np
import pytest
import mpmath as mp

import artref
from conftest import load_golden


def _rel(a, b):
    return np.abs(np.asarray(a) - b).max()/max(np.abs(b).max(), 1e-300)


@pytest.mark.parametrize("name", ["zoo", "human36_contact", "snake_loop", "balls", "simplearm_limits"])
def test_matrices_match_the_real_reference(name):
    model, tr = load_golden(name)
    gens = {"body": [], "aligned": [], "c0": [], "limdof": []}
    for i, s in enumerate(tr["full_steps"]):
        for w in range(tr["gpos_in"].shape[0]):
            g = tr["gpos_in"][w] if s == 0 else tr["gpos"][w, s - 1]
            v = tr["gvel_in"][w] if s == 0 else tr["gvel"][w, s - 1]
            r = artref.ArtRef(model.to_dict(), g, v, float(tr["dt"]), gens)
            with mp.workdps(artref.DPS):
                for k, ref in (("M", "mass"), ("N", "nleffects"), ("B", "viscosity"), ("Z", "impedance")):
                    assert _rel(artref.tofloat(getattr(r, k)), tr[ref][w, i]) <= 2e-14, (k, s, w)
                assert _rel(artref.tofloat(r.Zinv), tr["admittance"][w, i]) <= 64*artref.U*r.cond_Z()
                if "gforce_ctrl" in tr:
                    assert _rel(artref.tofloat(r.gforce), tr["gforce_ctrl"][w, s]) <= 2e-14


def test_50_digits_agree_with_100():
    model, tr = load_golden("human36_contact")
    gens = {"body": [1], "aligned": [0], "c0": [-1], "limdof": [10]}
    g, v = tr["gpos"][1, 149], tr["gvel"][1, 149]
    r50 = artref.ArtRef(model.to_dict(), g, v, 1e-3, gens)
    old = artref.DPS
    artref.DPS = 100
    try:
        r100 = artref.ArtRef(model.to_dict(), g, v, 1e-3, gens)
    finally:
        artref.DPS = old
    with mp.workdps(110):
        for a, b in ((r50.qfree, r100.qfree), (r50.Lam.reshape(-1), r100.Lam.reshape(-1))):
            scale = max(abs(x) for x in b)
            assert max(abs(x - y) for x, y in zip(a, b)) <= mp.mpf(10)**-40*scale
