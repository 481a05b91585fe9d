"""The fused prepare stage (world_fused_prepare + the Gauss-Seidel prologue) and the finish stage,
CPU build of the device routines (tests/hosttest), against the 50-digit reference of the impedance
solve (artref.py) on the families of artbanks.py: q_free, v0 = G q_free, EVERY entry of
Lambda = G Z^-1 G^T, the diagonal Delassus blocks A_cc of the active constraints (reference: from the
constraint Jacobians directly), and q'+ = q_free + Z^-1 G^T y with the joint integration.  Each within
the componentwise bound C u E(x) fixed in artref.py.  Mutations of the reference (artref.MUTATIONS) must make
the comparison fail."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "hosttest"))

import artbanks  # noqa: E402
import artref  # noqa: E402
import harness  # noqa: E402


def _dbl(hb, name, n):
    out = np.zeros((max(n, 1), 1))
    hb.L.ht_fused_dbl.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_void_p]
    assert hb.L.ht_fused_dbl(hb.h, name.encode(), n, out.ctypes.data) == 0
    return out[:n, 0].copy()


def generators(hb):
    """the generator layout; the counts first, then arrays of those sizes"""
    cnt = np.zeros(2, np.int32)
    hb.L.ht_generators.argtypes = [C.c_void_p] * 6
    hb.L.ht_generators(hb.h, cnt.ctypes.data, None, None, None, None)
    ng, NG = int(cnt[0]), int(cnt[1])
    arr = [np.zeros(max(k, 1), np.int32) for k in (ng, ng, ng, NG - 6*ng)]
    hb.L.ht_generators(hb.h, cnt.ctypes.data, *[a.ctypes.data for a in arr])
    return {"body": arr[0][:ng].tolist(), "aligned": arr[1][:ng].tolist(), "c0": arr[2][:ng].tolist(),
            "limdof": arr[3][:NG - 6*ng].tolist(), "ng": NG}


def host_readback(world, seed=0):
    """the host build's hand-over of one world, and its finish stage for a seeded y"""
    model = world["model"]
    if world.get("tau") is not None:        # artic_factor<true, false>: the applied-force build
        from test_applied_forces import AppliedHostBatch, applied_lib
        hb = AppliedHostBatch(model, 1)
        bodies = tuple(sorted(world["wrench"]))
        hb.bind_applied(world["tau"][:, None], np.array([world["wrench"][b] for b in bodies])[:, :, None], bodies)
        prep = applied_lib().ht_applied_fused_prepare
    else:
        hb = harness.HostBatch(model, 1)
        prep = hb.L.ht_fused_prepare
    prep.argtypes = [C.c_void_p, C.c_double]
    hb.gpos[:, 0], hb.gvel[:, 0] = world["gpos"], world["gvel"]
    hb.cforce[:len(world["cforce"]), 0] = world["cforce"]
    prep(hb.h, world["dt"])
    g = generators(hb)
    NG, n, nc = g["ng"], int(model.ndof), len(model.cons_type)
    rb = {"gens": g, "qfree": _dbl(hb, "fq", n), "v0": _dbl(hb, "fv0", NG),
          "lambda": _dbl(hb, "fLam", NG*NG).reshape(NG, NG), "delassus": _dbl(hb, "fAcc", 4*int(model.nrows)),
          "active": hb.iarr("factive", nc)[:, 0].copy()}
    y = np.random.default_rng(seed).normal(size=NG)*np.abs(rb["lambda"]).max()**-1*1e-2
    yb = y[:, None].copy()
    hb.L.ht_fused_dbl_set.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_void_p]
    hb.L.ht_fused_dbl_set(hb.h, b"fy", NG, yb.ctypes.data)
    hb.L.ht_fused_finish.argtypes = [C.c_void_p, C.c_double]
    hb.L.ht_fused_finish(hb.h, world["dt"])
    rb["y"], rb["gvel"], rb["gpos"] = y, hb.gvel[:, 0].copy(), hb.gpos[:, 0].copy()
    return rb


def ratios(world, rb, ref):
    """worst err / (C u E) of every compared quantity of one world"""
    Cc = ref["C"]
    out = {"qfree": artref.err_ratio(rb["qfree"], ref["qfree"], ref["E_qfree"], Cc),
           "v0": artref.err_ratio(rb["v0"], ref["v0"], ref["E_v0"], Cc),
           "lambda": artref.err_ratio(rb["lambda"], ref["Lam"], ref["E_Lam"], Cc)}
    model = world["model"]
    rows = np.asarray(model.cons_row).reshape(-1)
    worst = 0.
    for c, (A, E) in ref["acc"].items():
        d = A.shape[0]
        got = rb["delassus"][4*rows[c]:4*rows[c] + d*d].reshape(d, d)
        worst = max(worst, artref.err_ratio(got, A, E, Cc))
    out["delassus"] = worst
    if "finish" in ref and "gvel" in rb:
        qn, E, gp, Eg = ref["finish"]
        out["finish_v"] = artref.err_ratio(rb["gvel"], qn, E, Cc)
        out["finish_p"] = artref.err_ratio(rb["gpos"], gp, Eg, Cc)
    return out


def run_family(name, mutate=()):
    worlds = artbanks.family(name)
    rbs = [host_readback(w, k) for k, w in enumerate(worlds)]
    jobs = [artbanks.job(w, rb["gens"], np.flatnonzero(rb["active"]), rb["y"], mutate) for w, rb in zip(worlds, rbs)]
    refs = artref.run(jobs)
    return worlds, rbs, refs


@pytest.mark.parametrize("name", artbanks.FAMILIES)
def test_host_prepare_and_finish_vs_50_digits(name):
    worlds, rbs, refs = run_family(name)
    kz = artbanks.expect(name, worlds, refs, [rb["active"] for rb in rbs], [rb["gens"] for rb in rbs])
    worst = {}
    for w, rb, ref in zip(worlds, rbs, refs):
        for k, v in ratios(w, rb, ref).items():
            if v > worst.get(k, (0, ""))[0]:
                worst[k] = (v, w["tag"])
    print(name, "cond(Z) %.1e .. %.1e" % (min(kz), max(kz)), {k: "%.3g (%s)" % v for k, v in worst.items()})
    for k, (v, tag) in worst.items():
        assert v <= 1., "%s: %s err/(C u E) = %.3g in world %s" % (name, k, v, tag)


def test_unknown_family_raises():
    with pytest.raises(KeyError):
        artbanks.family("nonesuch")
    with pytest.raises(KeyError):
        artbanks.expect("nonesuch", [], [], [], [])


# each mutation of the REFERENCE (artref.MUTATIONS), the family built to resolve it, and what it must break
BITES = [("drop_N", "fixtures", "qfree"), ("drop_PD", "fixtures", "qfree"), ("drop_B", "fixtures", "qfree"),
         ("unrotated", "fixtures", "lambda"), ("lambda_T", "fixtures", "lambda"),
         ("flip_wrench", "instantiations", "qfree"), ("free_half_dt", "fixtures", "finish_p")]


@pytest.mark.parametrize("mutation,name,what", BITES)
def test_reference_mutations_bite(mutation, name, what):
    worlds, rbs, refs = run_family(name, (mutation,))
    worst = max(ratios(w, rb, ref)[what] for w, rb, ref in zip(worlds, rbs, refs))
    assert worst > 1., "%s undetected by %s (%s: %.3g)" % (mutation, name, what, worst)
