"""CPU tier: the host build (g++) of the small dense routines and of the soft-finger contact solve,
and the numpy oracle's SoftFingerContact.solve, against the 50-digit reference (tests/smallref.py) on
the seeded banks of tests/smallbanks.py; each family's liveness (it reaches the path it targets, its
ambiguity band stays small); and a check that the comparisons are live (a reference moved at one
boundary makes the family that targets it fail)."""
import numpy as np
import pytest

import smallbanks as banks
import smallcheck as chk
import smallref as ref

CONTACT = banks.contact_families()
SLIDE = banks.sliding_families()
POLY = banks.poly_families()
PINV = banks.pinv_families()
SOLVE = banks.solve_families()
EIG = banks.eig_families()
SE3 = banks.se3_families()
FRAMES = banks.frame_families()

# ceiling on the problems of a family inside the rounding band (either outcome accepted there).  Two families
# are all band by construction, and their values are compared nonetheless:
#  - pinv_rank: an exact zero singular value is computed with an absolute error of a few eps sigma_max, above
#    the 1e-15 sigma_max cut, so keeping or cutting it is not determined in float64 (numpy's pinv is in the
#    same position); the result must match the reference's or numpy's pseudo-inverse within 100 eps cond;
#  - eig_defective: a Jordan block of size m splits into m eigenvalues on a circle of radius ~eps^(1/m), real
#    or complex at random, so the count of real eigenvalues is not determined; every eigenvalue is still
#    compared, within 30 eps^(1/m) of the scale.
BAND_CEILING = {"contact_generic": 0.05, "contact_clamp": 0.1, "contact_release_edge": 0., "contact_static_edge": 0.1,
                "contact_yn_tiny": 0.1, "contact_eps": 0.1, "slide_generic": 0.05, "slide_zero_root": 0.,
                "slide_tangent": 0.5, "slide_yn_tiny": 0.1, "slide_no_root": 0.05, "slide_beyond_clamp": 0.05, "pinv_straddle": 0.34,
                "pinv_cond": 0., "pinv_rank": 1., "eig_defective": 1., "eig_companion": 0., "eig_balance": 0.,
                "eig_exceptional": 0.}


@pytest.fixture(scope="module")
def host():
    return chk.HostLib()


def _assert(rep):
    print(rep)
    assert not rep.bad, (rep.name, rep.bad[:5])
    ceil = BAND_CEILING.get(rep.name)
    if ceil is not None:
        assert rep.band <= ceil * rep.n, (rep.name, rep.band, rep.n)


def contact_ref(name):
    return chk.cached(("contact", name), lambda: chk.contact_refs(CONTACT[name]))


def contact_oracle(name):
    return chk.cached(("oracle", name), lambda: chk.oracle_softfinger(CONTACT[name]))


def run_contact(impl, fam):
    return impl.softfinger_solve(fam["v"], fam["A"], fam["P"], fam["sdist"], fam["mu"], fam["eps"], fam["dt"], fam["f0"])


@pytest.mark.parametrize("name", sorted(CONTACT))
def test_contact_host_vs_mp(host, name):
    fam = CONTACT[name]
    res = run_contact(host, fam)
    orc = contact_oracle(name)
    alt = [(np.array([o[0] for o in orc]), None)] if orc is not None else []
    _assert(chk.check_contact(name, fam, res, contact_ref(name), alt=alt))


@pytest.mark.parametrize("name", sorted(k for k in CONTACT if CONTACT[k].get("P_is_pinv", True)))
def test_contact_oracle_vs_mp(name):
    """the oracle's softfinger_solve (numpy, the restatement every world test trusts) on the same banks"""
    fam = CONTACT[name]
    orc = contact_oracle(name)
    n = len(orc)
    F = np.array([o[1] for o in orc])
    DF = np.array([o[2] for o in orc])
    BR = np.array([o[0] for o in orc])
    ST = np.array([ref.ST_EIG_NOROOT if o[3] is not None and not _has_root(o[3][0]) else 0 for o in orc])
    rep = chk.check_contact(name, fam, (F, DF, BR, ST), contact_ref(name), alt=[(BR, None)])
    _assert(rep)
    assert n == len(fam["v"])


def _has_root(B):
    S = np.linalg.eigvals(B)
    return bool(((S.imag == 0) & (S.real <= 0)).any())


def test_contact_families_reach_their_branches():
    br = {k: [r["br"] for r in contact_ref(k)] for k in CONTACT}
    assert set(br["contact_generic"]) == {1, 2, 3}
    rel = [r["rel"] for r in contact_ref("contact_release_edge")]
    assert sum(x == 0 for x in rel) >= 4 and sum(x > 0 for x in rel) >= 16 and sum(x < 0 for x in rel) >= 16
    st = [r.get("stat") for r in contact_ref("contact_static_edge")]
    assert sum(x == 0 for x in st) >= 6 and sum(x > 0 for x in st) >= 12 and sum(x < 0 for x in st) >= 12
    assert all(r["stat_bound"] == 0. for r in contact_ref("contact_static_edge"))
    assert all(r["rel_bound"] == 0. for r in contact_ref("contact_release_edge"))
    assert br["contact_eps"].count(3) >= 10 and br["contact_yn_tiny"].count(2) >= 4
    assert len(set(br["contact_static_edge"])) == 2
    # the clamp family: decided sliding problems without an admissible root (s = -1e10, EIG_NOROOT) and with
    # their root beyond the clamp
    cl = [r for r in contact_ref("contact_clamp") if r["br"] == 3 and chk._slide_decided(r["slide"])]
    assert sum(not r["slide"]["found"] for r in cl) >= 12
    assert sum(r["slide"]["found"] and r["slide"]["s"] < -ref.CLAMP for r in cl) >= 12
    assert all(r["status"] == (0 if r["slide"]["found"] else ref.ST_EIG_NOROOT) for r in cl)


def slide_ref(name):
    return chk.cached(("slide", name), lambda: chk.slide_refs(SLIDE[name]))


@pytest.mark.parametrize("name", sorted(SLIDE))
def test_sliding_root_host_vs_mp(host, name):
    fam = SLIDE[name]
    res = host.sliding_root(fam["A"], fam["alpha"], fam["mu"])
    _assert(chk.check_sliding_root(name, fam, res, slide_ref(name), alt=[(None, numpy_found(fam))]))


def numpy_found(fam):
    """whether numpy's eigvals of the float64 B (the oracle's path) finds an admissible root"""
    return np.array([_has_root(banks._np_sliding_matrix(a, x, m)) for a, x, m in zip(fam["A"], fam["alpha"], fam["mu"])])


def test_sliding_families_land_where_they_claim():
    z = slide_ref("slide_zero_root")
    assert sum(r["zero"] == 0 and r["exact"] for r in z) >= 6
    assert not any(r["found"] for r in slide_ref("slide_no_root"))
    assert sum(r["found"] and r["s"] < -ref.CLAMP for r in slide_ref("slide_beyond_clamp")) >= 20
    t = slide_ref("slide_tangent")
    def real_gap(r):
        re = sorted(x for x, y in r["eigs"] if y == 0.)
        return min([b - a for a, b in zip(re, re[1:])] or [np.inf])
    assert sum(r["imag"] < 1e-3 for r in t) >= 5 and sum(real_gap(r) < 1e-3 for r in t) >= 5


def test_bad_structured_path_falls_back_to_eig6(host):
    """sigma = 0: sliding_root_structured refuses the problem (on every call form), and eig_real_general6 --
    the fallback of softfinger_sliding -- gets B's eigenvalues (all 0) against the reference"""
    fam = banks.bad_sliding_family()
    S, FO, OK = host.sliding_root(fam["A"], fam["alpha"], fam["mu"])
    assert not OK.any()
    refs = chk.cached(("eig", "bad"), lambda: [chk.eig_ref(b) for b in fam["B"]])
    _assert(chk.check_eig("slide_bad_eig6", fam, host.eig6(fam["B"]), refs))


def poly_ref(name):
    return chk.cached(("poly", name), lambda: chk.poly_refs(POLY[name]))


def _poly_x(name):
    return np.array([(r["largest"] if r["largest"] is not None else 0.) + 1e-3 for r in poly_ref(name)])


@pytest.mark.parametrize("name", sorted(POLY))
def test_poly6_host_vs_mp(host, name):
    fam = POLY[name]
    res = host.poly6(fam["p"], _poly_x(name))
    _assert(chk.check_poly(name, fam, res, poly_ref(name)))
    fast_ok, _, positive, slow_n, _, _ = res
    n = len(fam["p"])
    # liveness: at least 90 % of the family takes the exit it targets (host counters for the recovery)
    if name == "poly_recover":
        assert host.recovered.sum() >= 0.9 * n, host.recovered.sum()
    elif name == "poly_positive":
        assert ((fast_ok == 0) & (positive == 1)).sum() >= 0.9 * n
    else:
        assert ((fast_ok == 0) & (positive == 0) & (slow_n > 0)).sum() >= 0.9 * n


def pinv_ref(name):
    return chk.cached(("pinv", name), lambda: chk.pinv_refs(PINV[name]))


@pytest.mark.parametrize("name", sorted(PINV))
def test_pinv_host_vs_mp(host, name):
    fam = PINV[name]
    out = host.pinv(fam["A"])
    npv = np.array([np.linalg.pinv(a) for a in fam["A"]])
    _assert(chk.check_pinv(name, fam, out, pinv_ref(name), alt=[npv]))
    if name == "pinv_cond":
        _, cond = host.inv_cond4(fam["A"])
        _assert(chk.check_cond(name + "_decision", fam, cond, [ref.cond1(a) for a in fam["A"]]))


def test_pinv_small_sizes(host):
    """1x1 (zero and not) and 3x3 against the reference"""
    a1 = np.array([[[0.]], [[2.5]], [[-1e-300]]])
    out = host.pinv(a1)
    assert out[0, 0, 0] == 0. and out[1, 0, 0] == 0.4 and out[2, 0, 0] == 1. / -1e-300
    rng = np.random.default_rng(9)
    a3 = rng.normal(size=(12, 3, 3))
    a3[::3, :, 2] = a3[::3, :, 0] * 2.
    _assert(chk.check_pinv("pinv3", {}, host.pinv(a3), [ref.pinv(a) for a in a3],
                           alt=[np.array([np.linalg.pinv(a) for a in a3])]))


@pytest.mark.parametrize("name", sorted(SOLVE))
def test_solve4_host_vs_mp(host, name):
    fam = SOLVE[name]
    res = host.solve4(fam["A"], fam["b"])
    refs = [ref.solve(a, b) if name != "solve_singular" else (None, np.inf) for a, b in zip(fam["A"], fam["b"])]
    _assert(chk.check_solve(name, fam, res, refs, singular=name == "solve_singular"))


def eig_ref(name):
    return chk.cached(("eig", name), lambda: [chk.eig_ref(a) for a in EIG[name]["A"]])


@pytest.mark.parametrize("name", sorted(EIG))
def test_eig6_host_vs_mp(host, name):
    fam = EIG[name]
    _assert(chk.check_eig(name, fam, host.eig6(fam["A"]), eig_ref(name)))


def test_se3_exp_host_vs_mp(host):
    fam = SE3["se3_switch"]
    refs = [ref.twist_exp(t) for t in fam["tw"]]
    _assert(chk.check_se3("se3_switch", fam, host.se3_exp(fam["tw"]), refs))
    assert sum(r["margin"] == 0 for r in refs) >= 3 and sum(not r["rodrigues"] for r in refs) >= 12


def test_zaligned_and_collide_host_vs_mp(host):
    fam = FRAMES["zaligned_ties"]
    refs = [ref.zaligned(z) for z in fam["z"]]
    assert sum(r["margin"] == 0 for r in refs) >= 10
    _assert(chk.check_zaligned("zaligned_ties", fam, host.zaligned(fam["z"]), refs))
    fam = FRAMES["collide"]
    refs = [ref.collide(p, c, h0, h1) for p, c, h0, h1 in zip(fam["pair"], fam["cd"], fam["H0"], fam["H1"])]
    assert sum(r.get("face", 1.) == 0 for r in refs) >= 2 and sum(r.get("inside", 1.) == 0 for r in refs) >= 4
    assert sum(r.get("sign", 1.) == 0 for r in refs) >= 2
    _assert(chk.check_collide("collide", fam, host.collide(fam["pair"], fam["cd"], fam["H0"], fam["H1"]), refs))


# ---------------------------------------------------------------------------------------------------
# the comparisons are live: a reference moved at one boundary fails the family that targets it
# ---------------------------------------------------------------------------------------------------
def test_moved_rcond_fails_the_straddle_family(host, monkeypatch):
    fam = PINV["pinv_straddle"]
    out = host.pinv(fam["A"])
    monkeypatch.setattr(ref, "RCOND", 1e-14)
    assert chk.check_pinv("pinv_straddle", fam, out, chk.pinv_refs(fam)).bad


def test_moved_series_switch_fails_the_se3_family(host, monkeypatch):
    fam = SE3["se3_switch"]
    out = host.se3_exp(fam["tw"])
    monkeypatch.setattr(ref, "SERIES_SWITCH", 2e-3)
    assert chk.check_se3("se3_switch", fam, out, [ref.twist_exp(t) for t in fam["tw"]]).bad


def test_strict_zero_inclusion_fails_the_zero_root_family(host, monkeypatch):
    fam = SLIDE["slide_zero_root"]
    res = host.sliding_root(fam["A"], fam["alpha"], fam["mu"])
    monkeypatch.setattr(ref, "INCLUSIVE_ZERO", False)
    assert chk.check_sliding_root("slide_zero_root", fam, res, chk.slide_refs(fam)).bad


def test_dropped_noroot_bit_or_wrong_clamped_force_fails_the_clamp_family(host):
    """the status rule and the force of the clamped solve are compared: clearing EIG_NOROOT on the no-root
    problems, or scaling the force of a clamped solve, is a violation"""
    fam = CONTACT["contact_clamp"]
    refs = contact_ref("contact_clamp")
    F, DF, BR, ST = run_contact(host, fam)
    noroot = np.array([r["br"] == 3 and not r["slide"]["found"] for r in refs])
    beyond = np.array([r["br"] == 3 and r["slide"]["found"] and r["slide"]["s"] < -ref.CLAMP for r in refs])
    rep = chk.check_contact("contact_clamp", fam, (F, DF, BR, ST), refs)
    assert not rep.bad
    decided = np.ones(len(refs), bool)
    decided[rep.band_idx] = False
    noroot &= decided
    beyond &= decided
    assert noroot.sum() >= 12 and beyond.sum() >= 12
    st = ST.copy()
    st[noroot] &= ~ref.ST_EIG_NOROOT
    rep = chk.check_contact("contact_clamp", fam, (F, DF, BR, st), refs)
    assert {b[0] for b in rep.bad if b[1] == "EIG_NOROOT"} == set(np.nonzero(noroot)[0])
    # (the force rule is 100 eps cond(A - s D): a 50 % error is inside it only where cond > 2e13)
    tight = np.array([r["br"] == 3 and 100 * chk.EPS * r["slide"]["cond2"] < 0.5 for r in refs])
    assert (noroot & tight).sum() >= 8 and (beyond & tight).sum() >= 8
    for sel in (noroot & tight, beyond & tight):
        f = F.copy()
        f[sel] *= 1.5
        rep = chk.check_contact("contact_clamp", fam, (f, f - fam["f0"], BR, ST), refs)
        assert {b[0] for b in rep.bad} == set(np.nonzero(sel)[0])
