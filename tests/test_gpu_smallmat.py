"""GPU tier: the device arithmetic of the soft-finger contact solve and of the small dense routines
(tests/devtest/arb_devtest.cu, one problem per thread) against the 50-digit reference on the banks of
tests/smallbanks.py, against the host build on discrete outcomes, across the three call forms of the
sliding solve (per lane, ballot mask, shared-memory queue), across lane positions and warp neighbours,
and in the variant builds of DESIGN 3.3 (positivity march and bracket recovery off; Laguerre step with
IEEE square root and division).  Run with -s for the per-family summary."""
import importlib.util
import os

import numpy as np
import pytest

import smallbanks as banks
import smallcheck as chk
import smallref as ref

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
_spec = importlib.util.spec_from_file_location("arb_devtest_harness", os.path.join(HERE, "devtest", "harness.py"))
devharness = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(devharness)

CONTACT = banks.contact_families()
SLIDE = banks.sliding_families()
POLY = banks.poly_families()
PINV = banks.pinv_families()
SOLVE = banks.solve_families()
EIG = banks.eig_families()
SE3 = banks.se3_families()
FRAMES = banks.frame_families()

VARIANTS = {"no_march_no_recover": ("ARB_POSITIVE_MARCH=0", "ARB_FASTROOT_RECOVER=0"),
            "ieee_laguerre": ("ARB_LAGUERRE_FAST=0",)}

import test_smallmat_banks as cpu  # noqa: E402  (shared reference caches and band ceilings)


@pytest.fixture(scope="module")
def dev():
    return devharness.DevLib()


@pytest.fixture(scope="module")
def host():
    return chk.HostLib()


def _assert(rep):
    cpu._assert(rep)


def _odd(fam, keys):
    """the bank padded by repeating its first problem so that N is not a multiple of 32"""
    n = len(fam[keys[0]])
    if n % 32:
        return fam
    out = dict(fam)
    for k in keys:
        out[k] = np.concatenate([fam[k], fam[k][:1]])
    return out


CKEYS = ("v", "A", "P", "sdist", "mu", "eps", "f0")


def _contact_run(dev, fam, mode=None):
    if mode is None:
        return dev.softfinger_solve(fam["v"], fam["A"], fam["P"], fam["sdist"], fam["mu"], fam["eps"], fam["dt"], fam["f0"])
    return dev.softfinger_fused(mode, fam["v"], fam["A"], fam["P"], fam["sdist"], fam["mu"], fam["eps"][0], fam["dt"],
                                fam["f0"])


@pytest.mark.parametrize("name", sorted(CONTACT))
def test_contact_device_vs_mp_and_host(dev, host, name):
    fam = CONTACT[name]
    n = len(fam["v"])
    pf = _odd(fam, CKEYS)
    refs = cpu.contact_ref(name)
    hb = cpu.run_contact(host, fam)
    orc = cpu.contact_oracle(name)
    alt = [(hb[2], hb[0])] + ([(np.array([o[0] for o in orc]), None)] if orc is not None else [])
    res = [a[:n] for a in _contact_run(dev, pf)]
    _assert(chk.check_contact(name, fam, res, refs, alt=alt))
    # the fused form, three call forms of the sliding solve: identical bits
    forms = [[a[:n] for a in _contact_run(dev, pf, mode)] for mode in (0, 1, 2)]
    for m in (1, 2):
        for a, b in zip(forms[0], forms[m]):
            assert np.array_equal(a, b, equal_nan=True), (name, m)
    rep = chk.check_contact(name + "/fused", fam, forms[0], refs, alt=alt)
    rep.name = name
    _assert(rep)
    # discrete outcomes of device and host builds agree wherever the reference decides them
    agree = (res[2] == hb[2]) | np.array([chk_band(r) for r in refs])
    assert agree.all(), np.nonzero(~agree)


def chk_band(r):
    if not (abs(r["rel"]) > r["rel_bound"] or r["rel_bound"] == 0.):
        return True
    if r["br"] != 1 and "stat" in r and not (abs(r["stat"]) > r["stat_bound"] or r["stat_bound"] == 0.):
        return True
    return r["br"] == 3 and not chk._slide_decided(r["slide"])


@pytest.mark.parametrize("name", sorted(SLIDE))
def test_sliding_root_device_vs_mp(dev, host, name):
    fam = SLIDE[name]
    n = len(fam["A"])
    pf = _odd(fam, ("A", "alpha", "mu"))
    hres = host.sliding_root(fam["A"], fam["alpha"], fam["mu"])
    alt = [(None, hres[1]), (None, cpu.numpy_found(fam))]
    for coop in (0, 1):
        res = [a[:n] for a in dev.sliding_root(pf["A"], pf["alpha"], pf["mu"], coop)]
        _assert(chk.check_sliding_root(name, fam, res, cpu.slide_ref(name), alt=alt))
        if coop:
            assert all(np.array_equal(a, b) for a, b in zip(res, prev)), name
        prev = res


def test_bad_structured_path_device(dev):
    fam = banks.bad_sliding_family()
    for coop in (0, 1):
        assert not dev.sliding_root(fam["A"], fam["alpha"], fam["mu"], coop)[2].any()
    refs = chk.cached(("eig", "bad"), lambda: [chk.eig_ref(b) for b in fam["B"]])
    _assert(chk.check_eig("slide_bad_eig6", fam, dev.eig6(fam["B"]), refs))


@pytest.mark.parametrize("name", sorted(POLY))
def test_poly6_device_vs_mp(dev, host, name):
    fam = POLY[name]
    n = len(fam["p"])
    x = cpu._poly_x(name)
    p = _odd(dict(p=fam["p"], x=x), ("p", "x"))
    res = [a[:n] for a in dev.poly6(p["p"], p["x"])]
    _assert(chk.check_poly(name, fam, res, cpu.poly_ref(name)))
    h = host.poly6(fam["p"], x)
    # exits.  The positivity march and the isolation count use IEEE operations only, and decide on margins far
    # from rounding on these banks: equal to the host build's.  The fast path's verdict is not a function with
    # a margin: it stops when |p| reaches its own rounding bound and certifies the iterate it stopped at, and
    # that iterate differs in the last bits between builds (FMA contraction, the MUFU seeds of the Laguerre
    # step); a verdict may then differ, the answer may not -- a root it returns is compared with the
    # reference above, on both builds.  The share of such differences is reported.
    for i in (2, 3):
        assert np.array_equal(res[i], h[i]), (name, i)
    print("%s: fast verdict differs from the host build on %d of %d" % (name, int((res[0] != h[0]).sum()), n))


@pytest.mark.parametrize("name", sorted(PINV))
def test_pinv_device_vs_mp(dev, host, name):
    fam = PINV[name]
    n = len(fam["A"])
    A = _odd(fam, ("A",))["A"]
    out = dev.pinv(A)[:n]
    npv = np.array([np.linalg.pinv(a) for a in fam["A"]])
    _assert(chk.check_pinv(name, fam, out, cpu.pinv_ref(name), alt=[npv, host.pinv(fam["A"])]))
    if name == "pinv_cond":
        _, cond = dev.inv_cond4(A)
        _assert(chk.check_cond(name + "_decision", fam, cond[:n], [ref.cond1(a) for a in fam["A"]]))


def test_pinv_small_sizes_device(dev):
    a1 = np.array([[[0.]], [[2.5]], [[-1e-300]]])
    out = dev.pinv(a1)
    assert out[0, 0, 0] == 0. and out[1, 0, 0] == 0.4 and out[2, 0, 0] == 1. / -1e-300
    rng = np.random.default_rng(9)
    a3 = rng.normal(size=(13, 3, 3))
    a3[::3, :, 2] = a3[::3, :, 0] * 2.
    _assert(chk.check_pinv("pinv3", {}, dev.pinv(a3), [ref.pinv(a) for a in a3],
                           alt=[np.array([np.linalg.pinv(a) for a in a3])]))


@pytest.mark.parametrize("name", sorted(SOLVE))
def test_solve4_device_vs_mp(dev, name):
    fam = SOLVE[name]
    res = dev.solve4(fam["A"], fam["b"])
    refs = [ref.solve(a, b) if name != "solve_singular" else (None, np.inf) for a, b in zip(fam["A"], fam["b"])]
    _assert(chk.check_solve(name, fam, res, refs, singular=name == "solve_singular"))


@pytest.mark.parametrize("name", sorted(EIG))
def test_eig6_device_vs_mp(dev, name):
    fam = EIG[name]
    _assert(chk.check_eig(name, fam, dev.eig6(fam["A"]), cpu.eig_ref(name)))


def test_se3_zaligned_collide_device_vs_mp(dev):
    fam = SE3["se3_switch"]
    _assert(chk.check_se3("se3_switch", fam, dev.se3_exp(fam["tw"]), [ref.twist_exp(t) for t in fam["tw"]]))
    fam = FRAMES["zaligned_ties"]
    _assert(chk.check_zaligned("zaligned_ties", fam, dev.zaligned(fam["z"]), [ref.zaligned(z) for z in fam["z"]]))
    fam = FRAMES["collide"]
    refs = [ref.collide(p, c, h0, h1) for p, c, h0, h1 in zip(fam["pair"], fam["cd"], fam["H0"], fam["H1"])]
    _assert(chk.check_collide("collide", fam, dev.collide(fam["pair"], fam["cd"], fam["H0"], fam["H1"]), refs))


def test_lane_position_and_neighbour_invariance(dev):
    """a probe problem at each of the 32 lane positions of a warp whose other lanes are drawn from the generic,
    boundary and clamp families (release, static, sliding with a root, with no admissible root and with its
    root beyond the clamp): bit-identical results in the phase form and in the three fused forms (DESIGN 3.2
    claims this of worlds).  (With ARB_SAMPLE_ROOT = 0, the default, the ballot mask changes only the early
    exits of sliding_root_structured; what this checks is that no call form depends on its neighbours.)"""
    names = ["contact_generic", "contact_release_edge", "contact_static_edge", "contact_yn_tiny", "contact_clamp"]
    fam = {k: np.concatenate([CONTACT[n][k] for n in names]) for k in CKEYS}
    fam["dt"] = banks.DT
    refs = sum((cpu.contact_ref(n) for n in names), [])
    br = np.array([r["br"] for r in refs])
    noroot = [k for k, r in enumerate(refs) if r["br"] == 3 and not r["slide"]["found"]]
    beyond = [k for k, r in enumerate(refs) if r["br"] == 3 and r["slide"]["found"] and r["slide"]["s"] < -ref.CLAMP]
    probes = [int(np.nonzero(br == b)[0][0]) for b in (1, 2, 3)] + [int(i) for i in np.nonzero(br == 3)[0][1:3]] + \
        [noroot[0], beyond[0]]
    pool = [k for k in range(len(br)) if k not in probes]
    rng = np.random.default_rng(3)
    idx = []
    for p in probes:
        for lane in range(32):
            warp = list(rng.choice(pool, size=32))
            warp[lane] = p
            idx += warp
    idx.append(pool[0])                          # N not a multiple of 32
    idx = np.array(idx)
    big = {k: fam[k][idx] for k in CKEYS}
    big["dt"] = fam["dt"]
    iso = {k: fam[k][probes] for k in CKEYS}
    iso["dt"] = fam["dt"]
    for mode in (None, 0, 1, 2):
        r_big = _contact_run(dev, big, mode)
        r_iso = _contact_run(dev, iso, mode)
        for j, p in enumerate(probes):
            at = np.nonzero(idx == p)[0]
            for a_big, a_iso in zip(r_big, r_iso):
                assert all(np.array_equal(a_big[i], a_iso[j]) for i in at), (mode, p)


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_variant_builds(dev, variant):
    """DESIGN 3.3 / 4: the variant builds give the same branches, found flags and status bits as the default
    build, and their s within the rule of the reference"""
    var = devharness.DevLib(VARIANTS[variant])
    for name in sorted(CONTACT):
        fam = _odd(CONTACT[name], CKEYS)
        a, b = _contact_run(dev, fam), _contact_run(var, fam)
        assert np.array_equal(a[2], b[2]) and np.array_equal(a[3], b[3]), (variant, name)
        n = len(CONTACT[name]["v"])
        _assert(chk.check_contact(name, CONTACT[name], [x[:n] for x in b], cpu.contact_ref(name), alt=[(a[2][:n], a[0][:n])]))
    for name in sorted(SLIDE):
        fam = SLIDE[name]
        n = len(fam["A"])
        pf = _odd(fam, ("A", "alpha", "mu"))
        a = dev.sliding_root(pf["A"], pf["alpha"], pf["mu"], 1)
        b = var.sliding_root(pf["A"], pf["alpha"], pf["mu"], 1)
        assert np.array_equal(a[1], b[1]) and np.array_equal(a[2], b[2]), (variant, name)
        _assert(chk.check_sliding_root(name, fam, [x[:n] for x in b], cpu.slide_ref(name), alt=[(None, a[1][:n])]))
