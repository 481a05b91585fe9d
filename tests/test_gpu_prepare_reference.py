"""The device's fused prepare stage through arb_get_fused (BatchedWorld.fused) against the 50-digit
reference of the impedance solve (artref.py), on the fixtures family of artbanks.py: q_free, v0, EVERY
entry of Lambda and the Delassus blocks of the active constraints within the bound C u E(x) of
artref.py; the finish stage from the read-back y; the read-backs' mapping through the world -> thread
assignment; the NaN rule of worlds without an active constraint and the refusal after a phase step."""
import numpy as np
import pytest
import artbanks
import artref

pytestmark = pytest.mark.gpu


def _batch(world, W=1):
    """a batch of W copies of the world, with its per-world inputs bound (so that the step runs the
    instantiation that reads them: applied forces artic_factor<true,false>, inertia or gravity <true,true>)"""
    from arboris_b200.batch import BatchedWorld
    bw = BatchedWorld(world["model"], W)
    bw.set_state(np.repeat(world["gpos"][:, None], W, 1), np.repeat(world["gvel"][:, None], W, 1),
                 np.repeat(world["cforce"][:, None], W, 1) if int(world["model"].nrows) else None)
    if world.get("tau") is not None:
        bodies = tuple(sorted(world["wrench"]))
        bw.set_applied_forces(np.repeat(world["tau"][:, None], W, 1),
                              np.repeat(np.array([world["wrench"][b] for b in bodies])[:, :, None], W, 2), bodies)
    if world.get("inertia") is not None:
        bodies, p = world["inertia"]
        bw.set_body_inertia(np.repeat(np.asarray(p)[:, :, None], W, 2), bodies)
    if world.get("gravity") is not None:
        bw.set_gravity(np.repeat(np.asarray(world["gravity"])[:, None], W, 1))
    return bw


@pytest.mark.parametrize("name", artbanks.FAMILIES)
def test_device_hand_over_vs_50_digits(name):
    worlds = artbanks.family(name)
    rbs, jobs = [], []
    for k, w in enumerate(worlds):
        bw = _batch(w)
        bw.begin_step(w["dt"])
        rb = {"gens": bw.generators(), "active": bw.constraints("active")[0].cpu().numpy()}
        for key in ("qfree", "v0", "lambda", "delassus", "y"):
            rb[key] = bw.fused(key)[0].cpu().numpy()
        rb["delassus"] = rb["delassus"].reshape(-1)
        bw.end_step(w["dt"])
        rb["gvel"], rb["gpos"] = bw.gvel[:, 0].cpu().numpy(), bw.gpos[:, 0].cpu().numpy()
        assert int(bw.status()[0]) == 0
        rbs.append(rb)
        jobs.append(artbanks.job(w, rb["gens"], np.flatnonzero(rb["active"]), rb["y"]))
        bw.close()
    refs = artref.run(jobs)
    kz = artbanks.expect(name, worlds, refs, [rb["active"] for rb in rbs], [rb["gens"] for rb in rbs])
    from test_prepare_reference import ratios
    worst = {}
    for w, rb, ref in zip(worlds, rbs, refs):
        for k, v in ratios(w, rb, ref).items():
            if v > worst.get(k, (0, ""))[0]:
                worst[k] = (v, w["tag"])
    print("device", name, "cond(Z) %.1e .. %.1e" % (min(kz), max(kz)), {k: "%.3g (%s)" % v for k, v in worst.items()})
    for k, (v, tag) in worst.items():
        assert v <= 1., "%s err/(C u E) = %.3g in world %s" % (k, v, tag)


def test_read_backs_map_through_the_assignment():
    """DISTINCT worlds (human36 states with different active sets, so that their sort keys differ and
    the sort permutes them): after arb_step with sort_period 2 every world's read-back is bit-identical to
    the same world's in a batch that never re-sorts, and to the world stepped alone; no two worlds'
    read-backs coincide, so a wrong world -> slot map cannot go unnoticed"""
    worlds = [x for x in artbanks.family("fixtures") if x["tag"] == "human36_contact64"]
    W = 96
    ids = np.arange(W) % len(worlds)
    gpos = np.stack([worlds[i]["gpos"] for i in ids], 1)
    gvel = np.stack([worlds[i]["gvel"] for i in ids], 1)*(1. + 1e-3*np.arange(W))   # every world its own state
    dt = worlds[0]["dt"]
    # (not the Delassus rows: those of inactive constraints are unspecified, left by whichever world last
    # held the slot)
    keys = ("qfree", "v0", "lambda", "y", "gframe")
    got = {}
    for period in (0, 2):
        from arboris_b200.batch import BatchedWorld
        bw = BatchedWorld(worlds[0]["model"], W)
        bw.set_option("sort_period", period)
        bw.set_state(gpos, gvel)
        bw.step(dt, 3)                          # re-sorts before steps 2 (sort_period 2)
        got[period] = {k: bw.fused(k).cpu().numpy() for k in keys}
        got[period]["state"] = (bw.gpos.cpu().numpy(), bw.gvel.cpu().numpy())
        bw.close()
    for k in keys:
        assert (got[0][k].view(np.int64) == got[2][k].view(np.int64)).all(), k
    q = got[2]["qfree"]
    assert len({q[w].tobytes() for w in range(W)}) == W
    for w in (0, 37, W - 1):                   # the world alone, from the same state
        from arboris_b200.batch import BatchedWorld
        bw = BatchedWorld(worlds[0]["model"], 1)
        bw.set_state(gpos[:, w:w + 1], gvel[:, w:w + 1])
        bw.step(dt, 3)
        for k in keys:
            a = bw.fused(k).cpu().numpy()[0]
            assert (a.view(np.int64) == got[2][k][w].view(np.int64)).all(), (w, k)
        bw.close()


def test_nan_rule_and_refusal():
    """a world without an active constraint: NaN for v0, Lambda, y and the Delassus blocks, q_free
    formed; the read-back refuses after a phase step, and K without the group prepare stage"""
    from arboris_b200._capi import ArbError
    w = [x for x in artbanks.family("fixtures") if x["tag"] == "human36_contact64"][0]
    bw = _batch(w, 2)
    g = bw.gpos.cpu().numpy()
    g[:, 1] = np.asarray(w["model"].gpos0)
    g[:, 1][[0, 1, 2, 4, 5, 6, 8, 9, 10]] = np.eye(3).reshape(-1)
    g[[3, 7, 11], 1] = 50.                                          # far above the ground: nothing active
    bw.set_state(g, np.zeros_like(bw.gvel.cpu().numpy()))
    bw.begin_step(1e-3)
    act = bw.constraints("active").cpu().numpy()
    assert act[0].any() and not act[1].any()
    for k in ("v0", "lambda", "y", "delassus"):
        a = bw.fused(k).cpu().numpy()
        assert np.isfinite(a[0]).all() and np.isnan(a[1]).all(), k
    assert np.isfinite(bw.fused("qfree").cpu().numpy()).all()
    with pytest.raises(ArbError):
        bw.fused("K")
    bw.end_step(1e-3)
    bw.set_option("force_phases", 1)
    bw.step(1e-3)
    with pytest.raises(ArbError):
        bw.fused("qfree")
    bw.close()
