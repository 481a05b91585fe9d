"""The fused step on the B200 on generated worlds (tests/genworlds.py), whose shapes reach kernel
variants no fixed fixture reaches: the unstaged Gauss-Seidel and the 64-bit cooperative mask past 32
constraints, the general staged instantiation, sorting, the group prepare stage with NG > 32 and its
fallback when the record does not fit in shared memory.

* arb_step against the oracle, teacher-forced, on a few worlds;
* the fused step against the four phase kernels (two independent algorithms) on every world of a
  batch of 1003;
* bit-identity of states, forces, branches and status after 50 free-running steps across the kernel
  options, batch sizes and batch positions;
* prepare_group against the lane stages (within 1e-10 where the group stage runs, bit-identical where
  it falls back).
"""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "hosttest"))
sys.path.insert(0, os.path.dirname(__file__))
import genworlds as G  # noqa: E402

pytestmark = pytest.mark.gpu

DT = G.DT
NSEED = 16          # distinct oracle-accepted states per world, tiled over the batch
W = 1003
NFREE = 50
WORLDS = sorted(G.CATALOGUE) + ["free%d" % s for s in G.FREE_SEEDS]


def rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max()/max(np.abs(b).max(), 1e-300)


_cache = {}


def world(name):
    if name not in _cache:
        spec = G.free_spec(int(name[4:])) if name.startswith("free") else G.CATALOGUE[name]
        model = G.build(spec, 0)
        if not name.startswith("free"):
            G.expect(name, model)
        gp, gv, _ = G.states(model, spec, 0, NSEED, steps=2)
        _cache[name] = (model, gp, gv)
    return _cache[name]


def batch(model, gp, gv, nworlds, **options):
    import torch
    from arboris_b200.batch import BatchedWorld
    bw = BatchedWorld(model, nworlds, device="cuda:0")
    for k, v in options.items():
        bw.set_option(k, v)
    reps = (nworlds + gp.shape[1] - 1)//gp.shape[1]
    bw.set_state(np.tile(gp, (1, reps))[:, :nworlds], np.tile(gv, (1, reps))[:, :nworlds])
    torch.cuda.synchronize()
    return bw


def snapshot(bw):
    import torch
    torch.cuda.synchronize()
    return {"gpos": bw.gpos.clone(), "gvel": bw.gvel.clone(), "cforce": bw.cforce.clone(),
            "active": bw.constraints("active").clone(), "branch": bw.constraints("branch").clone(),
            "status": bw.status().clone()}


def bits_equal(a, b):
    import torch
    if a.dtype == torch.float64:
        return bool(torch.equal(a.view(torch.int64), b.view(torch.int64)))
    return bool(torch.equal(a, b))


@pytest.mark.parametrize("name", WORLDS)
def test_arb_step_vs_oracle(name):
    """teacher-forced from the oracle's states: velocities, positions and forces within 1e-10,
    active sets and branches identical"""
    from oracle.arboris_oracle import OracleWorld
    model, gp, gv = world(name)
    nw, nc = 4, len(model.cons_type)
    bw = batch(model, gp[:, :nw], gv[:, :nw], nw)
    oracles = []
    for w in range(nw):
        o = OracleWorld(model.to_dict())
        o.gpos[:], o.gvel[:] = gp[:, w], gv[:, w]
        oracles.append(o)
    worst, flips = {}, 0
    for s in range(4):
        bw.set_state(np.stack([o.gpos for o in oracles], 1), np.stack([o.gvel for o in oracles], 1),
                     np.stack([o.cforce for o in oracles], 1) if model.nrows else None)
        bw.step(DT, 1)
        g, v, f = bw.get_state()
        act, br = bw.constraints("active").cpu().numpy(), bw.constraints("branch").cpu().numpy()
        for w, o in enumerate(oracles):
            o.step(DT)
            a = np.array(o.active, dtype=int)
            flips += int((act[w, :nc] != a).sum()) + int((br[w, :nc]*act[w, :nc] != np.array(o.branch)*a).sum())
            for k, x, r in (("gvel", v[:, w], o.gvel), ("gpos", g[:, w], o.gpos), ("cforce", f[:, w], o.cforce)):
                if r.size:
                    worst[k] = max(worst.get(k, 0.), rel(x, r))
    print("%s vs oracle: %s, flips %d" % (name, {k: "%.1e" % x for k, x in worst.items()}, flips))
    assert flips == 0
    assert not (bw.status().cpu().numpy() & 3).any()
    for k, x in worst.items():
        assert x <= 1e-10, (k, x)


@pytest.mark.parametrize("name", WORLDS)
def test_fused_vs_phase_kernels_every_world(name):
    """one step from the first state and one after 20 free steps, by both paths, on all 1003 worlds"""
    import torch
    model, gp, gv = world(name)
    bw = batch(model, gp, gv, W)
    worst, flips = 0., 0
    for lead in (0, 20):
        if lead:
            bw.step(DT, lead)
        good = torch.isfinite(bw.gvel).all(0)
        g0, v0, f0 = bw.gpos.clone(), bw.gvel.clone(), bw.cforce.clone()
        bw.set_option("force_phases", 1)
        bw.step(DT, 1)
        vp = bw.gvel.clone()
        ap, bp = bw.constraints("active").clone(), bw.constraints("branch").clone()
        bw.set_option("force_phases", 0)
        bw.gpos.copy_(g0); bw.gvel.copy_(v0); bw.cforce.copy_(f0)
        bw.step(DT, 1)
        af, bf = bw.constraints("active"), bw.constraints("branch")
        scale = vp.abs().amax(0).clamp_min(1e-3)
        dv = ((bw.gvel - vp).abs().amax(0)/scale)[good]
        worst = max(worst, dv.max().item())
        flips += int((ap != af)[good].sum()) + int(((bp != bf) & (af == 1))[good].sum())
        assert int(good.sum()) >= W//2, "most worlds stay finite"
    print("%s fused vs phases: max rel dv %.1e, flips %d" % (name, worst, flips))
    assert flips == 0
    assert worst <= 1e-10


VARIANTS = [("gs_stage", 0), ("gs_plain", 0), ("gs_coop", 1), ("sort_period", 0), ("sort_period", 1)]


@pytest.mark.parametrize("name", WORLDS)
def test_kernel_variants_bit_identical(name):
    """50 free-running steps: every option, batch size and batch position gives the same bits"""
    model, gp, gv = world(name)
    ref = batch(model, gp, gv, W)
    ref.step(DT, NFREE)
    r = snapshot(ref)
    # replicas of one state at different batch positions
    for k in ("gpos", "gvel", "cforce"):
        x = r[k][:, :W//NSEED*NSEED].reshape(r[k].shape[0], -1, NSEED)
        assert bits_equal(x, x[:, :1].expand_as(x).contiguous()), k
    for opt, val in VARIANTS:
        bw = batch(model, gp, gv, W, **{opt: val})
        bw.step(DT, NFREE)
        s = snapshot(bw)
        for k in r:
            assert bits_equal(s[k], r[k]), (opt, val, k)
    for nw in (1, 33):
        bw = batch(model, gp, gv, nw)
        bw.step(DT, NFREE)
        s = snapshot(bw)
        for k in r:
            x = r[k][..., :nw] if k in ("gpos", "gvel", "cforce") else r[k][:nw]
            assert bits_equal(s[k], x), (nw, k)


@pytest.mark.parametrize("name", WORLDS)
def test_prepare_group_vs_lane_stages(name):
    import torch
    model, gp, gv = world(name)
    supported = G.group_record_bytes(model) <= G.GROUP_SMEM_MAX
    ref = batch(model, gp, gv, W)
    bw = batch(model, gp, gv, W, prepare_group=1)
    nsteps = 1 if supported else 10      # (one step: two summation orders, compared at 1e-10)
    ref.step(DT, nsteps)
    bw.step(DT, nsteps)
    r, s = snapshot(ref), snapshot(bw)
    if not supported:       # the fallback: the lane stages themselves
        for k in r:
            assert bits_equal(s[k], r[k]), k
        return
    good = torch.isfinite(r["gvel"]).all(0)
    scale = r["gvel"].abs().amax(0).clamp_min(1e-3)
    dv = ((s["gvel"] - r["gvel"]).abs().amax(0)/scale)[good].max().item()
    print("%s prepare_group vs lanes: max rel dv %.1e" % (name, dv))
    assert bool(torch.equal(s["active"], r["active"]))
    assert dv <= 1e-10
