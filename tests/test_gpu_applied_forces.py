"""Per-world applied forces through ``BatchedWorld.set_applied_forces`` on the device: oracle parity
on every path that steps, independence from the thread assignment of the worlds, per-world effect,
and the refusals."""
import numpy as np
import pytest

from test_applied_forces import BODIES, DT, NSTEPS, NW, S0, _contact64, applied_forces, applied_oracle, rel

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a CUDA device")
    return torch


def _batch(model, W):
    from arboris_b200.batch import BatchedWorld
    return BatchedWorld(model, W, device="cuda:0")


@pytest.mark.parametrize("path", ["step", "begin_end", "phases", "step_phases"])
def test_applied_forces_vs_oracle_on_device(torch_cuda, path):
    """Teacher-forced from the oracle's states: velocities, positions and forces within 1e-10 relative,
    active sets and branches identical, World._gforce after update_controllers (phases) too."""
    model, tr = _contact64()
    W = NW
    tau, wrench = applied_forces(model, W)
    bw = _batch(model, W)
    if path == "step_phases":
        bw.set_option("force_phases", 1)
    bw.set_applied_forces(gforce=tau, wrench=wrench, bodies=BODIES)
    oracles = []
    for w in range(W):
        o = applied_oracle(model, tau[:, w], wrench[:, :, w], BODIES)
        o.gpos[:], o.gvel[:], o.cforce[:] = tr["gpos"][w, S0], tr["gvel"][w, S0], tr["cforce"][w, S0]
        oracles.append(o)
    worst, flips, nact = {}, 0, 0
    for s in range(NSTEPS):
        bw.set_state(np.stack([o.gpos for o in oracles], 1), np.stack([o.gvel for o in oracles], 1),
                     np.stack([o.cforce for o in oracles], 1))
        gf = None
        if path in ("step", "step_phases"):
            bw.step(DT, 1)
        elif path == "begin_end":
            bw.begin_step(DT)
            bw.end_step(DT)
        else:
            bw.update_dynamic()
            bw.update_controllers(DT)
            gf = bw.gforce().cpu().numpy()
            bw.update_constraints(DT)
            bw.integrate(DT)
        g, v, f = bw.get_state()
        act = bw.constraints("active").cpu().numpy()
        br = bw.constraints("branch").cpu().numpy()
        for w, o in enumerate(oracles):
            o.update_dynamic()
            o.update_controllers(DT)
            if gf is not None:
                worst["gforce"] = max(worst.get("gforce", 0.), rel(gf[w], o.gforce))
            o.update_constraints(DT)
            o.integrate(DT)
            a = np.array(o.active, dtype=int)
            flips += int((act[w] != a).sum()) + int((br[w]*act[w] != np.array(o.branch)*a).sum())
            nact += int(a.sum())
            worst["gvel"] = max(worst.get("gvel", 0.), rel(v[:, w], o.gvel))
            worst["gpos"] = max(worst.get("gpos", 0.), rel(g[:, w], o.gpos))
            worst["cforce"] = max(worst.get("cforce", 0.), rel(f[:, w], o.cforce))
    assert nact > 100
    assert flips == 0, "active set / branch flips: %d" % flips
    assert not (bw.status().cpu().numpy() & 3).any()
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


def _tiled(model, tr, reps):
    """reps copies of the 64 states at step S0, each world its own forces"""
    W = 64*reps
    gpos = np.tile(tr["gpos"][:, S0].T, reps)
    gvel = np.tile(tr["gvel"][:, S0].T, reps)
    cf = np.tile(tr["cforce"][:, S0].T, reps)
    tau, wrench = applied_forces(model, W, seed=1)
    return W, (gpos, gvel, cf), tau, wrench


def test_applied_forces_follow_the_world_not_the_slot(torch_cuda):
    """the fused stages run the worlds in sorted order when sort_period > 0: the forces are read by
    world, so 20 steps give the same state bit for bit as without sorting"""
    model, tr = _contact64()
    W, state, tau, wrench = _tiled(model, tr, 4)
    out = []
    for sort in (1, 0):
        bw = _batch(model, W)
        bw.set_option("sort_period", sort)
        bw.set_applied_forces(gforce=tau, wrench=wrench, bodies=BODIES)
        bw.set_state(*state)
        for _ in range(20):
            bw.step(DT, 1)
        out.append(bw.get_state() + (bw.constraints("branch").cpu().numpy(),))
    for a, b in zip(out[0], out[1]):
        assert a.tobytes() == b.tobytes()
    assert (out[0][3] == 3).any()        # some contact slides


def test_applied_forces_are_per_world_and_written_in_place(torch_cuda):
    """unbinding changes the result; zeroing the bound tensors in place gives the unbound result"""
    model, tr = _contact64()
    W, state, tau, wrench = _tiled(model, tr, 1)

    def run(bw):
        bw.set_state(*state)
        bw.step(DT, 5)
        return bw.get_state()

    bw = _batch(model, W)
    bw.set_applied_forces(gforce=tau, wrench=wrench, bodies=BODIES)
    pushed = run(bw)
    assert bw.applied_bodies == BODIES
    bw.applied_gforce.zero_()
    bw.applied_wrench.zero_()
    zeroed = run(bw)
    bw.set_applied_forces(gforce=False, wrench=False)
    assert bw.applied_gforce is None and bw.applied_wrench is None
    free = run(bw)
    for a, b in zip(zeroed, free):
        assert a.tobytes() == b.tobytes()
    d = np.abs(pushed[1] - free[1]).max(0)
    assert (d > 1e-6).all(), "every world moves under its own forces"
    # a force on one world only changes that world
    one = np.zeros((model.ndof, W))
    one[:, 7] = tau[:, 7]
    bw.set_applied_forces(gforce=one)
    single = run(bw)
    changed = np.abs(single[1] - free[1]).max(0) > 0
    assert changed[7] and changed.sum() == 1


def test_nan_force_flags_its_world_only(torch_cuda):
    model, tr = _contact64()
    W, state, tau, _ = _tiled(model, tr, 1)
    tau[5, 11] = np.nan
    for phases in (0, 1):
        bw = _batch(model, W)
        bw.set_option("force_phases", phases)
        bw.set_applied_forces(gforce=tau)
        bw.set_state(*state)
        bw.step(DT, 1)
        st = bw.status().cpu().numpy()
        assert st[11] & 1
        assert not (np.delete(st, 11) & 1).any()


def test_applied_forces_refusals(torch_cuda):
    from arboris_b200._capi import ArbError
    model, tr = _contact64()
    W = 8
    bw = _batch(model, W)
    with pytest.raises(ValueError):
        bw.set_applied_forces(gforce=np.zeros((model.ndof + 1, W)))
    with pytest.raises(ValueError):
        bw.set_applied_forces(wrench=np.zeros((2, 6, W)), bodies=(1,))
    for bodies in ((0,), (len(model.joint_type) + 1,), (3, 3)):
        with pytest.raises(ArbError):
            bw.set_applied_forces(wrench=np.zeros((len(bodies), 6, W)), bodies=bodies)
    assert bw.applied_wrench is None
    # the group prepare stage has no applied-force term: it refuses instead of ignoring them
    bw.set_option("prepare_group", 1)
    bw.set_applied_forces(gforce=np.ones((model.ndof, W)))
    with pytest.raises(ArbError, match="prepare_group"):
        bw.step(DT, 1)
    with pytest.raises(ArbError, match="prepare_group"):
        bw.begin_step(DT)
    bw.set_applied_forces(gforce=False)
    bw.step(DT, 1)
