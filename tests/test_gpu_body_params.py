"""Per-world body inertia and gravity through ``BatchedWorld.set_body_inertia`` / ``set_gravity`` on the
device: oracle parity on every path that steps and on the read-backs, mass-scaling invariance in one
batch, independence from the thread assignment and the Gauss-Seidel variant, a NaN confined to its
world, the refusals and the energy monitor."""
import numpy as np
import pytest

import bodyparams as bp

pytestmark = pytest.mark.gpu

NW = 8


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("GPU tests need a CUDA device")
    return torch


def _batch(model, W, **opts):
    from arboris_b200.batch import BatchedWorld
    bw = BatchedWorld(model, W, device="cuda:0")
    for k, v in opts.items():
        bw.set_option(k, v)
    return bw


@pytest.mark.parametrize("path", ["step", "begin_end", "phases", "step_phases"])
@pytest.mark.parametrize("name", ["human36_contact", "zoo", "snake_loop"])
def test_body_params_vs_oracle_on_device(torch_cuda, name, path):
    """teacher-forced from the oracle's states on each world's own model: within 1e-10 relative, no
    active-set or branch flip; on the phases M, N, gforce and every body's N_b as well"""
    model, st = bp.load(name, NW)
    bodies, P, G = bp.perturbed(model, NW, seed=1)
    bw = _batch(model, NW, **({"force_phases": 1} if path == "step_phases" else {}))
    bw.set_body_inertia(P, bodies)
    bw.set_gravity(G)
    oracles = [bp.oracle(model, bodies, P[:, :, w], G[:, w], [a[:, w] for a in st]) for w in range(NW)]
    nc, nr, nj = len(model.cons_type), model.nrows, len(model.joint_type)
    worst, flips = {}, 0
    for s in range(bp.NSTEPS):
        bw.set_state(np.stack([o.gpos for o in oracles], 1), np.stack([o.gvel for o in oracles], 1),
                     np.stack([o.cforce for o in oracles], 1).reshape(nr, NW) if nr else None)
        rb = None
        if path in ("step", "step_phases"):
            bw.step(bp.DT, 1)
        elif path == "begin_end":
            bw.begin_step(bp.DT)
            bw.end_step(bp.DT)
        else:
            bw.update_dynamic()
            bw.update_controllers(bp.DT)
            rb = (bw.matrix("mass").cpu().numpy(), bw.matrix("nleffects").cpu().numpy(), bw.gforce().cpu().numpy(),
                  [bw.body("nleffects", b).cpu().numpy() for b in range(1, nj + 1)])
            bw.update_constraints(bp.DT)
            bw.integrate(bp.DT)
        g, v, f = bw.get_state()
        if nc:
            act = bw.constraints("active").cpu().numpy()
            br = bw.constraints("branch").cpu().numpy()
        for w, o in enumerate(oracles):
            Mo, No, gfo = bp.oracle_step(o)
            if rb is not None:
                for k, a, b in (("M", rb[0][w], Mo), ("N", rb[1][w], No), ("gforce", rb[2][w], gfo)):
                    worst[k] = max(worst.get(k, 0.), bp.rel(a, b))
                for b in range(1, nj + 1):
                    if np.abs(o.body_nle[b]).max() > 0:
                        worst["N_b"] = max(worst.get("N_b", 0.), bp.rel(rb[3][b - 1][w], o.body_nle[b]))
            if nc:
                a = np.array(o.active, dtype=int)
                flips += int((act[w] != a).sum()) + int((br[w]*act[w] != np.array(o.branch)*a).sum())
            worst["gvel"] = max(worst.get("gvel", 0.), bp.rel(v[:, w], o.gvel))
            worst["gpos"] = max(worst.get("gpos", 0.), bp.rel(g[:, w], o.gpos))
            if nr:
                worst["cforce"] = max(worst.get("cforce", 0.), bp.rel(f[:, w], o.cforce))
    assert flips == 0, "active set / branch flips: %d" % flips
    assert not (bw.status().cpu().numpy() & 3).any()
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


def test_mass_scaling_in_one_batch(torch_cuda):
    """human36_free, all 17 bodies bound with k = 0.5, 1, 2, 4 times the model's parameters in one
    batch (one instantiation): every world equals the k = 1 world bit for bit after 20 steps, on the
    fused stages and on the phase kernels"""
    from arboris_b200 import massmatrix
    model, st = bp.load("human36_free", 1)
    W = 4*33
    st = [np.repeat(a, W, 1) for a in st]
    p0 = massmatrix.to_params(bp.body_masses(model))
    k = np.tile([0.5, 1., 2., 4.], W//4)
    P = p0[:, :, None]*k
    for phases in (0, 1):
        bw = _batch(model, W, force_phases=phases)
        bw.set_body_inertia(P, range(1, p0.shape[0] + 1))
        bw.set_state(*st)
        bw.step(bp.DT, 20)
        g, v, _ = bw.get_state()
        assert np.abs(v[:, 1]).max() > 0.1
        assert not bw.status().cpu().numpy().any()
        for w in range(W):
            assert g[:, w].tobytes() == g[:, 1].tobytes() and v[:, w].tobytes() == v[:, 1].tobytes(), w


def _tiled(name, reps, seed=3):
    model, st = bp.load(name, 64)
    W = 64*reps
    st = [np.tile(a, reps) for a in st]
    bodies, P, G = bp.perturbed(model, W, seed=seed)
    return model, W, st, bodies, P, G


def _run(model, W, st, bodies, P, G, nsteps=20, **opts):
    bw = _batch(model, W, **opts)
    bw.set_body_inertia(P, bodies)
    bw.set_gravity(G)
    bw.set_state(*st)
    for _ in range(nsteps):
        bw.step(bp.DT, 1)
    return bw.get_state() + (bw.constraints("branch").cpu().numpy(), bw.status().cpu().numpy())


def test_params_follow_the_world_not_the_slot(torch_cuda):
    """sorting (sort_period 1 against 0) and the Gauss-Seidel variants (staged, unstaged, cooperative)
    give the same 20 steps bit for bit with the parameters bound"""
    model, W, st, bodies, P, G = _tiled("human36_contact", 4)
    ref = _run(model, W, st, bodies, P, G, sort_period=0)
    assert (ref[3] == 3).any()        # some contact slides
    for opts in ({"sort_period": 1}, {"gs_stage": 0}, {"gs_plain": 0}, {"gs_coop": 1}):
        got = _run(model, W, st, bodies, P, G, **opts)
        for a, b in zip(got, ref):
            assert a.tobytes() == b.tobytes(), opts


def test_replicas_at_other_batch_positions(torch_cuda):
    """a world and its parameters moved to another column of the batch give the same result"""
    model, W, st, bodies, P, G = _tiled("human36_contact", 1)
    ref = _run(model, W, st, bodies, P, G)
    perm = np.random.default_rng(5).permutation(W)
    got = _run(model, W, [a[:, perm] for a in st], bodies, P[:, :, perm], G[:, perm])
    for a, b in zip(got[:3], ref[:3]):
        assert a.tobytes() == b[:, perm].tobytes()


def test_params_are_per_world_and_written_in_place(torch_cuda):
    """writing the model's own values into the bound tensors in place comes within rounding of the
    unbound step (human36's matrices are not exactly of the rigid-body form); a change in one world
    changes that world only"""
    from arboris_b200 import massmatrix
    model, W, st, bodies, P, G = _tiled("human36_contact", 1)
    bw = _batch(model, W)

    def run():
        bw.set_state(*st)
        bw.step(bp.DT, 5)
        return bw.get_state()

    free = run()
    bw.set_body_inertia(P, bodies)
    bw.set_gravity(G)
    moved = run()
    assert (np.abs(moved[1] - free[1]).max(0) > 1e-6).all(), "every world moves with its own parameters"
    assert bw.inertia_bodies == bodies
    p0 = massmatrix.to_params(bp.body_masses(model))
    bw.body_inertia.copy_(bw.body_inertia.new_tensor(np.repeat(p0[:, :, None], W, 2)))
    g0 = sum(float(c[0]) for t, c in zip(model.ctrl_type, model.ctrl_dbl) if int(t) == 0)*np.asarray(model.up)
    bw.gravity.copy_(bw.gravity.new_tensor(np.repeat(g0[:, None], W, 1)))
    own = run()
    assert bp.rel(own[1], free[1]) < 1e-9
    one = bw.body_inertia.clone()
    one[3, 0, 7] *= 2.
    bw.set_body_inertia(one)
    single = run()
    changed = np.abs(single[1] - own[1]).max(0) > 0
    assert changed[7] and changed.sum() == 1
    bw.set_body_inertia(False)
    bw.set_gravity(False)
    assert bw.body_inertia is None and bw.gravity is None
    for a, b in zip(run(), free):
        assert a.tobytes() == b.tobytes()


def test_nan_params_flag_their_world_only(torch_cuda):
    model, W, st, bodies, P, G = _tiled("human36_contact", 1)
    P[2, 4, 11] = np.nan
    G[1, 20] = np.nan
    for phases in (0, 1):
        bw = _batch(model, W, force_phases=phases)
        bw.set_body_inertia(P, bodies)
        bw.set_gravity(G)
        bw.set_state(*st)
        bw.step(bp.DT, 1)
        s = bw.status().cpu().numpy()
        assert s[11] & 1 and s[20] & 1
        assert not (np.delete(s, [11, 20]) & 1).any()


def test_body_params_refusals(torch_cuda):
    from arboris_b200._capi import ArbError
    from arboris_b200.flatten import FlatModel
    model, st = bp.load("human36_contact", 8)
    W = 8
    bw = _batch(model, W)
    with pytest.raises(ValueError):
        bw.set_body_inertia(np.zeros((2, 10, W)), (1,))
    with pytest.raises(ValueError):
        bw.set_gravity(np.zeros((3, W + 1)))
    for bodies in ((0,), (len(model.joint_type) + 1,), (3, 3)):
        with pytest.raises(ArbError):
            bw.set_body_inertia(np.zeros((len(bodies), 10, W)), bodies)
    assert bw.body_inertia is None
    d = model.to_dict()
    for k in ("ctrl_type", "ctrl_int", "ctrl_dbl"):
        d[k] = d[k][:0]
    with pytest.raises(ArbError, match="WeightController"):
        _batch(FlatModel.from_dict(d), W).set_gravity(np.zeros((3, W)))
    # the group prepare stage reads the model's inertia and gravity: it refuses
    bw.set_option("prepare_group", 1)
    for bind, unbind in ((lambda: bw.set_gravity(np.zeros((3, W))), lambda: bw.set_gravity(False)),
                         (lambda: bw.set_body_inertia(np.zeros((1, 10, W)), (2,)), lambda: bw.set_body_inertia(False))):
        bind()
        with pytest.raises(ArbError, match="prepare_group"):
            bw.step(bp.DT, 1)
        with pytest.raises(ArbError, match="prepare_group"):
            bw.begin_step(bp.DT)
        unbind()
        bw.step(bp.DT, 1)


def test_energy_monitor_with_bound_params(torch_cuda):
    """BatchedEnergyMonitor with per-world inertia and gravity against a numpy evaluation on each
    world's own matrices"""
    from arboris_b200 import massmatrix
    from arboris_b200.observers import BatchedEnergyMonitor
    model, W, st, bodies, P, G = _tiled("human36_contact", 1)
    bw = _batch(model, W)
    bw.set_body_inertia(P, bodies)
    bw.set_gravity(G)
    bw.set_state(*st)
    bw.step(bp.DT, 3)
    mon = BatchedEnergyMonitor()
    mon.init(bw, None)
    mon.update(bp.DT)
    mon.finish()
    bm = bp.body_masses(model)
    Ec, Ep = np.zeros(W), np.zeros(W)
    for b in range(1, len(bm) + 1):
        T = bw.body("twist", b).cpu().numpy()
        H = bw.body("pose", b).cpu().numpy()
        for w in range(W):
            M = massmatrix.from_params(P[bodies.index(b), :, w])
            Ec[w] += 0.5*T[w] @ M @ T[w]
            if M[3, 3] > 0:
                c = np.array([M[2, 4], M[0, 5], M[1, 3]])/M[3, 3]
                Ep[w] -= M[3, 3]*(H[w, :3, :3] @ c + H[w, :3, 3]) @ G[:, w]
    assert bp.rel(mon.kinetic_energy[0], Ec) < 1e-12
    assert bp.rel(mon.potential_energy[0], Ep) < 1e-12
