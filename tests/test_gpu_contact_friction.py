"""Per-world contact friction through ``BatchedWorld.set_contact_friction`` on the device: oracle parity
on every path that steps (and with the group prepare stage), independence from the Gauss-Seidel
variant, the thread assignment and the batch position, batches grouped by mu against batches built
with that mu, in-place writes, a NaN confined to its world, and the refusals."""
import numpy as np
import pytest

import contactfriction as cf

pytestmark = pytest.mark.gpu

NW = 8
FIXTURES = sorted(cf.FIXTURES)


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


@pytest.mark.parametrize("path", ["step", "begin_end", "phases", "step_phases", "step_group"])
@pytest.mark.parametrize("name", FIXTURES)
def test_friction_vs_oracle_on_device(torch_cuda, name, path):
    """teacher-forced from the oracle's states on each world's own model: within 1e-10 relative, no
    active-set or branch flip (step_group: the prepare_group option, which supports friction)"""
    model, st = cf.load(name, NW)
    cons, mu, full = cf.perturbed(model, NW, seed=1)
    opts = {"step_phases": {"force_phases": 1}, "step_group": {"prepare_group": 1}}.get(path, {})
    bw = _batch(model, NW, **opts)
    bw.set_contact_friction(mu, cons)
    oracles = [cf.oracle(model, full[:, w], [a[:, w] for a in st]) for w in range(NW)]
    nr = model.nrows
    worst, flips = {}, 0
    for s in range(cf.NSTEPS):
        bw.set_state(np.stack([o.gpos for o in oracles], 1), np.stack([o.gvel for o in oracles], 1),
                     np.stack([o.cforce for o in oracles], 1).reshape(nr, NW))
        if path in ("step", "step_phases", "step_group"):
            bw.step(cf.DT, 1)
        elif path == "begin_end":
            bw.begin_step(cf.DT)
            bw.end_step(cf.DT)
        else:
            bw.update_dynamic()
            bw.update_controllers(cf.DT)
            bw.update_constraints(cf.DT)
            bw.integrate(cf.DT)
        g, v, f = bw.get_state()
        act = bw.constraints("active").cpu().numpy()
        br = bw.constraints("branch").cpu().numpy()
        for w, o in enumerate(oracles):
            o.step(cf.DT)
            a = np.array(o.active, dtype=int)
            flips += int((act[w] != a).sum()) + int((br[w]*act[w] != np.array(o.branch)*a).sum())
            worst["gvel"] = max(worst.get("gvel", 0.), cf.rel(v[:, w], o.gvel))
            worst["gpos"] = max(worst.get("gpos", 0.), cf.rel(g[:, w], o.gpos))
            worst["cforce"] = max(worst.get("cforce", 0.), cf.rel(f[:, w], o.cforce))
    assert flips == 0, "active set / branch flips: %d" % flips
    assert not (bw.status().cpu().numpy() & 3).any()
    for k, v in worst.items():
        assert v <= 1e-10, (k, v)


def _tiled(name, reps, seed=3):
    model, st = cf.load(name, 64)
    W = 64*reps
    st = [np.tile(a, reps) for a in st]
    cons, mu, full = cf.perturbed(model, W, seed=seed)
    return model, W, st, cons, mu


def _run(model, W, st, cons, mu, nsteps=20, **opts):
    bw = _batch(model, W, **opts)
    if mu is not None:
        bw.set_contact_friction(mu, cons)
    bw.set_state(*st)
    for _ in range(nsteps):
        bw.step(cf.DT, 1)
    return bw.get_state() + (bw.constraints("branch").cpu().numpy(), bw.status().cpu().numpy())


@pytest.mark.parametrize("name", FIXTURES)
def test_friction_follows_the_world_not_the_slot(torch_cuda, name):
    """sort_period 0 and 2 (re-sorting every other step over 20 steps) and the Gauss-Seidel variants
    (staged, unstaged, general instantiation, cooperative) give the same bits with friction bound"""
    model, W, st, cons, mu = _tiled(name, 4)
    ref = _run(model, W, st, cons, mu, sort_period=0)
    if name != "nc_over_32":      # (the generated world's contacts have released by the last step)
        assert (ref[3] == 3).any()        # some contact slides
    for opts in ({"sort_period": 2}, {"gs_stage": 0}, {"gs_stage": 1}, {"gs_plain": 0}, {"gs_coop": 1},
                 {"gs_coop": 1, "sort_period": 2}):
        got = _run(model, W, st, cons, mu, **opts)
        for a, b in zip(got, ref):
            assert a.tobytes() == b.tobytes(), opts


def test_permuted_worlds_permute_the_results(torch_cuda):
    """the worlds of a batch and their mu permuted together: the results permuted, bit for bit"""
    model, W, st, cons, mu = _tiled("human36_contact", 2)
    ref = _run(model, W, st, cons, mu)
    perm = np.random.default_rng(5).permutation(W)
    got = _run(model, W, [a[:, perm] for a in st], cons, mu[:, perm])
    for a, b in zip(got[:3], ref[:3]):
        assert a.tobytes() == b[:, perm].tobytes()


@pytest.mark.parametrize("phases", [0, 1])
def test_groups_equal_batches_built_with_their_mu(torch_cuda, phases):
    """worlds grouped by four values of mu (all contacts): each group is, bit for bit, an unbound batch
    whose model has that mu"""
    model, st = cf.load("human36_contact", 64)
    values = (0.3, 0.6, 0.9, 1.4)
    W = 64*len(values)
    st4 = [np.tile(a, len(values)) for a in st]
    cs = cf.contacts(model)
    mu = np.repeat(np.repeat(np.array(values)[None, :], 64, 1), len(cs), 0)
    got = _run(model, W, st4, cs, mu, nsteps=10, force_phases=phases)
    for k, m in enumerate(values):
        ref = _run(cf.world_model(model, np.full(len(cs), m)), 64, st, None, None, nsteps=10, force_phases=phases)
        for a, b in zip(got[:3], ref[:3]):
            assert a[:, 64*k:64*(k + 1)].tobytes() == b.tobytes(), m


def test_in_place_write_takes_effect_at_the_next_step(torch_cuda):
    model, W, st, cons, mu = _tiled("human36_contact", 1)
    cs = cf.contacts(model)
    bw = _batch(model, W)
    bw.set_contact_friction(np.full((len(cs), W), 0.6), cs)
    assert bw.friction_constraints == tuple(cs) and bw.contact_indices() == cs
    bw.set_state(*st)
    bw.step(cf.DT, 1)
    mid = bw.get_state()
    ref = _batch(model, W)
    ref.set_contact_friction(np.full((len(cs), W), 0.6), cs)
    ref.set_state(*mid)
    ref.step(cf.DT, 1)
    same = ref.get_state()
    assert all(a.tobytes() == b.tobytes() for a, b in zip(bw.get_state(), mid))
    bw.contact_friction[:, 3] = 5.      # in place, between the two steps (world 3 slides at mu = 0.6)
    bw.step(cf.DT, 1)
    got = bw.get_state()
    changed = np.abs(got[1] - same[1]).max(0) > 0
    assert changed[3] and changed.sum() == 1
    bw.set_contact_friction(False)
    assert bw.contact_friction is None and bw.friction_constraints == ()


def test_nan_mu_flags_its_world_only(torch_cuda):
    """a NaN mu in world 3 (sliding contacts), on the fused stages and the phase kernels: only that
    world's status is set, the neighbours' bits are those of the batch without the NaN"""
    model, st = cf.load("human36_contact", 8)
    cs = cf.contacts(model)
    mu = np.full((len(cs), 8), 0.6)
    for phases in (0, 1):
        ref = _run(model, 8, st, cs, mu, nsteps=2, force_phases=phases)
        bad = mu.copy()
        bad[:, 3] = np.nan
        got = _run(model, 8, st, cs, bad, nsteps=2, force_phases=phases)
        assert got[4][3] != 0 and np.delete(got[4], 3).tobytes() == np.delete(ref[4], 3).tobytes()
        for a, b in zip(got[:3], ref[:3]):
            assert np.delete(a, 3, 1).tobytes() == np.delete(b, 3, 1).tobytes()


def test_friction_refusals_keep_the_binding(torch_cuda):
    from arboris_b200._capi import ArbError
    model, W, st, cons, mu = _tiled("human36_contact", 1)
    ref = _run(model, W, st, cons, mu, nsteps=3)
    bw = _batch(model, W)
    bw.set_contact_friction(mu, cons)
    with pytest.raises(ValueError):
        bw.set_contact_friction(np.ones((2, W)), (1,))
    limit = [c for c, t in enumerate(model.cons_type) if int(t) == 0][0]
    for ids, msg in (((len(model.cons_type),), "out of range"), ((-1,), "out of range"),
                     ((limit,), "not a contact"), ((2, 2), "twice")):
        with pytest.raises(ArbError, match=msg):
            bw.set_contact_friction(np.ones((len(ids), W)), ids)
    assert bw.friction_constraints == cons
    bw.set_state(*st)
    for _ in range(3):
        bw.step(cf.DT, 1)
    got = bw.get_state() + (bw.constraints("branch").cpu().numpy(), bw.status().cpu().numpy())
    for a, b in zip(got, ref):
        assert a.tobytes() == b.tobytes()
