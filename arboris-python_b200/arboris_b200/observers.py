"""Observers of batched worlds: the downstream consumers of the step.

Mirrors of the reference's ``arboris/observers.py`` for ``BatchedWorld``:

* ``BatchedHdf5Logger``  <- ``Hdf5Logger`` (observers.py:133-289): ``timeline``, ``gpositions/``,
  ``gvelocities/``, ``transforms/`` with the reference's names and shapes, plus ONE extra axis
  for the worlds right after the step axis (dropped with ``squeeze=True`` when one world is
  logged, which gives the reference's ``flat=True`` datasets: ``timeline``, per-joint ``gpositions`` /
  ``gvelocities``, ``transforms`` of the ground and of every moving body).  NOT written: the
  transforms of the contacts' ``MovingSubFrame``s (observers.py:238-239; the fused step does not
  materialise contact frames) and the ``model/`` group (``save_model``, observers.py:245-252).  h5py is not needed: the file is written
  by ``arboris_b200.h5write`` (or as ``.npz`` with the same keys).
* ``BatchedEnergyMonitor`` <- ``EnergyMonitor`` (observers.py:14-54), one value per world.

Like the reference's, they are called by ``simulate()`` between ``update_constraints`` and
``integrate`` (core.py:1360-1362) and therefore see the state at the START of the interval.
Both are "fused-compatible" (``fused_ok``): ``simulate()`` keeps the fused CUDA step
(``begin_step`` / ``end_step``) instead of the four materialising phase calls.  Samples are kept
on the device and copied to the host once, in ``finish()``.
"""
import numpy as np
import torch

from . import massmatrix
from .core import Observer
from .flatten import JOINT_NDOF, JOINT_NGPOS


def _world_index(worlds, nworlds, device):
    if worlds is None:
        idx = torch.arange(nworlds, device=device)
    elif isinstance(worlds, slice):
        idx = torch.arange(nworlds, device=device)[worlds]
    else:
        idx = torch.as_tensor(np.asarray(worlds, dtype=np.int64), device=device)
    assert idx.numel() > 0 and int(idx.min()) >= 0 and int(idx.max()) < nworlds
    return idx


class BatchedHdf5Logger(Observer):
    """Save the trajectories of (a subset of) the worlds of a ``BatchedWorld``.

    :param filename: output file; ``*.npz`` selects numpy's format, anything else HDF5
    :param group: sub-group of the file that receives the data (default ``"/"``)
    :param save_state: write ``gpositions`` and ``gvelocities``
    :param save_transforms: write ``transforms`` (absolute body poses, the reference's
        ``flat=True`` layout)
    :param worlds: indices (or slice) of the worlds to log; default all
    :param squeeze: drop the world axis when a single world is logged
    """
    fused_ok = True

    def __init__(self, filename, group="/", save_state=True, save_transforms=True,
                 worlds=None, squeeze=False):
        self._filename, self._group = filename, group
        self._save_state, self._save_transforms = save_state, save_transforms
        self._worlds, self._squeeze = worlds, squeeze
        self.root = None

    def init(self, world, timeline):
        self._world = world
        m = world.model
        self._nb_steps = len(timeline) - 1
        self._current_step = 0
        self._idx = _world_index(self._worlds, world.nworlds, world.device)
        nsel = int(self._idx.numel())
        kw = dict(dtype=torch.float64, device=world.device)
        self._timeline = np.zeros(self._nb_steps)
        if self._save_state:
            self._gpos = torch.empty((self._nb_steps, int(m.ngpos), nsel), **kw)
            self._gvel = torch.empty((self._nb_steps, int(m.ndof), nsel), **kw)
        if self._save_transforms:
            self._bodies = [k for k in range(1, len(m.joint_type) + 1)]
            self._poses = torch.empty((self._nb_steps, len(self._bodies), nsel, 4, 4), **kw)

    def update(self, dt):
        assert self._current_step < self._nb_steps
        w, s = self._world, self._current_step
        self._timeline[s] = w.current_time
        if self._save_state:
            self._gpos[s] = w.gpos[:, self._idx]
            self._gvel[s] = w.gvel[:, self._idx]
        if self._save_transforms:
            for i, k in enumerate(self._bodies):
                self._poses[s, i] = w.body("pose", k)[self._idx]
        self._current_step += 1

    def _names(self, names, prefix, n):
        out, seen = [], set()
        for i in range(n):
            nm = names[i] if i < len(names) and names[i] else "%s%d" % (prefix, i)
            while nm in seen:
                nm += "_"
            seen.add(nm)
            out.append(nm)
        return out

    def tree(self):
        """The logged data as the nested dict the file holds."""
        m = self._world.model
        n = self._current_step
        sq = self._squeeze and int(self._idx.numel()) == 1

        def fix(a):          # (steps, worlds, ...) or (steps, ...)
            return a[:, 0] if sq else a
        root = {"timeline": self._timeline[:n].copy()}
        nj = len(m.joint_type)
        if self._save_state:
            gp, gv = self._gpos[:n].cpu().numpy(), self._gvel[:n].cpu().numpy()
            gpos, gvel = {}, {}
            for j, name in enumerate(self._names(m.joint_names, "Joint", nj)):
                t = int(m.joint_type[j])
                g0, d0 = int(m.joint_gpos[j]), int(m.joint_dof[j])
                q = np.moveaxis(gp[:, g0:g0 + JOINT_NGPOS[t]], 1, 2)      # (steps, worlds, ngpos)
                if t == 0:
                    q = q.reshape(q.shape[:2] + (4, 4))
                gpos[name] = fix(q)
                gvel[name] = fix(np.moveaxis(gv[:, d0:d0 + JOINT_NDOF[t]], 1, 2))
            root["gpositions"], root["gvelocities"] = gpos, gvel
        if self._save_transforms:
            P = self._poses[:n].cpu().numpy()
            has_ground = len(m.body_names) == nj + 1
            names = self._names(list(m.body_names)[1:] if has_ground else list(m.body_names), "Body", nj)
            root["transforms"] = {name: fix(P[:, i]) for i, name in enumerate(names)}
            # the ground is a body too (World.iterbodies, observers.py:233-235): identity
            gname = (m.body_names[0] if has_ground and m.body_names[0] else "ground")
            if gname not in root["transforms"]:
                eye = np.broadcast_to(np.eye(4), P[:, 0].shape).copy()
                root["transforms"][gname] = fix(eye)
        for g in [g for g in self._group.split("/") if g][::-1]:
            root = {g: root}
        return root

    def finish(self):
        self.root = self.tree()
        if self._filename is None:
            return
        if str(self._filename).endswith(".npz"):
            flat = {}

            def walk(t, prefix):
                for k, v in t.items():
                    if isinstance(v, dict):
                        walk(v, prefix + k + "/")
                    else:
                        flat[prefix + k] = v
            walk(self.root, "")
            np.savez(self._filename, **flat)
        else:
            from . import h5write
            h5write.write(self._filename, self.root)


class BatchedEnergyMonitor(Observer):
    """Kinetic, potential and mechanical energy of every world at every step
    (``EnergyMonitor``, observers.py:14-54; the attribute names are the reference's).
    The kinetic energy ``gvel^T M gvel / 2`` is evaluated body by body,
    ``sum_b T_b^T M_b T_b / 2`` with ``T_b = J_b gvel``, so the mass matrix is not assembled.
    Bodies with per-world inertia (``BatchedWorld.set_body_inertia``) count with each world's own
    matrix, and with per-world gravity (``set_gravity``) the potential energy is
    ``-sum_b m_b g_w . p_com,b`` instead of ``9.81 sum_b m_b up . p_com,b``."""
    fused_ok = True

    def init(self, world, timeline):
        self._world = world
        m = world.model
        self.time = []
        self.kinetic_energy, self.potential_energy, self.mechanichal_energy = [], [], []
        dev = world.device
        M = np.asarray(m.body_mass, dtype=float).reshape(-1, 6, 6)
        self._bodies = [k for k in range(M.shape[0]) if np.any(M[k] != 0.)]
        self._M = torch.as_tensor(M, device=dev)
        com = np.zeros((M.shape[0], 4))
        com[:, 3] = 1.
        for k in self._bodies:
            mass = M[k][5, 5]
            if mass > 0:
                rx = M[k][0:3, 3:6]/mass            # massmatrix.principalframe: H[0:3,3]
                com[k, :3] = (rx[2, 1], rx[0, 2], rx[1, 0])
        self._com = torch.as_tensor(com, device=dev)
        self._up = torch.as_tensor(np.asarray(m.up, dtype=float), device=dev)

    def update(self, dt):
        w = self._world
        self.time.append(w.current_time)
        Ec = torch.zeros(w.nworlds, dtype=torch.float64, device=w.device)
        Ep = torch.zeros_like(Ec)
        bound = getattr(w, "inertia_bodies", ())
        g = getattr(w, "gravity", None)
        if not bound and g is None:
            for k in self._bodies:
                T = w.body("twist", k + 1)                       # (W, 6)
                Ec += 0.5*torch.einsum("wi,ij,wj->w", T, self._M[k], T)
                H = w.body("pose", k + 1)                        # (W, 4, 4)
                h = torch.einsum("wij,j->wi", H, self._com[k])[:, :3] @ self._up
                Ep += self._M[k][3, 3]*h
            Ep *= 9.81
        else:
            for k in sorted(set(self._bodies) | {b - 1 for b in bound}):
                if k + 1 in bound:                               # (W, 6, 6): the world's own M_b
                    M = massmatrix.from_params(w.body_inertia[bound.index(k + 1)].T)
                    m = M[:, 3, 3]
                    com = torch.stack((M[:, 2, 4], M[:, 0, 5], M[:, 1, 3]), 1)
                    com = torch.where((m > 0)[:, None], com/torch.where(m > 0, m, 1.)[:, None], 0.)
                    com = torch.cat((com, torch.ones_like(m)[:, None]), 1)
                else:
                    M = self._M[k].expand(w.nworlds, 6, 6)
                    m = M[:, 3, 3]
                    com = self._com[k].expand(w.nworlds, 4)
                T = w.body("twist", k + 1)
                Ec += 0.5*torch.einsum("wi,wij,wj->w", T, M, T)
                p = torch.einsum("wij,wj->wi", w.body("pose", k + 1), com)[:, :3]
                if g is None:
                    Ep += 9.81*m*(p @ self._up)
                else:
                    Ep -= m*(p*g.T).sum(1)
        self.kinetic_energy.append(Ec)
        self.potential_energy.append(Ep)
        self.mechanichal_energy.append(Ec + Ep)

    def finish(self):
        for name in ("kinetic_energy", "potential_energy", "mechanichal_energy"):
            v = getattr(self, name)
            setattr(self, name, torch.stack(v).cpu().numpy() if v else np.zeros((0, self._world.nworlds)))
