"""``BatchedWorld``: W independent worlds of one model stepping in lockstep on a GPU.

It exposes the reference's step API (``update_dynamic``, ``update_controllers``,
``update_constraints``, ``integrate``, and ``simulate()`` via
``arboris_b200.core.simulate``; reference core.py:682-980, 1334-1365) over
batched state, plus the fused ``step``.  PyTorch owns the device memory and the
stream; all arithmetic is in the CUDA library behind the C ABI
(``include/arboris_b200.h``), loaded with ctypes.  No CUDA library or no GPU ->
this module raises; there is no CPU path.

State tensors (fp64, device, world index fastest -- the layout the kernels
coalesce on):  ``gpos`` (ngpos, W), ``gvel`` (ndof, W), ``cforce`` (nrows, W).
"""
import ctypes as C

import numpy as np
import torch

from . import _capi
from .flatten import FlatModel, flatten, JOINT_NDOF, JOINT_NGPOS

MATRIX_IDS = {"mass": 0, "nleffects": 1, "viscosity": 2, "impedance": 3, "admittance": 4}
BODY_IDS = {"pose": (0, (4, 4)), "twist": (1, (6,)), "jacobian": (2, None),
            "djacobian": (3, None), "nleffects": (4, (6, 6))}


class BatchedWorld(object):
    def __init__(self, world_or_model, nworlds=1, device=None, stream=None):
        if isinstance(world_or_model, FlatModel):
            self.world, self.model = None, world_or_model
        else:
            self.world = world_or_model
            if hasattr(world_or_model, "init") and getattr(world_or_model, "_ndof", 0) == 0:
                world_or_model.init()
            self.model = flatten(world_or_model)
        if not torch.cuda.is_available():
            raise RuntimeError("arboris_b200 needs a CUDA device: the simulation step has no CPU path")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None \
            else torch.device(device)
        self.nworlds = int(nworlds)
        self._lib = _capi.load()
        m = self.model
        self._desc, self._keep = _capi.make_desc(m)
        h = C.c_void_p()
        _capi.check(self._lib, self._lib.arb_model_create(C.byref(self._desc), C.byref(h)))
        self._model_h = h
        self._stream = stream
        with torch.cuda.device(self.device):
            s = torch.cuda.current_stream(self.device) if stream is None else stream
            b = C.c_void_p()
            _capi.check(self._lib, self._lib.arb_batch_create(
                self._model_h, self.nworlds, self.device.index or 0,
                C.c_void_p(s.cuda_stream), C.byref(b)))
        self._batch_h = b
        W = self.nworlds
        kw = dict(dtype=torch.float64, device=self.device)
        self.gpos = torch.empty((m.ngpos, W), **kw)
        self.gvel = torch.empty((m.ndof, W), **kw)
        self.cforce = torch.zeros((max(int(m.nrows), 1), W), **kw)
        self._bind()
        self.set_state(np.repeat(np.asarray(m.gpos0)[:, None], W, 1),
                       np.repeat(np.asarray(m.gvel0)[:, None], W, 1),
                       np.repeat(np.asarray(m.cforce0)[:, None], W, 1) if m.nrows else None)
        self._current_time = 0.
        self._pinned = None
        self._ctrl_params = {}
        self.applied_gforce = self.applied_wrench = None
        self.applied_bodies = ()
        why = C.c_char_p()
        if self._lib.arb_batch_step_path(self._batch_h, C.byref(why)) == 0:
            # not silent: the fused stages fold controllers per dof; anything else runs the
            # (much slower) phase kernels
            import warnings
            warnings.warn("arboris_b200: step() runs the four phase kernels for this model, not the "
                          "fused stages (%s)" % (why.value or b"").decode(), RuntimeWarning, stacklevel=2)

    # ---- plumbing -----------------------------------------------------------------
    def _bind(self):
        _capi.check(self._lib, self._lib.arb_batch_bind_state(
            self._batch_h, self.gpos.data_ptr(), self.gvel.data_ptr(), self.cforce.data_ptr()))

    def _sync_stream(self):
        s = torch.cuda.current_stream(self.device) if self._stream is None else self._stream
        self._lib.arb_batch_set_stream(self._batch_h, C.c_void_p(s.cuda_stream))

    def set_option(self, name, value):
        """``force_phases`` / ``time_stages`` switches of ``arb_batch_set_option``."""
        _capi.check(self._lib, self._lib.arb_batch_set_option(
            self._batch_h, name.encode(), int(value)))

    def close(self):
        if getattr(self, "_batch_h", None):
            self._lib.arb_batch_destroy(self._batch_h)
            self._batch_h = None
        if getattr(self, "_model_h", None):
            self._lib.arb_model_destroy(self._model_h)
            self._model_h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    ndof = property(lambda self: int(self.model.ndof))
    current_time = property(lambda self: self._current_time)

    def init(self):
        """``World.init()`` of the batched world: the model is already flat."""

    # ---- state ----------------------------------------------------------------------
    def set_state(self, gpos=None, gvel=None, cforce=None):
        """Upload state given as (elem, W) arrays (numpy or torch)."""
        for dst, src in ((self.gpos, gpos), (self.gvel, gvel), (self.cforce, cforce)):
            if src is None:
                continue
            t = torch.as_tensor(np.ascontiguousarray(src) if isinstance(src, np.ndarray) else src,
                                dtype=torch.float64)
            if t.numel() == 0:
                continue
            dst[:t.shape[0]].copy_(t.reshape(t.shape[0], -1), non_blocking=False)

    def get_state(self):
        return self.gpos.cpu().numpy(), self.gvel.cpu().numpy(), \
            self.cforce[:int(self.model.nrows)].cpu().numpy()

    # ---- per-world controller parameters -------------------------------------------------------
    def pd_dofs(self):
        """dof of each row of the per-world PD parameter arrays (controllers in registration
        order, each controller's dofs in its own order)."""
        n = self._lib.arb_model_pd_dofs(self._model_h, None, 0)
        out = (C.c_int32*max(n, 1))()
        self._lib.arb_model_pd_dofs(self._model_h, out, n)
        return [int(out[i]) for i in range(n)]

    def set_controller_params(self, kp=None, kd=None, gpos_des=None, gvel_des=None):
        """Per-world ``kp``, ``kd`` (diagonal gains), ``gpos_des``, ``gvel_des`` of the
        ProportionalDerivativeControllers (reference controllers.py:63-159, one value per
        controller object there): arrays (npd, W), rows as ``pd_dofs()``.  ``None`` keeps what was
        bound before for that parameter; ``False`` goes back to the model's value."""
        npd = len(self.pd_dofs())
        for name, v in (("kp", kp), ("kd", kd), ("gpos_des", gpos_des), ("gvel_des", gvel_des)):
            if v is None:
                continue
            if v is False:
                self._ctrl_params.pop(name, None)
                continue
            t = torch.as_tensor(np.ascontiguousarray(v) if isinstance(v, np.ndarray) else v,
                                dtype=torch.float64).to(self.device).contiguous()
            if tuple(t.shape) != (npd, self.nworlds):
                raise ValueError("%s must have shape (%d, %d)" % (name, npd, self.nworlds))
            self._ctrl_params[name] = t
        ptr = [self._ctrl_params[k].data_ptr() if k in self._ctrl_params else None
               for k in ("kp", "kd", "gpos_des", "gvel_des")]
        _capi.check(self._lib, self._lib.arb_batch_bind_controller_params(self._batch_h, *ptr))

    # ---- per-world applied forces --------------------------------------------------------------
    def set_applied_forces(self, gforce=None, wrench=None, bodies=None):
        """Per-world forces of a controller added after the model's ones (what a reference
        ``Controller`` whose ``update`` returns ``(gforce, 0)`` adds):

        ``gforce``: (ndof, W) generalized forces;  ``wrench``: (len(bodies), 6, W) wrenches
        [torque; force] in ground axes acting at the origin of body ``bodies[i]`` (indices as in
        ``body()``, the ground excluded).  Numpy or torch; ``None`` keeps what is bound (``bodies``
        too), ``False`` unbinds (a wrench and its bodies together).  The bound fp64 device tensors
        are ``applied_gforce`` and ``applied_wrench`` (the argument itself when it already is one):
        write into them in place to change the forces between steps without another call."""
        W = self.nworlds

        def dev(v, shape, name):
            t = torch.as_tensor(np.ascontiguousarray(v) if isinstance(v, np.ndarray) else v,
                                dtype=torch.float64).to(self.device).contiguous()
            if tuple(t.shape) != shape:
                raise ValueError("%s must have shape %s, not %s" % (name, shape, tuple(t.shape)))
            return t

        g, wr, bd = self.applied_gforce, self.applied_wrench, self.applied_bodies
        if gforce is False:
            g = None
        elif gforce is not None:
            g = dev(gforce, (self.ndof, W), "gforce")
        if wrench is False:
            wr, bd = None, ()
        else:
            if bodies is not None:
                bd = tuple(int(b) for b in np.asarray(bodies).reshape(-1))
            if wrench is not None:
                wr = dev(wrench, (len(bd), 6, W), "wrench")
            elif wr is not None and tuple(wr.shape) != (len(bd), 6, W):
                raise ValueError("the bound wrench has %d bodies, not %d: pass the wrench with its bodies"
                                 % (wr.shape[0], len(bd)))
        ids = (C.c_int32*max(len(bd), 1))(*bd)
        self._sync_stream()         # (the body table is replaced in stream order)
        _capi.check(self._lib, self._lib.arb_batch_bind_applied_forces(
            self._batch_h, g.data_ptr() if g is not None else None, len(bd) if wr is not None else 0,
            ids, wr.data_ptr() if wr is not None else None))
        self.applied_gforce, self.applied_wrench = g, wr
        self.applied_bodies = bd if wr is not None else ()

    # ---- the four phases and the fused step ---------------------------------------------
    def update_dynamic(self):
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_update_dynamic(self._batch_h))

    def update_controllers(self, dt):
        assert dt > 0
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_update_controllers(self._batch_h, float(dt)))

    def update_constraints(self, dt):
        assert dt > 0
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_update_constraints(self._batch_h, float(dt)))

    def integrate(self, dt):
        assert dt > 0
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_integrate(self._batch_h, float(dt)))
        self._current_time += dt

    def step(self, dt, nsteps=1):
        """``nsteps`` iterations of the simulate() loop, fused on the device."""
        dts = np.full(nsteps, dt, dtype=np.float64) if np.isscalar(dt) else \
            np.ascontiguousarray(dt, dtype=np.float64)
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_step(
            self._batch_h, dts.ctypes.data_as(_capi.c_dblp), len(dts)))
        self._current_time += float(dts.sum())

    def begin_step(self, dt):
        """First half of one fused step: everything ``simulate()`` does before the observers
        run (update_dynamic, update_controllers, update_constraints; core.py:1357-1359).  The
        state is untouched; body poses / twists, active sets and constraint forces of this
        step can be read until ``end_step``."""
        assert dt > 0
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_step_begin(self._batch_h, float(dt)))

    def end_step(self, dt):
        """Second half: ``integrate(dt)`` (core.py:1362)."""
        assert dt > 0
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_step_end(self._batch_h, float(dt)))
        self._current_time += dt

    def step_host(self, gpos, gvel, cforce, dt, nsteps=1):
        """End-to-end call with HOST buffers (numpy (elem, W), updated in place):
        host->device copy of the state, ``nsteps`` steps, device->host copy."""
        dts = np.full(nsteps, dt, dtype=np.float64)
        self._sync_stream()
        cf = cforce.ctypes.data if cforce is not None and cforce.size else None
        _capi.check(self._lib, self._lib.arb_step_host(
            self._batch_h, gpos.ctypes.data, gvel.ctypes.data, cf,
            dts.ctypes.data_as(_capi.c_dblp), nsteps))
        self._current_time += float(dts.sum())

    def step_host_async(self, gpos, gvel, cforce, dt, nsteps=1):
        """Like ``step_host`` for column blocks of larger host arrays (numpy views
        ``big[:, w0:w1]`` of C-contiguous (elem, W_total) arrays, pinned for the copies to be
        asynchronous), without waiting: the copies and kernels are enqueued on this batch's
        stream.  ``synchronize()`` waits.  See ``HostPipeline``."""
        dts = np.full(nsteps, dt, dtype=np.float64)
        ld = gpos.strides[0]//8
        assert gpos.strides[1] == 8 and gvel.strides[1] == 8 and gvel.strides[0]//8 == ld
        self._sync_stream()
        cf = cforce.ctypes.data if cforce is not None and cforce.size else None
        if cf is not None:
            assert cforce.strides[0]//8 == ld
        _capi.check(self._lib, self._lib.arb_step_host_strided(
            self._batch_h, gpos.ctypes.data, gvel.ctypes.data, cf, ld,
            dts.ctypes.data_as(_capi.c_dblp), nsteps, 0))
        self._current_time += float(dts.sum())

    def synchronize(self):
        _capi.check(self._lib, self._lib.arb_batch_synchronize(self._batch_h))

    # ---- read-backs --------------------------------------------------------------------------
    def _range(self, w0, w1):
        w1 = self.nworlds if w1 is None else w1
        return int(w0), int(w1)

    def matrix(self, name, w0=0, w1=None):
        """(w1-w0, n, n) tensor of ``mass|nleffects|viscosity|impedance|admittance``."""
        w0, w1 = self._range(w0, w1)
        n = self.ndof
        out = torch.empty((w1 - w0, n, n), dtype=torch.float64, device=self.device)
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_get_matrix(
            self._batch_h, MATRIX_IDS[name], out.data_ptr(), w0, w1))
        return out

    mass = property(lambda self: self.matrix("mass"))
    nleffects = property(lambda self: self.matrix("nleffects"))
    viscosity = property(lambda self: self.matrix("viscosity"))
    impedance = property(lambda self: self.matrix("impedance"))
    admittance = property(lambda self: self.matrix("admittance"))

    def gforce(self, w0=0, w1=None):
        w0, w1 = self._range(w0, w1)
        out = torch.empty((w1 - w0, self.ndof), dtype=torch.float64, device=self.device)
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_get_vector(self._batch_h, 0, out.data_ptr(), w0, w1))
        return out

    def body(self, what, body, w0=0, w1=None):
        """``pose|twist|jacobian|djacobian|nleffects`` of body index ``body``
        (0 = ground) for worlds [w0, w1)."""
        w0, w1 = self._range(w0, w1)
        code, shape = BODY_IDS[what]
        if shape is None:
            shape = (6, self.ndof)
        out = torch.empty((w1 - w0,) + shape, dtype=torch.float64, device=self.device)
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_get_body(
            self._batch_h, code, int(body), out.data_ptr(), w0, w1))
        return out

    def constraints(self, what, w0=0, w1=None):
        """``active|branch`` (int32 (W, nc)), ``sdist`` (fp64 (W, nc)) or
        ``zidx`` (int32 (W, nc, 3))."""
        w0, w1 = self._range(w0, w1)
        nc = len(self.model.cons_type)
        code = {"active": 0, "branch": 1, "sdist": 2, "zidx": 3}[what]
        if what == "sdist":
            out = torch.zeros((w1 - w0, nc), dtype=torch.float64, device=self.device)
        elif what == "zidx":
            out = torch.zeros((w1 - w0, nc, 3), dtype=torch.int32, device=self.device)
        else:
            out = torch.zeros((w1 - w0, nc), dtype=torch.int32, device=self.device)
        if nc:
            self._sync_stream()
            _capi.check(self._lib, self._lib.arb_get_constraint(
                self._batch_h, code, out.data_ptr(), w0, w1))
        return out

    def status(self):
        """Per-world ARB_STATUS_* bits accumulated since the last call."""
        out = torch.zeros(self.nworlds, dtype=torch.int32, device=self.device)
        self._sync_stream()
        _capi.check(self._lib, self._lib.arb_batch_status(self._batch_h, out.data_ptr()))
        return out

    def stage_ms(self):
        """{prepare, gs, finish} device milliseconds accumulated since
        ``set_option("time_stages", 1)`` and the number of steps they cover."""
        out = (C.c_double*4)()
        _capi.check(self._lib, self._lib.arb_batch_stage_ms(self._batch_h, out))
        return {"prepare": out[0], "gs": out[1], "finish": out[2], "steps": int(out[3])}

    def launch_count(self):
        return int(self._lib.arb_batch_launch_count(self._batch_h))

    # ---- single-world synchronisation used by World.update_* ------------------------------
    def push_host_state(self, world):
        m = self.model
        gpos = np.zeros(m.ngpos)
        for k, j in enumerate(world.iterjoints()):
            v = np.asarray(j.gpos, dtype=float).reshape(-1)
            gpos[int(m.joint_gpos[k]):int(m.joint_gpos[k]) + v.size] = v
        cf = np.zeros(max(int(m.nrows), 1))
        for k, c in enumerate(world._constraints):
            f = np.asarray(c._force, dtype=float).reshape(-1)
            cf[int(m.cons_row[k]):int(m.cons_row[k]) + f.size] = f
        self.set_state(gpos[:, None], np.asarray(world._gvel, dtype=float)[:, None], cf[:, None])

    def pull_dynamic(self, world):
        world._mass[:] = self.matrix("mass")[0].cpu().numpy()
        world._nleffects[:] = self.matrix("nleffects")[0].cpu().numpy()
        world._viscosity[:] = self.matrix("viscosity")[0].cpu().numpy()
        for k, b in enumerate(world.iterbodies()):
            b._pose = self.body("pose", k)[0].cpu().numpy()
            b._twist = self.body("twist", k)[0].cpu().numpy()
            b._jacobian = self.body("jacobian", k)[0].cpu().numpy()
            b._djacobian = self.body("djacobian", k)[0].cpu().numpy()
            b._nleffects = self.body("nleffects", k)[0].cpu().numpy()

    def pull_controllers(self, world):
        world._impedance = self.matrix("impedance")[0].cpu().numpy()
        world._admittance = self.matrix("admittance")[0].cpu().numpy()
        world._gforce[:] = self.gforce()[0].cpu().numpy()

    def pull_constraints(self, world):
        m = self.model
        world._gforce[:] = self.gforce()[0].cpu().numpy()
        cf = self.cforce[:, 0].cpu().numpy()
        act = self.constraints("active")[0].cpu().numpy()
        sd = self.constraints("sdist")[0].cpu().numpy()
        for k, c in enumerate(world._constraints):
            r0 = int(m.cons_row[k])
            c._force[:] = cf[r0:r0 + c._force.size]
            c._is_active = bool(act[k])
            if hasattr(c, "_sdist"):
                c._sdist = float(sd[k])

    def pull_state(self, world):
        m = self.model
        gpos = self.gpos[:, 0].cpu().numpy()
        world._gvel[:] = self.gvel[:, 0].cpu().numpy()
        for k, j in enumerate(world.iterjoints()):
            g = int(m.joint_gpos[k])
            t = int(m.joint_type[k])
            if t == 0:
                j.gpos = gpos[g:g + 16].reshape(4, 4).copy()
            else:
                j.gpos[:] = gpos[g:g + JOINT_NDOF[t]]


class HostPipeline(object):
    """End-to-end stepping of HOST state: the worlds are split into ``chunks`` column blocks, each
    with its own ``BatchedWorld``, so that the host->device copy of one block, the kernels of
    another and the device->host copy of a third overlap (PCIe is full duplex; the step of 262144
    human36 worlds and the two 268 MB copies take about as long).
    ``gpos``, ``gvel``, ``cforce`` are C-contiguous (elem, W) numpy arrays over PINNED memory
    (e.g. ``torch.empty(...).pin_memory().numpy()``), updated in place."""

    def __init__(self, world_or_model, nworlds, chunks="auto", device=None, mode="serial",
                 compute_streams="priority"):
        """``chunks``: number of equal column blocks or their relative sizes (``shard.block_ranges``).
        ``mode="serial"`` (default): the kernels of ALL blocks on ``compute_streams`` streams (see below), block
        after block, the copies on two more streams ordered by events -- few kernels on the GPU at a
        time (kernels of different stages sharing an SM lose a fifth of their throughput once the
        worlds are sorted); with one compute stream every block and stage ends in a partial wave of
        CTAs that nothing fills, two or three streams measured best (profiles/README.md).
        ``mode="streams"``: one stream per block (copies and kernels of a block in order on it,
        ``arb_step_host_strided``)."""
        from .shard import block_ranges
        assert mode in ("streams", "serial")
        self.mode = mode
        self.nworlds = int(nworlds)
        if chunks == "auto":
            chunks = self.auto_chunks(self.nworlds)
        self.chunks = chunks
        self.ranges = block_ranges(self.nworlds, chunks)
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        serial = mode == "serial"
        # compute streams of the serial mode: "priority" (default) = one stream per block, earlier blocks
        # at higher priority, so that the blocks run nearly in order and the tail of a block's kernels
        # is filled by the next block's (end to end +1.7 %, queued calls +4 % against three plain streams,
        # profiles/README.md); an integer = that many plain streams, blocks assigned round robin
        if serial and compute_streams == "priority":
            ncs = len(self.ranges)
            lo, hi = -5, 0            # (cudaDeviceGetStreamPriorityRange on B200: greatest -5, least 0)
            self._css = [torch.cuda.Stream(dev, priority=max(lo, min(hi, -(ncs - 1 - i)))) for i in range(ncs)]
        elif serial:
            ncs = max(1, int(compute_streams))
            self._css = [torch.cuda.Stream(dev) for _ in range(ncs)]
        else:
            self._css = None
        self._hs = torch.cuda.Stream(dev) if serial else None            # host -> device copies
        self._ds = torch.cuda.Stream(dev) if serial else None            # device -> host copies
        first = BatchedWorld(world_or_model, self.ranges[0][1] - self.ranges[0][0], device=dev,
                             stream=self._css[0] if serial else torch.cuda.Stream(dev))
        self.model = first.model
        self.parts = [first] + [BatchedWorld(self.model, w1 - w0, device=dev,
                                             stream=self._css[(i + 1) % len(self._css)] if serial
                                             else torch.cuda.Stream(dev))
                                for i, (w0, w1) in enumerate(self.ranges[1:])]
        self._ev = [(torch.cuda.Event(), torch.cuda.Event()) for _ in self.parts] if serial else None
        self._ed = [torch.cuda.Event() for _ in self.parts] if serial else None     # copy-out of a block done
        torch.cuda.synchronize(dev)      # construction ran on the default stream

    @staticmethod
    def auto_chunks(nworlds):
        """Column blocks by batch size: a block should still fill the GPU (148 SMs x 256 resident
        worlds = 37888), so small batches are not split -- 32768 worlds per GPU (262144 over 8 GPUs)
        go through as ONE block (copy in, step, copy out: 3.7 ms instead of 8.1 ms in seven slivers),
        mid-sized ones as 1:2:1, large ones as the measured best 1:1:2:2:2:1:1."""
        if nworlds < 49152:
            return 1
        if nworlds < 163840:
            return (1, 2, 1)
        return (1, 1, 2, 2, 2, 1, 1)

    def set_option(self, name, value):
        for p in self.parts:
            p.set_option(name, value)

    def _copy(self, p, gpos, gvel, cforce, w0, w1, to_device, stream):
        ld = gpos.strides[0]//8
        assert gpos.strides[1] == 8 and gvel.strides[1] == 8 and gvel.strides[0]//8 == ld
        g, v = gpos[:, w0:w1], gvel[:, w0:w1]
        cf = None
        if cforce is not None and cforce.size:
            assert cforce.strides[0]//8 == ld
            cf = cforce[:, w0:w1].ctypes.data
        _capi.check(p._lib, p._lib.arb_state_copy_host_strided(
            p._batch_h, g.ctypes.data, v.ctypes.data, cf, ld, 1 if to_device else 0,
            C.c_void_p(stream.cuda_stream)))

    def _step_serial(self, gpos, gvel, cforce, dt, nsteps, sync=True):
        for (w0, w1), p, (eh, ec), ed in zip(self.ranges, self.parts, self._ev, self._ed):
            # (a block's copy-in waits for the copy-out of its previous call: the host arrays are
            # updated in place, and calls may be queued without waiting, see step)
            self._hs.wait_event(ed)
            self._copy(p, gpos, gvel, cforce, w0, w1, True, self._hs)
            eh.record(self._hs)
        for (w0, w1), p, (eh, ec), ed in zip(self.ranges, self.parts, self._ev, self._ed):
            p._stream.wait_event(eh)
            p.step(dt, nsteps)
            ec.record(p._stream)
            self._ds.wait_event(ec)
            self._copy(p, gpos, gvel, cforce, w0, w1, False, self._ds)
            ed.record(self._ds)
        if sync:
            self._ds.synchronize()

    def wait(self):
        """Block until every queued call has delivered its results to the host arrays."""
        if self.mode == "serial":
            self._ds.synchronize()
        else:
            for p in self.parts:
                p.synchronize()

    def step(self, gpos, gvel, cforce, dt, nsteps=1, sync=True):
        """Host arrays in, ``nsteps`` steps, host arrays out (in place).  ``sync=False`` (serial mode)
        queues the call and returns: the next call's copies of a block start as soon as that block's
        results of this call are on the host, while the later blocks of this call still compute --
        no idle GPU between calls.  The host arrays must not be touched until ``wait()``."""
        if self.mode == "serial":
            return self._step_serial(gpos, gvel, cforce, dt, nsteps, sync)
        for (w0, w1), p in zip(self.ranges, self.parts):
            p.step_host_async(gpos[:, w0:w1], gvel[:, w0:w1],
                              cforce[:, w0:w1] if cforce is not None and cforce.size else None, dt, nsteps)
        for p in self.parts:
            p.synchronize()

    def launch_count(self):
        return sum(p.launch_count() for p in self.parts)

    def close(self):
        for p in self.parts:
            p.close()
