"""ctypes binding of the C ABI declared in ``include/arboris_b200.h``.

Loads ``lib/libarboris_b200.so`` (built in-tree by ``__graft_entry__.build()``)
and declares every exported entry point.  There is no fallback: if the library
is missing or the CUDA device is unusable, importing the step raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# ARB_B200_LIB selects another build of the same library (A/B runs of kernel variants)
LIB_PATH = os.environ.get("ARB_B200_LIB") or os.path.join(_HERE, "lib", "libarboris_b200.so")

c_i32p = C.POINTER(C.c_int32)
c_dblp = C.POINTER(C.c_double)


class ModelDesc(C.Structure):
    """``arb_model_desc``"""
    _fields_ = [
        ("ndof", C.c_int32), ("ngpos", C.c_int32), ("njoints", C.c_int32),
        ("nconstraints", C.c_int32), ("ncontrollers", C.c_int32),
        ("nrows", C.c_int32), ("nblob", C.c_int32),
        ("joint_type", c_i32p), ("joint_parent", c_i32p), ("joint_dof", c_i32p),
        ("joint_gpos", c_i32p),
        ("joint_Hpr", c_dblp), ("joint_Hcn", c_dblp),
        ("body_mass", c_dblp), ("body_visc", c_dblp),
        ("cons_type", c_i32p), ("cons_int", c_i32p), ("cons_dbl", c_dblp),
        ("cons_row", c_i32p),
        ("ctrl_type", c_i32p), ("ctrl_int", c_i32p), ("ctrl_dbl", c_dblp),
        ("ctrl_blob", c_dblp),
        ("up", C.c_double*3),
    ]


def make_desc(model):
    """Build an ``arb_model_desc`` from a ``FlatModel``.  Returns (desc, keep):
    ``keep`` holds the numpy arrays the pointers refer to."""
    keep = []

    def ip(a):
        a = np.ascontiguousarray(a, dtype=np.int32).reshape(-1)
        if a.size == 0:
            a = np.zeros(1, np.int32)
        keep.append(a)
        return a.ctypes.data_as(c_i32p)

    def dp(a):
        a = np.ascontiguousarray(a, dtype=np.float64).reshape(-1)
        if a.size == 0:
            a = np.zeros(1, np.float64)
        keep.append(a)
        return a.ctypes.data_as(c_dblp)

    d = ModelDesc()
    d.ndof, d.ngpos, d.njoints = int(model.ndof), int(model.ngpos), len(model.joint_type)
    d.nconstraints, d.ncontrollers = len(model.cons_type), len(model.ctrl_type)
    d.nrows, d.nblob = int(model.nrows), int(np.asarray(model.ctrl_blob).size)
    d.joint_type, d.joint_parent = ip(model.joint_type), ip(model.joint_parent)
    d.joint_dof, d.joint_gpos = ip(model.joint_dof), ip(model.joint_gpos)
    d.joint_Hpr, d.joint_Hcn = dp(model.joint_Hpr), dp(model.joint_Hcn)
    d.body_mass, d.body_visc = dp(model.body_mass), dp(model.body_visc)
    d.cons_type, d.cons_int = ip(model.cons_type), ip(model.cons_int)
    d.cons_dbl, d.cons_row = dp(model.cons_dbl), ip(model.cons_row)
    d.ctrl_type, d.ctrl_int = ip(model.ctrl_type), ip(model.ctrl_int)
    d.ctrl_dbl, d.ctrl_blob = dp(model.ctrl_dbl), dp(model.ctrl_blob)
    for i in range(3):
        d.up[i] = float(model.up[i])
    return d, keep


# (name, restype, argtypes) of every symbol include/arboris_b200.h declares
_vp, _i64, _i32, _dbl = C.c_void_p, C.c_int64, C.c_int, C.c_double
SYMBOLS = [
    ("arb_last_error", C.c_char_p, []),
    ("arb_version", _i32, []),
    ("arb_model_create", _i32, [C.POINTER(ModelDesc), C.POINTER(_vp)]),
    ("arb_model_destroy", None, [_vp]),
    ("arb_batch_create", _i32, [_vp, _i64, _i32, _vp, C.POINTER(_vp)]),
    ("arb_batch_destroy", None, [_vp]),
    ("arb_batch_set_stream", _i32, [_vp, _vp]),
    ("arb_batch_set_option", _i32, [_vp, C.c_char_p, _i32]),
    ("arb_batch_bind_state", _i32, [_vp, _vp, _vp, _vp]),
    ("arb_batch_bind_controller_params", _i32, [_vp, _vp, _vp, _vp, _vp]),
    ("arb_model_pd_dofs", _i32, [_vp, c_i32p, _i32]),
    ("arb_batch_bind_applied_forces", _i32, [_vp, _vp, _i32, c_i32p, _vp]),
    ("arb_batch_bind_body_inertia", _i32, [_vp, _i32, c_i32p, _vp]),
    ("arb_batch_bind_gravity", _i32, [_vp, _vp]),
    ("arb_batch_bind_contact_friction", _i32, [_vp, _i32, c_i32p, _vp]),
    ("arb_batch_step_path", _i32, [_vp, C.POINTER(C.c_char_p)]),
    ("arb_update_dynamic", _i32, [_vp]),
    ("arb_update_controllers", _i32, [_vp, _dbl]),
    ("arb_update_constraints", _i32, [_vp, _dbl]),
    ("arb_integrate", _i32, [_vp, _dbl]),
    ("arb_step", _i32, [_vp, c_dblp, _i32]),
    ("arb_step_begin", _i32, [_vp, _dbl]),
    ("arb_step_end", _i32, [_vp, _dbl]),
    ("arb_step_host", _i32, [_vp, _vp, _vp, _vp, c_dblp, _i32]),
    ("arb_step_host_strided", _i32, [_vp, _vp, _vp, _vp, _i64, c_dblp, _i32, _i32]),
    ("arb_batch_synchronize", _i32, [_vp]),
    ("arb_state_copy_host_strided", _i32, [_vp, _vp, _vp, _vp, _i64, _i32, _vp]),
    ("arb_get_matrix", _i32, [_vp, _i32, _vp, _i64, _i64]),
    ("arb_get_vector", _i32, [_vp, _i32, _vp, _i64, _i64]),
    ("arb_get_body", _i32, [_vp, _i32, _i32, _vp, _i64, _i64]),
    ("arb_get_constraint", _i32, [_vp, _i32, _vp, _i64, _i64]),
    ("arb_get_fused", _i32, [_vp, _i32, _vp, _i64, _i64]),
    ("arb_model_generators", _i32, [_vp, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p, c_i32p]),
    ("arb_batch_status", _i32, [_vp, _vp]),
    ("arb_batch_launch_count", _i64, [_vp]),
    ("arb_batch_stage_ms", _i32, [_vp, c_dblp]),
    ("arb_measure_fp64_peak", _i32, [_i32, c_dblp]),
]

_lib = None


def load(path=None):
    """Load the shared library and attach prototypes (raises if it is missing)."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.isfile(p):
        raise ImportError(
            "CUDA library %s not found: run `python -c 'import __graft_entry__ as g; "
            "g.build()'` (there is no CPU fallback for the simulation step)" % p)
    lib = C.CDLL(p)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if path is None:
        _lib = lib
    return lib


class ArbError(RuntimeError):
    pass


def check(lib, rc):
    if rc != 0:
        msg = lib.arb_last_error()
        raise ArbError("arboris_b200 error %d: %s" % (rc, (msg or b"").decode()))
