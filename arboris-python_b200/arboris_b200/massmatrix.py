"""Host-side 6x6 spatial mass matrices for model building.

Same public names as the reference ``arboris/massmatrix.py`` (``transport`` :27,
``box`` :103, ``ellipsoid`` :124, ``cylinder`` :146, ``sphere`` :165).  Runs once
per model on the host; its outputs (body mass matrices) are constants of the
flattened model the CUDA kernels consume.  Twist/wrench order is [angular; linear].
"""
import numpy as np
from . import homogeneousmatrix as Hg


def ismassmatrix(M, semi=False):
    M = np.asarray(M)
    ok = (M.shape == (6, 6) and np.allclose(M, M.T)
          and np.allclose(M[3:, 3:], M[3, 3]*np.eye(3)))
    if not ok:
        return False
    ev = np.linalg.eigvalsh((M + M.T)/2)
    return bool((ev >= 0.).all() if semi else (ev > 0.).all())


def transport(M, H):
    """Express mass matrix ``M`` (frame a) in frame b, ``H = H_ab``."""
    assert ismassmatrix(M)
    Ad = Hg.adjoint(H)
    return Ad.T.dot(np.asarray(M).dot(Ad))


def _diag_inertia(ix, iy, iz, mass):
    return np.diag((ix, iy, iz, mass, mass, mass)).astype(float)


def box(half_extents, mass):
    x, y, z = half_extents
    k = mass/3.
    return _diag_inertia(k*(y**2 + z**2), k*(x**2 + z**2), k*(x**2 + y**2), mass)


def ellipsoid(radii, mass):
    x, y, z = radii
    k = mass/5.
    return _diag_inertia(k*(y**2 + z**2), k*(x**2 + z**2), k*(x**2 + y**2), mass)


def cylinder(length, radius, mass):
    """Homogeneous cylinder, symmetry axis along z."""
    itan = mass*(radius**2/4. + length**2/12.)
    return _diag_inertia(itan, itan, mass*radius**2/2., mass)


def sphere(radius, mass):
    i = 2.*mass*radius**2/5.
    return _diag_inertia(i, i, i, mass)


def to_params(M):
    """The 10 independent entries ``[m, m c_x, m c_y, m c_z, I_xx, I_yy, I_zz, I_xy, I_xz, I_yz]`` of
    rigid-body mass matrices ``M`` (..., 6, 6), [angular; linear] order: ``m = M[3,3]``, ``m c`` from
    ``M[0:3,3:6] = skew(m c)``, ``I = M[0:3,0:3]``.  The input of ``BatchedWorld.set_body_inertia``;
    vectorised over the leading axes.  ``from_params(to_params(M)) == M`` for matrices of that form."""
    M = np.asarray(M, dtype=float)
    return np.stack((M[..., 3, 3], M[..., 2, 4], M[..., 0, 5], M[..., 1, 3],
                     M[..., 0, 0], M[..., 1, 1], M[..., 2, 2], M[..., 0, 1], M[..., 0, 2], M[..., 1, 2]), -1)


# M.flat[i] = PARAM_SIGN[i] * [p, 0][PARAM_INDEX[i]]: placement and sign of the 10 parameters
PARAM_INDEX = np.array([4, 7, 8, 10, 3, 2,
                        7, 5, 9, 3, 10, 1,
                        8, 9, 6, 2, 1, 10,
                        10, 3, 2, 0, 10, 10,
                        3, 10, 1, 10, 0, 10,
                        2, 1, 10, 10, 10, 0])
PARAM_SIGN = np.array([1., 1., 1., 1., -1., 1.,
                       1., 1., 1., 1., 1., -1.,
                       1., 1., 1., -1., 1., 1.,
                       1., 1., -1., 1., 1., 1.,
                       -1., 1., 1., 1., 1., 1.,
                       1., -1., 1., 1., 1., 1.])


def from_params(p):
    """Mass matrices (..., 6, 6) of parameters ``p`` (..., 10) (``to_params``):
    ``[[I, skew(m c)], [skew(m c)^T, m 1]]``, placement and sign only, as the step assembles them.
    Numpy arrays or torch tensors."""
    if isinstance(p, np.ndarray) or not hasattr(p, "new_zeros"):
        p = np.asarray(p, dtype=float)
        q = np.concatenate((p, np.zeros(p.shape[:-1] + (1,))), -1)
        return (q[..., PARAM_INDEX]*PARAM_SIGN).reshape(p.shape[:-1] + (6, 6))
    import torch
    q = torch.cat((p, p.new_zeros(p.shape[:-1] + (1,))), -1)
    idx = torch.as_tensor(PARAM_INDEX, device=p.device)
    return (q[..., idx]*torch.as_tensor(PARAM_SIGN, dtype=p.dtype, device=p.device)).reshape(p.shape[:-1] + (6, 6))
