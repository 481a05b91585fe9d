"""TEST INFRASTRUCTURE ONLY: ctypes driver of the device unit harness (arb_devtest.cu).

Builds the harness with the package's nvcc flags (``__graft_entry__.NVCC_FLAGS``), plus optional
``-D`` defines for the variant builds, into ``tests/devtest/_build/`` (or a temporary directory when
the tree is read-only), and runs its kernels on torch CUDA tensors laid out element-major
``[elem][N]``, one problem per thread."""
import ctypes as C
import hashlib
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRC = os.path.join(HERE, "arb_devtest.cu")
CSRC = os.path.join(ROOT, "arboris-python_b200", "csrc")
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import __graft_entry__  # noqa: E402


def _outdir():
    d = os.path.join(HERE, "_build")
    try:
        os.makedirs(d, exist_ok=True)
        if os.access(d, os.W_OK):
            return d
    except OSError:
        pass
    d = os.path.join(tempfile.gettempdir(), "arb_devtest_%d" % os.getuid())
    os.makedirs(d, exist_ok=True)
    return d


def build(defines=()):
    """Compile the harness (``defines``: e.g. ``("ARB_LAGUERRE_FAST=0",)``); returns the library path."""
    defines = tuple(defines)
    tag = hashlib.sha1(" ".join(defines).encode()).hexdigest()[:10] if defines else "default"
    out = os.path.join(_outdir(), "libarb_devtest_%s.so" % tag)
    deps = [SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
    if os.path.isfile(out) and all(os.path.getmtime(out) >= os.path.getmtime(d) for d in deps):
        return out
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not os.path.isfile(nvcc):
        nvcc = "nvcc"
    tmp = out + ".%d.tmp" % os.getpid()
    subprocess.check_call([nvcc] + __graft_entry__.NVCC_FLAGS + ["-D" + d for d in defines] + ["-o", tmp, SRC],
                          cwd=HERE)
    os.replace(tmp, out)
    return out


class DevLib(object):
    """One build of the harness; every method takes numpy inputs shaped [N][...] (problem-major, the
    natural form of a bank) and returns numpy outputs [N][...]."""

    def __init__(self, defines=()):
        import torch
        self.torch = torch
        self.L = C.CDLL(build(defines))
        self.dev = torch.device("cuda:0")

    def _in(self, a, dtype=None):
        t = self.torch
        a = np.asarray(a, dtype=dtype or np.float64)
        n = a.shape[0]
        return t.from_numpy(np.ascontiguousarray(a.reshape(n, -1).T)).to(self.dev)

    def _out(self, n, k, dtype):
        return self.torch.zeros((k, n), dtype=dtype, device=self.dev)

    def _call(self, name, *args):
        ptrs = []
        for a in args:
            if hasattr(a, "data_ptr"):
                ptrs.append(C.c_void_p(a.data_ptr()))
            elif isinstance(a, float):
                ptrs.append(C.c_double(a))
            else:
                ptrs.append(C.c_int(int(a)))
        err = getattr(self.L, name)(*ptrs)
        assert err == 0, (name, err)
        self.torch.cuda.synchronize()

    @staticmethod
    def _np(t, *shape):
        a = t.cpu().numpy().T.copy()
        return a.reshape((a.shape[0],) + shape) if shape else a[:, 0]

    def softfinger_solve(self, v, A, P, sdist, mu, eps, dt, f0):
        t = self.torch
        n = len(v)
        f = self._in(f0)
        df = self._out(n, 4, t.float64)
        br, st = self._out(n, 1, t.int32), self._out(n, 1, t.int32)
        self._call("dt_softfinger_solve", n, self._in(v), self._in(A), self._in(P), self._in(sdist), self._in(mu),
                   self._in(eps), float(dt), f, df, br, st)
        return self._np(f, 4), self._np(df, 4), self._np(br), self._np(st)

    def softfinger_fused(self, mode, v, A, P, sdist, mu, eps3, dt, f0):
        """eps3: the one eps of the launch (3 doubles)."""
        t = self.torch
        n = len(v)
        sdist = np.asarray(sdist, np.float64)
        aux = np.stack([sdist, sdist/dt], axis=1)
        f = self._in(f0)
        df = self._out(n, 4, t.float64)
        br, st = self._out(n, 1, t.int32), self._out(n, 1, t.int32)
        e = t.tensor(np.asarray(eps3, np.float64), device=self.dev)
        self._call("dt_softfinger_fused", n, int(mode), self._in(v), self._in(A), self._in(P), self._in(aux),
                   self._in(mu), e, float(dt), f, df, br, st)
        return self._np(f, 4), self._np(df, 4), self._np(br), self._np(st)

    def sliding_root(self, A, alpha, mu, coop=0):
        t = self.torch
        n = len(A)
        s = self._out(n, 1, t.float64)
        found, ok = self._out(n, 1, t.int32), self._out(n, 1, t.int32)
        self._call("dt_sliding_root", n, int(coop), self._in(A), self._in(alpha), self._in(mu), s, found, ok)
        return self._np(s), self._np(found), self._np(ok)

    def poly6(self, p, x):
        t = self.torch
        n = len(p)
        o = [self._out(n, 1, t.int32), self._out(n, 1, t.float64), self._out(n, 1, t.int32),
             self._out(n, 1, t.int32), self._out(n, 1, t.float64), self._out(n, 1, t.int32)]
        self._call("dt_poly6", n, self._in(p), self._in(x), *o)
        return tuple(self._np(a) for a in o)    # fast_ok, fast_root, positive, slow_n, slow_root, certify

    def eig6(self, A):
        t = self.torch
        n = len(A)
        wr, wi, ok = self._out(n, 6, t.float64), self._out(n, 6, t.float64), self._out(n, 1, t.int32)
        self._call("dt_eig6", n, self._in(A), wr, wi, ok)
        return self._np(wr, 6), self._np(wi, 6), self._np(ok)

    def pinv(self, A):
        n, m = len(A), np.asarray(A).shape[1]
        out = self._out(n, m*m, self.torch.float64)
        self._call("dt_pinv", n, m, self._in(A), out)
        return self._np(out, m, m)

    def inv_cond4(self, A):
        n = len(A)
        out, cond = self._out(n, 16, self.torch.float64), self._out(n, 1, self.torch.float64)
        self._call("dt_inv_cond4", n, self._in(A), out, cond)
        return self._np(out, 4, 4), self._np(cond)

    def solve4(self, A, b):
        n = len(A)
        x, ok = self._out(n, 4, self.torch.float64), self._out(n, 1, self.torch.int32)
        self._call("dt_solve4", n, self._in(A), self._in(b), x, ok)
        return self._np(x, 4), self._np(ok)

    def se3_exp(self, tw):
        n = len(tw)
        out = self._out(n, 12, self.torch.float64)
        self._call("dt_se3_exp", n, self._in(tw), out)
        return self._np(out, 12)

    def zaligned(self, z):
        n = len(z)
        R, idx = self._out(n, 9, self.torch.float64), self._out(n, 3, self.torch.int32)
        self._call("dt_zaligned", n, self._in(z), R, idx)
        return self._np(R, 3, 3), self._np(idx, 3)

    def collide(self, pair, cd, H0, H1):
        t = self.torch
        n = len(pair)
        sd = self._out(n, 1, t.float64)
        c0, c1, zi = self._out(n, 12, t.float64), self._out(n, 12, t.float64), self._out(n, 3, t.int32)
        self._call("dt_collide", n, self._in(pair, np.int32), self._in(cd), self._in(H0), self._in(H1), sd, c0, c1, zi)
        return self._np(sd), self._np(c0, 12), self._np(c1, 12), self._np(zi, 3)
