"""
ORACLE -- TEST INFRASTRUCTURE ONLY.  PARITY UNPINNED.

CPU restatement of the algorithm behind gadfly's GP hot path.  The arithmetic
lives in celerite2 (external, un-pinned dependency of the reference,
pyproject.toml:20; not installable here), so this package restates celerite2's
published algorithm (SURVEY.md Appendix A) and is validated against dense
``numpy.linalg.cholesky`` on the kernel *definition* (``tests/test_oracle.py``).
The reference's own tests hold no golden vectors for this path (only the
statistical round trip gadfly/tests/test_core.py:17-49, which is reproduced in
``tests/``), hence "parity unpinned": every "matches celerite2" claim means
"matches this validated restatement".

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` /
``--impl reference`` legs may import this package.  ``gadfly_b200`` never does.

Layout
------
``terms_oracle``      numpy: SHO -> (a,b,c,d), exposure-time transform, PSD, k(tau)  [A.3-A.5]
``celerite_oracle.c`` C:     row generation, factor, solve/matmul sweeps, fused streams [A.2, A.6]
``dense``             numpy: dense covariance + Cholesky ground truth
"""
import atexit
import ctypes
import hashlib
import os
import platform
import shutil
import subprocess
import tempfile

import numpy as np

from . import terms_oracle  # noqa: F401
from . import dense  # noqa: F401

_HERE = os.path.dirname(os.path.abspath(__file__))
_libs = {}

_dp = ctypes.POINTER(ctypes.c_double)
_lp = ctypes.POINTER(ctypes.c_long)


def _cpu_tag():
    model = platform.processor() or ""
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags"):
                    model += line
                    break
    except OSError:
        pass
    return hashlib.sha1(model.encode()).hexdigest()[:12]


def build(fast=False):
    """Compile the C oracle with gcc (per host CPU for the -march=native build) into
    ``oracle/_build``.  In a read-only tree without a current build there, compile into a new
    private temporary directory of this process (removed at exit), so that nothing is written
    into the tree and no build is shared with another process or checkout."""
    name = "liboracle_fast.so" if fast else "liboracle.so"
    out = os.path.join(_HERE, "_build", _cpu_tag() if fast else "generic")
    path = os.path.join(out, name)
    src = os.path.join(_HERE, "celerite_oracle.c")
    if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
        if not os.access(_HERE, os.W_OK):
            out = tempfile.mkdtemp(prefix="gadfly_b200_oracle_")
            atexit.register(shutil.rmtree, out, True)
            path = os.path.join(out, name)
        os.makedirs(out, exist_ok=True)
        subprocess.check_call(["make", "-s", "-C", _HERE, f"OUT={out}", path])
    return path


def lib(fast=False):
    if fast not in _libs:
        L = ctypes.CDLL(build(fast))
        L.orc_factor.restype = ctypes.c_long
        L.orc_stream.restype = ctypes.c_long
        L.orc_max_threads.restype = ctypes.c_int
        _libs[fast] = L
    return _libs[fast]


def _p(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


class LinAlgError(Exception):
    pass


def celerite_matrices(coeffs, t, diag=None, ddiag=0.0):
    """(c[J], a[N], U[N,J], V[N,J]) for coefficient tuple (ar,cr,ac,bc,cc,dc)  [A.2]."""
    ar, cr, ac, bc, cc, dc = [_f64(x) for x in coeffs]
    t = _f64(t)
    N, Jr, Jc = len(t), len(ar), len(ac)
    J = Jr + 2 * Jc
    c = np.empty(J)
    a = np.empty(N)
    U = np.empty((N, J))
    V = np.empty((N, J))
    dg = None if diag is None else _f64(np.broadcast_to(diag, (N,)))
    lib().orc_matrices(ctypes.c_long(N), Jr, Jc, _p(t), _p(dg), ctypes.c_double(ddiag),
                       _p(ar), _p(cr), _p(ac), _p(bc), _p(cc), _p(dc), _p(c), _p(a), _p(U), _p(V))
    return c, a, U, V


def factor(t, c, a, U, V):
    """-> (d[N], W[N,J]); raises LinAlgError at the first non-positive pivot  [A.6]."""
    t, c, a, U, V = map(_f64, (t, c, a, U, V))
    N, J = U.shape
    d = np.empty(N)
    W = np.empty((N, J))
    flag = lib().orc_factor(ctypes.c_long(N), J, _p(t), _p(c), _p(a), _p(U), _p(V), _p(d), _p(W))
    if flag:
        raise LinAlgError(f"failed to factorize; d[{flag - 1}] <= 0")
    return d, W


def _sweep(fn, t, c, U, W, Y):
    t, c, U, W = map(_f64, (t, c, U, W))
    Y = _f64(Y)
    vec = Y.ndim == 1
    Y2 = Y.reshape(len(t), -1)
    Z = np.empty_like(Y2)
    N, J = U.shape
    fn(ctypes.c_long(N), J, Y2.shape[1], _p(t), _p(c), _p(U), _p(W), _p(np.ascontiguousarray(Y2)), _p(Z))
    return Z[:, 0] if vec else Z


def solve_lower(t, c, U, W, Y):
    return _sweep(lib().orc_solve_lower, t, c, U, W, Y)


def matmul_lower(t, c, U, W, Y):
    return _sweep(lib().orc_matmul_lower, t, c, U, W, Y)


def solve_upper(t, c, U, W, Y):
    return _sweep(lib().orc_solve_upper, t, c, U, W, Y)


def matmul_upper(t, c, U, W, Y):
    return _sweep(lib().orc_matmul_upper, t, c, U, W, Y)


class OracleGP:
    """celerite2.GaussianProcess restated on the functions above (reference call sites
    gadfly/gp.py:59,202,327,350,370,391).  ``kernel`` is anything with
    ``scan_coefficients() -> (ar,cr,ac,bc,cc,dc,ddiag)``-like data passed as a tuple."""

    def __init__(self, scan_coeffs, t, diag=None, mean=0.0):
        *coeffs, ddiag = scan_coeffs
        self.t = _f64(t)
        self.mean = mean
        self.c, self.a, self.U, self.V = celerite_matrices(coeffs, self.t, diag, ddiag)
        self.d, self.W = factor(self.t, self.c, self.a, self.U, self.V)
        self.log_det = float(np.sum(np.log(self.d)))
        self.norm = -0.5 * (self.log_det + len(self.t) * np.log(2 * np.pi))

    def log_likelihood(self, y):
        z = solve_lower(self.t, self.c, self.U, self.W, _f64(y) - self.mean)
        return float(self.norm - 0.5 * np.sum(z * z / self.d))

    def dot_tril(self, y):
        y = _f64(y)
        z = y * (np.sqrt(self.d) if y.ndim == 1 else np.sqrt(self.d)[:, None])
        return matmul_lower(self.t, self.c, self.U, self.W, z)

    def apply_inverse(self, y):
        y = _f64(y)
        z = solve_lower(self.t, self.c, self.U, self.W, y)
        z = z / (self.d if y.ndim == 1 else self.d[:, None])
        return solve_upper(self.t, self.c, self.U, self.W, z)

    def sample_from_normals(self, n, include_mean=True):
        """celerite2 ``sample`` given the N(0,1) draws it would have made
        (``dot_tril(n).T + mean``), then gadfly's mean subtraction (gadfly/gp.py:391-392)."""
        x = self.dot_tril(n).T
        if include_mean:
            x = x + self.mean
        return x - x.mean(axis=0 if x.ndim == 2 else None)


def stream(mode, scan_coeffs, t, y, diag=None, fast=False):
    """Fused streaming pass (nothing materialised).  mode 0 -> (logdet, quad, status);
    mode 1 -> (x, logdet, status)."""
    ar, cr, ac, bc, cc, dc, ddiag = scan_coeffs
    ar, cr, ac, bc, cc, dc = [_f64(v) for v in (ar, cr, ac, bc, cc, dc)]
    t, y = _f64(t), _f64(y)
    N = len(t)
    out = np.zeros(2)
    x = np.empty(N) if mode == 1 else None
    dg = None if diag is None else _f64(np.broadcast_to(diag, (N,)))
    flag = lib(fast).orc_stream(mode, ctypes.c_long(N), len(ar), len(ac), _p(t), _p(y), _p(dg),
                                ctypes.c_double(ddiag), _p(ar), _p(cr), _p(ac), _p(bc), _p(cc),
                                _p(dc), _p(out), _p(x))
    if mode == 0:
        return out[0], out[1], int(flag)
    return x, out[0], int(flag)


def log_likelihood_from_stream(logdet, quad, N):
    return -0.5 * quad - 0.5 * logdet - 0.5 * N * np.log(2 * np.pi)


def stream_batch(mode, n_off, t_off, j_off, t, y, ddiag, ac, bc, cc, dc, nthreads=0, fast=True):
    """Batched fused passes, one sequence per host thread (the timed CPU baseline)."""
    n_off = np.ascontiguousarray(n_off, dtype=np.int64)
    t_off = np.ascontiguousarray(t_off, dtype=np.int64)
    j_off = np.ascontiguousarray(j_off, dtype=np.int64)
    B = len(n_off) - 1
    t, y, ddiag, ac, bc, cc, dc = map(_f64, (t, y, ddiag, ac, bc, cc, dc))
    out = np.zeros((B, 2))
    status = np.zeros(B, dtype=np.int64)
    x = np.empty_like(y) if mode == 1 else None
    lib(fast).orc_stream_batch(mode, ctypes.c_long(B), n_off.ctypes.data_as(_lp),
                               t_off.ctypes.data_as(_lp), j_off.ctypes.data_as(_lp),
                               _p(t), _p(y), _p(ddiag), _p(ac), _p(bc), _p(cc), _p(dc),
                               _p(out), _p(x), status.ctypes.data_as(_lp), int(nthreads))
    return out, x, status


def max_threads():
    return int(lib(True).orc_max_threads())


def psd(base_coeffs, omega, delta=0.0):
    """Kernel PSD [A.5] on the un-convolved coefficients, times sinc^2(delta omega / 2)."""
    ar, cr, ac, bc, cc, dc = [_f64(v) for v in base_coeffs]
    omega = _f64(omega)
    out = np.empty_like(omega)
    lib().orc_psd(ctypes.c_long(omega.size), _p(omega), len(ar), len(ac), _p(ar), _p(cr), _p(ac),
                  _p(bc), _p(cc), _p(dc), ctypes.c_double(delta), _p(out))
    return out
