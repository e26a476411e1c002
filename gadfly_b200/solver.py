"""
ctypes binding of ``libgadfly_b200.so`` -- the C ABI declared in
``include/gadfly_b200.h`` -- plus the batch descriptors the library consumes.

This module is the only place the Python facade touches the GPU.  There is no
CPU fallback: if the shared library is missing or no CUDA device is visible,
every entry point raises :class:`SolverUnavailable`.

The functions mirror what gadfly reaches through celerite2 (reference call
sites in parentheses):

=====================  ==========================================================
``Solver.loglike``     ``GaussianProcess.compute`` + ``log_likelihood``
                       (gadfly/gp.py:59,202-204,350), fused, nothing materialised
``Solver.sample``      ``compute`` + ``dot_tril``/``sample`` (gadfly/gp.py:327,391)
``Solver.factor``      ``compute`` keeping d and W (gadfly/gp.py:202-204)
``Solver.sweep``       ``driver.solve_lower/matmul_lower/solve_upper/matmul_upper``
                       (gadfly/gp.py:327,350,370)
``Solver.psd``         ``kernel.get_psd`` (gadfly/psd.py:151, tests/test_core.py:34)
=====================  ==========================================================
"""
import ctypes
import os
import threading

import numpy as np

__all__ = ["Solver", "KernelBatch", "SolverUnavailable", "LinAlgError", "default_solver",
           "library_path", "DevicePointer", "GF_MAX_J", "FLAG_ASYNC", "FLAG_REFERENCE_ORDER"]

GF_MAX_J = 176          # widest state of the register-resident scans
GF_MAX_J_WIDE = 352     # widest state at all (slower kernel, state in L2-resident scratch)
FLAG_ASYNC = 1
FLAG_REFERENCE_ORDER = 2
FLAG_SHARED_Y = 4
FLAG_WIDE_KERNEL = 8
FLAG_BLOCKED = 16

# scan kernel that served a call (gf_last_scan_path; include/gadfly_b200.h GF_PATH_*)
PATH_NONE, PATH_FAST, PATH_SMALL, PATH_REF, PATH_WIDE, PATH_BLOCKED = -1, 0, 1, 2, 3, 4
PATH_NAMES = {PATH_NONE: "none", PATH_FAST: "scan_fast", PATH_SMALL: "scan_small", PATH_REF: "scan_ref",
              PATH_WIDE: "scan_wide", PATH_BLOCKED: "scan_blk"}

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBNAME = "libgadfly_b200.so"


class SolverUnavailable(RuntimeError):
    """The CUDA library (or a CUDA device) is not available; there is no CPU fallback."""


class LinAlgError(Exception):
    """The covariance matrix is not positive definite (a pivot d[n] <= 0);
    celerite2 raises ``driver.LinAlgError`` in the same situation."""


def library_path():
    """In-tree library; ``$GADFLY_B200_LIB`` selects another build of the same C ABI (kernel A/B
    experiments, tools/ab_scan.py)."""
    return os.environ.get("GADFLY_B200_LIB") or os.path.join(_HERE, _LIBNAME)


_lib = None
_lib_lock = threading.Lock()

_i64p = ctypes.POINTER(ctypes.c_int64)
_f64p = ctypes.c_void_p      # host or device address
_i32p = ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/gadfly_b200.h declares
_SIGNATURES = {
    "gf_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "gf_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "gf_synchronize": (ctypes.c_int, [ctypes.c_void_p]),
    "gf_last_error": (ctypes.c_char_p, [ctypes.c_void_p]),
    "gf_stream": (ctypes.c_void_p, [ctypes.c_void_p]),
    "gf_ticket": (ctypes.c_int64, [ctypes.c_void_p]),
    "gf_wait": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64]),
    "gf_wait_stream": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "gf_stream_wait": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "gf_device_info": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int),
                                      ctypes.POINTER(ctypes.c_double), ctypes.c_int]),
    "gf_launch_count": (ctypes.c_int64, [ctypes.c_void_p]),
    "gf_last_kernel_ms": (ctypes.c_float, [ctypes.c_void_p]),
    "gf_last_scan_path": (ctypes.c_int, [ctypes.c_void_p]),
    "gf_loglike_batched": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _i64p, _i64p, _i64p, _f64p, ctypes.c_int64, _f64p, _f64p,
        _f64p, _f64p, _f64p, _f64p, _i32p, ctypes.c_uint32]),
    "gf_sample_batched": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _i64p, _i64p, _i64p, _f64p, ctypes.c_int64, _f64p, _f64p,
        _f64p, _f64p, ctypes.c_uint64, ctypes.c_uint64, _f64p, _f64p, _i32p, ctypes.c_uint32]),
    "gf_sample_multi": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _i64p, _i64p, _i64p, _f64p, ctypes.c_int64, _f64p, _f64p,
        _f64p, ctypes.c_int64, _f64p, ctypes.c_uint64, ctypes.c_uint64, _f64p, _f64p, _i32p, ctypes.c_uint32]),
    "gf_loglike_multi": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _i64p, _i64p, _i64p, _f64p, ctypes.c_int64, _f64p, _f64p,
        _f64p, ctypes.c_int64, _f64p, _f64p, _f64p, _i32p, ctypes.c_uint32]),
    "gf_factor_batched": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _i64p, _i64p, _i64p, _i64p, _f64p, ctypes.c_int64, _f64p,
        _f64p, _f64p, _f64p, _f64p, _f64p, _i32p, ctypes.c_uint32]),
    "gf_sweep_batched": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, _i64p, _i64p, _i64p, _i64p, _f64p,
        ctypes.c_int64, _f64p, _f64p, _f64p, _f64p, ctypes.c_uint32]),
    "gf_psd_batched": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _i64p, _f64p, _f64p, _f64p, ctypes.c_int64, _f64p,
        ctypes.c_uint32]),
    "gf_power_spectrum_batched": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, _f64p, ctypes.c_double, ctypes.c_int, _f64p,
        ctypes.c_uint32]),
    "gf_bin_power_batched": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _i64p, _i64p, _f64p, _f64p,
        ctypes.c_double, _f64p, _f64p, ctypes.c_uint32]),
    "gf_feed_stars": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _f64p, _f64p, _f64p, _f64p, _f64p, ctypes.c_double, _f64p,
        ctypes.c_int64, _f64p, ctypes.c_int64, _f64p, ctypes.c_int64, _i64p, _f64p, _f64p, _f64p, _f64p,
        ctypes.c_uint32]),
    "gf_feed_sho": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _i64p, _f64p, _f64p, _f64p, _f64p, _f64p, ctypes.c_uint32]),
    "gf_bandpass_amplitude": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _f64p, ctypes.c_int64, _f64p, _f64p, _f64p, ctypes.c_uint32]),
    "gf_conditional_mean": (ctypes.c_int, [
        ctypes.c_void_p, ctypes.c_int64, _f64p, ctypes.c_int64, _f64p, ctypes.c_int64, _f64p,
        _f64p, _f64p, ctypes.c_uint32]),
}


def load_library(path=None):
    """dlopen the C-ABI library and bind every declared symbol (no GPU needed for this)."""
    global _lib
    with _lib_lock:
        if _lib is not None and path is None:
            return _lib
        path = path or library_path()
        if not os.path.exists(path):
            raise SolverUnavailable(
                f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; "
                f"g.build()'` (nvcc, sm_100a). gadfly_b200 has no CPU fallback.")
        try:
            L = ctypes.CDLL(path)
        except OSError as exc:  # pragma: no cover - e.g. libcudart missing
            raise SolverUnavailable(f"cannot load {path}: {exc}") from exc
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError if the header and the library disagree
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = L
        return L


# ---------------------------------------------------------------------------------------
# pointers: numpy arrays (host) or anything with ``data_ptr()`` (a torch CUDA/CPU tensor)
# ---------------------------------------------------------------------------------------
class DevicePointer:
    """A raw device (or pinned host) address with an element count, for callers that manage memory
    without torch (cuda-python, cupy ...).  Ordering against other streams is the caller's business
    (``Solver.stream``, gf_wait_stream / gf_stream_wait)."""

    def __init__(self, address, count, dtype=np.float64):
        self.address, self.count, self.dtype = int(address), int(count), dtype


def _addr(x, dtype=np.float64, count=None, name="array"):
    """(address, keepalive) of a contiguous float64/int32 buffer on host or device."""
    if x is None:
        return None, None
    if isinstance(x, DevicePointer):
        if x.dtype != dtype:
            raise TypeError(f"{name}: pointer to {x.dtype}, need {dtype}")
        if count is not None and x.count < count:
            raise ValueError(f"{name}: {x.count} elements, need {count}")
        return x.address, x
    if hasattr(x, "data_ptr"):  # torch tensor
        import torch
        want = {np.float64: torch.float64, np.int32: torch.int32, np.int64: torch.int64}[dtype]
        if x.dtype != want or not x.is_contiguous():
            raise TypeError(f"{name}: tensor must be contiguous {want}")
        if count is not None and x.numel() < count:
            raise ValueError(f"{name}: {x.numel()} elements, need {count}")
        return x.data_ptr(), x
    a = np.ascontiguousarray(x, dtype=dtype)
    if count is not None and a.size < count:
        raise ValueError(f"{name}: {a.size} elements, need {count}")
    return a.ctypes.data, a


def _out(x, shape, dtype=np.float64):
    """An output buffer: the caller's (tensor or ndarray, written in place) or a new ndarray."""
    if x is None:
        x = np.empty(shape, dtype=dtype)
    elif not hasattr(x, "data_ptr") and not isinstance(x, DevicePointer):
        if not (isinstance(x, np.ndarray) and x.dtype == dtype and x.flags.c_contiguous):
            raise TypeError("output must be a C-contiguous ndarray of the right dtype")
    addr, keep = _addr(x, dtype, int(np.prod(shape)))
    return x, addr


def _i64(a):
    a = np.ascontiguousarray(a, dtype=np.int64)
    return a, a.ctypes.data_as(_i64p)


class KernelBatch:
    """Flat coefficient arrays of B kernels, as the library wants them.

    ``coef``  [sum Jc, 4]  (a', b', c, d) of every complex term after the exposure-time
                           transform (real terms enter as (a, 0, c, 0));
    ``base``  [sum Jc, 4]  the un-convolved coefficients (PSD);
    ``j_off`` [B+1], ``ddiag`` [B], ``delta`` [B].
    """

    def __init__(self, kernels):
        kernels = list(kernels)
        coef, base, j_off, ddiag, delta = [], [], [0], [], []
        for k in kernels:
            ar, cr, ac, bc, cc, dc, dd = k.scan_coefficients()
            rows = [np.stack([ar, np.zeros_like(ar), cr, np.zeros_like(cr)], axis=1),
                    np.stack([ac, bc, cc, dc], axis=1)]
            coef.append(np.concatenate(rows, axis=0))
            bar, bcr, bac, bbc, bcc, bdc = k.base_coefficients()
            base.append(np.concatenate([
                np.stack([bar, np.zeros_like(bar), bcr, np.zeros_like(bcr)], axis=1),
                np.stack([bac, bbc, bcc, bdc], axis=1)], axis=0))
            j_off.append(j_off[-1] + len(ar) + len(ac))
            ddiag.append(dd)
            delta.append(k.exposure)
        self.B = len(kernels)
        self.coef = np.ascontiguousarray(np.concatenate(coef, axis=0) if coef else np.empty((0, 4)))
        self.base = np.ascontiguousarray(np.concatenate(base, axis=0) if base else np.empty((0, 4)))
        self.j_off = np.asarray(j_off, dtype=np.int64)
        self.ddiag = np.asarray(ddiag, dtype=np.float64)
        self.delta = np.asarray(delta, dtype=np.float64)
        if self.B and int(np.max(np.diff(self.j_off))) * 2 > GF_MAX_J_WIDE:
            raise ValueError(f"kernel state wider than GF_MAX_J_WIDE = {GF_MAX_J_WIDE}")

    @staticmethod
    def for_stars(mass, radius, temperature, luminosity, texp_s=60.0, bandpass='SOHO VIRGO', alpha=None,
                  solver=None):
        """Batched ``Hyperparameters.for_star`` + kernel assembly for arrays of stars
        (gadfly_b200/feeder.py): ~100x faster than one kernel object per star on the host; with
        ``solver=`` the same arithmetic runs on that solver's GPU (csrc/feed.cu)."""
        from .feeder import kernel_batch_for_stars
        return kernel_batch_for_stars(mass, radius, temperature, luminosity, texp_s=texp_s,
                                      bandpass=bandpass, alpha=alpha, solver=solver)

    @property
    def J(self):
        return 2 * np.diff(self.j_off)

    def take(self, idx):
        """Sub-batch (used to shard across ranks)."""
        out = object.__new__(KernelBatch)
        idx = np.asarray(idx, dtype=np.int64)
        widths = np.diff(self.j_off)[idx]
        rows = np.concatenate([np.arange(self.j_off[i], self.j_off[i + 1]) for i in idx]) \
            if len(idx) else np.empty(0, dtype=np.int64)
        out.B = len(idx)
        out.coef = np.ascontiguousarray(self.coef[rows])
        out.base = np.ascontiguousarray(self.base[rows])
        out.j_off = np.concatenate([[0], np.cumsum(widths)]).astype(np.int64)
        out.ddiag = self.ddiag[idx].copy()
        out.delta = self.delta[idx].copy()
        return out


class Geometry:
    """CSR description of a batch of light curves: n_off[B+1], t_off[B]."""

    def __init__(self, n_off, t_off, t_len):
        self.n_off = np.ascontiguousarray(n_off, dtype=np.int64)
        self.t_off = np.ascontiguousarray(t_off, dtype=np.int64)
        self.t_len = int(t_len)
        self.B = len(self.t_off)

    @classmethod
    def shared_t(cls, B, N):
        """B sequences on one common time grid of N points."""
        return cls(np.arange(B + 1, dtype=np.int64) * N, np.zeros(B, dtype=np.int64), N)

    @classmethod
    def ragged(cls, lengths):
        """Each sequence has its own time stamps, concatenated."""
        off = np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64)
        return cls(off, off[:-1].copy(), int(off[-1]))


class Solver:
    """One library handle (one CUDA stream) on one device."""

    def __init__(self, device=0):
        self._lib = load_library()
        h = ctypes.c_void_p()
        rc = self._lib.gf_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise SolverUnavailable(
                f"gf_create(device={device}) failed with code {rc}: no usable CUDA device. "
                f"gadfly_b200 has no CPU fallback.")
        self._h = h
        self._calls = 0
        self._inflight = []
        self._ticket_call = {}
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.gf_destroy(self._h)
            self._h = None

    def __del__(self):  # pragma: no cover
        try:
            self.close()
        except Exception:
            pass

    # -- bookkeeping -------------------------------------------------------------------
    def _check(self, rc):
        if rc != 0:
            msg = self._lib.gf_last_error(self._h)
            msg = msg.decode() if msg else ""
            if rc < 0:
                raise ValueError(f"gadfly_b200: argument error {rc}: {msg}")
            raise RuntimeError(f"gadfly_b200: CUDA error {rc}: {msg}")

    def synchronize(self):
        self._check(self._lib.gf_synchronize(self._h))
        self._inflight.clear()

    def ticket(self):
        """Mark "everything issued so far, copies back to host buffers included" (FLAG_ASYNC calls)."""
        t = int(self._lib.gf_ticket(self._h))
        if t <= 0:
            self._check(t)
        self._ticket_call[t] = self._calls
        return t

    def wait(self, ticket):
        """Block until the work marked by ``ticket`` has completed (later calls may still be running)."""
        self._check(self._lib.gf_wait(self._h, int(ticket)))
        upto = self._ticket_call.get(int(ticket))
        if upto is not None:
            self._inflight = [(c, a) for c, a in self._inflight if c > upto]
            self._ticket_call = {k: v for k, v in self._ticket_call.items() if k > int(ticket)}

    # Device buffers are touched on the handle's compute stream only (include/gadfly_b200.h,
    # "Streams"): whatever torch stream produced a CUDA tensor we are handed must be ordered
    # before our kernels, and torch work that follows an ASYNC call after them.
    @staticmethod
    def _cuda_tensors(xs):
        return [x for x in xs if x is not None and hasattr(x, "data_ptr") and getattr(x, "is_cuda", False)]

    def _order_before(self, *xs):
        ts = self._cuda_tensors(xs)
        if ts:
            import torch
            cur = torch.cuda.current_stream(ts[0].device).cuda_stream
            if cur != self.stream:
                self._check(self._lib.gf_wait_stream(self._h, ctypes.c_void_p(cur)))

    def _order_after(self, flags, *xs):
        # Host outputs of a FLAG_ASYNC call are written when the work completes (pageable ones in
        # gf_synchronize / gf_wait, from the library's pinned ring): keep them alive until then,
        # whatever the caller does with the returned arrays.
        if flags & FLAG_ASYNC:
            self._calls += 1
            host = [x for x in xs if isinstance(x, np.ndarray)]
            if host:
                self._inflight.append((self._calls, host))
        else:
            self._inflight.clear()
        ts = self._cuda_tensors(xs)
        if ts and (flags & FLAG_ASYNC):
            import torch
            cur = torch.cuda.current_stream(ts[0].device).cuda_stream
            if cur != self.stream:
                self._check(self._lib.gf_stream_wait(self._h, ctypes.c_void_p(cur)))

    @property
    def stream(self):
        return self._lib.gf_stream(self._h)

    @property
    def launch_count(self):
        return int(self._lib.gf_launch_count(self._h))

    @property
    def last_kernel_ms(self):
        return float(self._lib.gf_last_kernel_ms(self._h))

    def last_scan_path(self):
        """Name of the scan kernel that served the most recent scan launch on this handle
        (``"scan_fast"``, ``"scan_small"``, ``"scan_ref"``, ``"scan_wide"``, ``"scan_blk"``), or
        ``"none"`` before the first one."""
        return PATH_NAMES[int(self._lib.gf_last_scan_path(self._h))]

    def device_info(self, measure=False):
        sm = ctypes.c_int()
        fl = ctypes.c_double()
        self._check(self._lib.gf_device_info(self._h, ctypes.byref(sm), ctypes.byref(fl), int(measure)))
        return dict(sm_count=sm.value, fp64_flops=fl.value)

    # -- (f2) feeder -------------------------------------------------------------------
    def feed_stars(self, mass, radius, temperature, luminosity, delta, gran, modes, alpha=None,
                   wavelength_nm=550.0, want_sho=True):
        """Stellar parameters -> (j_off, sho, coef, base, ddiag) on the device (gf_feed_stars):
        batched ``Hyperparameters.for_star`` + kernel assembly.  ``gran`` [n_gran, 3] and ``modes``
        [n_modes, 4 + n_gran] are the star-independent solar tables (feeder.solar_tables())."""
        M, R, T, L, D = (np.ascontiguousarray(np.atleast_1d(x), dtype=np.float64)
                         for x in (mass, radius, temperature, luminosity, delta))
        B = len(M)
        assert len(R) == len(T) == len(L) == len(D) == B
        gran = np.ascontiguousarray(gran, dtype=np.float64)
        modes = np.ascontiguousarray(modes, dtype=np.float64)
        n_gran, n_modes = len(gran), len(modes)
        assert gran.shape == (n_gran, 3) and modes.shape == (n_modes, 4 + n_gran)
        al = None if alpha is None else np.ascontiguousarray(np.broadcast_to(alpha, (B,)), dtype=np.float64)
        cap = B * (n_gran + n_modes)
        j_off = np.zeros(B + 1, dtype=np.int64)
        sho = np.empty((cap, 3)) if want_sho else None
        coef = np.empty((cap, 4))
        base = np.empty((cap, 4))
        ddiag = np.empty(B)
        self._check(self._lib.gf_feed_stars(
            self._h, B, M.ctypes.data, R.ctypes.data, T.ctypes.data, L.ctypes.data,
            None if al is None else al.ctypes.data, float(wavelength_nm), D.ctypes.data,
            n_gran, gran.ctypes.data, n_modes, modes.ctypes.data, cap,
            j_off.ctypes.data_as(_i64p), None if sho is None else sho.ctypes.data, coef.ctypes.data,
            base.ctypes.data, ddiag.ctypes.data, 0))
        self._inflight.clear()
        n = int(j_off[-1])
        return j_off, (None if sho is None else sho[:n]), coef[:n], base[:n], ddiag

    def feed_sho(self, j_off, S0, w0, Q, delta):
        """(S0, w0, Q) in CSR layout -> (coef, base, ddiag) on the device (gf_feed_sho)."""
        j_off = np.ascontiguousarray(j_off, dtype=np.int64)
        B = len(j_off) - 1
        sho = np.ascontiguousarray(np.stack([S0, w0, Q], axis=1), dtype=np.float64)
        n = int(j_off[-1])
        assert sho.shape == (n, 3)
        D = np.ascontiguousarray(np.broadcast_to(delta, (B,)), dtype=np.float64)
        coef, base, ddiag = np.empty((n, 4)), np.empty((n, 4)), np.empty(B)
        self._check(self._lib.gf_feed_sho(self._h, B, j_off.ctypes.data_as(_i64p), sho.ctypes.data, D.ctypes.data,
                                          coef.ctypes.data, base.ctypes.data, ddiag.ctypes.data, 0))
        self._inflight.clear()
        return coef, base, ddiag

    def bandpass_amplitude(self, temperature, wl_um, transmittance):
        """Bandpass amplitude ratio (Morris+ 2020 Eqn 11) of B temperatures on the device."""
        T = np.ascontiguousarray(np.atleast_1d(temperature), dtype=np.float64)
        wl = np.ascontiguousarray(wl_um, dtype=np.float64)
        tr = np.ascontiguousarray(transmittance, dtype=np.float64)
        assert wl.shape == tr.shape and wl.ndim == 1
        out = np.empty(len(T))
        self._check(self._lib.gf_bandpass_amplitude(self._h, len(T), T.ctypes.data, len(wl), wl.ctypes.data,
                                                    tr.ctypes.data, out.ctypes.data, 0))
        self._inflight.clear()
        return out

    # -- K1 ----------------------------------------------------------------------------
    def loglike(self, kb, geom, t, y, diag=None, logdet=None, quad=None, status=None, flags=0):
        """-> (logdet[B], quad[B], status[B]); log L = -(quad + logdet + N log 2 pi)/2."""
        B = geom.B
        assert kb.B == B
        total = int(geom.n_off[-1])
        keep = []
        pt, k = _addr(t, count=geom.t_len, name="t"); keep.append(k)
        ny = geom.t_len if (flags & FLAG_SHARED_Y) else total     # y laid out like t
        py, k = _addr(y, count=ny, name="y"); keep.append(k)
        pd, k = _addr(diag, count=ny, name="diag"); keep.append(k)
        logdet, pl = _out(logdet, (B,))
        quad, pq = _out(quad, (B,))
        status, ps = _out(status, (B,), np.int32)
        n_off, pn = _i64(geom.n_off)
        t_off, pto = _i64(geom.t_off)
        j_off, pj = _i64(kb.j_off)
        self._order_before(t, y, diag, logdet, quad, status)
        self._check(self._lib.gf_loglike_batched(
            self._h, B, pn, pto, pj, pt, geom.t_len, py, pd, kb.coef.ctypes.data,
            kb.ddiag.ctypes.data, pl, pq, ps, flags))
        self._order_after(flags, logdet, quad, status)
        return logdet, quad, status

    # -- K2 ----------------------------------------------------------------------------
    def sample(self, kb, geom, t, diag=None, normals=None, seed=0, seq0=0, out=None, logdet=None,
               status=None, flags=0):
        """-> (x[sum N], logdet[B], status[B]) with x = L (sqrt(d) o n)."""
        B = geom.B
        assert kb.B == B
        total = int(geom.n_off[-1])
        keep = []
        pt, k = _addr(t, count=geom.t_len, name="t"); keep.append(k)
        pd, k = _addr(diag, count=total, name="diag"); keep.append(k)
        pn_, k = _addr(normals, count=total, name="normals"); keep.append(k)
        out, po = _out(out, (total,))
        logdet, pl = _out(logdet, (B,))
        status, ps = _out(status, (B,), np.int32)
        n_off, pn = _i64(geom.n_off)
        t_off, pto = _i64(geom.t_off)
        j_off, pj = _i64(kb.j_off)
        self._order_before(t, diag, normals, out, logdet, status)
        self._check(self._lib.gf_sample_batched(
            self._h, B, pn, pto, pj, pt, geom.t_len, pd, kb.coef.ctypes.data,
            kb.ddiag.ctypes.data, pn_, int(seed), int(seq0), po, pl, ps, flags))
        self._order_after(flags, out, logdet, status)
        return out, logdet, status

    # -- K1m / K2m: k right-hand sides per sequence on one factor ---------------------------
    def sample_multi(self, kb, geom, t, k, diag=None, normals=None, seed=0, seq0=0, out=None, logdet=None,
                     status=None, flags=0):
        """k realisations per sequence from ONE factor -> (x[sum N * k] laid out [b][r][n], logdet[B],
        status[B]).  ``normals`` (same layout) or Philox with realisation index seq0 + b k + r."""
        B, k = geom.B, int(k)
        assert kb.B == B and k >= 1
        total = int(geom.n_off[-1])
        keep = []
        pt, q = _addr(t, count=geom.t_len, name="t"); keep.append(q)
        pd, q = _addr(diag, count=total, name="diag"); keep.append(q)
        pn_, q = _addr(normals, count=total * k, name="normals"); keep.append(q)
        out, po = _out(out, (total * k,))
        logdet, pl = _out(logdet, (B,))
        status, ps = _out(status, (B,), np.int32)
        n_off, pn = _i64(geom.n_off)
        t_off, pto = _i64(geom.t_off)
        j_off, pj = _i64(kb.j_off)
        self._order_before(t, diag, normals, out, logdet, status)
        self._check(self._lib.gf_sample_multi(
            self._h, B, pn, pto, pj, pt, geom.t_len, pd, kb.coef.ctypes.data, kb.ddiag.ctypes.data, k,
            pn_, int(seed), int(seq0), po, pl, ps, flags))
        self._order_after(flags, out, logdet, status)
        return out, logdet, status

    def loglike_multi(self, kb, geom, t, y, k, diag=None, logdet=None, quad=None, status=None, flags=0):
        """k data vectors per sequence on ONE factor -> (logdet[B], quad[B * k], status[B])."""
        B, k = geom.B, int(k)
        assert kb.B == B and k >= 1
        total = int(geom.n_off[-1])
        keep = []
        pt, q = _addr(t, count=geom.t_len, name="t"); keep.append(q)
        py, q = _addr(y, count=total * k, name="y"); keep.append(q)
        pd, q = _addr(diag, count=total, name="diag"); keep.append(q)
        logdet, pl = _out(logdet, (B,))
        quad, pq = _out(quad, (B * k,))
        status, ps = _out(status, (B,), np.int32)
        n_off, pn = _i64(geom.n_off)
        t_off, pto = _i64(geom.t_off)
        j_off, pj = _i64(kb.j_off)
        self._order_before(t, y, diag, logdet, quad, status)
        self._check(self._lib.gf_loglike_multi(
            self._h, B, pn, pto, pj, pt, geom.t_len, pd, kb.coef.ctypes.data, kb.ddiag.ctypes.data, k,
            py, pl, pq, ps, flags))
        self._order_after(flags, logdet, quad, status)
        return logdet, quad, status

    # -- K3 ----------------------------------------------------------------------------
    def factor(self, kb, geom, t, diag=None, d=None, W=None, w_off=None, want_W=True, logdet=None,
               status=None, flags=0):
        """-> (d[sum N], W[sum N*J] or None, w_off, logdet[B], status[B])."""
        B = geom.B
        assert kb.B == B
        total = int(geom.n_off[-1])
        lengths = np.diff(geom.n_off)
        if w_off is None:
            w_off = np.concatenate([[0], np.cumsum(lengths * kb.J)]).astype(np.int64)
            w_total = int(w_off[-1])
            w_off = w_off[:-1]
        else:
            w_off = np.ascontiguousarray(w_off, dtype=np.int64)
            w_total = int(np.max(w_off + lengths * kb.J)) if B else 0
        keep = []
        pt, k = _addr(t, count=geom.t_len, name="t"); keep.append(k)
        pd, k = _addr(diag, count=total, name="diag"); keep.append(k)
        d, pdd = _out(d, (total,))
        if want_W or W is not None:
            W, pW = _out(W, (w_total,))
        else:
            pW = None
        logdet, pl = _out(logdet, (B,))
        status, ps = _out(status, (B,), np.int32)
        n_off, pn = _i64(geom.n_off)
        t_off, pto = _i64(geom.t_off)
        j_off, pj = _i64(kb.j_off)
        w_off_arr, pw = _i64(w_off)
        self._order_before(t, diag, d, W, logdet, status)
        self._check(self._lib.gf_factor_batched(
            self._h, B, pn, pto, pj, pw, pt, geom.t_len, pd, kb.coef.ctypes.data,
            kb.ddiag.ctypes.data, pdd, pW, pl, ps, flags))
        self._order_after(flags, d, W, logdet, status)
        return d, W, w_off_arr, logdet, status

    # -- K4 ----------------------------------------------------------------------------
    def sweep(self, op, kb, geom, w_off, t, W, Y, Z=None, flags=0):
        """op 0 solve_lower, 1 matmul_lower, 2 solve_upper, 3 matmul_upper; -> Z[sum N]."""
        B = geom.B
        assert kb.B == B
        total = int(geom.n_off[-1])
        keep = []
        pt, k = _addr(t, count=geom.t_len, name="t"); keep.append(k)
        pW, k = _addr(W, name="W"); keep.append(k)
        pY, k = _addr(Y, count=total, name="Y"); keep.append(k)
        Z, pZ = _out(Z, (total,))
        n_off, pn = _i64(geom.n_off)
        t_off, pto = _i64(geom.t_off)
        j_off, pj = _i64(kb.j_off)
        w_off, pw = _i64(w_off)
        self._order_before(t, W, Y, Z)
        self._check(self._lib.gf_sweep_batched(
            self._h, int(op), B, pn, pto, pj, pw, pt, geom.t_len, kb.coef.ctypes.data, pW, pY, pZ,
            flags))
        self._order_after(flags, Z)
        return Z

    # -- K5 ----------------------------------------------------------------------------
    def psd(self, kb, omega, out=None, n_omega=None, flags=0):
        """-> psd[B, F] of the (exposure-integrated) kernels at angular frequencies omega."""
        if n_omega is not None:
            F = int(n_omega)
        else:   # ndarray or device tensor
            F = int(omega.numel()) if hasattr(omega, "numel") else int(np.size(omega))
        pw, keep = _addr(omega, count=F, name="omega")
        out, po = _out(out, (kb.B, F))
        j_off, pj = _i64(kb.j_off)
        self._order_before(omega, out)
        self._check(self._lib.gf_psd_batched(
            self._h, kb.B, pj, kb.base.ctypes.data, kb.delta.ctypes.data, pw, F, po, flags))
        self._order_after(flags, out)
        return out


    # -- K7 ----------------------------------------------------------------------------
    def power_spectrum(self, flux, B, N, d, include_zero=False, out=None, flags=0):
        """-> power[B, N//2 (+1)] = |rfft(flux)|^2 d / sqrt(2 pi) / N (flux [B, N] in ppm, d in 1/uHz)."""
        nout = N // 2 + 1 - (0 if include_zero else 1)
        pf, keep = _addr(flux, count=B * N, name="flux")
        out, po = _out(out, (B, nout))
        self._order_before(flux, out)
        self._check(self._lib.gf_power_spectrum_batched(self._h, B, N, pf, float(d), int(include_zero), po, flags))
        self._order_after(flags, out)
        return out

    def bin_power(self, power, B, axis, lo, cnt, constant=1.0, stat=None, err=None, flags=0):
        """-> (stat[B, nb], err[B, nb]) for bins [lo[k], lo[k] + cnt[k]) of the shared axis[F]."""
        F = int(axis.numel()) if hasattr(axis, "numel") else int(np.size(axis))
        lo_a, plo = _i64(lo)
        cnt_a, pcnt = _i64(cnt)
        nb = len(lo_a)
        pa, k1 = _addr(axis, count=F, name="axis")
        pp, k2 = _addr(power, count=B * F, name="power")
        stat, ps = _out(stat, (B, nb))
        err, pe = _out(err, (B, nb))
        self._order_before(axis, power, stat, err)
        self._check(self._lib.gf_bin_power_batched(self._h, B, F, nb, plo, pcnt, pa, pp, float(constant), ps, pe, flags))
        self._order_after(flags, stat, err)
        return stat, err

    # -- K6 ----------------------------------------------------------------------------
    def conditional_mean(self, coef, t, ts, alpha, out=None, flags=0):
        """-> mu[M] = K(ts, t) alpha for the semiseparable kernel ``coef[Jc, 4]`` (a', b', c, d);
        ``t`` and ``ts`` sorted ascending (celerite2 general_matmul_lower + _upper)."""
        coef = np.ascontiguousarray(coef, dtype=np.float64).reshape(-1, 4)
        N = int(t.numel()) if hasattr(t, "numel") else int(np.size(t))
        M = int(ts.numel()) if hasattr(ts, "numel") else int(np.size(ts))
        pt, k1 = _addr(t, count=N, name="t")
        pts, k2 = _addr(ts, count=M, name="ts")
        pa, k3 = _addr(alpha, count=N, name="alpha")
        out, po = _out(out, (M,))
        self._order_before(t, ts, alpha, out)
        self._check(self._lib.gf_conditional_mean(
            self._h, N, pt, M, pts, coef.shape[0], coef.ctypes.data, pa, po, flags))
        self._order_after(flags, out)
        return out


_default = {}
_default_lock = threading.Lock()


def default_solver(device=None):
    """Process-wide solver for ``device`` (default: $LOCAL_RANK or 0)."""
    if device is None:
        device = int(os.environ.get("GADFLY_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    with _default_lock:
        if device not in _default:
            _default[device] = Solver(device)
        return _default[device]


def psd(kernels, omega):
    """PSD of each kernel on the shared grid ``omega`` (used by ``Term.get_psd``)."""
    kb = KernelBatch(kernels)
    return default_solver().psd(kb, np.ascontiguousarray(omega, dtype=np.float64))
