"""The kernels that run after a factor exists -- the four O(N J) sweeps (csrc/sweep.cu), the conditional
mean at new times (csrc/cond.cu) and the k-right-hand-side helpers (csrc/multi.cu with the virtual
sequences of api.cu run_multi) -- against an extended-precision reference of the same operation.

The reference is numpy ``longdouble`` (a 64-bit mantissa on x86-64) and takes the FP64 inputs the kernels
take.  It evaluates the operation as the kernels define it: phases are the FP64 products fl64(d t)
(``__dmul_rn`` in the kernels), their cos / sin are taken in longdouble; a step's decay is
exp(-c dt) of the FP64 difference dt of neighbouring stamps.  Next to every result runs a magnitude
run -- the same sums over |terms| -- which gives each element the scale its tolerance is relative to,
so that a bound does not depend on cancellation:

* matmul sweeps (ops 1, 3): componentwise forward error  |z - z_ref| <= tol * magnitude;
* solve sweeps (ops 0, 2): componentwise backward error  |L z - y| <= tol * (|y| + |L| |z|), with L
  applied in longdouble to the kernel's z (independent of cond(L)), and a normwise forward bound;
* conditional mean: |mu - mu_ref| <= tol * sum_m |alpha_m| sum_j e^{-c |tau|} (|a| + |b|);
* quad of loglike_multi: relative to sum z^2 / d of the longdouble solve.

Where the library promises bits (a sequence does not depend on its neighbours or its place in the
launch; sample_multi is Solver.sweep(1) of sqrt(d) n on the factor), the cases assert bit-identity.

The tests without the ``gpu`` mark check the reference itself: against a dense longdouble L, against
the FP64 oracle on the dense goldens, and against the kernel definition k(tau)."""
import numpy as np
import pytest

import gadfly_b200 as g
from gadfly_b200 import batch, philox
from gadfly_b200.solver import Geometry, KernelBatch
import oracle
from oracle import terms_oracle as T
from conftest import golden

LD = np.longdouble

# Bounds on error / magnitude per group.  Each is 20 ... 45x the worst ratio observed on one NVIDIA B200
# (1000 W power limit), given beside it; none may be looser than 100x that ratio or than 1e-11.
BOUND = {
    "sweep_matmul": 2e-14,       # 7.2e-16  ops 1, 3: componentwise forward error
    "sweep_solve": 1e-14,        # 2.3e-16  ops 0, 2: componentwise backward error
    "sweep_solve_fwd": 1e-13,    # 2.9e-15  ops 0, 2: normwise forward error
    "cond_mean": 2e-14,          # 9.8e-16
    "gp_alpha": 1e-14,           # 3.0e-16  apply_inverse inside predict: normwise forward error
    "multi_sample": 3e-14,       # 1.1e-15  Philox realisations against the longdouble matmul
    "quad": 5e-15,               # 2.0e-16  loglike_multi quad, relative
}
_WORST = {}


def _check(group, err, scale):
    """Assert |err| <= BOUND[group] * scale elementwise, and remember the worst ratio."""
    err = np.atleast_1d(np.abs(np.asarray(err, dtype=LD)).astype(np.float64))
    scale = np.broadcast_to(np.asarray(scale, dtype=LD).astype(np.float64), err.shape)
    if err.size == 0:
        return 0.0
    r = np.divide(err, scale, out=np.where(err > 0, np.inf, 0.0), where=scale > 0)
    worst = float(np.max(r))
    _WORST[group] = max(_WORST.get(group, 0.0), worst)
    assert worst <= BOUND[group], (group, worst, int(np.argmax(r)))
    return worst


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if _WORST:
        print("\nworst error / magnitude: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(_WORST.items())))


# ---- kernels and inputs -------------------------------------------------------------------------
@pytest.fixture(scope="module")
def kern(solar_kernel):
    """kern(J): a kernel of state width J -- the first J / 2 solar terms, or the solar kernel plus
    (J - 172) / 2 extra p-mode-like terms (solar p modes at half the power, shifted by 0.3 %)."""
    terms = list(solar_kernel.term.terms)
    pm = terms[6:]
    extra = [g.SHOTerm(S0=pm[i % len(pm)].S0 * 0.5, w0=pm[i % len(pm)].w0 * (1 + 0.003 * (1 + i // len(pm))),
                       Q=pm[i % len(pm)].Q) for i in range(91)]
    cache = {}

    def make(J):
        if J not in cache:
            k = g.StellarOscillatorKernel(terms=(terms + extra)[:J // 2], delta=solar_kernel.delta)
            assert k.J == J
            cache[J] = k
        return cache[J]
    return make


def _k0(k):
    sc = k.scan_coefficients()
    return float(np.sum(sc[0]) + np.sum(sc[2]) + sc[6])


def _times(cadence, N, seed=0):
    """uniform: 1-min cadence.  mixed: runs of 1-min and 3-min cadence with 1e-3 jitter, a 0.4 and a 40
    gap (every decay underflows over the latter).  bjd: BJD-like absolute stamps, phases near 1e9 rad."""
    if cadence == "uniform" or N == 0:
        return np.arange(N) * 6e-5
    rng = np.random.default_rng(seed)
    if cadence == "bjd":
        dt = np.where(np.arange(N) < N // 2, 6e-5, 1.2e-4) * (1 + 1e-3 * rng.standard_normal(N))
        return 2.1e5 + np.cumsum(dt)
    assert cadence == "mixed"
    dt = np.where(np.arange(N) % 11 < 6, 6e-5, 1.8e-4) * (1 + 1e-3 * rng.standard_normal(N))
    dt[N // 3] = 0.4
    dt[(2 * N) // 3] = 40.0
    return np.cumsum(dt)


def _diag(k, N, rng):
    """Heteroscedastic white noise of 1 ... 2 % of k(0): a well-conditioned system."""
    return _k0(k) * 1e-2 * (1 + rng.uniform(size=N))


def _take(kb, idx):
    """KernelBatch.take for many repeats (vectorised row gather)."""
    idx = np.asarray(idx, dtype=np.int64)
    widths = np.diff(kb.j_off)[idx]
    j_off = np.concatenate([[0], np.cumsum(widths)]).astype(np.int64)
    rows = np.repeat(kb.j_off[idx] - j_off[:-1], widths) + np.arange(j_off[-1])
    out = object.__new__(KernelBatch)
    out.B, out.j_off = len(idx), j_off
    out.coef = np.ascontiguousarray(kb.coef[rows])
    out.base = np.ascontiguousarray(kb.base[rows])
    out.ddiag, out.delta = kb.ddiag[idx].copy(), kb.delta[idx].copy()
    return out


# ---- the longdouble reference -------------------------------------------------------------------
def _rows(coef, t):
    """U rows [N, 2 Jc] (cos block | sin block) of the coefficient rows (a', b', c, d) at times t, and
    their elementwise magnitudes: phases fl64(d t), cos / sin in longdouble."""
    a, b = coef[:, 0].astype(LD), coef[:, 1].astype(LD)
    ph = np.multiply.outer(np.asarray(t, dtype=np.float64), coef[:, 3]).astype(LD)
    cs, sn = np.cos(ph), np.sin(ph)
    U = np.concatenate([a * cs + b * sn, a * sn - b * cs], axis=1)
    Um = np.concatenate([abs(a * cs) + abs(b * sn), abs(a * sn) + abs(b * cs)], axis=1)
    return U, Um


def _gap_decay(coef, t):
    """[N - 1, 2 Jc]: exp(-c dt) over the FP64 step dt = t[n] - t[n - 1]."""
    dt = np.diff(np.asarray(t, dtype=np.float64)).astype(LD)
    p = np.exp(-np.multiply.outer(dt, coef[:, 2].astype(LD)))
    return np.concatenate([p, p], axis=1)


def _chain(dot, upd, dec, y, solve):
    """F <- dec_m o (F + upd_{m-1} prev),  z_m = y_m -/+ dot_m . F  over the steps m of every row of a
    batch ([R, S, J2] arrays; dec[:, 0] is not used); prev = z (solve rows) or y."""
    R, S, _ = dot.shape
    F = np.zeros(dot.shape[::2], dtype=LD)
    z = np.zeros((R, S), dtype=LD)
    prev = np.zeros(R, dtype=LD)
    for m in range(S):
        if m:
            F = dec[:, m] * (F + upd[:, m - 1] * prev[:, None])
        acc = np.sum(dot[:, m] * F, axis=1)
        z[:, m] = np.where(solve, y[:, m] - acc, y[:, m] + acc)
        prev = np.where(solve, z[:, m], y[:, m])
    return z


def sweep_ref(op, items):
    """The O(N J) recurrence of csrc/sweep.cu in longdouble for a list of (coef[Jc, 4], t[N], W[N * 2 Jc],
    y[N]) -> [(z, mag)]: z = L^-1 y (op 0), L y (1), L^-T y (2), L^T y (3) with
    L = I + tril(U (W o decay)^T, -1); mag is the same recurrence as a product on |U|, |W|, |y|."""
    upper, solve = op >= 2, op in (0, 2)
    rows = []
    for coef, t, W, y in items:
        N, J2 = len(t), 2 * len(coef)
        U, Um = _rows(coef, t)
        Wl = np.asarray(W, dtype=np.float64).reshape(N, J2).astype(LD)
        p = _gap_decay(coef, t)
        y = np.asarray(y, dtype=np.float64).astype(LD)
        if upper:       # step m is sample N - 1 - m; the state enters through U, is read through W
            dot, upd, dotm, updm, p, y = Wl[::-1], U[::-1], abs(Wl[::-1]), Um[::-1], p[::-1], y[::-1]
        else:
            dot, upd, dotm, updm = U, Wl, Um, abs(Wl)
        dec = np.concatenate([np.zeros((1, J2), dtype=LD), p], axis=0)
        rows.append((dot, upd, dec, y, solve))
        rows.append((dotm, updm, dec, abs(y), False))
    S = max([len(r[3]) for r in rows] + [1])
    J2 = max([r[0].shape[1] for r in rows] + [2])
    R = len(rows)
    dot, upd, dec = (np.zeros((R, S, J2), dtype=LD) for _ in range(3))
    y = np.zeros((R, S), dtype=LD)
    for i, (a, b, c, v, _) in enumerate(rows):
        n, j = a.shape
        dot[i, :n, :j], upd[i, :n, :j], dec[i, :n, :j], y[i, :n] = a, b, c, v
    z = _chain(dot, upd, dec, y, np.array([r[4] for r in rows]))
    out = []
    for i in range(0, R, 2):
        n = len(rows[i][3])
        zi, mi = z[i, :n], z[i + 1, :n]
        out.append((zi[::-1], mi[::-1]) if upper else (zi, mi))
    return out


def dense_L(coef, t, W):
    """Dense longdouble L = I + tril(U (W o decay)^T, -1) and its magnitude I + tril(|U| (|W| o decay)^T, -1),
    the decay exp(-c (T_n - T_m)) taken once over the longdouble sum T of the FP64 steps."""
    N, J2 = len(t), 2 * len(coef)
    U, Um = _rows(coef, t)
    Wl = np.asarray(W, dtype=np.float64).reshape(N, J2).astype(LD)
    Tn = np.concatenate([[LD(0)], np.cumsum(np.diff(np.asarray(t, dtype=np.float64)).astype(LD))])
    c = np.concatenate([coef[:, 2], coef[:, 2]]).astype(LD)
    dec = np.exp(-np.maximum(Tn[:, None] - Tn[None, :], LD(0))[:, :, None] * c)
    eye = np.eye(N, dtype=LD)
    return (np.tril(np.einsum("nj,mj,nmj->nm", U, Wl, dec), -1) + eye,
            np.tril(np.einsum("nj,mj,nmj->nm", Um, abs(Wl), dec), -1) + eye)


def _tri_solve(L, y, lower):
    """Forward / backward substitution in longdouble on a unit-diagonal triangle."""
    N = len(y)
    z = np.zeros(N, dtype=LD)
    for i in (range(N) if lower else range(N - 1, -1, -1)):
        s = L[i, :i] @ z[:i] if lower else L[i, i + 1:] @ z[i + 1:]
        z[i] = y[i] - s
    return z


def cond_ref(coef, t, ts, alpha, rows=None):
    """mu[i] = sum_m alpha_m k(t*_i, t_m) in the product form of csrc/cond.cu (forward t_m <= t*, backward
    t_m > t*) and its magnitude sum_m |alpha_m| sum_j e^{-c |tau|} (|a| + |b|), for i in ``rows``."""
    rows = np.arange(len(ts)) if rows is None else np.asarray(rows)
    a, b, c = (coef[:, i].astype(LD) for i in range(3))
    cs_t, sn_t = (f(np.multiply.outer(t, coef[:, 3]).astype(LD)) for f in (np.cos, np.sin))
    Ut = (a * cs_t + b * sn_t, a * sn_t - b * cs_t)
    al = np.asarray(alpha, dtype=np.float64).astype(LD)
    tl = np.asarray(t, dtype=np.float64).astype(LD)
    mu = np.zeros(len(rows), dtype=LD)
    mag = np.zeros(len(rows), dtype=LD)
    ab = abs(a) + abs(b)
    step = max(1, int(4e6 // max(1, len(t) * len(coef))))
    for i0 in range(0, len(rows), step):
        r = rows[i0:i0 + step]
        tq = ts[r]
        ph = np.multiply.outer(tq, coef[:, 3]).astype(LD)
        cs, sn = np.cos(ph), np.sin(ph)
        tau = np.asarray(tq, dtype=np.float64).astype(LD)[:, None] - tl[None, :]     # [r, N]
        e = np.exp(-np.abs(tau)[:, :, None] * c)                                        # [r, N, Jc]
        fwd = (a * cs + b * sn)[:, None] * cs_t[None] + (a * sn - b * cs)[:, None] * sn_t[None]
        bwd = cs[:, None] * Ut[0][None] + sn[:, None] * Ut[1][None]
        k = e * np.where((t[None, :] <= tq[:, None])[:, :, None], fwd, bwd)
        mu[i0:i0 + step] = np.sum(k, axis=2) @ al
        mag[i0:i0 + step] = np.sum(e * ab, axis=2) @ abs(al)
    return mu, mag


# ---- CPU: the reference against independent evaluations -----------------------------------------
def _oracle_factor(k, t, diag):
    """(coef[Jc, 4] rows as KernelBatch lays them out, W[N, 2 Jc] in the library's layout, d) of the FP64
    oracle's factor."""
    sc = k.scan_coefficients()
    ogp = oracle.OracleGP(sc, t, diag=diag)
    Jr, Jc = len(sc[0]), len(sc[2])
    N = len(t)
    Wl = np.zeros((N, 2 * (Jr + Jc)))
    Wl[:, :Jr] = ogp.W[:, :Jr]                        # a real term is a row (a, 0, c, 0): its sin column is 0
    Wl[:, Jr:Jr + Jc] = ogp.W[:, Jr:Jr + Jc]
    Wl[:, 2 * Jr + Jc:] = ogp.W[:, Jr + Jc:]
    return KernelBatch([k]).coef, Wl, ogp


@pytest.mark.parametrize("cadence", ["uniform", "mixed", "bjd"])
@pytest.mark.parametrize("J", [2, 10, 64])
def test_reference_recurrence_equals_dense_longdouble(kern, J, cadence):
    """For N <= 200 the recurrence is L y, L^-1 y, L^T y, L^-T y of the dense longdouble L, to the
    longdouble level."""
    k = kern(J)
    rng = np.random.default_rng(J)
    N = 160
    t = _times(cadence, N, seed=J)
    coef, W, _ = _oracle_factor(k, t, _diag(k, N, rng))
    y = rng.standard_normal(N)
    L, Lm = dense_L(coef, t, W)
    yl = y.astype(LD)
    dense = [_tri_solve(L, yl, True), L @ yl, _tri_solve(L.T, yl, False), L.T @ yl]
    for op in range(4):
        (z, mag), = sweep_ref(op, [(coef, t, W, y)])
        M = Lm if op < 2 else Lm.T
        # the magnitude run is the product with the magnitude matrix, and bounds |L| |y|
        assert np.all(abs(mag - M @ abs(yl)) <= 1e-16 * mag), op
        assert np.all(abs(L if op < 2 else L.T) @ abs(yl) <= mag + 1e-16 * mag), op
        scale = M @ abs(z) if op in (0, 2) else mag
        assert np.all(abs(z - dense[op]) <= 1e-16 * scale), op


@pytest.mark.parametrize("name", ["sun_n384", "sun_ragged", "giant_n512", "gran_only"])
def test_reference_matches_fp64_oracle_sweeps(name):
    """On the dense goldens the longdouble recurrence agrees with the FP64 oracle's sweeps at FP64 level."""
    gd = golden(f"dense_{name}.npz")
    terms = [g.SHOTerm(S0=r[0], w0=r[1], Q=r[2]) for r in gd["sho"]]
    delta = float(gd["delta"])
    k = g.StellarOscillatorKernel(terms=terms, delta=delta) if delta > 0 else g.TermSum(*terms)
    t = gd["t"]
    coef, W, ogp = _oracle_factor(k, t, gd["diag"])
    y = np.random.default_rng(2).standard_normal(len(t))
    fns = [oracle.solve_lower, oracle.matmul_lower, oracle.solve_upper, oracle.matmul_upper]
    for op, fn in enumerate(fns):
        ref = fn(ogp.t, ogp.c, ogp.U, ogp.W, y)
        (z, mag), = sweep_ref(op, [(coef, t, W, y)])
        if op in (1, 3):
            assert np.all(abs(ref - z) <= 1e-13 * mag), op
        else:
            assert np.max(abs(ref - z)) <= 1e-11 * np.max(abs(z)), op


@pytest.mark.parametrize("J", [2, 64, 172])
def test_reference_conditional_mean_matches_kernel_definition(kern, J):
    """The product-form sum equals K(t*, t) alpha with K from the kernel definition at moderate t."""
    k = kern(J)
    coef = KernelBatch([k]).coef
    rng = np.random.default_rng(J)
    t = np.sort(rng.uniform(0, 0.05, 120))
    ts = np.sort(np.concatenate([rng.uniform(-0.01, 0.06, 40), t[::7], t[[3, 3]]]))
    alpha = rng.standard_normal(len(t))
    mu, mag = cond_ref(coef, t, ts, alpha)
    ref = T.get_value((np.empty(0), np.empty(0), *coef.T), ts[:, None] - t[None, :]) @ alpha
    assert np.all(abs(mu - ref) <= 1e-13 * mag)


# ---- GPU helpers --------------------------------------------------------------------------------
def _factored(solver, kernels, ts, seed=0):
    """Factor a ragged batch (heteroscedastic diag) -> dict(kb, geom, t, d, W, w_off, items) with
    items[b] = (coef, t, W) of sequence b."""
    rng = np.random.default_rng(seed)
    kb = KernelBatch(kernels)
    lengths = [len(x) for x in ts]
    geom = Geometry.ragged(lengths)
    t = np.concatenate(ts) if lengths else np.empty(0)
    diag = np.concatenate([_diag(k, len(x), rng) for k, x in zip(kernels, ts)])
    d, W, w_off, logdet, status = solver.factor(kb, geom, t, diag)
    assert np.all(status == 0)
    items = []
    for b, k in enumerate(kernels):
        J2 = int(kb.J[b])
        items.append((kb.coef[kb.j_off[b]:kb.j_off[b + 1]], ts[b], W[w_off[b]:w_off[b] + lengths[b] * J2]))
    return dict(kb=kb, geom=geom, t=t, d=d, W=W, w_off=w_off, items=items, logdet=logdet, diag=diag)


def _split(x, n_off):
    return [x[n_off[b]:n_off[b + 1]] for b in range(len(n_off) - 1)]


def _check_sweep(op, items, ys, zs):
    """Every sequence of one sweep launch against the reference (see the module docstring)."""
    refs = sweep_ref(op, [it + (y,) for it, y in zip(items, ys)])
    if op in (0, 2):
        back = sweep_ref(op + 1, [it + (z,) for it, z in zip(items, zs)])
    for b, (z, (zr, mag)) in enumerate(zip(zs, refs)):
        if len(z) == 0:
            continue
        zl = np.asarray(z, dtype=np.float64).astype(LD)
        if op in (1, 3):
            _check("sweep_matmul", zl - zr, mag)
        else:
            Lz, mag_z = back[b]
            yl = np.asarray(ys[b], dtype=np.float64).astype(LD)
            _check("sweep_solve", Lz - yl, abs(yl) + mag_z)
            _check("sweep_solve_fwd", np.max(abs(zl - zr)), np.max(abs(zr)))


# ---- GPU: the four sweeps -----------------------------------------------------------------------
SHORT = [1, 2, 7, 8, 9, 15, 16, 17, 30, 31, 32, 33]
WIDTHS = [2, 10, 64, 172, 176, 192, 194, 258, 352]
WITH_4099 = {10, 192, 194, 352}       # widths that also sweep N = 4099 (on the mixed cadence)


@pytest.mark.gpu
@pytest.mark.parametrize("cadence", ["uniform", "mixed", "bjd"])
@pytest.mark.parametrize("J", WIDTHS)
def test_sweeps_vs_longdouble(solver, kern, J, cadence):
    """All four ops at one width (so the launch uses that width's build: 3 terms per lane up to J = 192,
    6 from J = 194), every short length and a long one, through the host path and through device
    buffers with Z aliasing Y in place."""
    import torch
    lengths = SHORT + [241] + ([4099] if (J in WITH_4099 and cadence == "mixed") else [])
    ts = [_times(cadence, n, seed=n) for n in lengths]
    f = _factored(solver, [kern(J)] * len(lengths), ts, seed=J)
    rng = np.random.default_rng(J + 1)
    Y = rng.standard_normal(len(f["t"]))
    ys = _split(Y, f["geom"].n_off)
    for op in range(4):
        Z = solver.sweep(op, f["kb"], f["geom"], f["w_off"], f["t"], f["W"], Y)
        buf = torch.from_numpy(Y.copy()).cuda()
        solver.sweep(op, f["kb"], f["geom"], f["w_off"], f["t"], f["W"], buf, Z=buf)
        assert np.array_equal(buf.cpu().numpy(), Z), op
        _check_sweep(op, f["items"], ys, _split(Z, f["geom"].n_off))


@pytest.mark.gpu
def test_sweep_batch_shape(solver, kern):
    """One launch that mixes J = 2, 172 and 300 (the narrow sequences run in the 6-per-lane build), with
    zero-length sequences between non-empty ones, three sequences that share one t and one W
    (t_off, w_off repeated), and a zero-length sequence last: nothing is written past its offset."""
    import torch
    widths = [2, 172, 300, 2, 172, 300, 172]
    lengths = [33, 0, 241, 0, 17, 9, 0]
    ts = [_times("mixed", n, seed=i) for i, n in enumerate(lengths)]
    kernels = [kern(J) for J in widths]
    f = _factored(solver, kernels, ts, seed=5)
    kb, geom = f["kb"], f["geom"]
    # three extra sequences on the t and W of sequence 2 (J = 300, N = 241)
    kb2 = _take(kb, list(range(len(widths))) + [2, 2, 2])
    n_off = np.concatenate([geom.n_off, geom.n_off[-1] + np.arange(1, 4) * lengths[2]])
    t_off = np.concatenate([geom.t_off, [geom.t_off[2]] * 3])
    geom2 = Geometry(n_off, t_off, geom.t_len)
    w_off2 = np.concatenate([f["w_off"], [f["w_off"][2]] * 3])
    items = f["items"] + [f["items"][2]] * 3
    rng = np.random.default_rng(6)
    total = int(n_off[-1])
    Y = rng.standard_normal(total)
    ys = _split(Y, n_off)
    for op in range(4):
        Yd = torch.from_numpy(Y).cuda()
        Zd = torch.full((total + 64,), np.nan, dtype=torch.float64, device="cuda")
        solver.sweep(op, kb2, geom2, w_off2, f["t"], f["W"], Yd, Z=Zd)
        Z = Zd.cpu().numpy()
        assert np.all(np.isnan(Z[total:])), op
        Z = Z[:total]
        assert np.array_equal(Z, solver.sweep(op, kb2, geom2, w_off2, f["t"], f["W"], Y)), op
        _check_sweep(op, items, ys, _split(Z, n_off))


@pytest.mark.gpu
@pytest.mark.parametrize("build", ["narrow", "wide"])
def test_sweep_placement_past_the_grid_cap(solver, kern, build):
    """2 * 65535 + 5 shuffled copies of seven short items: every CTA sweeps two or three sequences, and
    each copy is bit-identical to its item swept alone, for all four ops.  ``narrow`` mixes widths up to
    J = 192 (3 terms per lane), ``wide`` has a J = 300 item (6 terms per lane for all)."""
    widths = [2, 10, 64, 172, 192, 34, 100] if build == "narrow" else [2, 10, 64, 300, 192, 34, 100]
    lengths = [3, 8, 17, 40, 9, 31, 24]
    ts = [_times(["uniform", "mixed", "bjd"][i % 3], n, seed=i) for i, n in enumerate(lengths)]
    f = _factored(solver, [kern(J) for J in widths], ts, seed=7)
    rng = np.random.default_rng(8)
    ys = [rng.standard_normal(n) for n in lengths]
    B = 2 * 65535 + 5
    idx = np.concatenate([np.arange(7), rng.integers(0, 7, B - 7)])
    rng.shuffle(idx)
    lens = np.asarray(lengths)[idx]
    n_off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    geom = Geometry(n_off, f["geom"].t_off[idx], f["geom"].t_len)
    kb = _take(f["kb"], idx)
    w_off = f["w_off"][idx]
    Y = np.concatenate([ys[i] for i in idx])
    for op in range(4):
        alone = [solver.sweep(op, f["kb"].take([i]), Geometry.ragged([lengths[i]]), [0], ts[i],
                              f["items"][i][2], ys[i]) for i in range(7)]
        Z = solver.sweep(op, kb, geom, w_off, f["t"], f["W"], Y)
        ref = np.concatenate([alone[i] for i in idx])
        bad = np.flatnonzero(Z != ref)
        assert bad.size == 0, (op, int(np.searchsorted(n_off, bad[0], side="right") - 1))
        _check_sweep(op, f["items"], ys, alone)


# ---- GPU: the conditional mean ------------------------------------------------------------------
def _new_times(t, M, rng):
    """Sorted new times: every observed time (M = "all") or M of them, duplicates, points wholly before
    and wholly after the data, points in the 40-unit gaps, and random points inside the span."""
    gaps = np.flatnonzero(np.diff(t) > 30)
    special = [t[[0, 0, len(t) // 2, len(t) // 2, -1]], [t[0] - 50.0, t[0] - 1e-4, t[-1] + 1e-4, t[-1] + 50.0]]
    special += [t[i] + np.array([1e-3, 20.0, t[i + 1] - t[i] - 1e-3]) for i in gaps]
    special = np.concatenate(special)
    if M == "all":
        return np.sort(np.concatenate([t, special, rng.uniform(t[0], t[-1], 40)]))
    if M <= 2:
        return np.sort(special[[2, 3]][:M]) if M == 2 else t[[len(t) // 2]]
    pool = np.concatenate([special, rng.choice(t, min(len(t), M // 2), replace=False)])
    return np.sort(np.concatenate([pool, rng.uniform(t[0], t[-1], M - len(pool))]))


def _rows_to_check(ts, t, Jc, budget=3e7, seed=0):
    """Every new time, or -- where the direct sum would be too long -- the first and last eight, every
    point before / after the data or tied to a stamp, and a random sample."""
    M = len(ts)
    if M * len(t) * Jc <= budget:
        return np.arange(M)
    n = max(16, int(budget // (len(t) * Jc)))
    tied = np.flatnonzero(np.isin(ts, t) | (ts < t[0]) | (ts > t[-1]))
    rng = np.random.default_rng(seed)
    pick = np.concatenate([np.arange(8), np.arange(M - 8, M), rng.choice(tied, min(len(tied), n // 2), False),
                           rng.choice(M, n // 2, replace=False)])
    return np.unique(pick)


COND_CASES = [  # (Jc, N, M, cadence)
    (1, 1, "all", "mixed"), (1, 2000, 500, "mixed"), (64, 2, 2, "mixed"), (64, 300, 1, "uniform"),
    (128, 300, "all", "mixed"), (128, 2000, 500, "bjd"), (129, 300, 500, "bjd"), (129, 2, "all", "uniform"),
    (176, 300, "all", "bjd"), (176, 2000, 500, "mixed"), (176, 1, 2, "bjd")]


@pytest.mark.gpu
@pytest.mark.parametrize("Jc,N,M,cadence", COND_CASES)
def test_conditional_mean_vs_longdouble(solver, kern, Jc, N, M, cadence):
    """cond_mean_kernel at widths around its pass boundary (128 terms per pass), at N and M down to 1,
    with ties, duplicates, points outside the data and in gaps where every decay underflows."""
    rng = np.random.default_rng(Jc * 7 + N)
    coef = KernelBatch([kern(2 * Jc)]).coef
    t = _times(cadence, N, seed=N)
    ts = _new_times(t, M, rng)
    alpha = rng.standard_normal(N)
    mu = solver.conditional_mean(coef, t, ts, alpha)
    assert mu.shape == ts.shape
    rows = _rows_to_check(ts, t, Jc)
    ref, mag = cond_ref(coef, t, ts, alpha, rows)
    _check("cond_mean", mu[rows] - ref, mag)


@pytest.mark.gpu
@pytest.mark.parametrize("J", [258, 352])
def test_predict_at_new_times_wide_kernels(solver, kern, J):
    """GaussianProcess.predict(y, t=...) with a factored kernel of J = 258 / 352 (its apply_inverse runs
    the 6-per-lane sweeps), and with ``kernel=`` narrower and wider than the factored one; M = 0."""
    k = kern(J)
    rng = np.random.default_rng(J)
    N = 400
    t = _times("mixed", N, seed=1)
    diag = _diag(k, N, rng)
    y = rng.standard_normal(N) * np.sqrt(_k0(k))
    gp = g.GaussianProcess(k, t=t, diag=diag, solver=solver)
    alpha = gp.apply_inverse(y)
    coef = KernelBatch([k]).coef
    W = gp._W.cpu().numpy()[:N * J]
    (z, _), = sweep_ref(0, [(coef, t, W, y)])
    (a_ref, _), = sweep_ref(2, [(coef, t, W, z / gp._d.astype(LD))])
    _check("gp_alpha", np.max(abs(alpha - a_ref)), np.max(abs(a_ref)))
    ts = _new_times(t, "all", rng)
    for kp in (None, kern(64), kern(352) if J < 352 else kern(172)):
        mu = gp.predict(y, t=ts, kernel=kp)
        cp = coef if kp is None else KernelBatch([kp]).coef
        rows = _rows_to_check(ts, t, len(cp))
        ref, mag = cond_ref(cp, t, ts, alpha, rows)
        _check("cond_mean", mu[rows] - ref, mag)
    assert gp.predict(y, t=np.empty(0)).shape == (0,)
    assert solver.conditional_mean(coef, t, np.empty(0), alpha).shape == (0,)


# ---- GPU: k right-hand sides on one factor ------------------------------------------------------
def _virtual(f, k):
    """run_multi's virtual batch v = b k + r: kernels, geometry, w_off, the sequence of each v, d[v]."""
    idx = np.repeat(np.arange(f["kb"].B), k)
    lengths = np.diff(f["geom"].n_off)[idx]
    geom = Geometry(np.concatenate([[0], np.cumsum(lengths)]).astype(np.int64), f["geom"].t_off[idx],
                    f["geom"].t_len)
    ds = _split(f["d"], f["geom"].n_off)
    d_v = np.concatenate([ds[b] for b in idx]) if len(idx) else np.empty(0)
    return _take(f["kb"], idx), geom, f["w_off"][idx], idx, d_v


def _sweep_below_cap(solver, op, f, kb_v, geom_v, w_off_v, Y):
    """Solver.sweep over the virtual batch in launches of at most 65535 sequences (one CTA each)."""
    out = []
    for a in range(0, kb_v.B, 65535):
        s = np.arange(a, min(kb_v.B, a + 65535))
        n0 = geom_v.n_off[s[0]]
        geom = Geometry(geom_v.n_off[s[0]:s[-1] + 2] - n0, geom_v.t_off[s], geom_v.t_len)
        out.append(solver.sweep(op, _take(kb_v, s), geom, w_off_v[s], f["t"], f["W"],
                                Y[n0:geom_v.n_off[s[-1] + 1]]))
    return np.concatenate(out)


def _check_multi(solver, f, k, check_v, seed=0):
    """sample_multi (external normals: bit-identical to Solver.sweep(1) of sqrt(d) n; Philox: the host
    generator's draws through the longdouble matmul) and loglike_multi (quad against the longdouble
    solve) on the factored batch ``f``, k realisations each; longdouble checks for ``check_v``."""
    kb_v, geom_v, w_off_v, idx, d_v = _virtual(f, k)
    kb, geom, t, diag = f["kb"], f["geom"], f["t"], f["diag"]
    rng = np.random.default_rng(seed)
    total = int(geom_v.n_off[-1])
    nrm = rng.standard_normal(total)
    x, logdet, status = solver.sample_multi(kb, geom, t, k, diag, normals=nrm)
    assert np.all(status == 0) and np.array_equal(logdet, f["logdet"])
    assert np.array_equal(x, _sweep_below_cap(solver, 1, f, kb_v, geom_v, w_off_v, np.sqrt(d_v) * nrm))
    # Philox: realisation v = b k + r draws sequence seq0 + v
    seq0 = 1000
    xp, _, status = solver.sample_multi(kb, geom, t, k, diag, seed=seed, seq0=seq0)
    assert np.all(status == 0)
    lens = np.diff(geom_v.n_off)
    ys = [np.sqrt(d_v[geom_v.n_off[v]:geom_v.n_off[v + 1]]) * philox.normals(seed, seq0 + v, lens[v])
          for v in check_v]
    refs = sweep_ref(1, [f["items"][idx[v]] + (y,) for v, y in zip(check_v, ys)])
    for v, (zr, mag) in zip(check_v, refs):
        _check("multi_sample", xp[geom_v.n_off[v]:geom_v.n_off[v + 1]].astype(LD) - zr, mag)
    # loglike_multi: quad[v] = sum z^2 / d with z = L^-1 y_v
    yq = rng.standard_normal(total)
    ld, quad, status = solver.loglike_multi(kb, geom, t, yq, k, diag)
    assert np.all(status == 0) and np.array_equal(ld, f["logdet"])
    z = _sweep_below_cap(solver, 0, f, kb_v, geom_v, w_off_v, yq)
    starts = geom_v.n_off[:-1]
    q64 = np.add.reduceat(z * z / d_v, np.minimum(starts, max(total - 1, 0))) if total else np.zeros(len(idx))
    q64 = np.where(lens > 0, q64, 0.0)
    assert np.all(abs(quad - q64) <= 1e-13 * q64)
    refs = sweep_ref(0, [f["items"][idx[v]] + (yq[geom_v.n_off[v]:geom_v.n_off[v + 1]],) for v in check_v])
    for v, (zr, _) in zip(check_v, refs):
        dv = d_v[geom_v.n_off[v]:geom_v.n_off[v + 1]].astype(LD)
        qref = np.sum(zr * zr / dv)
        _check("quad", LD(quad[v]) - qref, qref)
    return x, xp


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3])
def test_multi_rhs_ragged_mixed_widths(solver, kern, k):
    """A ragged batch of J = 2 ... 194 (6-per-lane sweeps) with a zero-length sequence, k = 1 and 3."""
    widths = [2, 64, 194, 172, 10]
    lengths = [17, 241, 33, 0, 9]
    ts = [_times(["mixed", "bjd", "uniform"][i % 3], n, seed=i) for i, n in enumerate(lengths)]
    f = _factored(solver, [kern(J) for J in widths], ts, seed=k)
    _check_multi(solver, f, k, np.arange(len(widths) * k), seed=k)


@pytest.mark.gpu
def test_multi_rhs_past_the_grid_cap(solver, kern):
    """B k = 3 * 21846 = 65538 virtual sequences (N = 16): the sweeps' CTAs and prep / quad's grid-stride
    loops take realisations on both sides of index 65535; batch.sample(size=k) at that size."""
    k, N = 21846, 16
    widths = [2, 10, 64]
    ts = [_times(c, N, seed=i) for i, c in enumerate(["uniform", "mixed", "bjd"])]
    kernels = [kern(J) for J in widths]
    f = _factored(solver, kernels, ts, seed=3)
    check_v = [0, 1, k - 1, k, 2 * k - 1, 2 * k, 65533, 65534, 65535, 65536, 65537]
    x, xp = _check_multi(solver, f, k, check_v, seed=9)
    rows, status = batch.sample(kernels, f["t"], f["diag"], lengths=[N] * 3, seed=9, seq0=1000, size=k,
                                solver=solver, subtract_mean=False)
    assert np.all(status == 0) and np.array_equal(np.concatenate([r.ravel() for r in rows]), xp)
    rows_m, _ = batch.sample(kernels, f["t"], f["diag"], lengths=[N] * 3, seed=9, seq0=1000, size=k,
                             solver=solver)
    for r, rm in zip(rows, rows_m):
        assert np.array_equal(rm, r - r.mean(axis=0, keepdims=True))


@pytest.mark.gpu
def test_gp_sample_more_realisations_than_the_grid(solver, kern):
    """GaussianProcess.sample(size=70000) at N = 24: every realisation is dot_tril of its normals alone."""
    k = kern(64)
    N, size = 24, 70000
    t = _times("mixed", N, seed=4)
    rng = np.random.default_rng(4)
    gp = g.GaussianProcess(k, t=t, diag=_diag(k, N, rng), solver=solver)
    np.random.seed(11)
    x = gp.sample(size=size)
    np.random.seed(11)
    n = np.random.randn(N, size)
    full = gp.dot_tril(n)
    ref = full.T + gp._mean_value
    assert np.array_equal(x, ref - ref.mean(axis=0))
    cols = np.unique(np.concatenate([[0, 1, 65534, 65535, 65536, size - 1], rng.choice(size, 10, False)]))
    coef = KernelBatch([k]).coef
    W = gp._W.cpu().numpy()[:N * 64]
    refs = sweep_ref(1, [(coef, t, W, np.sqrt(gp._d) * n[:, c]) for c in cols])
    for c, (zr, mag) in zip(cols, refs):
        assert np.array_equal(full[:, c], gp.dot_tril(n[:, c])), c
        _check("sweep_matmul", full[:, c].astype(LD) - zr, mag)
