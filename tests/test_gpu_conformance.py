"""Conformance of every scan path (csrc/scan_fast.cu, scan_small.cu, scan_blk.cu, and scan_ref.cu with
its register store "scan_ref" and its L2 store "scan_wide") to relations that hold EXACTLY, independent
of any reference implementation, plus the dispatch and length edges against the oracle.

* Amplitude: a', b', ddiag and diag times s = 2^e, y times 2^(e/2).  Every product and sum of the
  recurrence scales by a power of two, so IEEE rounding commutes with it: quad and the samples are
  bit-identical (after the rescale), d -> d s and W -> W / s bit for bit, and
  logdet -> logdet + N e ln 2.  Flux in ppm puts the pivots near 2^4 ... 2^16; other flux units move
  them by many binades, and a kernel that multiplies raw pivots overflows there.
* Time: t times 2^k, c and d divided by 2^k leaves every phase d t and decay c dt bit-identical.  An
  absolute time constant in the producer's path decisions (cadence tables, renormalisation) would
  show up here.
* Reversal: t -> (t_max - t) reversed and y reversed is the same covariance up to a permutation, so
  logdet and quad agree -- at a length where dense Cholesky is out of reach.
* Batch placement: the scans are persistent (CTAs / warps claim sequences from a queue and reuse
  shared memory, ring phases and flags between sequences); a sequence's result must not depend on
  which sequences ran before it on the same CTA.
* State stores: scan_ref.cu's two stores give a J <= 176 sequence the same bits.

Every case asserts which kernel served it (``Solver.last_scan_path``): a path added to ``PATHS`` is
covered by every parametrised case below."""
import ctypes
from collections import namedtuple

import numpy as np
import pytest

import gadfly_b200 as g
from gadfly_b200 import batch, solver as S
from gadfly_b200.solver import Geometry, KernelBatch
import oracle

pytestmark = pytest.mark.gpu
RTOL = 1e-9
LN2 = float(np.log(2.0))
EXPS = [-240, -128, -64, 64, 128, 240]

Path = namedtuple("Path", "flags widths modes")
ALL_MODES = ("loglike", "sample", "factor")
# name: (flags that select it, three state widths J a case may use, entry points it serves).  The
# LAST width is the one a single-kernel case uses; every width on its own selects the same path.
PATHS = {
    "scan_fast": Path(0, (34, 100, 172), ALL_MODES),
    "scan_small": Path(0, (18, 26, 32), ALL_MODES),
    "scan_ref": Path(S.FLAG_REFERENCE_ORDER, (10, 100, 172), ALL_MODES),
    "scan_wide": Path(0, (240, 300, 178), ALL_MODES),
    "scan_blk": Path(S.FLAG_BLOCKED, (10, 100, 172), ("loglike", "sample")),
}
PATH_MODES = [(p, m) for p in PATHS for m in PATHS[p].modes]


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


def _gappy(N, seed):
    rng = np.random.default_rng(seed)
    return np.cumsum(rng.choice([6e-5, 6e-5, 1.2e-4, 3e-3, 0.4], N))


def _cadence(name, seed=3):
    """Cadences that take the producer through its paths: the uniform 1-min table path; cadence
    changes, jitter inside and outside the first-order window and gaps; BJD-like absolute stamps."""
    if name == "uniform":
        return np.arange(2000) * 6e-5
    if name == "mixed":
        rng = np.random.default_rng(seed)
        dt = np.concatenate([
            np.full(200, 6e-5), np.full(150, 1.8e-3),
            np.full(100, 6e-5) * (1 + 1e-13 * rng.standard_normal(100)),
            np.full(100, 6e-5) * (1 + 1e-3 * rng.standard_normal(100)),
            [0.5], np.full(60, 6e-5), [40.0], np.full(60, 6e-5)])
        return np.cumsum(dt)
    assert name == "bjd"
    return 2.1e5 + np.arange(1500) * 6e-5


def _scaled(kernels, amp=None, lam=None):
    """KernelBatch of ``kernels`` with sequence b's a', b', ddiag times amp[b] and c, d divided by lam[b]."""
    kb = KernelBatch(kernels)
    for b in range(kb.B):
        rows = slice(int(kb.j_off[b]), int(kb.j_off[b + 1]))
        if amp is not None:
            kb.coef[rows, :2] *= amp[b]
            kb.ddiag[b] *= amp[b]
        if lam is not None:
            kb.coef[rows, 2:] /= lam[b]
    return kb


class _AmpKernel:
    """A kernel times s (what KernelBatch and GaussianProcess read of a kernel)."""

    def __init__(self, k, s):
        self.k, self.s = k, s

    @property
    def exposure(self):
        return self.k.exposure

    def scan_coefficients(self):
        ar, cr, ac, bc, cc, dc, dd = self.k.scan_coefficients()
        return ar * self.s, cr, ac * self.s, bc * self.s, cc, dc, dd * self.s

    def base_coefficients(self):
        ar, cr, ac, bc, cc, dc = self.k.base_coefficients()
        return ar * self.s, cr, ac * self.s, bc * self.s, cc, dc


def _run(solver, path, mode, kb, geom, t, data, diag, flags=0):
    """One scan call of ``mode`` on ``path``; asserts that ``path`` served it."""
    flags |= PATHS[path].flags
    if mode == "loglike":
        ld, q, st = solver.loglike(kb, geom, t, data, diag, flags=flags)
        out = dict(logdet=ld, quad=q, status=st)
    elif mode == "sample":
        x, ld, st = solver.sample(kb, geom, t, diag, normals=data, flags=flags)
        out = dict(x=x, logdet=ld, status=st)
    else:
        d, W, w_off, ld, st = solver.factor(kb, geom, t, diag, flags=flags)
        out = dict(d=d, W=W, w_off=w_off, logdet=ld, status=st)
    assert solver.last_scan_path() == path
    return out


def _seq(geom, b):
    return slice(int(geom.n_off[b]), int(geom.n_off[b + 1]))


def _wseq(out, geom, kb, b):
    w0 = int(out["w_off"][b])
    return slice(w0, w0 + int(geom.n_off[b + 1] - geom.n_off[b]) * int(kb.J[b]))


def _maxrel(a, b):
    return np.max(np.abs(np.asarray(a) - np.asarray(b))) / np.max(np.abs(b))


def _assert_logdet_shift(logdet, ld0, N, exps):
    for b, e in enumerate(exps, start=1):
        want = ld0 + N * e * LN2
        assert np.isfinite(logdet[b]) and abs(logdet[b] - want) <= 1e-13 * abs(want), (e, logdet[b], want)


# ---- a. amplitude ------------------------------------------------------------------------------
@pytest.mark.parametrize("path,mode", PATH_MODES)
def test_amplitude_scaling_is_exact(solver, kern, path, mode):
    k = kern(PATHS[path].widths[-1])
    N = 3000
    t = _gappy(N, 1)
    scales = [1.0] + [2.0 ** e for e in EXPS]
    roots = [1.0] + [2.0 ** (e // 2) for e in EXPS]
    B = len(scales)
    kb = _scaled([k] * B, amp=scales)
    geom = Geometry.shared_t(B, N)
    dg = np.full(N, 1e-3 * _k0(k))
    diag = np.concatenate([dg * s for s in scales])
    v = np.random.default_rng(2).standard_normal(N)
    data = {"loglike": np.concatenate([v * np.sqrt(_k0(k)) * r for r in roots]),
            "sample": np.tile(v, B), "factor": None}[mode]
    out = _run(solver, path, mode, kb, geom, t, data, diag)
    assert out["status"].tolist() == [0] * B
    _assert_logdet_shift(out["logdet"], out["logdet"][0], N, EXPS)
    for b in range(1, B):
        if mode == "loglike":
            assert out["quad"][b] == out["quad"][0], (EXPS[b - 1], out["quad"][b], out["quad"][0])
        elif mode == "sample":
            np.testing.assert_array_equal(out["x"][_seq(geom, b)], out["x"][_seq(geom, 0)] * roots[b])
        else:
            np.testing.assert_array_equal(out["d"][_seq(geom, b)], out["d"][_seq(geom, 0)] * scales[b])
            np.testing.assert_array_equal(out["W"][_wseq(out, geom, kb, b)],
                                          out["W"][_wseq(out, geom, kb, 0)] / scales[b])


def _amp_setup(kern, N=2000):
    k = kern(172)
    t = _gappy(N, 4)
    scales = [1.0] + [2.0 ** e for e in EXPS]
    roots = [1.0] + [2.0 ** (e // 2) for e in EXPS]
    dg = np.full(N, 1e-3 * _k0(k))
    y = np.random.default_rng(5).standard_normal(N) * np.sqrt(_k0(k))
    return k, t, scales, roots, dg, y


def test_amplitude_scaling_shared_y(solver, kern):
    """FLAG_SHARED_Y: y and diag addressed through t_off (each scaled copy on its own time block)."""
    k, t, scales, roots, dg, y = _amp_setup(kern)
    N, B = len(t), len(scales)
    kb = _scaled([k] * B, amp=scales)
    geom = Geometry.ragged([N] * B)
    ld, q, st = solver.loglike(kb, geom, np.tile(t, B), np.concatenate([y * r for r in roots]),
                               np.concatenate([dg * s for s in scales]), flags=S.FLAG_SHARED_Y)
    assert solver.last_scan_path() == "scan_fast"
    assert st.tolist() == [0] * B
    _assert_logdet_shift(ld, ld[0], N, EXPS)
    assert q.tolist() == [q[0]] * B


def test_amplitude_scaling_multi_rhs(solver, kern):
    """gf_sample_multi / gf_loglike_multi: the factor scan, then k sweeps per sequence on it."""
    k, t, scales, roots, dg, y = _amp_setup(kern)
    N, B, kk = len(t), len(scales), 3
    kb = _scaled([k] * B, amp=scales)
    geom = Geometry.shared_t(B, N)
    diag = np.concatenate([dg * s for s in scales])
    nrm = np.random.default_rng(6).standard_normal(kk * N)
    x, ld, st = solver.sample_multi(kb, geom, t, kk, diag, normals=np.tile(nrm, B))
    assert solver.last_scan_path() == "scan_fast"
    assert st.tolist() == [0] * B
    _assert_logdet_shift(ld, ld[0], N, EXPS)
    x = x.reshape(B, kk * N)
    for b in range(1, B):
        np.testing.assert_array_equal(x[b], x[0] * roots[b])
    ys = np.tile(y, kk) * 1.0
    ld2, q, st2 = solver.loglike_multi(kb, geom, t, np.concatenate([ys * r for r in roots]), kk, diag)
    assert solver.last_scan_path() == "scan_fast"
    assert st2.tolist() == [0] * B
    _assert_logdet_shift(ld2, ld2[0], N, EXPS)
    q = q.reshape(B, kk)
    for b in range(1, B):
        np.testing.assert_array_equal(q[b], q[0])


def test_amplitude_scaling_sweeps_on_stored_factor(solver, kern):
    """The four O(N J) sweeps on the stored factor: L = I + tril(U W^T) is invariant (U -> U s,
    W -> W / s), so every sweep of y 2^(e/2) is the sweep of y times 2^(e/2), bit for bit."""
    k, t, scales, roots, dg, y = _amp_setup(kern)
    N, B = len(t), len(scales)
    kb = _scaled([k] * B, amp=scales)
    geom = Geometry.shared_t(B, N)
    d, W, w_off, ld, st = solver.factor(kb, geom, t, np.concatenate([dg * s for s in scales]))
    assert solver.last_scan_path() == "scan_fast"
    assert st.tolist() == [0] * B
    Y = np.concatenate([y * r for r in roots])
    for op in range(4):
        Z = solver.sweep(op, kb, geom, w_off, t, W, Y).reshape(B, N)
        for b in range(1, B):
            np.testing.assert_array_equal(Z[b], Z[0] * roots[b], err_msg=f"op {op}, e = {EXPS[b - 1]}")


def test_amplitude_scaling_gaussian_process(solver, kern):
    """GaussianProcess.compute (factor on the default path), log_likelihood, dot_tril,
    apply_inverse and predict at the observed and at new times: mu scales by 2^(e/2)."""
    k, t, scales, roots, dg, y = _amp_setup(kern, N=1500)
    N = len(t)
    v = np.random.default_rng(7).standard_normal(N)
    tnew = np.sort(np.random.default_rng(8).uniform(t[0], t[-1], 300))
    gp0 = g.GaussianProcess(_AmpKernel(k, 1.0), t=t, diag=dg, solver=solver)
    assert solver.last_scan_path() == "scan_fast"
    ll0, mu0, mt0 = gp0.log_likelihood(y), gp0.predict(y), gp0.predict(y, t=tnew)
    dt0, ai0 = gp0.dot_tril(v), gp0.apply_inverse(y)
    for e, s, r in zip(EXPS, scales[1:], roots[1:]):
        gp = g.GaussianProcess(_AmpKernel(k, s), t=t, diag=dg * s, solver=solver)
        assert solver.last_scan_path() == "scan_fast"
        want = gp0._log_det + N * e * LN2
        assert np.isfinite(gp._log_det) and abs(gp._log_det - want) <= 1e-13 * abs(want), e
        # log L is a difference of terms of size |logdet|: relative to that
        assert abs(gp.log_likelihood(y * r) - (ll0 - 0.5 * N * e * LN2)) <= 1e-13 * abs(want), e
        np.testing.assert_array_equal(gp.predict(y * r), mu0 * r, err_msg=str(e))
        np.testing.assert_array_equal(gp.predict(y * r, t=tnew), mt0 * r, err_msg=str(e))
        np.testing.assert_array_equal(gp.dot_tril(v), dt0 * r, err_msg=str(e))
        np.testing.assert_array_equal(gp.apply_inverse(y * r), ai0 * (r / s), err_msg=str(e))


# ---- b. scan_blk's exponent sum past 2^31 -------------------------------------------------------
def test_blocked_scan_exponent_sum_past_2_31(solver, solar_kernel):
    """N = 2^24 pivots near 2^(+-240): the sum of their binary exponents passes 2^31.  The three
    scales share one launch (one sequence per CTA); no oracle needed."""
    N = 1 << 24
    t = np.arange(N) * 6e-5
    exps = [240, -240]
    scales = [1.0] + [2.0 ** e for e in exps]
    roots = [1.0] + [2.0 ** (e // 2) for e in exps]
    kb = _scaled([solar_kernel] * 3, amp=scales)
    y = np.random.default_rng(9).standard_normal(N) * 300.0
    ld, q, st = solver.loglike(kb, Geometry.shared_t(3, N), t, np.concatenate([y * r for r in roots]),
                               np.concatenate([np.full(N, 25.0 * s) for s in scales]), flags=S.FLAG_BLOCKED)
    assert solver.last_scan_path() == "scan_blk"
    assert st.tolist() == [0, 0, 0]
    _assert_logdet_shift(ld, ld[0], N, exps)
    assert q[1] == q[0] and q[2] == q[0]


# ---- c. time scaling ---------------------------------------------------------------------------
@pytest.mark.parametrize("cadence", ["uniform", "mixed", "bjd"])
@pytest.mark.parametrize("path", list(PATHS))
def test_time_scaling_is_exact(solver, kern, path, cadence):
    k = kern(PATHS[path].widths[-1])
    t = _cadence(cadence)
    N = len(t)
    lams = [1.0, 2.0 ** -10, 2.0 ** 10]
    B = len(lams)
    kb = _scaled([k] * B, lam=lams)
    geom = Geometry.ragged([N] * B)
    ts = np.concatenate([t * lam for lam in lams])
    dg = np.full(N, 1e-3 * _k0(k))
    diag = np.tile(dg, B)
    v = np.random.default_rng(10).standard_normal(N)
    for mode in PATHS[path].modes:
        data = {"loglike": np.tile(v * np.sqrt(_k0(k)), B), "sample": np.tile(v, B), "factor": None}[mode]
        out = _run(solver, path, mode, kb, geom, ts, data, diag)
        assert out["status"].tolist() == [0] * B, mode
        assert out["logdet"].tolist() == [out["logdet"][0]] * B, mode
        for b in range(1, B):
            if mode == "loglike":
                assert out["quad"][b] == out["quad"][0]
            elif mode == "sample":
                np.testing.assert_array_equal(out["x"][_seq(geom, b)], out["x"][_seq(geom, 0)])
            else:
                np.testing.assert_array_equal(out["d"][_seq(geom, b)], out["d"][_seq(geom, 0)])
                np.testing.assert_array_equal(out["W"][_wseq(out, geom, kb, b)], out["W"][_wseq(out, geom, kb, 0)])


# ---- d. batch placement ------------------------------------------------------------------------
Item = namedtuple("Item", "J t diag v ok")


def _items(kern, path):
    """Seven distinct sequences: three widths, lengths 0 / 1 / 9 / 65 / 1000 / 4097, gappy cadences,
    and one that is not positive definite (diag negative from the middle)."""
    J = PATHS[path].widths
    rng = np.random.default_rng(11)
    specs = [(J[0], 0, "u"), (J[1], 1, "u"), (J[2], 9, "u"), (J[0], 65, "g"), (J[1], 1000, "u"),
             (J[0], 4097, "g"), (J[2], 65, "npd")]
    items = []
    for Jw, N, kind in specs:
        k0 = _k0(kern(Jw))
        t = _gappy(N, int(rng.integers(1 << 30))) if kind == "g" else 3.0 + np.arange(N) * 6e-5
        dg = np.full(N, 1e-3 * k0)
        if kind == "npd":
            dg[N // 2:] = -10.0 * k0
        items.append(Item(Jw, t, dg, rng.standard_normal(N), kind != "npd"))
    return items


def _batch_of(kern, items, idx):
    kb = KernelBatch([kern(items[i].J) for i in sorted(set(idx))])
    pos = {i: p for p, i in enumerate(sorted(set(idx)))}
    kb = kb.take([pos[i] for i in idx])
    geom = Geometry.ragged([len(items[i].t) for i in idx])
    cat = lambda f: np.concatenate([f(items[i]) for i in idx])    # noqa: E731
    return kb, geom, cat(lambda it: it.t), cat(lambda it: it.diag), cat(lambda it: it.v)


@pytest.mark.parametrize("path,mode", PATH_MODES)
def test_result_independent_of_batch_placement(solver, kern, path, mode):
    """B = 2 x SMs + 5 sequences (scan_small: more than its 12 warps x SMs) drawn from seven items in
    a shuffled order: every copy of an item bit-identical to every other and to the item run alone.
    One launch each; normals are passed, so the Philox sequence id does not enter."""
    items = _items(kern, path)
    sm = solver.device_info()["sm_count"]
    B = (12 * sm + 5) if path == "scan_small" else (2 * sm + 5)
    rng = np.random.default_rng(12)
    idx = np.concatenate([np.arange(len(items)), rng.integers(0, len(items), B - len(items))])
    rng.shuffle(idx)
    idx = [int(i) for i in idx]

    def call(ix):
        kb, geom, t, diag, v = _batch_of(kern, items, ix)
        data = {"loglike": v * 300.0, "sample": v, "factor": None}[mode]
        return kb, geom, _run(solver, path, mode, kb, geom, t, data, diag)

    kb, geom, out = call(idx)
    alone = [call([i]) for i in range(len(items))]
    for b, i in enumerate(idx):
        kb1, geom1, ref = alone[i]
        assert out["status"][b] == ref["status"][0], (b, i)
        assert (out["status"][b] == 0) == items[i].ok, (b, i)
        if not items[i].ok:
            continue
        assert out["logdet"][b] == ref["logdet"][0], (b, i)
        if len(items[i].t) == 0:
            assert out["logdet"][b] == 0.0
        if mode == "loglike":
            assert out["quad"][b] == ref["quad"][0], (b, i)
        elif mode == "sample":
            np.testing.assert_array_equal(out["x"][_seq(geom, b)], ref["x"], err_msg=f"{b} {i}")
        else:
            np.testing.assert_array_equal(out["d"][_seq(geom, b)], ref["d"], err_msg=f"{b} {i}")
            np.testing.assert_array_equal(out["W"][_wseq(out, geom, kb, b)], ref["W"][_wseq(ref, geom1, kb1, 0)],
                                          err_msg=f"{b} {i}")


# ---- e. dispatch and length edges --------------------------------------------------------------
def _against_oracle(solver, path, kernels, t, diag, flags=0, seed=13):
    """loglike, sample and factor of ``kernels`` on the shared cadence t against the oracle."""
    B, N = len(kernels), len(t)
    kb = KernelBatch(kernels)
    geom = Geometry.shared_t(B, N)
    rng = np.random.default_rng(seed)
    nrm = [rng.standard_normal(N) for _ in range(B)]
    scans = [k.scan_coefficients() for k in kernels]
    refs = [oracle.stream(1, sc, t, n, diag=dg) for sc, n, dg in zip(scans, nrm, diag)]
    modes = PATHS[path].modes
    x = _run(solver, path, "sample", kb, geom, t, np.concatenate(nrm), np.concatenate(diag), flags)
    y = np.concatenate([r[0] for r in refs])
    ll = _run(solver, path, "loglike", kb, geom, t, y, np.concatenate(diag), flags)
    fa = _run(solver, path, "factor", kb, geom, t, None, np.concatenate(diag), flags) if "factor" in modes else None
    for b in range(B):
        xr, ldr, st = refs[b]
        assert st == 0
        assert x["status"][b] == 0 and ll["status"][b] == 0
        assert _maxrel(x["x"][_seq(geom, b)], xr) <= RTOL, b
        o_ld, o_q, _ = oracle.stream(0, scans[b], t, xr, diag=diag[b])
        assert ll["logdet"][b] == pytest.approx(o_ld, rel=RTOL) and ll["quad"][b] == pytest.approx(o_q, rel=RTOL), b
        assert x["logdet"][b] == pytest.approx(o_ld, rel=RTOL)
        if fa is not None:
            assert fa["status"][b] == 0 and fa["logdet"][b] == pytest.approx(o_ld, rel=RTOL)
            assert _maxrel(fa["d"][_seq(geom, b)], oracle.OracleGP(scans[b], t, diag=diag[b]).d) <= RTOL


@pytest.mark.parametrize("J,path", [(32, "scan_small"), (34, "scan_fast"), (174, "scan_fast"), (176, "scan_fast"),
                                    (178, "scan_wide"), (350, "scan_wide"), (352, "scan_wide")])
def test_dispatch_width_edges(solver, kern, J, path):
    k = kern(J)
    t = _gappy(300, J)
    _against_oracle(solver, path, [k], t, [np.full(300, 1e-3 * _k0(k))])


@pytest.mark.parametrize("J,path", [(34, "scan_fast"), (176, "scan_fast"), (178, "scan_wide")])
def test_dispatch_two_term_sequence_beside_a_wider_one(solver, kern, J, path):
    ks = [kern(2), kern(J)]
    t = _gappy(257, J + 1)
    _against_oracle(solver, path, ks, t, [np.full(257, 1e-3 * _k0(k)) for k in ks])


def test_dispatch_refuses_wider_than_352(solver, kern, solar_kernel):
    too_wide = g.StellarOscillatorKernel(terms=list(kern(352).term.terms) + [g.SHOTerm(S0=1.0, w0=50.0, Q=3.0)],
                                         delta=solar_kernel.delta)
    assert too_wide.J == 354
    with pytest.raises(ValueError):
        KernelBatch([too_wide])
    # the raw C ABI: GF_E_TOO_WIDE, before anything is launched
    N, Jc = 16, 177
    n_off = np.array([0, N], dtype=np.int64)
    t_off = np.zeros(1, dtype=np.int64)
    j_off = np.array([0, Jc], dtype=np.int64)
    coef = np.ascontiguousarray(np.tile(KernelBatch([solar_kernel]).coef[:1], (Jc, 1)))
    ddiag, t, y = np.zeros(1), np.arange(N) * 6e-5, np.zeros(N)
    ld, q, x, st = np.zeros(1), np.zeros(1), np.zeros(N), np.zeros(1, dtype=np.int32)
    p64 = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))     # noqa: E731
    lib = solver._lib
    rc = lib.gf_loglike_batched(solver._h, 1, p64(n_off), p64(t_off), p64(j_off), t.ctypes.data, N, y.ctypes.data,
                                None, coef.ctypes.data, ddiag.ctypes.data, ld.ctypes.data, q.ctypes.data,
                                st.ctypes.data, 0)
    assert rc == -3                      # GF_E_TOO_WIDE
    rc = lib.gf_sample_batched(solver._h, 1, p64(n_off), p64(t_off), p64(j_off), t.ctypes.data, N, None,
                               coef.ctypes.data, ddiag.ctypes.data, None, 0, 0, x.ctypes.data, ld.ctypes.data,
                               st.ctypes.data, 0)
    assert rc == -3


LENGTHS = [0, 1, 2, 7, 8, 9, 63, 64, 65, 129]


@pytest.mark.parametrize("path", list(PATHS))
def test_length_edges(solver, kern, path):
    """N around the row-ring half and the log flush (8), scan_blk's block (4), the 32-row flushes and
    the 64-step renormalisation, in one ragged batch, against the oracle; N = 0 gives zeros."""
    k = kern(PATHS[path].widths[-1])
    B = len(LENGTHS)
    ts = [_gappy(n, 20 + n) if n % 2 else np.arange(n) * 6e-5 for n in LENGTHS]
    dgs = [np.full(n, 1e-3 * _k0(k)) for n in LENGTHS]
    rng = np.random.default_rng(14)
    nrm = [rng.standard_normal(n) for n in LENGTHS]
    kb = KernelBatch([k] * B)
    geom = Geometry.ragged(LENGTHS)
    t, diag = np.concatenate(ts), np.concatenate(dgs)
    sc = k.scan_coefficients()
    x = _run(solver, path, "sample", kb, geom, t, np.concatenate(nrm), diag)
    xr = [oracle.stream(1, sc, ts[b], nrm[b], diag=dgs[b])[0] if LENGTHS[b] else np.zeros(0) for b in range(B)]
    ll = _run(solver, path, "loglike", kb, geom, t, np.concatenate(xr), diag)
    fa = _run(solver, path, "factor", kb, geom, t, None, diag) if "factor" in PATHS[path].modes else None
    for b, n in enumerate(LENGTHS):
        assert x["status"][b] == 0 and ll["status"][b] == 0, n
        if n == 0:
            assert ll["logdet"][b] == 0.0 and ll["quad"][b] == 0.0 and x["logdet"][b] == 0.0
            continue
        assert _maxrel(x["x"][_seq(geom, b)], xr[b]) <= RTOL, n
        o_ld, o_q, _ = oracle.stream(0, sc, ts[b], xr[b], diag=dgs[b])
        assert ll["logdet"][b] == pytest.approx(o_ld, rel=RTOL, abs=1e-12), n
        assert ll["quad"][b] == pytest.approx(o_q, rel=RTOL), n
        if fa is not None:
            assert fa["status"][b] == 0
            assert _maxrel(fa["d"][_seq(geom, b)], oracle.OracleGP(sc, ts[b], diag=dgs[b]).d) <= RTOL, n


@pytest.mark.parametrize("path,mode", PATH_MODES)
def test_zero_length_sequence_writes_nothing(solver, kern, path, mode):
    """A sequence of length 0 between two others: status 0, logdet 0, quad 0, no element of the
    outputs written (NaN-filled device buffers with a guard band past n_off[B]), neighbours
    bit-identical to the batch without it."""
    import torch
    k = kern(PATHS[path].widths[-1])
    rng = np.random.default_rng(15)
    lens = [50, 0, 70]
    t = np.concatenate([_gappy(50, 1), np.zeros(0), _gappy(70, 2)])
    dg = np.full(120, 1e-3 * _k0(k))
    v = rng.standard_normal(120)
    data = {"loglike": v * 300.0, "sample": v, "factor": None}[mode]
    guard = 64
    dev = f"cuda:{solver.device}"
    flags = PATHS[path].flags

    def go(lengths):
        B = len(lengths)
        kb, geom = KernelBatch([k] * B), Geometry.ragged(lengths)
        total = int(geom.n_off[-1])
        if mode == "loglike":
            ld = torch.full((B + guard,), float("nan"), dtype=torch.float64, device=dev)
            q = torch.full((B + guard,), float("nan"), dtype=torch.float64, device=dev)
            _, _, st = solver.loglike(kb, geom, t, data, dg, logdet=ld, quad=q, flags=flags)
            res = dict(logdet=ld, quad=q, status=st)
        elif mode == "sample":
            x = torch.full((total + guard,), float("nan"), dtype=torch.float64, device=dev)
            _, ld, st = solver.sample(kb, geom, t, dg, normals=data, out=x, flags=flags)
            res = dict(x=x, logdet=ld, status=st)
        else:
            w_total = int(np.sum(np.asarray(lengths) * kb.J))
            d = torch.full((total + guard,), float("nan"), dtype=torch.float64, device=dev)
            W = torch.full((w_total + guard,), float("nan"), dtype=torch.float64, device=dev)
            w_off = np.concatenate([[0], np.cumsum(np.asarray(lengths) * kb.J)])[:-1]
            _, _, _, ld, st = solver.factor(kb, geom, t, dg, d=d, W=W, w_off=w_off, flags=flags)
            res = dict(d=d, W=W, logdet=ld, status=st, w_total=w_total)
        torch.cuda.synchronize(dev)
        assert solver.last_scan_path() == path
        return {key: (val.cpu().numpy() if hasattr(val, "cpu") else val) for key, val in res.items()}

    r3, r2 = go(lens), go([50, 70])
    assert r3["status"].tolist() == [0, 0, 0] and r2["status"].tolist() == [0, 0]
    assert r3["logdet"][1] == 0.0
    assert r3["logdet"][0] == r2["logdet"][0] and r3["logdet"][2] == r2["logdet"][1]
    if mode == "loglike":
        assert r3["quad"][1] == 0.0 and r3["quad"][0] == r2["quad"][0] and r3["quad"][2] == r2["quad"][1]
        assert np.all(np.isnan(r3["logdet"][3:])) and np.all(np.isnan(r3["quad"][3:]))
    elif mode == "sample":
        np.testing.assert_array_equal(r3["x"], r2["x"])          # guard band included: NaN == NaN here
        assert np.all(np.isnan(r3["x"][120:])) and not np.any(np.isnan(r3["x"][:120]))
    else:
        np.testing.assert_array_equal(r3["d"], r2["d"])
        np.testing.assert_array_equal(r3["W"], r2["W"])
        assert np.all(np.isnan(r3["d"][120:])) and np.all(np.isnan(r3["W"][r3["w_total"]:]))
        assert not np.any(np.isnan(r3["W"][:r3["w_total"]]))


# ---- f. status ---------------------------------------------------------------------------------
@pytest.mark.parametrize("path,mode", PATH_MODES)
def test_status_first_non_positive_pivot(solver, kern, path, mode):
    """diag turning negative at row 0, at a middle row and at row N - 1, between healthy sequences:
    status = the oracle's 1 + index of the first non-positive pivot; the healthy neighbours are
    bit-identical to a run in which nothing fails.  (Outputs after a failure are unspecified.)"""
    k = kern(PATHS[path].widths[-1])
    k0 = _k0(k)
    N = 200
    t = _gappy(N, 16)
    sc = k.scan_coefficients()
    bad_rows = {1: 0, 3: 97, 5: N - 1}
    B = 7
    dg = np.full(N, 1e-3 * k0)
    clean = [dg] * B
    broken = [dg] * B
    for b, row in bad_rows.items():
        d = dg.copy()
        d[row:] = -10.0 * k0
        broken[b] = d
    v = np.random.default_rng(17).standard_normal(B * N)
    data = {"loglike": v * np.sqrt(k0), "sample": v, "factor": None}[mode]
    kb, geom = KernelBatch([k] * B), Geometry.shared_t(B, N)
    ok = _run(solver, path, mode, kb, geom, t, data, np.concatenate(clean))
    bad = _run(solver, path, mode, kb, geom, t, data, np.concatenate(broken))
    assert ok["status"].tolist() == [0] * B
    for b in range(B):
        if b in bad_rows:
            want = oracle.stream(0, sc, t, np.zeros(N), diag=broken[b])[2]
            assert want == bad_rows[b] + 1
            assert bad["status"][b] == want, (b, bad["status"][b], want)
            continue
        assert bad["status"][b] == 0 and bad["logdet"][b] == ok["logdet"][b], b
        if mode == "loglike":
            assert bad["quad"][b] == ok["quad"][b]
        elif mode == "sample":
            np.testing.assert_array_equal(bad["x"][_seq(geom, b)], ok["x"][_seq(geom, b)])
        else:
            np.testing.assert_array_equal(bad["d"][_seq(geom, b)], ok["d"][_seq(geom, b)])
            np.testing.assert_array_equal(bad["W"][_wseq(bad, geom, kb, b)], ok["W"][_wseq(ok, geom, kb, b)])


# ---- g. time reversal --------------------------------------------------------------------------
@pytest.mark.parametrize("path", list(PATHS))
def test_time_reversal_invariance(solver, kern, path):
    """N = 2^16 with gaps: logdet and quad of the reversed sequence (t_max - t, reversed; y
    reversed) equal the forward ones -- the same matrix up to a permutation.  y is a draw of the
    process (on the same path), so quad is well conditioned (the oracle agrees with itself to 1e-12
    on the log-det and 1e-11 on quad here)."""
    k = kern(PATHS[path].widths[-1])
    N = 1 << 16
    t = _gappy(N, 18)
    tr = (t[-1] - t)[::-1].copy()
    dgr = np.full(N, 1e-3 * _k0(k))
    dgr[: N // 3] *= 2.0                  # a diagonal that is not constant, reversed with the data
    y = _run(solver, path, "sample", KernelBatch([k]), Geometry.shared_t(1, N), t,
             np.random.default_rng(19).standard_normal(N), dgr)["x"]
    kb = KernelBatch([k, k])
    geom = Geometry.ragged([N, N])
    out = _run(solver, path, "loglike", kb, geom, np.concatenate([t, tr]), np.concatenate([y, y[::-1]]),
               np.concatenate([dgr, dgr[::-1]]))
    assert out["status"].tolist() == [0, 0]
    assert out["logdet"][1] == pytest.approx(out["logdet"][0], rel=1e-10)
    assert out["quad"][1] == pytest.approx(out["quad"][0], rel=1e-10)


# ---- batch.sample(size=k) --------------------------------------------------------------------
@pytest.mark.parametrize("path", [p for p in PATHS if "factor" in PATHS[p].modes])
def test_sample_size_k_matches_oracle(solver, kern, path):
    """``batch.sample(..., size=k)``: k realisations per unit on one factor, with the reference's
    mean subtraction across the realisations (celerite2 sample(size=k) is [k, N]; gadfly subtracts
    its mean over axis 0), against OracleGP.sample_from_normals on the same normals."""
    k = kern(PATHS[path].widths[-1])
    N, B, kk = 300, 2, 5
    t = _gappy(N, 21)
    dg = np.full(N, 1e-3 * _k0(k))
    nrm = np.random.default_rng(22).standard_normal(B * kk * N)
    rows, st = batch.sample([k] * B, t, np.tile(dg, (B, 1)), normals=nrm, size=kk, solver=solver,
                            flags=PATHS[path].flags)
    assert solver.last_scan_path() == path
    assert st.tolist() == [0] * B and rows.shape == (B, kk, N)
    ogp = oracle.OracleGP(k.scan_coefficients(), t, diag=dg)
    for b in range(B):
        n = nrm[b * kk * N:(b + 1) * kk * N].reshape(kk, N).T          # [N, k], as np.random.randn(N, k)
        ref = ogp.sample_from_normals(n)                                # [k, N]
        scale = np.max(np.abs(ogp.dot_tril(n)))
        assert np.max(np.abs(rows[b] - ref)) <= RTOL * scale, b
        np.testing.assert_allclose(rows[b].mean(axis=0), 0.0, atol=1e-12 * scale)


# ---- h. the two state stores of the reference-order kernel ---------------------------------------
@pytest.mark.parametrize("mode", ["loglike", "sample", "philox", "factor"])
@pytest.mark.parametrize("J", [100, 172])
def test_reference_order_state_stores_agree(solver, kern, J, mode):
    """scan_ref_kernel keeps the J x J state in registers ("scan_ref") or, in a batch with a kernel
    wider than 176, in L2-resident scratch ("scan_wide").  Both stores run the same per-tile
    expressions and folds in the same order, so a J <= 176 sequence run alone under
    FLAG_REFERENCE_ORDER and beside a J = 300 kernel gives the same bits.  ("philox": sampling with
    the normals drawn in the kernel; the sequence is index 0 of both batches.)"""
    N, n2 = 3000, 64
    k, wide = kern(J), kern(300)
    t = _gappy(N, 23)
    dg = 1e-3 * _k0(k) * (1.0 + np.random.default_rng(24).uniform(0.0, 2.0, N))
    dg2 = np.full(n2, 1e-3 * _k0(wide))
    v = np.random.default_rng(25).standard_normal(N + n2)
    scan_mode = "sample" if mode == "philox" else mode
    data = {"loglike": np.concatenate([v[:N] * np.sqrt(_k0(k)), v[N:] * np.sqrt(_k0(wide))]),
            "sample": v, "philox": None, "factor": None}[mode]
    alone = _run(solver, "scan_ref", scan_mode, KernelBatch([k]), Geometry.shared_t(1, N), t,
                 None if data is None else data[:N], dg)
    kb, geom = KernelBatch([k, wide]), Geometry.ragged([N, n2])
    both = _run(solver, "scan_wide", scan_mode, kb, geom, np.concatenate([t, _gappy(n2, 26)]), data,
                np.concatenate([dg, dg2]))
    assert alone["status"][0] == 0 and both["status"].tolist() == [0, 0]
    assert both["logdet"][0] == alone["logdet"][0]
    if mode == "loglike":
        assert both["quad"][0] == alone["quad"][0]
    elif scan_mode == "sample":
        np.testing.assert_array_equal(both["x"][:N], alone["x"])
    else:
        np.testing.assert_array_equal(both["d"][:N], alone["d"])
        np.testing.assert_array_equal(both["W"][:N * J], alone["W"])
