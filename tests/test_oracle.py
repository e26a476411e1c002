"""CPU tests of the oracle itself: the restated recurrences against dense Cholesky of the
kernel definition, against the committed golden vectors, and the term algebra against its
defining integrals and the reference's closed-form PSD."""
import numpy as np
import pytest

import oracle
from oracle import terms_oracle as T, dense
from conftest import golden

CASES = ["sun_n384", "sun_ragged", "giant_n512", "gran_only"]


def _scan(g):
    coeffs = T.sho_sum([tuple(r) for r in g["sho"]])
    return coeffs, T.scan_coefficients(coeffs, float(g["delta"]))


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_dense_golden(name):
    g = golden(f"dense_{name}.npz")
    coeffs, scan = _scan(g)
    gp = oracle.OracleGP(scan, g["t"], diag=g["diag"])
    assert gp.d[0] == pytest.approx(float(g["d0"]) + 0.0, rel=1e-14)
    assert gp.log_det == pytest.approx(float(g["logdet"]), rel=1e-11)
    assert gp.log_likelihood(g["y"]) == pytest.approx(float(g["loglike"]), rel=1e-10)
    x = gp.dot_tril(g["normals"])
    assert np.max(np.abs(x - g["dot_tril"])) <= 2e-9 * np.max(np.abs(g["dot_tril"]))
    ai = gp.apply_inverse(g["y"])
    assert np.max(np.abs(ai - g["apply_inverse"])) <= 1e-7 * np.max(np.abs(g["apply_inverse"]))


@pytest.mark.parametrize("name", CASES)
def test_stream_equals_materialised(name):
    """The fused streaming pass is the same arithmetic as matrices -> factor -> sweep."""
    g = golden(f"dense_{name}.npz")
    _, scan = _scan(g)
    gp = oracle.OracleGP(scan, g["t"], diag=g["diag"])
    logdet, quad, status = oracle.stream(0, scan, g["t"], g["y"], diag=g["diag"])
    assert status == 0
    assert logdet == pytest.approx(gp.log_det, rel=1e-13)   # np.sum is pairwise, the stream sequential
    ll = oracle.log_likelihood_from_stream(logdet, quad, len(g["t"]))
    assert ll == pytest.approx(gp.log_likelihood(g["y"]), rel=1e-13)
    x, _, _ = oracle.stream(1, scan, g["t"], g["normals"], diag=g["diag"])
    np.testing.assert_allclose(x, gp.dot_tril(g["normals"]), rtol=0, atol=1e-12 * np.max(np.abs(x)))


def test_matrix_sweeps_multi_rhs():
    g = golden("dense_gran_only.npz")
    _, scan = _scan(g)
    gp = oracle.OracleGP(scan, g["t"], diag=g["diag"])
    Y = np.random.default_rng(1).standard_normal((len(g["t"]), 3))
    Z = oracle.solve_lower(gp.t, gp.c, gp.U, gp.W, Y)
    back = oracle.matmul_lower(gp.t, gp.c, gp.U, gp.W, Z)
    np.testing.assert_allclose(back, Y, rtol=0, atol=1e-10)
    Zu = oracle.solve_upper(gp.t, gp.c, gp.U, gp.W, Y)
    np.testing.assert_allclose(oracle.matmul_upper(gp.t, gp.c, gp.U, gp.W, Zu), Y, rtol=0, atol=1e-10)
    for k in range(3):
        np.testing.assert_allclose(Z[:, k], oracle.solve_lower(gp.t, gp.c, gp.U, gp.W, Y[:, k]))


def test_non_positive_definite_is_reported():
    coeffs = T.sho_sum([(1.0, 2.0, 3.0)])
    scan = T.scan_coefficients(coeffs, None)
    t = np.array([0.0, 0.0, 1.0])   # duplicated time stamp, no jitter: singular
    with pytest.raises(oracle.LinAlgError):
        oracle.OracleGP(scan, t)
    _, _, status = oracle.stream(0, scan, t, np.ones(3))
    assert status == 2


def test_exposure_transform_matches_defining_integral():
    """A.4 closed forms = delta^-2 int (delta-|x|) k(tau+x) dx, on well-conditioned terms."""
    coeffs = T.sho_sum([(3.0, 40.0, 2.5), (1.0, 900.0, 30.0), (2.0, 5.0, 0.3)])
    delta = 7e-3
    for tau in [0.0, 2e-3, 6.9e-3, 7e-3, 1.1e-2, 0.3]:
        closed = T.get_value_convolved(coeffs, delta, tau)[0]
        quad = dense.exposure_integral(coeffs, delta, tau)
        assert closed == pytest.approx(quad, rel=2e-10), tau
    scan = T.scan_coefficients(coeffs, delta)
    k0 = np.sum(scan[0]) + np.sum(scan[2]) + scan[6]
    assert k0 == pytest.approx(dense.exposure_integral(coeffs, delta, 0.0), rel=2e-10)


def test_psd_golden_from_reference_closed_form():
    """Golden vectors produced by the reference's own ``_sho_psd`` (gadfly/core.py:33-41).

    celerite2's general (a, b, c, d) PSD formula (A.5) loses a factor ~min(Q^2, (w0^2/(w^2-w0^2))^2)
    of precision to cancellation next to a resonance (p-mode Q ~ 2.6e3 -> ~1e-9); the closed form
    does not.  So: 1e-12 below 800 uHz (far from every p-mode), 1e-8 inside the p-mode forest."""
    g = golden("ref_sho_psd.npz")
    coeffs = T.sho_sum([tuple(r) for r in g["params"]])
    far = g["omega"] < 2 * np.pi * 800.0
    for fn in (T.psd, oracle.psd):
        got = fn(coeffs, g["omega"])
        np.testing.assert_allclose(got[far], g["psd_sum"][far], rtol=1e-12)
        np.testing.assert_allclose(got, g["psd_sum"], rtol=1e-8)
    for row, idx in zip(g["psd_terms"], [0, 4, 5, 40, 85]):
        one = T.sho_sum([tuple(g["params"][idx])])
        # a single term also carries the rounding residue of (a c - b d) w^2 (exactly 0 in
        # exact arithmetic) far above its own w0: relative eps (w / w0)^2
        np.testing.assert_allclose(oracle.psd(one, g["omega"]), row, rtol=1e-8)
        np.testing.assert_allclose(T.sho_psd(g["omega"], *g["params"][idx]), row, rtol=1e-15)


def test_psd_exposure_sinc():
    coeffs = T.sho_sum([(3.0, 40.0, 2.5)])
    w = np.array([0.0, 1.0, 1e3, 1e5])
    np.testing.assert_allclose(oracle.psd(coeffs, w, 6e-5), T.psd_convolved(coeffs, 6e-5, w), rtol=1e-14)


def test_fast_build_agrees_with_reproducible_build():
    g = golden("dense_sun_n384.npz")
    _, scan = _scan(g)
    a = oracle.stream(0, scan, g["t"], g["y"], fast=False)
    b = oracle.stream(0, scan, g["t"], g["y"], fast=True)
    assert a[0] == pytest.approx(b[0], rel=1e-12) and a[1] == pytest.approx(b[1], rel=1e-9)
    n_off = np.array([0, 384, 768])
    out, x, status = oracle.stream_batch(0, n_off, [0, 0], [0, 86, 172], g["t"], np.tile(g["y"], 2),
                                         [scan[6]] * 2, *[np.tile(scan[i], 2) for i in (2, 3, 4, 5)],
                                         fast=False)
    assert status.tolist() == [0, 0] and out[0, 0] == a[0] and out[1, 1] == a[1]


# ---- ground truth from the kernel DEFINITION in extended precision (tools/make_golden_definition.py:
# (S0, w0, Q) -> dense exposure-integrated covariance by quadrature -> longdouble Cholesky; nothing of
# oracle/ or gadfly_b200/ is involved in producing it) ------------------------------------------------
# tolerances: (log-det, log-likelihood, samples and K^-1 y).  Measured deviations of the oracle: logL
# <= 2e-12, samples <= 5e-10 on the three well-conditioned cases; at the 1-min exposure 2.8e-9 on the
# samples (the slowest granulation term's a' carries celerite2's own FP64 cancellation, SURVEY.md 0.6).
DEF_CASES = [("def_solar_200s", 1e-10, 1e-10, 1e-9), ("def_subgiant", 1e-10, 1e-10, 1e-9),
             ("def_giant", 1e-10, 1e-10, 1e-9), ("def_solar_sc", 1e-9, 1e-10, 2e-8)]


@pytest.mark.parametrize("name,tol_ld,tol_ll,tol_x", DEF_CASES)
def test_oracle_matches_definition_golden(name, tol_ld, tol_ll, tol_x):
    g = golden(name + ".npz")
    coeffs = T.sho_sum(list(zip(g["S0"], g["w0"], g["Q"])))
    scan = T.scan_coefficients(coeffs, float(g["delta"]))
    # k(0) of the exposure-integrated kernel: sum a' + ddiag  (A.4)
    assert np.sum(scan[2]) + scan[6] == pytest.approx(float(g["k0"]), rel=10 * tol_ld)
    gp = oracle.OracleGP(scan, g["t"], diag=g["diag"])
    assert gp.log_det == pytest.approx(float(g["logdet"]), rel=tol_ld)
    assert gp.log_likelihood(g["y"]) == pytest.approx(float(g["logl"]), rel=tol_ll)
    x = gp.dot_tril(g["normals"])
    assert np.max(np.abs(x - g["x"])) <= tol_x * np.max(np.abs(g["x"]))
    ai = gp.apply_inverse(g["y"])
    assert np.max(np.abs(ai - g["alpha"])) <= tol_x * np.max(np.abs(g["alpha"]))
    # the fused streams
    logdet, quad, status = oracle.stream(0, scan, g["t"], g["y"], diag=g["diag"])
    assert status == 0 and quad == pytest.approx(float(g["quad"]), rel=100 * tol_ll)


# ---- exact relations the GPU conformance suite (tests/test_gpu_conformance.py) asserts of every scan
# kernel: the oracle obeys them too, so they are properties of the recurrence, not of one kernel -------
def _gappy_case(N=1500):
    g = golden("dense_sun_n384.npz")
    _, scan = _scan(g)
    rng = np.random.default_rng(1)
    t = np.cumsum(rng.choice([6e-5, 6e-5, 1.2e-4, 3e-3, 0.4], N))
    diag = np.full(N, 25.0)
    diag[:N // 3] = 40.0
    return scan, t, diag, rng.standard_normal(N) * 300.0, rng.standard_normal(N)


def test_oracle_amplitude_scaling_is_exact():
    """a', b', ddiag, diag times s = 2^e and y times 2^(e/2): quad and the samples bit-identical after
    the rescale, d -> d s, U -> U s, W -> W / s bit for bit, logdet -> logdet + N e ln 2."""
    scan, t, diag, y, nrm = _gappy_case()
    ar, cr, ac, bc, cc, dc, dd = scan
    N = len(t)
    ld0, q0, st0 = oracle.stream(0, scan, t, y, diag=diag)
    x0 = oracle.stream(1, scan, t, nrm, diag=diag)[0]
    gp0 = oracle.OracleGP(scan, t, diag=diag)
    assert st0 == 0
    for e in (-240, -128, 128, 240):
        s, r = 2.0 ** e, 2.0 ** (e // 2)
        sc = (ar * s, cr, ac * s, bc * s, cc, dc, dd * s)
        ld, q, st = oracle.stream(0, sc, t, y * r, diag=diag * s)
        x, ldx, _ = oracle.stream(1, sc, t, nrm, diag=diag * s)
        assert st == 0 and q == q0, e
        np.testing.assert_array_equal(x, x0 * r)
        want = ld0 + N * e * np.log(2.0)
        assert abs(ld - want) <= 1e-13 * abs(want) and ldx == ld, e
        gp = oracle.OracleGP(sc, t, diag=diag * s)
        np.testing.assert_array_equal(gp.d, gp0.d * s)
        np.testing.assert_array_equal(gp.U, gp0.U * s)
        np.testing.assert_array_equal(gp.W, gp0.W / s)
        np.testing.assert_array_equal(gp.dot_tril(nrm), gp0.dot_tril(nrm) * r)
        np.testing.assert_array_equal(gp.apply_inverse(y * r), gp0.apply_inverse(y) / r)


def test_oracle_time_scaling_is_exact():
    """t times 2^k with c, d divided by 2^k: logdet, quad, samples and the factor bit-identical."""
    scan, t, diag, y, nrm = _gappy_case()
    ar, cr, ac, bc, cc, dc, dd = scan
    ld0, q0, _ = oracle.stream(0, scan, t, y, diag=diag)
    x0 = oracle.stream(1, scan, t, nrm, diag=diag)[0]
    gp0 = oracle.OracleGP(scan, t, diag=diag)
    for k in (-10, 10):
        lam = 2.0 ** k
        sc = (ar, cr / lam, ac, bc, cc / lam, dc / lam, dd)
        ld, q, st = oracle.stream(0, sc, t * lam, y, diag=diag)
        assert st == 0 and ld == ld0 and q == q0, k
        np.testing.assert_array_equal(oracle.stream(1, sc, t * lam, nrm, diag=diag)[0], x0)
        gp = oracle.OracleGP(sc, t * lam, diag=diag)
        np.testing.assert_array_equal(gp.d, gp0.d)
        np.testing.assert_array_equal(gp.W, gp0.W)


def test_oracle_time_reversal_invariance():
    """(t_max - t) reversed, y and diag reversed: the same matrix up to a permutation, so logdet and
    quad agree to rounding (measured: 9e-13 and 2e-11 at this length)."""
    scan, t, diag, y, _ = _gappy_case(1 << 16)
    ld0, q0, _ = oracle.stream(0, scan, t, y, diag=diag, fast=True)
    ld, q, st = oracle.stream(0, scan, (t[-1] - t)[::-1], y[::-1], diag=diag[::-1], fast=True)
    assert st == 0
    assert ld == pytest.approx(ld0, rel=1e-10) and q == pytest.approx(q0, rel=1e-10)
