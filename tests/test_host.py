"""CPU tests of the host side: the hyper-parameter feeder, kernel objects, the C-ABI library's
symbol table, batch descriptors and sharding (incl. a world-size-2 gloo gather)."""
import ctypes
import os
import re
import subprocess
import sys
import warnings

import numpy as np
import pytest

import gadfly_b200 as g
from gadfly_b200 import batch, scale, solver, units as u
from conftest import ROOT, golden
from oracle import terms_oracle as T


# ---- feeder: reference gadfly/tests/test_core.py:52-73, test_sun.py:11-19 ----------------
def test_scaling_relations_to_solar():
    should_be_ones = np.array([
        scale.amplitude_with_wavelength('SOHO VIRGO', 5777 * u.K),
        scale.nu_max(1 * u.M_sun, 5777 * u.K, 1 * u.R_sun),
        scale.delta_nu(1 * u.M_sun, 1 * u.R_sun),
        scale.tau_gran(1.0, 5777.0, 1.0),
        scale.granulation_amplitude(1.0, 5777.0, 1.0),
        scale.p_mode_amplitudes(1.0, 5777.0, 1.0),
    ])
    np.testing.assert_allclose(should_be_ones, 1)
    assert scale.amplitude_with_wavelength('SOHO VIRGO', 5777 * u.K) == 1.0


def test_p_mode_frequencies_present():
    from gadfly_b200.sun import broomhall_p_mode_freqs
    nu, ell = broomhall_p_mode_freqs()
    assert len(nu) == 81 and np.bincount(ell).tolist() == [22, 21, 20, 18]
    # the reference's own check (gadfly/tests/test_sun.py:6-19)
    for f in [3033.886, 3082.471, 3098.327, 3160.028, 3168.773, 3217.916]:
        np.testing.assert_allclose(f, nu[np.argmin(np.abs(nu - f))])
    assert 900 < nu.min() < 1100 and 3900 < nu.max() < 4100


def test_for_sun_terms_match_reference_solar_fit():
    """for_star at exactly solar inputs: 5 granulation + 81 p-mode terms, granulation terms
    identical to the reference JSON, p-mode frequencies = 2 pi x the BiSON table."""
    hp = g.Hyperparameters.for_sun()
    assert len(hp) == 86
    ref = golden("ref_sho_psd.npz")["params"]
    got = np.array([[p['hyperparameters'][k] for k in ('S0', 'w0', 'Q')] for p in hp])
    np.testing.assert_allclose(got[:5], ref[:5], rtol=1e-14)
    np.testing.assert_allclose(got[5:, 1], ref[5:, 1], rtol=1e-14)
    assert np.all(got[:, 2] >= 0.5)          # complex (underdamped) terms only
    assert np.all(got[:, 0] > 0)
    k = g.SolarOscillatorKernel(texp=1 * u.min, bandpass='SOHO VIRGO')
    assert k.J == 172 and k.delta == pytest.approx(6e-5)


@pytest.mark.parametrize("star,nterms", [((0.9, 10.0, 4919.0, 52.3), 62), ((1.0, 1.0, 5777.0, 1.0), 86)])
def test_for_star_term_counts(star, nterms):
    hp = g.Hyperparameters.for_star(*star, bandpass='SOHO VIRGO', quiet=True)
    assert len(hp) == nterms


def test_kernel_defaults_warn_and_add():
    hp = g.Hyperparameters.for_sun()
    with pytest.warns(g.GadflyUserWarning):
        k = g.StellarOscillatorKernel(hp)
    assert k.delta == pytest.approx(6e-5)
    shot = g.ShotNoiseKernel(S0=2.0, w0=g.ShotNoiseKernel.w0, Q=0.5)
    both = k + shot
    assert isinstance(both, g.StellarOscillatorKernel)
    assert len(both.term.terms) == 87 and both.delta == k.delta and both.J == 174
    assert both.name == "Shot noise"


def test_term_algebra_matches_oracle(solar_kernel):
    sho = [(t.S0, t.w0, t.Q) for t in solar_kernel.term.terms]
    coeffs = T.sho_sum(sho)
    for a, b in zip(solar_kernel.base_coefficients(), coeffs):
        np.testing.assert_array_equal(a, b)
    mine = solar_kernel.scan_coefficients()
    ref = T.scan_coefficients(coeffs, solar_kernel.delta)
    for a, b in zip(mine[:6], ref[:6]):
        np.testing.assert_array_equal(a, b)      # bit-identical: same expression order
    assert mine[6] == ref[6]
    ar, cr, _, _, _, _ = g.SHOTerm(S0=1.0, w0=2.0, Q=0.3).get_coefficients()
    assert len(ar) == 2 and len(cr) == 2


def test_kernel_batch_layout(solar_kernel, giant_kernel):
    kb = solver.KernelBatch([solar_kernel, giant_kernel, g.SHOTerm(S0=1.0, w0=2.0, Q=0.3)])
    assert kb.j_off.tolist() == [0, 86, 148, 150] and kb.J.tolist() == [172, 124, 4]
    assert kb.coef.shape == (150, 4) and kb.base.shape == (150, 4)
    assert kb.delta.tolist() == [6e-5, 6e-5, 0.0] and kb.ddiag[2] == 0.0
    assert np.all(kb.coef[148:, 1] == 0) and np.all(kb.coef[148:, 3] == 0)   # real terms
    sub = kb.take([1, 1, 0])
    assert sub.j_off.tolist() == [0, 62, 124, 210]
    np.testing.assert_array_equal(sub.coef[:62], kb.coef[86:148])


# ---- the C ABI ---------------------------------------------------------------------------
def test_library_exports_every_declared_symbol(built):
    header = open(os.path.join(ROOT, "include", "gadfly_b200.h")).read()
    declared = set(re.findall(r"\b(gf_[a-z_0-9]+)\s*\(", header))
    assert declared == set(solver._SIGNATURES), declared ^ set(solver._SIGNATURES)
    lib = ctypes.CDLL(built)
    for name in declared:
        assert hasattr(lib, name), name
    out = subprocess.run(["nm", "-D", "--defined-only", built], capture_output=True, text=True).stdout
    exported = set(re.findall(r" T (gf_[a-z_0-9]+)", out))
    assert declared <= exported
    assert solver.load_library() is not None


def test_library_has_sm100a_code(built):
    out = subprocess.run(["cuobjdump", "-lelf", built], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_cpu_fallback_when_library_missing(tmp_path):
    with pytest.raises(solver.SolverUnavailable):
        solver.load_library(str(tmp_path / "libmissing.so"))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "gadfly_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f
                assert "liboracle" not in src, f


# ---- sharding ----------------------------------------------------------------------------
def test_shard_bounds_balance_cost():
    cost = np.array([1.0] * 10 + [10.0] * 2)
    b = batch.shard_bounds(cost, 2)
    assert b[0] == 0 and b[-1] == 12 and abs(cost[:b[1]].sum() - cost[b[1]:].sum()) <= 10
    for world in (1, 2, 3, 8):
        b = batch.shard_bounds(np.ones(100), world)
        assert np.all(np.diff(b) >= 100 // world) and b[-1] == 100
    assert batch.shard(7, 2, 4) == (4, 5) or sum(hi - lo for lo, hi in [batch.shard(7, r, 4) for r in range(4)]) == 7
    assert batch.shard_bounds([], 4).tolist() == [0] * 5


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {root!r})
import numpy as np
import torch.distributed as dist
from gadfly_b200 import batch
dist.init_process_group("gloo", init_method="tcp://127.0.0.1:{port}", rank=int(sys.argv[1]), world_size=2)
rank = dist.get_rank()
B = 11
cost = np.arange(1, B + 1, dtype=float)
lo, hi = batch.shard(B, rank, 2, cost)
local = np.arange(lo, hi, dtype=np.float64) * 1.5        # stands in for per-unit logL
full = batch.gather_concat(local)
status = batch.gather_concat(np.full(hi - lo, rank, dtype=np.int32))
assert full.tolist() == (np.arange(B) * 1.5).tolist(), full
assert status.tolist() == [0] * batch.shard(B, 0, 2, cost)[1] + [1] * (B - batch.shard(B, 0, 2, cost)[1])
# with the shard boundaries known to every rank (no size exchange), and a torch tensor as input
import torch
bounds = batch.shard_bounds(cost, 2)
full2 = batch.gather_concat(torch.as_tensor(local), bounds=bounds)
assert full2.tolist() == full.tolist()
# an empty shard on one rank
e = batch.gather_concat(np.arange(3.0) if rank == 0 else np.empty(0))
assert e.tolist() == [0.0, 1.0, 2.0]
dist.barrier(); dist.destroy_process_group()
print("ok", rank, lo, hi)
"""


def test_gather_world_size_2_gloo(tmp_path):
    port = 29000 + os.getpid() % 2000
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER.format(root=ROOT, port=port))
    procs = [subprocess.Popen([sys.executable, str(script), str(r)], stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=180)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "ok" in o


# ---- facade argument checking that needs no GPU -----------------------------------------
def test_gp_usage_before_compute_raises(solar_kernel):
    gp = g.GaussianProcess(solar_kernel)
    with pytest.raises(RuntimeError):
        gp.log_likelihood(np.zeros(3))
    with pytest.raises(RuntimeError):
        gp.sample()
    with pytest.raises(ValueError):
        gp.compute(np.array([0.0, 2.0, 1.0]))
    with pytest.raises(ValueError):
        gp.compute(np.zeros((2, 2)))


def test_sample_mean_subtraction_refuses_async(solar_kernel):
    """batch.sample subtracts the mean on the host: with FLAG_ASYNC the draws are not there yet."""
    t = np.arange(16) * 6e-5
    for size in (None, 3):
        with pytest.raises(ValueError, match="FLAG_ASYNC"):
            batch.sample([solar_kernel], t, size=size, flags=solver.FLAG_ASYNC)


def test_power_spectrum_fft_normalisation():
    rng = np.random.default_rng(0)
    t = np.arange(4096) / 1440.0                # 1-min cadence in days
    flux = rng.standard_normal(4096) * 100.0
    ps = g.PowerSpectrum.from_light_curve(t, flux)
    d = 60e-6
    assert ps.frequency[0] == pytest.approx(1 / (4096 * d)) and len(ps.power) == 2048
    # Parseval with the reference's normalisation (gadfly/psd.py:576-586)
    assert np.sum(ps.power) * 2 / (d / np.sqrt(2 * np.pi)) == pytest.approx(np.sum(flux ** 2), rel=0.02)
    b = ps.bin(10)
    assert len(b.frequency) == 10 and b.error is not None
    assert len(ps.cutout(100 * u.uHz, 1000 * u.uHz).frequency) < len(ps.frequency)


def test_batched_feeder_matches_per_star():
    """gadfly_b200/feeder.py (SURVEY 8f-2) against Hyperparameters.for_star + StellarOscillatorKernel
    + KernelBatch star by star: same terms kept, coefficients to a few ulp (the diagonal correction
    is a cancelling sum: compared on the scale of k(0))."""
    import warnings
    from gadfly_b200 import feeder
    stars = [(1.0, 1.0, 5777.0, 1.0), (0.9, 10.0, 4919.0, 52.3), (1.32, 11.26, 4923.0, 66.8),
             (1.1, 1.6, 6100.0, 3.2), (2.0, 20.7, 4364.0, 146.0), (0.9, 1.4, 5500.0, 2.2)]
    M, R, T, L = (np.array(x) for x in zip(*stars))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        kernels = [g.StellarOscillatorKernel(
            g.Hyperparameters.for_star(m, r, t, l, bandpass='SOHO VIRGO', quiet=True), texp=1 * u.min)
            for m, r, t, l in stars]
    from gadfly_b200.solver import KernelBatch
    ref = KernelBatch(kernels)
    hpb = feeder.for_stars(M, R, T, L)
    got = feeder.kernel_batch_from_sho(hpb, kernels[0].delta)
    assert np.array_equal(got.j_off, ref.j_off)
    assert got.j_off[1] == 86 and got.j_off[2] - got.j_off[1] == 62      # Sun, KIC 9333184
    np.testing.assert_allclose(got.base, ref.base, rtol=1e-11)
    np.testing.assert_allclose(got.coef, ref.coef, rtol=1e-11)
    k0 = np.array([ref.coef[ref.j_off[b]:ref.j_off[b + 1], 0].sum() for b in range(ref.B)])
    assert np.all(np.abs(got.ddiag - ref.ddiag) <= 1e-9 * k0)
    assert np.array_equal(got.delta, ref.delta)
    # the reference's list-of-dicts view of one star
    sun = hpb.star(0)
    assert len(sun) == 86 and sun[0]['hyperparameters']['Q'] == pytest.approx(0.6)
    # one-call form, and the alpha override
    kb = KernelBatch.for_stars(M, R, T, L, texp_s=60.0)
    np.testing.assert_allclose(kb.coef, ref.coef, rtol=1e-11)
    kb2 = KernelBatch.for_stars(M, R, T, L, alpha=2.0)
    gran = slice(0, 5)
    np.testing.assert_allclose(kb2.base[gran, 0], 2.0 * kb.base[gran, 0], rtol=1e-13)

    # a tabulated (non-flat) bandpass: the batched amplitude ratio equals the per-star quadrature
    class Band:
        wavelength = np.linspace(0.4, 0.9, 200) * u.um
        transmittance = np.exp(-0.5 * ((np.linspace(0.4, 0.9, 200) - 0.65) / 0.1) ** 2)
        mean_wavelength = 0.65 * u.um
    many = scale.amplitude_with_wavelength_many(Band, T)
    one = np.array([scale.amplitude_with_wavelength(Band, t) for t in T])
    np.testing.assert_allclose(many, one, rtol=1e-14)
    assert np.array_equal(scale.amplitude_with_wavelength_many('SOHO VIRGO', T), np.ones(len(T)))


def test_get_value_matches_oracle_and_defining_integral(solar_kernel):
    """Term.get_value / TermConvolution.get_value (celerite2 API used by the predictive variance):
    both branches of the exposure-integrated kernel against the oracle, k(0) against the scan's
    diagonal, and one overlapping-exposure lag against the defining integral."""
    from oracle import dense
    base = solar_kernel.base_coefficients()
    delta = solar_kernel.delta
    tau = np.concatenate([np.linspace(0.0, 0.99 * delta, 7), [delta], np.linspace(1.01 * delta, 0.3, 40)])
    got = solar_kernel.get_value(tau)
    np.testing.assert_allclose(got, T.get_value_convolved(base, delta, tau), rtol=1e-10)
    np.testing.assert_allclose(solar_kernel.get_value(-tau), got, rtol=0)           # even in tau
    scan = solar_kernel.scan_coefficients()
    assert got[0] == pytest.approx(np.sum(scan[2]) + scan[6], rel=1e-8)               # k(0) = sum a' + ddiag
    assert solar_kernel.get_value(0.4 * delta) == pytest.approx(
        float(dense.exposure_integral(base, delta, 0.4 * delta)), rel=1e-7)
    plain = solar_kernel.term
    np.testing.assert_allclose(plain.get_value(tau), T.get_value(plain.base_coefficients(), tau), rtol=1e-13)
    over = g.SHOTerm(S0=3.0, w0=2.0, Q=0.3)                                          # real terms
    np.testing.assert_allclose(over.get_value(tau), T.get_value(over.base_coefficients(), tau), rtol=1e-13)
    assert solar_kernel.get_value(np.zeros((2, 3))).shape == (2, 3)


def test_for_star_matches_independent_evaluation():
    """(S0, w0, Q) of ``Hyperparameters.for_star`` against tests/golden/for_star.json: the scaling
    relations of the reference (gadfly/core.py:107-333, scale.py) evaluated independently, scalar by
    scalar in 40-digit mpmath, from the reference's own data files (tools/make_forstar_fixture.py);
    the per-star path and the batched feeder."""
    import json
    import os
    import warnings
    import gadfly_b200 as g
    from gadfly_b200 import feeder
    with open(os.path.join(os.path.dirname(__file__), "golden", "for_star.json")) as fh:
        stars = json.load(fh)["stars"]
    assert stars["Sun"]["n_terms"] == 86 and stars["KIC 9333184"]["n_terms"] == 62
    names = list(stars)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        hpb = feeder.for_stars(*[[stars[n][k] for n in names]
                                 for k in ("mass", "radius", "temperature", "luminosity")])
        for b, name in enumerate(names):
            st = stars[name]
            hp = g.Hyperparameters.for_star(st["mass"], st["radius"], st["temperature"], st["luminosity"],
                                            bandpass="SOHO VIRGO")
            assert len(hp) == st["n_terms"]
            for key in ("S0", "w0", "Q"):
                got = np.array([p["hyperparameters"][key] for p in hp])
                np.testing.assert_allclose(got, st[key], rtol=1e-12, err_msg=f"{name} {key}")
            sl = slice(hpb.j_off[b], hpb.j_off[b + 1])
            for key, arr in (("S0", hpb.S0), ("w0", hpb.w0), ("Q", hpb.Q)):
                np.testing.assert_allclose(arr[sl], st[key], rtol=1e-12, err_msg=f"batched {name} {key}")


def test_bench_dump_output_sample_dtype_and_size(tmp_path):
    """bench.py --dump-outputs: an array longer than DUMP_ELEMS is stored as the same seeded sample of
    its elements whatever its type (numpy / torch) and shape, every array in float64, and the twelve
    arrays the bench writes stay under 64 MB."""
    import torch
    import bench
    big = np.arange(3 * bench.DUMP_ELEMS, dtype=np.float64) * 0.5
    bench.dump_output(str(tmp_path / "a"), "x", big)
    bench.dump_output(str(tmp_path / "b"), "x", torch.as_tensor(big).reshape(3, -1))
    a, b = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "b" / "x.npy")
    assert a.dtype == np.float64 and a.shape == (bench.DUMP_ELEMS,)
    np.testing.assert_array_equal(a, b)
    assert np.all(np.diff(a) > 0) and np.all(np.isin(a, big))        # distinct input elements, in order
    assert 12 * os.path.getsize(tmp_path / "a" / "x.npy") < 64 << 20
    bench.dump_output(str(tmp_path / "a"), "status", torch.tensor([0, 2, -1], dtype=torch.int32))
    s = np.load(tmp_path / "a" / "status.npy")
    assert s.dtype == np.float64 and s.tolist() == [0.0, 2.0, -1.0]


def test_bench_rejects_bad_arguments(monkeypatch):
    import bench
    for argv in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "d"]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
        with pytest.raises(SystemExit):
            bench.parse()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "5", "--dump-outputs", "d"])
    a = bench.parse()
    assert a.steps == 5 and a.dump_outputs == "d"


def test_oracle_build_in_read_only_tree_is_private(tmp_path, monkeypatch):
    """Without a current build in oracle/_build and without write access to oracle/, the oracle is
    compiled into a new private temporary directory per call: nothing goes into the tree, and no
    build is shared with another process or checkout."""
    import shutil
    import oracle
    tree = tmp_path / "oracle"
    tree.mkdir()
    for f in ("Makefile", "celerite_oracle.c"):
        shutil.copy(os.path.join(ROOT, "oracle", f), tree / f)
    monkeypatch.setattr(oracle, "_HERE", str(tree))
    tree.chmod(0o555)
    if os.getuid() == 0:                        # permission bits do not bind root
        monkeypatch.setattr(oracle.os, "access", lambda path, mode: False)
    paths = []
    try:
        paths = [oracle.build(fast=False), oracle.build(fast=False)]
        assert paths[0] != paths[1]
        for p in paths:
            d = os.path.dirname(p)
            assert not p.startswith(str(tree)) and os.stat(d).st_mode & 0o077 == 0
            assert os.stat(d).st_uid == os.getuid()
            ctypes.CDLL(p).orc_max_threads()
        assert sorted(os.listdir(tree)) == ["Makefile", "celerite_oracle.c"]
    finally:
        tree.chmod(0o755)
        for p in paths:
            shutil.rmtree(os.path.dirname(p), ignore_errors=True)


def test_bin_ranges_match_host_binning():
    """The index ranges handed to the device binning kernel are scipy.stats.binned_statistic's bins
    (what ``bin_power_spectrum`` uses on the host): every point in exactly one bin, the last edge
    closed on the right, points on an inner edge in the bin to its right."""
    from gadfly_b200 import psd as P
    rng = np.random.default_rng(1)
    for axis in (np.log10(np.fft.rfftfreq(5000, 6e-5)[1:]), np.sort(rng.uniform(0, 10, 777)),
                 np.linspace(0.0, 1.0, 101)):
        for bins in (1, 7, 15, 100):
            edges, lo, cnt = P.bin_ranges(axis, bins)
            assert cnt.sum() == len(axis) and np.all(lo[1:] == lo[:-1] + cnt[:-1]) and lo[0] == 0
            which = np.searchsorted(edges, axis, side='right') - 1
            which[axis == edges[-1]] = bins - 1
            for k in range(bins):
                assert np.array_equal(np.flatnonzero(which == k), np.arange(lo[k], lo[k] + cnt[k]))
