"""Staging of every C ABI entry point: each buffer may be pageable host memory, pinned host memory or
device memory, and a call may block or return at once (FLAG_ASYNC).  Whatever the mix, the outputs must
be bit-identical to those of the all-pageable blocking call, and the call must count the same launches
and report the same scan path.

One row per entry point.  Each row is run
- with every buffer pinned, then with every buffer on the device (except the arrays the library reads
  on the host: the offset arrays, bin power's lo / cnt and the j_off gf_feed_stars writes), then with
  device inputs and pageable outputs, then with pageable inputs and device outputs, and all pageable;
  each once blocking and once with FLAG_ASYNC followed by gf_synchronize;
- as three FLAG_ASYNC calls back to back with different inputs and distinct pageable outputs, issued
  while the handle's compute stream is held, then one gf_synchronize: both buffers of every staging
  slot and the pinned ring of small outputs are in use.

The entry points are called through ``Solver._lib`` with raw addresses, so that every buffer of every
entry point (the feeders' too) can be placed anywhere."""
import ctypes
import functools

import numpy as np
import pytest

from gadfly_b200 import solver as S
from gadfly_b200.feeder import solar_tables
from gadfly_b200.solver import Geometry, KernelBatch

pytestmark = pytest.mark.gpu

_i64p = ctypes.POINTER(ctypes.c_int64)

# scan rows: three light curves of one time grid, at overlapping offsets
LENGTHS = [300, 217, 401]
T_OFF = np.array([0, 100, 50], dtype=np.int64)
T_LEN = 500
N_OFF = np.concatenate([[0], np.cumsum(LENGTHS)]).astype(np.int64)
TOTAL = int(N_OFF[-1])
B = len(LENGTHS)
K = 3                                    # right-hand sides of the multi rows


class Row:
    def __init__(self, name, make, call, launches, path=None, host=()):
        self.name, self.make, self.call = name, make, call
        self.launches, self.path, self.host = launches, path, set(host)

    def __repr__(self):
        return self.name


@functools.lru_cache(maxsize=None)
def _scan_setup():
    import gadfly_b200 as g
    kern = g.SolarOscillatorKernel(texp=1 * g.units.min, bandpass='SOHO VIRGO')
    kb = KernelBatch([kern] * B)
    t = np.arange(T_LEN) * 6e-5
    return kb, t


def _rng(row, variant):
    return np.random.default_rng([sum(map(ord, row)), variant])


def _scan_inputs(name, variant, y_len=TOTAL):
    kb, t = _scan_setup()
    rng = _rng(name, variant)
    return dict(n_off=N_OFF, t_off=T_OFF, j_off=kb.j_off, t=t, coef=kb.coef, ddiag=kb.ddiag,
                diag=rng.uniform(20.0, 40.0, y_len)), rng


def _out(shape, dtype=np.float64):
    return np.full(shape, -7, dtype=dtype)


# ---- rows -----------------------------------------------------------------------------------------
def make_loglike(variant, shared=False):
    inp, rng = _scan_inputs("loglike" + "s" * shared, variant, T_LEN if shared else TOTAL)
    inp["y"] = rng.standard_normal(T_LEN if shared else TOTAL) * 300.0
    return inp, dict(logdet=_out(B), quad=_out(B), status=_out(B, np.int32)), {}


def call_loglike(L, h, p, q, s, flags):
    return L.gf_loglike_batched(h, B, q("n_off"), q("t_off"), q("j_off"), p("t"), T_LEN, p("y"), p("diag"),
                                p("coef"), p("ddiag"), p("logdet"), p("quad"), p("status"), flags)


def make_sample(variant, philox=False):
    inp, rng = _scan_inputs("sample" + "p" * philox, variant)
    if not philox:
        inp["normals"] = rng.standard_normal(TOTAL)
    return inp, dict(out=_out(TOTAL), logdet=_out(B), status=_out(B, np.int32)), dict(seed=11 + variant)


def call_sample(L, h, p, q, s, flags):
    return L.gf_sample_batched(h, B, q("n_off"), q("t_off"), q("j_off"), p("t"), T_LEN, p("diag"), p("coef"),
                               p("ddiag"), p("normals"), s["seed"], 5, p("out"), p("logdet"), p("status"), flags)


def _w_off():
    kb, _ = _scan_setup()
    w = np.concatenate([[0], np.cumsum(np.diff(N_OFF) * kb.J)]).astype(np.int64)
    return w[:-1].copy(), int(w[-1])


def make_factor(variant):
    inp, rng = _scan_inputs("factor", variant)
    inp["w_off"], w_len = _w_off()
    return inp, dict(d=_out(TOTAL), W=_out(w_len), logdet=_out(B), status=_out(B, np.int32)), {}


def call_factor(L, h, p, q, s, flags):
    return L.gf_factor_batched(h, B, q("n_off"), q("t_off"), q("j_off"), q("w_off"), p("t"), T_LEN, p("diag"),
                               p("coef"), p("ddiag"), p("d"), p("W"), p("logdet"), p("status"), flags)


@functools.lru_cache(maxsize=None)
def _factor():
    """W of the scan rows' batch, for the sweeps."""
    kb, t = _scan_setup()
    inp, _, _ = make_factor(0)
    geom = Geometry(N_OFF, T_OFF, T_LEN)
    d, W, w_off, logdet, status = S.default_solver().factor(kb, geom, t, diag=inp["diag"])
    assert np.all(status == 0)
    return W


def make_sweep(variant, alias):
    kb, t = _scan_setup()
    rng = _rng("sweep", variant)
    inp = dict(n_off=N_OFF, t_off=T_OFF, j_off=kb.j_off, w_off=_w_off()[0], t=t, coef=kb.coef, W=_factor())
    y = rng.standard_normal(TOTAL) * 100.0
    if alias:
        return inp, dict(Z=y), {}
    inp["Y"] = y
    return inp, dict(Z=_out(TOTAL)), {}


def call_sweep(op, alias):
    def call(L, h, p, q, s, flags):
        Y = p("Z") if alias else p("Y")
        return L.gf_sweep_batched(h, op, B, q("n_off"), q("t_off"), q("j_off"), q("w_off"), p("t"), T_LEN,
                                  p("coef"), p("W"), Y, p("Z"), flags)
    return call


@functools.lru_cache(maxsize=None)
def _two_kernels():
    import gadfly_b200 as g
    solar = g.SolarOscillatorKernel(texp=1 * g.units.min, bandpass='SOHO VIRGO')
    hp = g.Hyperparameters.for_star(0.9, 10.0, 4919.0, 52.3, bandpass='SOHO VIRGO', quiet=True)
    return KernelBatch([solar, g.StellarOscillatorKernel(hp, texp=1 * g.units.min)])


def make_psd(variant):
    kb = _two_kernels()
    omega = 2 * np.pi * np.sort(_rng("psd", variant).uniform(0.5, 6000.0, 400))
    return dict(j_off=kb.j_off, base=kb.base, delta=kb.delta, omega=omega), dict(out=_out((2, 400))), {}


def call_psd(L, h, p, q, s, flags):
    return L.gf_psd_batched(h, 2, q("j_off"), p("base"), p("delta"), p("omega"), 400, p("out"), flags)


def make_cond(variant):
    kb, _ = _scan_setup()
    rng = _rng("cond", variant)
    t = np.sort(rng.uniform(0.0, 0.03, 300))
    ts = np.sort(rng.uniform(0.0, 0.03, 150))
    coef = np.ascontiguousarray(kb.coef[kb.j_off[0]:kb.j_off[1]])
    return dict(t=t, ts=ts, coef=coef, alpha=rng.standard_normal(300)), dict(mu=_out(150)), dict(Jc=len(coef))


def call_cond(L, h, p, q, s, flags):
    return L.gf_conditional_mean(h, 300, p("t"), 150, p("ts"), s["Jc"], p("coef"), p("alpha"), p("mu"), flags)


def make_sample_multi(variant):
    inp, rng = _scan_inputs("sample_multi", variant)
    inp["normals"] = rng.standard_normal(TOTAL * K)
    return inp, dict(out=_out(TOTAL * K), logdet=_out(B), status=_out(B, np.int32)), {}


def call_sample_multi(L, h, p, q, s, flags):
    return L.gf_sample_multi(h, B, q("n_off"), q("t_off"), q("j_off"), p("t"), T_LEN, p("diag"), p("coef"),
                             p("ddiag"), K, p("normals"), 3, 0, p("out"), p("logdet"), p("status"), flags)


def make_loglike_multi(variant):
    inp, rng = _scan_inputs("loglike_multi", variant)
    inp["y"] = rng.standard_normal(TOTAL * K) * 300.0
    return inp, dict(logdet=_out(B), quad=_out(B * K), status=_out(B, np.int32)), {}


def call_loglike_multi(L, h, p, q, s, flags):
    return L.gf_loglike_multi(h, B, q("n_off"), q("t_off"), q("j_off"), p("t"), T_LEN, p("diag"), p("coef"),
                              p("ddiag"), K, p("y"), p("logdet"), p("quad"), p("status"), flags)


def make_power(variant):
    flux = _rng("power", variant).standard_normal((3, 1000)) * 100.0
    return dict(flux=flux), dict(power=_out((3, 500))), {}


def call_power(L, h, p, q, s, flags):
    return L.gf_power_spectrum_batched(h, 3, 1000, p("flux"), 1.0 / 1440.0, 0, p("power"), flags)


def make_bin(variant):
    rng = _rng("bin", variant)
    lo = np.arange(12, dtype=np.int64) * 40
    cnt = np.full(12, 40, dtype=np.int64)
    cnt[3] = 7
    inp = dict(lo=lo, cnt=cnt, axis=np.linspace(1.0, 5000.0, 500), power=rng.uniform(0.5, 2.0, (3, 500)))
    return inp, dict(stat=_out((3, 12)), err=_out((3, 12))), {}


def call_bin(L, h, p, q, s, flags):
    return L.gf_bin_power_batched(h, 3, 500, 12, q("lo"), q("cnt"), p("axis"), p("power"), 1.5, p("stat"),
                                  p("err"), flags)


STARS = np.array([(1.0, 1.0, 5777.0, 1.0), (1.1, 1.6, 6100.0, 3.2), (0.9, 1.4, 5500.0, 2.2)])


def make_feed_stars(variant):
    gran, modes, _ = solar_tables()
    M, R, T, Lum = (STARS[:, i] * (1 + 0.01 * variant) for i in range(4))
    nb = len(STARS)
    cap = nb * (len(gran) + len(modes))
    inp = dict(mass=M, radius=R, temperature=T, luminosity=Lum, alpha=np.full(nb, 1.0 + 0.01 * variant),
               delta=np.full(nb, 6e-5), gran=gran, modes=modes)
    outs = dict(j_off=_out(nb + 1, np.int64), sho=_out((cap, 3)), coef=_out((cap, 4)), base=_out((cap, 4)),
                ddiag=_out(nb))
    return inp, outs, dict(n_gran=len(gran), n_modes=len(modes), cap=cap)


def call_feed_stars(L, h, p, q, s, flags):
    return L.gf_feed_stars(h, len(STARS), p("mass"), p("radius"), p("temperature"), p("luminosity"), p("alpha"),
                           550.0, p("delta"), s["n_gran"], p("gran"), s["n_modes"], p("modes"), s["cap"],
                           q("j_off"), p("sho"), p("coef"), p("base"), p("ddiag"), flags)


def make_feed_sho(variant):
    rng = _rng("feed_sho", variant)
    j_off = np.array([0, 3, 7], dtype=np.int64)
    sho = np.stack([rng.uniform(1.0, 10.0, 7), rng.uniform(100.0, 3000.0, 7), rng.uniform(0.6, 50.0, 7)], axis=1)
    return (dict(j_off=j_off, sho=sho, delta=np.array([6e-5, 2e-5])),
            dict(coef=_out((7, 4)), base=_out((7, 4)), ddiag=_out(2)), {})


def call_feed_sho(L, h, p, q, s, flags):
    return L.gf_feed_sho(h, 2, q("j_off"), p("sho"), p("delta"), p("coef"), p("base"), p("ddiag"), flags)


def make_bandpass(variant):
    rng = _rng("bandpass", variant)
    wl = np.linspace(0.35, 1.0, 200)
    inp = dict(temperature=rng.uniform(4000.0, 7000.0, 5), wl=wl, tr=np.exp(-((wl - 0.6) / 0.15) ** 2))
    return inp, dict(out=_out(5)), {}


def call_bandpass(L, h, p, q, s, flags):
    return L.gf_bandpass_amplitude(h, 5, p("temperature"), 200, p("wl"), p("tr"), p("out"), flags)


SCAN_HOST = ("n_off", "t_off", "j_off", "w_off")
ROWS = [
    Row("loglike", make_loglike, call_loglike, 1, "scan_fast", SCAN_HOST),
    Row("loglike_shared_y", functools.partial(make_loglike, shared=True),
        lambda L, h, p, q, s, f: call_loglike(L, h, p, q, s, f | S.FLAG_SHARED_Y), 1, "scan_fast", SCAN_HOST),
    Row("sample_normals", make_sample, call_sample, 1, "scan_fast", SCAN_HOST),
    Row("sample_philox", functools.partial(make_sample, philox=True), call_sample, 1, "scan_fast", SCAN_HOST),
    Row("factor_W", make_factor, call_factor, 1, "scan_fast", SCAN_HOST),
] + [
    Row(f"sweep{op}_{'alias' if alias else 'separate'}", functools.partial(make_sweep, alias=alias),
        call_sweep(op, alias), 1, None, SCAN_HOST)
    for op in range(4) for alias in (False, True)
] + [
    Row("psd", make_psd, call_psd, 1, None, ("j_off",)),
    Row("conditional_mean", make_cond, call_cond, 2),
    Row("sample_multi", make_sample_multi, call_sample_multi, 3, "scan_fast", SCAN_HOST),
    Row("loglike_multi", make_loglike_multi, call_loglike_multi, 3, "scan_fast", SCAN_HOST),
    Row("power_spectrum", make_power, call_power, 1),
    Row("bin_power", make_bin, call_bin, 1, None, ("lo", "cnt")),
    Row("feed_stars", make_feed_stars, call_feed_stars, 2, None, ("j_off",)),
    Row("feed_sho", make_feed_sho, call_feed_sho, 1, None, ("j_off",)),
    Row("bandpass_amplitude", make_bandpass, call_bandpass, 1),
]


# ---- placement and one call -----------------------------------------------------------------------
def _place(a, where):
    import torch
    if where == "pageable":
        return np.array(a, copy=True)
    x = torch.from_numpy(np.ascontiguousarray(a))
    return x.pin_memory() if where == "pinned" else x.cuda()


def _addr(x):
    return x.data_ptr() if hasattr(x, "data_ptr") else x.ctypes.data


def _numpy(x):
    return x.cpu().numpy().copy() if hasattr(x, "data_ptr") else x.copy()


def _placed(row, variant, inputs_at, outputs_at):
    """-> (every buffer of the call by name, names of the outputs, scalars).  The buffers must stay
    alive until the call has been synchronised."""
    import torch
    inp, outs, scalars = row.make(variant)
    bufs = {k: _place(v, "pageable" if k in row.host else inputs_at) for k, v in inp.items()}
    bufs.update({k: _place(v, "pageable" if k in row.host else outputs_at) for k, v in outs.items()})
    # torch's copies before the library's streams (torch's stream only: a device-wide synchronise
    # would also wait for calls of the library still in flight)
    torch.cuda.current_stream().synchronize()
    return bufs, list(outs), scalars


def _call(solver, row, placed, flags):
    """Issue the call; -> launch delta."""
    L, h = solver._lib, solver._h
    bufs, _, scalars = placed
    p = lambda k: _addr(bufs[k]) if k in bufs else None                        # noqa: E731
    q = lambda k: ctypes.cast(ctypes.c_void_p(_addr(bufs[k])), _i64p)          # noqa: E731
    n0 = int(L.gf_launch_count(h))
    rc = row.call(L, h, p, q, scalars, flags)
    assert rc == 0, (row.name, rc, L.gf_last_error(h))
    return int(L.gf_launch_count(h)) - n0


def _check_path(solver, row, before):
    got = S.PATH_NAMES[int(solver._lib.gf_last_scan_path(solver._h))]
    assert got == (row.path or before), (row.name, got)


def _assert_same(row, what, got, ref):
    for k in ref:
        a, b = np.ascontiguousarray(got[k]), np.ascontiguousarray(ref[k])
        assert a.shape == b.shape and np.array_equal(a.view(np.uint8), b.view(np.uint8)), \
            (row.name, what, k, np.max(np.abs(a.astype(np.float64) - b.astype(np.float64))))


PLACEMENTS = [("pageable", "pageable"), ("pinned", "pinned"), ("device", "device"),
              ("device", "pageable"), ("pageable", "device")]


@pytest.mark.parametrize("row", ROWS, ids=lambda r: r.name)
def test_staging_is_transparent(solver, row):
    L, h = solver._lib, solver._h
    path0 = S.PATH_NAMES[int(L.gf_last_scan_path(h))]

    def blocking(variant):
        bufs, outs, _ = placed = _placed(row, variant, "pageable", "pageable")
        assert _call(solver, row, placed, 0) == row.launches, row.name
        _check_path(solver, row, path0)
        return {k: _numpy(bufs[k]) for k in outs}

    ref = blocking(0)
    for inputs_at, outputs_at in PLACEMENTS:
        for flags in (0, S.FLAG_ASYNC):
            bufs, outs, _ = placed = _placed(row, 0, inputs_at, outputs_at)
            n = _call(solver, row, placed, flags)
            if flags:
                assert L.gf_synchronize(h) == 0
            assert n == row.launches, (row.name, inputs_at, outputs_at, flags, n)
            _check_path(solver, row, path0)
            _assert_same(row, (inputs_at, outputs_at, flags), {k: _numpy(bufs[k]) for k in outs}, ref)

    # Three calls in flight on one handle, each with its own inputs and pageable outputs.  The handle's
    # compute stream is held behind a ~50 ms spin on a torch stream, so that no kernel of the three runs
    # before all are issued: the second call finds every buffer of the first still in use and takes the
    # other buffer of each slot, and the third waits for the first's.  (The feeders wait for their own
    # kernels inside the call, so only their outputs are in flight together.)
    import torch
    refs = [blocking(v) for v in (1, 2, 3)]
    placed = [_placed(row, v, "pageable", "pageable") for v in (1, 2, 3)]
    hold = torch.cuda.Stream()
    with torch.cuda.stream(hold):
        torch.cuda._sleep(100_000_000)
    assert L.gf_wait_stream(h, ctypes.c_void_p(hold.cuda_stream)) == 0
    launches = [_call(solver, row, pl, S.FLAG_ASYNC) for pl in placed]
    assert L.gf_synchronize(h) == 0
    for v, (bufs, outs, _), n, r in zip((1, 2, 3), placed, launches, refs):
        assert n == row.launches
        _assert_same(row, ("async", v), {k: bufs[k] for k in outs}, r)
    _check_path(solver, row, path0)
