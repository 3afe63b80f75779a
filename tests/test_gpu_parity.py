"""GPU parity: CUDA path (through the C-ABI) vs the CPU oracle and the golden
fixtures generated from the reference.  Tolerances follow BASELINE.json's
north star: bit-exact index/mask arrays, <= 1e-5 relative (max-norm) for FFT
floats, <= 1e-5 element-wise relative for eigenvalues."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import complex_digest         # noqa: E402
from oracle import dynspec_oracle as DO   # noqa: E402
from oracle import thth_oracle as TO      # noqa: E402

RTOL = 1e-5


def maxrel(a, b):
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


@pytest.fixture(scope="module")
def sb():
    import scintools_b200
    from scintools_b200 import _device
    _device.device()
    return scintools_b200


@pytest.fixture(scope="module")
def sample(golden_dir):
    g = np.load(os.path.join(golden_dir, "thth_sample_64x150.npz"))
    npad = int(g["npad"])
    d0 = g["dspec2"] - g["dspec2"].mean()
    CS = TO.conjugate_spectrum(d0, npad, 0.0)
    return g, CS


def test_thth_indices_bit_exact(sb, sample):
    g, CS = sample
    thth = sb.ththmod
    for eta in (float(g["eta_a"]), float(g["eta_b"]), 12.5, 99.9):
        th, ti, fi, pn = TO.thth_indices(g["tau"], g["fd"], eta, g["edges"])
        m, gti, gfi, gpn = thth.thth_map(CS, g["tau"], g["fd"], eta, g["edges"],
                                         return_indices=True)
        assert np.array_equal(gti, ti.astype(np.int32))
        assert np.array_equal(gfi, fi.astype(np.int32))
        assert np.array_equal(gpn, pn)
        assert np.array_equal(thth.th_points(g["tau"], g["fd"], eta, g["edges"]),
                              TO.th_points(g["tau"], g["fd"], eta, g["edges"]))


def test_thth_map_values(sb, sample):
    g, CS = sample
    thth = sb.ththmod
    for tag in ("a", "b"):
        eta = float(g["eta_" + tag])
        red, er = thth.thth_redmap(CS, g["tau"], g["fd"], eta, g["edges"])
        # the reference's map, rebuilt by the oracle and checked bit for bit against
        # the digest the fixture keeps of it
        ref, _ = TO.thth_redmap(CS, g["tau"], g["fd"], eta, g["edges"])
        assert complex_digest(ref) == str(g["red_%s_sha256" % tag])
        assert red.shape == ref.shape
        assert maxrel(red, ref) < 1e-6
        assert np.array_equal((red == 0), (ref == 0))
        assert np.array_equal(er, g["edges_red_" + tag])
    full = thth.thth_map(CS, g["tau"], g["fd"], 30.0, g["edges"], hermetian=False)
    assert maxrel(full, TO.thth_map(CS, g["tau"], g["fd"], 30.0, g["edges"], False)) < 1e-6


def test_eta_sweep_golden(sb, sample):
    g, CS = sample
    eigs, info = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], g["etas"], g["edges"],
                                      return_info=True)
    rel = np.abs(eigs - g["eigs"]) / g["eigs"]
    assert rel.max() < RTOL, rel.max()
    assert (info["status"] == 0).all()
    assert info["iters"].max() < 64
    # N_red shrinks with eta exactly like the reference crop
    nred = np.array([TO.th_points(g["tau"], g["fd"], e, g["edges"]).sum()
                     for e in g["etas"]])
    assert np.array_equal(info["nred"], nred)
    # documented known answer (thth_intro.rst:101-104): eta ~ 44 s^3
    assert abs(g["etas"][np.argmax(eigs)] - 44.0) < 2.0
    assert sb.ththmod.Eval_calc(CS, g["tau"], g["fd"], g["etas"][37], g["edges"]) == \
        pytest.approx(g["eigs"][37], rel=RTOL)


def test_eta_sweep_incoherent(sb, sample):
    g, CS = sample
    tau_mask = 0.5
    CSm = CS.copy()
    CSm[np.abs(g["tau"]) < tau_mask] = 0
    eigs = sb.ththmod.eta_sweep(np.abs(CSm), g["tau"], g["fd"], g["inc_etas"],
                                g["edges"], coher=True)
    assert (np.abs(eigs - g["inc_eigs"]) / g["inc_eigs"]).max() < RTOL
    eigs2 = sb.ththmod.eta_sweep(CSm, g["tau"], g["fd"], g["inc_etas"],
                                 g["edges"], coher=False)
    assert (np.abs(eigs2 - g["inc_eigs"]) / g["inc_eigs"]).max() < RTOL


def test_eta_sweep_failure_modes(sb, sample):
    g, CS = sample
    thth = sb.ththmod
    # edges far wider than the fd axis: numpy raises IndexError -> NaN
    wide = np.linspace(-6.0, 6.0, 64)
    ref = TO.eta_sweep(CS, g["tau"], g["fd"], np.array([20.0, 50.0]), wide)
    got, info = thth.eta_sweep(CS, g["tau"], g["fd"], np.array([20.0, 50.0]), wide,
                               return_info=True)
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    if ok.any():
        assert (np.abs(got[ok] - ref[ok]) / ref[ok]).max() < RTOL
    # all-zero spectrum: NaN start vector -> NaN
    z = thth.eta_sweep(np.zeros_like(CS), g["tau"], g["fd"], np.array([40.0]), g["edges"])
    assert np.isnan(z).all()
    with pytest.raises(Exception):
        thth.Eval_calc(np.zeros_like(CS), g["tau"], g["fd"], 40.0, g["edges"])


def _dyn(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _ds(sb, dyn, dt, df):
    nf, nt = dyn.shape
    bd = sb.BasicDyn(dyn, times=dt * np.arange(nt), freqs=1400 + df * np.arange(nf),
                     dt=dt, df=df)
    return sb.Dynspec(dyn=bd, verbose=False)


def _check_db(got_db, ref_db, rtol=RTOL, db_tol=2e-4):
    lin_g, lin_r = 10 ** (got_db / 10), 10 ** (ref_db / 10)
    assert maxrel(lin_g, lin_r) < rtol
    big = lin_r > 1e-3 * lin_r.max()
    # dB error = 4.34 * relative power error: absolute 1e-4 dB on significant bins
    assert np.max(np.abs(got_db[big] - ref_db[big])) < db_tol


@pytest.mark.parametrize("name", ["sspec_acf_48x80.npz", "sspec_acf_64x128.npz"])
def test_sspec_acf_golden(sb, golden_dir, name):
    g = _dyn(golden_dir, name)
    ds = _ds(sb, g["dyn"], float(g["dt"]), float(g["df"]))
    ds.calc_sspec()
    assert ds.sspec.shape == g["sspec"].shape
    assert np.array_equal(ds.fdop, g["fdop"]) and np.array_equal(ds.tdel, g["tdel"])
    _check_db(ds.sspec, g["sspec"])
    ds.calc_acf()
    assert ds.acf.shape == g["acf"].shape
    assert maxrel(ds.acf, g["acf"]) < RTOL
    raw = ds.calc_acf(input_dyn=g["dyn"] - g["dyn"].mean(), normalise=False)
    assert maxrel(raw, DO.calc_acf(g["dyn"], normalise=False)) < RTOL


def test_acf_sspec_method(sb, golden_dir):
    g = _dyn(golden_dir, "sspec_acf_48x80.npz")
    ds = _ds(sb, g["dyn"], float(g["dt"]), float(g["df"]))
    ds.calc_acf(method="sspec")
    assert ds.acf.shape == g["acf_sspec"].shape
    assert maxrel(ds.acf, g["acf_sspec"]) < RTOL


def test_sspec_variants(sb, golden_dir):
    g = _dyn(golden_dir, "sspec_acf_48x80.npz")
    ds = _ds(sb, g["dyn"], float(g["dt"]), float(g["df"]))
    _, _, pw = ds.calc_sspec(prewhite=True, return_sspec=True)
    # prewhite differences / transforms / post-darkens in float64 on the device
    _check_db(pw, g["sspec_prewhite"])
    _, td, full = ds.calc_sspec(halve=False, window="blackman", window_frac=0.25,
                                return_sspec=True)
    assert np.array_equal(td, g["tdel_full"])
    _check_db(full, g["sspec_full_blackman"])
    _, _, nw = ds.calc_sspec(window=None, return_sspec=True)
    _check_db(nw, g["sspec_nowindow"])
    with pytest.raises(RuntimeError):
        ds.calc_sspec(prewhite=True, halve=False)


@pytest.mark.parametrize("shape,npad", [((8, 16), 3), ((64, 128), 3), ((32, 512), 1),
                                        ((256, 64), 0), ((128, 2048), 3)])
def test_conjugate_spectrum(sb, shape, npad):
    rng = np.random.default_rng(5)
    d = rng.normal(size=shape)
    d -= d.mean()
    f = 1400 + 0.05 * np.arange(shape[0])
    tau = TO.fft_axis(f, "us", npad)
    for pad_value, mask in ((0.0, 0.0), (0.37, 0.0), (None, 2.0)):
        ref = TO.conjugate_spectrum(d, npad, pad_value, tau, mask)
        for half in (False, True):
            got = sb.ththmod.conjugate_spectrum(d, npad, pad_value, tau, mask,
                                                half=half).numpy()
            assert got.shape == ref.shape
            assert maxrel(got, ref) < RTOL
            if mask:
                assert np.array_equal(got == 0, ref == 0)


@pytest.mark.parametrize("shape,npad", [((64, 150), 3), ((10, 7), 1), ((33, 100), 2),
                                        ((128, 75), 3), ((50, 64), 0)])
def test_conjugate_spectrum_any_size(sb, shape, npad):
    """Non power-of-two padded sizes (chirp-z path), incl. odd lengths."""
    rng = np.random.default_rng(6)
    d = rng.normal(size=shape)
    d -= d.mean()
    f = 1400 + 0.05 * np.arange(shape[0])
    tau = TO.fft_axis(f, "us", npad)
    for pad_value, mask in ((0.0, 0.0), (None, 0.0), (0.21, 1.5)):
        ref = TO.conjugate_spectrum(d, npad, pad_value, tau, mask)
        got = sb.ththmod.conjugate_spectrum(d, npad, pad_value, tau, mask).numpy()
        assert got.shape == ref.shape
        assert maxrel(got, ref) < RTOL
        if mask:
            assert np.array_equal(got == 0, ref == 0)


def test_single_search_tutorial_chunk(sb, golden_dir):
    """The reference's own tutorial chunk (64 x 150, npad=3 -> 256 x 600 CS)
    end to end on the GPU against the reference's single_search output."""
    g = np.load(os.path.join(golden_dir, "thth_sample_64x150.npz"))
    d0 = g["dspec2"] - g["dspec2"].mean()
    res = sb.ththmod.single_search([d0, g["freq"], g["time"], g["etas"], g["edges"],
                                    None, False, 0.1, int(g["npad"]), True, 0.0, False])
    assert (np.abs(res[4] - g["ss_eigs"]) / g["ss_eigs"]).max() < RTOL
    assert res[0] == pytest.approx(float(g["ss_eta_fit"]), rel=1e-4)
    assert abs(res[0] - 44.0) < 2.0
    inc = sb.ththmod.single_search([d0, g["freq"], g["time"], g["inc_etas"], g["edges"],
                                    None, False, 0.1, int(g["npad"]), False, 0.5, False])
    assert (np.abs(inc[4] - g["inc_eigs"]) / g["inc_eigs"]).max() < RTOL


def test_half_plane_sweep_matches_full(sb):
    """The sweep on the Hermitian half-plane CS equals the sweep on the full
    array, including gathers that land on negative fd (edges wider than fd)."""
    rng = np.random.default_rng(9)
    nf, nt, npad = 32, 64, 1
    d = rng.normal(size=(nf, nt))
    d -= d.mean()
    t = np.arange(nt) * 10.0
    f = 1400 + 0.1 * np.arange(nf)
    fd = TO.fft_axis(t, "mHz", npad)
    tau = TO.fft_axis(f, "us", npad)
    thth = sb.ththmod
    full = thth.conjugate_spectrum(d, npad, 0.0, half=False)
    half = thth.conjugate_spectrum(d, npad, 0.0, half=True)
    for lim in (20.0, 60.0, 110.0):      # 110 > fd range: wraps to negative fd
        edges = np.linspace(-lim, lim, 64)
        etas = np.linspace(0.0005, 0.004, 12)
        a, ia = thth.eta_sweep(full, tau, fd, etas, edges, return_info=True)
        b, ib = thth.eta_sweep(half, tau, fd, etas, edges, return_info=True)
        ref = TO.eta_sweep(full.numpy(), tau, fd, etas, edges)
        assert np.array_equal(np.isnan(a), np.isnan(b))
        assert np.array_equal(np.isnan(a), np.isnan(ref))
        ok = ~np.isnan(a)
        assert np.allclose(a[ok], b[ok], rtol=1e-6)
        if ok.any():
            assert (np.abs(a[ok] - ref[ok]) / np.abs(ref[ok])).max() < RTOL
        m1 = thth.thth_map(full, tau, fd, etas[3], edges) if not np.isnan(a[3]) else None
        if m1 is not None:
            m2 = thth.thth_map(half, tau, fd, etas[3], edges)
            assert maxrel(m2, m1) < 1e-6


def test_single_search_end_to_end(sb, golden_dir):
    """Power-of-two chunk: CS on the GPU + sweep + host parabola fit."""
    rng = np.random.default_rng(3)
    nf, nt, npad = 64, 128, 3
    t = np.arange(nt) * 20.0
    f = 1400.0 + np.arange(nf) * 0.05
    eta_true = 30.0
    fdk = rng.uniform(-6, 6, 24)
    ak = (rng.normal(size=24) + 1j * rng.normal(size=24)) * np.exp(-(fdk / 3) ** 2)
    E = sum(a * np.exp(2j * np.pi * (k * 1e-3 * t[None, :] - eta_true * k ** 2 * (f[:, None] - f[0])))
            for a, k in zip(ak, fdk))
    dyn = np.abs(E) ** 2
    dyn += rng.normal(0, 0.05 * dyn.mean(), dyn.shape)
    d0 = dyn - dyn.mean()
    edges = np.linspace(-8, 8, 256)
    etas = np.linspace(15, 60, 46)
    ref = TO.single_search(d0, f, t, etas, edges, 0.1, npad, True, 0.0)
    got = sb.ththmod.single_search([d0, f, t, etas, edges, None, False, 0.1, npad,
                                    True, 0.0, False])
    assert (np.abs(got[4] - ref[4]) / ref[4]).max() < RTOL
    assert got[0] == pytest.approx(ref[0], rel=1e-4)
    assert got[1] == pytest.approx(ref[1], rel=5e-2)
    assert abs(got[0] - eta_true) / eta_true < 0.1


def test_batch_arc_pipeline(sb):
    """Config-5 style unit at reduced size: sspec + acf + curvature for a batch
    of dynspecs; curvatures agree with the oracle's single_search."""
    from scintools_b200.pipeline import batch_arc_pipeline
    nf, nt, npad = 64, 128, 3
    t = np.arange(nt) * 20.0
    f = 1400.0 + np.arange(nf) * 0.05
    edges = np.linspace(-8, 8, 128)
    etas = np.linspace(15, 60, 24)
    dyns = []
    for seed in range(3):
        rng = np.random.default_rng(1000 + seed)
        fdk = rng.uniform(-6, 6, 16)
        ak = (rng.normal(size=16) + 1j * rng.normal(size=16)) * np.exp(-(fdk / 3) ** 2)
        E = sum(a * np.exp(2j * np.pi * (k * 1e-3 * t[None, :] - 30.0 * k ** 2 * (f[:, None] - f[0])))
                for a, k in zip(ak, fdk))
        dyns.append(np.abs(E) ** 2)
    fit, sig = batch_arc_pipeline(dyns, f, t, etas, edges, npad=npad)
    assert fit.shape == (3,)
    for i, d in enumerate(dyns):
        ref = TO.single_search(d - d.mean(), f, t, etas, edges, 0.1, npad, True, 0.0)
        assert fit[i] == pytest.approx(ref[0], rel=1e-3)


def test_dynspec_thetatheta_chunks(sb):
    """Dynspec.prep_thetatheta / thetatheta_single / fit_thetatheta on a 2x2
    chunk grid against the oracle's single_search per chunk and the reference's
    weighted A/f^2 combination (dynspec.py:1724-1744)."""
    rng = np.random.default_rng(21)
    nf, nt = 128, 256
    t = np.arange(nt) * 20.0
    f = 1400.0 + np.arange(nf) * 0.05
    fdk = rng.uniform(-6, 6, 24)
    ak = (rng.normal(size=24) + 1j * rng.normal(size=24)) * np.exp(-(fdk / 3) ** 2)
    E = sum(a * np.exp(2j * np.pi * (k * 1e-3 * t[None, :] - 30.0 * k ** 2 * (f[:, None] - f[0])))
            for a, k in zip(ak, fdk))
    dyn = np.abs(E) ** 2 + rng.normal(0, 0.02, (nf, nt))
    ds = sb.Dynspec(dyn=sb.BasicDyn(dyn, times=t, freqs=f, dt=20.0, df=0.05), verbose=False)
    ds.prep_thetatheta(cwf=64, cwt=128, eta_min=15.0, eta_max=60.0, nedge=128,
                       edges_lim=8.0, fw=0.2, npad=3)
    assert (ds.ncf_fit, ds.nct_fit) == (2, 2)
    etas, eigs, popt = ds.thetatheta_single(cf=1, ct=0)
    fs, ts = slice(64, 128), slice(0, 128)
    d2 = dyn[fs, ts] - dyn[fs, ts].mean()
    e_ref = TO.eta_grid(ds.eta_min, ds.eta_max, ds.fw, ds.fref, f[fs].mean())
    assert np.array_equal(etas, e_ref)
    CS = TO.conjugate_spectrum(d2, 3, 0.0)
    ref = TO.eta_sweep(CS, TO.fft_axis(f[fs], "us", 3), TO.fft_axis(t[ts], "mHz", 3), e_ref,
                       ds.edges * (f[fs].mean() / ds.fref))
    assert (np.abs(eigs - ref) / ref).max() < RTOL
    ds.fit_thetatheta()
    assert ds.eta_evo.shape == (2, 2)
    for cf in range(2):
        for ct in range(2):
            fs, ts = slice(cf * 64, (cf + 1) * 64), slice(ct * 128, (ct + 1) * 128)
            d2 = dyn[fs, ts] - dyn[fs, ts].mean()
            r = TO.single_search(d2, f[fs], t[ts],
                                 TO.eta_grid(ds.eta_min, ds.eta_max, ds.fw, ds.fref, f[fs].mean()),
                                 ds.edges * (f[fs].mean() / ds.fref), ds.fw, 3, True, 0.0)
            assert ds.eta_evo[cf, ct] == pytest.approx(r[0], rel=1e-3)
    f0 = ds.f0s[:, None]
    ok = np.isfinite(ds.eta_evo) * np.isfinite(ds.eta_evo_err)
    A = (np.sum(ds.eta_evo[ok] / (f0 * ds.eta_evo_err)[ok] ** 2) /
         np.sum(1 / ((f0 ** 2) * ds.eta_evo_err)[ok] ** 2))
    assert ds.ththeta == pytest.approx(A / ds.fref ** 2, rel=1e-12)
    with pytest.raises(ValueError):
        ds.fit_thetatheta(pool=object())


def test_column_limited_cs(sb):
    """conjugate_spectrum(ncols_keep=needed_fd_columns(...)) gives the same
    sweep as the full CS, and refuses a theta grid wider than it was built for."""
    rng = np.random.default_rng(31)
    nf, nt, npad = 64, 256, 3
    d = rng.normal(size=(nf, nt))
    d -= d.mean()
    t = np.arange(nt) * 10.0
    f = 1400 + 0.1 * np.arange(nf)
    fd = TO.fft_axis(t, "mHz", npad)
    tau = TO.fft_axis(f, "us", npad)
    thth = sb.ththmod
    edges = np.linspace(-6, 6, 128)
    keep = thth.needed_fd_columns(fd, edges)
    assert keep is not None and keep < fd.shape[0] // 2
    etas = np.linspace(0.005, 0.05, 10)
    full = thth.conjugate_spectrum(d, npad, 0.0)
    lim = thth.conjugate_spectrum(d, npad, 0.0, ncols_keep=keep)
    a = thth.eta_sweep(full, tau, fd, etas, edges)
    b = thth.eta_sweep(lim, tau, fd, etas, edges)
    assert np.array_equal(a, b)
    with pytest.raises(ValueError):
        thth.eta_sweep(lim, tau, fd, etas, np.linspace(-12, 12, 128))
    with pytest.raises(ValueError):
        lim.numpy()
    assert thth.needed_fd_columns(fd, np.linspace(-60, 60, 64)) is None


def test_eta_sweep_persistent_grid(sb, sample, monkeypatch):
    """SB_EIG_PERSIST: a few persistent CTAs walk all curvatures (ring state
    carried from one matrix to the next)."""
    g, CS = sample
    monkeypatch.setenv("SB_EIG_PERSIST", "7")
    eigs, info = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], g["etas"], g["edges"],
                                      return_info=True)
    assert (np.abs(eigs - g["eigs"]) / g["eigs"]).max() < RTOL
    assert (info["status"] == 0).all()
    wide = np.linspace(-6.0, 6.0, 64)
    r2 = TO.eta_sweep(CS, g["tau"], g["fd"], np.array([20.0, 50.0, 30.0]), wide)
    e2 = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], np.array([20.0, 50.0, 30.0]), wide)
    assert np.array_equal(np.isnan(e2), np.isnan(r2))


def test_eta_sweep_batched_slab(sb, sample, monkeypatch):
    """Force the theta-theta matrix slab to a few MB so the sweep runs in many
    build+eigen batches; results must not change."""
    g, CS = sample
    ref, _ = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], g["etas"][::3], g["edges"],
                                  return_info=True)
    monkeypatch.setenv("SB_SWEEP_SLAB_MB", "5")      # 2 matrices of 2 MB per batch
    got, info = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], g["etas"][::3], g["edges"],
                                     return_info=True)
    assert np.array_equal(got, ref)
    assert (info["status"] == 0).all()


def test_thin_thetatheta(sb, golden_dir):
    """two_curve_map / singularvalue_calc / single_search_thin against the
    reference's own outputs (tutorial chunk, run through the units shim)."""
    g = np.load(os.path.join(golden_dir, "thth_sample_64x150.npz"))
    t = np.load(os.path.join(golden_dir, "thth_thin_64x150.npz"))
    thth = sb.ththmod
    d0 = g["dspec2"] - g["dspec2"].mean()
    CS = TO.conjugate_spectrum(d0, int(g["npad"]), 0.0)
    eta = float(t["eta_map"])
    red, er1, er2 = thth.two_curve_map(CS, g["tau"], g["fd"], eta, t["edges"], eta, t["arc"])
    assert red.shape == t["red"].shape
    assert np.array_equal(er1, t["er1"]) and np.array_equal(er2, t["er2"])
    assert maxrel(red, t["red"].astype(np.complex128)) < 2e-6
    assert np.array_equal(red == 0, t["red"] == 0)
    sv, info = thth.thin_sweep(CS, g["tau"], g["fd"], t["etas"], t["edges"], t["arc"],
                               float(t["cut"]), return_info=True)
    assert (np.abs(sv - t["sv"]) / t["sv"]).max() < RTOL
    assert (info["status"] == 0).all()
    assert thth.singularvalue_calc(CS, g["tau"], g["fd"], t["etas"][5], t["edges"],
                                   t["etas"][5], t["arc"], float(t["cut"])) == \
        pytest.approx(t["sv"][5], rel=RTOL)
    arc, cut = t["arc"], float(t["cut"])
    res = thth.single_search_thin([d0, g["freq"], g["time"], t["etas"], t["edges"], None,
                                   False, 0.2, int(g["npad"]), True, False, arc, cut])
    assert (np.abs(res[4] - t["ss_eigs"]) / t["ss_eigs"]).max() < RTOL
    assert res[0] == pytest.approx(float(t["ss_eta_fit"]), rel=1e-4)
    inc = thth.single_search_thin([d0, g["freq"], g["time"], t["inc_etas"], t["edges"], None,
                                   False, 0.2, int(g["npad"]), False, False, arc, 0.0])
    assert (np.abs(inc[4] - t["inc_eigs"]) / t["inc_eigs"]).max() < RTOL


def test_thin_random_vs_oracle(sb):
    rng = np.random.default_rng(55)
    nf, nt, npad = 32, 128, 1
    d = rng.normal(size=(nf, nt))
    d -= d.mean()
    t = np.arange(nt) * 10.0
    f = 1400 + 0.2 * np.arange(nf)
    fd = TO.fft_axis(t, "mHz", npad)
    tau = TO.fft_axis(f, "us", npad)
    cs = sb.ththmod.conjugate_spectrum(d, npad, 0.0)
    CS = cs.numpy()
    edges = np.linspace(-20, 20, 90)
    arc = edges[np.abs(edges) < 11]
    etas = np.linspace(0.002, 0.02, 9)
    got = sb.ththmod.thin_sweep(cs, tau, fd, etas, edges, arc, 1.5)
    ref = TO.thin_sweep(CS, tau, fd, etas, edges, arc, 1.5)
    assert (np.abs(got - ref) / ref).max() < RTOL


def test_dynspec_thetatheta_thin(sb):
    """fitting_proc='thin' through Dynspec (dynspec.py:1480-1515, 1593-1600,
    1701-1708) against the oracle's thin sweep."""
    rng = np.random.default_rng(22)
    nf, nt = 64, 256
    t = np.arange(nt) * 20.0
    f = 1400.0 + np.arange(nf) * 0.05
    fdk = rng.uniform(-6, 6, 24)
    ak = (rng.normal(size=24) + 1j * rng.normal(size=24)) * np.exp(-(fdk / 3) ** 2)
    E = sum(a * np.exp(2j * np.pi * (k * 1e-3 * t[None, :] - 30.0 * k ** 2 * (f[:, None] - f[0])))
            for a, k in zip(ak, fdk))
    dyn = np.abs(E) ** 2 + rng.normal(0, 0.02, (nf, nt))
    ds = sb.Dynspec(dyn=sb.BasicDyn(dyn, times=t, freqs=f, dt=20.0, df=0.05), verbose=False)
    ds.prep_thetatheta(cwt=128, eta_min=15.0, eta_max=60.0, nedge=128, edges_lim=8.0,
                       fw=0.2, npad=3, fitting_proc='thin', arclet_lim=3.0, center_cut=0.3)
    assert (ds.arclet_lim, ds.center_cut) == (3.0, 0.3)
    etas, eigs, popt = ds.thetatheta_single(cf=0, ct=1)
    ts = slice(128, 256)
    d2 = dyn[:, ts] - dyn[:, ts].mean()
    CS = TO.conjugate_spectrum(d2, 3, 0.0)
    tau, fd = TO.fft_axis(f, "us", 3), TO.fft_axis(t[ts], "mHz", 3)
    edges = ds.edges * (f.mean() / ds.fref)
    arc = edges[np.abs(edges) < 3.0]
    ref = TO.thin_sweep(CS, tau, fd, etas, edges, arc, 0.3)
    assert (np.abs(eigs - ref) / ref).max() < RTOL
    ds.fit_thetatheta()
    r = TO.peak_fit(etas, ref, ds.fw)
    assert ds.eta_evo[0, 1] == pytest.approx(r[0], rel=1e-3)


@pytest.mark.parametrize("cluster", ["0", "1", "2", "3", "5", "6", "8"])
def test_eta_sweep_solver_variants(sb, sample, monkeypatch, cluster):
    """The on-chip cluster solver (eig_cluster.cu) at every cluster size and
    the streaming solver (SB_EIG_CLUSTER=0) agree with the reference eigenvalues;
    failure modes are reported identically."""
    g, CS = sample
    monkeypatch.setenv("SB_EIG_CLUSTER", cluster)
    eigs, info = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], g["etas"], g["edges"],
                                      return_info=True)
    rel = np.abs(eigs - g["eigs"]) / g["eigs"]
    assert rel.max() < RTOL, rel.max()
    assert (info["status"] == 0).all()
    assert info["iters"].max() < 64
    # incoherent + masked rows, and a sweep with failing curvatures
    CSm = CS.copy()
    CSm[np.abs(g["tau"]) < 0.5] = 0
    inc = sb.ththmod.eta_sweep(CSm, g["tau"], g["fd"], g["inc_etas"], g["edges"], coher=False)
    assert (np.abs(inc - g["inc_eigs"]) / g["inc_eigs"]).max() < RTOL
    wide = np.linspace(-6.0, 6.0, 64)
    r2 = TO.eta_sweep(CS, g["tau"], g["fd"], np.array([20.0, 50.0]), wide)
    e2 = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], np.array([20.0, 50.0]), wide)
    assert np.array_equal(np.isnan(e2), np.isnan(r2))
    z = sb.ththmod.eta_sweep(np.zeros_like(CS), g["tau"], g["fd"], np.array([40.0]), g["edges"])
    assert np.isnan(z).all()


def test_search_batch_matches_single_search(sb, golden_dir):
    """search_batch (upload of the next chunk on a copy stream) returns exactly
    what a loop over single_search returns."""
    g = np.load(os.path.join(golden_dir, "thth_sample_64x150.npz"))
    d0 = g["dspec2"] - g["dspec2"].mean()
    pars = [[d0 * s, g["freq"], g["time"], g["etas"], g["edges"], None, False, 0.2,
             int(g["npad"]), True, 0.0, False] for s in (1.0, 2.0, 0.5)]
    pars[1][0] = pars[1][0].astype(np.float32)
    a = sb.ththmod.search_batch(pars)
    b = [sb.ththmod.single_search(p) for p in pars]
    for x, y in zip(a, b):
        assert np.allclose(x[4], y[4], rtol=1e-6, atol=0)
        assert x[0] == pytest.approx(y[0], rel=1e-6)


@pytest.mark.parametrize("env", [{}, {"SB_EIG_FP32": "1"}, {"SB_EIG_RTOL_R": "0"}])
def test_eta_sweep_mixed_precision_solver(sb, sample, monkeypatch, env):
    """Default solver (eig_bf16.cu: bf16 Lanczos iteration + fp32 Rayleigh
    quotient), the fp32 streaming solver (SB_EIG_FP32=1) and the default solver
    with its fp32 continuation forced on every curvature (SB_EIG_RTOL_R=0)."""
    g, CS = sample
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    eigs, info = sb.ththmod.eta_sweep(CS, g["tau"], g["fd"], g["etas"], g["edges"],
                                      return_info=True)
    assert (np.abs(eigs - g["eigs"]) / g["eigs"]).max() < RTOL
    assert (info["status"] == 0).all()
    # slowly converging random spectrum (small gaps, many steps)
    rng = np.random.default_rng(77)
    R = rng.normal(size=CS.shape) + 1j * rng.normal(size=CS.shape)
    etas = g["etas"][::16]
    got = sb.ththmod.eta_sweep(R, g["tau"], g["fd"], etas, g["edges"])
    ref = TO.eta_sweep(R, g["tau"], g["fd"], etas, g["edges"])
    assert (np.abs(got - ref) / ref).max() < RTOL
    z = sb.ththmod.eta_sweep(np.zeros_like(CS), g["tau"], g["fd"], np.array([40.0]), g["edges"])
    assert np.isnan(z).all()


def test_scale_dyn_lambda(sb, golden_dir, monkeypatch):
    g = np.load(os.path.join(golden_dir, "scale_dyn_40x24.npz"))
    dyn = g["dyn"]
    nf, nt = dyn.shape
    for flip in (False, True):
        d, f = (dyn[::-1].copy(), g["freqs"][::-1].copy()) if flip else (dyn, g["freqs"])
        ds = sb.Dynspec(dyn=sb.BasicDyn(d, times=float(g["dt"]) * np.arange(nt), freqs=f,
                                        dt=float(g["dt"]), df=float(g["df"])), verbose=False)
        ds.scale_dyn(scale="lambda")
        assert np.array_equal(ds.lam, g["lam"]) and ds.dlam == float(g["dlam"])
        assert maxrel(ds.lamdyn, g["lamdyn"]) < RTOL
    ds.calc_sspec(lamsteps=True)
    lin_g, lin_r = 10 ** (ds.lamsspec / 10), 10 ** (g["lamsspec"] / 10)
    assert maxrel(lin_g, lin_r) < 1e-4
