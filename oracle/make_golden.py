"""Generate tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference/scintools, via oracle/ref_loader.py) on seeded inputs.

TEST INFRASTRUCTURE (see oracle/__init__.py).  Run in the build container only:

    python -m oracle.make_golden

The fixtures are committed; the GPU box never needs /root/reference.  Every
fixture stores the inputs and the reference's outputs, so
tests/test_oracle_golden.py can check the numpy restatements against them and
the gpu tests can check the CUDA path against both.
"""
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")

from oracle import complex_digest, ref_loader  # noqa: E402


def _ref_dynspec(pkg, dyn, dt, df, f0=1400.0):
    nf, nt = dyn.shape
    freqs = f0 + df * np.arange(nf)
    times = dt * np.arange(nt)
    bd = pkg.dynspec.BasicDyn(dyn, name="golden", header=["golden"],
                              times=times, freqs=freqs, nchan=nf, nsub=nt,
                              bw=df * nf, df=df, freq=float(np.mean(freqs)),
                              tobs=dt * nt, dt=dt, mjd=60000)
    return pkg.dynspec.Dynspec(dyn=bd, verbose=False, process=False)


def golden_sspec_acf(pkg):
    """calc_sspec / calc_acf on a non power-of-two exponential field."""
    rng = np.random.default_rng(1)
    nf, nt, dt, df = 48, 80, 10.0, 0.1
    dyn = rng.exponential(1.0, (nf, nt))
    ds = _ref_dynspec(pkg, dyn.copy(), dt, df)
    ds.calc_sspec()
    out = dict(dyn=dyn, dt=dt, df=df, sspec=ds.sspec, fdop=ds.fdop,
               tdel=ds.tdel)
    ds.calc_acf()
    out["acf"] = ds.acf
    fd, td, sec = ds.calc_sspec(prewhite=True, return_sspec=True)
    out["sspec_prewhite"] = sec
    fd, td, sec = ds.calc_sspec(halve=False, window="blackman",
                                window_frac=0.25, return_sspec=True)
    out["sspec_full_blackman"] = sec
    out["tdel_full"] = td
    fd, td, sec = ds.calc_sspec(window=None, return_sspec=True)
    out["sspec_nowindow"] = sec
    ds.calc_acf(method="sspec")
    out["acf_sspec"] = ds.acf
    np.savez_compressed(os.path.join(GOLD, "sspec_acf_48x80.npz"), **out)
    # power-of-two case (C1 of BASELINE.json at reduced size)
    rng = np.random.default_rng(11)
    dyn = rng.exponential(1.0, (64, 128))
    ds = _ref_dynspec(pkg, dyn.copy(), dt, df)
    ds.calc_sspec()
    ds.calc_acf()
    np.savez_compressed(os.path.join(GOLD, "sspec_acf_64x128.npz"), dyn=dyn,
                        dt=dt, df=df, sspec=ds.sspec, fdop=ds.fdop,
                        tdel=ds.tdel, acf=ds.acf)


def golden_c1(pkg):
    """BASELINE.json configs[0]: Dynspec.calc_sspec on a 256x256 synthetic dynamic spectrum
    (the reference's own CPU case).  The input is regenerated from its seed by the test; the
    fixture keeps the axes, a decimated copy of the secondary spectrum, three full rows and
    the float64 sum."""
    rng = np.random.default_rng(256)
    nf, nt, dt, df = 256, 256, 8.0, 0.125
    dyn = rng.exponential(1.0, (nf, nt))
    ds = _ref_dynspec(pkg, dyn.copy(), dt, df)
    ds.calc_sspec()
    sec = np.asarray(ds.sspec)
    np.savez_compressed(os.path.join(GOLD, "c1_sspec_256x256.npz"), seed=256, nf=nf, nt=nt,
                        dt=dt, df=df, shape=np.array(sec.shape), fdop=ds.fdop, tdel=ds.tdel,
                        sspec_dec=sec[::3, ::5], rows=np.array([0, 1, sec.shape[0] - 1]),
                        sspec_rows=sec[[0, 1, sec.shape[0] - 1], :],
                        finite_sum=float(np.sum(sec[np.isfinite(sec)])))


def golden_thth(pkg):
    """ththmod on a chunk of Sample_Data.npz (tutorial recipe,
    docs/source/tutorials/thth_intro.rst:238-310) with seeded noise."""
    u = sys.modules["astropy.units"]
    thth = pkg.ththmod
    arch = np.load(os.path.join(ref_loader.REFERENCE_ROOT, "scintools",
                                "examples", "data", "ththsims",
                                "Sample_Data.npz"))
    rng = np.random.default_rng(7)
    wf = arch["Espec"]
    dspec = np.abs(wf) ** 2 + rng.normal(0, 20, wf.shape)
    cwf, npad = 64, 3
    dspec2 = np.copy(dspec[:cwf])
    freq2 = arch["f_MHz"][:cwf]
    time2 = arch["t_s"]
    mn = dspec2.mean()
    pad = np.pad(dspec2 - mn, ((0, npad * cwf), (0, npad * dspec2.shape[1])),
                 mode="constant", constant_values=0)
    CS = np.fft.fftshift(np.fft.fft2(pad))
    fd = thth.fft_axis(time2 * u.s, u.mHz, npad)
    tau = thth.fft_axis(freq2 * u.MHz, u.us, npad)
    edges = np.linspace(-0.4, 0.4, 512)
    etas = np.linspace(12.5, 100.0, 100)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        eigs = np.array([thth.Eval_calc(CS, tau, fd, e * u.s ** 3,
                                        edges * u.mHz) for e in etas])
        # index arrays + maps for two curvatures (full and cropped regime); the
        # complex128 maps (4 + 1 MB) are kept as shape + digest of their exact bytes
        extra = {}
        for tag, eta in (("a", etas[10]), ("b", etas[80])):
            red, er = thth.thth_redmap(CS, tau, fd, eta * u.s ** 3,
                                       edges * u.mHz)
            extra["eta_" + tag] = eta
            extra["red_%s_shape" % tag] = np.array(np.shape(red))
            extra["red_%s_sha256" % tag] = complex_digest(red)
            extra["edges_red_" + tag] = np.asarray(er.value)
        # single_search end-to-end (pads with dspec2.mean(); coherent)
        d0 = dspec2 - mn
        res = thth.single_search([d0, freq2 * u.MHz, time2 * u.s,
                                  etas * u.s ** 3, edges * u.mHz, None, False,
                                  0.1, npad, True, 0 * u.us, False])
        res_inc = thth.single_search([d0, freq2 * u.MHz, time2 * u.s,
                                      etas[::4] * u.s ** 3, edges * u.mHz,
                                      None, False, 0.1, npad, False,
                                      0.5 * u.us, False])
    np.savez_compressed(
        os.path.join(GOLD, "thth_sample_64x150.npz"),
        dspec2=dspec2, freq=freq2, time=time2, npad=npad, edges=edges,
        etas=etas, eigs=eigs, fd=np.asarray(fd.value),
        tau=np.asarray(tau.value),
        ss_eta_fit=float(res[0].value), ss_eta_sig=float(res[1].value),
        ss_eigs=np.asarray(res[4]),
        inc_etas=etas[::4], inc_eigs=np.asarray(res_inc[4]),
        inc_eta_fit=float(np.asarray(getattr(res_inc[0], "value",
                                             res_inc[0]))),
        **extra)
    print("thth: peak eta = %.3f (tutorial states ~44)" %
          etas[np.argmax(eigs)])
    # axes of the notebook's Dynspec (THTHSample.ipynb cell 13) for the
    # prep_thetatheta known-answer tests
    np.savez_compressed(os.path.join(GOLD, "sample_axes.npz"),
                        f_MHz=arch["f_MHz"], t_s=arch["t_s"])


def golden_thin(pkg):
    """two_curve_map / singularvalue_calc / single_search_thin on the tutorial
    chunk (reference run through the units shim)."""
    u = sys.modules["astropy.units"]
    thth = pkg.ththmod
    g = np.load(os.path.join(GOLD, "thth_sample_64x150.npz"))
    d0 = g["dspec2"] - g["dspec2"].mean()
    npad = int(g["npad"])
    pad = np.pad(d0, ((0, npad * d0.shape[0]), (0, npad * d0.shape[1])))
    CS = np.fft.fftshift(np.fft.fft2(pad))
    tau, fd = g["tau"] * u.us, g["fd"] * u.mHz
    edges = np.linspace(-0.4, 0.4, 512)
    arc = edges[np.abs(edges) < 0.25]
    etas = np.linspace(20.0, 80.0, 25)
    cut = 0.02
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        sv = np.array([thth.singularvalue_calc(CS, tau, fd, e * u.s ** 3, edges * u.mHz,
                                               e * u.s ** 3, arc * u.mHz, cut * u.mHz)
                       for e in etas])
        red, er1, er2 = thth.two_curve_map(CS, tau, fd, etas[8] * u.s ** 3, edges * u.mHz,
                                           etas[8] * u.s ** 3, arc * u.mHz)
        res = thth.single_search_thin([d0, g["freq"] * u.MHz, g["time"] * u.s,
                                       etas * u.s ** 3, edges * u.mHz, None, False, 0.2,
                                       npad, True, False, arc * u.mHz, cut * u.mHz])
        res_inc = thth.single_search_thin([d0, g["freq"] * u.MHz, g["time"] * u.s,
                                           etas[::3] * u.s ** 3, edges * u.mHz, None, False,
                                           0.2, npad, False, False, arc * u.mHz, 0 * u.mHz])
    np.savez_compressed(os.path.join(GOLD, "thth_thin_64x150.npz"), edges=edges, arc=arc,
                        etas=etas, cut=cut, sv=sv, eta_map=etas[8],
                        red=np.asarray(red).astype(np.complex64),
                        er1=np.asarray(er1.value), er2=np.asarray(er2.value),
                        ss_eigs=np.asarray(res[4]),
                        ss_eta_fit=float(np.asarray(getattr(res[0], "value", res[0]))),
                        inc_etas=etas[::3], inc_eigs=np.asarray(res_inc[4]))
    print("thin: peak eta = %.2f" % etas[np.argmax(sv)])


def golden_retrieval(pkg):
    """rev_map / modeler / single_chunk_retrieval on a 64 x 128 piece of the
    tutorial chunk (padded CS 256 x 512).  Eigenvector-dependent outputs are
    stored as computed (their global phase is arbitrary: ARPACK start vector)."""
    u = sys.modules["astropy.units"]
    thth = pkg.ththmod
    g = np.load(os.path.join(GOLD, "thth_sample_64x150.npz"))
    d0 = g["dspec2"][:, :128]
    d0 = d0 - d0.mean()
    time, freq = g["time"][:128], g["freq"]
    npad = int(g["npad"])
    eta = 44.0
    edges = np.linspace(-0.4, 0.4, 256)
    fd = thth.fft_axis(time * u.s, u.mHz, npad)
    tau = thth.fft_axis(freq * u.MHz, u.us, npad)
    pad = np.pad(d0, ((0, npad * d0.shape[0]), (0, npad * d0.shape[1])),
                 mode="constant", constant_values=d0.mean())
    CS = np.fft.fftshift(np.fft.fft2(pad))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        thth_red, thth2_red, recov, model, edges_red, w, V = thth.modeler(
            CS, tau, fd, eta * u.s ** 3, edges * u.mHz)
        res = thth.single_chunk_retrieval([d0, edges * u.mHz, time * u.s, freq * u.MHz,
                                           eta * u.s ** 3, 0, 0, npad, 0 * u.us, False])
        # a generic (non rank-1) map through rev_map, both symmetries
        rng = np.random.default_rng(5)
        n = thth_red.shape[0]
        tt = (rng.normal(size=(n, n)) + 1j * rng.normal(size=(n, n)))
        rv_h = thth.rev_map(tt, tau, fd, eta * u.s ** 3, edges_red, hermetian=True)
        rv_n = thth.rev_map(tt, tau, fd, eta * u.s ** 3, edges_red, hermetian=False)
    # the maps that do not depend on the eigenvector (thth_red, rv_h, rv_n: 0.56 MB
    # compressed) are kept as shape + digest of their exact complex128 bytes
    pinned = {}
    for key, a in (("thth_red", thth_red), ("rv_h", rv_h), ("rv_n", rv_n)):
        pinned[key + "_shape"] = np.array(np.shape(a))
        pinned[key + "_sha256"] = complex_digest(a)
    np.savez_compressed(
        os.path.join(GOLD, "retrieval_64x128.npz"), d0=d0, time=time, freq=freq, npad=npad,
        eta=eta, edges=edges, tau=np.asarray(tau.value), fd=np.asarray(fd.value),
        edges_red=np.asarray(edges_red.value), w=float(w), V=np.asarray(V).astype(np.complex64),
        recov=np.asarray(recov).astype(np.complex64), model=np.asarray(model).astype(np.float32),
        model_E=np.asarray(res[0]).astype(np.complex64), tt_seed=5, **pinned)
    print("retrieval: n_red = %d, w = %.4g, |model_E| max = %.3f" %
          (thth_red.shape[0], w, np.abs(res[0]).max()))


def golden_retrieval_tutorial(pkg):
    """modeler / single_chunk_retrieval on the full 64 x 150 tutorial chunk
    (padded CS 256 x 600: NOT powers of two -> chirp-z inverse FFT)."""
    u = sys.modules["astropy.units"]
    thth = pkg.ththmod
    g = np.load(os.path.join(GOLD, "thth_sample_64x150.npz"))
    d0 = g["dspec2"] - g["dspec2"].mean()
    npad = int(g["npad"])
    eta = 44.0
    edges = np.linspace(-0.4, 0.4, 256)
    fd = thth.fft_axis(g["time"] * u.s, u.mHz, npad)
    tau = thth.fft_axis(g["freq"] * u.MHz, u.us, npad)
    pad = np.pad(d0, ((0, npad * d0.shape[0]), (0, npad * d0.shape[1])),
                 mode="constant", constant_values=d0.mean())
    CS = np.fft.fftshift(np.fft.fft2(pad))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        out = thth.modeler(CS, tau, fd, eta * u.s ** 3, edges * u.mHz)
        res = thth.single_chunk_retrieval([d0, edges * u.mHz, g["time"] * u.s, g["freq"] * u.MHz,
                                           eta * u.s ** 3, 0, 0, npad, 0 * u.us, False])
    np.savez_compressed(os.path.join(GOLD, "retrieval_64x150.npz"), eta=eta, edges=edges,
                        w=float(out[5]), model_crop=np.asarray(out[3])[:64, :150].astype(np.float32),
                        model_E=np.asarray(res[0]).astype(np.complex64))
    print("retrieval tutorial: n_red = %d" % out[0].shape[0])


def golden_wavefield(pkg):
    """mosaic + Dynspec.calc_wavefield(gs=True) of the reference on preset
    (random) chunks: deterministic, no eigenvectors involved."""
    rng = np.random.default_rng(17)
    ncf, nct, cwf, cwt = 3, 3, 16, 32
    chunks = rng.normal(size=(ncf, nct, cwf, cwt)) + 1j * rng.normal(size=(ncf, nct, cwf, cwt))
    nf, nt = (ncf - 1) * (cwf // 2) + cwf, (nct - 1) * (cwt // 2) + cwt     # 32 x 64
    dyn = rng.exponential(1.0, (nf + 3, nt + 5))
    dyn[4, 7] = np.nan
    dyn[9, 11] = -0.5
    ds = _ref_dynspec(pkg, dyn, 10.0, 0.1)
    ds.chunks = chunks.copy()
    mos = pkg.ththmod.mosaic(chunks)
    ds.calc_wavefield(gs=True, niter=2)
    np.savez_compressed(os.path.join(GOLD, "wavefield_gs_32x64.npz"), chunks=chunks, dyn=dyn,
                        freqs=np.asarray(ds.freqs), dt=10.0, df=0.1, niter=2,
                        mosaic=mos, wavefield=np.asarray(ds.wavefield))
    print("wavefield: |W| max %.3f" % np.abs(ds.wavefield).max())


def golden_scale_dyn(pkg):
    """Dynspec.scale_dyn(scale='lambda') + calc_sspec(lamsteps=True) of the
    reference (oracle pin for SURVEY 8f rank 3; no CUDA row yet)."""
    rng = np.random.default_rng(23)
    nf, nt, dt, df = 40, 24, 10.0, 0.8
    dyn = rng.exponential(1.0, (nf, nt))
    ds = _ref_dynspec(pkg, dyn.copy(), dt, df, f0=1250.0)
    ds.scale_dyn(scale="lambda")
    out = dict(dyn=dyn, dt=dt, df=df, freqs=np.asarray(ds.freqs), lamdyn=ds.lamdyn,
               lam=ds.lam, dlam=ds.dlam)
    ds.calc_sspec(lamsteps=True)
    out.update(lamsspec=ds.lamsspec, beta=ds.beta, fdop=ds.fdop)
    np.savez_compressed(os.path.join(GOLD, "scale_dyn_40x24.npz"), **out)
    print("scale_dyn: lamdyn", ds.lamdyn.shape, "dlam %.3e" % ds.dlam)


def golden_norm_sspec(pkg):
    """Dynspec.norm_sspec of the reference with an explicit curvature (oracle pin
    for SURVEY 8f rank 2; no CUDA row yet)."""
    rng = np.random.default_rng(29)
    nf, nt, dt, df = 64, 96, 10.0, 0.1
    dyn = rng.exponential(1.0, (nf, nt))
    ds = _ref_dynspec(pkg, dyn.copy(), dt, df)
    ds.calc_sspec()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ds.norm_sspec(eta=0.4, lamsteps=False, plot=False, cutmid=2, startbin=2)
    np.savez_compressed(os.path.join(GOLD, "norm_sspec_64x96.npz"), dyn=dyn, dt=dt, df=df,
                        eta=0.4, cutmid=2, startbin=2, freq=float(ds.freq),
                        sspec=ds.sspec, fdop=ds.fdop, tdel=ds.tdel,
                        normsspec=np.ma.filled(ds.normsspec, np.nan),
                        mask=np.ma.getmaskarray(ds.normsspec),
                        normsspecavg=np.ma.filled(ds.normsspecavg, np.nan),
                        normsspec_fdop=ds.normsspec_fdop, normsspec_tdel=ds.normsspec_tdel,
                        powerspectrum=np.ma.filled(ds.powerspectrum, np.nan))
    print("norm_sspec:", np.shape(ds.normsspec))


def golden_fit_arc(pkg):
    """Dynspec.fit_arc of the reference (dynspec.py:970-1346) on a 1-D-screen dynamic
    spectrum with a clear arc, wavelength steps (the mode prep_thetatheta uses,
    dynspec.py:1458-1466: scale_dyn + calc_sspec(lamsteps=True) + norm_sspec):
    default call, asymmetric fit, explicit curvature range + log parabola; plus the
    norm_sspec products of the default call (oracle pin for SURVEY 8f rank 2).
    (lamsteps=False needs hand-tuned curvature ranges in the reference and reads
    self.beta anyway, :1089; norm_sspec(lamsteps=False) is pinned by norm_sspec_64x96.)"""
    rng = np.random.default_rng(41)
    nf, nt, dt, df, f0 = 128, 160, 8.0, 0.25, 1300.0
    eta_true = 0.35                                         # us / mHz^2
    nimg = 200
    fdk = rng.uniform(-14.0, 14.0, nimg)
    ak = (rng.normal(size=nimg) + 1j * rng.normal(size=nimg)) * np.exp(-(fdk / 7.0) ** 2)
    ak[0] += 12.0
    fdk[0] = 0.0
    t = dt * np.arange(nt)
    f = df * np.arange(nf)
    E = sum(a * np.exp(2j * np.pi * (fd_ * 1e-3 * t[None, :] - eta_true * fd_ ** 2 * f[:, None]))
            for a, fd_ in zip(ak, fdk))
    dyn = np.abs(E) ** 2
    dyn = dyn + rng.normal(0.0, 0.02 * dyn.mean(), dyn.shape)
    out = dict(dyn=dyn, dt=dt, df=df, f0=f0, eta_true=eta_true)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ds = _ref_dynspec(pkg, dyn.copy(), dt, df, f0)
        ds.fit_arc(lamsteps=True, plot=False)
        out.update(betaeta=ds.betaeta, betaetaerr=ds.betaetaerr, betaetaerr2=ds.betaetaerr2,
                   noise=ds.noise, eta_array=ds.eta_array,
                   norm_sspec_avg=np.ma.filled(ds.norm_sspec_avg, np.nan),
                   nsa=np.ma.filled(ds.normsspecavg, np.nan), nsf=ds.normsspec_fdop,
                   nst=ds.normsspec_tdel, powerspectrum=np.ma.filled(ds.powerspectrum, np.nan),
                   lamsspec=ds.lamsspec, beta=ds.beta, fdop=ds.fdop, tdel=ds.tdel,
                   freq=float(ds.freq), prob_eta_peak=np.ma.filled(ds.prob_eta_peak, np.nan))
        ds.fit_arc(lamsteps=True, asymm=True, plot=False, nsmooth=7, low_power_diff=-2.0,
                   high_power_diff=-1.0)
        out.update(betaeta_left=ds.betaeta_left, betaeta_right=ds.betaeta_right,
                   betaetaerr_left=ds.betaetaerr_left, betaetaerr_right=ds.betaetaerr_right)
        ds.fit_arc(lamsteps=True, numsteps=4000, etamin=300.0, etamax=12000.0,
                   log_parabola=True, plot=False, weighted=True, cutmid=5, startbin=4)
        out.update(betaeta_log=ds.betaeta, betaetaerr_log=ds.betaetaerr,
                   betaetaerr2_log=ds.betaetaerr2)
    np.savez_compressed(os.path.join(GOLD, "fit_arc_128x160.npz"), **out)
    print("fit_arc: betaeta %.2f +- %.2f (parabola %.2f), left %.2f right %.2f, log %.2f"
          % (out["betaeta"], out["betaetaerr"], out["betaetaerr2"], out["betaeta_left"],
             out["betaeta_right"], out["betaeta_log"]))


def golden_sim(pkg):
    """scint_sim.Simulation at 64^2 / 32x96, seeded (legacy MT19937)."""
    Sim = pkg.scint_sim.Simulation
    out = {}
    cfgs = {
        "iso": dict(mb2=2, ns=64, nf=8, dlam=0.25, seed=1),
        "aniso": dict(mb2=20, ar=2, psi=30, nx=32, ny=96, nf=4, dlam=0.33,
                      seed=5, inner=0.01),
        "lam": dict(mb2=2, ns=64, nf=4, dlam=0.25, seed=3, lamsteps=True),
        "aniso2": dict(mb2=20, ar=2, psi=30, nx=32, ny=128, nf=4, dlam=0.33,
                       seed=5, inner=0.01),
        "strong": dict(mb2=200, ns=128, nf=6, dlam=0.1, seed=11, ar=1.5, psi=-20),
    }
    for tag, kw in cfgs.items():
        s = Sim(verbose=False, **kw)
        for name in ("w", "xyp", "xyi", "spe", "spi", "dyn", "freqs",
                     "times"):
            out[tag + "_" + name] = np.asarray(getattr(s, name))
        out[tag + "_eta"] = s.eta
        out[tag + "_df"] = s.df
    np.savez_compressed(os.path.join(GOLD, "sim_small.npz"), **out)
    import json
    with open(os.path.join(GOLD, "sim_small_cfg.json"), "w") as f:
        json.dump(cfgs, f, indent=1)


def main():
    os.makedirs(GOLD, exist_ok=True)
    pkg = ref_loader.load()
    only = sys.argv[1:]
    if not only or "sspec" in only:
        golden_sspec_acf(pkg)
    if not only or "c1" in only:
        golden_c1(pkg)
    if not only or "thth" in only:
        golden_thth(pkg)
    if not only or "thin" in only:
        golden_thin(pkg)
    if not only or "retrieval" in only:
        golden_retrieval(pkg)
    if not only or "tutorial" in only:
        golden_retrieval_tutorial(pkg)
    if not only or "wavefield" in only:
        golden_wavefield(pkg)
    if not only or "scale" in only:
        golden_scale_dyn(pkg)
    if not only or "norm" in only:
        golden_norm_sspec(pkg)
    if not only or "fitarc" in only:
        golden_fit_arc(pkg)
    if not only or "sim" in only:
        golden_sim(pkg)
    for fn in sorted(os.listdir(GOLD)):
        size = os.path.getsize(os.path.join(GOLD, fn))
        print(fn, size // 1024, "KiB")
        # committed fixtures stay under 1 MB each: shrink or split what grows past it
        assert size < 1000000, "%s is %d bytes" % (fn, size)


if __name__ == "__main__":
    main()
