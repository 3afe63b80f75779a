"""CPU: the C-ABI library loads and exports every symbol include/*.h declares
(no compute calls without a GPU)."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    txt = open(os.path.join(ROOT, "include", "scint_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(sb_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_header_symbols():
    import __graft_entry__ as g
    g.build()
    from scintools_b200 import _lib
    names = _declared()
    assert len(names) >= 8
    for n in names:
        assert hasattr(_lib.lib, n), "missing export %s" % n
    assert set(_lib.EXPORTS) == set(names)
    assert _lib.lib.sb_abi_version() >= 1


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from scintools_b200 import _device
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _device.device()


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "scintools_b200")
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dp, fn)).read()
                assert "import oracle" not in src and "from oracle" not in src, fn


def test_host_axes_match_oracle():
    import numpy as np
    from oracle import thth_oracle as TO
    from scintools_b200 import ththmod as thth
    t = np.arange(150) * 28.7
    f = 1400 + 0.0321 * np.arange(64)
    for pad in (0, 3):
        assert np.array_equal(thth.fft_axis(t, "mHz", pad), TO.fft_axis(t, "mHz", pad))
        assert np.array_equal(thth.fft_axis(f, "us", pad), TO.fft_axis(f, "us", pad))
    e = np.linspace(-0.4, 0.4, 512)
    assert np.array_equal(thth.theta_centres(e), TO.theta_centres(e))
    fd, tau = TO.fft_axis(t, "mHz"), TO.fft_axis(f, "us")
    assert np.array_equal(thth.min_edges(0.3, fd, tau, 50.0), TO.min_edges(0.3, fd, tau, 50.0))


def test_prep_thetatheta_notebook_kats():
    """Known answers printed in the reference's own notebook
    (scintools/examples/THTHSample.ipynb cells 13-20): edge counts and the
    first curvatures of the per-chunk eta grids.  Host logic only."""
    import numpy as np
    from scintools_b200 import BasicDyn, Dynspec
    ax = np.load(os.path.join(ROOT, "tests", "golden", "sample_axes.npz"))
    f, t = ax["f_MHz"], ax["t_s"]
    dyn = np.ones((f.shape[0], t.shape[0]))
    ds = Dynspec(dyn=BasicDyn(dyn, times=t, freqs=f, nsub=t.shape[0], nchan=f.shape[0],
                              dt=t[1] - t[0], df=f[1] - f[0]), verbose=False)
    assert ds.df == 0.12511455278581707 and ds.dt == 289.8978362416107
    # cell 20
    ds.prep_thetatheta(cwf=64, edges_lim=.3, eta_min=30, eta_max=50)
    assert (ds.cwf, ds.cwt, ds.ncf_fit, ds.nct_fit) == (64, 150, 16, 1)
    assert ds.fref == 1396.0 and (ds.eta_min, ds.eta_max) == (30.0, 50.0)
    assert ds.edges.shape[0] == 302
    etas = ds._chunk_etas(f[:64].mean())
    np.testing.assert_allclose(etas[:3], [32.75781486, 33.08757201, 33.42064867], rtol=2e-9)
    # cell 18 (eta_max there came from the Hough prior: pass the printed value)
    ds.prep_thetatheta(cwf=128, edges_lim=.3, eta_min=30, eta_max=109.11037416158051)
    assert (ds.ncf_fit, ds.ncf_ret) == (8, 15)
    assert ds.edges.shape[0] == 1318
    etas = ds._chunk_etas(f[:128].mean())
    np.testing.assert_allclose(etas[:2], [32.56235154, 32.88990503], rtol=2e-9)


def test_host_mosaic_matches_reference(golden_dir):
    """ththmod.mosaic / mask_func are sequential host numpy in the product too
    (ththmod.py:1478-1554): check them against the reference's own output."""
    import numpy as np
    from scintools_b200 import ththmod
    g = np.load(os.path.join(golden_dir, "wavefield_gs_32x64.npz"))
    mos = ththmod.mosaic(g["chunks"])
    assert mos.shape == g["mosaic"].shape
    assert np.abs(mos - g["mosaic"]).max() < 1e-13 * np.abs(g["mosaic"]).max()
    x = ththmod.mask_func(8)
    assert x[0] == 0.0 and np.all(np.diff(x) > 0) and x[-1] < 1.0


def test_thin_and_retrieval_fail_loudly_without_device(golden_dir):
    """The widened rows have no CPU fallback either."""
    import numpy as np
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from scintools_b200 import ththmod
    g = np.load(os.path.join(golden_dir, "retrieval_64x128.npz"))
    with pytest.raises(RuntimeError):
        ththmod.rev_map(np.ones(tuple(g["thth_red_shape"]), complex), g["tau"], g["fd"],
                        float(g["eta"]), g["edges_red"])
    with pytest.raises(RuntimeError):
        ththmod.thin_sweep(np.zeros((256, 512), complex), g["tau"], g["fd"],
                           np.array([40.0]), g["edges"], g["edges"][60:200], 0.0)


def test_spline_tables_match_scipy(golden_dir):
    """Host half of scale_dyn (round-2 candidate): the column-independent
    not-a-knot spline tables, applied with numpy exactly as csrc/scale_dyn.cu
    applies them, reproduce scipy's interp1d(kind='cubic') and the reference's
    lamdyn (tests/golden/scale_dyn_40x24.npz)."""
    import numpy as np
    from scipy.constants import c
    from scintools_b200.dynspec import Dynspec
    g = np.load(os.path.join(golden_dir, "scale_dyn_40x24.npz"))
    freqs, dyn = g["freqs"], g["dyn"]
    lam_eq = np.flipud(g["lam"])
    feq = np.round(np.divide(c, lam_eq) / 10 ** 6, 6)
    feq = np.clip(feq, freqs.min(), freqs.max())
    T = Dynspec._spline_tables(freqs, feq)
    n = len(freqs)
    y = dyn
    d = np.zeros_like(y)
    M = np.zeros_like(y)
    prev = np.zeros(y.shape[1])
    for i in range(1, n - 1):
        r = (y[i + 1] - y[i]) * T["g"][i] - (y[i] - y[i - 1]) * T["g"][i - 1]
        prev = (r - T["a"][i] * prev) * T["inv"][i]
        d[i] = prev
    nxt = np.zeros(y.shape[1])
    for i in range(n - 2, 0, -1):
        nxt = d[i] - T["cp"][i] * nxt
        M[i] = nxt
    M[0] = (1 + T["p0"]) * M[1] - T["p0"] * M[2]
    M[n - 1] = (1 + T["pn"]) * M[n - 2] - T["pn"] * M[n - 3]
    W, idx = T["W"], T["idx"]
    out = (W[:, 0, None] * y[idx] + W[:, 1, None] * y[idx + 1] +
           W[:, 2, None] * M[idx] + W[:, 3, None] * M[idx + 1])
    lamdyn = np.flipud(out)
    assert lamdyn.shape == g["lamdyn"].shape
    assert np.abs(lamdyn - g["lamdyn"]).max() < 1e-12 * np.abs(g["lamdyn"]).max()


def test_thetatheta_chunks_plumbing(monkeypatch):
    """Host logic of Dynspec.thetatheta_chunks / calc_wavefield with the device
    call replaced: chunk order, slices, curvature scaling, mosaic shape."""
    import numpy as np
    import scintools_b200 as sb
    from scintools_b200 import ththmod
    rng = np.random.default_rng(0)
    nf, nt = 64, 128
    dyn = rng.exponential(1.0, (nf, nt))
    t = np.arange(nt) * 20.0
    f = 1400.0 + np.arange(nf) * 0.05
    ds = sb.Dynspec(dyn=sb.BasicDyn(dyn, times=t, freqs=f, dt=20.0, df=0.05), verbose=False)
    ds.prep_thetatheta(cwf=32, cwt=64, eta_min=15.0, eta_max=60.0, nedge=96, edges_lim=8.0,
                       fw=0.2, npad=3)
    ds.ththeta = 30.0
    seen = []

    def fake(params):
        d2, edges, time2, freq2, eta, idx_t, idx_f, npad, mask, verbose = params
        seen.append((idx_f, idx_t, float(eta), float(freq2.mean()), float(time2[0])))
        return (np.full(d2.shape, idx_f + 10 * idx_t + 1j * d2[0, 0]), idx_f, idx_t)

    monkeypatch.setattr(ththmod, "single_chunk_retrieval", fake)
    ds.calc_wavefield()
    assert ds.chunks.shape == (3, 3, 32, 64)
    assert [(s[0], s[1]) for s in seen] == [(cf, ct) for cf in range(3) for ct in range(3)]
    for cf in range(3):
        for ct in range(3):
            fs = slice(cf * 16, cf * 16 + 32)
            ts = slice(ct * 32, ct * 32 + 64)
            d2 = dyn[fs, ts] - dyn[fs, ts].mean()
            assert ds.chunks[cf, ct, 0, 0] == cf + 10 * ct + 1j * d2[0, 0]
    fm = f[16:48].mean()
    assert seen[3][2] == 30.0 * (ds.fref / fm) ** 2 and seen[3][3] == fm
    assert ds.wavefield.shape == (64, 128)
