"""CPU emulation of barrier-free CUDA kernels (tests/host_emu/*.cpp compile the
.cu source with g++ and run every thread sequentially).  Used for round-2
candidates that could not be run on a GPU in round 1: it checks the device
code's arithmetic and indexing, not its performance."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "host_emu")


def _build(name):
    src = os.path.join(EMU, name + ".cpp")
    out = os.path.join(EMU, "_build", name + ".so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    csrc = os.path.join(ROOT, "scintools_b200", "csrc")
    newest = max([os.path.getmtime(os.path.join(csrc, f)) for f in os.listdir(csrc)] +
                 [os.path.getmtime(os.path.join(EMU, f)) for f in os.listdir(EMU)
                  if f.endswith((".cpp", ".h"))])
    if not os.path.exists(out) or os.path.getmtime(out) < newest:
        subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC",
                        "-x", "c++", src, "-o", out], check=True)
    return ctypes.CDLL(out)


@pytest.mark.parametrize("flip", [0, 1])
def test_scale_dyn_kernels_on_host(golden_dir, flip):
    """csrc/scale_dyn.cu (spline_moments_kernel + spline_eval_kernel) run on the
    CPU reproduce the reference's lamdyn (scale_dyn_40x24 fixture) to fp32."""
    from scipy.constants import c
    from scintools_b200.dynspec import Dynspec
    lib = _build("scale_dyn_emu")
    g = np.load(os.path.join(golden_dir, "scale_dyn_40x24.npz"))
    freqs, dyn = g["freqs"], g["dyn"]
    nf, nt = dyn.shape
    lam_eq = np.flipud(g["lam"])
    feq = np.clip(np.round(np.divide(c, lam_eq) / 10 ** 6, 6), freqs.min(), freqs.max())
    T = Dynspec._spline_tables(freqs, feq)
    d32 = np.ascontiguousarray(dyn[::-1] if flip else dyn, dtype=np.float32)
    f32 = lambda v: np.ascontiguousarray(v, dtype=np.float32)
    a, cp, inv, gg, W = f32(T["a"]), f32(T["cp"]), f32(T["inv"]), f32(T["g"]), f32(T["W"])
    idx = np.ascontiguousarray(T["idx"], dtype=np.int32)
    nlam = len(feq)
    M = np.zeros((nf, nt), np.float32)
    out = np.zeros((nlam, nt), np.float32)
    P = lambda x: x.ctypes.data_as(ctypes.c_void_p)
    lib.emu_scale_dyn.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int] + \
        [ctypes.c_void_p] * 4 + [ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_void_p,
                                 ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.emu_scale_dyn(P(d32), nf, nt, flip, P(a), P(cp), P(inv), P(gg), float(T["p0"]),
                      float(T["pn"]), P(idx), P(W), nlam, P(M), P(out))
    ref = g["lamdyn"]
    assert out.shape == ref.shape
    assert np.abs(out - ref).max() < 1e-5 * np.abs(ref).max()


def test_bf16_pack_kernel_on_host():
    """csrc/bf16_pack.cuh: round-to-nearest-even bf16 of (re, im), no overflow to
    inf, compared with torch.bfloat16."""
    import torch
    src = os.path.join(EMU, "bf16_pack_emu.cpp")
    out = os.path.join(EMU, "_build", "bf16_pack_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", out],
                   check=True)
    lib = ctypes.CDLL(out)
    rng = np.random.default_rng(0)
    n = 5000
    x = (rng.normal(size=2 * n) * 10.0 ** rng.uniform(-20, 20, 2 * n)).astype(np.float32)
    x[:8] = [0.0, -0.0, 1.0, -1.0, 3.3895314e38, -3.3895314e38, 1.0039062, 1.0117188]  # near max, ties
    xb = np.ascontiguousarray(x)
    packed = np.zeros(n, np.uint32)
    lib.emu_pack_bf16.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_long]
    lib.emu_pack_bf16(xb.ctypes.data_as(ctypes.c_void_p), packed.ctypes.data_as(ctypes.c_void_p), n)
    re = ((packed & 0xffff).astype(np.uint32) << 16).view(np.float32)
    im = (packed & 0xffff0000).view(np.float32)
    ref = torch.from_numpy(xb).to(torch.bfloat16).to(torch.float32).numpy()
    ref = np.where(np.isinf(ref), np.sign(ref) * np.float32(3.3895314e38), ref)   # we clamp, torch overflows
    assert np.array_equal(re, ref[0::2])
    assert np.array_equal(im, ref[1::2])


@pytest.mark.parametrize("n0,n1,c0,c1", [(12, 10, 0, 0), (9, 20, 5, 7), (16, 15, 16, 4)])
def test_chirp_ifft2_functors_on_host(n0, n1, c0, c1):
    """The chirp-z any-size inverse FFT (dynspec.cu::ifft2_c2c_any): tables and
    load / store functors of csrc/chirp.cuh around a reference DFT reproduce
    numpy's ifft2(ifftshift(x)) (and ifft2(conj x) for the Gerchberg-Saxton
    forward step), crop and scale included."""
    src = os.path.join(EMU, "chirp_ifft2_emu.cpp")
    out = os.path.join(EMU, "_build", "chirp_ifft2_emu.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src, "-o", out],
                   check=True)
    lib = ctypes.CDLL(out)
    lib.emu_ifft2_any.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 5 + [ctypes.c_double] + \
        [ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
    rng = np.random.default_rng(n0 * 100 + n1)
    x = (rng.normal(size=(n0, n1)) + 1j * rng.normal(size=(n0, n1))).astype(np.complex64)
    cc0, cc1 = (c0 or n0), (c1 or n1)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    got = np.zeros((cc0, cc1), np.complex64)
    lib.emu_ifft2_any(P(x), n0, n1, 1, c0, c1, 3.0, 0, 0, P(got))
    ref = 3.0 * np.fft.ifft2(np.fft.ifftshift(x))[:cc0, :cc1]
    assert np.abs(got - ref).max() < 2e-5 * np.abs(ref).max()
    gotr = np.zeros((cc0, cc1), np.float32)
    lib.emu_ifft2_any(P(x), n0, n1, 0, c0, c1, 1.0, 1, 0, P(gotr))
    refr = np.fft.ifft2(x).real[:cc0, :cc1]
    assert np.abs(gotr - refr).max() < 2e-5 * np.abs(refr).max()
    lib.emu_ifft2_any(P(x), n0, n1, 0, c0, c1, 1.0, 0, 1, P(got))
    refc = np.fft.ifft2(np.conj(x))[:cc0, :cc1]
    assert np.abs(got - refc).max() < 2e-5 * np.abs(refc).max()


def _triangles(golden_dir, etas_idx):
    """theta-theta matrices as thth_build_kernel lays them out: [ld][ld] float2,
    strict upper triangle valid, diagonal and columns >= n zero, the rest junk."""
    from oracle import thth_oracle as TO
    g = np.load(os.path.join(golden_dir, "thth_sample_64x150.npz"))
    d0 = g["dspec2"] - g["dspec2"].mean()
    CS = TO.conjugate_spectrum(d0, int(g["npad"]), 0.0)
    mats = [TO.thth_redmap(CS, g["tau"], g["fd"], g["etas"][i], g["edges"])[0] for i in etas_idx]
    ld = 32 * ((max(m.shape[0] for m in mats) + 31) // 32)
    M = np.full((len(mats), ld, ld), np.nan + 1j * np.nan, dtype=np.complex64)   # junk everywhere
    nred = np.zeros(len(mats), np.int32)
    for e, A in enumerate(mats):
        n = A.shape[0]
        nred[e] = n
        up = np.triu(A, 1).astype(np.complex64)
        blk = np.zeros((n, ld), np.complex64)
        blk[:, :n] = up
        iu = np.triu_indices(n, 0)
        rows = np.arange(n)[:, None]
        cols = np.arange(ld)[None, :]
        keep = cols >= rows                       # diagonal and everything right of it
        M[e, :n][keep] = blk[keep]
    return g, M, nred, ld


def _sweep_emu_lib(slots=0):
    """tests/host_emu/sweep_emu.cpp compiled for the CPU; slots > 0 shrinks the
    Lanczos-basis capacity of eig_half.cu so that its fp32 restart is taken."""
    src = os.path.join(EMU, "sweep_emu.cpp")
    out = os.path.join(EMU, "_build", "sweep_emu%s.so" % ("_s%d" % slots if slots else ""))
    os.makedirs(os.path.dirname(out), exist_ok=True)
    csrc = os.path.join(ROOT, "scintools_b200", "csrc")
    newest = max(os.path.getmtime(os.path.join(csrc, f)) for f in os.listdir(csrc))
    newest = max(newest, os.path.getmtime(os.path.join(EMU, "simt.h")))
    if not os.path.exists(out) or os.path.getmtime(out) < max(newest, os.path.getmtime(src)):
        subprocess.run(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-shared", "-fPIC"] +
                       (["-DSB_EB_SLOTS=%d" % slots] if slots else []) +
                       ["-x", "c++", src, "-o", out], check=True)
    return ctypes.CDLL(out)


@pytest.mark.parametrize("mixed,slots", [(0, 0), (1, 0), (2, 0), (1, 3), (3, 0), (3, 3)])
def test_default_sweep_kernels_on_host(golden_dir, mixed, slots):
    """The device code of the curvature sweep (csrc/thth.cu: thth_prep_kernel,
    thth_indexerr_kernel, thth_build_kernel; csrc/eig_half.cu) under the SIMT
    emulator, launch geometry as in sb::eta_sweep, against the reference: cropped
    sizes bit-exact, eigenvalues to 1e-5.  mixed=0: the fp32 streaming solver
    thth_eig_kernel<256, TMA, 2> (SB_EIG_FP32=1); mixed=1: the default solver
    with the packed-FMA mat-vec (fp16 iteration + fp32 Rayleigh quotient); mixed=2: its
    fp32 continuation forced on every curvature; mixed=3: the tensor-core mat-vec on the
    block layout of the fp16 copy (ldmatrix / mma.sync emulated lane-exactly);
    slots=3: the fp32 restart (basis slots exhausted)."""
    from oracle import thth_oracle as TO
    lib = _sweep_emu_lib(slots)
    g = np.load(os.path.join(golden_dir, "thth_sample_64x150.npz"))
    d0 = g["dspec2"] - g["dspec2"].mean()
    CS = TO.conjugate_spectrum(d0, int(g["npad"]), 0.0)
    cs32 = np.ascontiguousarray(CS.astype(np.complex64))
    tau, fd = g["tau"], g["fd"]
    th = TO.theta_centres(g["edges"])
    sel = [5, 37, 60, 90]
    etas = np.ascontiguousarray(g["etas"][sel])
    neta = len(sel)
    eigs = np.zeros(neta)
    status = np.zeros(neta, np.int32)
    nred = np.zeros(neta, np.int32)
    iters = np.zeros(neta, np.int32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    c_ll, c_d, c_i, vp = ctypes.c_longlong, ctypes.c_double, ctypes.c_int, ctypes.c_void_p
    lib.emu_eta_sweep.argtypes = [vp, c_ll, c_ll, c_ll, c_i, c_d, c_d, c_d, c_d, c_d, c_d, vp, c_i,
                                  c_i, vp, c_i, c_d, c_i, c_i, vp, vp, vp, vp, vp]
    ld = 32 * ((len(th) + 31) // 32)
    Mout = np.zeros((neta, ld, ld), np.complex64)
    rc = lib.emu_eta_sweep(P(cs32), CS.shape[0], CS.shape[1], CS.shape[1], 0, float(tau[0]),
                           float(np.diff(tau).mean()), float(abs(tau.max())), float(fd[0]),
                           float(np.diff(fd).mean()), float(abs(fd.max()) / 2), P(th), len(th), 1,
                           P(etas), neta, 2e-5, 0, mixed, P(eigs), P(status), P(nred), P(iters),
                           P(Mout))
    assert rc == 0
    want_n = [int(TO.th_points(tau, fd, e, g["edges"]).sum()) for e in etas]
    assert list(nred) == want_n
    assert (status == 0).all()
    # the triangle written by thth_build_kernel against the reference's thth_redmap:
    # same gathered bins (any wrong bin is an O(1) error), fp32 rounding only
    for e in range(neta):
        A = TO.thth_redmap(CS, tau, fd, etas[e], g["edges"])[0]
        n = A.shape[0]
        up = np.triu(A, 1)
        got = np.triu(Mout[e, :n, :n], 1)
        assert np.abs(got - up).max() <= 1e-6 * np.abs(up).max()
        assert np.all(Mout[e, :n, :n][np.diag_indices(n)] == 0)
    ref = g["eigs"][sel]
    assert (np.abs(eigs - ref) / ref).max() < 1e-5, (eigs, ref)


def test_thin_kernels_on_host(golden_dir):
    """csrc/thin.cu (prep, index check, two-curvature gather, sigma_max by
    Lanczos on A^H A) under the SIMT emulator against the reference's
    singularvalue_calc values (tests/golden/thth_thin_64x150.npz)."""
    from oracle import thth_oracle as TO
    lib = _build("thin_emu")
    g = np.load(os.path.join(golden_dir, "thth_sample_64x150.npz"))
    t = np.load(os.path.join(golden_dir, "thth_thin_64x150.npz"))
    d0 = g["dspec2"] - g["dspec2"].mean()
    CS = TO.conjugate_spectrum(d0, int(g["npad"]), 0.0)
    cs32 = np.ascontiguousarray(CS.astype(np.complex64))
    tau, fd = g["tau"], g["fd"]
    e1, e2 = t["edges"], t["arc"]
    th1 = np.ascontiguousarray((e1[1:] + e1[:-1]) / 2)
    th2 = np.ascontiguousarray((e2[1:] + e2[:-1]) / 2)
    sel = [2, 8, 15]
    etas = np.ascontiguousarray(t["etas"][sel])
    neta = len(sel)
    sv = np.zeros(neta)
    status = np.zeros(neta, np.int32)
    n1r = np.zeros(neta, np.int32)
    n2r = np.zeros(neta, np.int32)
    iters = np.zeros(neta, np.int32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    c_ll, c_d, c_i, vp = ctypes.c_longlong, ctypes.c_double, ctypes.c_int, ctypes.c_void_p
    lib.emu_thin_sweep.argtypes = [vp, c_ll, c_ll, c_d, c_d, c_d, c_d, c_d, vp, c_i, vp, c_i, c_d,
                                   c_i, vp, vp, c_i, c_d, c_i, vp, vp, vp, vp, vp]
    rc = lib.emu_thin_sweep(P(cs32), CS.shape[0], CS.shape[1], float(tau[1]),
                            float(np.diff(tau).mean()), float(tau.max()), float(fd[1]),
                            float(np.diff(fd).mean()), P(th1), len(th1), P(th2), len(th2),
                            float(t["cut"]), 0, P(etas), P(etas), neta, 2e-5, 0, P(sv), P(status),
                            P(n1r), P(n2r), P(iters))
    assert rc == 0
    assert (status == 0).all(), status
    ref = t["sv"][sel]
    assert (np.abs(sv - ref) / ref).max() < 1e-5, (sv, ref)


@pytest.mark.parametrize("nedge,half,coherent,mixed", [(42, 0, 1, 0), (72, 1, 1, 0), (34, 0, 0, 0),
                                                      (66, 1, 1, 1), (50, 1, 1, 2), (66, 1, 1, 3),
                                                      (42, 0, 1, 3), (34, 0, 0, 3)])
def test_default_sweep_kernels_on_host_random(nedge, half, coherent, mixed):
    """Random small spectra through the emulated sweep kernels: full and
    Hermitian-half CS layouts, incoherent mode, odd / cropped theta grids,
    curvatures that fail (NaN) -- against the numpy oracle."""
    from oracle import thth_oracle as TO
    lib = _build("sweep_emu")
    rng = np.random.default_rng(nedge)
    nf, nt, npad = 16, 64, 1
    d = rng.normal(size=(nf, nt))
    d -= d.mean()
    t = np.arange(nt) * 10.0
    f = 1400 + 0.2 * np.arange(nf)
    fd = TO.fft_axis(t, "mHz", npad)
    tau = TO.fft_axis(f, "us", npad)
    CS = TO.conjugate_spectrum(d, npad, 0.0)
    src = CS if coherent else np.abs(CS)
    edges = np.linspace(-22, 22, nedge)
    etas = np.ascontiguousarray(np.array([0.002, 0.006, 0.02, 5.0]))
    ref = TO.eta_sweep(src, tau, fd, etas, edges)
    if half:        # unshifted fd >= 0 columns of the fftshifted array, like DeviceCS
        nfd = CS.shape[1]
        cols = np.fft.ifftshift(CS, axes=1)[:, :nfd // 2 + 1]
        pitch = nfd // 2 + 16
        buf = np.zeros((CS.shape[0], pitch), np.complex64)
        buf[:, :nfd // 2 + 1] = cols
    else:
        pitch = CS.shape[1]
        buf = np.ascontiguousarray(CS.astype(np.complex64))
    th = TO.theta_centres(edges)
    neta = len(etas)
    eigs = np.zeros(neta)
    status = np.zeros(neta, np.int32)
    nred = np.zeros(neta, np.int32)
    iters = np.zeros(neta, np.int32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    c_ll, c_d, c_i, vp = ctypes.c_longlong, ctypes.c_double, ctypes.c_int, ctypes.c_void_p
    lib.emu_eta_sweep.argtypes = [vp, c_ll, c_ll, c_ll, c_i, c_d, c_d, c_d, c_d, c_d, c_d, vp, c_i,
                                  c_i, vp, c_i, c_d, c_i, c_i, vp, vp, vp, vp, vp]
    ld = 32 * ((len(th) + 31) // 32)
    Mout = np.zeros((neta, ld, ld), np.complex64)
    rc = lib.emu_eta_sweep(P(buf), CS.shape[0], CS.shape[1], pitch, half, float(tau[0]),
                           float(np.diff(tau).mean()), float(abs(tau.max())), float(fd[0]),
                           float(np.diff(fd).mean()), float(abs(fd.max()) / 2), P(th), len(th),
                           coherent, P(etas), neta, 2e-5, 0, mixed, P(eigs), P(status), P(nred),
                           P(iters), P(Mout))
    assert rc == 0
    for e in range(neta):       # built triangle vs the reference's thth_redmap (cropped sizes vary)
        try:
            A = TO.thth_redmap(src, tau, fd, etas[e], edges)[0]
        except Exception:
            continue
        n = A.shape[0]
        if n < 2 or status[e] != 0:
            continue
        up = np.triu(A, 1)
        got = np.triu(Mout[e, :n, :n], 1)
        assert np.abs(got - up).max() <= 1e-6 * max(np.abs(up).max(), 1e-30)
    want_n = [int(TO.th_points(tau, fd, e, edges).sum()) for e in etas]
    assert list(nred) == want_n
    assert np.array_equal(np.isnan(eigs), np.isnan(ref)), (eigs, ref, status)
    ok = ~np.isnan(ref)
    assert (np.abs(eigs[ok] - ref[ok]) / ref[ok]).max() < 1e-5, (eigs, ref)


def test_retrieval_kernels_on_host(golden_dir):
    """csrc/retrieval.cu under the SIMT emulator: the histogram2d scatter
    (bit-exact bins) and the top-eigenpair kernel against the reference's
    rev_map / modeler outputs (tests/golden/retrieval_64x128.npz)."""
    from oracle import retrieval_maps
    from oracle import thth_oracle as TO
    lib = _build("retrieval_emu")
    g = np.load(os.path.join(golden_dir, "retrieval_64x128.npz"))
    maps = retrieval_maps(g)
    tau, fd, eta = g["tau"], g["fd"], float(g["eta"])
    th = TO.theta_centres(g["edges_red"])
    n = len(th)
    rng = np.random.default_rng(int(g["tt_seed"]))
    tt = (rng.normal(size=(n, n)) + 1j * rng.normal(size=(n, n))).astype(np.complex64)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    c_d, c_i, vp = ctypes.c_double, ctypes.c_int, ctypes.c_void_p
    lib.emu_rev_map.argtypes = [vp, c_i, vp, c_d, c_d, c_d, c_i, c_d, c_d, c_i, c_i, vp]
    for herm, key in ((1, "rv_h"), (0, "rv_n")):
        out = np.zeros((len(tau), len(fd)), np.complex64)
        lib.emu_rev_map(P(np.ascontiguousarray(tt)), n, P(th), eta, float(tau[0]),
                        float(tau[1] - tau[0]), len(tau), float(fd[0]), float(fd[1] - fd[0]),
                        len(fd), herm, P(out))
        ref = maps[key]
        assert np.array_equal(out == 0, ref == 0)
        assert np.abs(out - ref).max() < 1e-5 * np.abs(ref).max()
    A = np.ascontiguousarray(maps["thth_red"].astype(np.complex64))
    w = np.zeros(1)
    V = np.zeros(n, np.complex64)
    info = np.zeros(2, np.int32)
    lib.emu_herm_eigvec.argtypes = [vp, c_i, c_i, c_d, c_i, vp, vp, vp]
    lib.emu_herm_eigvec(P(A), n, n, 1e-7, 96, P(w), P(V), P(info))
    assert w[0] == pytest.approx(float(g["w"]), rel=1e-5)
    Vr = g["V"].astype(complex)
    z = np.vdot(V, Vr)
    assert np.abs(V * (z / abs(z)) - Vr).max() < 3e-5 * np.abs(Vr).max()


@pytest.mark.parametrize("mixed", [0, 1, 3])
def test_slowly_converging_curvature_on_host(golden_dir, mixed):
    """Regression for the round-1 stopping bug (lanczos.cuh: the residual estimate
    collapsed to 0 at the first range rescaling of the Sturm sequence, step ~21 for
    eigenvalues ~3e7): curvature 121 of the full-size bench workload needs 38 Lanczos
    steps (the top Ritz value plateaus 0.5 % low for steps 13-20).  Both solvers must
    reach the dense eigenvalue."""
    lib = _sweep_emu_lib(0)
    g = np.load(os.path.join(golden_dir, "thth_hard_511.npz"))
    n, ld = int(g["n"]), 512
    M = np.zeros((1, ld, ld), np.complex64)
    M[0][np.triu_indices(n, 1)[0], np.triu_indices(n, 1)[1]] = g["upper"]
    nred = np.array([n], np.int32)
    eigs = np.zeros(1)
    st = np.zeros(1, np.int32)
    it = np.zeros(1, np.int32)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    lib.emu_eig_triangles.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_double, ctypes.c_int, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p]
    lib.emu_eig_triangles(P(M), ld, P(nred), 1, mixed, 2e-5, 0, P(eigs), P(st), P(it))
    assert st[0] == 0
    assert abs(eigs[0] - float(g["top"])) / float(g["top"]) < 1e-6, (eigs, it)
    assert it[0] > 30
