#!/usr/bin/env python
"""Benchmark of the theta-theta curvature sweep (BASELINE.json metric:
"theta-theta eta-trials/sec on 4096x8192 dynspec").

One *step* = one pass of the hot path over one dynamic spectrum:
  conjugate spectrum of the 4096x8192 chunk (npad=3 -> 16384x32768 c64, 4.3 GB)
  + dominant-eigenvalue sweep over 1024 curvatures on a 512-point theta grid
  (+ one all-gather of the per-eta eigenvalues when N > 1).
Weak scaling: every rank sweeps 1024 etas of a global N x 1024 log grid,
interleaved over the ranks (the CS is recomputed per rank; no data-path
collective); a strong-scaling leg over a fixed 8192-eta grid is reported too.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                  [--dump-outputs DIR]

The b200 arm reports device-resident throughput (`value`), end-to-end
throughput through the public API with pinned host buffers (`e2e`), the
roofline of the dominant kernel and a CPU baseline measured in the same run.
The reference arm times the reference's CPU algorithm (oracle port:
numpy gather + scipy ARPACK, pocketfft CS) on the host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "theta-theta eta-trials/sec on 4096x8192 dynspec"
NF, NT, NPAD = 4096, 8192, 3
NETA, NEDGE = 1024, 512
ETA_TRUE = 0.08          # s^3
DT, DF = 10.0, 0.03125   # s, MHz
EDGE_LIM = 10.0          # mHz
FW = 0.1
WORKLOAD = ("C3 eta-sweep: 4096x8192 dynspec (1-D screen, 64 images, eta_true=0.08 s^3), "
            "npad=3 -> CS 16384x32768, 512-pt theta grid, 1024 etas per GPU")


def make_dynspec(seed=3, nf=NF, nt=NT):
    """SURVEY.md section 8(d) C3: 64-image 1-D screen, eta_true = 0.08 s^3.
    E(f,t) = sum_k a_k exp(2 pi i (fd_k t - tau_k f)) is separable per image,
    so it is one (nf x 64) @ (64 x nt) product."""
    rng = np.random.default_rng(seed)
    nimg = 64
    fdk = rng.uniform(-8.0, 8.0, nimg)                       # mHz
    ak = (rng.normal(size=nimg) + 1j * rng.normal(size=nimg)) / np.sqrt(2)
    ak = ak * np.exp(-(fdk / 4.0) ** 2)
    tauk = ETA_TRUE * fdk ** 2                               # us
    t = DT * np.arange(nt)
    f = DF * np.arange(nf)                                   # MHz offset
    U = np.exp(2j * np.pi * 1e-3 * fdk[:, None] * t[None, :])
    V = np.exp(-2j * np.pi * tauk[None, :] * f[:, None]) * ak[None, :]
    E = (V.astype(np.complex64) @ U.astype(np.complex64))
    dyn = (E.real ** 2 + E.imag ** 2).astype(np.float32)
    dyn += rng.normal(0.0, 0.2 * dyn.mean(), dyn.shape).astype(np.float32)
    dyn -= dyn.mean()
    return dyn, 1400.0 + f, t


def eta_grid(n_total):
    return np.logspace(np.log10(ETA_TRUE / 2), np.log10(2 * ETA_TRUE), n_total)


def peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi sampling in the background (started well before the timed
    region so that it is already polling); `stop(t0, t1)` keeps the samples
    whose timestamp falls inside the timed window (wall clock), falling back to
    the samples taken under load (power above half of the maximum seen)."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "20"],
                stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self, t0=None, t1=None):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        time.sleep(0.05)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                 "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(parts[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(parts[1]), float(parts[2]), float(parts[3]),
                             [nm for nm, v in zip(names, parts[4:8])
                              if v.lower().startswith("active")]))
            except ValueError:
                continue
        os.unlink(self.f.name)
        if not rows:
            return out
        sel = [r for r in rows if t0 is not None and t0 - 0.03 <= r[0] <= t1 + 0.03]
        how = "timed window"
        if not sel:
            pmax = max(r[3] for r in rows)
            sel = [r for r in rows if r[3] >= 0.5 * pmax]
            how = "samples under load around the timed window"
        reasons = sorted({x for r in sel for x in r[4]})
        return {"sm_mhz": float(np.median([r[1] for r in sel])),
                "sm_max_mhz": float(max(r[2] for r in sel)), "reasons": reasons,
                "power_w_max": float(max(r[3] for r in sel)),
                "samples": len(sel), "from": how}


# --------------------------------------------------------------------------
# CPU arms (oracle port of the reference algorithm)
# --------------------------------------------------------------------------
_G = {}


def _pool_init():
    """One BLAS/OpenMP thread per pool worker (no oversubscription)."""
    try:
        from threadpoolctl import threadpool_limits
        _G["limited"] = threadpool_limits(1)
    except Exception:
        _G["limited"] = True


def _eval_one(eta):
    from oracle import thth_oracle as TO
    try:
        return TO.Eval_calc(_G["CS"], _G["tau"], _G["fd"], eta, _G["edges"])
    except Exception:
        return float("nan")


class CpuSweep:
    """The reference's eta loop (ththmod.py:789-799) on the host cores.

    procs == 1: the as-shipped serial loop, one BLAS thread (numpy.fft and the
    eta loop of the reference are single-threaded).  procs > 1: the reference's
    own parallel mode, a process pool (dynspec.py:1715-1719 maps chunks over a
    pool; here the pool maps the eta-trials of one chunk).  The pool is created
    ONCE (fork: the workers share the CS copy-on-write) and re-used by every
    timed step; workers run one BLAS thread each."""

    def __init__(self, CS, tau, fd, edges, procs):
        _G.update(CS=CS, tau=tau, fd=fd, edges=edges)
        self.procs = procs
        self.pool = None
        self.limit = None
        if procs > 1:
            import multiprocessing as mp
            self.pool = mp.get_context("fork").Pool(procs, initializer=_pool_init)
        else:
            try:
                from threadpoolctl import threadpool_limits
                self.limit = threadpool_limits(1)
            except Exception:
                self.limit = None

    def run(self, etas):
        """Returns (seconds, eigs) for len(etas) eta-trials."""
        t0 = time.perf_counter()
        if self.pool is None:
            eigs = [_eval_one(e) for e in etas]
        else:
            eigs = self.pool.map(_eval_one, list(etas), chunksize=1)
        return time.perf_counter() - t0, np.array(eigs)

    def close(self):
        if self.pool is not None:
            self.pool.close()
            self.pool.join()
        if self.limit is not None and hasattr(self.limit, "restore_original_limits"):
            self.limit.restore_original_limits()


def reference_arm(args):
    """`--impl reference`: the reference's CPU algorithm (oracle port: numpy gather +
    scipy ARPACK eigsh, scipy pocketfft CS) on all host cores.  One step = a
    bounded sample of the C3 workload: `per_worker` eta-trials per pool worker,
    drawn from the same eta grid; the CS FFT (once per 1024 etas in the real
    workload) is timed once and charged pro rata to every step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import scipy.fft as sfft
    from oracle import thth_oracle as TO
    cores = len(os.sched_getaffinity(0))
    dyn, freq, t = make_dynspec()
    fd = TO.fft_axis(t, "mHz", NPAD)
    tau = TO.fft_axis(freq, "us", NPAD)
    edges = np.linspace(-EDGE_LIM, EDGE_LIM, NEDGE)
    pad = np.zeros(((NPAD + 1) * NF, (NPAD + 1) * NT), dtype=np.float32)
    pad[:NF, :NT] = dyn
    sfft.fft2(pad[:256, :256], workers=cores)               # thread-pool warm-up
    t0 = time.perf_counter()
    CS = sfft.fftshift(sfft.fft2(pad, workers=cores))       # pocketfft, c64
    t_cs = time.perf_counter() - t0
    del pad
    etas = eta_grid(NETA * args.gpus)
    per_worker = 8
    nsamp = per_worker * cores
    rng = np.random.default_rng(0)
    sweep = CpuSweep(CS, tau, fd, edges, cores)
    times = []
    for it in range(max(1, args.warmup) + args.steps):      # >= 1 warm-up step (page-in, BLAS init)
        sel = np.sort(rng.choice(len(etas), nsamp, replace=len(etas) < nsamp))
        dt_, _ = sweep.run(etas[sel])
        if it >= max(1, args.warmup):
            times.append(dt_)
    sweep.close()
    # as-shipped single process (serial eta loop), same grid
    one = CpuSweep(CS, tau, fd, edges, 1)
    one.run(etas[:1])
    sel1 = np.linspace(0, len(etas) - 1, 8).astype(int)
    t_one, _ = one.run(etas[sel1])
    one.close()
    cs_share = t_cs * nsamp / NETA                           # one CS per 1024 eta-trials
    per_step = float(np.mean(times)) + cs_share
    value = nsamp / per_step
    sample = ("%d eta-trials per step (%d per worker) over a persistent %d-process fork pool, "
              "1 BLAS thread each, on the full-size CS; + %.3f s per step = the CS FFT "
              "(scipy pocketfft c64, %d threads: %.1f s per 1024 etas) pro rata"
              % (nsamp, per_worker, cores, cs_share, cores, t_cs))
    line = {
        "impl": "reference", "metric": METRIC, "value": value,
        "unit": "eta-trials/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": max(1, args.warmup), "ms_per_step": per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "note": "reference algorithm (numpy gather + scipy ARPACK "
                           "eigsh) via the oracle port; astropy unavailable"},
        "cpu_baseline": {"value": value, "unit": "eta-trials/s", "cores": cores,
                         "kind": "port", "sample": sample,
                         "step_spread": [float(min(times)), float(max(times))],
                         "single_process": {"value": len(sel1) / t_one, "cores": 1,
                                            "sample": "8 eta-trials, serial loop, 1 BLAS "
                                                      "thread (as shipped), CS FFT not counted"}},
        "e2e": {"value": value, "unit": "eta-trials/s",
                "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------
PROF_NAMES = ["cs_rows", "cs_colA", "cs_colB", "thth_prep", "thth_build",
              "thth_eig", "sspec", "acf", "sim_screen", "sim_freq"]
NETA_STRONG = 8192       # fixed global grid of the strong-scaling leg


def ncu_traffic(kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, read at
    run time from the committed summary of the `ncu --set full` capture of this
    same command (profiles/r2_ncu_traffic.json, written by profiles/ncu_traffic.py
    from the .ncu-rep).  None when the capture does not list the kernel."""
    path = os.path.join(ROOT, "profiles", "r2_ncu_traffic.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        return d["kernels"][kernel]["dram_bytes"], "profiles/r2_ncu_traffic.json (%s)" % d.get("source", "")
    except Exception:
        return None, "no committed ncu capture lists this kernel"


def collect_prof(L, _lib):
    ms = np.zeros(16)
    cnt = np.zeros(16, dtype=np.int32)
    _lib.check(L.sb_profile_collect(ms.ctypes.data, cnt.ctypes.data, 16))
    return ms, cnt


CS_SAMPLE = 1 << 20      # CS points written by --dump-outputs (8 MB)


def dump_outputs(out_dir, buf, d_cs, ncols):
    """What the last timed step computed, as DIR/<name>.npy: the sweep's per-eta
    outputs in full (float64) and a fixed, seeded sample of the conjugate spectrum
    (the fd >= 0 columns it computed; float32 [re, im] pairs), for comparing the
    outputs of two builds run with the same arguments."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name in ("eigs", "stat", "nred", "iters"):
        np.save(os.path.join(out_dir, name + ".npy"),
                buf[name].cpu().numpy().astype(np.float64))
    rng = np.random.default_rng(0)
    rows = torch.from_numpy(rng.integers(0, d_cs.shape[0], CS_SAMPLE)).to(d_cs.device)
    cols = torch.from_numpy(rng.integers(0, ncols, CS_SAMPLE)).to(d_cs.device)
    np.save(os.path.join(out_dir, "cs_sample.npy"), d_cs[rows, cols].cpu().numpy())


def b200_arm(args):
    import torch
    import torch.distributed as dist
    from scintools_b200 import _device as D
    from scintools_b200 import _lib
    from scintools_b200 import ththmod as thth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = D.device()
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    clocks = ClockSampler(local)      # polling from the start; windowed later
    dyn, freq, t = make_dynspec()
    fd = np.asarray(thth.fft_axis(t, "mHz", NPAD))
    tau = np.asarray(thth.fft_axis(freq, "us", NPAD))
    edges = np.linspace(-EDGE_LIM, EDGE_LIM, NEDGE)
    # weak scaling: a global grid of world x 1024 curvatures, INTERLEAVED over the
    # ranks (rank r sweeps etas_all[r::world]) so that every rank gets the same mix
    # of easy (near the peak) and hard curvatures
    etas_all = eta_grid(NETA * world)
    etas = np.ascontiguousarray(etas_all[rank::world])

    # device-resident inputs
    d_dyn = D.upload(dyn)
    ntau, nfd = (NPAD + 1) * NF, (NPAD + 1) * NT
    pitch = nfd // 2 + 16          # Hermitian half-plane CS (fd >= 0)
    d_cs = D.empty((ntau, pitch, 2), torch.float32)
    # the sweep gathers at fd = theta_j - theta_i <= 2*EDGE_LIM: only those fd
    # columns of the CS are computed (exactly what single_search does)
    keep = thth.needed_fd_columns(fd, edges) or 0
    d_bound = D.empty((1,), torch.float32)      # L1 bound of |CS| (scale of the solver's fp16 copy)
    cs = thth.DeviceCS(d_cs, nfd=nfd, ncols_valid=keep or None, bound=d_bound)
    geom = thth._Geom(cs, tau, fd, edges, True)
    stream = D.stream_ptr()
    L = _lib.lib

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_leg(etas_local):
        n = len(etas_local)
        buf = dict(n=n, etas=D.upload(np.ascontiguousarray(etas_local)),
                   eigs=D.empty((n,), torch.float64), stat=D.empty((n,), torch.int32),
                   nred=D.empty((n,), torch.int32), iters=D.empty((n,), torch.int32),
                   gathered=D.empty((world * n,), torch.float64) if world > 1 else None)

        def step():
            _lib.check(L.sb_cs_f32(d_dyn.data_ptr(), NF, NT, NPAD, 0.0, 0, 1, pitch, keep,
                                   d_cs.data_ptr(), stream))
            _lib.check(L.sb_cs_bound_f32(d_dyn.data_ptr(), NF, NT, NPAD, 0.0, d_bound.data_ptr(),
                                         stream))
            _lib.check(L.sb_eta_sweep(geom.ref, buf["etas"].data_ptr(), n, thth.DEFAULT_TOL,
                                      0, buf["eigs"].data_ptr(), buf["stat"].data_ptr(),
                                      buf["nred"].data_ptr(), buf["iters"].data_ptr(), stream))
            if world > 1:
                dist.all_gather_into_tensor(buf["gathered"], buf["eigs"])
        return buf, step

    def timed(step, warmup, steps):
        """W warm-up steps, then K steps between barrier + synchronize; device time by
        CUDA events, max over ranks; per-kernel CUDA-event times, max over ranks."""
        for _ in range(warmup):
            step()
        sync_all()
        launches0 = L.sb_launch_count()
        L.sb_profile_enable(1)
        ev0 = torch.cuda.Event(enable_timing=True)
        ev1 = torch.cuda.Event(enable_timing=True)
        sync_all()
        wall0 = time.time()
        ev0.record()
        for _ in range(steps):
            step()
        ev1.record()
        sync_all()
        wall1 = time.time()
        launches = int(L.sb_launch_count() - launches0)
        pm, pc = collect_prof(L, _lib)
        L.sb_profile_enable(0)
        # per-kernel device time PER STEP (a kernel may be launched several times per
        # step: column chunks of the CS, eta batches of a long sweep)
        per = torch.tensor(np.concatenate(([ev0.elapsed_time(ev1)], pm / steps)),
                           device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(per, op=dist.ReduceOp.MAX)
        per = per.cpu().numpy()
        kern = {n_: float(per[1 + i]) for i, n_ in enumerate(PROF_NAMES) if pc[i]}
        return float(per[0]) / steps, kern, launches, (wall0, wall1)

    # ---- headline (weak) leg ------------------------------------------------
    wbuf, wstep = make_leg(etas)
    ms_step, kern, launches, (wall0, wall1) = timed(wstep, args.warmup, args.steps)
    clk = clocks.stop(wall0, wall1)
    if args.dump_outputs and rank == 0:
        # before the strong leg, which reuses d_cs
        dump_outputs(args.dump_outputs, wbuf, d_cs, keep or nfd // 2 + 1)
    value = world * NETA / (ms_step * 1e-3)
    eigs = wbuf["eigs"].cpu().numpy()
    nred = wbuf["nred"].cpu().numpy().astype(np.int64)
    iters = wbuf["iters"].cpu().numpy()
    status = wbuf["stat"].cpu().numpy()

    # algorithmic bytes of one launch of the sweep kernels: one c64 gather of the
    # strict upper triangle + one f64 eigenvalue per eta (SURVEY.md 8d)
    alg_bytes = float(np.sum(8 * nred * (nred - 1) // 2 + 8))
    dom = max((k for k in kern if k.startswith("thth")), key=lambda k: kern[k])
    peak, peak_src = peak_hbm()
    ach = alg_bytes / (kern[dom] * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic(dom)
    roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak,
                "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": alg_bytes,
                "note": "iterative solver: every Lanczos step streams the triangle once "
                        "(scaled fp16 copy in 512-byte blocks for the tensor-core mat-vec, 0.54 MB at "
                        "N=511, ~19 steps + 1 surplus step of the deferred convergence check) + "
                        "one fp32 pass for the Rayleigh quotient "
                        "= `traffic`; kernel_ms = CUDA events on the launching stream per step, "
                        "max over ranks",
                "kernel_ms": kern}

    # ---- strong-scaling leg: fixed 8192-eta grid split over the ranks ----------
    strong = None
    if not args.no_strong:
        es_all = eta_grid(NETA_STRONG)
        sbuf, sstep = make_leg(es_all[rank::world])
        s_ms, s_kern, _, _ = timed(sstep, 2, max(2, args.steps // 2))
        strong = {"etas_total": NETA_STRONG, "etas_per_gpu": sbuf["n"], "ms_per_step": s_ms,
                  "value": NETA_STRONG / (s_ms * 1e-3), "unit": "eta-trials/s",
                  "scaling": "strong", "kernel_ms": s_kern,
                  "note": "same step (CS recomputed on every rank + sweep + all-gather) over a "
                          "FIXED grid of 8192 curvatures interleaved over the ranks"}
        del sbuf

    # ---- end to end through the public API, pinned host input ----------
    def e2e_leg(h_dyn):
        """ththmod.search_batch over `steps` chunks: every chunk's dynamic spectrum is
        copied from pinned host memory inside the timed region (the copy of chunk i+1
        overlaps the sweep of chunk i), eigenvalues come back to the host, the
        parabola fit runs on the host."""
        params = [h_dyn, freq, t, etas, edges, None, False, FW, NPAD, True, 0.0, False]
        thth.search_batch([params] * 2)
        vals = []
        for _ in range(3):      # a leg is ~30 ms at 5 steps: median of three (host jitter)
            sync_all()
            t0 = time.perf_counter()
            res = thth.search_batch([params] * args.steps)
            torch.cuda.synchronize()
            dt_ = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(dt_, op=dist.ReduceOp.MAX)
            vals.append(world * NETA / (float(dt_.item()) / args.steps))
        return sorted(vals)[1], res[-1]

    h32 = torch.from_numpy(dyn).pin_memory()
    e2e_val, res = e2e_leg(h32.numpy())
    e2e = {"value": e2e_val, "unit": "eta-trials/s",
           "h2d_bytes_per_step": int(dyn.nbytes + etas.nbytes + 8 * (NEDGE - 1)),
           "d2h_bytes_per_step": int(8 * NETA),
           "api": "scintools_b200.ththmod.search_batch([params] * steps) (the loop of "
                  "Dynspec.fit_thetatheta) incl. host parabola fit; dyn float32 in pinned "
                  "host memory; median of three timed batches of `steps` chunks",
           "eta_fit": float(res[0])}
    e2e_f64 = None
    if not args.no_extra:
        h64 = torch.from_numpy(dyn.astype(np.float64)).pin_memory()
        v64, _ = e2e_leg(h64.numpy())
        e2e_f64 = {"value": v64, "unit": "eta-trials/s",
                   "h2d_bytes_per_step": int(8 * dyn.size + etas.nbytes + 8 * (NEDGE - 1)),
                   "d2h_bytes_per_step": int(8 * NETA),
                   "note": "same call with the reference's dtype: float64 host dynamic "
                           "spectrum (narrowed to fp32 on the device)"}
        del h64
    del h32

    line = None
    if rank == 0:
        cpu = None
        if world == 1 and not args.no_cpu:
            cpu = cpu_baseline_leg(thth, dyn, tau, fd, edges, etas, eigs)
        extra = None
        if world == 1 and not args.no_extra:
            extra = other_configs(peak)
        line = {
            "metric": METRIC, "value": value, "unit": "eta-trials/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "etas_total": world * NETA,
                       "cs": "fd>=0 half stored (2.15 GB c64), recomputed every step; "
                             "%d of %d fd>=0 columns computed (those the 512-pt theta grid "
                             "can reach)" % (keep or nfd // 2 + 1, nfd // 2 + 1),
                       "l2": "inputs larger than L2 (CS half-plane 2.15 GB, matrices 1.6 GB)",
                       "tol": thth.DEFAULT_TOL,
                       "parallelism": "global eta grid interleaved over the ranks, CS "
                                      "replicated, one NCCL all-gather of eigenvalues per step"},
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "e2e_f64": e2e_f64,
            "strong": strong, "extra": extra,
            "gpu_launches": launches, "clocks": clk,
            "sweep": {"nred_min": int(nred.min()), "nred_max": int(nred.max()),
                      "iters_mean": float(iters.mean()), "iters_max": int(iters.max()),
                      "iters_hist": {"<=20": int((iters <= 20).sum()),
                                     "21-24": int(((iters > 20) & (iters <= 24)).sum()),
                                     "25-32": int(((iters > 24) & (iters <= 32)).sum()),
                                     ">32": int((iters > 32).sum())},
                      "status_nonzero": int((status != 0).sum()),
                      "eta_peak": float(etas[np.nanargmax(eigs)])},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def cpu_baseline_leg(thth, dyn, tau, fd, edges, etas, eigs):
    """cpu_baseline of the b200 arm: the oracle port on ONE host core (the
    as-shipped serial eta loop), 1 warm-up + 24 eta-trials (about 10-20 s)."""
    full = thth.conjugate_spectrum(dyn, NPAD, 0.0)      # all columns, for the CPU leg
    CS_host = full.numpy().astype(np.complex64)
    del full
    one = CpuSweep(CS_host, tau, fd, edges, 1)
    one.run(etas[:1])
    sel = np.linspace(0, NETA - 1, 24).astype(int)
    secs, ref = one.run(etas[sel])
    one.close()
    rel = np.abs(eigs[sel] - ref) / np.abs(ref)
    return {"value": len(sel) / secs, "unit": "eta-trials/s", "cores": 1, "kind": "port",
            "sample": "24 of 1024 eta-trials after 1 warm-up trial (oracle Eval_calc: numpy "
                      "gather + scipy ARPACK, 1 BLAS thread) on the GPU-built 16384x32768 "
                      "CS; the CPU fft2 of the CS is not counted",
            "max_rel_err_vs_gpu": float(np.nanmax(rel))}


def other_configs(peak):
    """BASELINE.json configs 2 and 4 in the same process (rank 0, one GPU):
    C2 calc_sspec / calc_acf on a 4096x8192 dynamic spectrum, C4 one 8192^2
    Simulation realisation (8 frequencies timed).  Device ms = CUDA events of the
    library call (sb_profile); e2e ms = the public API call from pinned host
    float32 memory to the host result; frac = algorithmic bytes (SURVEY.md 8d)
    / device time / measured HBM peak."""
    import torch
    from scintools_b200 import _lib, BasicDyn, Dynspec
    from scintools_b200.scint_sim import Simulation
    L = _lib.lib
    rng = np.random.default_rng(2)
    dyn = torch.from_numpy(rng.exponential(1.0, (NF, NT)).astype(np.float32)).pin_memory().numpy()
    ds = Dynspec(dyn=BasicDyn(dyn, times=10.0 * np.arange(NT), freqs=1400 + DF * np.arange(NF),
                              dt=10.0, df=DF), verbose=False)

    def prof(fn, reps):
        fn()
        torch.cuda.synchronize()
        L.sb_profile_enable(1)
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) / reps
        ms, cnt = collect_prof(L, _lib)
        L.sb_profile_enable(0)
        return wall, ms, cnt

    out = {}
    w, ms, cnt = prof(lambda: ds.calc_sspec(dtype=np.float32), 3)
    tms = ms[6] / cnt[6]
    alg = 4 * NF * NT + 4 * NF * 2 * NT
    out["c2_sspec"] = {"device_ms": tms, "e2e_ms": w * 1e3, "algorithmic_bytes": alg,
                       "achieved_GBs": alg / tms / 1e6, "frac": alg / tms / 1e6 / peak}
    w, ms, cnt = prof(lambda: ds.calc_acf(dtype=np.float32), 3)
    tms = ms[7] / cnt[7]
    alg = 4 * NF * NT + 4 * 2 * NF * 2 * NT
    out["c2_acf"] = {"device_ms": tms, "e2e_ms": w * 1e3, "algorithmic_bytes": alg,
                     "achieved_GBs": alg / tms / 1e6, "frac": alg / tms / 1e6 / peak}
    del ds, dyn
    nfreq, n = 8, 8192
    w, ms, cnt = prof(lambda: Simulation(mb2=2, ns=n, nf=nfreq, dlam=0.25, seed=1,
                                         device_rng=True), 1)
    per_f = ms[9] / cnt[9]
    out["c4_sim"] = {"ns": n, "nf_timed": nfreq, "screen_ms": ms[8] / cnt[8],
                     "per_freq_ms": per_f, "e2e_s": w,
                     "per_freq_algorithmic_bytes": 52 * n * n,
                     "achieved_GBs": 52 * n * n / per_f / 1e6,
                     "frac": 52 * n * n / per_f / 1e6 / peak,
                     "realisation_nf256_est_s": (ms[8] / cnt[8] + 256 * per_f) / 1e3,
                     "note": "the library reads 20 n^2 B per frequency (collapsed inverse, "
                             "DESIGN.md); frac is quoted against the faithful plan's 52 n^2"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu", action="store_true",
                    help="skip the cpu_baseline leg (profiling runs)")
    ap.add_argument("--no-strong", action="store_true",
                    help="skip the strong-scaling leg (profiling runs)")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip e2e_f64 and the C2/C4 extra configs (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed as "
                         "DIR/<name>.npy (b200 arm; rank 0's share when --gpus > 1)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        return reference_arm(args)
    return b200_arm(args)


if __name__ == "__main__":
    sys.exit(main())
