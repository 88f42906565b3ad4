#!/usr/bin/env python
"""bench.py -- Navier2D timesteps/s on B200 (BASELINE.json metric), one JSON line on stdout.

  python bench.py --gpus N --steps K --warmup W [--config C2|C3|C4|C1] [--impl reference] [--dump-outputs DIR]

A "step" is one `Navier2D::update()` (src/navier_stokes/navier.rs:438-466) on synthetic fields:
constructor defaults, physical fields U(-0.1, 0.1) from numpy default_rng(1/2/3), forward().
Default workload at every N: BASELINE configs[3] = confined 4097 x 4097 Chebyshev x Chebyshev, Ra 1e9, dt 1e-4
(the configuration the metric "at 1/2/4/8 B200" and the north-star roofline target are quoted on; it fits one GPU).
--config C2 = configs[1] (1025 x 1025), C3 = configs[2] (periodic 2048 x 1025), C1 = configs[0] (129 x 129).

value  : steps/s with state resident in HBM, CUDA events on the library's stream, max over ranks.
e2e    : the same step through the public API with HOST state: every step uploads the four
         spectral state arrays from pinned host memory, steps, and downloads them again.
roofline: HBM-bound lane kernels: algorithmic bytes per step (SURVEY 8d: 728 N) / time in lane kernels.
ops    : ms / transform and ms / solve (the second half of BASELINE.json's metric): forward, backward, to_ortho, from_ortho,
         gradient, HholtzAdi and Poisson on standalone fields of the benchmarked size, each against its algorithmic bytes.
cpu_baseline / --impl reference: the C++/OpenMP restatement of the reference's update() (oracle/cpu_restated.cpp: one
         pass per reference call, lane-parallel, OpenBLAS DGEMM) timed on the host cores (the Rust reference cannot be
         built in this image: no cargo/rustc).
parity_check: 2 steps of a 257 x 129 problem on the same ranks against the numpy oracle (smooth state: 1e-10; white noise:
         max(1e-10, 10 x the oracle's own response to a last-bit change of its input)); parity_check_workload: the
         benchmarked configuration itself against the C++ restatement (1 GPU).
--dump-outputs DIR: the four spectral state arrays (temp, velx, vely, pres) as the last timed step left them, written to
         DIR/<name>.npy (see dump_outputs), so that two builds can be compared output for output on identical inputs.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
if os.environ.get("OMP_NUM_THREADS") == "1" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
    # torchrun pins OMP_NUM_THREADS=1; the (untimed) host LAPACK setup of the Poisson solver is minutes at one thread: give every
    # rank its share of the host cores before numpy / OpenBLAS load
    os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // int(os.environ["WORLD_SIZE"])))
os.environ.setdefault("OMP_WAIT_POLICY", "PASSIVE")   # CPU arm: idle OpenMP threads must not spin against OpenBLAS's own pool

CONFIGS = {
    # name: (nx, ny, ra, dt, periodic)
    "C1": (129, 129, 1e5, 1e-2, False),
    "C2": (1025, 1025, 1e7, 1e-3, False),
    "C3": (2048, 1025, 1e7, 1e-3, True),
    "C4": (4097, 4097, 1e9, 1e-4, False),
    "C5": (8192, 4097, 1e10, 5e-5, True),   # BASELINE configs[4]
    "C6": (8193, 8193, 1e10, 5e-5, False),  # north_star scaling case (8193^2 confined); host LAPACK setup takes minutes (cached via B2_EIG_CACHE)
}


def config_dict(cfg):
    """`config` of the JSON line: identical in both arms (the repo arm's run details go to `run`)."""
    nx, ny = CONFIGS[cfg][:2]
    return {"workload": workload_name(cfg), "config": cfg,
            "l2": "per-step working set (~30 arrays x 8N bytes) exceeds the 126 MB L2; no explicit flush" if nx * ny > 600000 else "fits L2"}


def workload_name(cfg):
    nx, ny, ra, dt, per = CONFIGS[cfg]
    return f"Navier2D {'periodic' if per else 'confined'} {nx}x{ny} {'Fourier' if per else 'Cheb'}xCheb Ra={ra:g} dt={dt:g}"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def cpu_restated(cfg, eig, threads=0):
    """The C++/OpenMP restatement of the reference's update() (oracle/cpu_restated.cpp: one pass per reference call,
    lane-parallel like rayon, OpenBLAS DGEMM) on the host cores, constructor defaults + init_random(0.1)."""
    from oracle import cpu_restated as cr

    nx, ny, ra, dt, per = CONFIGS[cfg]
    nav = cr.Navier2D(nx, ny, ra, 1.0, dt, 1.0, "rbc", periodic=per, pois_eig=eig, threads=threads)
    nav.init_random(0.1)
    return nav


def time_cpu(nav, steps, warmup):
    nav.update(max(1, warmup))
    t0 = time.perf_counter()
    nav.update(steps)
    return (time.perf_counter() - t0) / steps


def cpu_ops(nav, calls=3):
    """ms / transform and ms / solve of the CPU restatement (same operators, same spaces as the repo arm's `ops`)."""
    sec = nav.time_ops(calls)
    ms = {k: 1e3 * v for k, v in sec.items()}
    return {"ms_per_transform": {"forward": ms["forward"], "backward": ms["backward"]},
            "ms_per_solve": {"hholtz_adi": ms["hholtz_adi"], "poisson": ms["poisson"]},
            "ms_per_projection": {k: ms[k] for k in ("to_ortho", "from_ortho", "gradient_10", "gradient_02")},
            "calls": calls, "threads": nav.threads}


def cpu_best_threads(cfg, eig):
    """Thread count of the CPU arm: the reference runs its `*_par` passes on the rayon pool and OpenBLAS on its own threads -- more
    threads is not always faster (on the 128-thread GPU host the all-threads run of 1025^2 was 14x slower than one thread), so the
    baseline is timed at the best count of a short doubling sweep, one step each, and the sweep is reported."""
    cores = os.cpu_count() or 1
    cands, t = [], 4
    while t < cores:
        cands.append(t); t *= 2
    cands.append(cores)
    best, best_s, tried = 1, None, {}
    for t in [1] + cands:
        nav = cpu_restated(cfg, eig, threads=t)
        s = time_cpu(nav, 1, 1)
        del nav
        tried[t] = round(s, 4)
        if best_s is None or s < best_s:
            best, best_s = t, s
        elif t > 1 and s > 1.5 * best_s:
            break   # past the knee
    return best, tried


def host_eig(cfg):
    """Host LAPACK setup of the confined Poisson solver for the CPU arm (scipy, parity blocks; not timed)."""
    nx, ny, ra, dt, per = CONFIGS[cfg]
    if per:
        return None
    from oracle import rustpde_oracle as o

    f = o.Field2(o.Space2(o.cheb_neumann(nx), o.cheb_neumann(ny)))
    mass, lap, _, _ = f.ingredients_for_poisson(0)
    lam, fwd, bwd = o.parity_eig(lap, mass)
    if abs(lam[0]) < 1e-10:
        lam = lam - 1e-10
    return lam, fwd, bwd


def run_reference(args):
    """--impl reference: the reference's CPU algorithm on the box's host cores.  The Rust reference cannot be built in
    this image (no cargo/rustc), so the arm is the C++/OpenMP restatement that keeps the reference's pass structure
    (oracle/cpu_restated.cpp), all host threads, the driver's --steps / --warmup."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.config
    eig = host_eig(cfg)
    threads, tried = cpu_best_threads(cfg, eig)
    nav = cpu_restated(cfg, eig, threads=threads)
    sec = time_cpu(nav, args.steps, args.warmup)
    v = 1.0 / sec
    try:
        ops = cpu_ops(nav)
    except Exception as ex:  # noqa: BLE001 - the step line must still be printed
        ops = {"error": repr(ex)}
    line = {
        "impl": "reference", "metric": "Navier2D timesteps/sec", "value": v, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * sec, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(cfg),
        "cpu_baseline": {"value": v, "unit": "steps/s", "cores": nav.threads, "kind": "port", "flavour": "restated-c++",
                         "openblas_dgemm": nav.blas,
                         "sample": f"{args.steps} full update() steps of the C++/OpenMP restatement of the reference's pass structure "
                                   f"(reference Rust toolchain absent), {nav.threads} threads (best of the sweep)",
                         "threads_tried_s_per_step": tried, "host_cores": os.cpu_count()},
        "e2e": {"value": v, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "ops": ops,
    }
    print(json.dumps(line), flush=True)


def time_ops(b2, ctx, cfg, eig, peak_gbs, world=1, calls=10, dist=None):
    """ms / transform and ms / solve (BASELINE.json's metric names them next to timesteps/s; the reference's own harnesses are
    benches/benchmark_transform.rs and benchmark_solver.rs): the field operators and the two solvers of the step on standalone
    fields of the benchmarked size, each timed alone with CUDA events on the library's stream (`calls` back-to-back calls after
    2 warm-ups, results written into preallocated arrays).  `hbm_frac` = SURVEY 8(d)'s algorithmic bytes of the operator
    (2 sweeps x read + write = 32 N bytes; confined Poisson 48 N + 16 (nx-2)^2) / time / measured HBM peak; the confined Poisson
    solve is bound by its two FP64 GEMMs, not by HBM (see roofline.gemm)."""
    nx, ny, ra, dt, per = CONFIGS[cfg]
    N = nx * ny
    b0 = b2.fourier_r2c(nx) if per else b2.cheb_dirichlet(nx)
    p0 = b2.fourier_r2c(nx) if per else b2.cheb_neumann(nx)
    f = b2.Field2(b2.Space2(b0, b2.cheb_dirichlet(ny), ctx=ctx))       # the space of temp / velx / vely (navier.rs:232-244)
    fp = b2.Field2(b2.Space2(p0, b2.cheb_neumann(ny), ctx=ctx))        # the space of pres / pseu
    f.vhat = np_zeros_like_vhat(f)
    ortho = b2.DeviceArray(f.space, b2.ORTHO)
    ortho_p = b2.DeviceArray(fp.space, b2.ORTHO)
    out_p = b2.DeviceArray(fp.space, b2.SPECTRAL)
    out_h = b2.DeviceArray(f.space, b2.SPECTRAL)
    hh = b2.HholtzAdi(f, [dt * 1e-3, dt * 1e-3])
    po = b2.Poisson(fp, [1.0, 1.0], eig=eig) if not per else b2.Poisson(fp, [1.0, 1.0])

    def timed(fn):
        fn(); fn()
        ctx.sync()
        ctx.timer_start()
        for _ in range(calls):
            fn()
        return ctx.timer_stop() / calls

    ms = {
        "backward": timed(f.backward),
        "forward": timed(f.forward),
        "to_ortho": timed(lambda: f.to_ortho(out=ortho)),
        "from_ortho": timed(lambda: f.from_ortho(ortho)),
        "gradient_10": timed(lambda: f.gradient((1, 0), None, out=ortho)),
        "gradient_02": timed(lambda: f.gradient((0, 2), None, out=ortho)),
        "hholtz_adi": timed(lambda: hh.solve(ortho, out_h)),
        "poisson": timed(lambda: po.solve(ortho_p, out_p)),
    }
    if dist is not None:   # device time of the slowest rank, as for the step
        import torch

        t = torch.tensor([ms[k] for k in sorted(ms)], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = {k: float(v) for k, v in zip(sorted(ms), t)}
    alg = {k: 32.0 * N / world for k in ms}
    if not per:
        alg["poisson"] = (48.0 * N + 16.0 * (nx - 2) ** 2) / world
    frac = {k: (alg[k] / (ms[k] * 1e-3) / 1e9 / peak_gbs) if ms[k] > 0 else None for k in ms}
    for o_ in (hh, po, ortho, ortho_p, out_p, out_h, f, fp):
        o_.close()
    return {"ms_per_transform": {"forward": ms["forward"], "backward": ms["backward"]},
            "ms_per_solve": {"hholtz_adi": ms["hholtz_adi"], "poisson": ms["poisson"]},
            "ms_per_projection": {k: ms[k] for k in ("to_ortho", "from_ortho", "gradient_10", "gradient_02")},
            "hbm_frac": frac, "alg_bytes": alg, "calls": calls,
            "note": "standalone operator calls (2 lane passes each: along y, transposing store, along x, transposing store back); "
                    "forward / backward include the composite <-> orthonormal projection; inside update() they are fused into the "
                    "27 lane passes of the step, so these do not add up to ms_per_step"}


DUMP_BYTES = 64 * 10**6


def dump_outputs(arrays, out_dir, budget=DUMP_BYTES):
    """Write every array to out_dir/<name>.npy in float64 (complex arrays as [..., 2] = real, imaginary part), at most
    `budget` bytes in all.  An array larger than its even share of the budget is replaced by a fixed sample of its flattened
    entries, the same in every run: positions drawn without replacement by numpy default_rng(0), in ascending order."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    share = budget // len(arrays) - 4096   # room for the .npy header
    for name, a in arrays.items():
        a = np.asarray(a)
        cx = np.iscomplexobj(a)
        width = 16 if cx else 8   # bytes per entry in the file
        if a.size * width > share:
            flat = a.reshape(-1)
            a = flat[np.sort(np.random.default_rng(0).choice(flat.size, share // width, replace=False))]
        out = np.stack([a.real, a.imag], axis=-1) if cx else a
        np.save(os.path.join(out_dir, f"{name}.npy"), out.astype(np.float64, copy=False))


def np_zeros_like_vhat(f):
    """a smooth, non-trivial spectral state for the standalone operator timings (timing is data-independent)"""
    import numpy as np

    a = f.vhat
    i = np.arange(a.shape[0])[:, None]; j = np.arange(a.shape[1])[None, :]
    return (1.0 / (1.0 + i + j) ** 2).astype(a.dtype)


def parity_small(b2, ctx, dist):
    """2 steps of a 257 x 129 confined problem on the SAME ranks / context as the timed run, gathered and compared with
    the numpy oracle (navier.rs:438-466 / navier_stokes_mpi/navier.rs:497-522).  Cheap; runs before the timing.
    Two initial states: the reference example's smooth modes (strict: 1e-10) and the bench's white noise, whose step is
    conditioned well above rounding (the projection cancels a large divergent part): bounded by max(1e-10, 10 x yardstick),
    the yardstick being the oracle against itself when the same input is changed in the last bit (the rule of
    tests/gpu_checks.check_navier_white_noise)."""
    import numpy as np

    from oracle import rustpde_oracle as o

    nx, ny = 257, 129
    eig = b2.poisson_eig(b2.CHEB_NEUMANN, nx, 1.0)

    def rel(got, ref):
        return max(float(np.abs(got[k] - v).max() / np.abs(v).max()) for k, v in ref.items())

    def noise(perturb):
        out = {}
        for name, seed in (("temp", 1), ("velx", 2), ("vely", 3)):
            f = np.random.default_rng(seed).uniform(-0.1, 0.1, size=(nx, ny))
            out[name] = f * (1.0 + 4e-16 * np.random.default_rng(100 + seed).standard_normal((nx, ny))) if perturb else f
        return out

    def oracle_run(init, perturb=False):
        ref = o.Navier2D(nx, ny, 1e5, 1.0, 1e-2, 1.0, "rbc", pois_eig=eig)
        if init == "smooth":
            ref.set_velocity(0.2, 1.0, 1.0); ref.set_temperature(0.2, 1.0, 1.0)
        else:
            for name, f in noise(perturb).items():
                fld = getattr(ref, name)
                fld.v = f
                fld.forward()
        for _ in range(2):
            ref.update()
        return ref.state()

    out = {"world": ctx.nranks, "config": "confined 257x129, 2 steps, vs numpy oracle (same host eigendecomposition on both sides)", "tol": 1e-10}
    for init in ("smooth", "random"):
        nav = b2.Navier2D(nx, ny, 1e5, 1.0, 1e-2, 1.0, "rbc", ctx=ctx, pois_eig=eig, init_random=False)
        if init == "smooth":
            nav.set_velocity(0.2, 1.0, 1.0); nav.set_temperature(0.2, 1.0, 1.0)
        else:
            nav.init_random(0.1)   # U(-0.1, 0.1) from default_rng(1 / 2 / 3): the arrays of noise(False)
        nav.update(2)
        got = nav.gather_state()
        nav.close()
        ref = oracle_run(init)
        err = rel(got, ref)
        if init == "smooth":
            out["smooth_state_rel_err"] = err
            assert err < 1e-10, f"parity check failed (smooth state, {ctx.nranks} ranks): {err}"
        else:
            yard = rel(oracle_run(init, True), ref)
            out["worst_rel_err"] = err
            out["random_state"] = {"rel_err": err, "yardstick": yard, "bound": max(1e-10, 10.0 * yard),
                                   "note": "white noise: bounded by max(1e-10, 10 x the oracle's own response to a last-bit change of the input)"}
            assert err < max(1e-10, 10.0 * yard), f"parity check failed (white-noise state, {ctx.nranks} ranks): {err} (yardstick {yard})"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-ops", action="store_true", help="skip the standalone ms/transform, ms/solve timings")
    ap.add_argument("--ops-calls", type=int, default=10, help="timed calls per standalone operator")
    ap.add_argument("--ops-multi", action="store_true", help="also time the standalone operators on N > 1 ranks (slab fields)")
    ap.add_argument("--no-parity", action="store_true", help="skip the in-run parity checks (small multi-rank problem; workload vs CPU restatement)")
    ap.add_argument("--mode", type=int, default=1, help="1 fused+graph (default), 3 fused without graph, 0 one pass pair per reference call")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the state arrays of the last timed step to DIR/<name>.npy (float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.config is None:
        # BASELINE.json quotes its metric "at 1/2/4/8 B200" on configs[3] = confined 4097 x 4097 (C4), which fits one GPU
        # and is the size the north-star roofline target is stated on: the same workload at every N, so that the
        # driver's 1 -> 8 series is a strong-scaling series of one problem.  --config C2 / C3 / C1 run the others.
        args.config = "C4"
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    import numpy as np
    import torch

    import rustpde_mpi_b200 as b2

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world == 1 and args.gpus > 1:
        raise SystemExit("launch with torch.distributed.run for --gpus > 1")
    cfg = args.config
    nx, ny, ra, dt, per = CONFIGS[cfg]
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group(backend="cpu:gloo,cuda:nccl")
        heap = ((160 if args.ops_multi else 110) * (nx + 64) * (ny + 64) * 8) // world + (64 << 20)
        ctx = b2.Context.distributed(local, heap)
    else:
        ctx = b2.Context(local)

    def fence():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    parity = None if args.no_parity else parity_small(b2, ctx, dist)   # same ranks, same context, before the timing
    t_setup = time.perf_counter()
    eig = None if per else b2.poisson_eig(b2.CHEB_NEUMANN, nx, 1.0)   # host LAPACK setup (not timed)
    nav = b2.Navier2D(nx, ny, ra, 1.0, dt, 1.0, "rbc", periodic=per, ctx=ctx, pois_eig=eig)
    nav.init_random(0.1)
    nav.set_mode(args.mode)
    setup_s = time.perf_counter() - t_setup
    N = nx * ny

    # ---- device-resident timing ----
    sampler = ClockSampler(local)
    sampler.start()
    nav.update(args.warmup)
    ctx.sync()
    fence()
    l0 = ctx.launch_count()
    t_a = time.time()
    ctx.timer_start()
    nav.update(args.steps)
    ms = ctx.timer_stop()
    fence()
    t_b = time.time()
    # copied here: the clock, GEMM and e2e passes below step the same solver further
    outputs = (nav.gather_state() if dist is not None else nav.state()) if args.dump_outputs else None
    if dist is not None:  # device time of the slowest rank
        t = torch.tensor([ms], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    launches = ctx.launch_count() - l0
    ms_per_step = ms / args.steps
    value = 1e3 / ms_per_step
    # keep the same loop running until nvidia-smi (100 ms period) has seen >= 1.5 s of it
    n_more = 0
    burst = max(1, args.steps // 4)
    if dist is None:
        while time.time() - t_a < 1.5:
            nav.update(burst); ctx.sync(); n_more += 1
    else:
        # multi-rank: every rank must issue the same number of steps, so the count comes from the all-reduced step time
        # (identical on every rank), not from the local wall clock: ~2 s of the loop, nvidia-smi needs a few 100 ms to start
        for _ in range(min(2000, max(4, int(math.ceil(2000.0 / (burst * ms_per_step)))))):
            nav.update(burst); ctx.sync(); n_more += 1
    clocks = sampler.stop()
    clocks["note"] = f"sampled every 100 ms from warm-up through the timed region ({(t_b - t_a) * 1e3:.0f} ms) and {n_more} continuation bursts of the same loop"
    # GEMM share of the step (separate short pass: event pairs around the two gemm_pb_kernel launches, no graph replay)
    n_prof = max(2, min(args.steps, 10))
    ctx.profile(True)
    nav.update(n_prof)
    gemm_ms = ctx.profile(False) / n_prof * args.steps
    div = nav.div_norm()
    assert np.isfinite(div), "NaN divergence"

    # ---- roofline of the HBM-bound lane kernels (SURVEY 8d work model) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    lane_ms = (ms - gemm_ms) / args.steps
    alg_bytes = 728.0 * N / world   # per GPU
    achieved = alg_bytes / (lane_ms * 1e-3) / 1e9
    traffic = None   # only a capture of THIS config on ONE GPU counts (profiles/traffic.json is written by tools/gpu_profile.sh)
    if world == 1:
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(cfg, {}).get("dram_bytes_per_step")
        except Exception:  # noqa: BLE001
            pass
    info = nav.info()
    if per:
        gemm_flop = 0.0
    elif info["parity_blocks"]:   # two GEMM pairs on the parity blocks (half the flops of the dense products)
        gemm_flop = 2.0 * 2.0 * info["P1"] * (info["ce"] ** 2 + info["co"] ** 2) / world
    else:
        gemm_flop = 4.0 * info["m0"] ** 2 * info["P1"] / world
    # FP64 GEMM denominator: a plain library DGEMM of the Poisson products' shape, measured here (MEASURED_PEAKS.json has none)
    fp64_peak = None
    if gemm_flop > 0:
        try:
            m = 2048
            a = torch.randn(m, m, dtype=torch.float64, device="cuda"); bm = torch.randn(m, 4096, dtype=torch.float64, device="cuda")
            torch.matmul(a, bm); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                torch.matmul(a, bm)
            e1.record(); torch.cuda.synchronize()
            fp64_peak = 5 * 2.0 * m * m * 4096 / (e0.elapsed_time(e1) * 1e-3) / 1e12
            del a, bm
        except Exception:  # noqa: BLE001
            fp64_peak = None
    gemm_tf = (gemm_flop / (gemm_ms / args.steps * 1e-3) / 1e12) if gemm_ms > 0 else None
    t_hbm = alg_bytes / (peak * 1e9) * 1e3
    t_gemm = (gemm_flop / (fp64_peak * 1e12) * 1e3) if (fp64_peak and gemm_flop) else 0.0
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": "MEASURED_PEAKS.json (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                "kernel": "lane_kernel (all per-axis passes of one step)", "alg_bytes_per_step": alg_bytes,
                "lane_ms_per_step": lane_ms, "gemm_ms_per_step": gemm_ms / args.steps,
                "lane_ms_note": "step time minus the time inside the Poisson GEMMs (FP64-peak-bound, measured with events in a separate un-captured pass)",
                "gemm": {"achieved": gemm_tf, "peak": fp64_peak, "unit": "TFLOP/s", "frac": (gemm_tf / fp64_peak) if (gemm_tf and fp64_peak) else None,
                         "peak_source": "library DGEMM 2048x2048x4096 (torch.matmul f64) timed in this run", "flop_per_step": gemm_flop,
                         "parity_block_gemms": bool(info["parity_blocks"])},
                "whole_step": {"bound_ms": t_hbm + t_gemm, "measured_ms": ms_per_step, "frac": (t_hbm + t_gemm) / ms_per_step,
                               "note": "algorithmic bytes / measured HBM peak + GEMM flops / measured DGEMM rate, over the measured step"},
                "traffic_note": "dram__bytes_read+write summed over the lane-kernel launches of one step (ncu --set full, this config, 1 GPU)" if traffic else None}

    # ---- end to end with host-resident state (pinned), copies inside the timed region ----
    e2e, e2e_error = None, None
    if not args.no_e2e:
        try:
            names = ("temp", "velx", "vely", "pres")
            host = {}
            for k in names:
                a = getattr(nav, k).vhat
                t = torch.from_numpy(a.view(np.float64) if a.dtype == np.complex128 else a).clone().pin_memory()
                host[k] = (t, a.dtype, a.shape)
            nbytes = sum(t.numel() * 8 for t, _, _ in host.values())
            k_e2e = max(3, min(args.steps, 10))

            def e2e_step():
                for k in names:
                    t, dt_, sh = host[k]
                    arr = t.numpy().view(dt_).reshape(sh)
                    getattr(nav, k).vhat = arr
                nav.update(1)
                for k in names:
                    t, dt_, sh = host[k]
                    getattr(nav, k).vhat_into(t.numpy().view(dt_).reshape(sh))   # straight into the pinned buffer

            e2e_step()
            fence()
            ctx.timer_start()
            for _ in range(k_e2e):
                e2e_step()
            ms2 = ctx.timer_stop()   # CUDA events on the library's stream around the whole loop (copies included)
            fence()
            if dist is not None:
                t = torch.tensor([ms2, float(nbytes)], dtype=torch.float64)
                tm = t.clone()
                dist.all_reduce(tm, op=dist.ReduceOp.MAX)
                dist.all_reduce(t, op=dist.ReduceOp.SUM)
                ms2, nbytes = float(tm[0]), int(t[1])
            e2e = {"value": 1e3 / (ms2 / k_e2e), "unit": "steps/s", "h2d_bytes_per_step": nbytes, "d2h_bytes_per_step": nbytes,
                   "steps": k_e2e}
        except Exception as ex:  # noqa: BLE001 - the device-resident line must still be printed
            e2e, e2e_error = None, repr(ex)

    # ---- CPU baseline: the C++/OpenMP restatement of the reference's pass structure, bounded sample; the same run is the
    # parity check of the BENCHMARKED configuration (k steps from the same synthetic initial state on both sides) ----
    cpu, parity_workload = None, None
    if not args.no_cpu_baseline and world == 1:
        n_cpu = {"C1": 20, "C2": 5, "C3": 5}.get(cfg, 3)
        cpu_threads, cpu_tried = cpu_best_threads(cfg, eig)
        cnav = cpu_restated(cfg, eig, threads=cpu_threads)
        sec = time_cpu(cnav, n_cpu, 1)
        cpu = {"value": 1.0 / sec, "unit": "steps/s", "cores": cnav.threads, "kind": "port", "flavour": "restated-c++",
               "openblas_dgemm": cnav.blas,
               "sample": f"{n_cpu} full update() steps (after 1 warm-up) of the C++/OpenMP restatement of the reference's pass structure at the same config, {cnav.threads} threads ({sec * n_cpu:.1f} s)",
               "threads_tried_s_per_step": cpu_tried, "host_cores": os.cpu_count()}
        try:
            cpu["ops"] = cpu_ops(cnav)
        except Exception as ex:  # noqa: BLE001
            cpu["ops"] = {"error": repr(ex)}
        if nx * ny <= 1100 * 1100:   # the 1-thread figure (README's OPENBLAS_NUM_THREADS=1 mode) where it costs seconds
            cpu["value_1thread"] = 1.0 / cpu_tried[1]
            del cnav
            cnav = cpu_restated(cfg, eig, threads=cpu_threads)
            cnav.update(1 + n_cpu)
        if not args.no_parity:
            def rel(gs, cs):
                return {k: float(np.abs(gs[k] - v).max() / np.abs(v).max()) for k, v in cs.items()}

            nav.init_random(0.1)
            nav.pres.vhat = np.zeros_like(nav.pres.vhat)
            nav.update(1 + n_cpu)
            e_rand = rel(nav.state(), cnav.state())
            del cnav
            # the same configuration from the reference example's smooth state (examples/navier_rbc.rs:18-22): the strict bound
            cnav = cpu_restated(cfg, eig, threads=cpu_threads)
            cnav.set_velocity(0.2, 1.0, 1.0); cnav.set_temperature(0.2, 1.0, 1.0)
            cnav.update(2)
            nav.set_velocity(0.2, 1.0, 1.0); nav.set_temperature(0.2, 1.0, 1.0)
            nav.pres.vhat = np.zeros_like(nav.pres.vhat)
            nav.update(2)
            e_smooth = rel(nav.state(), cnav.state())
            parity_workload = {"config": cfg, "against": "oracle/cpu_restated.cpp (checked against the numpy oracle in tests/)",
                               "smooth_state": {"steps": 2, "worst_rel_err": max(e_smooth.values()), "per_field": e_smooth, "tol": 1e-10},
                               "random_state": {"steps": 1 + n_cpu, "worst_rel_err": max(e_rand.values()), "per_field": e_rand, "tol": 1e-6,
                                                "note": "white-noise fields: the projection step cancels a large divergent part, two CPU restatements "
                                                        "already differ by ~1e-8 on 1025^2 (tests/test_gpu_parity_large.py)"},
                               "note": "both sides get the same host eigendecomposition of the Poisson operator (DESIGN.md, Poisson parity)"}
            assert max(e_smooth.values()) < 1e-10 and max(e_rand.values()) < 1e-6, parity_workload
        del cnav

    # ---- ms / transform, ms / solve (the metric's second half): standalone operators on the benchmarked size ----
    ops, ops_error = None, None
    if not args.no_ops and (world == 1 or args.ops_multi):   # N > 1: opt-in (--ops-multi); the slab operators are covered by tests/test_gpu_multi.py
        try:
            ops = time_ops(b2, ctx, cfg, eig, peak, world, calls=max(1, args.ops_calls), dist=dist)
        except Exception as ex:  # noqa: BLE001 - the step line must still be printed
            ops, ops_error = None, repr(ex)

    line = {
        "metric": "Navier2D timesteps/sec", "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_dict(cfg),
        "run": {"parallelism": "1 GPU" if world == 1 else f"{world} GPUs, slab decomposition, peer-store transposes over NVLink",
                "schedule": {1: "fused, CUDA-graph replay", 3: "fused, no graph", 0: "one pass pair per reference call"}.get(args.mode, str(args.mode)),
                "launches_per_step": nav.launches_per_step(), "parallel_branches": bool(info["branches"])},
        "clocks": clocks, "e2e": e2e, "e2e_error": e2e_error, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu,
        "parity_check": parity, "parity_check_workload": parity_workload, "ops": ops, "ops_error": ops_error,
        "setup_s": setup_s, "div_norm": div,
    }
    if rank == 0:
        if outputs is not None:
            dump_outputs(outputs, args.dump_outputs)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
