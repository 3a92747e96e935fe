#!/usr/bin/env python
"""Benchmark of the reduced-order frequency-sweep hot path (BASELINE.json metric: reduced-sweep freq points/sec).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload cfg3|cfg2|cfg5|mid|small] [--dump-outputs DIR]

One "step" = one pass of the four hot stages over one synthetic batch: orthonormalise the snapshot block
(CholeskyQR2 + SVD of R), Galerkin-project Ct/Tt/WP, solve every reduced system, evaluate the S-parameters.
The default workload is the configuration the metric and the north-star target are quoted on (BASELINE configs[2]:
N = 1M DOF, r = 256, 4 ports, 100k sweep points); it fits one B200.  ``--gpus N`` STRONG-scales it: the same global
problem at every N, rows of the snapshot block / operators and the sweep points block-sharded over the ranks, r x r
partials all-reduced, Q halo rows exchanged, S-parameters all-gathered.

``value`` = sweep points of the whole job / device time of K steps (inputs resident in HBM, max over ranks);
``e2e``   = the same through the reference-facing Python call with HOST (pinned) inputs, H2D/D2H inside the timing;
``parity``= the S-parameters of the timed configuration against the CPU restatement of the reference (oracle/);
``--impl reference`` times that CPU restatement (numpy/scipy = the library calls the pure-Python reference makes)
on all host cores of rank 0, each step a bounded sample of the same global workload.
``--dump-outputs DIR`` writes what the last timed step returned as .npy files: the inputs are seeded, so two builds run with the
same arguments can be compared output for output.
"""
from __future__ import annotations

import os
import sys


def _host_cores() -> int:
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


# torchrun exports OMP_NUM_THREADS=1 to every rank.  The CPU legs (reference arm, cpu_baseline, parity) run on rank 0 only
# and use all the host cores the process may run on -- set before numpy / OpenBLAS are loaded, and recorded in the line.
if int(os.environ.get("RANK", "0")) == 0:
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(_host_cores())

import argparse
import json
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: GLOBAL grid (nx, ny, nz), r, ports, GLOBAL sweep points; cpu_points = points the CPU legs solve (scaled linearly)
    "cfg3": dict(grid=(25, 20, 2000), r=256, m=4, f=100000, cpu_points=200,
                 desc="BASELINE configs[2]: synthetic N=1M DOF, r=256, 4 ports, 100k freq points (the configuration the metric "
                      "and the north-star target are quoted on); strong scaling over the GPUs"),
    "cfg2": dict(grid=(20, 10, 1000), r=64, m=2, f=10000, cpu_points=2000,
                 desc="BASELINE configs[1]: synthetic curl-curl FEM N=200k DOF, r=64 basis, 2 ports, 10k freq points"),
    "cfg5": dict(grid=(25, 20, 8000), r=512, m=8, f=1000000, cpu_points=40,
                 desc="BASELINE configs[4]: dense wideband sweep N=4M DOF, r=512, 8 ports, 1M freq points, row-sharded projection"),
    "mid": dict(grid=(10, 8, 250), r=64, m=2, f=1024, cpu_points=1024, desc="parity-sized workload (N=20k, r=64, 2 ports, 1024 points)"),
    "small": dict(grid=(5, 4, 100), r=16, m=2, f=512, cpu_points=512, desc="smoke-sized workload"),
}
METRIC = "reduced-sweep freq points/sec"
UNIT = "points/s"
FP64_PEAK_FALLBACK = 37.05   # TFLOP/s, DMMA m8n8k4 issue loop measured on this pool's B200 in round 1 (profiles/r01_fp64_peaks.jsonl)
SNAP_BLOCKS = 8              # the global snapshot block is 8 seeded row blocks, whatever the number of ranks
EPS = float(np.finfo(np.float64).eps)
# --dump-outputs: bytes per written array and its row list (60 MiB in all with the four reduced operators at r <= 512: under 64 MB)
DUMP_CAP = {"gsm": 28 << 20, "q": 12 << 20, "info": 4 << 20}
DUMP_CAP_OTHER = 4 << 20


def workload_config(name, wl, n):
    """The ``config`` object of the JSON line -- identical for the b200 and the reference arm."""
    return {"workload": name + ": " + wl["desc"], "N_dof_total": int(n), "r": wl["r"], "ports": wl["m"], "freq_points_total": wl["f"],
            "scaling": "strong: one global problem, rows and sweep points block-sharded over the GPUs",
            "l2": "inputs larger than L2 (snapshot block %.0f MB complex128 + operators); no flush" % (n * wl["r"] * 16 / 1e6)}


def snapshot_rows(n, r, lo, hi):
    """Rows [lo, hi) of the global synthetic snapshot block: SNAP_BLOCKS independently seeded row blocks (SURVEY 8d)."""
    from morfem_b200 import synthetic, dist as mfd
    parts = []
    for b in range(SNAP_BLOCKS):
        b0, b1 = mfd.even_split(n, SNAP_BLOCKS, b)
        s0, s1 = max(lo, b0), min(hi, b1)
        if s1 > s0:
            blk = synthetic.snapshot_matrix(b1 - b0, r, seed=1000 + b, decay_decades=6.0)
            parts.append(blk[s0 - b0:s1 - b0])
    return np.ascontiguousarray(np.concatenate(parts, axis=0)) if len(parts) != 1 else np.ascontiguousarray(parts[0])


def build_operators(wl):
    from morfem_b200 import synthetic
    nx, ny, nz = wl["grid"]
    ct, tt = synthetic.waveguide_operators(nx, ny, nz)
    n = ct.shape[0]
    wp = synthetic.port_matrix(n, wl["m"], 19)
    in_c, in_gamma, in_b = synthetic.driver_scaled(ct, tt, wp)
    f = synthetic.frequency_points(wl["f"])
    return in_c, in_gamma, in_b, f, n


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""
    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTE = {"sw_power_cap": 0x4, "hw_power_brake": 0x80, "sync_boost": 0x10, "applications_clocks": 0x2}

    def __init__(self, device_index, period=0.02):
        super().__init__(daemon=True)
        self.period = period
        self.samples, self.reasons = [], set()
        self.max_mhz = None
        self.ok = False
        self._stop_evt = threading.Event()
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(device_index).uuid)
            try:
                self.h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception as exc:  # pragma: no cover - no GPU
            self.err = repr(exc)

    def sample(self):
        nv = self.nv
        self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
        except Exception:
            mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
        for name, bit in {**self.BAD, **self.NOTE}.items():
            if mask & bit:
                self.reasons.add(name)

    def run(self):
        while self.ok and not self._stop_evt.is_set():
            try:
                self.sample()
            except Exception:
                break
            self._stop_evt.wait(self.period)

    def stop(self):
        self._stop_evt.set()
        if self.is_alive():
            self.join(timeout=2)
        if self.ok and not self.samples:
            try:
                self.sample()
            except Exception:
                pass
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------ CPU legs (oracle)
def sample_indices(f_total, count):
    return np.unique(np.linspace(0, f_total - 1, min(int(count), int(f_total))).astype(np.int64))


def cpu_stage12(in_c, in_gamma, in_b, s):
    """Stages 1 + 2 of the CPU restatement of the reference on the given rows (implementation.py:226, :181-184)."""
    from scipy.sparse import csc_array
    from oracle import reference_path as orc
    t0 = time.perf_counter()
    q = orc.orthonormal_basis(s)
    t1 = time.perf_counter()
    red = orc.galerkin_projection(q, in_c, csc_array(in_c.shape), in_gamma, in_b)
    t2 = time.perf_counter()
    return red, {"basis_s": t1 - t0, "projection_s": t2 - t1}


def cpu_sweep(fs, red):
    """Stages 3 + 4 of the CPU restatement on the points ``fs`` (implementation.py:189-194, test_helpers.py:60-65)."""
    from oracle import reference_path as orc
    a0_r, a1_r, a2_r, b_r = red
    t0 = time.perf_counter()
    x = orc.reduced_sweep(fs, a0_r, a1_r, a2_r, b_r, lambda t: 1.0, lambda t: t, lambda t: t ** 2, orc.b_coefficient)
    t1 = time.perf_counter()
    gsm = orc.scattering_sweep(fs, x, b_r)
    t2 = time.perf_counter()
    return gsm, {"sweep_s_per_point": (t1 - t0) / fs.size, "gsm_s_per_point": (t2 - t1) / fs.size, "points_sampled": int(fs.size)}


def system_conds(fs, red):
    from oracle import reference_path as orc
    a0_r, a1_r, a2_r, _ = red
    return np.array([np.linalg.cond(orc.system_matrix(1.0, t, t ** 2, a0_r, a1_r, a2_r)) for t in fs])


def snapshot_cond(s):
    """cond(S) from the eigenvalues of the Gram matrix (an estimate good to a few digits for cond up to ~1e7)."""
    w = np.linalg.eigvalsh(s.T @ s)
    return float(np.sqrt(w[-1] / max(w[0], w[-1] * 1e-15)))


def per_point_rel(new, ref):
    new = np.asarray(new).reshape(new.shape[0], -1)
    ref = np.asarray(ref).reshape(ref.shape[0], -1)
    return np.linalg.norm(new - ref, axis=1) / np.linalg.norm(ref, axis=1)


def blas_threads():
    try:
        import threadpoolctl
        return max([p.get("num_threads", 1) for p in threadpoolctl.threadpool_info()] + [1])
    except Exception:
        return _host_cores()


def run_reference(args, name, wl, rank, world):
    """The reference's CPU implementation of the path (oracle port: the reference is pure Python, its arithmetic is the very
    numpy/scipy calls made here), all host cores, the same GLOBAL workload at every N.  One step = a bounded sample:
    stages 1+2 on the leading ``cpu_rows`` rows (cost linear in N, scaled), stages 3+4 on ``cpu_points`` points (scaled)."""
    if rank != 0:
        return
    nx, ny, nz = wl["grid"]
    n = nx * ny * nz
    r = wl["r"]
    # the row sample is a shorter waveguide of the same cross-section (same band structure and non-zeros per row, so the same
    # cost per row), with its own port matrix so that the sampled reduced model is a regular one
    nz_s = min(nz, max(2 * 19 // (nx * ny) + 2, args.cpu_rows // (nx * ny)))
    sub_c, sub_g, sub_b, f, rows = build_operators(dict(wl, grid=(nx, ny, nz_s)))
    s = snapshot_rows(n, r, 0, rows)
    idx = sample_indices(f.size, args.cpu_points or wl["cpu_points"])
    fs = f[idx]

    def one_step():
        red, t12 = cpu_stage12(sub_c, sub_g, sub_b, s)
        _, t34 = cpu_sweep(fs, red)
        t12["step_s_full"] = (t12["basis_s"] + t12["projection_s"]) * (n / rows) + (t34["sweep_s_per_point"] + t34["gsm_s_per_point"]) * f.size
        t12.update(t34)
        return t12

    for _ in range(args.warmup):
        one_step()
    times = []
    t_start = time.perf_counter()
    for _ in range(args.steps):
        times.append(one_step())
    wall = time.perf_counter() - t_start
    step_s = float(np.mean([t["step_s_full"] for t in times]))
    value = f.size / step_s
    cores = blas_threads()
    sample = (f"per step: stages 1+2 on the leading {rows} of {n} rows (r={r}; cost linear in N, scaled by {n / rows:.1f}), stages 3+4 on "
              f"{fs.size} of {f.size} points scaled linearly; numpy/scipy = the reference's own library calls (oracle port), real float64 "
              f"(the reference's dtype), {cores} BLAS threads on {_host_cores()} host cores")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": step_s * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(name, wl, n),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "stages": {"basis_ms_full": float(np.mean([t["basis_s"] for t in times])) * 1e3 * n / rows,
                       "projection_ms_full": float(np.mean([t["projection_s"] for t in times])) * 1e3 * n / rows,
                       "sweep_us_per_point": float(np.mean([t["sweep_s_per_point"] for t in times])) * 1e6,
                       "gsm_us_per_point": float(np.mean([t["gsm_s_per_point"] for t in times])) * 1e6},
            "wall_s": wall}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------- B200 arm
def measure_fp64_peak():
    """FP64 tensor-pipe (DMMA) peak measured live by the library's issue-loop kernel (mf_peak_dmma_tflops)."""
    import ctypes
    import torch
    from morfem_b200 import _ffi
    lib = _ffi.load()
    out = ctypes.c_double(0.0)
    try:
        st = lib.mf_peak_dmma_tflops(4096, ctypes.byref(out), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    except AttributeError:
        return FP64_PEAK_FALLBACK, "fallback: 37.05 TFLOP/s measured in round 1 (profiles/r01_fp64_peaks.jsonl)"
    if st != 0 or not (out.value > 1.0):
        return FP64_PEAK_FALLBACK, "fallback: 37.05 TFLOP/s measured in round 1 (profiles/r01_fp64_peaks.jsonl)"
    return float(out.value), ("FP64 tensor-pipe (DMMA m8n8k4) issue-loop peak measured in this run by mf_peak_dmma_tflops; "
                             "MEASURED_PEAKS.json holds no FP64 figure and its bf16 figure does not bound an FP64 kernel")


def dump_outputs(out_dir, arrays):
    """Write every tensor of ``arrays`` as ``out_dir/<name>.npy`` in float64, complex ones with a trailing (real, imag) axis.  An
    array above its byte cap keeps a sample of its leading-axis rows drawn with a fixed seed (the same rows on every run with the
    same arguments), listed in ``<name>_rows.npy``."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if t is None:                                         # an all-zero operator is returned as None
            continue
        cap = DUMP_CAP.get(name, DUMP_CAP_OTHER)
        row_bytes = max(1, t[0].numel()) * (16 if t.is_complex() else 8)
        if t.shape[0] * row_bytes > cap:
            keep = cap // (row_bytes + 8)                     # the row list counts against the cap too
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
            np.save(os.path.join(out_dir, name + "_rows.npy"), rows.astype(np.float64))
        a = t.cpu().numpy()
        if np.iscomplexobj(a):
            a = np.stack((a.real, a.imag), axis=-1)
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


def make_path(wl_ops, rank, world):
    from scipy.constants import pi, epsilon_0
    from scipy.sparse import csc_array
    from morfem_b200 import dist as mfd, implementation as impl, test_helpers as th
    in_c, in_gamma, in_b, f, n = wl_ops
    cb = impl.coefficient_array(th.b_coefficient, f)
    coeffs = [np.ones_like(f), f, f ** 2, cb, 2 * pi * f * epsilon_0]
    return mfd.ShardedHotPath([in_c, csc_array(in_c.shape), in_gamma], in_b, n, f.size, coeffs)


def parity_small(world, rank, dev, real):
    """N > 1: before timing, the sharded path on a reduced-size GLOBAL problem against the CPU oracle on rank 0 -- halo-window
    SpMM, all-reduced Gram / projection partials and the gathered S-parameters, on the hardware the timing runs on."""
    import torch
    import torch.distributed as dist
    from morfem_b200 import device as dv, dist as mfd
    wl = WORKLOADS["mid"]
    ops = build_operators(wl)
    in_c, in_gamma, in_b, f, n = ops
    path = make_path(ops, rank, world)
    lo, hi = mfd.even_split(n, world, rank)
    s_dev = dv.real_or_complex_to_device(snapshot_rows(n, wl["r"], lo, hi), dev, widen=not real)
    gsm, q, red, res = path.step(s_dev, want_x=False, gather=True)
    torch.cuda.synchronize()
    out = None
    if rank == 0:
        s_glob = snapshot_rows(n, wl["r"], 0, n)
        ref_red, _ = cpu_stage12(in_c, in_gamma, in_b, s_glob)
        ref_gsm, _ = cpu_sweep(f, ref_red)
        cond = system_conds(f, ref_red)
        tol = np.maximum(1e-10, 50 * EPS * np.maximum(cond, snapshot_cond(s_glob)))
        err = per_point_rel(gsm.cpu().numpy(), ref_gsm)
        out = {"workload": "mid: " + wl["desc"] + f", sharded over {world} ranks", "max_rel_err": float(err.max()), "points": int(f.size),
               "tol_max": float(tol.max()), "worst_err_over_tol": float((err / tol).max()), "ok": bool(np.all(err < tol))}
    ok = torch.tensor([1 if (out is None or out["ok"]) else 0], device=dev)
    dist.broadcast(ok, 0)
    if int(ok.item()) != 1:
        raise SystemExit(f"bench: multi-rank parity against the CPU oracle FAILED: {out}")
    del path
    return out


def run_b200(args, name, wl, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from scipy.sparse import csc_array
    from morfem_b200 import device as dv, dist as mfd, _ffi, test_helpers as th

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    _ffi.load()
    fp64_peak, fp64_src = measure_fp64_peak()

    # "c128" (default, the north star's arithmetic): the real synthetic data embedded in complex128, complex128 kernels
    # throughout.  The synthetic operators and snapshots are real, like the reference's data (main.py:21-23), so "auto" /
    # "f64" run the real float64 twins -- what the public API selects by itself for such inputs; the default run times
    # that path too and reports it under "other_dtype".
    real = args.dtype in ("auto", "f64")

    parity_pre = parity_small(world, rank, dev, real) if (world > 1 and not args.no_parity) else None

    ops = build_operators(wl)
    in_c, in_gamma, in_b, f, n = ops
    r, m = wl["r"], wl["m"]
    path = make_path(ops, rank, world)
    row0, row1 = mfd.even_split(n, world, rank)
    s_loc = snapshot_rows(n, r, row0, row1)
    s_dev = dv.real_or_complex_to_device(s_loc, dev, widen=not real)
    f_total = f.size

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    use_graph = not args.no_graph and (world == 1 or path.graph_capable)

    def make_step(s_in):
        def step():
            if use_graph:
                return path.step_graph(s_in, want_x=False)        # whole step replayed from one CUDA graph
            return path.step_deferred(s_in, want_x=False, gather=True)   # eager launches, CholeskyQR2 flags verified after the loop
        return step

    def check_flags(what):
        ok = (path.verify() is None) if use_graph else path.verify_deferred()
        if not ok:
            raise SystemExit(f"bench: optimistic CholeskyQR2 failed verification on the synthetic snapshot block ({what})")

    def timed(step, k, w):
        for _ in range(w):
            out_ = step()
        barrier()
        l0 = _ffi.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            out_ = step()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / k, out_, _ffi.launch_count() - l0

    step = make_step(s_dev)
    warm = max(args.warmup, 3)
    for _ in range(warm):
        out = step()
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_step, out, launches = timed(step, args.steps, 0)
    clocks = sampler.stop()
    check_flags("timed loop")
    if args.dump_outputs and rank == 0:
        gsm_o, q_o, red_o, res_o = out
        dump_outputs(args.dump_outputs, {"gsm": gsm_o, "q": q_o, "a0_r": red_o[0], "a1_r": red_o[1], "a2_r": red_o[2], "b_r": red_o[3],
                                         "info": res_o.info})
    if use_graph:
        launches = args.steps * path.launches_per_graph          # a replay launches the captured kernels without passing the ABI counter
    value = f_total / (ms_step * 1e-3)
    gsm_dev = out[0].clone()                                   # small copies: `out` pins the static outputs of the captured step
    reduced_dev = [None if o is None else o.clone() for o in out[2]]
    del out

    # ---- parity of the timed configuration against the CPU restatement of the reference (rank 0, sampled points)
    parity, cpu_baseline = None, None
    if rank == 0 and not args.no_parity:
        idx = sample_indices(f_total, args.cpu_points or wl["cpu_points"])
        fs = f[idx]
        g_gpu = gsm_dev[torch.from_numpy(idx).to(dev)].cpu().numpy()
        red_gpu = [np.zeros((r, r)) if o is None else o.cpu().numpy() for o in reduced_dev[:3]] + [reduced_dev[3].cpu().numpy()]
        red_gpu = [np.ascontiguousarray(a.real) for a in red_gpu]          # real data stays exactly real on the complex128 path
        # (a) stage isolated: the CPU sweep (lu_factor/lu_solve + the S-parameter algebra) on the reduced model the GPU produced
        g_iso, t34 = cpu_sweep(fs, red_gpu)
        cond = system_conds(fs, red_gpu)
        tol_iso = np.maximum(1e-10, 20 * EPS * cond)
        e_iso = per_point_rel(g_gpu, g_iso)
        parity = {"points": int(fs.size), "tol": "max(1e-10, 20 eps cond(A(t))) per point (stage isolated); chained: eps-level "
                  "changes of S move span(S) by eps cond(S), so max(1e-10, 50 eps max(cond(A(t)), cond(S)))",
                  "stage_isolated": {"max_rel_err": float(e_iso.max()), "median_rel_err": float(np.median(e_iso)), "tol_max": float(tol_iso.max()),
                                     "worst_err_over_tol": float((e_iso / tol_iso).max()), "cond_max": float(cond.max())}}
        ok = bool(np.all(e_iso < tol_iso))
        full = args.parity == "full" or (args.parity == "auto" and world == 1 and n * r * r <= 1.1e6 * 256 * 256)
        if full:
            # (b) chained: the whole path on the CPU (svd, projection, LU sweep, S-parameters) -- also the cpu_baseline figure
            s_glob = s_loc if world == 1 else snapshot_rows(n, r, 0, n)
            ref_red, t12 = cpu_stage12(in_c, in_gamma, in_b, s_glob)
            g_ref, t34 = cpu_sweep(fs, ref_red)
            cond_ref = system_conds(fs, ref_red)
            cond_s = snapshot_cond(s_glob)
            tol_ch = np.maximum(1e-10, 50 * EPS * np.maximum(cond_ref, cond_s))
            e_ch = per_point_rel(g_gpu, g_ref)
            parity["chained"] = {"max_rel_err": float(e_ch.max()), "median_rel_err": float(np.median(e_ch)), "tol_max": float(tol_ch.max()),
                                 "worst_err_over_tol": float((e_ch / tol_ch).max()), "cond_S": cond_s}
            parity["max_rel_err"] = float(e_ch.max())
            ok = ok and bool(np.all(e_ch < tol_ch))
            step_s = t12["basis_s"] + t12["projection_s"] + (t34["sweep_s_per_point"] + t34["gsm_s_per_point"]) * f_total
            cpu_baseline = {"value": f_total / step_s, "unit": UNIT, "cores": blas_threads(), "kind": "port",
                            "sample": f"one pass: stages 1+2 in full (N={n}, r={r}: svd {t12['basis_s']:.2f} s, projection {t12['projection_s']:.2f} s), "
                                      f"stages 3+4 on {t34['points_sampled']} of {f_total} points ({t34['sweep_s_per_point'] * 1e6:.0f} + "
                                      f"{t34['gsm_s_per_point'] * 1e6:.0f} us/point) scaled linearly; real float64 like the reference"}
            del s_glob
        else:
            parity["max_rel_err"] = float(e_iso.max())
        parity["ok"] = ok
        if parity_pre is not None:
            parity["multi_rank_small_problem"] = parity_pre
    if not args.no_parity:
        flag = torch.tensor([1 if (parity is None or parity["ok"]) else 0], device=dev)
        if world > 1:
            dist.broadcast(flag, 0)
        if int(flag.item()) != 1:
            raise SystemExit(f"bench: parity against the CPU oracle FAILED: {json.dumps(parity)}")

    # ---- the same timed loop on the other arithmetic type (same data; complex128 kernels <-> real float64 twins)
    alt = None
    if not args.no_alt_dtype:
        s_alt = dv.real_or_complex_to_device(s_loc, dev, widen=real)
        ms_alt, out_alt, _ = timed(make_step(s_alt), args.steps, warm)
        check_flags("alternate dtype")
        if rank == 0:
            da = per_point_rel(out_alt[0][::max(1, f_total // 512)].cpu().numpy(), gsm_dev[::max(1, f_total // 512)].cpu().numpy())
        alt = {"dtype": "c128" if real else "f64", "value": f_total / (ms_alt * 1e-3), "unit": UNIT, "ms_per_step": ms_alt,
               "max_rel_diff_vs_primary": float(da.max()) if rank == 0 else None,
               "note": "same workload and timed loop on the other arithmetic type: " +
                       ("real data embedded in complex128, complex128 kernels throughout (the north star's kernels)" if real
                        else "real float64 twins of every kernel (the reference's own dtype)")}
        del s_alt, out_alt
        path.drop_graph()

    # ---- per-kernel and per-stage timing (CUDA events on the launching stream, separate pass over the same steps)
    prof_steps = max(1, min(args.steps, 3))
    for _ in range(2):                                        # eager warm-up (the timed loop above may have been graph replays)
        path.step(s_dev, want_x=False, gather=True)
    barrier()
    dv.timer = dv.KernelTimer()
    path.stage_events = []
    for _ in range(prof_steps):
        path.step(s_dev, want_x=False, gather=True)           # eager: per-kernel events cannot be recorded inside a replay
    agg = dv.timer.summary()
    dv.timer = None
    # basis and projection overlap (the SVD rotation runs on a side stream under the SpMMs), so they are timed together
    stage_ms = {"basis_plus_projection": 0.0, "sweep": 0.0, "gather": 0.0}
    for ev in path.stage_events:
        for i, key in enumerate(("basis_plus_projection", "sweep", "gather")):
            stage_ms[key] += ev[i].elapsed_time(ev[i + 1]) / prof_steps
    path.stage_events = None
    have_peaks = os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json"))
    hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"] if have_peaks else 6650.0
    peak_src = "MEASURED_PEAKS.json hbm_gbs (measured)" if have_peaks else "fallback 6650 GB/s"
    kernels = {}
    dominant, dom_ms, all_ms = None, -1.0, 0.0
    for kname, a in agg.items():
        ms_call = a["ms"] / a["calls"]
        kernels[kname] = {"calls_per_step": a["calls"] / prof_steps, "ms_per_call": ms_call, "ms_per_step": a["ms"] / prof_steps,
                          "GBps": a["bytes"] / a["calls"] / ms_call / 1e6 if ms_call > 0 else None,
                          "TFLOPs": a["flops"] / a["calls"] / ms_call / 1e9 if ms_call > 0 else None}
        all_ms += a["ms"]
        if a["ms"] > dom_ms:
            dominant, dom_ms = kname, a["ms"]
    traffic, traffic_src = None, None
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        ent = tr.get(f"{name}:{'f64' if real else 'c128'}:{dominant}")
        if ent:
            traffic, traffic_src = ent["bytes_per_point"] * (f_total / world), ent["source"]
    except Exception:
        pass
    roof = None
    if dominant is not None:
        a = agg[dominant]
        ms_call = kernels[dominant]["ms_per_call"]
        t_mem = a["bytes"] / a["calls"] / (hbm_peak * 1e9)
        t_flop = a["flops"] / a["calls"] / (fp64_peak * 1e12)
        share = {"share_of_timed_kernels": dom_ms / all_ms, "share_of_step": (dom_ms / prof_steps) / ms_step,
                 "traffic_source": traffic_src or "no ncu capture of this kernel at this size is committed"}
        if t_flop >= t_mem:
            ach = a["flops"] / a["calls"] / (ms_call * 1e-3) / 1e12
            roof = {"kernel": dominant, "bound": "tensor", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s", "frac": ach / fp64_peak,
                    "traffic": traffic, "peak_source": fp64_src, **share}
        else:
            ach = a["bytes"] / a["calls"] / (ms_call * 1e-3) / 1e9
            roof = {"kernel": dominant, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                    "traffic": traffic, "peak_source": peak_src, **share}

    # ---- end to end through the reference-facing call, host (pinned) buffers in, host array out (rank-local job)
    e2e = None
    if world == 1:
        def pin(a):
            return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()

        def pinned_csc(a):
            a = csc_array(a)
            return csc_array((pin(a.data), pin(a.indices.astype(np.int32)), pin(a.indptr.astype(np.int32))), shape=a.shape)

        s_host = pin(s_loc)
        c_host, g_host, b_host = pinned_csc(in_c), pinned_csc(in_gamma), pinned_csc(in_b)
        out_pinned = torch.empty((f_total, m, m), dtype=torch.complex128).pin_memory()
        k_e2e = max(3, min(args.steps, 20 if ms_step < 50 else 5))
        # the call allocates its device buffers on two streams (compute and upload): start from an empty cache and warm the
        # allocator's per-stream pools up, otherwise some timed calls pay a cudaMalloc (seen as 20-50 ms outliers)
        path.drop_graph()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        for _ in range(6 if ms_step < 50 else 3):
            th.model_order_reduction_gsm_from_snapshots(f, s_host, c_host, g_host, b_host, pinned_out=out_pinned, real_path=real)
        torch.cuda.synchronize()
        import gc
        gc.collect()
        gc.disable()                                           # no collector pause inside the few-millisecond calls
        dv.transfer_bytes["h2d"] = dv.transfer_bytes["d2h"] = 0
        per_call = []
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            tc = time.perf_counter()
            gsm_host = th.model_order_reduction_gsm_from_snapshots(f, s_host, c_host, g_host, b_host, pinned_out=out_pinned, real_path=real)
            per_call.append(time.perf_counter() - tc)           # the call returns after its blocking download
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / k_e2e
        e2e = {"value": f_total / dt, "unit": UNIT, "h2d_bytes_per_step": dv.transfer_bytes["h2d"] // k_e2e,
               "d2h_bytes_per_step": dv.transfer_bytes["d2h"] // k_e2e, "ms_per_step": dt * 1e3, "steps": k_e2e,
               "ms_per_call_median": float(np.median(per_call)) * 1e3, "ms_per_call_max": float(np.max(per_call)) * 1e3,
               "ms_per_call": [round(t * 1e3, 3) for t in per_call],
               "call": "morfem_b200.test_helpers.model_order_reduction_gsm_from_snapshots (host ndarrays / scipy csc in pinned memory)"}
        # PCIe floor of that call: nothing but the same pinned host buffers copied to the device (what bounds e2e)
        bufs = [torch.from_numpy(s_host)] + [torch.from_numpy(np.asarray(x)) for a_ in (c_host, g_host, b_host) for x in (a_.data, a_.indices, a_.indptr)]
        dsts = [torch.empty_like(b_, device=dev) for b_ in bufs]
        torch.cuda.synchronize()
        c0_, c1_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0_.record()
        for _ in range(3):
            for d_, b_ in zip(dsts, bufs):
                d_.copy_(b_, non_blocking=True)
        c1_.record()
        torch.cuda.synchronize()
        copy_ms = c0_.elapsed_time(c1_) / 3
        copy_bytes = sum(b_.numel() * b_.element_size() for b_ in bufs)
        e2e["h2d_copy_floor"] = {"ms": copy_ms, "bytes": copy_bytes, "GBps": copy_bytes / copy_ms / 1e6,
                                 "note": "the same pinned input buffers copied host->device with nothing else running"}
        del dsts
        gc.enable()
        # sanity: the e2e result equals the device-resident result
        sub = slice(None, None, max(1, f_total // 2048))
        d_e2e = per_point_rel(gsm_host[sub], gsm_dev[sub].cpu().numpy())
        e2e["max_rel_diff_vs_device_resident"] = float(d_e2e.max())
        if not np.all(d_e2e < 1e-8):
            raise SystemExit("bench: e2e and device-resident S-parameters disagree")
    else:
        # N > 1: the public multi-GPU call is ShardedHotPath.step on device-resident shards; its e2e adds the per-rank
        # snapshot upload and the S-parameter download
        s_host = torch.from_numpy(np.ascontiguousarray(s_loc)).pin_memory()
        out_pinned = torch.empty((f_total, m, m), dtype=torch.complex128).pin_memory()
        k_e2e = max(3, min(args.steps, 10))
        path.drop_graph()                                      # the eager calls below allocate their own buffers: give the graph's pool back first
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        for _ in range(2):
            path.step(s_dev, want_x=False, gather=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(k_e2e):
            sd = s_host.to(dev, non_blocking=False)
            if not real:
                sd = sd.to(torch.complex128)
            gsm_all = path.step(sd, want_x=False, gather=True)[0]
            out_pinned.copy_(gsm_all)
        barrier()
        dt = (time.perf_counter() - t0) / k_e2e
        tt_ = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt_, op=dist.ReduceOp.MAX)
        dt = float(tt_.item())
        e2e = {"value": f_total / dt, "unit": UNIT, "h2d_bytes_per_step": int(s_host.numel() * 8) * world, "d2h_bytes_per_step": int(out_pinned.numel() * 16),
               "ms_per_step": dt * 1e3, "steps": k_e2e, "call": "morfem_b200.dist.ShardedHotPath.step (per-rank snapshot rows from pinned host memory)"}

    # ---- stages 1+2 alone, device timed (CUDA graph where the step is captured; else eager launches)
    bp_alone_ms = None
    try:
        def step12():
            if use_graph:
                return path.step_graph(s_dev, want_x=False, skip_sweep=True)
            return path.step(s_dev, want_x=False, gather=False, optimistic=True, skip_sweep=True)
        bp_alone_ms, _, _ = timed(step12, args.steps, 3)
        path.drop_graph()
    except Exception as exc:                                  # pragma: no cover - reported, not fatal
        bp_alone_ms = None
        print(f"bench: stage-1/2 timing failed: {exc!r}", file=sys.stderr)

    # ---- stages 1+2 against their composite roofline (SURVEY.md 8d): per kernel
    #      max(algorithmic bytes / measured HBM peak, flops / measured FP64 peak), complex128 operands, real operator values
    sweep_ms_alone = kernels.get("sweep_lu_gsm", {}).get("ms_per_step")
    bp_roof = None
    if sweep_ms_alone:
        n_loc = n / world
        wbytes = 16.0 if not real else 8.0
        fl = 1.0 if not real else 0.25                            # real twins: a quarter of the flops
        bw, p64 = hbm_peak * 1e9, fp64_peak * 1e12
        t_roof = max(6 * wbytes * n_loc * r / bw, 20.0 * n_loc * r * r * fl / p64)                       # CholeskyQR2 + rotation
        for a_ in (in_c, in_gamma):
            nnz_loc = a_.nnz / world
            t_roof += max((nnz_loc * 12.0 + 4.0 * (n_loc + 1) + 2 * wbytes * n_loc * r) / bw, (2.0 if real else 4.0) * nnz_loc * r / p64)   # SpMM (real operator values)
            t_roof += max((2 * wbytes * n_loc * r + wbytes * r * r) / bw, 8.0 * n_loc * r * r * fl / p64)     # Q^T (A Q)
        bp_ms = ms_step - sweep_ms_alone - stage_ms["gather"]
        bp_roof = {"ms": bp_alone_ms, "t_roof_ms": t_roof * 1e3, "frac": t_roof * 1e3 / bp_alone_ms if bp_alone_ms else None,
                   "ms_in_step": bp_ms, "frac_in_step": t_roof * 1e3 / bp_ms if bp_ms > 0 else None,
                   "note": "ms: stages 1+2 timed alone on the device (max over ranks); ms_in_step: whole timed step minus "
                           "the sweep kernel timed alone; roofline = sum over kernels of max(bytes/HBM, flops/FP64) per GPU (SURVEY 8d)"}

    # ---- secondary line: BASELINE configs[1] (N=200k, r=64, 2 ports, 10k points), same timed loop, single GPU only
    secondary = None
    if world == 1 and name != "cfg2" and not args.no_secondary:
        del path, s_dev
        torch.cuda.empty_cache()
        wl2 = WORKLOADS["cfg2"]
        ops2 = build_operators(wl2)
        path2 = make_path(ops2, 0, 1)
        s2 = dv.real_or_complex_to_device(snapshot_rows(ops2[4], wl2["r"], 0, ops2[4]), dev, widen=not real)

        def step2():
            return path2.step_graph(s2, want_x=False) if use_graph else path2.step_deferred(s2, want_x=False, gather=True)
        ms2, out2, _ = timed(step2, max(args.steps, 20), 3)
        ok2 = (path2.verify() is None) if use_graph else path2.verify_deferred()
        idx2 = sample_indices(wl2["f"], 256)
        red2 = [np.zeros((wl2["r"], wl2["r"])) if o is None else np.ascontiguousarray(o.cpu().numpy().real) for o in out2[2][:3]]
        red2.append(np.ascontiguousarray(out2[2][3].cpu().numpy().real))
        g2, _ = cpu_sweep(ops2[3][idx2], red2)
        e2 = per_point_rel(out2[0][torch.from_numpy(idx2).to(dev)].cpu().numpy(), g2)
        tol2 = np.maximum(1e-10, 20 * EPS * system_conds(ops2[3][idx2], red2))
        secondary = {"cfg2": {"config": workload_config("cfg2", wl2, ops2[4]), "value": wl2["f"] / (ms2 * 1e-3), "unit": UNIT, "ms_per_step": ms2,
                              "dtype": "c128" if not real else "f64", "cholqr2_flags_ok": bool(ok2),
                              "parity_stage_isolated": {"max_rel_err": float(e2.max()), "worst_err_over_tol": float((e2 / tol2).max()), "points": int(idx2.size)}}}

    if rank == 0:
        sweep_k = kernels.get("sweep_lu_gsm", {})
        cfg = workload_config(name, wl, n)
        cfg.update({"N_dof_per_gpu": n // world, "step": "basis (CholeskyQR2+SVD) + projection + reduced solves + S-parameters" +
                    (", replayed from one CUDA graph" if use_graph else ", eager launches"),
                    "parallelism": "rows of Q/operators and sweep points block-sharded over %d GPU(s)" % world})
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "c128" if not real else "f64", "data": "synthetic",
                "config": cfg,
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu_baseline, "parity": parity,
                "other_dtype": alt,
                "basis_plus_projection": bp_roof,
                "stages": {"basis_plus_projection_ms": stage_ms["basis_plus_projection"], "sweep_ms": stage_ms["sweep"],
                           "gather_ms": stage_ms["gather"],
                           "sweep_kernel_points_per_s_per_gpu": (f_total / world) / (sweep_k["ms_per_step"] * 1e-3) if sweep_k.get("ms_per_step") else None},
                "kernels": kernels, "secondary": secondary}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS))
    ap.add_argument("--r", type=int, default=0, help="override the basis size of the workload (BASELINE configs[3]: r = 16..512 at N = 1M)")
    ap.add_argument("--points", type=int, default=0, help="override the number of sweep points of the workload")
    ap.add_argument("--ports", type=int, default=0, help="override the number of ports of the workload")
    ap.add_argument("--cpu-points", type=int, default=0, help="sweep points the CPU legs solve (scaled to the full axis); 0 = per workload")
    ap.add_argument("--cpu-rows", type=int, default=62500, help="rows of the snapshot block / operators the reference arm's stages 1+2 run on per step")
    ap.add_argument("--parity", default="auto", choices=["auto", "full", "isolated"],
                    help="full: the whole path on the CPU once (svd of the full snapshot block: ~30 s at cfg3) -- default at N=1; "
                         "isolated: CPU sweep on the reduced model the GPU produced")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the cfg2 line reported under 'secondary'")
    ap.add_argument("--dtype", default="c128", choices=["auto", "c128", "f64"],
                    help="c128: complex128 kernels throughout (north star); f64: the real float64 twins (the reference's own dtype; "
                         "valid because the synthetic operators and snapshots are real, like the reference's data)")
    ap.add_argument("--no-alt-dtype", action="store_true", help="skip the second timed loop on the other arithmetic type")
    ap.add_argument("--no-graph", action="store_true", help="run the eager (adaptive CholeskyQR) step instead of the CUDA-graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (S-parameters, basis, reduced operators, per-point "
                         "pivot info) as DIR/<name>.npy in float64, complex arrays with a trailing (real, imag) axis; a larger array "
                         "keeps a fixed seeded sample of its rows (DIR/<name>_rows.npy), 64 MB in all.  With --gpus N > 1, rank 0 "
                         "writes and the basis and pivot info are its own shard")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the b200 path; the reference arm times a sample of the workload")
    wl = dict(WORKLOADS[args.workload])
    if args.r or args.points or args.ports:
        wl["r"], wl["f"], wl["m"] = args.r or wl["r"], args.points or wl["f"], args.ports or wl["m"]
        wl["desc"] += f" [overridden: r={wl['r']}, {wl['m']} ports, {wl['f']} points -- BASELINE configs[3], basis-size sweep]"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, args.workload, wl, rank, world)
        return
    if world != args.gpus:
        raise SystemExit(f"bench.py: --gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
    run_b200(args, args.workload, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
