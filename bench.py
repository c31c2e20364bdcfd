#!/usr/bin/env python
"""Benchmark of the per-voxel T2 fit: masked-voxel fits per second (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c1|c2|c3|c4|c5] [--solver auto|fast|lbfgsb|lbfgsb_dense] [--impl reference]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--config (default c2 = BASELINE.json configs[1], the configuration the metric is quoted on; the other four are the remaining
BASELINE configs, each with its own roofline / parity / cpu_baseline blocks, run by hand and logged in profiles/):

  c1  64^3 x 4 TE, sphere mask, gaussian LF --no_prior            volume step, fast solver (the reference-runnable case)
  c2  256^3 x 5 TE, ellipsoid brain mask, gaussian LF --no_prior  volume step, fast solver            [HEADLINE]
  c3  160x256x256 x 12 TE phantom, gaussian_rician --no_prior      volume step, L-BFGS-B solver, dense-matrix form (the reference's own
                                                                  optimiser: the loosely converged 3-parameter maps need its path;
                                                                  `other_solvers`: scipy's compact form, and the fast minimiser)
  c4  64 volumes 160^3 x 6 TE, gaussian --no_prior                 t2map_series from HOST arrays, volumes dealt round-robin to ranks
  c5  512^3 x 16 TE unmasked, gaussian_rician --no_prior           ONE job strong-scaled over contiguous slabs + all-gather of T2 / S0

One *pass* = the hot block of process_t2maps for one volume (run_t2mapping.py:411-461): zero the four dense maps, fit every
masked voxel, residual epilogue, scatter into the dense maps, flags / iteration counts / final errors per voxel.  One *step* =
`passes_per_step` back-to-back passes (chosen so that one step lasts >= 30 ms whatever K is, so that the default 20 timed steps
last >= 0.6 s: a c2 pass is 67 us, and a timed region of 20 x 67 us cannot be cross-checked against a wall clock).

--dump-outputs DIR (volume configurations c1 / c2 / c3 on one GPU): after the timed steps, what the last pass handed its caller --
the four dense maps and the per-voxel fun / nit / status -- at a fixed, seeded sample of the masked voxels, as DIR/<name>.npy
(see dump_outputs).  The inputs are seeded, so two builds run with the same arguments can be compared array for array.

  value     N = 1: whole-job fits/s of the step above with the volume resident in HBM.
            N > 1: the PRODUCT's multi-GPU path -- ONE job of N volume-sized slabs, every rank holds only its slab, fits it
            (compact results written straight into its chunk of the gather buffers) and the (t2, k, res, status) vectors are
            all-gathered in place (NCCL over NVLink) INSIDE the timed step; full-vector equality with the ranks' local results is
            asserted.  `replicas` beside it: N independent dense-map steps (no gather), as round 1 reported.
  e2e       the same metric through fit_voxels_batch() with HOST (page-locked) numpy buffers, host<->device traffic inside.
  roofline  dominant kernel of the step against the measured HBM peak (algorithmic bytes / launch time from CUDA events).
  parity    a sample of the workload fitted by the oracle port (scipy exactly as fit_voxel drives it) vs the default solver.
  cpu_baseline  the oracle port on a bounded sample, all host cores.

--impl reference: the reference's own CPU implementation of the path (oracle port: scipy.optimize L-BFGS-B + multiprocessing
over all host cores), each step a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os

# the CPU arm forks scipy workers: BLAS must be single-threaded BEFORE numpy loads it (SURVEY.md section 6:
# without this the forked workers oversubscribe the cores and the baseline collapses 50x)
for _v in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS"):
    os.environ.setdefault(_v, "1")
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "masked_voxel_T2_fits_per_sec"
UNIT = "fits/s"
CONFIGS = {
    "c1": dict(kind="volume", fit="gaussian", solver="fast",
               workload="c1: 64x64x64 x 4 TE, sphere mask, gaussian 2-param fit, LF preset, --no_prior"),
    "c2": dict(kind="volume", fit="gaussian", solver="fast",
               workload="c2: 256x256x256 x 5 TE adult-brain, ellipsoid mask, gaussian 2-param fit, LF preset, --no_prior"),
    "c3": dict(kind="volume", fit="gaussian_rician", solver="lbfgsb_dense",
               workload="c3: 160x256x256 x 12 TE NIST phantom, Rician data, gaussian_rician 3-param fit, LF preset, --no_prior"),
    "c4": dict(kind="series", fit="gaussian", solver="fast",
               workload="c4: 64 fetal-brain volumes 160x160x160 x 6 TE, gaussian 2-param fit, LF preset, --no_prior, from host arrays"),
    "c5": dict(kind="slab", fit="gaussian_rician", solver="lbfgsb_dense",
               workload="c5: 512x512x512 x 16 TE unmasked, Rician data, gaussian_rician 3-param fit, LF preset, --no_prior, slab-partitioned"),
}
LB_SOLVERS = ("lbfgsb", "lbfgsb_dense")
LB_WHAT = {"lbfgsb": "the reference's own optimiser, scipy's compact 2m x 2m form restated operation by operation (FP64 L-BFGS-B, lbfgsb_kernel)",
           "lbfgsb_dense": "the reference's own optimiser with the limited-memory matrix as the dense n x n matrix it represents "
                           "(FP64 L-BFGS-B, lbfgsb_dense_kernel): same algorithm, objectives, differences, line search and stopping tests"}
LB_KERNEL = {"lbfgsb": "lbfgsb_kernel<%s> (one thread per voxel, FP64, compact matrices in local memory)",
             "lbfgsb_dense": "lbfgsb_dense_kernel<%s> (one thread per voxel, FP64, dense n x n matrix, state in registers + 480 B of pairs)"}
SCALE = float(os.environ.get("T2FIT_BENCH_SCALE", "1.0"))       # shrinks every spatial axis (smoke runs of the bench itself)
MIN_STEP_S = float(os.environ.get("T2FIT_BENCH_MIN_STEP_S", "0.03"))
DUMP_SAMPLE = 1 << 20           # masked voxels written by --dump-outputs: 7 float32 + 1 float64 arrays of 2^20 = 36 MB


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d["hbm_gbs"]), "sm_max_mhz": float(d.get("sm_max_mhz", 1965.0)), "src": "measured"}
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# workloads
# ---------------------------------------------------------------------------------------------------
def make_volume_workload(cfg_name, index):
    """(flat f32 [N,E], mask_indices int64 [M], TEeffs) of volume `index` of a volume-kind configuration."""
    from fetal_t2mapping_b200 import synth
    y, mask, te, _ = synth.make_volume(cfg_name, scale=SCALE, volume_index=index)
    flat = np.ascontiguousarray(y.reshape(-1, te.size))
    idx = np.flatnonzero(mask.reshape(-1)).astype(np.int64)
    return flat, idx, te


def c5_te():
    return np.linspace(100.0, 700.0, 16)


def c5_rows_host(n, seed=4):
    """A host sample of c5-like rows (same distributions as the device generator) for the CPU arm."""
    rng = np.random.default_rng(seed)
    te = c5_te().astype(np.float32)
    t2 = np.exp(rng.uniform(np.log(10.0), np.log(2000.0), n)).astype(np.float32)
    s0 = rng.uniform(300.0, 3000.0, n).astype(np.float32)
    s = s0[:, None] * np.exp(-te[None, :] / t2[:, None])
    n1 = rng.standard_normal(s.shape).astype(np.float32) * 20.0
    n2 = rng.standard_normal(s.shape).astype(np.float32) * 20.0
    return np.sqrt((s + n1) ** 2 + n2 ** 2).astype(np.float32)


def c5_rows_device(torch, dev, first, count, n_total):
    """Rows [first, first + count) of the c5 volume, generated on the device in chunks (8.6 GB at full size); the generator is
    seeded per 2^20-voxel block so that any rank can make any slab."""
    te = torch.tensor(c5_te(), device=dev, dtype=torch.float32)
    y = torch.empty((count, 16), dtype=torch.float32, device=dev)
    blk = 1 << 20
    b0 = first // blk
    while b0 * blk < first + count:
        lo, hi = max(first, b0 * blk), min(first + count, (b0 + 1) * blk, n_total)
        g = torch.Generator(device=dev).manual_seed(1000 + b0)
        m = min(blk, n_total - b0 * blk)
        t2v = torch.exp(torch.empty(m, device=dev).uniform_(float(np.log(10.0)), float(np.log(2000.0)), generator=g))
        s0 = torch.empty(m, device=dev).uniform_(300.0, 3000.0, generator=g)
        s = s0[:, None] * torch.exp(-te[None, :] / t2v[:, None])
        rows = torch.sqrt((s + torch.randn((m, 16), device=dev, generator=g) * 20.0) ** 2 +
                          (torch.randn((m, 16), device=dev, generator=g) * 20.0) ** 2)
        y[lo - first:hi - first] = rows[lo - b0 * blk:hi - b0 * blk]
        del t2v, s0, s, rows
        b0 += 1
    return y


def cpu_rows_for(cfg_name, n, seed=11):
    """A seeded random sample of n masked rows of the configuration's workload (host), TEeffs."""
    if cfg_name == "c5":
        return c5_rows_host(n, seed), c5_te()
    flat, idx, te = make_volume_workload("c4" if cfg_name == "c4" else cfg_name, 0)
    rng = np.random.default_rng(seed)
    pick = np.sort(rng.choice(idx, size=min(n, idx.size), replace=False))
    return np.ascontiguousarray(flat[pick]), te


def oracle_fit(rows, te, fit, procs, mode="verbatim", starts=None):
    from oracle import fit_oracle as fo
    _, fp = fo.preset(fit, "lf")
    t0 = time.perf_counter()
    p, ok, nit, fun, _ = fo.fit_rows_oracle(rows, te, fit, fp, False, False, mode=mode, procs=procs, starts=starts)
    return dict(params=p, ok=ok, nit=nit, fun=fun, dt=time.perf_counter() - t0, rate=rows.shape[0] / (time.perf_counter() - t0))


def host_procs():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


# ---------------------------------------------------------------------------------------------------
# the reference arm
# ---------------------------------------------------------------------------------------------------
def run_reference(args):
    """scipy L-BFGS-B driven exactly as fit_voxel drives it, Pool over all host cores (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    cfg = CONFIGS[args.config]
    procs = host_procs()
    pool_rows, te = cpu_rows_for(args.config, 40000, seed=5)
    probe = oracle_fit(pool_rows[:256 * min(procs, 8)], te, cfg["fit"], procs)
    budget_s = float(os.environ.get("T2FIT_REF_BUDGET_S", "100"))
    per_step = int(np.clip(budget_s * probe["rate"] / max(1, args.steps + args.warmup), 256, 20000))
    rng = np.random.default_rng(200)

    def sample():
        return np.ascontiguousarray(pool_rows[np.sort(rng.choice(pool_rows.shape[0], size=min(per_step, pool_rows.shape[0]), replace=False))])
    for _ in range(args.warmup):
        oracle_fit(sample(), te, cfg["fit"], procs)
    t_tot, n_tot = 0.0, 0
    for _ in range(args.steps):
        rows = sample()
        r = oracle_fit(rows, te, cfg["fit"], procs)
        t_tot += r["dt"]
        n_tot += rows.shape[0]
    value = n_tot / t_tot
    import scipy
    smp = f"{per_step} masked voxels per step (seeded random sample of the workload), {args.steps} steps"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / max(1, args.steps), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "sample": smp, "scipy": scipy.__version__, "numpy": np.__version__},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": procs, "kind": "port", "sample": smp},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# the CUDA arm
# ---------------------------------------------------------------------------------------------------
class Ctx:
    pass


def gpu_setup(args):
    import torch
    import torch.distributed as dist
    import fetal_t2mapping_b200 as t2
    c = Ctx()
    c.rank = int(os.environ.get("RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    if c.world != args.gpus and c.world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={c.world}")
    torch.cuda.set_device(c.local)
    c.dev = torch.device("cuda", c.local)
    if c.world > 1:
        dist.init_process_group("nccl", device_id=c.dev)
    c.lib = t2.init(c.local)
    c.torch, c.dist, c.t2 = torch, dist, t2
    c.stream = torch.cuda.current_stream(c.dev)
    # OMP_NUM_THREADS=1 above is for the forked scipy workers of the CPU arm; torch's own host copies (the loader's casts into
    # page-locked planes) get the cores back
    torch.set_num_threads(max(1, host_procs() // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", c.world)))))
    return c


def barrier(c):
    if c.world > 1:
        c.dist.barrier()
    c.torch.cuda.synchronize()


def max_over_ranks(c, *vals):
    if c.world == 1:
        return [float(v) for v in vals]
    t = c.torch.tensor(list(vals), device=c.dev, dtype=c.torch.float64)
    c.dist.all_reduce(t, op=c.dist.ReduceOp.MAX)
    return [float(v) for v in t]


def sum_over_ranks(c, v):
    if c.world == 1:
        return int(v)
    t = c.torch.tensor([int(v)], device=c.dev, dtype=c.torch.int64)
    c.dist.all_reduce(t)
    return int(t[0])


def time_steps(c, step, steps, passes, finish=None):
    """K steps of `passes` passes between two CUDA events on the launching stream, barrier + synchronize on both sides;
    returns the max over ranks of the elapsed milliseconds.  No events inside: a pair around every launch was measured to
    stretch a 68 us c2 pass to 125 us."""
    torch = c.torch
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier(c)
    e0.record(c.stream)
    for _ in range(steps):
        for _ in range(passes):
            step()
    if finish is not None:
        finish()                                  # e.g. make the stream wait for collectives still in flight
    e1.record(c.stream)
    barrier(c)
    return max_over_ranks(c, e0.elapsed_time(e1))[0]


def pick_passes(c, step, finish=None):
    """passes per step so that one step lasts >= MIN_STEP_S (same on every rank); independent of the step count, so that
    --steps K times K steps of the same size."""
    torch = c.torch
    for _ in range(3):
        step()
    if finish is not None:
        finish()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = 6
    e0.record(c.stream)
    for _ in range(n):
        step()
    if finish is not None:
        finish()
    e1.record(c.stream)
    torch.cuda.synchronize()
    per = max_over_ranks(c, e0.elapsed_time(e1) / n)[0] * 1e-3
    return int(np.clip(np.ceil(MIN_STEP_S / max(per, 1e-7)), 1, 5000))


def slab_hashes(torch, fields, bounds):
    """[world, F] int64: per slab and field the sum of the raw 32-bit patterns (uint8: of the bytes) -- equal tables mean
    equal vectors for the purpose of 'the gather delivered what the owner computed'."""
    rows = []
    for a, b in bounds:
        row = []
        for f in fields:
            v = f[a:b]
            row.append(v.view(torch.int32).to(torch.int64).sum() if v.dtype == torch.float32 else v.to(torch.int64).sum())
        rows.append(torch.stack(row))
    return torch.stack(rows)


def dump_outputs(torch, out_dir, maps, idx_d, per_voxel):
    """--dump-outputs: the dense maps (t2, k, sigma, res) and the per-voxel outputs (fun, nit, status) of the last pass at a
    fixed, seeded sample of DUMP_SAMPLE masked voxels (all of them if there are fewer), as float32 .npy files;
    voxel_index.npy (float64, exact) holds each sampled voxel's flat index in the volume.  Off-mask voxels are left out:
    the bench asserts that they are zero."""
    m = idx_d.numel()
    pick = np.arange(m) if m <= DUMP_SAMPLE else np.sort(np.random.default_rng(0).choice(m, DUMP_SAMPLE, replace=False))
    pick_d = torch.from_numpy(pick).to(idx_d.device)
    vox_d = idx_d[pick_d]
    arrays = {"voxel_index": vox_d.to(torch.float64)}
    arrays.update({name: maps[i][vox_d] for i, name in enumerate(("t2", "k", "sigma", "res"))})
    arrays.update({name: v[pick_d].to(torch.float32) for name, v in per_voxel.items()})
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def parity_block(c, cfg, rows, te, oracle, solver):
    """Delta-T2 of the CUDA solver(s) against the reference's scipy fit of the same rows, on all sampled voxels and on the
    converged ones (reference success and a tight restart from its own answer moves T2 by <= 1e-4, SURVEY 7.3)."""
    from oracle import fit_oracle as fo
    t2 = c.t2
    _, fp = t2.preset(cfg["fit"], True)
    ref_t2 = oracle["params"][:, 1]
    out = {"sample": int(rows.shape[0]), "reference": "oracle port = scipy L-BFGS-B exactly as fit_voxel calls it",
           "reference_success": float(np.mean(oracle["ok"])), "converged_share": float(np.mean(oracle["converged"][:oracle["conv_n"]])),
           "converged_classified_on": int(oracle["conv_n"])}
    names = [solver] + [s for s in ("fast", "lbfgsb_dense", "lbfgsb") if s != solver and not (s == "fast" and cfg["fit"] == "rician")]
    for name in names:
        rr = t2.fit_voxels_batch(rows, None, te, cfg["fit"], fp, prior=False, norm=False, solver=name)
        rel = np.abs(rr.t2.astype(np.float64) - ref_t2) / np.abs(ref_t2)
        cv = oracle["converged"]
        out[name] = {"t2_rel_le_1e-3_all": float(np.mean(rel <= 1e-3)), "t2_rel_le_1e-3_converged": float(np.mean(rel[cv] <= 1e-3)) if cv.any() else None,
                     "t2_rel_median": float(np.median(rel)), "t2_rel_p999": float(np.quantile(rel, 0.999)),
                     "success_equal": bool(np.array_equal(rr.status == 0, oracle["ok"])), "default": name == solver}
        if name in LB_SOLVERS:
            out[name]["nit_equal"] = float(np.mean(rr.nit == oracle["nit"]))
            out[name]["note"] = LB_WHAT[name]
        else:
            out[name]["note"] = ("bounded minimiser (multi-start), NOT the reference's point: the reference stops at ftol=gtol=1e-2"
                                 if cfg["fit"] != "gaussian" else "bounded minimiser = the reference's point up to its stopping error (ftol=1e-6)")
    return out


def cpu_leg(args, cfg):
    """CPU baseline + the oracle fits the parity block needs; BEFORE CUDA is initialised (the oracle forks workers)."""
    procs = host_procs()
    rows_all, te = cpu_rows_for(args.config, 200000)
    probe = oracle_fit(rows_all[:64 * procs], te, cfg["fit"], procs)
    n_s = int(os.environ.get("T2FIT_CPU_SAMPLE", "0")) or int(np.clip(12.0 * probe["rate"], 512, rows_all.shape[0]))
    rows = np.ascontiguousarray(rows_all[:n_s])
    o = oracle_fit(rows, te, cfg["fit"], procs)
    from oracle import fit_oracle as fo
    _, fp = fo.preset(cfg["fit"], "lf")
    n_c = min(rows.shape[0], 4000)                 # the converged classification costs a second (tight) fit: bounded
    conv = np.zeros(rows.shape[0], bool)
    good = np.isfinite(o["params"]).all(axis=1)
    starts = np.where(good[:, None], o["params"], np.array(fp["initial_guess"], float)[None, :])
    cs, _ = fo.converged_set(rows[:n_c], te, cfg["fit"], fp, False, False, starts[:n_c], (o["ok"] & good)[:n_c], procs=procs)
    conv[:n_c] = cs
    o["converged"] = conv
    o["conv_n"] = n_c
    import scipy
    base = {"value": o["rate"], "unit": UNIT, "cores": procs, "kind": "port",
            "sample": f"{rows.shape[0]} seeded random masked voxels of the same workload, {o['dt']:.1f} s, scipy {scipy.__version__} "
                      f"L-BFGS-B via multiprocessing.Pool({procs})"}
    return base, rows, te, o


def bench_volume(args, cfg):
    cpu = cpu_leg(args, cfg) if (int(os.environ.get("RANK", "0")) == 0 and int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_cpu_baseline) else None
    c = gpu_setup(args)
    torch, t2, lib = c.torch, c.t2, c.lib
    import ctypes as C
    from fetal_t2mapping_b200 import _abi
    from fetal_t2mapping_b200 import distributed as D
    from fetal_t2mapping_b200.api import _fill_problem
    fit = cfg["fit"]
    solver = cfg["solver"] if args.solver == "auto" else args.solver
    _, fp = t2.preset(fit, True)
    flat, idx, te = make_volume_workload(args.config, c.rank)
    n_vox, n_echo = flat.shape
    m = idx.size
    mono = fit == "gaussian"
    y_d = torch.from_numpy(flat).to(c.dev)
    idx_d = torch.from_numpy(idx).to(c.dev)
    maps = torch.empty((4, n_vox), dtype=torch.float32, device=c.dev)
    mask_np = np.zeros(n_vox, np.uint8)
    mask_np[idx] = 1
    mask_d = torch.from_numpy(mask_np).to(c.dev)          # the (union) mask volume, reshaped_mask of :412
    fun_d = torch.empty(m, dtype=torch.float32, device=c.dev)
    nit_d = torch.empty(m, dtype=torch.int32, device=c.dev)
    st_d = torch.empty(m, dtype=torch.uint8, device=c.dev)
    cnt_d = torch.zeros(4, dtype=torch.int64, device=c.dev)
    p, o = _abi.Problem(), _abi.Outputs()
    keep = _fill_problem(p, fit, fp, te, False, False, 0, 0.0, "auto", solver)
    p.echoes, p.memory, p.layout, p.mask_idx = y_d.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_AOS, idx_d.data_ptr()
    p.n_vox, p.n_fit = n_vox, m
    o.t2, o.k, o.sigma, o.res = maps[0].data_ptr(), maps[1].data_ptr(), maps[2].data_ptr(), maps[3].data_ptr()
    o.fun, o.nit, o.status, o.dense = fun_d.data_ptr(), nit_d.data_ptr(), st_d.data_ptr(), 1
    o.zero_fill_mask = mask_d.data_ptr()                 # np.zeros_like x4 (:415-418) done by the fit launch itself
    o.counts_dev = cnt_d.data_ptr()
    fill_in_fit = mono and solver == "fast" and os.environ.get("T2FIT_FILL", "fused") != "stream"

    def dense_pass():
        rc = lib.t2fit_run(C.byref(p), C.byref(o), c.stream.cuda_stream)
        if rc:
            raise RuntimeError(lib.t2fit_last_error())

    # ---- the product's multi-GPU step: slab-only inputs, compact results straight into the gather buffers, in-place all-gather
    sharded = None
    if c.world > 1:
        sizes = torch.zeros(c.world, dtype=torch.int64, device=c.dev)
        sizes[c.rank] = m
        c.dist.all_reduce(sizes)
        sizes_l = [int(v) for v in sizes.tolist()]
        # ONE job of `world` slabs: rank r's slab = the first m_s masked voxels of its volume, m_s = the common 128-aligned slab
        # length (distributed.slab_bounds cuts at multiples of 128: at most 127 of a volume's 1.6 M masked voxels are left out)
        m_s = (min(sizes_l) // D.ALIGN) * D.ALIGN
        L, n_job = m_s, c.world * m_s
        assert D.slab_bounds(n_job, c.world)[c.rank] == (c.rank * L, (c.rank + 1) * L)
        names = ["t2", "k", "res", "status"] + ([] if mono else ["sigma"])
        rows_d = y_d[idx_d[:m_s]].contiguous()                    # what a loader hands this rank: the rows of its slab, nothing else
        scnt = torch.zeros(4, dtype=torch.int64, device=c.dev)
        # TWO buffer sets: the all-gather of pass i (NCCL's stream) overlaps the fit of pass i+1 (compute stream), as
        # distributed.SlabPipeline does for a stream of jobs; the structs of the fit call are built once per set (this loop
        # issues a pass every ~50-100 us)
        sets = []
        for _ in range(2):
            bufs = {n: torch.zeros(c.world * L, dtype=torch.uint8 if n == "status" else torch.float32, device=c.dev) for n in names}
            mine = {n: bufs[n][c.rank * L:(c.rank + 1) * L] for n in names}
            p2, o2 = _abi.Problem(), _abi.Outputs()
            k2 = _fill_problem(p2, fit, fp, te, False, False, 0, 0.0, "auto", solver)
            p2.echoes, p2.memory, p2.layout, p2.mask_idx = rows_d.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_AOS, None
            p2.n_vox, p2.n_fit = m_s, m_s
            o2.t2, o2.k, o2.res, o2.status = mine["t2"].data_ptr(), mine["k"].data_ptr(), mine["res"].data_ptr(), mine["status"].data_ptr()
            o2.sigma = None if mono else mine["sigma"].data_ptr()
            o2.dense, o2.counts_dev = 0, scnt.data_ptr()
            sets.append({"bufs": bufs, "mine": mine, "p": p2, "o": o2, "keep": k2, "pending": None})
        bufs, mine = sets[0]["bufs"], sets[0]["mine"]
        state = {"i": 0}

        def fit_set(st):
            rc = lib.t2fit_run(C.byref(st["p"]), C.byref(st["o"]), c.stream.cuda_stream)
            if rc:
                raise RuntimeError(lib.t2fit_last_error())

        def fit_only_pass():
            fit_set(sets[0])

        try:                                                      # one NCCL group launch for the fields of a pass if torch offers it
            from torch.distributed import _coalescing_manager

            def gather_async(st):
                with _coalescing_manager(device=c.dev, async_ops=True) as cm:
                    for n in names:
                        c.dist.all_gather_into_tensor(st["bufs"][n], st["mine"][n])
                return [cm]
            for w in gather_async(sets[0]):
                w.wait()
            torch.cuda.synchronize()
            coalesced = True
        except Exception:
            coalesced = False

            def gather_async(st):
                return [c.dist.all_gather_into_tensor(st["bufs"][n], st["mine"][n], async_op=True) for n in names]

        def wait_set(st):
            if st["pending"]:
                for w in st["pending"]:
                    w.wait()                                      # the compute stream waits for that set's gathers; the host does not
                st["pending"] = None

        def sharded_pass():                                       # pipelined: gather(i) || fit(i+1)
            st = sets[state["i"] & 1]
            state["i"] += 1
            wait_set(st)                                          # its buffers are about to be overwritten
            fit_set(st)
            st["pending"] = gather_async(st)

        def sharded_finish():
            for st in sets:
                wait_set(st)

        def single_job_pass():                                    # one job alone: fit, then its gather, nothing overlapped
            fit_set(sets[0])
            for w in gather_async(sets[0]):
                w.wait()

        # the all-gather FUSED into the fit kernels (distributed.FusedAllGather): peer stores from the epilogue + a one-element
        # all-reduce as the barrier; falls back to the NCCL path on every rank if CUDA IPC is not available
        fa = None
        try:
            fa = D.FusedAllGather(n_job, fit)
            ok_f = 1
        except Exception as ex:
            ok_f, fused_err = 0, repr(ex)
        okt = torch.tensor([ok_f], device=c.dev, dtype=torch.int32)
        c.dist.all_reduce(okt, op=c.dist.ReduceOp.MIN)
        if int(okt[0]) == 0:
            fa = None

        # multicast buffers (NVSwitch replicates one store into every rank's buffer): checked against the owners' slabs BEFORE
        # anything is timed; any difference on any rank -> the unicast CUDA-IPC form on every rank
        fused_note = None
        if fa is not None and fa.multicast:
            bounds_f = [(r * L, (r + 1) * L) for r in range(c.world)]
            ok_m = 1
            for _ in range(3):                                    # both buffer sets
                rf = fa.result(fa.submit(rows_d, te, fp, prior=False, norm=False, solver=solver))
                torch.cuda.synchronize()
                tab = slab_hashes(torch, [rf[n][c.rank * L:(c.rank + 1) * L] for n in names], [(0, m_s)])[0]
                tabs = torch.zeros((c.world, len(names)), dtype=torch.int64, device=c.dev)
                c.dist.all_gather_into_tensor(tabs, tab)
                ok_m &= int(torch.equal(tabs, slab_hashes(torch, [rf[n] for n in names], bounds_f)))
            okt = torch.tensor([ok_m], device=c.dev, dtype=torch.int32)
            c.dist.all_reduce(okt, op=c.dist.ReduceOp.MIN)
            if int(okt[0]) == 0:
                fused_note = "multicast stores did not reproduce the owners' slabs on this node: unicast peer stores used"
                fa.close()
                fa = D.FusedAllGather(n_job, fit, multicast="off")

        def fused_pass():
            fa.submit(rows_d, te, fp, prior=False, norm=False, solver=solver)

        fa2 = None                                                # the literal "gather of the parameter maps": T2 and S0 only
        if fa is not None:
            try:
                fa2 = D.FusedAllGather(n_job, fit, gather=("t2", "k"))
                ok2 = 1
            except Exception:
                ok2 = 0
            okt = torch.tensor([ok2], device=c.dev, dtype=torch.int32)
            c.dist.all_reduce(okt, op=c.dist.ReduceOp.MIN)
            if int(okt[0]) == 0:
                fa2 = None

        def fused_pass_t2s0():
            fa2.submit(rows_d, te, fp, prior=False, norm=False, solver=solver)

    sampler = ClockSampler(c.local) if c.rank == 0 else None
    if sampler:
        sampler.start()
    main_pass = (fused_pass if fa is not None else sharded_pass) if c.world > 1 else dense_pass
    main_finish = (None if fa is not None else sharded_finish) if c.world > 1 else None
    for _ in range(max(3, args.warmup)):
        main_pass()
    passes = pick_passes(c, main_pass, main_finish)
    for _ in range(max(3, args.warmup)):                  # W warm-up STEPS of the final shape
        for _ in range(min(passes, 50)):
            main_pass()
    if main_finish:
        main_finish()
    elapsed_ms = time_steps(c, main_pass, args.steps, passes, main_finish)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs:                                 # the maps still hold the last timed pass (one GPU: dense_pass)
        dump_outputs(torch, args.dump_outputs, maps, idx_d, {"fun": fun_d, "nit": nit_d, "status": st_d})
    m_total = sum_over_ranks(c, m_s if c.world > 1 else m)
    value = m_total * args.steps * passes / (elapsed_ms * 1e-3)
    pass_ms = elapsed_ms / (args.steps * passes)

    extra = {}
    if c.world > 1:
        # the gather delivered, bit for bit, what every owner computed (every rank checks every slab) -- for both forms
        bounds = [(r * L, (r + 1) * L) for r in range(c.world)]

        def check_gathered(full, local):
            local_tab = slab_hashes(torch, [local[n] for n in names], [(0, m_s)])[0]
            tabs = torch.zeros((c.world, len(names)), dtype=torch.int64, device=c.dev)
            c.dist.all_gather_into_tensor(tabs, local_tab)
            return bool(torch.equal(tabs, slab_hashes(torch, [full[n] for n in names], bounds)))
        for _ in range(4):                                # (the timed loop may have ended on either buffer set)
            sharded_pass()
        sharded_finish()
        torch.cuda.synchronize()
        ok_g = all(check_gathered(st["bufs"], {n: st["mine"][n] for n in names}) for st in sets)
        # and the slab fit itself equals the single-GPU dense-map fit of the same volume
        dense_pass()
        torch.cuda.synchronize()
        sel = idx_d[:m_s]
        fit_ok = bool(torch.equal(mine["t2"][:m_s], maps[0][sel])) and bool(torch.equal(mine["res"][:m_s], maps[3][sel])) \
            and bool(torch.equal(mine["status"][:m_s], st_d[:m_s]))
        ok_fused = None
        if fa is not None:
            s0 = fa.submit(rows_d, te, fp, prior=False, norm=False, solver=solver)
            rf = fa.result(s0)
            torch.cuda.synchronize()
            ok_fused = check_gathered(rf, {n: rf[n][c.rank * L:(c.rank + 1) * L] for n in names}) and \
                all(bool(torch.equal(rf[n], bufs[n][:n_job])) for n in names)
        ok_all = torch.tensor([int(ok_g and fit_ok and ok_fused is not False)], device=c.dev, dtype=torch.int32)
        c.dist.all_reduce(ok_all, op=c.dist.ReduceOp.MIN)
        assert int(ok_all[0]) == 1, "sharded fit + gather differs from the single-GPU fit"
        p_fit = pick_passes(c, fit_only_pass)
        fit_ms = time_steps(c, fit_only_pass, args.steps, p_fit) / (args.steps * p_fit)
        p_one = pick_passes(c, single_job_pass)
        one_ms = time_steps(c, single_job_pass, args.steps, p_one) / (args.steps * p_one)
        p_pipe = pick_passes(c, sharded_pass, sharded_finish)
        pipe_ms = time_steps(c, sharded_pass, args.steps, p_pipe, sharded_finish) / (args.steps * p_pipe)
        p_rep = pick_passes(c, dense_pass)
        rep_ms = time_steps(c, dense_pass, args.steps, p_rep) / (args.steps * p_rep)
        bytes_in = sum((c.world - 1) * L * (1 if n == "status" else 4) for n in names)
        extra["sharded"] = {"form": "fused all-gather" if fa is not None else "NCCL all-gather, pipelined",
                            "op": ("fit of the rank's slab; the kernel epilogue stores the compact results (" + ", ".join(names) + "; status as uint8) into "
                                   "its own buffer and, over NVLink, into every peer's buffer (" + ("float fields: ONE store per value to the buffers' NVSwitch "
                                   "multicast address, replicated by the switch; status: unicast peer stores" if fa.multicast else "CUDA-IPC peer stores")
                                   + "); a one-element NCCL all-reduce ordered after the kernels is the barrier (distributed.FusedAllGather)") if fa is not None else
                                  "fit + in-place NCCL all_gather_into_tensor per field, two buffer sets (distributed.SlabPipeline)",
                            "ms_per_pass": pass_ms, "fit_only_ms": fit_ms, "gather_bytes_received_per_rank": int(bytes_in),
                            "gather_gbs_received_per_rank": bytes_in / max(pass_ms, 1e-9) / 1e6,
                            "equals_single_gpu_fit": True, "gathered_equals_owner": True, "voxels_per_rank": m_s,
                            "note": "every rank ends with the full vectors: it RECEIVES (N-1) slabs per pass, which bounds the pass at "
                                    "(N-1) * slab * 13 B / NVLink ingest whatever the fit costs (DESIGN.md section 5)"}
        extra["sharded_nccl"] = {"op": "fit + in-place NCCL all_gather_into_tensor per field (" + ("one coalesced group launch" if coalesced else "one launch per field")
                                       + "), status as uint8", "pipelined_ms_per_pass": pipe_ms, "pipelined_value": m_total / (pipe_ms * 1e-3),
                                 "single_job_ms": one_ms, "single_job_gather_ms": one_ms - fit_ms, "single_job_value": m_total / (one_ms * 1e-3),
                                 "gather_gbs_received_per_rank_single_job": bytes_in / max(one_ms - fit_ms, 1e-9) / 1e6,
                                 "what": "pipelined: the gather of pass i overlaps the fit of pass i+1; single job: nothing overlapped"}
        if fa2 is not None:
            s2 = fa2.submit(rows_d, te, fp, prior=False, norm=False, solver=solver)
            r2 = fa2.result(s2)
            torch.cuda.synchronize()
            ok2 = all(bool(torch.equal(r2[n], bufs[n][:n_job])) for n in ("t2", "k"))
            okt = torch.tensor([int(ok2)], device=c.dev, dtype=torch.int32)
            c.dist.all_reduce(okt, op=c.dist.ReduceOp.MIN)
            assert int(okt[0]) == 1, "fused gather of T2 / S0 differs"
            p2s = pick_passes(c, fused_pass_t2s0)
            t2s0_ms = time_steps(c, fused_pass_t2s0, args.steps, p2s) / (args.steps * p2s)
            extra["sharded_t2_s0_only"] = {"value": m_total / (t2s0_ms * 1e-3), "ms_per_pass": t2s0_ms,
                                           "gather_bytes_received_per_rank": int((c.world - 1) * L * 8),
                                           "what": "the same fused all-gather moving only the PARAMETER maps (T2 and S0, 8 B per voxel: the 'final "
                                                   "gather of the parameter maps' of BASELINE.json read literally); res and status stay with the slab's owner"}
            fa2.close()
        if fa is not None:
            extra["sharded"]["multicast"] = bool(fa.multicast)
            if fused_note:
                extra["sharded"]["multicast_note"] = fused_note
        if fa is None:
            extra["sharded"]["fused_unavailable"] = fused_err if not ok_f else "CUDA IPC failed on another rank"
        extra["replicas"] = {"value": sum_over_ranks(c, m) / (rep_ms * 1e-3), "ms_per_pass": rep_ms,
                             "what": "N independent dense-map passes (zero-fill + fit + scatter of one volume per rank), no gather -- round 1's value"}
        if fa is not None:
            fa.close()
    else:
        fit_ms = None

    # ---- sanity of the timed result + roofline numerators
    dense_pass()
    torch.cuda.synchronize()
    cnt = [int(v) for v in cnt_d.cpu()]
    nit = nit_d.cpu().numpy().astype(np.int64)
    status = st_d.cpu().numpy()
    n_failed = int((status != 0).sum())
    assert cnt[0] == 0 and cnt[3] == 0
    t2v = maps[0][idx_d].cpu().numpy()
    ok_v = status == 0
    assert np.isfinite(t2v).all() and t2v[ok_v].min() >= 10 - 1e-3 and t2v[ok_v].max() <= 2000 + 1e-3
    assert bool((maps[:, mask_d == 0] == 0).all()), "dense maps are not zero off-mask"
    if mono:
        assert n_failed <= 1e-5 * m, f"bench workload produced {n_failed} failed voxels"
    peaks = measured_peaks()
    info = t2.device_info()
    traffic = {}
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.isfile(tp):
        traffic = json.load(open(tp))
    per_fit = 4.0 * n_echo + 8 + 4 * (3 if mono else 4) + 1 + 4 + 4      # echoes + int64 index in; maps + status, nit, fun out
    step_bytes = float(m) * per_fit + float(n_vox) + 4.0 * (3 * (n_vox - m) + n_vox if mono else 4 * (n_vox - m))
    # the dense pass alone (at N > 1 the timed step is the sharded one; the replicas block has timed it)
    dense_ms = extra["replicas"]["ms_per_pass"] if c.world > 1 else pass_ms
    ach = step_bytes / (dense_ms * 1e-3) / 1e9
    kernel_name = ("fit_kernel<mono2,E=%d,AoS,FILL> (one launch per pass: fit + zero-fill of the dense maps)" % n_echo if fill_in_fit else
                   ((LB_KERNEL[solver] % fit) + " || zero_fill_kernel" if solver in LB_SOLVERS
                    else "floor_queue_kernel || zero_fill_kernel" if not mono else "fit_kernel || zero_fill_kernel"))
    roofline = {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"],
                "traffic": traffic.get("step_dram_bytes") if (args.config == "c2" and fill_in_fit) else None, "peak_src": peaks["src"],
                "kernel": kernel_name, "kernel_ms": dense_ms, "algorithmic_bytes": step_bytes,
                "bytes_per_fit": per_fit, "dense_map_bytes": step_bytes - float(m) * per_fit,
                # the same launch on SURVEY 8(d)'s per-fit accounting alone (4E + 4(P+1) + 1 bytes per masked voxel, without the
                # zero-fill of the dense maps and without index / nit / fun): what share of the HBM peak the FITS themselves use
                "per_fit_accounting": {"bytes_per_fit": 4.0 * n_echo + 4 * (3 if mono else 4) + 1,
                                       "achieved": float(m) * (4.0 * n_echo + 4 * (3 if mono else 4) + 1) / (dense_ms * 1e-3) / 1e9,
                                       "frac": float(m) * (4.0 * n_echo + 4 * (3 if mono else 4) + 1) / (dense_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]}}
    if solver == "lbfgsb":
        roofline["note"] = ("the L-BFGS-B kernel is bound by the latency of its own per-thread optimiser state (~7 KB / voxel in local "
                            "memory, DRAM-resident at 896 threads / SM), not by HBM bandwidth or a math pipe: frac is the "
                            "algorithmic-bytes figure the contract asks for, not a utilisation (DESIGN.md section 4)")
    if solver == "lbfgsb_dense":
        roofline["note"] = ("the dense L-BFGS-B kernel is not HBM-bound: ncu puts it at 33 % issue-active, FP64 pipe 20 %, 17 of 32 lanes "
                            "active (every lane is somewhere else in its optimiser), stalls = instruction fetch + dependent FP64 chains "
                            "+ the correction pairs in local memory; frac is the algorithmic-bytes figure the contract asks for, not "
                            "a utilisation (DESIGN.md section 4, profiles/r02_lbfgsb_dense_*)")
    roof_fp32 = None
    if mono and solver == "fast":
        wm = t2.work_model("gaussian", n_echo)
        o_fit = _abi.Outputs()
        o_fit.t2, o_fit.k, o_fit.sigma, o_fit.res = o.t2, o.k, None, o.res
        o_fit.fun, o_fit.nit, o_fit.status, o_fit.dense = o.fun, o.nit, o.status, 1
        o_fit.counts_dev = cnt_d.data_ptr()

        def plain_pass():
            lib.t2fit_run(C.byref(p), C.byref(o_fit), c.stream.cuda_stream)
        pp = pick_passes(c, plain_pass)
        plain_ms = time_steps(c, plain_pass, max(3, args.steps // 4), pp) / (max(3, args.steps // 4) * pp)
        flops = float((wm["flop_fixed"] + wm["flop_per_pass"] * nit).sum())
        mufu = float((wm["mufu_fixed"] + wm["mufu_per_pass"] * nit).sum())
        fp32_peak = info["sm_count"] * 128 * 2 * peaks["sm_max_mhz"] * 1e6 / 1e12
        mufu_peak = info["sm_count"] * 16 * peaks["sm_max_mhz"] * 1e6 / 1e12
        roof_fp32 = {"bound": "fp32", "achieved": flops / (plain_ms * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFLOP/s",
                     "frac": flops / (plain_ms * 1e-3) / 1e12 / fp32_peak, "kernel": "fit_kernel<mono2> alone (dense scatter, no zero-fill)",
                     "kernel_ms": plain_ms, "mufu_frac": mufu / (plain_ms * 1e-3) / 1e12 / mufu_peak,
                     "passes_per_voxel": float(nit.mean()), "flop_per_voxel": flops / m,
                     "hbm_gbs": float(m) * per_fit / (plain_ms * 1e-3) / 1e9}

    # ---- end to end through the public API with HOST buffers (numpy in, numpy out), every call: inputs from page-locked host
    # memory to the GPU, fit, results back into host arrays
    def time_e2e(a_flat, a_idx, want, steps, windows=3):
        t_w, n_w = time.perf_counter(), 0
        while n_w < 3 or time.perf_counter() - t_w < 0.5:
            r_ = t2.fit_voxels_batch(a_flat, a_idx, te, fit, fp, prior=False, norm=False, solver=solver, want=want)
            n_w += 1
        dts = []
        for _ in range(windows):
            barrier(c)
            t0_ = time.perf_counter()
            for _ in range(steps):
                r_ = t2.fit_voxels_batch(a_flat, a_idx, te, fit, fp, prior=False, norm=False, solver=solver, want=want)
                _ = float(r_.res[0])
            torch.cuda.synchronize()
            dts.append(max_over_ranks(c, time.perf_counter() - t0_)[0])
        return float(np.median(dts)), r_, dts

    e2e_steps = max(3, min(args.steps, 20)) if solver != "lbfgsb" else 2
    flat_p = t2.pinned_array(None, like=flat)
    idx32_p = t2.pinned_array(None, like=idx.astype(np.int32))
    n_out = 3 if mono else 4
    e2e_s, r, wins = time_e2e(flat_p, idx32_p, ("status",), e2e_steps)
    assert np.array_equal(r.t2, t2v), "e2e path and device path disagree"
    e2e = {"value": m_total * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(m * (n_echo * 4 + 4)),
           "d2h_bytes_per_step": int(m * (4 * n_out + 1)), "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
           "windows_ms_per_step": [round(1e3 * w / e2e_steps, 4) for w in wins],
           "path": "fit_voxels_batch(page-locked numpy [N,E], int32 mask_indices, want=('status',)) -> numpy t2, k, res"
                   + ("" if mono else ", sigma") + ", status: ONE kernel gathers the masked rows and the index vector straight from host "
                   "memory over PCIe and stores the results straight back into page-locked numpy arrays; a step here is ONE call"}
    idx_p = t2.pinned_array(None, like=idx)
    full_s, r, _ = time_e2e(flat_p, idx_p, ("nit", "fun", "status"), e2e_steps)
    e2e["all_outputs_int64_indices"] = {"value": m_total * e2e_steps / full_s, "ms_per_step": 1e3 * full_s / e2e_steps,
                                        "h2d_bytes_per_step": int(m * (n_echo * 4 + 8)), "d2h_bytes_per_step": int(m * (4 * n_out + 4 + 4 + 1)),
                                        "what": "everything fit_voxel returns per voxel (+ nit, fun), np.where's int64 indices -- round 1's e2e"}
    pg_s, r, _ = time_e2e(flat, idx, ("nit", "fun", "status"), e2e_steps)
    e2e["pageable_input"] = {"value": m_total * e2e_steps / pg_s, "ms_per_step": 1e3 * pg_s / e2e_steps}
    if c.world > 1:
        # strong-scaled single volume: every rank reads 1/N of the masked rows of volume 0 from its own host copy
        flat0, idx0, _ = make_volume_workload(args.config, 0)
        f0p = t2.pinned_array(None, like=flat0)
        a0, b0 = D.slab_bounds(idx0.size, c.world)[c.rank]
        i0p = t2.pinned_array(None, like=idx0[a0:b0].astype(np.int32))
        s_s, _, _ = time_e2e(f0p, i0p, ("status",), e2e_steps)
        e2e["strong_single_volume"] = {"value": idx0.size * e2e_steps / s_s, "ms_per_volume": 1e3 * s_s / e2e_steps,
                                       "what": "ONE volume, each rank fits 1/N of its masked rows from host memory (results stay in each rank's host arrays)"}
        del f0p, flat0
    del flat_p

    # ---- the other solver on the same device-resident workload (secondary, outside the timed region)
    other, others = None, []
    if not args.no_secondary and c.rank == 0:
        for oth in [s_ for s_ in ("lbfgsb_dense", "lbfgsb", "fast") if s_ != solver and not (s_ == "fast" and fit == "rician")]:
            try:
                best = 1e30
                for _ in range(2):
                    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    g0.record(c.stream)
                    ro = t2.fit_voxels_batch(y_d, idx_d, te, fit, fp, prior=False, norm=False, solver=oth, check_bounds=False)
                    g1.record(c.stream)
                    torch.cuda.synchronize()
                    best = min(best, g0.elapsed_time(g1))
                t2o = ro.t2.cpu().numpy()
                others.append({"solver": oth, "fits_per_s": m / (best * 1e-3), "ms_per_volume": best, "mean_nit": float(ro.nit.float().mean()),
                               "success": float((ro.status == 0).float().mean()),
                               "t2_within_1e-3_of_default_solver": float(np.mean(np.abs(t2o - t2v) <= 1e-3 * np.abs(t2v))),
                               "what": LB_WHAT.get(oth, "float32 Newton / LM" + (" multi-start: the bounded minimiser, NOT the reference's loosely converged point" if fit != "gaussian" else ": the bounded minimiser"))})
            except Exception as ex:
                others.append({"solver": oth, "error": repr(ex)})
        other = others[0] if others else None

    parity = None
    if cpu is not None:
        try:
            parity = parity_block(c, cfg, cpu[1], cpu[2], cpu[3], solver)
        except Exception as ex:
            parity = {"error": repr(ex)}

    if c.rank == 0:
        launches = 1 if fill_in_fit else 2
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": c.world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if solver == "fast" else "f64", "data": "synthetic",
                "config": {"workload": cfg["workload"], "solver": solver, "passes_per_step": passes, "ms_per_pass": pass_ms,
                           "masked_voxels_per_gpu": int(m_s if c.world > 1 else m), "failed_voxels": n_failed, "volume_voxels_per_gpu": int(n_vox), "n_echo": int(n_echo),
                           "l2": "inputs + outputs of a pass (%.0f MB) exceed the 126 MB L2" % ((flat.nbytes + 16.0 * n_vox) / 1e6),
                           "timed_region_s": elapsed_ms * 1e-3,
                           "step": ("%d back-to-back passes; a pass = " % passes) + (
                               "ONE job of %d slabs: fit of the rank's slab + all-gather of the result vectors to every rank (see `sharded.form`)" % c.world if c.world > 1 else
                               "zero the four dense maps + fit + residuals + scatter of one volume"),
                           "scale": SCALE},
                "roofline": roofline, "roofline_fp32": roof_fp32, "cpu_baseline": cpu[0] if cpu else None, "parity": parity,
                "other_solver": other, "other_solvers": others, "e2e": e2e, "gpu_launches": int(args.steps * passes * (launches if c.world == 1 else 1)),
                "clocks": clocks, "device": info["name"]}
        line.update(extra)
        print(json.dumps(line), flush=True)
    if c.world > 1:
        c.dist.destroy_process_group()
    del keep


def bench_series(args, cfg):
    """c4: a batch of volumes through t2map_series from host arrays; volume v goes to rank v % world."""
    cpu = cpu_leg(args, cfg) if (int(os.environ.get("RANK", "0")) == 0 and int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_cpu_baseline) else None
    c = gpu_setup(args)
    torch, t2 = c.torch, c.t2
    from fetal_t2mapping_b200 import synth
    n_vol = int(os.environ.get("T2FIT_BENCH_C4_VOLUMES", "64"))
    _, fp = t2.preset("gaussian", True)
    mine, te = [], None
    distinct = {}
    for v in range(c.rank, n_vol, c.world):
        key = v % 8                                             # 8 distinct synthetic volumes, reused (host memory)
        if key not in distinct:
            y, mask, te, _ = synth.make_volume("c4", scale=SCALE, volume_index=key)
            distinct[key] = ([np.ascontiguousarray(y[..., e]) for e in range(y.shape[-1])], [mask.astype(np.uint8)] * y.shape[-1], int(mask.sum()))
        mine.append(distinct[key])
    if te is None:
        te = synth.make_volume("c4", scale=0.1)[2]
    m_local = sum(v[2] for v in mine)
    vols = [(v[0], v[1]) for v in mine]

    def one_pass():
        acc = 0.0
        for mp in t2.t2map_series(vols, te, "gaussian", fp, prior=False, depth=3, route=os.environ.get("T2FIT_BENCH_C4_ROUTE", "auto")):
            acc += float(mp.t2[mp.t2.shape[0] // 2, 0, 0])       # consume the maps as process_t2maps does, then drop them
        return acc
    sampler = ClockSampler(c.local) if c.rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(3, args.warmup)):
        one_pass()
    barrier(c)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        one_pass()
    torch.cuda.synchronize()
    dt = max_over_ranks(c, time.perf_counter() - t0)[0]
    clocks = sampler.stop() if sampler else None
    m_total = sum_over_ranks(c, m_local)
    value = m_total * args.steps / dt
    n_vox = int(np.prod(vols[0][0][0].shape)) if vols else 0
    n_echo = len(te)
    peaks = measured_peaks()
    # device part of one volume (PLANES layout, dense maps + fused fill), events around it
    dev_ms = None
    if vols:
        planes = torch.stack([torch.from_numpy(a.reshape(-1)) for a in vols[0][0]]).to(c.dev)
        mk = torch.from_numpy(vols[0][1][0].reshape(-1)).to(c.dev)
        idx = t2.mask_indices_device(mk.reshape(vols[0][0][0].shape))
        import ctypes as C
        from fetal_t2mapping_b200 import _abi
        from fetal_t2mapping_b200.api import _fill_problem
        p, o = _abi.Problem(), _abi.Outputs()
        keep = _fill_problem(p, "gaussian", fp, te, False, False, 0, 0.0, "auto", "fast")
        maps = torch.empty((4, n_vox), dtype=torch.float32, device=c.dev)
        st = torch.empty(idx.numel(), dtype=torch.uint8, device=c.dev)
        cnt = torch.zeros(4, dtype=torch.int64, device=c.dev)
        p.echoes, p.memory, p.layout, p.ld, p.mask_idx = planes.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_PLANES, n_vox, idx.data_ptr()
        p.n_vox, p.n_fit = n_vox, idx.numel()
        o.t2, o.k, o.sigma, o.res = (maps[i].data_ptr() for i in range(4))
        o.status, o.dense, o.zero_fill_mask, o.counts_dev = st.data_ptr(), 1, mk.data_ptr(), cnt.data_ptr()

        def dev_pass():
            c.lib.t2fit_run(C.byref(p), C.byref(o), c.stream.cuda_stream)
        pp = pick_passes(c, dev_pass)
        dev_ms = time_steps(c, dev_pass, 3, pp) / (3 * pp)
        mv = idx.numel()
        step_bytes = mv * (4.0 * n_echo + 8 + 12 + 1) + n_vox + 4.0 * (3 * (n_vox - mv) + n_vox)
        del keep
    if c.rank == 0:
        ach = step_bytes / (dev_ms * 1e-3) / 1e9 if dev_ms else None
        h2d = sum(a.nbytes for a in vols[0][0]) + sum(a.nbytes for a in vols[0][1]) if vols else 0
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": c.world, "steps": args.steps, "warmup": max(3, args.warmup),
                "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": cfg["workload"], "solver": "fast", "volumes": n_vol, "volumes_per_rank": len(vols),
                           "masked_voxels_total": m_total, "volume_voxels": n_vox, "n_echo": n_echo, "timed_region_s": dt, "scale": SCALE,
                           "step": "the whole batch once: per volume cast into page-locked planes, H2D, mask union + indices, fit into "
                                   "zero-filled dense maps, D2H of the four maps (t2map_series, 3 volumes in flight)",
                           "ms_per_volume": 1e3 * dt / args.steps / max(1, len(vols))},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"] if ach else None,
                             "traffic": None, "kernel": "fit_kernel<mono2,E=%d,PLANES,FILL> (device part of one volume)" % n_echo, "kernel_ms": dev_ms,
                             "note": "the series is bound by the host side (cast into pinned planes) and PCIe, not by this kernel"},
                "cpu_baseline": cpu[0] if cpu else None,
                "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": int(h2d * len(vols)), "d2h_bytes_per_step": int((16 + 1) * n_vox * len(vols)),
                        "path": "t2map_series IS the end-to-end path: host arrays in, host maps out"},
                "gpu_launches": int(args.steps * len(vols) * 5), "clocks": clocks, "device": t2.device_info()["name"]}
        print(json.dumps(line), flush=True)
    if c.world > 1:
        c.dist.destroy_process_group()


def bench_slab(args, cfg):
    """c5: ONE unmasked volume strong-scaled over contiguous slabs, all-gather of the T2 / S0 vectors inside the step."""
    cpu = cpu_leg(args, cfg) if (int(os.environ.get("RANK", "0")) == 0 and int(os.environ.get("WORLD_SIZE", "1")) == 1 and not args.no_cpu_baseline) else None
    c = gpu_setup(args)
    torch, t2 = c.torch, c.t2
    from fetal_t2mapping_b200 import distributed as D
    from fetal_t2mapping_b200.api import fit_voxels_into
    side = max(16, int(round(512 * SCALE)))
    n = side ** 3
    fit = cfg["fit"]
    solver = cfg["solver"] if args.solver == "auto" else args.solver
    _, fp = t2.preset(fit, True)
    te = c5_te()
    L = D.slab_length(n, c.world)
    a, b = D.slab_bounds(n, c.world)[c.rank]
    rows = c5_rows_device(torch, c.dev, a, b - a, n)
    names = ["t2", "k"]                                            # "NCCL gather of T2/S0 maps" (BASELINE config 5)
    bufs = {k: torch.zeros(c.world * L, dtype=torch.float32, device=c.dev) for k in names}
    mine = {k: bufs[k][c.rank * L:(c.rank + 1) * L] for k in names}
    loc = {k: torch.empty(max(b - a, 1), dtype=torch.float32 if k != "status" else torch.uint8, device=c.dev) for k in ("sigma", "res", "status")}
    outp = {"t2": mine["t2"].data_ptr(), "k": mine["k"].data_ptr(), "sigma": loc["sigma"].data_ptr(), "res": loc["res"].data_ptr(),
            "status": loc["status"].data_ptr()}
    cnt = torch.zeros(4, dtype=torch.int64, device=c.dev)

    def fit_pass():
        fit_voxels_into(rows, None, te, fit, fp, False, False, outp, solver=solver, counts=cnt)

    def one_pass():
        fit_pass()
        if c.world > 1:
            for k in names:
                c.dist.all_gather_into_tensor(bufs[k], mine[k])
    sampler = ClockSampler(c.local) if c.rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(max(1, min(3, args.warmup))):
        one_pass()
    elapsed_ms = time_steps(c, one_pass, args.steps, 1)
    clocks = sampler.stop() if sampler else None
    fit_ms = time_steps(c, fit_pass, max(1, args.steps // 2), 1) / max(1, args.steps // 2)
    value = n * args.steps / (elapsed_ms * 1e-3)
    ok = True
    if c.world > 1:
        tabs = torch.zeros((c.world, 2), dtype=torch.int64, device=c.dev)
        c.dist.all_gather_into_tensor(tabs, slab_hashes(torch, [mine[k] for k in names], [(0, b - a)])[0])
        got = slab_hashes(torch, [bufs[k] for k in names], D.slab_bounds(n, c.world))
        ok = bool(torch.equal(tabs, got))
        assert ok, "gathered T2 / S0 differ from what the owners computed"
    status = loc["status"][:b - a]
    failed = sum_over_ranks(c, int((status != 0).sum()))
    peaks = measured_peaks()
    per_fit = 4.0 * 16 + 4 * 4 + 1
    if c.rank == 0:
        ach = (b - a) * per_fit / (fit_ms * 1e-3) / 1e9
        step_ms = elapsed_ms / args.steps
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": c.world, "steps": args.steps, "warmup": max(1, min(3, args.warmup)),
                "ms_per_step": step_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32" if solver == "fast" else "f64", "data": "synthetic (generated on the device)",
                "config": {"workload": cfg["workload"], "solver": solver, "voxels": n, "voxels_per_rank": b - a, "n_echo": 16, "scale": SCALE,
                           "failed_voxels": failed, "timed_region_s": elapsed_ms * 1e-3,
                           "step": "fit of the rank's contiguous slab + in-place NCCL all-gather of the T2 and S0 vectors (every rank ends with both full maps)"},
                "sharded": {"fit_ms": fit_ms, "gather_ms": step_ms - fit_ms, "gather_bytes_received_per_rank": int((c.world - 1) * L * 8),
                            "gathered_equals_owner": ok},
                "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": ach / peaks["hbm_gbs"], "traffic": None,
                             "kernel": (LB_KERNEL[solver] % "gaussian_rician" if solver in LB_SOLVERS else "floor_queue_kernel<16,AoS> (multi-start)"),
                             "kernel_ms": fit_ms, "bytes_per_fit": per_fit,
                             "note": "not HBM-bound: instruction issue at 17 of 32 active lanes, FP64 pipe 20 % (lbfgsb_dense) / latency of the per-thread optimiser state (lbfgsb) / issue slots (fast); see DESIGN.md section 4"},
                "cpu_baseline": cpu[0] if cpu else None, "parity": None,
                "e2e": None, "gpu_launches": int(args.steps), "clocks": clocks, "device": t2.device_info()["name"]}
        if cpu is not None:
            try:
                line["parity"] = parity_block(c, cfg, cpu[1], cpu[2], cpu[3], solver)
            except Exception as ex:
                line["parity"] = {"error": repr(ex)}
        # end to end: a 2^20-voxel host slab of the same distribution through the public API
        try:
            hr = t2.pinned_array(None, like=c5_rows_host(1 << 20, seed=9))
            best = 1e30
            for _ in range(3):
                t0 = time.perf_counter()
                r = t2.fit_voxels_batch(hr, None, te, fit, fp, prior=False, norm=False, solver=solver, want=("status",))
                _ = float(r.res[0])
                best = min(best, time.perf_counter() - t0)
            line["e2e"] = {"value": (1 << 20) / best, "unit": UNIT, "h2d_bytes_per_step": int((1 << 20) * 64), "d2h_bytes_per_step": int((1 << 20) * 17),
                           "what": "one call on a 2^20-voxel host slab (page-locked), one GPU"}
        except Exception as ex:
            line["e2e"] = {"error": repr(ex)}
        print(json.dumps(line), flush=True)
    if c.world > 1:
        c.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--solver", default="auto", choices=["auto", "fast", "lbfgsb", "lbfgsb_dense"])
    ap.add_argument("--no-cpu-baseline", dest="no_cpu_baseline", action="store_true")
    ap.add_argument("--no-secondary", dest="no_secondary", action="store_true")
    ap.add_argument("--no-lbfgsb", dest="no_secondary", action="store_true")      # round-1 name of --no-secondary
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed pass as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or CONFIGS[args.config]["kind"] != "volume" or args.gpus != 1):
        ap.error("--dump-outputs is available for the volume configurations (c1, c2, c3) of the CUDA arm on one GPU")
    if args.impl == "reference":
        run_reference(args)
        return
    cfg = CONFIGS[args.config]
    {"volume": bench_volume, "series": bench_series, "slab": bench_slab}[cfg["kind"]](args, cfg)


if __name__ == "__main__":
    main()
