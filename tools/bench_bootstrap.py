"""Cost of the parametric bootstrap (DESIGN.md section 13) at B = 200 replicates per voxel, pass by pass, in one GPU run.

    python tools/bench_bootstrap.py [--out profiles/r05_bench_bootstrap.json] [--reps 3] [--n-rep 200]

Configurations (device-resident inputs, the solvers bench.py uses for them, --no_prior box):
    c2      256^3 x 5 TE adult brain, ~1.6 M masked voxels, gaussian, fast solver
    c3      160x256x256 x 12 TE NIST phantom, gaussian_rician, lbfgsb_dense solver
    rician  a slab of 2^20 voxels x 16 TE (Rician data as c5), rician, lbfgsb_dense solver

Every voxel's replicates are generated, refitted and summarised in one chunk (the buffers fit in HBM here), so the three
passes are timed on their own: t2fit_bootstrap_replicates (the generator), t2fit_run on the M * B replicate rows (the
refit), t2fit_bootstrap_stats.  Every timed pass is preceded by a 512 MB write that evicts the L2.  Times are CUDA events
around single passes, median over --reps (the refit of the L-BFGS-B configurations runs once).  The card name and power
limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import fetal_t2mapping_b200 as t2                                      # noqa: E402
from fetal_t2mapping_b200 import _abi, api, presets                    # noqa: E402
from bench_interval import Flush, card, time_pass                      # noqa: E402
from fetal_t2mapping_b200 import synth                                 # noqa: E402


def volume(name, dev):
    if name in ("c2", "c3"):
        y, mask, te, _ = synth.make_volume(name, scale=1.0)
        fit, solver = ("gaussian", "fast") if name == "c2" else ("gaussian_rician", "lbfgsb_dense")
        flat = torch.from_numpy(np.ascontiguousarray(y.reshape(-1, te.size))).to(dev)
        idx = torch.from_numpy(np.flatnonzero(mask.reshape(-1)).astype(np.int64)).to(dev)
        return fit, solver, te, flat, idx
    n, te = 1 << 20, np.linspace(100.0, 700.0, 16)
    g = torch.Generator(device=dev).manual_seed(4)
    ted = torch.tensor(te, device=dev, dtype=torch.float32)
    t2v = torch.exp(torch.empty(n, device=dev).uniform_(np.log(30.0), np.log(300.0), generator=g))
    s0 = torch.empty(n, device=dev).uniform_(550.0, 900.0, generator=g)
    s = s0[:, None] * torch.exp(-ted[None, :] / t2v[:, None])
    flat = torch.sqrt((s + 20.0 * torch.randn((n, te.size), device=dev, generator=g)) ** 2 +
                      (20.0 * torch.randn((n, te.size), device=dev, generator=g)) ** 2).contiguous()
    return "rician", "lbfgsb_dense", te, flat, None


def run_config(name, lib, flush, reps, B):
    dev = torch.device("cuda", 0)
    fit, solver, te, flat, idx = volume(name, dev)
    _, fp = presets.preset(fit, True)
    P = 2 if fit == "gaussian" else 3
    r = t2.fit_voxels_batch(flat, idx, te, fit, fp, prior=False, solver=solver)        # the maps being bootstrapped
    params = [r.k, r.t2, r.sigma if P == 3 else None]
    p = _abi.Problem()
    keep = [api._fill_problem(p, fit, fp, te, False, False, 0, 0.0, "auto", solver), api._device_rows(p, flat, idx)]
    m, E = p.n_fit, p.n_echo
    rows = torch.empty((m * B, E), dtype=torch.float32, device=dev)
    rep = torch.empty((P, m * B), dtype=torch.float32, device=dev)
    rst = torch.empty(m * B, dtype=torch.uint8, device=dev)
    outs = [torch.empty(3 * m, device=dev), torch.empty(3 * m, device=dev), torch.empty(m, device=dev), torch.empty(m, device=dev),
            torch.empty(m, dtype=torch.int32, device=dev), torch.empty(m, dtype=torch.int32, device=dev)]
    cnt = torch.zeros(4, dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    ptr = lambda t: t.data_ptr() if t is not None else None

    def gen():
        _abi.check(lib, lib.t2fit_bootstrap_replicates(C.byref(p), *[ptr(a) for a in params], None, None, 0, B,
                                                       rows.data_ptr(), stream), "t2fit_bootstrap_replicates")

    def refit():
        out = {"t2": rep[1].data_ptr(), "k": rep[0].data_ptr(), "sigma": rep[2].data_ptr() if P == 3 else None, "res": None,
               "status": rst.data_ptr()}
        api.fit_voxels_into(rows, None, te, fit, fp, False, False, out, solver=solver, counts=cnt)

    def stats():
        _abi.check(lib, lib.t2fit_bootstrap_stats(p.model, m, B, rep[0].data_ptr(), rep[1].data_ptr(),
                                                  rep[2].data_ptr() if P == 3 else None, rst.data_ptr(), 0.95,
                                                  *[o.data_ptr() for o in outs], stream), "t2fit_bootstrap_stats")
    gen_us, gen_all = time_pass(gen, flush, reps)
    fit_us, fit_all = time_pass(refit, flush, reps if solver == "fast" else 1)
    st_us, st_all = time_pass(stats, flush, reps)
    n_used = outs[4].cpu().numpy()
    sd_t2 = outs[1].view(3, m)[1].cpu().numpy()
    n_fits = m * B
    out = {"config": name, "fit": fit, "solver": solver, "voxels": m, "n_echo": E, "n_rep": B, "replicate_fits": n_fits,
           "replicate_row_bytes": n_fits * E * 4,
           "generator_us": gen_us, "refit_us": fit_us, "stats_us": st_us, "total_us": gen_us + fit_us + st_us,
           "generator_rows_per_s": n_fits / (gen_us * 1e-6), "generator_write_GBps": n_fits * E * 4 / (gen_us * 1e-6) / 1e9,
           "refit_fits_per_s": n_fits / (fit_us * 1e-6), "stats_voxels_per_s": m / (st_us * 1e-6),
           "n_used_share": float(n_used.sum() / n_fits), "t2_sd_finite_share": float(np.isfinite(sd_t2).mean()),
           "median_t2_sd_ms": float(np.nanmedian(sd_t2)),
           "generator_us_all": gen_all, "refit_us_all": fit_all, "stats_us_all": st_all}
    print(json.dumps({k: v for k, v in out.items() if not k.endswith("_all")}), flush=True)
    del keep, rows, rep, rst, outs, r, params, flat, idx
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--n-rep", type=int, default=200)
    ap.add_argument("--configs", default="c2,c3,rician")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_bootstrap needs a CUDA device")
    lib = t2.init(0)
    info = {"card": card(), "device": t2.device_info(),
            "l2": "each timed pass follows a 512 MB write (L2 evicted)", "results": []}
    print(info["card"], flush=True)
    flush = Flush(torch.device("cuda", 0))
    for name in a.configs.split(","):
        info["results"].append(run_config(name, lib, flush, a.reps, a.n_rep))
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
