"""Cost of the standard-error pass (t2fit_stderr) against the fit pass of the same configuration, in one GPU run.

    python tools/bench_stderr.py [--out profiles/r03_bench_stderr.json] [--reps 20]

Configurations (device-resident inputs, the solvers bench.py uses for them):
    c2      256^3 x 5 TE adult brain, ~1.6 M masked voxels, gaussian, fast solver; dense [n_vox] maps in and out
    c3      160x256x256 x 12 TE NIST phantom, gaussian_rician, lbfgsb_dense solver; dense maps
    rician  a slab of 2^22 voxels x 16 TE (Rician data as c5), rician, lbfgsb_dense solver; compact outputs

Every timed pass is preceded by a 512 MB write that evicts the 126 MB L2, so each pass reads its inputs from HBM (the c2 and
c3 echo volumes are 335 / 252 MB; the rician slab 268 MB).  Times are CUDA events around single passes, median over --reps.
Work counted per voxel (see WORK below): algorithmic bytes 4E + 8P + index (echoes and parameters in, standard errors out)
and the FP64 operations of csrc/t2fit_stderr.cuh.  The card name and power limit are read in the same run.
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
from fetal_t2mapping_b200 import _abi, api, presets, synth             # noqa: E402
from bench_interval import Flush, card, time_pass                      # noqa: E402

HBM_PEAK = 7.7e12          # B/s, NVIDIA HGX B200 data sheet, one GPU
FP64_PEAK = 37e12          # FLOP/s FP64, the same data sheet (296 TFLOP/s for eight GPUs)

# FP64 work per echo of voxel_stderr, counted from csrc/t2fit_stderr.cuh (FMA = 2 FLOP; division, sqrt and exp counted as
# calls: each is a multi-instruction FP64 sequence on the device -- exp ~ 20 DFMA-class instructions, div / sqrt ~ 10).
#   gaussian:        m, J (3 MUL), J'J (3 FMA), residual (SUB + FMA)                              -> 12 FLOP, div 1, exp 1
#   gaussian_rician: k u^2, m (2 MUL + MUL + FMA), J (3 MUL), J'J (6 FMA), residual (SUB + FMA)   -> 23 FLOP, div 4, sqrt 1, exp 1
#   rician:          m, x, derivative terms (~40 FLOP), H (6 entries, ~20 FLOP), Bessel ratio: two Chebyshev series of
#                    25-30 terms (~3 FLOP per term)                                              -> ~230 FLOP, div 8, sqrt 0-2, exp 1
WORK = {"gaussian": dict(flop=12, div=1, sqrt=0, exp=1, P=2),
        "gaussian_rician": dict(flop=23, div=4, sqrt=1, exp=1, P=3),
        "rician": dict(flop=230, div=8, sqrt=1, exp=1, P=3)}
# per voxel after the echo loop: scaled Cholesky of a 2x2 / 3x3 matrix and the diagonal of its inverse
FIXED = {2: dict(flop=12, div=4, sqrt=4), 3: dict(flop=40, div=8, sqrt=6)}
CALL_FLOP = {"div": 10, "sqrt": 10, "exp": 20}          # FP64 instruction-equivalents of one call, for the FP64 roofline


def run_config(name, lib, flush, reps_fit, reps_se):
    dev = torch.device("cuda", 0)
    if name in ("c2", "c3"):
        y, mask, te, _ = synth.make_volume(name, scale=1.0)
        fit, solver = ("gaussian", "fast") if name == "c2" else ("gaussian_rician", "lbfgsb_dense")
        flat = torch.from_numpy(np.ascontiguousarray(y.reshape(-1, te.size))).to(dev)
        idx = torch.from_numpy(np.flatnonzero(mask.reshape(-1)).astype(np.int64)).to(dev)
        del y
        dense = 1
    else:
        fit, solver, dense = "rician", "lbfgsb_dense", 0
        n, te = 1 << 22, np.linspace(100.0, 700.0, 16)
        g = torch.Generator(device=dev).manual_seed(4)
        ted = torch.tensor(te, device=dev, dtype=torch.float32)
        t2v = torch.exp(torch.empty(n, device=dev).uniform_(np.log(30.0), np.log(300.0), generator=g))
        s0 = torch.empty(n, device=dev).uniform_(550.0, 900.0, generator=g)
        s = s0[:, None] * torch.exp(-ted[None, :] / t2v[:, None])
        flat = torch.sqrt((s + 20.0 * torch.randn((n, te.size), device=dev, generator=g)) ** 2 +
                          (20.0 * torch.randn((n, te.size), device=dev, generator=g)) ** 2).contiguous()
        del t2v, s0, s
        idx = None
    n_vox, E = flat.shape
    m = n_vox if idx is None else idx.numel()
    _, fp = presets.preset(fit, True)
    p, o = _abi.Problem(), _abi.Outputs()
    keep = api._fill_problem(p, fit, fp, te, False, False, 0, 0.0, "auto", solver)
    p.echoes, p.memory, p.layout, p.ld = flat.data_ptr(), _abi.MEM_DEVICE, _abi.LAYOUT_AOS, 0
    p.mask_idx = idx.data_ptr() if idx is not None else None
    p.n_vox, p.n_fit = n_vox, m
    size = n_vox if dense else m
    maps = torch.zeros((4, size), dtype=torch.float32, device=dev)
    se = torch.zeros((3, size), dtype=torch.float32, device=dev)
    status = torch.empty(m, dtype=torch.uint8, device=dev)
    cnt = torch.zeros(4, dtype=torch.int64, device=dev)
    o.t2, o.k, o.sigma, o.res = (maps[i].data_ptr() for i in range(4))
    if fit == "gaussian":
        o.sigma = None
    o.status, o.dense, o.counts_dev = status.data_ptr(), dense, cnt.data_ptr()
    stream = torch.cuda.current_stream(dev).cuda_stream

    def fit_pass():
        _abi.check(lib, lib.t2fit_run(C.byref(p), C.byref(o), stream), "t2fit_run")

    def se_pass():
        api._stderr_launch(lib, p, fit, [maps[1].data_ptr(), maps[0].data_ptr(), maps[2].data_ptr()], dense,
                           [se[1].data_ptr(), se[0].data_ptr(), se[2].data_ptr()], stream)
    fit_us, fit_all = time_pass(fit_pass, flush, reps_fit)
    se_us, se_all = time_pass(se_pass, flush, reps_se)
    sel = (idx if idx is not None else slice(None))
    se_t2 = se[0][sel] if dense else se[0]
    nan_share = float(torch.isnan(se_t2).float().mean())
    w = WORK[fit]
    P = w["P"]
    fx = FIXED[P]
    idx_bytes = 8 if idx is not None else 0
    bytes_pv = 4 * E + 8 * P + idx_bytes
    flop_pv = E * w["flop"] + fx["flop"]
    calls_pv = {k: E * w.get(k, 0) + fx.get(k, 0) for k in ("div", "sqrt", "exp")}
    eq_flop_pv = flop_pv + sum(CALL_FLOP[k] * v for k, v in calls_pv.items())
    t = se_us * 1e-6
    mem_frac = m * bytes_pv / t / HBM_PEAK
    fp_frac = m * eq_flop_pv / t / FP64_PEAK
    out = {"config": name, "fit": fit, "solver_of_fit_pass": solver, "n_vox": n_vox, "voxels": m, "n_echo": E, "dense": bool(dense),
           "fit_us_per_pass": fit_us, "stderr_us_per_pass": se_us, "stderr_over_fit": se_us / fit_us,
           "fit_voxels_per_s": m / (fit_us * 1e-6), "stderr_voxels_per_s": m / t,
           "bytes_per_voxel": bytes_pv, "hbm_bytes_per_s": m * bytes_pv / t, "hbm_fraction": mem_frac,
           "fp64_flop_per_voxel": flop_pv, "fp64_calls_per_voxel": calls_pv, "fp64_flop_equiv_per_voxel": eq_flop_pv,
           "fp64_fraction": fp_frac, "bound": "memory" if mem_frac >= fp_frac else "FP64 compute",
           "stderr_nan_share": nan_share, "fit_us_all": fit_all, "stderr_us_all": se_all}
    print(json.dumps({k: v for k, v in out.items() if not k.endswith("_all")}), flush=True)
    del keep
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--configs", default="c2,c3,rician")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_stderr needs a CUDA device")
    lib = t2.init(0)
    info = {"card": card(), "device": t2.device_info(), "hbm_peak_Bps": HBM_PEAK, "fp64_peak_flops": FP64_PEAK,
            "l2": "each timed pass follows a 512 MB write (L2 evicted)", "results": []}
    print(info["card"], flush=True)
    flush = Flush(torch.device("cuda", 0))
    for name in a.configs.split(","):
        info["results"].append(run_config(name, lib, flush, max(3, a.reps // 4) if name != "c2" else a.reps, a.reps))
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
