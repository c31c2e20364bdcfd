"""Cost of the T2 interval pass (t2fit_t2_interval) against the fit pass of the same configuration, in one GPU run.

    python tools/bench_interval.py [--out profiles/r04_bench_interval.json] [--reps 5]

Configurations (device-resident inputs, the solvers bench.py uses for them):
    c2      256^3 x 5 TE adult brain, ~1.6 M masked voxels, gaussian, fast solver; dense [n_vox] maps
    c3      160x256x256 x 12 TE NIST phantom, gaussian_rician, lbfgsb_dense solver; dense maps
    rician  a slab of 2^20 voxels x 16 TE (Rician data as c5), rician, lbfgsb_dense solver; compact outputs

The interval pass runs at the default grid (G = 64) and level 0.95 on the --no_prior box, as the fit pass does.  Every timed
pass is preceded by a 512 MB write that evicts the 126 MB L2.  Times are CUDA events around single passes, median over
--reps.  The card name and power limit are read in the same run.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import fetal_t2mapping_b200 as t2                                      # noqa: E402
from fetal_t2mapping_b200 import _abi, api, presets, synth             # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


class Flush:
    def __init__(self, dev):
        self.buf = torch.empty(1 << 29, dtype=torch.uint8, device=dev)

    def __call__(self):
        self.buf.fill_(1)


def time_pass(fn, flush, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b) * 1e3)
    return float(np.median(ts)), [round(t, 1) for t in ts]


def run_config(name, lib, flush, reps_fit, reps_iv):
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
        n, te = 1 << 20, np.linspace(100.0, 700.0, 16)
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
    iv = torch.zeros((3, size), dtype=torch.float32, device=dev)
    ivf = torch.zeros(size, dtype=torch.uint8, device=dev)
    q = api._interval_q(fit, E, 0.95)
    status = torch.empty(m, dtype=torch.uint8, device=dev)
    cnt = torch.zeros(4, dtype=torch.int64, device=dev)
    o.t2, o.k, o.sigma, o.res = (maps[i].data_ptr() for i in range(4))
    if fit == "gaussian":
        o.sigma = None
    o.status, o.dense, o.counts_dev = status.data_ptr(), dense, cnt.data_ptr()
    stream = torch.cuda.current_stream(dev).cuda_stream

    def fit_pass():
        _abi.check(lib, lib.t2fit_run(C.byref(p), C.byref(o), stream), "t2fit_run")

    def iv_pass():
        api._interval_launch(lib, p, q, 64, dense, [iv[0].data_ptr(), iv[1].data_ptr(), iv[2].data_ptr(), ivf.data_ptr()],
                             None, stream)
    fit_us, fit_all = time_pass(fit_pass, flush, reps_fit)
    iv_us, iv_all = time_pass(iv_pass, flush, reps_iv)
    sel = (idx if idx is not None else slice(None))
    fl = (ivf[sel] if dense else ivf).cpu().numpy()
    lo, hi, best = ((iv[j][sel] if dense else iv[j]).cpu().numpy() for j in range(3))
    ok = (fl & 8) == 0
    out = {"config": name, "fit": fit, "solver_of_fit_pass": solver, "n_vox": n_vox, "voxels": m, "n_echo": E,
           "dense": bool(dense), "n_grid": 64, "level": 0.95,
           "fit_us_per_pass": fit_us, "interval_us_per_pass": iv_us, "interval_over_fit": iv_us / fit_us,
           "fit_voxels_per_s": m / (fit_us * 1e-6), "interval_voxels_per_s": m / (iv_us * 1e-6),
           "flag_share": {str(b): float(np.mean(fl & b != 0)) for b in (1, 2, 4, 8)},
           "median_width_ms": float(np.median(hi[ok] - lo[ok])) if ok.any() else None,
           "fit_us_all": fit_all, "interval_us_all": iv_all}
    print(json.dumps({k: v for k, v in out.items() if not k.endswith("_all")}), flush=True)
    del keep
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--configs", default="c2,c3,rician")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_interval needs a CUDA device")
    lib = t2.init(0)
    info = {"card": card(), "device": t2.device_info(),
            "l2": "each timed pass follows a 512 MB write (L2 evicted)", "results": []}
    print(info["card"], flush=True)
    flush = Flush(torch.device("cuda", 0))
    for name in a.configs.split(","):
        info["results"].append(run_config(name, lib, flush, a.reps, a.reps))
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
