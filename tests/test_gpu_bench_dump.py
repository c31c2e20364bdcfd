"""bench.py --dump-outputs writes what the timed pass computed: on a small c1 volume (fewer masked voxels than the dump's
sample, so all of them) every array equals what fit_voxels_batch returns for the same seeded volume."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import ROOT

pytestmark = pytest.mark.gpu


def test_dump_outputs_equal_the_public_api(gpu_lib, tmp_path):
    torch = pytest.importorskip("torch")
    t2 = gpu_lib
    from fetal_t2mapping_b200 import synth
    out = tmp_path / "dump"
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", "c1", "--steps", "2",
                          "--warmup", "1", "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(out)],
                         cwd=tmp_path, env=dict(os.environ, T2FIT_BENCH_SCALE="0.25"), capture_output=True, text=True)
    assert run.returncode == 0, run.stderr[-3000:]
    got = {f[:-len(".npy")]: np.load(out / f) for f in os.listdir(out)}
    assert sorted(got) == ["fun", "k", "nit", "res", "sigma", "status", "t2", "voxel_index"]

    y, mask, te, _ = synth.make_volume("c1", scale=0.25)
    idx = np.flatnonzero(mask.reshape(-1))
    assert got["voxel_index"].dtype == np.float64 and np.array_equal(got["voxel_index"], idx)
    r = t2.fit_voxels_batch(torch.from_numpy(y.reshape(-1, te.size)).cuda(), torch.from_numpy(idx).cuda(), te, "gaussian",
                            t2.preset("gaussian", True)[1], prior=False, norm=False, solver="fast")
    torch.cuda.synchronize()
    for name in ("t2", "k", "sigma", "res", "fun", "nit", "status"):
        v = getattr(r, name)
        want = (v.cpu().numpy() if hasattr(v, "cpu") else np.asarray(v)).astype(np.float32)
        assert got[name].dtype == np.float32 and np.array_equal(got[name], want), name
