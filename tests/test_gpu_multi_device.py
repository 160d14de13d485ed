"""One thread, two devices: the library keeps its scratch, error flag, SM count and shared-memory limits per device
(DeviceCtx), so running every op and the engine on cuda:0, then cuda:1, then cuda:0 again gives the same results each time.
Skipped on machines with fewer than two CUDA devices."""
import numpy as np
import pytest
import torch

from points2surf_b200 import ops, synth
from points2surf_b200.train_ops import CudaPrims

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason='needs two CUDA devices')]
SEED = 40938661


def run_on(dev, cloud, sd, mats):
    v = synth.VARIANTS['vanilla']
    pts = torch.from_numpy(cloud).to(dev)
    out = {}
    lin = ops.query_grid(pts, 64, 3)
    q = ops.query_points(lin, 64)
    out['grid'] = lin
    out['knn_ids'], out['knn_patch'], out['knn_radius'] = ops.knn_patch(pts, q[:2048], 300)
    out['sub_ids'] = ops.subsample(pts, q[:512], 1000, False, SEED)     # weighted, 10 000 points: the cell kernel
    eng = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], device=torch.device(dev).index, precision='tc',
                     guard_band=0.05)
    out['rec_lin'], out['rec_sdf'] = eng.reconstruct(pts, 64, 3, v['uniform_subsample'], SEED, batch=4096)
    out['guard_count'] = torch.tensor(eng.last_guard_count())
    eng.close()
    out['vol'], iters = ops.sdf_to_volume(out['rec_lin'], out['rec_sdf'], 64, 5, 13.0)
    out['iters'] = torch.tensor(iters)
    out['verts'], out['faces'] = ops.marching_cubes(out['vol'])
    out['samples'] = ops.mesh_sample(out['verts'], out['faces'], 20000, seed=1)
    metric = ops.chamfer_hausdorff(out['samples'], pts)
    prims = CudaPrims()
    A, W, B = (torch.from_numpy(m).to(dev) for m in mats)
    out['gemm_nt'] = prims.gemm_nt(A, W)            # tensor-core kernel, no bias (the zero-bias scratch)
    gemm_tn = prims.gemm_tn(A, B)                   # tensor-core kernel
    return {k: t.cpu() for k, t in out.items()}, metric, gemm_tn.cpu()


def test_one_thread_alternating_devices():
    cloud = synth.make_cloud('sphere', 10000, seed=0)
    sd = synth.make_state_dict('vanilla', 6)
    rng = np.random.RandomState(3)
    mats = (rng.randn(8192, 256).astype(np.float32), rng.randn(512, 256).astype(np.float32),
            rng.randn(8192, 128).astype(np.float32))
    runs = [run_on(dev, cloud, sd, mats) for dev in ('cuda:0', 'cuda:1', 'cuda:0')]
    out0, metric0, tn0 = runs[0]
    assert out0['grid'].numel() > 4096 and out0['rec_lin'].numel() == out0['grid'].numel() and out0['faces'].numel() > 0
    for out, metric, tn in runs[1:]:
        for k in out0:
            assert torch.equal(out[k], out0[k]), k
        # the distance sums and the split-M weight-gradient tiles are accumulated with atomics: equal to round-off
        assert metric.keys() == metric0.keys()
        for k in metric0:
            assert metric[k] == pytest.approx(metric0[k], rel=1e-12), k
        assert torch.allclose(tn, tn0, rtol=1e-5, atol=1e-4)
