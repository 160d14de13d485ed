"""Parity of the HEADLINE configuration (VERDICT r01 item 1): bench.py's exact workload -- synth.make_cloud('sphere', 10000,
seed=0), the bench's calibrated checkpoint, precision 'tc' with the default guard band 0.05, default batch 8192 -- through the
fused pipeline `Engine.reconstruct`, compared with the CPU oracle (fp32 torch-CPU network on cKDTree patches) on a strided
sample of queries, with the GPU's own sub-sample ids (the Philox stream is a different stream than MT19937 by design).

Stated bars
  * sign class: identical to the fp32 oracle on every sampled query whose oracle |sign logit| exceeds 2e-3 (the agreement
    bar between two fp32 implementations, tests/test_gpu_parity.py) -- inside and outside the guard band;
  * |d SDF|: stated in VOXELS of the grid (voxel = 2 / res).  The tensor-core path uses fp16 operands (11-bit significand)
    with fp32 accumulation; the reference's own stock GPU path is cuDNN Conv1d with TF32 operands (same significand).  The
    bar is therefore expressed against the oracle with TF32-rounded conv operands (`conv_tf32=True`): the engine's maximum
    deviation from the fp32 oracle must stay within MAX_VOXELS[res] and within 2x the TF32 reference's own maximum deviation
    measured on the same queries (+0.02 voxel).
"""
import os
import sys

import numpy as np
import pytest
import torch

from oracle import p2s_oracle as orc
from points2surf_b200 import synth, ops

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
SEED = 40938661          # bench.py --seed default
FP32_AMBIGUOUS = 2e-3    # |sign logit| below which two fp32 implementations may disagree on the sign
MAX_VOXELS = {128: 0.4, 256: 0.6}   # max |d SDF| of the tc engine vs the fp32 oracle, in voxels (measured: see DESIGN.md section 2)


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def bench_engine(variant, **kw):
    """The checkpoint bench.py times: make_workload's seeds + the GPU-calibrated output bias."""
    v = synth.VARIANTS[variant]
    sd = synth.make_state_dict(variant, 6 if variant == 'vanilla' else 4)
    bench.calibrate_output_bias(sd, variant, 0)
    return sd, ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], precision='tc', guard_band=0.05, **kw)


def oracle_sdf(sd, variant, cloud, qpts, sub_ids, conv_tf32=False, chunk=256):
    v = synth.VARIANTS[variant]
    kd = orc.make_kdtree(cloud)
    logits = np.empty((len(qpts), 2), np.float32)
    radius = np.empty((len(qpts),), np.float32)
    for b in range(0, len(qpts), chunk):
        pr = [orc.knn_patch(cloud, kd, q, 300)[1:] for q in qpts[b:b + chunk]]
        radius[b:b + chunk] = [r for _, r in pr]
        logits[b:b + chunk] = orc.model_forward(sd, np.stack([p for p, _ in pr]), cloud[sub_ids[b:b + chunk]], qpts[b:b + chunk],
                                                v['use_point_stn'], v['shared_transformer'], conv_tf32=conv_tf32)
    return logits, orc.post_process(logits, radius)


def check_against_oracle(tag, sd, variant, cloud, res, lin, sdf, first, sel, n_tf32):
    v = synth.VARIANTS[variant]
    pts = cu(cloud)
    voxel = 2.0 / res
    qpts_dev = ops.query_points(lin, res)
    qpts = qpts_dev.cpu().numpy()
    # the fused pipeline's query set is the oracle's (bit-exact), in np.nonzero order
    assert np.array_equal(qpts[sel], orc.query_grid(cloud, res, 3)[first + sel])
    ids = np.empty((len(sel), 1000), np.int32)
    for j, i in enumerate(sel):
        ids[j] = ops.subsample(pts, qpts_dev[i:i + 1], 1000, bool(v['uniform_subsample']), SEED, query_index_base=first + int(i)).cpu().numpy()[0]
    logits_o, sdf_o = oracle_sdf(sd, variant, cloud, qpts[sel], ids)
    got = sdf.cpu().numpy()[sel]
    decided = np.abs(logits_o[:, 1]) > FP32_AMBIGUOUS
    mism = int(((got >= 0) != (sdf_o >= 0))[decided].sum())
    in_band = np.abs(logits_o[:, 1]) < 0.05
    dv = np.abs(np.abs(got) - np.abs(sdf_o)) / voxel
    print('%s: %d queries sampled, %d inside the guard band, %d fp32-ambiguous, sign mismatches %d; |dSDF| max %.4f mean %.5f voxel'
          % (tag, len(sel), int(in_band.sum()), int((~decided).sum()), mism, dv.max(), dv.mean()))
    assert mism == 0
    assert (got[~decided] != 0).all()                      # ambiguous ones still carry a sign
    assert dv.max() <= MAX_VOXELS[res], dv.max()
    if n_tf32:
        _, sdf_t = oracle_sdf(sd, variant, cloud, qpts[sel[:n_tf32]], ids[:n_tf32], conv_tf32=True)
        dt = np.abs(np.abs(sdf_t) - np.abs(sdf_o[:n_tf32])) / voxel
        de = dv[:n_tf32]
        print('%s: on %d queries -- tc engine |dSDF| max %.4f mean %.5f voxel; TF32-conv reference (stock cuDNN arithmetic) max %.4f mean %.5f voxel'
              % (tag, n_tf32, de.max(), de.mean(), dt.max(), dt.mean()))
        assert de.max() <= 2.0 * dt.max() + 0.02, (de.max(), dt.max())
        assert de.mean() <= 2.0 * dt.mean() + 0.002, (de.mean(), dt.mean())
    return mism, float(dv.max())


def test_headline_vanilla_res128_all_queries():
    """BASELINE configs[1] literally: vanilla, 10k-pt cloud, grid_res 128, every query on the GPU; 4096 checked on the CPU."""
    cloud = synth.make_cloud('sphere', 10000, seed=0)
    sd, eng = bench_engine('vanilla')
    lin, sdf = eng.reconstruct(cu(cloud), 128, 3, 0, SEED)
    Q = lin.numel()
    assert Q > 5 * 8192                                       # several default batches
    n_guard = eng.last_guard_count()
    print('res 128: Q = %d, guard-band recompute %d queries (%.2f %%)' % (Q, n_guard, 100.0 * n_guard / Q))
    sel = np.linspace(0, Q - 1, 4096).astype(np.int64)
    check_against_oracle('vanilla res128', sd, 'vanilla', cloud, 128, lin, sdf, 0, sel, n_tf32=512)
    # a batch > 8192 crosses the chunk loop of forward_tc_core; results do not depend on the batch partition
    lin2, sdf2 = eng.reconstruct(cu(cloud), 128, 3, 0, SEED, batch=20000)
    assert torch.equal(lin, lin2)
    a, b = sdf.cpu().numpy(), sdf2.cpu().numpy()
    assert np.array_equal(np.sign(a), np.sign(b))
    assert np.abs(a - b).max() <= 1e-6
    eng.close()


def test_guard_band_recomputes_every_query_over_several_batches():
    """A guard band wider than any |sign logit|: every batch flags all its queries into the slab-wide list (at the batch's
    offset), and all of them are recomputed in split precision, in batches of the same size.  The result must not depend on
    the batch size."""
    cloud = synth.make_cloud('sphere', 10000, seed=0)
    sd, eng = bench_engine('vanilla')
    eng.set_precision('tc', guard_band=1e9)
    lin, sdf = eng.reconstruct(cu(cloud), 128, 3, 0, SEED)
    Q = lin.numel()
    assert eng.last_guard_count() == Q
    lin2, sdf2 = eng.reconstruct(cu(cloud), 128, 3, 0, SEED, batch=3000)
    assert Q > 4 * 3000
    assert eng.last_guard_count() == Q
    assert torch.equal(lin, lin2)
    a, b = sdf.cpu().numpy(), sdf2.cpu().numpy()
    assert np.array_equal(np.sign(a), np.sign(b))
    assert np.abs(a - b).max() <= 1e-6
    eng.close()


def test_headline_vanilla_res256_slab():
    """The bench line's own resolution: a 20 000-query slab (three default batches) of the res-256 band."""
    cloud = synth.make_cloud('sphere', 10000, seed=0)
    sd, eng = bench_engine('vanilla')
    Qall = ops.query_grid(cu(cloud), 256, 3).numel()
    first = Qall // 3
    lin, sdf = eng.reconstruct(cu(cloud), 256, 3, 0, SEED, first_query=first, num_queries=20000)
    assert lin.numel() == 20000
    sel = np.linspace(0, 19999, 1024).astype(np.int64)
    check_against_oracle('vanilla res256 slab', sd, 'vanilla', cloud, 256, lin, sdf, first, sel, n_tf32=256)
    eng.close()


def test_headline_max_res128():
    cloud = synth.make_cloud('sphere', 10000, seed=0)
    sd, eng = bench_engine('max')
    lin, sdf = eng.reconstruct(cu(cloud), 128, 3, 1, SEED)
    sel = np.linspace(0, lin.numel() - 1, 1024).astype(np.int64)
    check_against_oracle('max res128', sd, 'max', cloud, 128, lin, sdf, 0, sel, n_tf32=256)
    eng.close()
