"""GPU parity tests: the CUDA path, called through the C ABI (points2surf_b200.ops -> ctypes ->
libp2s_b200.so), against the oracle and the committed golden vectors.
Integer / index work must be bit-exact; floating point tolerances are stated per test."""
import numpy as np
import pytest
import torch

from oracle import p2s_oracle as orc
from points2surf_b200 import synth, ops
from helpers import load_golden, golden_model_case, calibrated_state_dict

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def make_engine(sd, variant, **kw):
    v = synth.VARIANTS[variant]
    return ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], **kw)


# ------------------------------------------------------------------ a7 / a8 : network
# fp32 path tolerance: |logit error| <= 2e-3 absolute on logits of magnitude O(1..30) (fp32 FMA with a
# different summation order than the CPU BLAS); sign class must be identical on the golden batch.
@pytest.mark.parametrize('variant', ['vanilla', 'max', 'uniform'])
def test_forward_fp32_matches_golden(variant):
    sd, inp, g = golden_model_case(variant)
    eng = make_engine(sd, variant)
    out = eng.forward(cu(inp['patch_pts_ps']), cu(inp['pts_sub_sample_ms']), cu(inp['imp_surf_query_point_ms'])).cpu().numpy()
    err = np.abs(out - g['logits']).max()
    assert err < 2e-3, err
    assert ((out[:, 1] >= 0) == (g['logits'][:, 1] >= 0)).all()
    # host-buffer entry point gives the same bits as the device entry point
    out_h = eng.forward_host(inp['patch_pts_ps'], inp['pts_sub_sample_ms'], inp['imp_surf_query_point_ms'])
    assert np.array_equal(out, out_h)
    sdf = ops.sdf_from_logits(cu(g['logits']), cu(g['radius'])).cpu().numpy()
    np.testing.assert_allclose(sdf, g['sdf'], rtol=2e-6, atol=1e-8)
    assert np.array_equal(np.sign(sdf), np.sign(g['sdf']))


def test_forward_fp32_ragged_batch_and_no_mutation():
    # batch sizes around the internal chunking (256) and a batch of 1; inputs must not be modified
    sd = calibrated_state_dict('vanilla', 21)
    eng = make_engine(sd, 'vanilla')
    inp = synth.make_model_inputs(300, seed=5)
    pa, su, qu = cu(inp['patch_pts_ps']), cu(inp['pts_sub_sample_ms']), cu(inp['imp_surf_query_point_ms'])
    su_before = su.clone()
    full = eng.forward(pa, su, qu)
    assert torch.equal(su, su_before)
    one = eng.forward(pa[257:258], su[257:258], qu[257:258])
    assert torch.allclose(full[257:258], one, atol=1e-4)
    ref = orc.model_forward(sd, inp['patch_pts_ps'][250:262], inp['pts_sub_sample_ms'][250:262],
                            inp['imp_surf_query_point_ms'][250:262], 1, 1)
    assert np.abs(full[250:262].cpu().numpy() - ref).max() < 2e-3
    assert eng.forward(pa[:0], su[:0], qu[:0]).shape == (0, 2)


def test_nan_logit_becomes_one():
    lg = cu(np.array([[np.nan, 1.0], [0.5, -1.0]], np.float32))
    sdf = ops.sdf_from_logits(lg, cu(np.array([0.1, 0.2], np.float32))).cpu().numpy()
    assert sdf[0] == 1.0 and sdf[1] < 0


# ------------------------------------------------------------------ a1 : candidate grid (bit-exact)
@pytest.mark.parametrize('kind,n,res,eps', [('sphere', 10000, 64, 3), ('torus', 4000, 48, 4), ('box', 3000, 40, 2),
                                            ('sphere', 2000, 32, 5), ('sphere', 300, 16, 1), ('box', 5000, 127, 3)])
def test_query_grid_bit_exact(kind, n, res, eps):
    cloud = synth.make_cloud(kind, n, seed=2)
    lin = ops.query_grid(cu(cloud), res, eps)
    idx = orc.query_grid_indices(cloud, res, eps)
    ref_lin = (idx[:, 0] * res + idx[:, 1]) * res + idx[:, 2]
    assert np.array_equal(lin.cpu().numpy().astype(np.int64), ref_lin)
    q = ops.query_points(lin, res).cpu().numpy()
    assert np.array_equal(q, orc.query_grid(cloud, res, eps))


def test_query_grid_golden_counts():
    g = load_golden('grid.npz')
    for name, kind, n, res, eps in (('sphere64e3', 'sphere', 10000, 64, 3), ('torus48e4', 'torus', 4000, 48, 4)):
        lin = ops.query_grid(cu(synth.make_cloud(kind, n, seed=2)), res, eps).cpu().numpy().astype(np.int64)
        assert len(lin) == int(g[name + '_count'])
        assert np.bitwise_xor.reduce(lin) == int(g[name + '_lin_xor'])


def test_query_grid_points_outside_cube_are_ignored():
    cloud = synth.make_cloud('sphere', 1000, seed=3)
    bad = np.concatenate([cloud, np.array([[1.5, 0, 0], [0, -1.2, 0], [0, 0, 1.0]], np.float32)])
    a = ops.query_grid(cu(cloud), 32, 3).cpu().numpy()
    b = ops.query_grid(cu(bad), 32, 3).cpu().numpy()
    assert np.array_equal(a, b)


# ------------------------------------------------------------------ a4 / a5 : kNN patch (bit-exact)
def test_knn_patch_golden():
    g = load_golden('assembly.npz')
    cloud, res, k = g['cloud'], int(g['res']), int(g['k'])
    qpts = orc.volume_space_to_model_space(g['query_idx'].astype(np.int64), res).astype(np.float32)
    ids, patch, radius = ops.knn_patch(cu(cloud), cu(qpts[:6]), k)
    assert np.array_equal(ids.cpu().numpy(), g['patch_ids'])          # same order as cKDTree (ascending distance)
    assert np.array_equal(radius.cpu().numpy(), g['radius'])
    assert np.array_equal(patch.cpu().numpy(), g['patch_ps'])


def test_knn_patch_vs_oracle_many_queries():
    cloud = synth.make_cloud('torus', 7000, seed=4)
    qpts = orc.query_grid(cloud, 32, 3)
    sel = np.random.RandomState(0).choice(len(qpts), 400, replace=False)
    q = qpts[sel]
    ids, patch, radius = ops.knn_patch(cu(cloud), cu(q), 300)
    ids, patch, radius = ids.cpu().numpy(), patch.cpu().numpy(), radius.cpu().numpy()
    kd = orc.make_kdtree(cloud)
    for i in range(len(q)):
        oid, ops_, orad = orc.knn_patch(cloud, kd, q[i], 300)
        _, d2 = orc.knn_bruteforce(cloud, q[i], 300)
        assert set(ids[i].tolist()) == set(oid.tolist())
        gd = ((cloud[ids[i]].astype(np.float64) - q[i].astype(np.float64)) ** 2).sum(1)
        assert np.array_equal(gd, d2)                   # ascending, identical float64 distances
        assert radius[i] == orad
        if np.all(np.diff(d2) > 0):                      # no exact ties -> order is unique
            assert np.array_equal(ids[i], oid)
            assert np.array_equal(patch[i], ops_)


def test_knn_small_k_and_duplicates():
    rng = np.random.RandomState(1)
    cloud = rng.uniform(-0.9, 0.9, (500, 3)).astype(np.float32)
    cloud[100:110] = cloud[100]                          # exact duplicates -> ties
    q = cloud[100:101] + np.float32(0.01)
    ids, patch, radius = ops.knn_patch(cu(cloud), cu(q), 8)
    bid, d2 = orc.knn_bruteforce(cloud, q[0], 8)
    gd = ((cloud[ids[0].cpu().numpy()].astype(np.float64) - q[0].astype(np.float64)) ** 2).sum(1)
    assert np.array_equal(gd, d2)
    with pytest.raises(ops.P2SError):
        ops.knn_patch(cu(cloud[:5]), cu(q), 8)           # N < k: the reference would index out of range


# ------------------------------------------------------------------ a6 : sub-sample
def test_subsample_uniform_properties():
    cloud = synth.make_cloud('sphere', 5000, seed=1)
    q = cu(orc.query_grid(cloud, 16, 3)[:64])
    a = ops.subsample(cu(cloud), q, 1000, True, seed=7).cpu().numpy()
    assert a.shape == (64, 1000) and a.min() >= 0 and a.max() < 5000
    # counter-based: independent of how the query list is split
    b = ops.subsample(cu(cloud), q[10:20], 1000, True, seed=7, query_index_base=10).cpu().numpy()
    assert np.array_equal(a[10:20], b)
    assert not np.array_equal(a, ops.subsample(cu(cloud), q, 1000, True, seed=8).cpu().numpy())
    # uniform over ids: chi-square-ish bound on bucket counts (64000 draws over 50 buckets)
    cnt = np.bincount(a.ravel() // 100, minlength=50)
    assert abs(cnt - 1280).max() < 6 * np.sqrt(1280)


def test_subsample_weighted_is_without_replacement_and_matches_reference_law():
    # inclusion frequencies of the GPU sampler vs RandomState.choice(replace=False, p) on a small cloud
    rng = np.random.RandomState(3)
    cloud = rng.uniform(-0.9, 0.9, (40, 3)).astype(np.float32)
    qp = np.array([[0.3, -0.2, 0.1]], np.float32)
    trials = 4000
    q = cu(np.repeat(qp, trials, axis=0))
    ids = ops.subsample(cu(cloud), q, 10, False, seed=11).cpu().numpy()
    assert all(len(set(r.tolist())) == 10 for r in ids)
    freq_gpu = np.bincount(ids.ravel(), minlength=40) / trials
    prob = orc.sub_sample_probabilities(cloud, qp[0])
    rs = np.random.RandomState(5)
    ref = np.stack([rs.choice(40, size=10, replace=False, p=prob) for _ in range(trials)])
    freq_ref = np.bincount(ref.ravel(), minlength=40) / trials
    # binomial std of an inclusion frequency ~ sqrt(.25*.75/4000) = 0.007; two estimates -> 5 sigma = 0.05
    assert np.abs(freq_gpu - freq_ref).max() < 0.05, np.abs(freq_gpu - freq_ref).max()
    # and the law is really non-uniform (near points favoured)
    near = np.argsort(np.linalg.norm(cloud - qp[0], axis=1))
    assert freq_gpu[near[:10]].mean() > freq_gpu[near[-10:]].mean() + 0.1


# The weighted sampler picks its kernel from the cloud size (N points, S drawn; the shared-memory cache holds 4 B per point,
# at most 160 KB): the cell index when N >= 2 S and N <= 40 960, the exponential clocks with the cache when N < 2 S and
# N <= 40 960, the clocks without the cache above 40 960 points.
@pytest.mark.parametrize('law,surface', [((40, 10), (10000, 1000)), ((40, 25), (1500, 1000)), (None, (50000, 1000))],
                         ids=['cells', 'clocks-cached', 'clocks-uncached'])
def test_subsample_weighted_kernels_realise_the_reference_law(law, surface):
    if law is not None:
        # law on a small cloud: inclusion frequencies vs RandomState.choice(replace=False, p)
        n, S = law
        rng = np.random.RandomState(3)
        cloud = rng.uniform(-0.9, 0.9, (n, 3)).astype(np.float32)
        qp = np.array([[0.3, -0.2, 0.1]], np.float32)
        trials = 4000
        ids = ops.subsample(cu(cloud), cu(np.repeat(qp, trials, axis=0)), S, False, seed=11).cpu().numpy()
        assert all(len(set(r.tolist())) == S for r in ids)
        freq = np.bincount(ids.ravel(), minlength=n) / trials
        prob = orc.sub_sample_probabilities(cloud, qp[0])
        rs = np.random.RandomState(5)
        ref = np.stack([rs.choice(n, size=S, replace=False, p=prob) for _ in range(trials)])
        dev_max = np.abs(freq - np.bincount(ref.ravel(), minlength=n) / trials).max()
        assert dev_max < 0.05, dev_max
        near = np.argsort(np.linalg.norm(cloud - qp[0], axis=1))
        assert freq[near[:10]].mean() > freq[near[-10:]].mean() + 0.1
    # a surface cloud: distinct ids in range, near points favoured, slabs reproduce the whole
    n, S = surface
    cloud = synth.make_cloud('sphere', n, seed=0)
    q = cloud[:64] * np.float32(0.97)
    a = ops.subsample(cu(cloud), cu(q), S, False, seed=7).cpu().numpy()
    assert a.min() >= 0 and a.max() < n and all(len(set(r.tolist())) == S for r in a)
    b = ops.subsample(cu(cloud), cu(q[10:20]), S, False, seed=7, query_index_base=10).cpu().numpy()
    assert np.array_equal(np.sort(a[10:20], axis=1), np.sort(b, axis=1))
    d = np.linalg.norm(cloud[a[0]] - q[0], axis=1)
    assert d.mean() < np.linalg.norm(cloud - q[0], axis=1).mean()


def test_subsample_requires_enough_points():
    cloud = synth.make_cloud('sphere', 100, seed=1)
    with pytest.raises(ops.P2SError):
        ops.subsample(cu(cloud), cu(cloud[:2]), 1000, True, seed=1)


# ------------------------------------------------------------------ a10 / a11 : volume (bit-exact)
@pytest.mark.parametrize('name', ['sphere', 'noisy'])
def test_sign_propagation_golden(name):
    g = load_golden('volume.npz')
    res = int(g[name + '_res'])
    idx = orc.model_space_to_volume_space(g[name + '_qpts'], res)
    lin = ((idx[:, 0] * res + idx[:, 1]) * res + idx[:, 2]).astype(np.int32)
    vol, iters = ops.sdf_to_volume(cu(lin), cu(g[name + '_dist']), res, 5, 13.0)
    ref = np.clip(g[name + '_vol'], -1.0, 1.0)
    assert np.array_equal(vol.cpu().numpy(), ref)
    assert iters == int(g[name + '_iters'])
    vol2, _ = ops.sdf_to_volume(cu(lin), cu(g[name + '_dist']), res, 3, 5.0)
    assert np.array_equal(vol2.cpu().numpy(), np.clip(g[name + '_vol_s3t5'], -1.0, 1.0))


# res % 4 == 0 and sigma <= 5 take the word-wide kernels, the rest the scalar ones
# res % 32 == 0 with sigma 5 takes the row-vector path (full tiles, 16-byte row loads, packed-byte votes)
@pytest.mark.parametrize('res,sigma,thr', [(24, 5, 13), (33, 4, 9), (48, 5, 26), (20, 2, 3), (36, 4, 9), (44, 7, 40), (64, 1, 1), (52, 3, 5),
                                           (32, 5, 13), (64, 5, 13), (64, 5, 0.5), (96, 5, 13), (128, 5, 13), (64, 5, 200)])
def test_sign_propagation_vs_oracle(res, sigma, thr):
    cloud = synth.make_cloud('torus', 4000, seed=9)
    qpts = orc.query_grid(cloud, res, 3)
    rng = np.random.RandomState(res)
    d = (rng.standard_normal(len(qpts)) * 0.05).astype(np.float32)
    d[np.linalg.norm(qpts, axis=1) < 0.4] *= np.sign(d[np.linalg.norm(qpts, axis=1) < 0.4])   # mostly + inside
    ref = orc.sdf_to_volume(d, qpts, res, sigma, thr)
    idx = orc.model_space_to_volume_space(qpts, res)
    lin = ((idx[:, 0] * res + idx[:, 1]) * res + idx[:, 2]).astype(np.int32)
    vol, _ = ops.sdf_to_volume(cu(lin), cu(d), res, sigma, float(thr))
    assert np.array_equal(vol.cpu().numpy().astype(np.float64), ref)


@pytest.mark.parametrize('res,noise,thr', [(32, 0.0, 13), (64, 0.0, 13), (64, 0.02, 13), (96, 0.01, 13), (128, 0.005, 13), (64, 0.0, 0.5), (64, 0.02, 20)])
def test_sign_propagation_row_vector_path_vs_oracle(res, noise, thr):
    # a real signed-distance band (sphere + noise): the fronts travel through the whole volume, volumes AND iteration counts
    # must equal the reference algorithm's
    cloud = synth.make_cloud('sphere', 6000, seed=4)
    qpts = orc.query_grid(cloud, res, 3)
    rng = np.random.RandomState(res + int(noise * 1000))
    r0 = float(np.linalg.norm(cloud, axis=1).mean())
    d = (np.linalg.norm(qpts, axis=1) - r0 + noise * rng.standard_normal(len(qpts))).astype(np.float32)
    vol_ref = orc.add_samples_to_volume(np.zeros((res,) * 3), qpts, d)
    vol_ref, it_ref = orc.propagate_sign(vol_ref, 5, thr)
    assert it_ref >= 3
    idx = orc.model_space_to_volume_space(qpts, res)
    lin = ((idx[:, 0] * res + idx[:, 1]) * res + idx[:, 2]).astype(np.int32)
    vol, iters = ops.sdf_to_volume(cu(lin), cu(d), res, 5, float(thr))
    assert iters == it_ref
    assert np.array_equal(vol.cpu().numpy().astype(np.float64), np.clip(vol_ref, -1.0, 1.0))


def test_all_zero_band_is_reported():
    lin = cu(np.arange(10, dtype=np.int32))
    vol, iters = ops.sdf_to_volume(lin, cu(np.zeros(10, np.float32)), 8, 5, 13.0)
    assert iters == -1


# ------------------------------------------------------------------ fused pipeline
@pytest.mark.parametrize('variant', ['vanilla', 'max'])
def test_reconstruct_matches_stagewise_oracle(variant):
    v = synth.VARIANTS[variant]
    sd = calibrated_state_dict(variant, 31)
    eng = make_engine(sd, variant)
    cloud = synth.make_cloud('sphere', 3000, seed=6)
    res, eps, seed = 16, 3, 1234
    lin, sdf = eng.reconstruct(cu(cloud), res, eps, v['uniform_subsample'], seed)
    idx = orc.query_grid_indices(cloud, res, eps)
    assert np.array_equal(lin.cpu().numpy().astype(np.int64), (idx[:, 0] * res + idx[:, 1]) * res + idx[:, 2])
    # replay a few queries on the CPU with the GPU's own sub-sample ids (RNG streams differ by design)
    qpts = orc.query_grid(cloud, res, eps)
    sel = [0, 1, len(qpts) // 2, len(qpts) - 1]
    sub_ids = ops.subsample(cu(cloud), cu(qpts), 1000, bool(v['uniform_subsample']), seed).cpu().numpy()
    kd = orc.make_kdtree(cloud)
    patches, radii = zip(*[(orc.knn_patch(cloud, kd, qpts[i], 300)[1:]) for i in sel])
    logits = orc.model_forward(sd, np.stack(patches), cloud[sub_ids[sel]], qpts[sel], v['use_point_stn'], v['shared_transformer'])
    ref = orc.post_process(logits, np.array(radii))
    got = sdf.cpu().numpy()[sel]
    np.testing.assert_allclose(got, ref, rtol=0, atol=2e-4)
    # slab sharding (multi-GPU tile mode) reproduces the same numbers
    lin2, sdf2 = eng.reconstruct(cu(cloud), res, eps, v['uniform_subsample'], seed, first_query=100, num_queries=50)
    assert torch.equal(lin2, lin[100:150]) and torch.allclose(sdf2, sdf[100:150], atol=1e-6)
    # host entry point
    lin3, sdf3 = eng.reconstruct_host(cloud, res, eps, v['uniform_subsample'], seed, cap=len(qpts))
    assert np.array_equal(lin3, lin.cpu().numpy()) and np.allclose(sdf3, sdf.cpu().numpy(), atol=1e-6)


# ------------------------------------------------------------------ a12 : marching cubes (oracle unpinned vs skimage)
# vertices: fp32 interpolation on both sides, tolerance 1e-6 absolute in model space; faces: identical indices.
@pytest.mark.parametrize('case', ['sphere', 'noise', 'propagated', 'all_cases'])
def test_marching_cubes_matches_oracle(case):
    from oracle import mc_oracle as mc
    from oracle import mc_topo
    if case == 'all_cases':
        # every corner-sign configuration with random magnitudes (ambiguous faces on both sides of the decider), exact zeros
        vol = mc_topo.all_cases_volume(0)
    elif case == 'sphere':
        R = 40
        g = (np.arange(R) + 0.5) / R * 2 - 1
        X, Y, Z = np.meshgrid(g, g, g, indexing='ij')
        vol = (0.55 - np.sqrt(X ** 2 + Y ** 2 + Z ** 2)).astype(np.float32)
    elif case == 'noise':
        rng = np.random.RandomState(0)
        vol = rng.standard_normal((19, 19, 19)).astype(np.float32)
        vol[[0, -1], :, :] = -1; vol[:, [0, -1], :] = -1; vol[:, :, [0, -1]] = -1
        vol[3, 3, 3] = 0; vol[5, 5, 5] = 0
    else:
        g = load_golden('volume.npz')
        vol = np.clip(g['noisy_vol'], -1, 1)
    v, f = ops.marching_cubes(cu(vol), 0.0)
    vo, fo = mc.marching_cubes(vol, 0.0)
    assert v.shape == vo.shape and f.shape == fo.shape
    assert np.array_equal(f.cpu().numpy(), fo)
    np.testing.assert_allclose(v.cpu().numpy(), vo, rtol=0, atol=1e-6)
    assert mc.mesh_is_closed(f.cpu().numpy())
    # the table-free second restatement (oracle/mc_topo.py: polygons traced on the cell values, asymptotic decider on
    # ambiguous faces) shares nothing with tools/gen_mc_tables.py: same vertices, same triangles
    vt, ft, st = mc_topo.marching_cubes(vol, 0.0, 'asymptotic', return_stats=True)
    assert np.array_equal(v.cpu().numpy(), vt) or np.abs(v.cpu().numpy() - vt).max() <= 1e-6
    assert np.array_equal(mc_topo.triangle_set(f.cpu().numpy()), mc_topo.triangle_set(ft))
    # and where the classic rule (always separate the positive corners) would have given another mesh
    vc, fc = mc_topo.marching_cubes(vol, 0.0, 'separate_positive')
    same = np.array_equal(mc_topo.triangle_set(fc), mc_topo.triangle_set(ft))
    print('%s: %d cells, %d with ambiguous faces, %d with more than one sheet; Euler characteristic asymptotic %d / classic %d; '
          'classic rule gives %s mesh' % (case, st['cells'], st['ambiguous_face_cells'], st['multi_sheet_cells'],
                                          mc_topo.euler_characteristic(len(vt), ft), mc_topo.euler_characteristic(len(vc), fc),
                                          'the same' if same else 'a different'))


def test_marching_cubes_empty_volume():
    v, f = ops.marching_cubes(cu(np.full((8, 8, 8), -1.0, np.float32)), 0.0)
    assert v.shape[0] == 0 and f.shape[0] == 0


def test_mesh_chamfer_against_analytic_sphere():
    # end of the chain on an analytic SDF band: scatter -> sign propagation -> MC; Chamfer (reference definition,
    # source/base/evaluation.py:222-256, 10k samples per side) to the true sphere below 1% of the diameter per sample
    res = 64
    cloud = synth.make_cloud('sphere', 10000, seed=0, noise=0.0)
    lin = ops.query_grid(cu(cloud), res, 3)
    q = ops.query_points(lin, res).cpu().numpy()
    d = (0.5 - np.linalg.norm(q, axis=1)).astype(np.float32)
    vol, iters = ops.sdf_to_volume(lin, cu(d), res, 5, 13.0)
    v, f = ops.marching_cubes(vol, 0.0)
    v, f = v.cpu().numpy(), f.cpu().numpy()
    rng = np.random.RandomState(0)
    s_mesh = orc.sample_mesh_surface(v, f, 10000, rng)
    dd = rng.standard_normal((10000, 3))
    s_ref = 0.5 * dd / np.linalg.norm(dd, axis=1, keepdims=True)
    assert orc.chamfer(s_mesh, s_ref) / 20000 < 0.01


# ------------------------------------------------------------------ a7 on the tensor-core path
# fp16 operands (11-bit significand, like the TF32 the reference's cuDNN convs use on Ampere+), fp32 accumulate.
# Tolerances (stated): max features within 2e-2 * max|feature| of the fp32 oracle; logits within
# 3e-2 * max(1, max|logit|); with the guard band on, the sign class is exact.
@pytest.mark.parametrize('variant', ['vanilla', 'max', 'uniform'])
def test_forward_tc_matches_oracle(variant):
    sd, inp, g = golden_model_case(variant)
    v = synth.VARIANTS[variant]
    eng = make_engine(sd, variant, precision='tc', guard_band=0.0)
    args = (cu(inp['patch_pts_ps']), cu(inp['pts_sub_sample_ms']), cu(inp['imp_surf_query_point_ms']))
    out, aux = eng.forward_with_aux(*args)
    # the aux tap observes the production head: the same logits, bit for bit, as a plain forward
    assert torch.equal(out, eng.forward(*args))
    ref, raux = orc.model_forward(sd, inp['patch_pts_ps'], inp['pts_sub_sample_ms'], inp['imp_surf_query_point_ms'],
                                  v['use_point_stn'], v['shared_transformer'], return_aux=True)
    if 'trans' in raux:
        terr = np.abs(aux['trans'].cpu().numpy() - raux['trans']).max()
        print('trans err', terr)
        assert terr < 2e-2
    for k in ('feat_global_max', 'feat_local_max'):
        a, r = aux[k].cpu().numpy(), raux[k]
        err = np.abs(a - r).max() / np.abs(r).max()
        print(variant, k, 'rel err', err)
        assert err < 2e-2, (k, err)
    out = out.cpu().numpy()
    err = np.abs(out - ref).max()
    print(variant, 'logit err', err, 'scale', np.abs(ref).max())
    assert err < 3e-2 * max(1.0, np.abs(ref).max()), err


def test_forward_tc_guard_band_makes_signs_exact():
    sd = calibrated_state_dict('vanilla', 21)
    inp = synth.make_model_inputs(200, seed=5)
    args = (cu(inp['patch_pts_ps']), cu(inp['pts_sub_sample_ms']), cu(inp['imp_surf_query_point_ms']))
    eng32 = make_engine(sd, 'vanilla', precision='fp32')
    ref = eng32.forward(*args).cpu().numpy()
    eng = make_engine(sd, 'vanilla', precision='tc', guard_band=0.0)
    raw = eng.forward(*args).cpu().numpy()
    err = np.abs(raw - ref).max()
    print('tc vs fp32 logit err', err, 'scale', np.abs(ref).max())
    band = max(4.0 * err, 1e-3)
    eng.set_precision('tc', guard_band=band)
    out = eng.forward(*args).cpu().numpy()
    n_guard = eng.last_guard_count()
    assert ((out[:, 1] >= 0) == (ref[:, 1] >= 0)).all()
    inside = np.abs(raw[:, 1]) < band
    assert n_guard == int(inside.sum())
    # recomputed queries come from the split-precision tensor-core path: fp32-level agreement with the fp32 FMA path
    assert np.abs(out[inside] - ref[inside]).max() < 2e-3 if inside.any() else True
    # ragged batch sizes through the tile scheduler (B not a multiple of the CTA count; B = 1)
    for B in (1, 3, 75, 149):
        o = eng.forward(args[0][:B], args[1][:B], args[2][:B]).cpu().numpy()
        assert np.abs(o - ref[:B]).max() < max(4.0 * err, 1e-3) + 1e-4


def test_reconstruct_tc_close_to_fp32():
    sd = calibrated_state_dict('vanilla', 31)
    cloud = synth.make_cloud('sphere', 3000, seed=6)
    e32 = make_engine(sd, 'vanilla', precision='fp32')
    etc = make_engine(sd, 'vanilla', precision='tc', guard_band=0.05)
    lin_a, sdf_a = e32.reconstruct(cu(cloud), 16, 3, 0, 99)
    lin_b, sdf_b = etc.reconstruct(cu(cloud), 16, 3, 0, 99)
    assert torch.equal(lin_a, lin_b)
    a, b = sdf_a.cpu().numpy(), sdf_b.cpu().numpy()
    assert np.array_equal(np.sign(a), np.sign(b))
    assert np.abs(a - b).max() < 1e-2   # |d| = tanh(l0)^2 r with r ~ 0.4: a logit error of 0.03 moves the SDF by < 1e-2


def test_subsample_weighted_large_cloud_uncached_path():
    # N * 4 B > 160 KB: the kernel recomputes the clocks per pass instead of caching them in shared memory
    rng = np.random.RandomState(2)
    cloud = rng.uniform(-0.9, 0.9, (50000, 3)).astype(np.float32)
    q = cu(cloud[:5] + np.float32(0.01))
    ids = ops.subsample(cu(cloud), q, 1000, False, seed=3).cpu().numpy()
    assert ids.min() >= 0 and ids.max() < 50000
    assert all(len(set(r.tolist())) == 1000 for r in ids)
    d = np.linalg.norm(cloud[ids[0]] - cloud[0], axis=1)
    assert d.mean() < np.linalg.norm(cloud - cloud[0], axis=1).mean()      # near points are favoured


@pytest.mark.parametrize('variant', ['vanilla', 'max', 'uniform'])
def test_split_precision_tensor_core_path_matches_fp32(variant):
    # a guard band wider than any logit sends every query through the accurate (hi/lo split, 3 MMAs per k-step)
    # tensor-core path: it must agree with the fp32 FMA path to fp32 round-off, not to fp16 round-off
    sd, inp, g = golden_model_case(variant)
    args = (cu(inp['patch_pts_ps']), cu(inp['pts_sub_sample_ms']), cu(inp['imp_surf_query_point_ms']))
    ref = make_engine(sd, variant, precision='fp32').forward(*args).cpu().numpy()
    eng = make_engine(sd, variant, precision='tc', guard_band=1e9)
    out = eng.forward(*args).cpu().numpy()
    assert eng.last_guard_count() == 8
    err = np.abs(out - ref).max()
    print(variant, 'split-precision logit err vs fp32 path', err, 'vs oracle', np.abs(out - g['logits']).max())
    assert err < 2e-3, err
    assert np.abs(out - g['logits']).max() < 3e-3
    # a larger ragged batch (several CTAs per stream, partial streams)
    sd2 = calibrated_state_dict(variant, 21)
    inp2 = synth.make_model_inputs(45, seed=9)
    a2 = (cu(inp2['patch_pts_ps']), cu(inp2['pts_sub_sample_ms']), cu(inp2['imp_surf_query_point_ms']))
    r2 = make_engine(sd2, variant, precision='fp32').forward(*a2).cpu().numpy()
    o2 = make_engine(sd2, variant, precision='tc', guard_band=1e9).forward(*a2).cpu().numpy()
    assert np.abs(o2 - r2).max() < 2e-3


# ------------------------------------------------------------------ section 8f-2: other patch / sub-sample sizes
# (small_kNN: 75-point patches; ragged tile tails on every path: 75, 200, 511 are no multiples of the 128-point tile)
@pytest.mark.parametrize('variant,P,S', [('uniform', 75, 1000), ('vanilla', 200, 500), ('max', 511, 300)])
def test_other_patch_and_subsample_sizes(variant, P, S):
    v = synth.VARIANTS[variant]
    sd = synth.make_state_dict(variant, seed=77)
    inp = synth.make_model_inputs(24, points_per_patch=P, sub_sample_size=S, seed=78)
    ref = orc.model_forward(sd, inp['patch_pts_ps'], inp['pts_sub_sample_ms'], inp['imp_surf_query_point_ms'],
                            v['use_point_stn'], v['shared_transformer'])
    args = (cu(inp['patch_pts_ps']), cu(inp['pts_sub_sample_ms']), cu(inp['imp_surf_query_point_ms']))
    scale = max(1.0, np.abs(ref).max())
    e32 = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], points_per_patch=P, sub_sample_size=S, precision='fp32')
    assert np.abs(e32.forward(*args).cpu().numpy() - ref).max() < 2e-3 * scale
    etc = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], points_per_patch=P, sub_sample_size=S, precision='tc',
                     guard_band=0.0)
    assert np.abs(etc.forward(*args).cpu().numpy() - ref).max() < 3e-2 * scale
    etc.set_precision('tc', guard_band=1e9)            # every query through the split-precision recompute path
    assert np.abs(etc.forward(*args).cpu().numpy() - ref).max() < 2e-3 * scale
    # the assembly kernels at the same sizes: exact kNN order and radius against the brute-force oracle
    cloud = synth.make_cloud('torus', 2500, seed=79)
    q = cloud[:40] + 0.01
    ids, patch, radius = ops.knn_patch(cu(cloud), cu(q.astype(np.float32)), P)
    for i in range(0, 40, 7):
        rid = orc.knn_bruteforce(cloud, q[i].astype(np.float32), P)
        assert np.array_equal(ids[i].cpu().numpy(), np.asarray(rid[0] if isinstance(rid, tuple) else rid).astype(np.int32))
    with pytest.raises(ops.P2SError):
        ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], points_per_patch=2000, sub_sample_size=S)   # documented limit 1536


def test_large_knn_1200_point_patches():
    """experiments/train_p2s_large_kNN.sh: points_per_patch 1200 (per-branch QSTN topology) on all three network paths and
    through the kNN kernel's 2048-candidate instantiation."""
    variant, P, S = 'uniform', 1200, 1000
    v = synth.VARIANTS[variant]
    sd = synth.make_state_dict(variant, seed=81)
    inp = synth.make_model_inputs(12, points_per_patch=P, sub_sample_size=S, seed=82)
    ref = orc.model_forward(sd, inp['patch_pts_ps'], inp['pts_sub_sample_ms'], inp['imp_surf_query_point_ms'],
                            v['use_point_stn'], v['shared_transformer'])
    args = (cu(inp['patch_pts_ps']), cu(inp['pts_sub_sample_ms']), cu(inp['imp_surf_query_point_ms']))
    scale = max(1.0, np.abs(ref).max())
    e32 = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], points_per_patch=P, sub_sample_size=S, precision='fp32')
    assert np.abs(e32.forward(*args).cpu().numpy() - ref).max() < 2e-3 * scale
    etc = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], points_per_patch=P, sub_sample_size=S, precision='tc', guard_band=0.0)
    assert np.abs(etc.forward(*args).cpu().numpy() - ref).max() < 3e-2 * scale
    etc.set_precision('tc', guard_band=1e9)
    assert np.abs(etc.forward(*args).cpu().numpy() - ref).max() < 2e-3 * scale
    cloud = synth.make_cloud('torus', 6000, seed=83)
    q = orc.query_grid(cloud, 24, 3)[::37][:48]
    ids, patch, radius = ops.knn_patch(cu(cloud), cu(q), P)
    ids, patch, radius = ids.cpu().numpy(), patch.cpu().numpy(), radius.cpu().numpy()
    kd = orc.make_kdtree(cloud)
    for i in range(len(q)):
        oid, ops_, orad = orc.knn_patch(cloud, kd, q[i], P)
        bid, d2 = orc.knn_bruteforce(cloud, q[i], P)
        gd = ((cloud[ids[i]].astype(np.float64) - q[i].astype(np.float64)) ** 2).sum(1)
        assert np.array_equal(gd, d2) and radius[i] == orad
        if np.all(np.diff(d2) > 0):
            assert np.array_equal(ids[i], oid) and np.array_equal(patch[i], ops_)
    # fused pipeline at this patch size
    lin, sdf = etc.reconstruct(cu(cloud), 16, 3, 1, 5)
    assert torch.isfinite(sdf).all() and lin.numel() == len(orc.query_grid(cloud, 16, 3))

