"""Drop-in for source/points_to_surf_eval.py: same CLI (parse_arguments), same entry point
(points_to_surf_eval(eval_opt)), same output tree -- the per-query DataLoader + model loop
(points_to_surf_eval.py:337-404) is replaced by the fused B200 pipeline (one C-ABI call per shape).

Outputs per shape, as in the reference (points_to_surf_eval.py:199-294):
  <outdir>/{rec|eval}/eval/<name>.xyz.npy, .xyz.txt      signed distance per query
  <outdir>/{rec|eval}/vis/<name>.ply                      coloured query points
  <outdir>/rec/query_pts_ms/<name>.xyz.npy, rec/dist_ms/<name>.xyz.npy, rec/query_pts_ms_vis/<name>.ply

With torch.distributed initialised (one rank per GPU), shapes are sharded round-robin over ranks; there is no
data-path collective (every shape is independent).
"""
import argparse
import os
import random

import numpy as np
import torch

from . import ops
from . import samplers
from . import sdf as p2s_sdf
from .weights import strip_module_prefix


def parse_arguments(args=None):
    """The reference's flags, verbatim (source/points_to_surf_eval.py:16-65), plus --precision / --guard_band."""
    parser = argparse.ArgumentParser()
    parser.add_argument('--indir', type=str, default='datasets/abc_minimal', help='input folder (meshes)')
    parser.add_argument('--outdir', type=str, default='results', help='output folder (estimated point cloud properties)')
    parser.add_argument('--dataset', nargs='+', type=str, default=['testset.txt'], help='shape set file name')
    parser.add_argument('--reconstruction', type=bool, default=False, help='do reconstruction instead of evaluation')
    parser.add_argument('--query_grid_resolution', type=int, default=None, help='resolution of sampled volume used for reconstruction')
    parser.add_argument('--epsilon', type=int, default=None, help='neighborhood size for reconstruction')
    parser.add_argument('--certainty_threshold', type=float, default=None, help='')
    parser.add_argument('--sigma', type=int, default=None, help='')
    parser.add_argument('--up_sampling_factor', type=int, default=10, help='unused (kept for CLI compatibility)')
    parser.add_argument('--modeldir', type=str, default='models', help='model folder')
    parser.add_argument('--models', type=str, default='p2s_vanilla', help='names of trained models, can evaluate multiple models')
    parser.add_argument('--modelpostfix', type=str, default='_model.pth', help='model file postfix')
    parser.add_argument('--parampostfix', type=str, default='_params.pth', help='parameter file postfix')
    parser.add_argument('--gpu_idx', type=int, default=0, help='CUDA device index (there is no CPU path)')
    parser.add_argument('--sparse_patches', type=int, default=False, help='unused (kept for CLI compatibility)')
    parser.add_argument('--sampling', type=str, default='full', help='only "full" is supported')
    parser.add_argument('--patches_per_shape', type=int, default=1000, help='number of patches evaluated in each shape (only for sequential_shapes_random_patches)')
    parser.add_argument('--query_points_per_patch', type=int, default=1, help='number of query points per patch')
    parser.add_argument('--sub_sample_size', type=int, default=500, help='unused: the training value is taken from the params file')
    parser.add_argument('--seed', type=int, default=40938661, help='manual seed')
    parser.add_argument('--batchSize', type=int, default=0, help='queries per network batch, 0 = library default')
    parser.add_argument('--workers', type=int, default=0, help='unused: there is no DataLoader on this path')
    parser.add_argument('--cache_capacity', type=int, default=100, help='unused (kept for CLI compatibility)')
    parser.add_argument('--precision', type=str, default='tc', choices=['tc', 'fp32'], help='tensor-core fp16/fp32-acc or fp32 FMA')
    parser.add_argument('--guard_band', type=float, default=0.05, help='|sign logit| below which a query is recomputed in split precision')
    opt = parser.parse_args(args=args)
    if len(opt.dataset) == 1:
        opt.dataset = opt.dataset[0]
    return opt


def _load_train_opt(param_filename):
    # pickled argparse.Namespace (points_to_surf_train.py:420): needs weights_only=False under torch >= 2.6
    train_opt = torch.load(param_filename, weights_only=False)
    if not hasattr(train_opt, 'single_transformer'):
        train_opt.single_transformer = 0
    if not hasattr(train_opt, 'shared_transformer'):
        train_opt.shared_transformer = False
    return train_opt


def _check_supported(train_opt, eval_opt):
    outs = list(train_opt.outputs)
    if 'imp_surf' in outs or 'imp_surf_magnitude' not in outs or 'imp_surf_sign' not in outs:
        raise ValueError('Unsupported outputs %s: need imp_surf_magnitude + imp_surf_sign' % outs)
    if getattr(train_opt, 'sym_op', 'max') != 'max':
        raise ValueError('Unsupported symmetric operation: %s' % train_opt.sym_op)
    if getattr(train_opt, 'single_transformer', 0):
        raise ValueError('Unsupported option: single_transformer=1')
    if getattr(train_opt, 'fixed_subsample', 0) and not getattr(train_opt, 'uniform_subsample', 0):
        raise ValueError('Unsupported option: fixed_subsample=1 with the distance-weighted sub-sample (only with uniform_subsample=1)')
    if eval_opt.sampling not in ('full', 'sequential_shapes_random_patches'):
        raise ValueError('Unknown sampling strategy: %s' % eval_opt.sampling)
    if eval_opt.sampling != 'full' and eval_opt.reconstruction:
        raise ValueError('Unsupported option: --sampling %s with --reconstruction (a partial band cannot be meshed)' % eval_opt.sampling)


def _shape_names(indir, dataset):
    with open(os.path.join(indir, dataset)) as f:
        names = [x.strip() for x in f.readlines()]
    return list(filter(None, names))


def _load_pts(indir, name):
    pts = np.load(os.path.join(indir, '04_pts', name + '.xyz.npy'))
    if pts.shape[1] > 3:
        pts = pts[:, 0:3]
    if pts.dtype != np.float32:
        print('Warning: pts_np must be converted to float32: {}'.format(name))
        pts = pts.astype(np.float32)
    return np.ascontiguousarray(pts)


def _random_rotations(rng, n):
    """trimesh.transformations.random_rotation_matrix(rng.rand(3)) per query (data_loader.py:381-393)."""
    r = rng.rand(n, 3)
    r1, r2 = np.sqrt(1.0 - r[:, 0]), np.sqrt(r[:, 0])
    t1, t2 = 2.0 * np.pi * r[:, 1], 2.0 * np.pi * r[:, 2]
    q = np.stack([np.cos(t2) * r2, np.sin(t1) * r1, np.cos(t1) * r1, np.sin(t2) * r2], axis=1)
    q = q * np.sqrt(2.0 / (q * q).sum(axis=1, keepdims=True))
    o = q[:, :, None] * q[:, None, :]
    R = np.empty((n, 3, 3))
    R[:, 0, 0] = 1.0 - o[:, 2, 2] - o[:, 3, 3]; R[:, 0, 1] = o[:, 1, 2] - o[:, 3, 0]; R[:, 0, 2] = o[:, 1, 3] + o[:, 2, 0]
    R[:, 1, 0] = o[:, 1, 2] + o[:, 3, 0]; R[:, 1, 1] = 1.0 - o[:, 1, 1] - o[:, 3, 3]; R[:, 1, 2] = o[:, 2, 3] - o[:, 1, 0]
    R[:, 2, 0] = o[:, 1, 3] - o[:, 2, 0]; R[:, 2, 1] = o[:, 2, 3] + o[:, 1, 0]; R[:, 2, 2] = 1.0 - o[:, 1, 1] - o[:, 2, 2]
    return R.astype(np.float32)


def _rotate_inputs(patch, sub, q, R):
    """trafo.transform_points(x, rand_rot) = (R x^T)^T for the patch, the sub-sample and the query point
    (data_loader.py:385-393; the reference computes in float64 and casts to float32, here float32 throughout)."""
    Rt = R.transpose(1, 2)
    return (torch.matmul(patch, Rt).contiguous(), torch.matmul(sub, Rt).contiguous(),
            torch.matmul(q.unsqueeze(1), Rt).squeeze(1).contiguous())


def _fixed_sub(pts_dev, n, sub_sample_size):
    """[n,S,3]: the one fixed uniform sub-sample of the shape, for every query (samplers.fixed_uniform_subsample_ids)."""
    ids = torch.from_numpy(samplers.fixed_uniform_subsample_ids(pts_dev.shape[0], sub_sample_size).astype(np.int64)).to(pts_dev.device)
    return pts_dev.index_select(0, ids).unsqueeze(0).expand(n, -1, -1).contiguous()


def _patches(pts_dev, q, train_opt, seed, query_index_base=0):
    """-> (patch_pts_ps [n,P,3], radius [n] or None for fixed-radius patches)."""
    patch_radius = float(getattr(train_opt, 'patch_radius', 0.0))
    if patch_radius > 0.0:       # radius ablations: ball query, fixed-radius normalisation, |d| not rescaled (eval.py:364-368)
        _, patch, _, _ = ops.ball_patch(pts_dev, q, train_opt.points_per_patch, patch_radius, seed, query_index_base=query_index_base)
        return patch, None
    _, patch, radius = ops.knn_patch(pts_dev, q, train_opt.points_per_patch)
    return patch, radius


def _reconstruct_fixed_subsample(eng, train_opt, eval_opt, pts_dev):
    """Reconstruction pass of a model trained with --fixed_subsample 1 (uniform): the fused pipeline draws a sub-sample per
    query, so this variant runs stage by stage -- candidate grid, patches, the ONE fixed sub-sample, network, post-process."""
    lin = ops.query_grid(pts_dev, eval_opt.query_grid_resolution, eval_opt.epsilon)
    q_all = ops.query_points(lin, eval_opt.query_grid_resolution)
    bs = eval_opt.batchSize if eval_opt.batchSize > 0 else 4096
    out = []
    for b0 in range(0, q_all.shape[0], bs):
        q = q_all[b0:b0 + bs].contiguous()
        patch, radius = _patches(pts_dev, q, train_opt, eval_opt.seed, query_index_base=b0)
        sub = _fixed_sub(pts_dev, q.shape[0], train_opt.sub_sample_size)
        out.append(ops.sdf_from_logits(eng.forward(patch, sub, q), radius))
    sdf = torch.cat(out) if out else torch.zeros((0,), dtype=torch.float32, device=pts_dev.device)
    return lin, sdf


def _eval_given_queries(eng, train_opt, eval_opt, pts_dev, query_pts, dev):
    """Non-reconstruction pass (full_eval.py:31-41): queries from 05_query_pts, random rotation augmentation
    of patch / sub-sample / query like the reference's dataset does when reconstruction is False."""
    q = torch.from_numpy(np.ascontiguousarray(query_pts, dtype=np.float32)).to(dev)
    patch, radius = _patches(pts_dev, q, train_opt, eval_opt.seed)
    uniform = bool(getattr(train_opt, 'uniform_subsample', 0))
    if getattr(train_opt, 'fixed_subsample', 0):
        sub = _fixed_sub(pts_dev, q.shape[0], train_opt.sub_sample_size)
    else:
        sub = ops.gather_points(pts_dev, ops.subsample(pts_dev, q, train_opt.sub_sample_size, uniform, eval_opt.seed))
    R = torch.from_numpy(_random_rotations(np.random.RandomState(eval_opt.seed), q.shape[0])).to(dev)
    patch, sub, qr = _rotate_inputs(patch, sub, q, R)
    out = []
    bs = eval_opt.batchSize if eval_opt.batchSize > 0 else 4096
    for b0 in range(0, q.shape[0], bs):
        out.append(eng.forward(patch[b0:b0 + bs], sub[b0:b0 + bs], qr[b0:b0 + bs]))
    return ops.sdf_from_logits(torch.cat(out), radius)


def points_to_surf_eval(eval_opt):
    models = eval_opt.models.split()
    if eval_opt.seed < 0:
        eval_opt.seed = random.randint(1, 10000)
    if not torch.cuda.is_available() or eval_opt.gpu_idx < 0:
        raise ops.P2SError('points2surf_b200 needs a CUDA device (--gpu_idx >= 0): there is no CPU fallback')
    rank, world = 0, 1
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        rank, world = torch.distributed.get_rank(), torch.distributed.get_world_size()
    dev_index = eval_opt.gpu_idx if world == 1 else int(os.environ.get('LOCAL_RANK', rank))
    dev = torch.device('cuda', dev_index)
    torch.cuda.set_device(dev)

    for model_name in models:
        print('Random Seed: %d' % eval_opt.seed)
        random.seed(eval_opt.seed)
        torch.manual_seed(eval_opt.seed)
        model_filename = os.path.join(eval_opt.modeldir, model_name + eval_opt.modelpostfix)
        param_filename = os.path.join(eval_opt.modeldir, model_name + eval_opt.parampostfix)
        train_opt = _load_train_opt(param_filename)
        _check_supported(train_opt, eval_opt)
        state = strip_module_prefix(torch.load(model_filename, map_location='cpu'))
        eng = ops.Engine(state, train_opt.use_point_stn, train_opt.shared_transformer,
                         points_per_patch=train_opt.points_per_patch, sub_sample_size=train_opt.sub_sample_size,
                         net_size=getattr(train_opt, 'net_size', 1024), device=dev_index,
                         precision=getattr(eval_opt, 'precision', 'tc'), guard_band=getattr(eval_opt, 'guard_band', 0.05))
        uniform = bool(getattr(train_opt, 'uniform_subsample', 0))
        model_out_dir = os.path.join(eval_opt.outdir, 'rec' if eval_opt.reconstruction else 'eval')
        os.makedirs(model_out_dir, exist_ok=True)
        names = _shape_names(eval_opt.indir, eval_opt.dataset)
        print(f'evaluating {len(names)} shapes')
        shape_patch_inds = None
        if eval_opt.sampling == 'sequential_shapes_random_patches':     # points_to_surf_eval.py:130-136
            counts = [int(np.load(os.path.join(eval_opt.indir, '05_query_pts', n + '.ply.npy'), mmap_mode='r').shape[0]) for n in names]
            from types import SimpleNamespace
            sampler = samplers.SequentialShapeRandomPointcloudPatchSampler(
                SimpleNamespace(shape_names=names, shape_patch_count=counts), patches_per_shape=eval_opt.patches_per_shape,
                seed=eval_opt.seed, sequential_shapes=True, identical_epochs=False)
            list(iter(sampler))
            shape_patch_inds = sampler.shape_patch_inds
        # shapes are independent: greedy LPT over ranks by the candidate-query count in reconstruction mode (the cheap grid
        # kernel gives Q before any network work), round-robin otherwise; every rank derives the same table
        mine = None
        if world > 1 and eval_opt.reconstruction:
            from . import sharding
            loads = [int(ops.query_grid(torch.from_numpy(_load_pts(eval_opt.indir, n)).to(dev), eval_opt.query_grid_resolution,
                                        eval_opt.epsilon).numel()) for n in names]
            mine = set(sharding.shapes_for_rank(len(names), rank, world, loads=loads))
        for si, name in enumerate(names):
            if (si not in mine) if mine is not None else (si % world != rank):
                continue
            pts = _load_pts(eval_opt.indir, name)
            pts_dev = torch.from_numpy(pts).to(dev)
            if eval_opt.reconstruction and getattr(train_opt, 'fixed_subsample', 0):
                lin, sdf = _reconstruct_fixed_subsample(eng, train_opt, eval_opt, pts_dev)
                query_pts = ops.query_points(lin, eval_opt.query_grid_resolution).cpu().numpy()
            elif eval_opt.reconstruction:
                lin, sdf = eng.reconstruct(pts_dev, eval_opt.query_grid_resolution, eval_opt.epsilon, uniform,
                                           eval_opt.seed, batch=eval_opt.batchSize,
                                           patch_radius=float(getattr(train_opt, 'patch_radius', 0.0)))
                query_pts = ops.query_points(lin, eval_opt.query_grid_resolution).cpu().numpy()
            else:
                query_pts = np.load(os.path.join(eval_opt.indir, '05_query_pts', name + '.ply.npy')).astype(np.float32)
                if shape_patch_inds is not None:
                    inds = np.asarray(shape_patch_inds[si], dtype=np.int64)
                    query_pts = np.ascontiguousarray(query_pts[inds])
                    np.savetxt(os.path.join(model_out_dir, name + '.idx'), inds, fmt='%d')   # points_to_surf_eval.py:292-294
                sdf = _eval_given_queries(eng, train_opt, eval_opt, pts_dev, query_pts, dev)
            imp_surf_np_ms = sdf.cpu().numpy()
            os.makedirs(os.path.join(model_out_dir, 'eval'), exist_ok=True)
            np.save(os.path.join(model_out_dir, 'eval', name + '.xyz.npy'), imp_surf_np_ms)
            np.savetxt(os.path.join(model_out_dir, 'eval', name + '.xyz.txt'), imp_surf_np_ms)
            p2s_sdf.visualize_query_points(query_pts, imp_surf_np_ms, os.path.join(model_out_dir, 'vis', name + '.ply'))
            if eval_opt.reconstruction:
                imp_surf_np_ms[np.isnan(imp_surf_np_ms)] = 1.0
                os.makedirs(os.path.join(model_out_dir, 'query_pts_ms'), exist_ok=True)
                np.save(os.path.join(model_out_dir, 'query_pts_ms', name + '.xyz.npy'), query_pts)
                os.makedirs(os.path.join(model_out_dir, 'dist_ms'), exist_ok=True)
                np.save(os.path.join(model_out_dir, 'dist_ms', name + '.xyz.npy'), imp_surf_np_ms)
                p2s_sdf.visualize_query_points(query_pts, imp_surf_np_ms,
                                               os.path.join(model_out_dir, 'query_pts_ms_vis', name + '.ply'))
        eng.close()


if __name__ == '__main__':
    points_to_surf_eval(parse_arguments())
