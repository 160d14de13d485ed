#!/usr/bin/env python
"""bench.py -- SDF queries/s of the Points2Surf reconstruction hot path on B200 (BASELINE.json metric).

One "step" = one pass of the hot path over one shape: point cloud -> candidate grid -> per query
(kNN-300 patch, 1000-point sub-sample, PointNet stacks, |SDF|+sign) -> SDF band of Q queries.
Workload (config.workload): vanilla model (shared QSTN, distance-weighted sub-sample), one synthetic
10k-point cloud per GPU, grid_res 256, epsilon 3 -- the model/cloud of BASELINE.json configs[1] at the
grid resolution its `metric` is quoted on; with --gpus N every rank reconstructs its own shape (weak scaling,
no data-path collective, like configs[2]).

  value : whole-job queries/s, cloud already resident in HBM when the timed region starts (device entry point)
  e2e   : the same metric through the host-buffer C-ABI call (p2s_reconstruct_host): pinned host cloud in,
          SDF band + voxel indices out, copies inside the timed region
  roofline     : the dominant kernel (tensor-core PointNet pass) against MEASURED_PEAKS.json
  cpu_baseline : the oracle port of the reference's CPU path on a bounded sample of the same queries

`--impl reference` times the reference's own CPU algorithm (oracle port: scipy cKDTree + NumPy sampling +
torch-CPU network, all host threads) on bounded samples of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_PER_QUERY = {'vanilla': 1.1407e9, 'max': 0.7768e9}   # SURVEY.md section 8(d), eval mode, BN folded, un-padded


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--model', default='vanilla', choices=['vanilla', 'max'])
    ap.add_argument('--grid_res', type=int, default=256)
    ap.add_argument('--epsilon', type=int, default=3)
    ap.add_argument('--points', type=int, default=10000)
    ap.add_argument('--precision', default='auto', choices=['auto', 'tc', 'fp32'])
    ap.add_argument('--guard_band', type=float, default=None)
    ap.add_argument('--skip_mesh_stage', action='store_true', help='do not run the volume / marching-cubes stage (for kernel launch lists of the queries/s step)')
    ap.add_argument('--mix_shapes', action='store_true', help='sphere / torus / box per rank instead of same-size spheres')
    ap.add_argument('--cpu_sample', type=int, default=256, help='queries in the bounded CPU-baseline sample')
    ap.add_argument('--seed', type=int, default=40938661)
    ap.add_argument('--batch', type=int, default=0, help='queries per network batch (0 = library default 8192)')
    ap.add_argument('--workload', default='headline', choices=['headline', 'sharded'],
                    help="'sharded': only the shape-sharded job (configs 3 / 5: --model, --shapes_per_gpu, --grid_res), shapes/s")
    ap.add_argument('--shapes_per_gpu', type=int, default=2)
    ap.add_argument('--skip_sharded', action='store_true', help='headline run without the sharded-job / tile-sharded sections')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write what the last timed step returned on rank 0 (voxel_index, sdf) as DIR/<name>.npy, for output-for-output "
                         "comparison of two builds on the same seeded workload")
    return ap.parse_args()


def dist_env():
    return int(os.environ.get('RANK', 0)), int(os.environ.get('LOCAL_RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))


def make_workload(args, rank):
    from points2surf_b200 import synth
    # weak scaling: every rank reconstructs a shape of the same kind and size (sphere, different seed), so the per-GPU
    # work is fixed as N grows; --mix_shapes gives the sphere / torus / box mix of SURVEY config 3 (unequal Q per rank)
    kinds = ['sphere', 'torus', 'box'] if args.mix_shapes else ['sphere']
    cloud = synth.make_cloud(kinds[rank % len(kinds)], args.points, seed=rank)
    sd = synth.make_state_dict(args.model, 6 if args.model == 'vanilla' else 4)
    return cloud, sd


# ----------------------------------------------------------------------------------------------------
# CPU side: oracle port of the reference path (test infrastructure used as the timed CPU baseline)
# ----------------------------------------------------------------------------------------------------
_ASM = {}


def _assemble_chunk(job):
    """Worker of the assembly pool (the reference runs PointcloudPatchDataset.__getitem__ in DataLoader worker processes,
    source/points_to_surf_eval.py:141-147)."""
    from oracle import p2s_oracle as orc
    idx, seed = job
    g = _ASM
    rng = np.random.RandomState(seed)
    return [orc.assemble_query(g['cloud'], g['kd'], g['qpts'][i], 300, 1000, rng, g['uniform']) for i in idx]


def cpu_reference_rate(args, cloud, sd, n_queries, fc4_bias=None, threads=None, workers=None):
    """queries/s of the reference algorithm on the host cores for `n_queries` queries of this workload: per-query assembly
    in `workers` processes (like the reference's DataLoader workers), network with `threads` torch threads."""
    import multiprocessing as mp
    import torch
    from oracle import p2s_oracle as orc
    from points2surf_b200 import synth
    v = synth.VARIANTS[args.model]
    cores = os.cpu_count() or 1
    threads = threads or cores
    workers = workers if workers is not None else max(1, min(cores - 1, 32))
    torch.set_num_threads(threads)
    if fc4_bias is not None:
        sd = dict(sd)
        sd['fc4.bias'] = torch.from_numpy(np.asarray(fc4_bias, dtype=np.float32))
    t0 = time.perf_counter()
    qpts = orc.query_grid(cloud, args.grid_res, args.epsilon)
    t_grid = time.perf_counter() - t0
    Q = len(qpts)
    sel = np.linspace(0, Q - 1, n_queries).astype(np.int64)
    kd = orc.make_kdtree(cloud)
    _ASM.update(cloud=cloud, kd=kd, qpts=qpts, uniform=bool(v['uniform_subsample']))
    t0 = time.perf_counter()
    if workers > 1 and n_queries >= 2 * workers:
        jobs = [(c, args.seed + j) for j, c in enumerate(np.array_split(sel, workers))]
        try:
            with mp.get_context('fork').Pool(workers) as pool:   # fork: the cloud / kd-tree are inherited, not pickled
                items = [it for part in pool.map_async(_assemble_chunk, jobs).get(timeout=180) for it in part]
        except Exception:                                        # a stuck or failed pool must not cost the bench line
            workers = 1
            items = _assemble_chunk((sel, args.seed))
    else:
        items = _assemble_chunk((sel, args.seed))
    patch = np.stack([it['patch_pts_ps'] for it in items])
    sub = np.stack([it['pts_sub_sample_ms'] for it in items])
    rad = np.array([it['patch_radius_ms'] for it in items])
    t_asm = time.perf_counter() - t0
    t0 = time.perf_counter()
    logits = orc.model_forward(sd, patch, sub, qpts[sel], v['use_point_stn'], v['shared_transformer'])
    sdf = orc.post_process(logits, rad)
    t_net = time.perf_counter() - t0
    # candidate grid is a per-shape cost: charge the sample its share
    total = t_asm + t_net + t_grid * (n_queries / max(Q, 1))
    return dict(value=n_queries / total, cores=cores, threads=threads, workers=workers, Q=Q, t_assemble_s=t_asm,
                t_network_s=t_net, t_grid_s=t_grid, sdf_checksum=float(np.abs(sdf).sum()))


def best_cpu_threads(args, cloud, sd):
    """Give the CPU arm its best configuration: probe the torch thread count on a 32-query sample."""
    cores = os.cpu_count() or 1
    best, best_rate = cores, 0.0
    for t in sorted({min(cores, c) for c in (8, 16, 32, 64, cores)}):
        r = cpu_reference_rate(args, cloud, sd, 32, threads=t)
        if r['value'] > best_rate:
            best, best_rate = t, r['value']
    return best, best_rate


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    cloud, sd = make_workload(args, 0)
    # bounded sample per step: size it from a 32-query probe so that the whole --warmup/--steps run ends in ~3 minutes
    threads, probe_rate = best_cpu_threads(args, cloud, sd)
    budget_s = 150.0
    args.cpu_sample = int(max(16, min(args.cpu_sample, probe_rate * budget_s / max(1, args.warmup + args.steps))))
    rates = []
    r = None
    for i in range(args.warmup + args.steps):
        r = cpu_reference_rate(args, cloud, sd, args.cpu_sample, threads=threads)
        if i >= args.warmup:
            rates.append(r['value'])
    value = float(np.mean(rates))
    line = {
        'impl': 'reference', 'metric': 'SDF queries/sec at grid_res=%d' % args.grid_res, 'value': value,
        'unit': 'queries/s', 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * args.cpu_sample / value, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, r['Q']),
        'cpu_baseline': {'value': value, 'unit': 'queries/s', 'cores': r['cores'], 'threads_used': max(r['threads'], r['workers']), 'kind': 'port',
                         'sample': '%d queries evenly spaced over the %d-query band per step (oracle port: scipy cKDTree kNN + '
                                   'NumPy RandomState sub-sample in %d worker processes, torch-CPU fp32 network on %d threads)'
                                   % (args.cpu_sample, r['Q'], r['workers'], r['threads'])},
        'e2e': {'value': value, 'unit': 'queries/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    if world > 1:
        # the CPU arm does not scale with --gpus: one host, rank 0 alone ran (the other ranks exited without work)
        line['cpu_baseline']['hosts'] = 1
        line['cpu_baseline']['sample'] += '; launched with %d ranks: rank 0 alone ran on this single host' % world
    print(json.dumps(line))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each array as out_dir/<name>.npy: floating arrays as float32, integer arrays as float64 (exact below 2^53).
    The arrays share their first axis.  Above DUMP_LIMIT_BYTES in all, a fixed, seeded subset of rows is written instead,
    with its row numbers as row_index.npy, so that runs with the same arguments dump the same rows."""
    arrays = {k: np.asarray(a, np.float32 if np.issubdtype(a.dtype, np.floating) else np.float64) for k, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.nbytes // max(n, 1) for a in arrays.values())
    keep = DUMP_LIMIT_BYTES // (row_bytes + 8)
    if n > keep:
        rows = np.sort(np.random.RandomState(0).choice(n, keep, replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays['row_index'] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + '.npy'), a)


def workload_config(args, Q):
    return {'workload': '%s model, 1 synthetic %d-pt %s cloud per GPU, grid_res=%d, epsilon=%d, kNN 300 + 1000-pt sub-sample'
                        % (args.model, args.points, 'sphere/torus/box' if args.mix_shapes else 'sphere', args.grid_res, args.epsilon),
            'queries_per_shape': int(Q), 'l2': 'flushed between timed iterations (256 MiB write)'}


def calibrate_output_bias(sd, model, device_index):
    """Centre the output bias of the rand-init checkpoint on a calibration batch (GPU fp32 path) so that the sign
    classes are mixed; modifies `sd` in place and returns the new bias.  tests/test_gpu_headline.py builds the
    bench's exact checkpoint through this function."""
    import torch
    from points2surf_b200 import ops, synth
    v = synth.VARIANTS[model]
    dev = torch.device('cuda', device_index)
    eng = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], device=device_index, precision='fp32')
    cal = synth.make_model_inputs(64, seed=777)
    raw = eng.forward(*(torch.from_numpy(cal[k]).to(dev) for k in ('patch_pts_ps', 'pts_sub_sample_ms', 'imp_surf_query_point_ms')))
    fc4_bias = (sd['fc4.bias'].numpy() - raw.median(dim=0).values.cpu().numpy()).astype(np.float32)
    eng.close()
    sd['fc4.bias'] = torch.from_numpy(fc4_bias)
    return fc4_bias


# ----------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(',')])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for j, n in enumerate(names) if any(s[2 + j].lower().startswith('active') for s in self.samples if len(s) > 2 + j)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                'reasons': reasons, 'samples': len(self.samples)}



# ----------------------------------------------------------------------------------------------------
# Sharded jobs (SURVEY section 8e), each timed end to end on the device: CUDA events around the rank's own work
# including the final gather, barrier on both sides, max over ranks.
# ----------------------------------------------------------------------------------------------------
def _timed_region(fn, dev, world, dist):
    import torch
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = fn()
    e1.record()
    torch.cuda.synchronize()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item()), out


def run_sharded_job(model, shapes_per_gpu, res, eps, seed, points, precision, guard, rank, world, dev, dist):
    """Shape-level sharding (BASELINE configs 3 and 5): shapes_per_gpu * world synthetic shapes (sphere / torus / box mix),
    greedy LPT assignment by the candidate-query count of the grid kernel, every rank runs the WHOLE pipeline for its shapes
    (queries -> SDF band -> sign propagation -> marching cubes), meshes gathered to rank 0 point-to-point.  The checkpoint
    has the fitted last layer so that a surface is meshed."""
    import torch
    from points2surf_b200 import ops, synth, sharding
    v = synth.VARIANTS[model]
    kinds = ['sphere', 'torus', 'box']
    n_shapes = shapes_per_gpu * world
    clouds = [torch.from_numpy(synth.make_cloud(kinds[i % 3], points, seed=i)).to(dev) for i in range(n_shapes)]
    loads = [int(ops.query_grid(c, res, eps).numel()) for c in clouds]          # every rank computes the same table
    bins, tot = sharding.lpt_assign(loads, world)
    mine = bins[rank]
    sd = synth.make_state_dict(model, 6 if model == 'vanilla' else 4, fitted=True)
    eng = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], device=dev.index, precision=precision, guard_band=guard)

    def one(i):
        lin, sdf = eng.reconstruct(clouds[i], res, eps, v['uniform_subsample'], seed, cap=loads[i])
        vol, _ = ops.sdf_to_volume(lin, sdf, res, 5, 13.0)
        mv, mf = ops.marching_cubes(vol, 0.0)
        return (i, mv, mf)

    def job():
        meshes = [one(i) for i in mine]
        return sharding.gather_meshes(meshes, dst=0)

    if mine:
        one(mine[0])                                   # warm-up: workspaces, NCCL channels
    job()
    ms, got = _timed_region(job, dev, world, dist)
    eng.close()
    res_d = {'workload': '%d shapes (%d per GPU; sphere / torus / box, %d points each), %s model with fitted last layer, grid_res %d, '
                         'epsilon %d: queries -> SDF band -> sign propagation -> marching cubes -> meshes gathered on rank 0; '
                         'LPT assignment by candidate-query count' % (n_shapes, shapes_per_gpu, points, model, res, eps),
             'shapes': n_shapes, 'ms': ms, 'shapes_per_s': n_shapes / (ms * 1e-3), 'queries': int(sum(loads)),
             'queries_per_s': sum(loads) / (ms * 1e-3), 'lpt_max_over_mean_load': max(tot) / (sum(tot) / world)}
    if rank == 0:
        res_d['meshes_on_rank0'] = len(got)
        res_d['mesh_bytes'] = int(sum(m[1].numel() * 4 + m[2].numel() * 4 for m in got))
        res_d['faces_total'] = int(sum(m[2].shape[0] for m in got))
    return res_d


def run_tile_sharded(eng, pts, res, eps, uniform, seed, Q, rank, world, dev, dist):
    """Tile-level sharding of ONE shape (strong scaling): rank r reconstructs a contiguous slab of the ordered query list,
    the SDF band is gathered point-to-point on rank 0, which runs sign propagation and marching cubes."""
    from points2surf_b200 import ops, sharding
    first, count = sharding.query_slab(Q, rank, world)
    counts = [sharding.query_slab(Q, r, world)[1] for r in range(world)]

    def job():
        lin, sdf = eng.reconstruct(pts, res, eps, uniform, seed, first_query=first, num_queries=count)
        band = sharding.gather_band(sdf, counts, dst=0) if world > 1 else sdf
        if rank == 0:
            lin_all = ops.query_grid(pts, res, eps) if world > 1 else lin
            vol, _ = ops.sdf_to_volume(lin_all, band, res, 5, 13.0)
            return ops.marching_cubes(vol, 0.0)
        return None

    job()
    ms, out = _timed_region(job, dev, world, dist)
    return {'workload': 'one shape, ordered query list cut into %d contiguous slabs, band gathered on rank 0 which meshes it' % world,
            'queries': int(Q), 'ms': ms, 'queries_per_s': Q / (ms * 1e-3), 'shapes_per_s': 1e3 / ms,
            'faces': int(out[1].shape[0]) if out is not None else None}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from points2surf_b200 import ops, synth, _lib
    rank, local_rank, world = dist_env()
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device: there is no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    v = synth.VARIANTS[args.model]
    cloud, sd = make_workload(args, rank)
    precision = args.precision
    if precision == 'auto':
        precision = 'tc'
    guard = args.guard_band if args.guard_band is not None else (0.05 if precision == 'tc' else 0.0)
    if args.workload == 'sharded':
        # BASELINE configs 3 / 5 on their own: e.g. --model max --grid_res 256 --shapes_per_gpu 1 (config 3 at --gpus 8),
        # --model vanilla --grid_res 512 --shapes_per_gpu 8 (config 5 at --gpus 8).  Metric: shapes/s reconstructed.
        sampler = ClockSampler(local_rank)
        sampler.start()
        job = run_sharded_job(args.model, args.shapes_per_gpu, args.grid_res, args.epsilon, args.seed, args.points, precision, guard,
                              rank, world, dev, dist)
        sampler.stop_flag = True
        sampler.join(timeout=2)
        if rank == 0:
            print(json.dumps({'metric': 'shapes/sec reconstructed at grid_res=%d (marching cubes and mesh gather included)' % args.grid_res,
                              'value': job['shapes_per_s'], 'unit': 'shapes/s', 'n_gpus': world, 'steps': 1, 'warmup': 1,
                              'ms_per_step': job['ms'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                              'dtype': 'f16 operands / f32 accumulate (tcgen05)', 'data': 'synthetic', 'config': {'workload': job['workload']},
                              'clocks': sampler.summary(), 'sharded_job': job}))
        if world > 1:
            dist.destroy_process_group()
        return

    fc4_bias = calibrate_output_bias(sd, args.model, local_rank)
    eng = ops.Engine(sd, v['use_point_stn'], v['shared_transformer'], device=local_rank, precision=precision, guard_band=guard)

    pts = torch.from_numpy(cloud).to(dev)
    Q = int(ops.query_grid(pts, args.grid_res, args.epsilon).numel())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    host_cloud = torch.from_numpy(cloud).pin_memory()
    host_lin = torch.empty(Q, dtype=torch.int32).pin_memory()
    host_sdf = torch.empty(Q, dtype=torch.float32).pin_memory()

    def step_dev():
        return eng.reconstruct(pts, args.grid_res, args.epsilon, v['uniform_subsample'], args.seed, cap=Q, batch=args.batch)

    def step_host():
        return eng.reconstruct_host(host_cloud.numpy(), args.grid_res, args.epsilon, v['uniform_subsample'], args.seed, cap=Q,
                                    out_lin=host_lin.numpy(), out_sdf=host_sdf.numpy(), batch=args.batch)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, host=False):
        for _ in range(warmup):
            fn()
        barrier()
        ops.launch_count(reset=True)
        if not host:
            eng.profile_enable(precision == 'tc')
        total_ms = 0.0
        out = None
        for _ in range(steps):
            flush.zero_()
            torch.cuda.synchronize()
            if host:
                t0 = time.perf_counter()
                out = fn()
                total_ms += (time.perf_counter() - t0) * 1e3     # the host call returns after its D2H completed
            else:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = fn()
                e1.record()
                torch.cuda.synchronize()
                total_ms += e0.elapsed_time(e1)
        barrier()
        launches = ops.launch_count()
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, out

    try:
        peaks_hbm = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs']
    except Exception:
        peaks_hbm = 6576.1   # B200_PROFILING.md fallback (measured copy bandwidth of this pool)
    sampler = ClockSampler(local_rank)
    sampler.start()
    dev_ms, launches, (lin_last, sdf_last) = timed(step_dev, args.steps, max(args.warmup, 3))
    guard_total = eng.last_guard_count() if precision == 'tc' else 0   # warm-up + timed steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'voxel_index': lin_last.cpu().numpy(), 'sdf': sdf_last.cpu().numpy()})

    prof = eng.profile_get() if precision == 'tc' else None
    eng.profile_enable(False)
    # second half of the metric ("shapes/sec reconstructed"): SDF band -> volume -> sign propagation -> marching cubes,
    # measured on this rank's shape outside the queries/s region (HBM/L2-bound byte kernels, SURVEY section 8d)
    mesh_stage = None
    if not args.skip_mesh_stage:
        from points2surf_b200 import sharding
        # the timed checkpoint is rand-init (calibrated bias): its SDF describes no surface.  The mesh stage runs on the
        # SDF of the same architecture with the fitted last layer (synth.fitted_fc4), so that sign propagation and
        # marching cubes see a surface-like band and a real mesh comes out.
        sd_fit = synth.make_state_dict(args.model, 6 if args.model == 'vanilla' else 4, fitted=True)
        eng_fit = ops.Engine(sd_fit, v['use_point_stn'], v['shared_transformer'], device=local_rank, precision=precision, guard_band=guard)
        lin, sdf = eng_fit.reconstruct(pts, args.grid_res, args.epsilon, v['uniform_subsample'], args.seed, cap=Q)
        eng_fit.close()
        res = args.grid_res
        for _ in range(2):
            vol, iters = ops.sdf_to_volume(lin, sdf, res, 5, 13.0)
            mv, mf = ops.marching_cubes(vol, 0.0)
        barrier()
        # five timed repetitions, median of each stage (single 2-3 ms calls next to the clock sampler are noisy)
        tv, tm = [], []
        for _ in range(5):
            e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
            e0.record()
            vol, iters = ops.sdf_to_volume(lin, sdf, res, 5, 13.0)
            e1.record()
            mv, mf = ops.marching_cubes(vol, 0.0)
            e2.record()
            torch.cuda.synchronize()
            tv.append(e0.elapsed_time(e1)); tm.append(e1.elapsed_time(e2))
        t_vol, t_mc = sorted(tv)[2], sorted(tm)[2]
        # final mesh gather to rank 0 (NCCL over NVLink; the only data-path communication of the sharded run)
        t_gather, gathered = 0.0, 1
        if world > 1:
            sharding.gather_meshes([(rank, mv, mf)], dst=0)   # warm-up (NCCL channel setup)
            barrier()
            t0 = time.perf_counter()
            got = sharding.gather_meshes([(rank, mv, mf)], dst=0)
            barrier()
            t_gather = (time.perf_counter() - t0) * 1e3
            gathered = len(got) if rank == 0 else 0
        tt = torch.tensor([t_vol + t_mc, t_gather], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        vox = float(res) ** 3
        mesh_stage = {'sign_propagation_ms': t_vol, 'sign_propagation_iterations': int(iters),
                      'sign_propagation_GBps': vox * 2.0 * (max(iters, 0) + 1) / (t_vol * 1e-3) / 1e9,
                      'sign_propagation_frac_of_hbm_peak': vox * 2.0 * (max(iters, 0) + 1) / (t_vol * 1e-3) / 1e9 / float(peaks_hbm),
                      'marching_cubes_ms': t_mc, 'verts': int(mv.shape[0]), 'faces': int(mf.shape[0]),
                      'marching_cubes_GBps': (vox * 4.0 * 2 + vox * 20.0 + mv.shape[0] * 12.0 + mf.shape[0] * 12.0) / (t_mc * 1e-3) / 1e9,
                      'bytes_model': 'sign propagation: SURVEY 8d algorithmic bytes = res^3 * 2 B per vote evaluation (iterations + 1; the whole scatter/init/propagate/finalize call is timed, median of 5); MC: res^3 * (2 x 4 B volume reads + 20 B scan scratch) + mesh bytes',
                      'mesh_gather_ms': float(tt[1].item()), 'meshes_on_rank0': gathered,
                      'shapes_per_s_incl_mesh': world * 1e3 / (dev_ms / args.steps + float(tt[0].item()) + float(tt[1].item()))}
    sampler.stop_flag = True
    sampler.join(timeout=2)
    sharded_job = tile_sharded = None
    if not args.skip_sharded:
        # config 3 analogue (max model, mixed shapes, LPT, whole pipeline + mesh gather timed) and strong scaling of one shape
        # (a failure in these add-on sections must not take the headline line with it: it is reported in their place)
        try:
            sharded_job = run_sharded_job('max', args.shapes_per_gpu, args.grid_res, args.epsilon, args.seed, args.points, precision, guard,
                                          rank, world, dev, dist)
        except Exception as e:  # noqa: BLE001
            sharded_job = {'error': '%s: %s' % (type(e).__name__, e)}
        try:
            sd_fit = synth.make_state_dict(args.model, 6 if args.model == 'vanilla' else 4, fitted=True)
            eng_fit = ops.Engine(sd_fit, v['use_point_stn'], v['shared_transformer'], device=local_rank, precision=precision, guard_band=guard)
            pts0 = torch.from_numpy(synth.make_cloud('sphere', args.points, seed=0)).to(dev)     # the same shape on every rank
            Q0 = int(ops.query_grid(pts0, args.grid_res, args.epsilon).numel())
            tile_sharded = run_tile_sharded(eng_fit, pts0, args.grid_res, args.epsilon, v['uniform_subsample'], args.seed, Q0, rank, world, dev, dist)
            eng_fit.close()
        except Exception as e:  # noqa: BLE001
            tile_sharded = {'error': '%s: %s' % (type(e).__name__, e)}
    e2e_ms, _, _ = timed(step_host, args.steps, 1, host=True)
    guard_frac = guard_total / max(Q * (args.steps + max(args.warmup, 3)), 1)

    q_total = torch.tensor([Q], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(q_total)
    q_total = float(q_total.item())
    value = q_total * args.steps / (dev_ms * 1e-3)
    e2e_value = q_total * args.steps / (e2e_ms * 1e-3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        roofline = None
        if prof and prof['launches'] > 0:
            peak = peaks.get('bf16_tflops_sustained') or 1400.0
            ach = prof['flops'] / (prof['ms'] * 1e-3) / 1e12
            traffic = None   # per-launch DRAM bytes come from an `ncu --set full` capture (profiles/), not from this run
            roofline = {'bound': 'tensor', 'kernel': prof['kernel'], 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s',
                        'frac': ach / peak, 'traffic': traffic,
                        'peak_source': 'MEASURED_PEAKS.json bf16_tflops_sustained (of measured)' if peaks else 'fallback 1.4 PFLOP/s sustained (of fallback)',
                        'flops_per_launch': prof['flops'] / prof['launches'], 'ms_per_launch': prof['ms'] / prof['launches'],
                        'share_of_step': prof['ms'] / dev_ms}
        if args.cpu_sample > 0 and world == 1:
            cpu_threads, _ = best_cpu_threads(args, cloud, sd)
            cpu = cpu_reference_rate(args, cloud, sd, args.cpu_sample, fc4_bias=fc4_bias, threads=cpu_threads)
        else:
            cpu = dict(value=None, cores=os.cpu_count(), threads=0, workers=0, t_assemble_s=0.0, t_network_s=0.0)
        line = {
            'metric': 'SDF queries/sec at grid_res=%d' % args.grid_res, 'value': value, 'unit': 'queries/s',
            'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': dev_ms / args.steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f16 operands / f32 accumulate (tcgen05); hi/lo split f16 (fp32-level) for FC tails and guard-band recompute' if precision == 'tc' else 'f32',
            'data': 'synthetic', 'config': dict(workload_config(args, Q), precision=precision, guard_band=guard,
                                                guard_recompute_fraction=guard_frac),
            'e2e': {'value': e2e_value, 'unit': 'queries/s', 'h2d_bytes_per_step': int(cloud.nbytes), 'd2h_bytes_per_step': int(Q * 8)},
            'gpu_launches': int(launches),
            'clocks': sampler.summary(),
            'roofline': roofline,
            'cpu_baseline': {'value': cpu['value'], 'unit': 'queries/s', 'cores': cpu['cores'], 'threads_used': max(cpu['threads'], cpu['workers']), 'kind': 'port',
                             'sample': '%d queries evenly spaced over the band (assembly in %d worker processes %.2fs, network on %d torch threads %.2fs)'
                                       % (args.cpu_sample, cpu['workers'], cpu['t_assemble_s'], cpu['threads'], cpu['t_network_s'])},
            'tensor_flops_per_s': value * FLOP_PER_QUERY[args.model],
            'mesh_stage': mesh_stage,
            'sharded_job': sharded_job,
            'tile_sharded_one_shape': tile_sharded,
        }
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_b200(a)
