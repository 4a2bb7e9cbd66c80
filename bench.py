#!/usr/bin/env python
"""Bench of the SHERF render hot path (ImportanceRenderer.forward + NeRFDecoder + ray marcher) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step = one pass of the hot path over N_gpus novel views of BASELINE.json configs[1]
(512x512 RenderPeople-shape, 64 samples/ray, one subject / one observation), synthetic seeded inputs.
With N > 1 (torchrun, one rank per GPU) the step's N x 262 144 rays are sharded across the ranks -- by default at view
granularity (rank r renders view r: the shard of the ray batch it owns), and the step ends with ONE all-gather of the
rendered tiles so that every rank holds all N images (weak scaling: N views on N GPUs).  `--shard tiles` instead
deals every view's rays to all ranks in interleaved 256-ray tiles with one all-gather per view (the single-view
latency mode of sherf_b200.dist.render_sharded).
Prints one JSON line (see README / DESIGN.md "Measurement").  `--dump-outputs DIR` also writes what the last timed step computed as
DIR/rgb.npy, DIR/depth.npy, DIR/acc.npy (float32, [views, rays, channels]); the inputs are seeded, so two builds run with the same
arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, S = 512, 512, 64
WORKLOAD = 'configs[1]: 512x512 RenderPeople-shape, 64 samples/ray, 1 subject novel view'
FLOP_PER_POINT = 429_248          # SURVEY.md 8(d): MLP MACs x 2 per decoded (surviving) sample
# the fused tcgen05 decoder kernel covers pts_linears[0..7], feature_linear, alpha_linear, views_linear, rgb_linear (triplane.py:293-314)
FLOP_PER_POINT_FUSED = 2 * (71 * 128 + 4 * 128 * 128 + 199 * 128 + 2 * 128 * 128 + 128 * 128 + 128 + 187 * 64 + 64 * 3)
GATHER_BYTES_PER_POINT = 8752     # SURVEY.md 8(d): tri-plane 1536 + 2-D feature 1024 + rgb 48 + 3-D pyramid 6144 bytes of taps per surviving sample (L2 -> SM traffic)
TF32_OVER_BF16 = 0.5              # dense TF32 tensor peak is half the bf16 peak (B200_PROFILING.md table: 1.1 vs 2.25 PF)
# DRAM bytes the path NEEDS per view (DESIGN.md section 4): per ray 28 B in + 20 B out; per surviving sample the 8 B of its compacted
# index pair written + read by the cull and the decoder-input tile (576 B) written by the front kernel and read by the decoder; once per
# view the feature tensors it actually touches (the scene is 25 + 17 + 3 + 270 MB; first touch of every line it needs)
NEEDED_DRAM_BYTES_PER_RAY = 48
NEEDED_DRAM_BYTES_PER_POINT = 2 * (8 + 576)
SCENE_BYTES = (3 * 32 * 256 * 256 + 64 * 256 * 256 + 3 * 512 * 512) * 4


def common_config(world, importance):
    """The workload description BOTH arms print (the driver compares the two `config` objects); arm-specific facts go under `arm`."""
    return {'workload': WORKLOAD if not importance else f'configs[4] shape on this GPU count: 512x512, {S}+{importance} coarse+fine importance sampling',
            'H': H, 'W': W, 'samples_per_ray': S, 'importance_samples_per_ray': importance, 'views_per_step': world,
            'parallelism': 'single GPU' if world == 1 else f'dp{world}: the step\'s {world} views are sharded over {world} ranks, one all-gather of the rendered tiles per step',
            'l2': 'working set of one view > 126 MB L2, plus an explicit 256 MiB flush between timed steps (outside the events)'}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='sherf_b200', choices=['sherf_b200', 'reference'])
    ap.add_argument('--precision', default='bf16x3', choices=['fp32', 'tf32', 'tf32x3', 'bf16x3'],
                    help="MLP arithmetic: tf32x3 = error-compensated 3xTF32 on tcgen05 (fp32-grade parity, default); fp32 = CUDA cores")
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-training-step', action='store_true', help='skip the (untimed) forward + backward measurement of the line\'s `training_step` key')
    ap.add_argument('--gpu-eager-baseline', action='store_true',
                    help='also time oracle/port.py (the reference path written as eager PyTorch) on this GPU for one full view (BASELINE.md 3.4)')
    ap.add_argument('--importance', type=int, default=0,
                    help='fine (importance) samples per ray; 64 = BASELINE configs[4] on one GPU (not the headline workload: the default is configs[1])')
    ap.add_argument('--shard', default='views', choices=['views', 'tiles'], help='N>1: ray-batch sharding granularity')
    ap.add_argument('--ref-rays', type=int, default=0, help='--impl reference: rays per step (0 = sized for a few minutes in total)')
    ap.add_argument('--ref-dump', default='', help='--impl reference: write the ray indices and the rendered outputs of the last step here (torch.save)')
    ap.add_argument('--dump-outputs', default='', metavar='DIR',
                    help='write rgb / depth / acc of the last timed step to DIR/<name>.npy (float32, [views, rays, channels])')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    return args


DUMP_BYTES_MAX = 64 << 20


def dump_outputs(out_dir, images):
    """images: [views, rays, 5] (rgb, depth, acc), the rendered outputs of one step.  Whole views only: when they exceed DUMP_BYTES_MAX the
    first views that fit are written."""
    import numpy as np
    x = images.detach().float().cpu().numpy()
    x = x[:max(1, DUMP_BYTES_MAX // (x[0].size * 4))]
    os.makedirs(out_dir, exist_ok=True)
    for name, sl in (('rgb', slice(0, 3)), ('depth', slice(3, 4)), ('acc', slice(4, 5))):
        np.save(os.path.join(out_dir, name + '.npy'), np.ascontiguousarray(x[..., sl]))


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'tensor_tflops': d.get('bf16_tflops_sustained', d['bf16_tflops']), 'src': 'measured (MEASURED_PEAKS.json, bf16 sustained)'}
    return {'hbm_gbs': 6650.0, 'tensor_tflops': 1400.0, 'src': 'fallback (B200_PROFILING.md)'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx, self.skip = [], None, gpu_index, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '5',
                                          '-i', str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 10.0 and self.proc.poll() is None:
                time.sleep(0.01)                      # NVML init takes ~0.5-1 s: it must be over BEFORE the timed region starts
        except Exception:
            self.proc = None

    def mark(self):
        """rows collected so far are idle-GPU samples; only later ones describe the timed region"""
        self.skip = len(self.rows)

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        self.rows = self.rows[self.skip:] or self.rows
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 8 and r[1].replace('.', '').isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 8 and r[2].replace('.', '').isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4:8]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def make_views(n_views, model):
    """One subject / observation, n_views novel target cameras.  Returns (base scene, list of per-view ray dicts), CPU tensors."""
    from sherf_b200 import synthetic as SY
    base = SY.make_scene(SY.SceneSpec(H=H, W=W, samples=S, seed=0, cam_azim_deg=25.0), model)
    views = [{k: base[k] for k in ('ray_origins', 'ray_directions', 'near', 'far')}]
    for v in range(1, n_views):
        sc = SY.make_scene(SY.SceneSpec(H=H, W=W, samples=S, seed=0, cam_azim_deg=25.0 + 360.0 * v / n_views), model, rays_only=True)
        views.append({k: sc[k] for k in ('ray_origins', 'ray_directions', 'near', 'far')})
    return base, views


def reference_cpu_rate(model, n_rays_target, threads, base=None, n_importance=0):
    """Times the reference's CPU path on a strided subset of the same 512x512x64 rays.  Where the reference's own files are available
    (oracle/_ref, materialised by oracle/make_ref.py, or /root/reference) this is the REFERENCE's own ImportanceRenderer.forward +
    NeRFDecoder + MipRayMarcher2, unmodified, under the shims of oracle/ref_shim.py (kind 'reference'; pytorch3d's knn_points is the
    shim's brute-force stand-in and dominates the time); otherwise the restatement oracle/port.py (kind 'port').
    Returns (rate, seconds, description, ray indices, outputs of those rays, importance draws, kind)."""
    import torch
    from sherf_b200 import synthetic as SY
    from sherf_b200 import dist as sd
    from sherf_b200.triplane import hot_path_modules
    from oracle import port, ref_shim
    torch.set_num_threads(threads)
    if base is None:
        base = SY.make_scene(SY.SceneSpec(H=H, W=W, samples=S, seed=0), model)
    stride = max(1, int(round((H * W / n_rays_target) ** 0.5)))
    idx = (torch.arange(0, H, stride)[:, None] * W + torch.arange(0, W, stride)[None, :]).reshape(-1)
    sub = dict(base)
    for k in ('ray_origins', 'ray_directions', 'near', 'far'):
        sub[k] = base[k][:, idx].contiguous()
    sub['rendering_options'] = dict(base['rendering_options'], depth_resolution_importance=n_importance)
    u = torch.rand(idx.numel(), n_importance, generator=torch.Generator().manual_seed(0)) if n_importance else None
    ren, dec = hot_path_modules(model, seed=0, dense_sigma=True)
    mt = SY.smpl_model_to_torch(model)
    if ref_shim.available():
        kind = 'reference'
        rren, rdec = ref_shim.build_reference(mt, 0)
        missing, unexpected = rren.load_state_dict({k: v for k, v in ren.state_dict().items() if not k.startswith('encoder_3d')}, strict=False)
        assert not unexpected, unexpected
        rdec.load_state_dict(dec.state_dict())
        t0 = time.perf_counter()
        out = ref_shim.render_importance(rren, rdec, sub, u) if n_importance else ref_shim.render(rren, rdec, sub)
        dt = time.perf_counter() - t0
    else:
        kind = 'port'
        wts = port.hot_path_state_dict(ren, dec)
        clamp = sd.depth_range(base['near'], base['far'], S)         # ray_marcher.py:57 is global over the full view
        t0 = time.perf_counter()
        out = port.render_forward(wts, mt, sub, importance_u=u, depth_clamp=clamp)
        dt = time.perf_counter() - t0
    n = idx.numel() * (S + n_importance)
    desc = f'{idx.numel()} rays (every {stride}th pixel in x and y of the 512x512 view) x {S + n_importance} samples = {n} ray-samples'
    return n / dt, dt, desc, idx, out, u, kind


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the path on the host cores (rank 0 only), each step a bounded sample
    of the same workload.  GPUs are hidden from this process, so the reference's hard-coded .cuda() calls are the identity (shim 3)."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    os.environ['CUDA_VISIBLE_DEVICES'] = ''
    import torch
    from sherf_b200 import synthetic as SY
    model = SY.make_smpl_model(0)
    threads = min(os.cpu_count() or 1, 32)      # the chunked brute-force KNN stand-in stops scaling (and regresses) beyond ~32 threads
    budget = 150.0 / max(1, args.steps + args.warmup)                 # seconds per step
    n_rays = args.ref_rays or int(min(16384, max(256, budget * 9000 / S)))      # ~9e3 ray-samples/s/8 cores measured in the build container
    base = SY.make_scene(SY.SceneSpec(H=H, W=W, samples=S, seed=0), model)
    rates, last, kind = [], None, 'port'
    for i in range(args.warmup + args.steps):
        rate, dt, sample, idx, out, u, kind = reference_cpu_rate(model, n_rays, threads, base, args.importance)
        if i >= args.warmup:
            rates.append((rate, dt))
        last = sample
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, torch.cat([out[0], out[1], out[2]], -1))
    if args.ref_dump:
        torch.save({'idx': idx, 'rgb': out[0], 'depth': out[1], 'acc': out[2], 'u': u, 'kind': kind, 'rate': rates[-1][0], 'seconds': rates[-1][1],
                    'sample': last, 'threads': threads}, args.ref_dump)
    value = sum(r for r, _ in rates) / len(rates)
    what = ('the reference\'s own ImportanceRenderer.forward + NeRFDecoder + MipRayMarcher2 (unmodified files under oracle/ref_shim.py; knn_points = brute-force stand-in for pytorch3d)'
            if kind == 'reference' else 'oracle/port.py (CPU restatement; the reference files were not available)')
    line = {
        'impl': 'reference', 'metric': 'ray_samples_per_sec', 'value': value, 'unit': 'ray-samples/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * sum(d for _, d in rates) / len(rates), 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': common_config(args.gpus, args.importance),
        'arm': {'what': what, 'step': 'bounded sample of the workload: ' + last, 'host_threads': threads},
        'cpu_baseline': {'value': value, 'unit': 'ray-samples/s', 'cores': threads, 'kind': kind, 'sample': last},
        'e2e': {'value': value, 'unit': 'ray-samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_subprocess(importance, n_rays=4096):
    """The bench's cpu_baseline leg: the reference arm in its OWN process (GPUs hidden, torch.Tensor.cuda shimmed there only), one
    step on `n_rays` rays; returns its dump (ray indices, outputs, rate)."""
    import tempfile
    import torch
    dump = os.path.join(tempfile.mkdtemp(prefix='sherf_ref_'), 'ref.pt')
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--ref-rays', str(n_rays),
           '--ref-dump', dump, '--importance', str(importance)]
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')}
    r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=1500)
    if r.returncode != 0 or not os.path.exists(dump):
        raise RuntimeError('reference arm failed: ' + r.stderr[-2000:])
    return torch.load(dump)


# Kernels of the point stages by library stage-timer index (include/sherf_b200.h: sherf_last_stage_ms): what bounds each, and its
# ALGORITHMIC work per surviving sample (DESIGN.md section 4).  The roofline object reports the one with the largest time share.
KERNELS = {
    2: dict(name='k_front_fused (warp + 3 gathers + conv1d_projection/reprojection + LayerNorm-1; tcgen05 kind::f16 bf16 split products)', bound='hbm',
            bytes_per_point=8 + 32 + 384 + 125,
            note='needed DRAM bytes per surviving sample: 8 B compacted index pair in, 32 B geometry + 384 B tokens out, ~125 B of first-touch feature lines (ncu dram read of the gather, profiles/); the 8 752 B of taps per sample are L2 -> SM traffic, not DRAM'),
    5: dict(name='k_decoder_pp (tcgen05 kind::f16 bf16 split products, whole NeRFDecoder, two 128-point tiles in flight per SM)', bound='tensor',
            flop_per_point=FLOP_PER_POINT_FUSED, issued=3),
    6: dict(name='k_xformer_bf16 (3-token transformer + decoder-input assembly; tcgen05 kind::f16 bf16 split products, two CTAs per SM)', bound='tensor',
            flop_per_point=2 * 25440, issued=3),
    7: dict(name='k_fusion_fused (conv1d_projection / reprojection + LayerNorm-1, tcgen05 kind::tf32 3xTF32)', bound='tensor', flop_per_point=2 * (18432 + 9216),
            issued=3, tf32=True),
}


def measured_traffic(kernel_key, points_per_launch):
    """DRAM bytes per launch of the named kernel from the committed ncu capture of this build (profiles/ncu_traffic.json, written by
    tools/ncu_traffic.py from `ncu --set full`: dram__bytes_read.sum + dram__bytes_write.sum); None when there is no capture."""
    p = os.path.join(ROOT, 'profiles', 'ncu_traffic.json')
    if not os.path.exists(p):
        return None, None
    d = json.load(open(p)).get(str(kernel_key))
    if not d:
        return None, None
    return d['dram_bytes_per_point'] * points_per_launch, d.get('source')


def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    import torch
    import torch.distributed as dist
    from sherf_b200 import synthetic as SY, _lib
    from sherf_b200 import dist as sd
    from sherf_b200.triplane import hot_path_modules

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    assert world == args.gpus or world == 1, f'--gpus {args.gpus} but WORLD_SIZE={world}'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.load()
    lib.sherf_set_profiling(1)

    model = SY.make_smpl_model(0)
    base, views = make_views(world, model)
    ren, dec = hot_path_modules(model, seed=0, mlp_precision=args.precision, dense_sigma=True)
    ren, dec = ren.to(dev), dec.to(dev)

    def mv(x):
        if torch.is_tensor(x):
            return x.to(dev)
        if isinstance(x, dict):
            return {k: mv(v) for k, v in x.items()}
        if isinstance(x, list):
            return [mv(v) for v in x]
        return x
    scene = {k: mv(v) for k, v in base.items()}
    scene['rendering_options']['depth_resolution_importance'] = args.importance      # draws: torch.rand on the device inside forward (renderer.py:526)
    N = H * W
    clamp = [sd.depth_range(v['near'], v['far'], S) for v in views]
    # this rank's tiles of every view (device resident for `value`, pinned host copies for `e2e`)
    by_tiles = world > 1 and args.shard == 'tiles'
    my_views = list(range(world)) if (by_tiles or world == 1) else [rank]
    idx = sd.shard_indices(N, rank, world) if by_tiles else torch.arange(N)
    shard_host = [{k: views[v][k][:, idx].contiguous().pin_memory() for k in views[v]} for v in my_views]
    shard_dev = [{k: t.to(dev) for k, t in sh.items()} for sh in shard_host]
    pose_host = {k: base['input_data'][k].pin_memory() for k in ('vertices',)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)                   # > 126 MB L2

    def render(sh, v, use_clamp=by_tiles):
        return ren(scene['planes'], scene['obs_input_img'], scene['obs_input_feature'], scene['volumes'], None, scene['obs_sp_input'],
                   dec, sh['ray_origins'], sh['ray_directions'], sh['near'], sh['far'], scene['input_data'], scene['rendering_options'],
                   depth_clamp=clamp[v] if use_clamp else None)

    stage_ms = [0.0] * 8
    host_us = [0.0] * 5             # C-side issue / sync / issue / total, and the Python wrapper around it
    launches = [0]
    points = [0]
    phase = {'render': [], 'collective': [], 'h2d': [], 'd2h': []}                  # (start, end) CUDA-event pairs, filled when `split` is on
    split = [False]
    overlap_gather = [False]                                                          # on only inside the device-timed loop

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    pending = []                                                                      # all-gathers in flight: (work, output, source)

    def drain_gathers():
        while pending:
            pending.pop(0)[0].wait()                                                    # the CURRENT STREAM waits (no host wait)

    def gather_views(local):
        """view-granular sharding: one all-gather of the rendered [N,5] tiles -> every rank holds all `world` images.  In the timed loop the
        all-gather of step i is left in flight while step i + 1 renders (views are independent; NCCL runs it on its own stream): the current
        stream only waits for it behind the NEXT render, and the last one is drained inside the last step's timed window."""
        full = local.new_empty(world * N, 5)
        src = local.contiguous()
        if split[0] or not overlap_gather[0]:
            drain_gathers()
            dist.all_gather_into_tensor(full, src)
            return full
        drain_gathers()                                                                 # step i - 1's gather: it had this step's render to finish
        pending.append((dist.all_gather_into_tensor(full, src, async_op=True), full, src))
        return full

    def step_device():
        outs = []
        for j, v in enumerate(my_views):
            t_py = time.perf_counter()
            a = ev() if split[0] else None
            rgb, depth, acc = render(shard_dev[j], v)
            host_us[4] += (time.perf_counter() - t_py) * 1e6
            for s_ in range(4):
                host_us[s_] += lib.sherf_last_host_us(s_)
            for s_ in range(8):
                stage_ms[s_] += lib.sherf_last_stage_ms(s_)
            launches[0] += ren.last_launches
            points[0] += ren.last_num_points
            local = torch.cat([rgb[0], depth[0], acc[0]], -1)
            b = ev() if split[0] else None
            outs.append(sd.all_gather_tiles(local, N) if by_tiles else (gather_views(local) if world > 1 else local))
            if split[0]:
                phase['render'].append((a, b))
                phase['collective'].append((b, ev()))
        return outs

    def step_e2e(host_out):
        """rays / near / far / posed vertices from pinned host memory -> device, render through the public API, all-gather, and this
        rank's OWN rendered view (the N ranks together: every image exactly once) -> pinned host memory."""
        for j, v in enumerate(my_views):
            a = ev() if split[0] else None
            sh = {k: t.to(dev, non_blocking=True) for k, t in shard_host[j].items()}
            scene['input_data']['vertices'] = pose_host['vertices'].to(dev, non_blocking=True)
            b = ev() if split[0] else None
            rgb, depth, acc = render(sh, v)
            local = torch.cat([rgb[0], depth[0], acc[0]], -1)
            c = ev() if split[0] else None
            if by_tiles:
                full = sd.all_gather_tiles(local, N)
                d = ev() if split[0] else None
                if v % world == rank:                                   # view v's assembled image is written out by one rank
                    host_out[v].copy_(full, non_blocking=True)
            elif world > 1:
                full = gather_views(local)
                d = ev() if split[0] else None
                host_out[rank].copy_(full[rank * N:(rank + 1) * N], non_blocking=True)
            else:
                d = c
                host_out[v].copy_(local, non_blocking=True)
            if split[0]:
                phase['h2d'].append((a, b)); phase['render'].append((b, c)); phase['collective'].append((c, d)); phase['d2h'].append((d, ev()))
        torch.cuda.current_stream().synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last_result = [None]                                                              # what the last step of the latest timed() returned

    def timed(fn, k):
        """k steps, each bracketed by CUDA events on the launching stream, L2 flushed between steps (outside the events).  The host does not
        wait for a step before it enqueues the next one (one synchronize after the k-th): launches are asynchronous in a real pipeline too,
        and with N ranks a per-step host wait turns every rank's host jitter into waiting time of its peers inside the all-gather
        (measured at N = 2: 3.36 ms per step against 3.0-3.05 ms of render + 0.1 ms of all-gather).  ImportanceRenderer.forward itself still
        waits for its survivor count inside every call; the end-to-end step reads its result on the host inside every step."""
        evs = []
        for i in range(k):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last_result[0] = fn()
            if i == k - 1:
                drain_gathers()                                                         # nothing escapes the K timed windows
            e1.record()
            evs.append((e0, e1))
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / k

    def phase_means():
        torch.cuda.synchronize()
        out = {k: (sum(a.elapsed_time(b) for a, b in v) / max(1, len(v)) * len(my_views)) for k, v in phase.items() if v}
        for v in phase.values():
            v.clear()
        return out

    for _ in range(args.warmup):
        step_device()
    # the timed steps run with the library's per-stage event timers OFF (they cost ~60 host-side event records per forward);
    # the stage split reported next to `value` comes from the same number of extra, untimed steps with the timers on
    lib.sherf_set_profiling(0)
    step_device()
    launches[0] = 0
    points[0] = 0
    host_us[:] = [0.0] * 5
    # clocks: ONE sampler (rank 0), started and past its NVML initialisation BEFORE the barrier that opens the timed region
    clocks = ClockSampler(local_rank) if rank == 0 else None
    if clocks:
        clocks.start()
    barrier()
    if clocks:
        clocks.mark()
    overlap_gather[0] = world > 1 and not by_tiles
    ms = timed(step_device, args.steps)
    # the images of the last timed step: [N, 5] per view rendered here, or [world * N, 5] all-gathered
    timed_images = torch.cat(last_result[0]).view(-1, N, 5)
    overlap_gather[0] = False
    barrier()
    clk = clocks.stop() if clocks else None
    n_launch_timed, n_points_timed = launches[0], points[0]
    host_timed = [h / (args.steps * len(my_views)) for h in host_us]
    # untimed extra steps: (a) per-phase CUDA events (render vs collective), (b) the library's per-stage timers
    split[0] = True
    for _ in range(args.steps):
        flush.zero_()
        step_device()
    split_dev = phase_means()
    split[0] = False
    lib.sherf_set_profiling(1)
    step_device()
    stage_ms[:] = [0.0] * 8
    for _ in range(args.steps):
        flush.zero_()
        step_device()
    launches[0], points[0] = n_launch_timed, n_points_timed
    lib.sherf_set_profiling(0)
    host_out = [torch.empty(N, 5).pin_memory() for _ in range(world)]
    for _ in range(args.warmup):
        step_e2e(host_out)
    barrier()
    ms_e2e = timed(lambda: step_e2e(host_out), args.steps)
    barrier()
    split[0] = True
    for _ in range(args.steps):
        flush.zero_()
        step_e2e(host_out)
    split_e2e = phase_means()
    split[0] = False

    # ---- N > 1: ONE view strong-scaled over all ranks in interleaved 256-ray tiles (sherf_b200.dist), checked on the hardware against
    #      the same view rendered by rank 0 alone: the gathered image must equal it bit for bit ----
    strong = None
    if world > 1 and not by_tiles:
        idx_t = sd.shard_indices(N, rank, world)
        sh_t = {k: views[0][k][:, idx_t].contiguous().to(dev) for k in views[0]}

        def one_view_sharded():
            rgb, depth, acc = render(sh_t, 0, use_clamp=True)
            return sd.all_gather_tiles(torch.cat([rgb[0], depth[0], acc[0]], -1), N)
        for _ in range(args.warmup):
            one_view_sharded()
        barrier()
        ms_t = timed(one_view_sharded, args.steps)
        barrier()
        img = one_view_sharded()
        full0 = {k: views[0][k].to(dev) for k in views[0]}
        r0 = render(full0, 0, use_clamp=False)
        ref_img = torch.cat([r0[0][0], r0[1][0], r0[2][0]], -1)
        for _ in range(2):
            render(full0, 0, use_clamp=False)
        ms_1 = timed(lambda: render(full0, 0, use_clamp=False), args.steps)
        same = bool(torch.equal(img, ref_img))
        tt = torch.tensor([ms_t, -ms_1 if rank else ms_1, 0.0 if same else 1.0], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        strong = {'what': f'view 0 (512x512x{S}) dealt to {world} ranks in interleaved 256-ray tiles, one all-gather of 20 B/ray', 'ms_per_view_sharded': float(tt[0]),
                  'ms_per_view_one_gpu': float(tt[1]), 'speedup': float(tt[1]) / float(tt[0]), 'efficiency': float(tt[1]) / float(tt[0]) / world,
                  'gathered_image_equals_single_gpu_render_bitwise_on_every_rank': float(tt[2]) == 0.0}

    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    per_rank = None
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        mine = {'rank': rank, 'step_ms': ms, 'device': split_dev, 'e2e_step_ms': ms_e2e, 'e2e': split_e2e}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
    ms, ms_e2e = float(t[0]), float(t[1])

    if rank == 0:
        pk = peaks()
        samples_per_step = world * N * (S + args.importance)
        calls = args.steps * len(my_views)
        mlp_ms = stage_ms[3] / calls
        p_call = points[0] / calls
        chunk_cap = int(os.environ.get('SHERF_CHUNK_CAP', 0)) or 524288       # api.cu chunk_cap_limit()
        n_launch = max(1, -(-int(p_call) // chunk_cap))
        per_stage = {i: stage_ms[i] / calls for i in range(8)}
        # ---- roofline of the kernel with the largest time share among the point-stage kernels ----
        cand = {k: per_stage[k] for k in KERNELS if per_stage[k] > 0}
        roof = None
        if cand:
            top = max(cand, key=cand.get)
            info, t_ms = KERNELS[top], cand[top]
            traffic, traffic_src = measured_traffic(top, p_call / n_launch)
            if info['bound'] == 'tensor':
                peak = pk['tensor_tflops'] * (TF32_OVER_BF16 if info.get('tf32') else 1.0)
                ach = p_call * info['flop_per_point'] / (t_ms * 1e-3) / 1e12
                roof = {'bound': 'tensor', 'kernel': info['name'], 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak,
                        'issued_frac': info['issued'] * ach / peak,
                        'algorithmic': f'{info["flop_per_point"]} FLOP per surviving sample x {p_call:.0f} samples per view; {n_launch} launches per view, avg {1e3 * t_ms / n_launch:.0f} us (CUDA events on the launching stream, stage timers)',
                        'peak_source': pk['src'] + (' x 0.5 (dense TF32 rate)' if info.get('tf32') else '') + '; useful FLOPs counted once, issued_frac counts the 3 MMAs of every split product'}
            else:
                ach = p_call * info['bytes_per_point'] / (t_ms * 1e-3) / 1e9
                roof = {'bound': 'hbm', 'kernel': info['name'], 'achieved': ach, 'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': ach / pk['hbm_gbs'],
                        'algorithmic': f'{info["bytes_per_point"]} B per surviving sample x {p_call:.0f} samples per view; {n_launch} launches per view, avg {1e3 * t_ms / n_launch:.0f} us (CUDA events on the launching stream, stage timers). {info["note"]}',
                        'peak_source': pk['src'].replace('bf16 sustained', 'STREAM-style copy'),
                        'l2_to_sm_GBps': p_call * GATHER_BYTES_PER_POINT / (t_ms * 1e-3) / 1e9}
            roof['time_share_of_step'] = t_ms * len(my_views) / ms if world == 1 else t_ms / ms
            roof['traffic'] = traffic
            roof['traffic_source'] = traffic_src
            # SURVEY 8(d)'s two PATH-level numbers: the whole step against the tensor and the HBM roofline
            decoded_per_s = p_call * len(my_views) / (ms * 1e-3) if world == 1 else p_call / (ms * 1e-3)
            needed = N * NEEDED_DRAM_BYTES_PER_RAY + p_call * NEEDED_DRAM_BYTES_PER_POINT + SCENE_BYTES
            roof['path'] = {'achieved_tensor': decoded_per_s * FLOP_PER_POINT / 1e12 / pk['tensor_tflops'],
                            'achieved_tensor_point_stages': (p_call * FLOP_PER_POINT / ((per_stage[2] + mlp_ms) * 1e-3) / 1e12 / pk['tensor_tflops']) if mlp_ms > 0 else None,
                            'achieved_hbm': needed / (ms / len(my_views) * 1e-3 if world == 1 else ms * 1e-3) / 1e9 / pk['hbm_gbs'],
                            'needed_dram_bytes_per_view': needed,
                            'note': 'achieved_tensor = decoded samples/s x 429 248 FLOP / measured bf16 peak (whole step; _point_stages: front + transformer + decoder kernels only -- the 429 248 FLOP include conv1d_projection / reprojection, which now run inside the front kernel next to the gathers); achieved_hbm = DRAM bytes the path needs per view / step time / measured copy bandwidth'}
        h2d_rank = sum(t_.numel() * 4 for sh in shard_host for t_ in sh.values()) + pose_host['vertices'].numel() * 4 * len(my_views)
        line = {
            'metric': 'ray_samples_per_sec', 'value': samples_per_step / (ms * 1e-3), 'unit': 'ray-samples/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': {'fp32': 'f32', 'tf32': 'tf32', 'tf32x3': 'tf32x3 (3xTF32 split products, fp32 accumulate; fp32-grade)',
                                                'bf16x3': 'bf16x3 (bf16 hi/lo split products on tcgen05 kind::f16, 16 significand bits per operand, fp32 accumulate) in every linear layer'}[args.precision],
            'data': 'synthetic',
            'config': common_config(world, args.importance),
            'arm': {'mlp_precision': args.precision, 'surviving_points_per_view': p_call * world if by_tiles else p_call,
                    'sharding': ('single GPU' if world == 1 else (f'256-ray tiles of every view dealt to {world} ranks, one all-gather per view' if by_tiles else
                                 f'view granularity (rank r renders view r), one all_gather_into_tensor of the rendered [N,5] tiles per step; in the device-timed loop the all-gather of step i overlaps the render of step i + 1 and the last one is drained inside the last timed window'))},
            'e2e': {'value': samples_per_step / (ms_e2e * 1e-3), 'unit': 'ray-samples/s', 'h2d_bytes_per_step': h2d_rank * world,
                    'd2h_bytes_per_step': world * N * 5 * 4, 'ms_per_step': ms_e2e,
                    'note': 'per step and rank: pinned-host rays/near/far/vertices -> device, ImportanceRenderer.forward via the C ABI, all-gather (N>1), the rank\'s own rendered rgb+depth+acc -> pinned host; bytes are totals over the ranks'},
            'gpu_launches': launches[0],
            'host_us_per_view_call': {'c_issue_until_sync': host_timed[0], 'c_blocked_in_sync': host_timed[1], 'c_issue_point_stages': host_timed[2],
                                      'c_total': host_timed[3], 'python_forward_total': host_timed[4],
                                      'note': 'timed steps are enqueued without a host wait between them: the host runs one step ahead of the GPU, so c_blocked_in_sync '
                                              '(the wait for the survivor-count event inside the call) is mostly the previous step still executing, not idle GPU time'},
            'clocks': clk,
            'stages_ms_per_view_call': {n: stage_ms[i] / calls for i, n in enumerate(['prologue+layout', 'cull+compact', 'front:warp+gather+fusion', 'point stages total', 'composite', 'mlp:decoder_kernel', 'mlp:transformer_kernel', 'mlp:fusion_kernel(legacy)'])},
            'point_stages_tflops': p_call * FLOP_PER_POINT / ((per_stage[2] + mlp_ms) * 1e-3) / 1e12 if mlp_ms > 0 else 0.0,
            'roofline': roof,
            'decoded_samples_per_sec': points[0] / args.steps * world / (ms * 1e-3),      # surviving samples through the MLP stack (rank 0's count x ranks)
        }
        if per_rank is not None:
            line['per_rank_ms'] = per_rank
            slow = max(per_rank, key=lambda r_: r_['device'].get('render', 0.0))
            line['scaling_limiter'] = {'slowest_rank_render_ms': slow['device'].get('render'), 'max_collective_ms': max(r_['device'].get('collective', 0.0) for r_ in per_rank),
                                       'note': 'device split from untimed extra steps with per-phase CUDA events; collective_ms of a rank includes waiting for the slowest rank\'s render'}
        if strong is not None:
            line['strong_scaling_one_view'] = strong
        if world == 1 and not args.no_cpu_baseline:
            # the reference's own CPU implementation of the path, in its own process (GPUs hidden), on 4 096 rays of the same view
            ref = cpu_baseline_subprocess(args.importance)
            idx, u_sub = ref['idx'], ref['u']
            line['cpu_baseline'] = {'value': ref['rate'], 'unit': 'ray-samples/s', 'cores': ref['threads'], 'kind': ref['kind'], 'sample': ref['sample'], 'seconds': ref['seconds']}
            # BASELINE.json's second metric: PSNR of our image against the reference's, on the rays the reference just rendered
            # (outside the timed region; the full 262 144-ray reference image would take the CPU ~20 minutes)
            import math
            u_full = None
            if args.importance:
                u_full = torch.rand(N, args.importance, device=dev)
                u_full[idx.to(dev)] = u_sub.to(dev)
            got = ren(scene['planes'], scene['obs_input_img'], scene['obs_input_feature'], scene['volumes'], None, scene['obs_sp_input'], dec,
                      shard_dev[0]['ray_origins'], shard_dev[0]['ray_directions'], shard_dev[0]['near'], shard_dev[0]['far'],
                      scene['input_data'], scene['rendering_options'], importance_u=u_full)[0][0].cpu()[idx]
            ref_img = ref['rgb'][0]
            hit = base['mask_at_box'].reshape(-1)[idx].bool()

            def psnr(a, b):
                mse = float(((a - b) ** 2).mean()) if a.numel() else 0.0
                return round(10 * math.log10(4.0 / max(mse, 1e-20)), 2)               # images span (-1, 1)
            line['psnr_vs_reference'] = {'all_pixels_db': psnr(got, ref_img), 'mask_at_box_db': psnr(got[hit], ref_img[hit]),
                                         'pixels': int(idx.numel()), 'mask_at_box_pixels': int(hit.sum()),
                                         'rgb_linf': float((got - ref_img).abs().max()), 'against': ref['kind'],
                                         'note': 'our render vs the cpu_baseline arm\'s image on its ray sample (test_loop.py:36-37,222-223 metric)'}
        if world == 1 and not args.importance and not args.no_training_step:
            # the training use of the same path (SURVEY 8 f2), outside the timed region: forward + the reference's reconstruction loss
            # (loss.py:150-151,167) + loss.backward() with every hot-path parameter and the five feature tensors requiring grad
            import copy
            ren_t, dec_t = copy.deepcopy(ren).train().requires_grad_(True), copy.deepcopy(dec).train().requires_grad_(True)
            leaves = [scene['planes'].clone().requires_grad_(True), scene['obs_input_feature'].clone().requires_grad_(True)] + \
                     [v.clone().requires_grad_(True) for v in scene['volumes']]
            tgt = torch.rand(1, N, 3, device=dev)

            def train_step():
                rgb, depth, acc = ren_t(leaves[0], scene['obs_input_img'], leaves[1], leaves[2:], None, scene['obs_sp_input'], dec_t,
                                        shard_dev[0]['ray_origins'], shard_dev[0]['ray_directions'], shard_dev[0]['near'], shard_dev[0]['far'],
                                        scene['input_data'], scene['rendering_options'])
                loss = 100 * ((rgb / 2 + 0.5 - tgt) ** 2).mean() + 10 * ((acc - 1) ** 2).mean()
                loss.backward()
                return loss
            for _ in range(2):
                train_step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                loss_t = train_step()
            e1.record()
            e1.synchronize()
            ms_t = e0.elapsed_time(e1) / 3
            line['training_step'] = {'ms_per_view': ms_t, 'ray_samples_per_sec': N * S / (ms_t * 1e-3), 'backward_launches': getattr(ren_t, 'last_backward_launches', None),
                                     'loss': float(loss_t), 'gradients': '39 hot-path parameters + tri-planes + 2-D feature map + 3 volume levels',
                                     'arithmetic': 'recompute-in-backward; GEMMs 3xTF32 on tcgen05 (csrc/backward_umma.cu, mlp_umma.cu)',
                                     'note': 'forward + loss (loss.py:150-151,167) + loss.backward() through ImportanceRenderer.forward, same view and weights; '
                                             'CUDA-event timed over 3 steps after 2 warm-up steps, outside the timed region of `value`'}
            del ren_t, dec_t, leaves
        if world == 1 and args.gpu_eager_baseline:
            # BASELINE.md 3.4: "the reference on the same box in GPU-eager mode": the reference's own ImportanceRenderer.forward (oracle/_ref
            # under the shims; knn_points = chunked brute force where the real reference calls pytorch3d's CUDA KNN), eager PyTorch on this GPU
            from oracle import port, ref_shim
            mt = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in SY.smpl_model_to_torch(model).items()}
            sc_full = dict(scene)
            for k in ('ray_origins', 'ray_directions', 'near', 'far'):
                sc_full[k] = shard_dev[0][k]
            sc_full['rendering_options'] = dict(scene['rendering_options'], depth_resolution_importance=0)
            if ref_shim.available():
                kind = 'reference'
                rren, rdec = ref_shim.build_reference(mt, 0)
                rren.load_state_dict({k: v for k, v in ren.state_dict().items() if not k.startswith('encoder_3d')}, strict=False)
                rdec.load_state_dict(dec.state_dict())
                rren, rdec = rren.to(dev), rdec.to(dev)
                run_ref = lambda: ref_shim.render(rren, rdec, sc_full)
            else:
                kind = 'port'
                wts = {k: v.to(dev) for k, v in port.hot_path_state_dict(ren, dec).items()}
                run_ref = lambda: port.render_forward(wts, mt, sc_full)
            run_ref()                                                               # warm-up (cuBLAS / cuSOLVER handles, allocator)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            ref_out = run_ref()
            e1.record()
            e1.synchronize()
            secs = e0.elapsed_time(e1) * 1e-3
            ours = ren(scene['planes'], scene['obs_input_img'], scene['obs_input_feature'], scene['volumes'], None, scene['obs_sp_input'], dec,
                       shard_dev[0]['ray_origins'], shard_dev[0]['ray_directions'], shard_dev[0]['near'], shard_dev[0]['far'],
                       scene['input_data'], sc_full['rendering_options'])
            line['gpu_eager_baseline'] = {'value': N * S / secs, 'unit': 'ray-samples/s', 'seconds_per_view': secs, 'kind': kind,
                                          'what': 'the reference\'s own forward as eager PyTorch on this GPU, one full 512x512x64 view (brute-force knn stand-in)' if kind == 'reference'
                                          else 'oracle/port.py as eager PyTorch on this GPU, one full 512x512x64 view',
                                          'peak_mem_GB': torch.cuda.max_memory_allocated() / 1e9,
                                          'rgb_linf_vs_cuda_path_full_view': float((ours[0] - ref_out[0]).abs().max()),
                                          'acc_linf_vs_cuda_path_full_view': float((ours[2] - ref_out[2]).abs().max()),
                                          'rays_beyond_1e-4': float(((ours[0] - ref_out[0]).abs().amax(-1) > 1e-4).float().mean())}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, timed_images)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
