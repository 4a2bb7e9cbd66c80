"""Nearest-vertex search: per-cell candidate lists against the grid searches, in one process, over the bench workload.

    python tools/bench_nn_lists.py [--importance 64] [--rounds 3] [--iters 20] [--modes lists,legacy] [--out FILE]

Renders bench.py's 512x512x64 view (same seeded inputs) and alternates the modes round by round: `legacy` sets SHERF_NN_LEGACY=1 (the
grid searches), `lists` clears it (the library reads the switch on every call).  Per mode it reports the library's per-stage CUDA-event
times (sherf_last_stage_ms, mean over the rounds), the kernel times of one profiled round (torch.profiler, summed per kernel name and
divided by the renders), and, for the list path, the list statistics of the last render (sherf_nn_list_stats: candidate samples of the
cull, sub-cells, mean / max list length, overflow fraction).  Prints one JSON object.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

STAGES = ['prologue+layout', 'cull+compact', 'front:warp+gather+fusion', 'point stages total', 'composite', 'mlp:decoder_kernel',
          'mlp:transformer_kernel', 'mlp:fusion_kernel(legacy)']
KERNELS = ['k_cull_candidates', 'k_cull_search', 'k_compact', 'k_front_fused', 'k_nnl_', 'k_grid_']


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--importance', type=int, default=0)
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--modes', default='lists,legacy')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    import torch
    from torch.profiler import profile, ProfilerActivity
    from sherf_b200 import synthetic as SY, _lib
    from sherf_b200.triplane import hot_path_modules
    import bench

    dev = torch.device('cuda', 0)
    lib = _lib.load()
    model = SY.make_smpl_model(0)
    base, _ = bench.make_views(1, model)
    ren, dec = hot_path_modules(model, seed=0, mlp_precision='bf16x3', dense_sigma=True)
    ren, dec = ren.to(dev), dec.to(dev)

    def mv(x):
        if torch.is_tensor(x):
            return x.to(dev)
        if isinstance(x, dict):
            return {k: mv(v) for k, v in x.items()}
        if isinstance(x, list):
            return [mv(v) for v in x]
        return x
    sc = {k: mv(v) for k, v in base.items()}
    sc['rendering_options']['depth_resolution_importance'] = args.importance

    def render():
        return ren(sc['planes'], sc['obs_input_img'], sc['obs_input_feature'], sc['volumes'], None, sc['obs_sp_input'], dec,
                   sc['ray_origins'], sc['ray_directions'], sc['near'], sc['far'], sc['input_data'], sc['rendering_options'])

    stats_fn = getattr(lib, 'sherf_nn_list_stats', None)
    if stats_fn is not None:
        stats_fn.restype = ctypes.c_int
        stats_fn.argtypes = [ctypes.POINTER(ctypes.c_double)]

    def set_mode(m):
        if m == 'legacy':
            os.environ['SHERF_NN_LEGACY'] = '1'
        else:
            os.environ.pop('SHERF_NN_LEGACY', None)

    modes = args.modes.split(',')
    res = {m: {'stage_ms': [0.0] * 8, 'ms_per_render': [], 'kernels_us': {}, 'points': None} for m in modes}
    for m in modes:                                   # warm every mode
        set_mode(m)
        for _ in range(3):
            render()
    torch.cuda.synchronize()
    for r in range(args.rounds):
        for m in modes:
            set_mode(m)
            lib.sherf_set_profiling(1)
            for _ in range(args.iters):
                render()
                for s in range(8):
                    res[m]['stage_ms'][s] += lib.sherf_last_stage_ms(s) / (args.iters * args.rounds)
            lib.sherf_set_profiling(0)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                render()
            e1.record()
            torch.cuda.synchronize()
            res[m]['ms_per_render'].append(e0.elapsed_time(e1) / args.iters)
            res[m]['points'] = int(ren.last_num_points)
    for m in modes:
        set_mode(m)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(args.iters):
                render()
            torch.cuda.synchronize()
        k = {}
        for e in prof.key_averages():
            t = getattr(e, 'self_device_time_total', None)
            if t is None:
                t = getattr(e, 'self_cuda_time_total', 0.0)
            for pat in KERNELS:
                if pat in e.key and t > 0:
                    name = e.key.split('(')[0].replace('void ', '').replace('sherf::', '')
                    k[name] = k.get(name, 0.0) + t / args.iters
        res[m]['kernels_us'] = {n: round(v, 2) for n, v in sorted(k.items())}
        if m != 'legacy' and stats_fn is not None:
            render()
            torch.cuda.synchronize()
            buf = (ctypes.c_double * 16)()
            if stats_fn(buf) == 0:
                res[m]['list_stats'] = {'cull_candidates': buf[0], 'cull_subcells': buf[1], 'cull_mean_len': buf[2], 'cull_max_len': buf[3],
                                        'cull_overflow_frac': buf[4], 'canon_subcells': buf[5], 'canon_mean_len': buf[6],
                                        'canon_max_len': buf[7], 'canon_overflow_frac': buf[8], 'capacity': buf[9]}
        res[m]['stage_ms'] = {n: round(v, 4) for n, v in zip(STAGES, res[m]['stage_ms'])}
    set_mode(modes[0])
    out = {'gpu': torch.cuda.get_device_name(0), 'importance': args.importance, 'rounds': args.rounds, 'iters': args.iters, 'modes': res}
    try:
        import subprocess
        out['power_limit'] = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:  # noqa: BLE001
        out['power_limit'] = None
    line = json.dumps(out)
    print(line, flush=True)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
