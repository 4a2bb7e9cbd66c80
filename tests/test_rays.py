"""Dataset-side ray setup (SURVEY.md 8f rank 3): sherf_generate_rays against the dataset's numpy code.

CPU: sherf_b200.synthetic.get_rays_np / near_far_np (the restatement that travels) == the reference's own get_rays /
get_near_far (RenderPeople_dataset.py:14-27, 68-101), bit for bit, on the answers stored in tests/golden/reference_dataset_calls.npz.
GPU: the CUDA kernel against the restatement -- origins / directions within 1 float32 ulp (fp64 inside, like numpy; BLAS
may fuse the 3-term dot products differently), hit mask equal except for rays grazing a box face within 1e-6, near / far
within 1e-6 relative on the common hits.
"""
import os

import numpy as np
import pytest
import torch

from sherf_b200 import synthetic as S
from oracle.gen_golden_reference_calls import sample_index

RAY_CASES = [(32, 48), (45, 31)]           # (H, W) of the cameras _camera(H, W, seed = case index) makes
RAY_SAMPLE = 256                           # pixels of each camera whose reference ray direction is stored
SMPL_VERTEX_SAMPLE = 512                   # vertices of each posed body whose reference answer is stored


def reference_calls():
    from conftest import GOLDEN_DIR
    return np.load(os.path.join(GOLDEN_DIR, 'reference_dataset_calls.npz'))


def _camera(H, W, seed):
    rng = np.random.default_rng(seed)
    a = rng.uniform(0, 2 * np.pi)
    centre = rng.uniform(-0.2, 0.2, 3)
    eye = centre + 3.0 * np.array([np.sin(a), 0.2, np.cos(a)])
    R, T = S._look_at(eye, centre)
    K = np.array([[1.2 * W, 0, W / 2], [0, 1.2 * W, H / 2], [0, 0, 1]], np.float64)
    bounds = np.stack([centre - np.array([0.5, 0.9, 0.3]), centre + np.array([0.5, 0.9, 0.3])], 0).astype(np.float32)
    return K, R, T, bounds


def test_restatement_matches_reference_dataset_code():
    g = reference_calls()
    for seed, (H, W) in enumerate(RAY_CASES):
        K, R, T, bounds = _camera(H, W, seed)
        ro2, rd2 = S.get_rays_np(H, W, K, R, T)
        assert np.array_equal(np.broadcast_to(g[f'rays{seed}/origin'], (H, W, 3)), ro2)
        assert np.array_equal(g[f'rays{seed}/dirs'], rd2.reshape(-1, 3)[sample_index(H * W, RAY_SAMPLE, seed).numpy()])
        # the reference fed its own rays to get_near_far; on the sampled pixels they are bit-identical to these
        o32, d32 = ro2.reshape(-1, 3).astype(np.float32), rd2.reshape(-1, 3).astype(np.float32)
        hit = np.unpackbits(g[f'rays{seed}/hit'])[:H * W].astype(bool)
        near, far = g[f'rays{seed}/near'], g[f'rays{seed}/far']
        n2, f2, h2 = S.near_far_np(bounds, o32.copy(), d32.copy())
        assert np.array_equal(hit, h2) and hit.any() and not hit.all()
        assert np.array_equal(near, n2[hit]) and np.array_equal(far, f2[hit])
        assert np.all(n2[~hit] == 0) and np.all(f2[~hit] == 1)                 # RenderPeople_dataset.py:129-134


@pytest.mark.gpu
@pytest.mark.parametrize('H,W', [(64, 64), (360, 640), (37, 53)])
def test_generate_rays_against_numpy(H, W):
    from sherf_b200.rays import generate_rays
    K, R, T, bounds = _camera(H, W, H * 1000 + W)
    out = generate_rays(H, W, K, R, T, bounds, 'cuda:0')
    ro, rd = S.get_rays_np(H, W, K, R, T)
    o32, d32 = ro.reshape(-1, 3).astype(np.float32), rd.reshape(-1, 3).astype(np.float32)
    near, far, hit = S.near_far_np(bounds, o32.copy(), d32.copy())
    go, gd = out['ray_o_all'][0, 0].cpu().numpy(), out['ray_d_all'][0, 0].cpu().numpy()
    gn, gf = out['near_all'][0, 0, :, 0].cpu().numpy(), out['far_all'][0, 0, :, 0].cpu().numpy()
    gh = out['mask_at_box_all'][0, 0].cpu().numpy()
    ulp = np.spacing(np.abs(d32).max())
    assert np.abs(go - o32).max() <= np.spacing(np.abs(o32).max())
    assert np.abs(gd - d32).max() <= ulp
    same = gh == hit
    both = gh & hit
    print(f'\n[{H}x{W}] exact dirs {float((gd == d32).mean()):.5f}, hit mask equal {float(same.mean()):.6f}, hits {int(hit.sum())}, '
          f'near rel {float((np.abs(gn - near)[both] / near[both]).max()):.2e}')
    assert same.mean() >= 0.9995 and hit.any() and not hit.all()
    assert (np.abs(gn - near)[both] / near[both]).max() <= 1e-6 and (np.abs(gf - far)[both] / far[both]).max() <= 1e-6
    assert np.all(gn[~gh] == 0) and np.all(gf[~gh] == 1)


@pytest.mark.gpu
def test_render_from_generated_rays(smpl_model):
    """End to end: rays made on the device feed ImportanceRenderer.forward and give the image of the host-made rays."""
    from conftest import scene_to
    from sherf_b200.rays import generate_rays
    from sherf_b200.triplane import hot_path_modules
    dev = torch.device('cuda:0')
    spec = S.SceneSpec(H=48, W=64, samples=24, seed=8)
    cpu_scene = S.make_scene(spec, smpl_model)
    cam = cpu_scene['camera']
    scene = scene_to(cpu_scene, dev)
    rays = generate_rays(spec.H, spec.W, cam['K'], cam['R'], cam['T'], cam['bounds'], dev)
    ren, dec = hot_path_modules(smpl_model, seed=0, dense_sigma=True)
    ren, dec = ren.to(dev), dec.to(dev)

    def render(o, d, n, f):
        return ren(scene['planes'], scene['obs_input_img'], scene['obs_input_feature'], scene['volumes'], None, scene['obs_sp_input'], dec,
                   o, d, n, f, scene['input_data'], scene['rendering_options'])
    a = render(scene['ray_origins'], scene['ray_directions'], scene['near'], scene['far'])
    b = render(rays['ray_o_all'][:, 0], rays['ray_d_all'][:, 0], rays['near_all'][:, 0], rays['far_all'][:, 0])
    assert float((rays['ray_d_all'][:, 0] - scene['ray_directions']).abs().max()) <= 1e-6
    bad = ((a[0] - b[0]).abs().amax(-1) > 1e-4).float().mean()
    assert float(bad) <= 2e-3 and float(a[2].max()) > 0.2


@pytest.mark.gpu
def test_render_sequence_single_gpu(smpl_model):
    """configs[3] in miniature on one GPU: a 3-frame novel-pose sequence of one observed subject streamed through
    dist.render_sequence (device-made rays, per-frame pose upload only) == rendering every frame from host-made rays."""
    from conftest import scene_to
    from sherf_b200 import dist as sd
    from sherf_b200.triplane import hot_path_modules
    dev = torch.device('cuda:0')
    H, W = 36, 64                                                   # 640x360 / 10
    static = S.make_scene(S.SceneSpec(H=H, W=W, samples=24, seed=8, random_global_R=True), smpl_model)
    frames, hosts = [], []
    for f in range(3):
        other = S.make_scene(S.SceneSpec(H=H, W=W, samples=24, seed=40 + f, random_global_R=True, cam_azim_deg=10.0 + 50 * f), smpl_model)
        frames.append({'params': other['input_data']['params'], 'vertices': other['input_data']['vertices'], 'camera': other['camera']})
        hosts.append(other)
    scene = scene_to(static, dev)
    ren, dec = hot_path_modules(smpl_model, seed=0, dense_sigma=True)
    ren, dec = ren.to(dev), dec.to(dev)
    outs = sd.render_sequence(ren, dec, scene, frames, H, W)
    assert len(outs) == 3
    for f, o in enumerate(outs):
        h = scene_to(hosts[f], dev)
        idt = dict(scene['input_data'])
        idt['params'], idt['vertices'] = h['input_data']['params'], h['input_data']['vertices']
        rgb, depth, acc = ren(scene['planes'], scene['obs_input_img'], scene['obs_input_feature'], scene['volumes'], None, scene['obs_sp_input'],
                              dec, h['ray_origins'], h['ray_directions'], h['near'], h['far'], idt, scene['rendering_options'])
        bad = ((o[:, :3] - rgb[0]).abs().amax(-1) > 1e-4).float().mean()
        assert float(bad) <= 2e-3, (f, float(bad))
        assert float(acc.max()) > 0.2


@pytest.mark.gpu
def test_sampler_writes_test_loop_style_outputs(smpl_model, tmp_path):
    """sherf_b200.sample.render_orbit (SURVEY 8f rank 4): novel views through the public API, files named and encoded like
    test_loop.py:197,218-222 writes its predictions."""
    from PIL import Image
    from conftest import scene_to
    from sherf_b200.sample import render_orbit, to8b
    from sherf_b200.triplane import hot_path_modules
    dev = torch.device('cuda:0')
    H = W = 32
    scene = scene_to(S.make_scene(S.SceneSpec(H=H, W=W, samples=16, seed=8), smpl_model), dev)
    ren, dec = hot_path_modules(smpl_model, seed=0, dense_sigma=True)
    outs = render_orbit(ren.to(dev), dec.to(dev), scene, 3, H, W, str(tmp_path), pose_index=7)
    assert len(outs) == 3 and all(o.shape == (H * W, 5) for o in outs)
    for v, o in enumerate(outs):
        png = np.asarray(Image.open(tmp_path / f'frame0007_view{v:04d}.png'))
        assert png.shape == (H, W, 3) and png.dtype == np.uint8
        assert np.array_equal(png, to8b((o[:, :3].reshape(H, W, 3) / 2 + 0.5).cpu().numpy()))
        assert np.array_equal(np.load(tmp_path / f'frame0007_view{v:04d}_acc.npy'), o[:, 4].reshape(H, W).cpu().numpy())
    assert float(torch.stack([o[:, 4].max() for o in outs]).max()) > 0.2          # the body is visible from the orbit


def smpl_inputs():
    """Three random (poses, shapes) of the synthetic body."""
    rng = np.random.default_rng(3)
    out = []
    for _ in range(3):
        poses = rng.normal(0, 0.3, 72).astype(np.float32)
        shapes = rng.normal(0, 0.7, 10).astype(np.float32)
        out.append((poses, shapes))
    return out


def test_smpl_forward_restatement_matches_reference_class(smpl_model):
    """synthetic.smpl_forward_np (what the GPU SMPL forward, sherf_smpl_vertices, is checked against) == the reference's own
    `SMPL.__call__` (sherf/smpl/smpl_numpy.py:46-98) on the synthetic body, loaded through its own pickle path (the reference's answer is
    stored for a fixed sample of the vertices)."""
    want = reference_calls()['smpl/vertices']
    idx = sample_index(S.V, SMPL_VERTEX_SAMPLE, 3).numpy()
    for (poses, shapes), w in zip(smpl_inputs(), want):
        got = S.smpl_forward_np(smpl_model, poses, shapes)[idx]
        assert np.abs(got - w).max() <= 2e-7, np.abs(got - w).max()   # cv2.Rodrigues rounds R to float32, the restatement keeps float64
