"""CPU tests of the checker itself: oracle/port.py against the golden fixtures made from the reference's own code: whole renders
(oracle/gen_golden.py) and single reference functions on fresh inputs (oracle/gen_golden_reference_calls.py)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_CASES, load_golden
from sherf_b200 import synthetic as S
from oracle import port, ref_shim
from oracle.gen_golden import checksum
from oracle.gen_golden_reference_calls import sample_index

SAMPLE_IMPORTANCE_ROWS = 50          # rays of each sample_importance case whose reference answer is stored


def reference_calls():
    from conftest import GOLDEN_DIR
    return np.load(os.path.join(GOLDEN_DIR, 'reference_oracle_calls.npz'))


@pytest.mark.parametrize('case', GOLDEN_CASES)
def test_port_matches_reference_golden(case, smpl_model, smpl_model_t):
    g = load_golden(case)
    scene = S.make_scene(g['scene_spec'], smpl_model)
    assert checksum(scene) == str(g['input_sha256']), 'synthetic scene is not bit-reproducible from its seed'
    rgb, depth, acc, st = port.render_forward(g['weights'], smpl_model_t, scene, return_stages=True)
    N, S_ = scene['ray_origins'].shape[1], g['scene_spec'].samples
    gold_mask = np.unpackbits(g['mask_bits'])[:N * S_].astype(bool)
    assert np.array_equal(st['mask'].numpy(), gold_mask)                      # bit-exact cull mask
    assert np.array_equal(st['id1'][st['sel']].numpy(), g['id1'].astype(np.int64))
    assert np.array_equal(st['id3'].numpy(), g['id3'].astype(np.int64))
    assert np.abs(st['can'].numpy() - g['can']).max() <= 2e-6
    assert np.abs(st['cdir'].numpy() - g['cdir']).max() <= 2e-6
    assert np.abs(st['uv'].numpy() - g['uv']).max() <= 5e-4
    k = g['f2d_head'].shape[0]
    assert np.abs(st['f2d'][:k].numpy() - g['f2d_head']).max() <= 5e-4     # = uv error x gradient of the N(0,1) map
    assert np.abs(st['f3d_raw'][:k].numpy() - g['f3raw_head']).max() <= 5e-4     # voxel-coordinate rounding x gradient of the N(0,1) volume
    assert np.abs(st['tok_post'][:k, :2].reshape(k, 64).numpy() - g['tok01_head']).max() <= 5e-4
    assert np.abs(st['sigma'].numpy() - g['sigma']).max() <= 1e-3
    assert np.abs(st['rgb'].numpy() - g['rgb_pts']).max() <= 1e-5
    assert np.abs(rgb[0].numpy() - g['rgb']).max() <= 1e-5
    assert np.abs(acc[0].numpy() - g['acc']).max() <= 1e-5
    assert np.abs(depth[0].numpy() - g['depth']).max() <= 1e-5


def test_port_matches_live_reference(smpl_model, smpl_model_t):
    """A fresh scene, not one of the render fixtures, through the reference's forward (weights: the seed-4 set stored with the importance
    fixture, density head scaled like every fixture)."""
    g, w = reference_calls(), load_golden('importance_28x20x16p12')['weights']
    scene = S.make_scene(S.SceneSpec(H=20, W=28, samples=12, seed=9, random_global_R=True), smpl_model)
    assert checksum(scene) == str(g['live/input_sha256'])
    got = port.render_forward(w, smpl_model_t, scene)
    for a, b in zip([g['live/rgb'], g['live/depth'], g['live/acc']], got):
        assert a.shape == tuple(b.shape)
        assert float(np.abs(a - b.numpy()).max()) <= 1e-5
    assert float(g['live/acc'].max()) > 0.2          # the body is actually visible


def test_port_importance_matches_golden(smpl_model, smpl_model_t):
    """SURVEY a13: coarse + fine pass.  The fixture comes from the repaired composition of the reference's own
    sample_importance / sample_pdf / unify_samples / ray marcher (oracle/ref_shim.render_importance)."""
    from oracle.gen_golden import importance_u
    g = load_golden('importance_28x20x16p12')
    scene = S.make_scene(g['scene_spec'], smpl_model)
    assert checksum(scene) == str(g['input_sha256'])
    n_imp = int(g['n_importance'])
    scene['rendering_options']['depth_resolution_importance'] = n_imp
    u = importance_u(scene['ray_origins'].shape[1], n_imp, int(g['u_seed']))
    rgb, depth, acc, st = port.render_forward(g['weights'], smpl_model_t, scene, return_stages=True, importance_u=u)
    assert np.abs(st['coarse_weights'].numpy() - g['coarse_weights']).max() <= 2e-6
    assert np.abs(st['t_fine'].numpy() - g['t_fine']).max() <= 5e-6
    assert np.array_equal(st['fine']['mask'].view(-1, n_imp).numpy(), g['sigma_fine'] != -80.0)       # fine cull mask
    assert np.abs(rgb[0].numpy() - g['rgb']).max() <= 1e-5
    assert np.abs(acc[0].numpy() - g['acc']).max() <= 1e-5
    assert np.abs(depth[0].numpy() - g['depth']).max() <= 1e-5


def test_port_importance_matches_live_reference(smpl_model, smpl_model_t):
    """A fresh scene through the reference's repaired coarse + fine pass (oracle/ref_shim.render_importance; weights: the seed-1 set stored with
    the ragged fixture)."""
    g, w = reference_calls(), load_golden('ragged_45x38x24_R_white')['weights']
    scene = S.make_scene(S.SceneSpec(H=18, W=22, samples=10, seed=17, white_back=True), smpl_model)
    assert checksum(scene) == str(g['live_importance/input_sha256'])
    scene['rendering_options']['depth_resolution_importance'] = 7
    u = torch.rand(18 * 22, 7, generator=torch.Generator().manual_seed(5))
    got = port.render_forward(w, smpl_model_t, scene, return_stages=True, importance_u=u)
    for a, b in zip([g['live_importance/rgb'], g['live_importance/depth'], g['live_importance/acc']], got[:3]):
        assert a.shape == tuple(b.shape)
        assert float(np.abs(a - b.numpy()).max()) <= 1e-5
    assert float(np.abs(g['live_importance/t_fine'] - got[3]['t_fine'].numpy()).max()) <= 5e-6


def test_sample_importance_properties():
    """Inverse-CDF sampling (renderer.py:483-542): samples stay inside the mid-point bins, follow the weights, and the bin
    index returned is searchsorted(right=True)."""
    depths = port.sample_depths(torch.tensor([1.0, 2.0]), torch.tensor([2.0, 4.0]), 8)
    w = torch.zeros(2, 8)
    w[0, 3] = 1.0                                   # all the mass on sample 3 of ray 0; ray 1 uniform
    u = torch.rand(2, 64, generator=torch.Generator().manual_seed(0))
    t, inds = port.sample_importance(depths, w, 64, u)
    mid = 0.5 * (depths[:, :-1] + depths[:, 1:])
    assert torch.all(t >= mid[:, :1] - 1e-6) and torch.all(t <= mid[:, -1:] + 1e-6)
    assert float(((t[0] > mid[0, 1]) & (t[0] < mid[0, 4])).float().mean()) > 0.9      # smoothing spreads the peak over 3 bins
    assert int(inds.min()) >= 1 and int(inds.max()) <= 6


def test_knn_tie_break_smallest_index():
    v = torch.tensor([[0., 0, 0], [1, 0, 0], [1, 0, 0], [0, 0, 0]])
    q = torch.tensor([[0.1, 0, 0], [0.9, 0, 0], [0.5, 0, 0]])
    d2, idx = port.knn1(q, v)
    assert idx.tolist() == [0, 1, 0]
    d2s, idxs, _ = ref_shim.knn_points_bruteforce(q[None], v[None])
    assert idxs[0, :, 0].tolist() == [0, 1, 0] and torch.equal(d2s[0, :, 0], d2)


def test_positional_encoding_layout():
    x = torch.tensor([[0.3, -0.2, 0.7]])
    e = port.positional_encoding(x, 2)[0]
    want = torch.cat([x[0], torch.sin(x[0]), torch.sin(x[0] + torch.pi * 0.5), torch.sin(2 * x[0]), torch.sin(2 * x[0] + torch.pi * 0.5)])
    assert torch.allclose(e, want, atol=1e-7)


def test_composite_background_and_clamp():
    depths = port.sample_depths(torch.tensor([0.0, 2.0]), torch.tensor([1.0, 3.0]), 4)
    colors = torch.zeros(2, 4, 3)
    sigma = torch.full((2, 4), -80.0)
    sigma[1, 1] = 50.0
    colors[1, 1] = torch.tensor([0.2, 0.4, 0.6])
    rgb, depth, w = port.composite(colors, sigma, depths, torch.tensor([[0., 0, 1], [0, 0, 2]]), white_back=False)
    assert torch.all(rgb[0] == -1) and float(depth[0]) == 3.0           # empty ray: nan -> inf -> clamp to max(depths)
    assert float(w[1].sum()) == pytest.approx(1.0, abs=1e-6)
    assert torch.allclose(rgb[1], torch.tensor([0.2, 0.4, 0.6]) * 2 - 1, atol=1e-5)


def sample_importance_inputs(S_, SF):
    """300 rays of random ray-marcher weights (every fourth ray all zero) and the uniform draws standing for torch.rand."""
    g = torch.Generator().manual_seed(S_ * 100 + SF)
    n = 300
    near = torch.rand(n, generator=g) + 0.5
    far = near + torch.rand(n, generator=g) * 2 + 0.1
    depths = port.sample_depths(near, far, S_)
    w = torch.rand(n, S_, generator=g) ** 6
    w[::4] = 0
    u = torch.rand(n, SF, generator=g)
    return near, far, depths, w, u


@pytest.mark.parametrize('S_,SF', [(16, 12), (64, 64), (5, 9)])
def test_sample_importance_matches_reference_function(S_, SF):
    """port.sample_importance against the reference's OWN sample_importance / sample_pdf (renderer.py:483-542) on random ray-marcher
    weights, with torch.rand (:526) returning the same draws: identical bins, depths to the last few ulp (the reference's answer is stored
    for a fixed sample of the rays)."""
    near, far, depths, w, u = sample_importance_inputs(S_, SF)
    want = torch.from_numpy(reference_calls()[f'sample_importance/{S_}_{SF}'])
    got, bins = port.sample_importance(depths, w, SF, u)
    assert float((got[sample_index(got.shape[0], SAMPLE_IMPORTANCE_ROWS, S_ * 100 + SF)] - want).abs().max()) <= 1e-6 * float((far - near).max())
    assert int(bins.min()) >= 1 and int(bins.max()) <= S_ - 2


def composite_inputs():
    """Random colours / densities / depths, incl. sigma = -80 "culled" samples and empty rays."""
    g = torch.Generator().manual_seed(11)
    n, S1, S2 = 200, 16, 12
    d1 = port.sample_depths(torch.rand(n, generator=g) + 0.5, torch.rand(n, generator=g) + 2.0, S1)
    d2 = d1[:, :1] + torch.rand(n, S2, generator=g) * (d1[:, -1:] - d1[:, :1])
    c1, c2 = torch.rand(n, S1, 3, generator=g), torch.rand(n, S2, 3, generator=g)
    s1, s2 = torch.randn(n, S1, generator=g) * 20, torch.randn(n, S2, generator=g) * 20
    s1[torch.rand(n, S1, generator=g) < 0.5] = -80.0
    s1[::7] = -80.0
    s2[::7] = -80.0
    rays_d = torch.randn(n, 3, generator=g)
    return d1, d2, c1, c2, s1, s2, rays_d


@pytest.mark.parametrize('white', [False, True])
def test_composite_and_unify_match_reference_functions(white):
    """port.composite == the reference's MipRayMarcher2 (ray_marcher.py:25-64) and port.unify_samples == ImportanceRenderer.unify_samples
    (renderer.py:446-456) on random colours / densities / depths (incl. sigma = -80 "culled" samples and empty rays).  unify_samples
    permutes the concatenated samples: the fixture holds the permutation it applied."""
    g = reference_calls()
    d1, d2, c1, c2, s1, s2, rays_d = composite_inputs()
    ref_rgb, ref_depth, ref_w = (torch.from_numpy(g[f'composite/{int(white)}/{k}']) for k in ('rgb', 'depth', 'weights'))
    rgb, depth, w = port.composite(c1, s1, d1, rays_d, white)
    assert float((rgb - ref_rgb).abs().max()) <= 1e-6 and float((w - ref_w).abs().max()) <= 1e-6
    assert torch.equal(depth, ref_depth)
    perm = torch.from_numpy(g['unify/permutation']).long()
    ad, as_ = torch.cat([d1, d2], 1).gather(1, perm), torch.cat([s1, s2], 1).gather(1, perm)
    ac = torch.cat([c1, c2], 1).gather(1, perm[..., None].expand(-1, -1, 3))
    pd, pc, ps = port.unify_samples(d1, c1, s1, d2, c2, s2)
    assert torch.equal(pd, ad) and torch.equal(pc, ac) and torch.equal(ps, as_)
    got2 = port.composite(pc, ps, pd, rays_d, white)
    assert float((got2[0] - torch.from_numpy(g[f'composite/{int(white)}/rgb_unified'])).abs().max()) <= 1e-6


def test_branch_free_erf_of_the_transformer_kernel():
    """csrc/xformer_bf16.cu: xb_erf -- the GELU's erf as 1 - exp(-|x| q(|x|)) with a degree-7 q on [0, 4].  The same fp32 arithmetic in numpy
    against scipy's erf: absolute error <= 2e-7 everywhere (the kernel's header states 1.6e-7), and the GELU built from it within 5e-7
    absolute of the exact one, and within 3e-7 relative for x > 0 (for x < 0 the `1 + erf` cancellation is the reference formula's own)."""
    import re
    from scipy.special import erf
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'sherf_b200', 'csrc', 'xformer_bf16.cu')).read()
    body = src[src.index('float xb_erf(float x)'):src.index('return copysignf')]
    coef = [np.float32(c) for c in re.findall(r'(-?\d+\.\d+(?:e-?\d+)?)f[;,)]', body) if c != '4.0']
    assert len(coef) == 8, coef
    x = np.linspace(-6, 6, 2000001).astype(np.float32)
    t = np.minimum(np.abs(x), np.float32(4.0))
    q = np.full_like(t, coef[0])
    for c in coef[1:]:
        q = (q * t + c).astype(np.float32)
    e = np.copysign((np.float32(1.0) - np.exp((-t * q).astype(np.float32)).astype(np.float32)).astype(np.float32), x)
    err = np.abs(e.astype(np.float64) - erf(x.astype(np.float64)))
    assert err.max() <= 2e-7, err.max()
    xs = x.astype(np.float64)
    g_ref = 0.5 * xs * (1 + erf(xs / np.sqrt(2)))
    arg = (x * np.float32(0.70710678118654752440)).astype(np.float32)
    ta = np.minimum(np.abs(arg), np.float32(4.0))
    qa = np.full_like(ta, coef[0])
    for c in coef[1:]:
        qa = (qa * ta + c).astype(np.float32)
    ea = np.copysign((np.float32(1.0) - np.exp((-ta * qa).astype(np.float32)).astype(np.float32)).astype(np.float32), arg)
    g = (np.float32(0.5) * x * (np.float32(1.0) + ea)).astype(np.float32)
    d = np.abs(g.astype(np.float64) - g_ref)
    assert d.max() <= 5e-7, d.max()
    big = np.abs(g_ref) > 1e-3
    assert (d[big] / np.abs(g_ref[big])).max() <= 2e-4          # the cancellation in 1 + erf(x) for x << 0 is the reference formula's own
    pos = xs > 0                                                # no cancellation on this side: fp32-grade relative accuracy
    assert (d[pos & big] / np.abs(g_ref[pos & big])).max() <= 3e-7


def test_training_step_fixture_is_complete_and_its_weights_regenerate():
    """tests/golden/training_step_32x32x16.npz (oracle/gen_golden_training.py: the reference's own synthesis + renderer + SparseConvNet + decoder in
    train(), loss.backward()): 80 parameter gradients + tri-planes + feature map, the volume-gradient taps of the three dense levels, BatchNorm
    statistics; the initial state it was produced from regenerates from the stored tensors + the encoder seed (checksum)."""
    import os
    import numpy as np
    from conftest import GOLDEN_DIR
    from oracle import sparse_encoder as SE
    from oracle.gen_golden_training import state_checksum
    from sherf_b200.renderer import SparseConvNet
    g = np.load(os.path.join(GOLDEN_DIR, 'training_step_32x32x16.npz'))
    grads = [k for k in g.files if k.startswith('g/') or k.startswith('gs/')]
    assert len(grads) == 39 + 39 + 2 + 2
    assert sum(k.split('/', 1)[1].startswith('renderer.encoder_3d.') for k in grads) == 39
    assert all(np.isfinite(g[k]).all() and np.abs(g[k]).max() > 0 for k in grads)
    for l in range(3):
        assert g[f'gvol{l}/zyx'].shape[0] == g[f'gvol{l}/g'].shape[0] > 100 and g[f'gvol{l}/g'].shape[1] == (32, 64, 96)[l]
    assert len([k for k in g.files if k.startswith('stat/')]) >= 13 * 3          # running mean / var / batch counter of every BatchNorm the step ran
    state = {k[2:]: torch.from_numpy(g[k]) for k in g.files if k.startswith('w/')}
    torch.manual_seed(0)
    enc = SparseConvNet(4)
    enc.load_state_dict(SE.random_state_dict(enc, int(g['enc_seed'])))
    state.update({'renderer.encoder_3d.' + k: v.clone() for k, v in enc.state_dict().items()})
    assert state_checksum(state) == str(g['state_sha256'])
