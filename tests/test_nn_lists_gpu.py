"""GPU tests of the nearest-vertex candidate lists (common.cuh: NnLists): the cull's knn #1 and the front kernel's knn #3 over per-sub-cell
lists must choose exactly the vertices the grid searches choose (SHERF_NN_LEGACY=1), so the ids, the surviving points and the images
are bit-identical between the two.  Covers the bench-size view, other seeds / poses / azimuths, the importance pass, a list capacity of
one (every sub-cell overflows to the grid search) and exact ties between coincident vertices (the smallest id wins)."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import scene_to
from sherf_b200 import synthetic as S

pytestmark = pytest.mark.gpu


def render(ren, dec, scene, debug):
    torch.manual_seed(0)                     # the importance pass draws its uniforms on the device inside forward
    out = ren(scene['planes'], scene['obs_input_img'], scene['obs_input_feature'], scene['volumes'], None, scene['obs_sp_input'], dec,
              scene['ray_origins'], scene['ray_directions'], scene['near'], scene['far'], scene['input_data'], scene['rendering_options'],
              debug=debug)
    torch.cuda.synchronize()
    return out


def list_stats():
    from sherf_b200 import _lib
    buf = (ctypes.c_double * 16)()
    assert _lib.load().sherf_nn_list_stats(buf) == 0
    return {'candidates': buf[0], 'cull_subcells': buf[1], 'cull_overflow': buf[4], 'canon_subcells': buf[5], 'canon_overflow': buf[8],
            'cap': buf[9]}


def both_paths(monkeypatch, ren, dec, scene, cap=None):
    """(lists, legacy) runs of the same forward: (rgb, depth, acc), debug taps, list statistics of the list run."""
    res = []
    for legacy in (False, True):
        monkeypatch.delenv('SHERF_NN_LEGACY', raising=False)
        monkeypatch.delenv('SHERF_NN_LIST_CAP', raising=False)
        if legacy:
            monkeypatch.setenv('SHERF_NN_LEGACY', '1')
        elif cap is not None:
            monkeypatch.setenv('SHERF_NN_LIST_CAP', str(cap))
        dbg = {'max_feat_points': 1}
        out = render(ren, dec, scene, dbg)
        res.append((out, dbg, None if legacy else list_stats()))
    monkeypatch.delenv('SHERF_NN_LEGACY', raising=False)
    monkeypatch.delenv('SHERF_NN_LIST_CAP', raising=False)
    return res


def assert_same(a, b):
    (oa, da, _), (ob, db, _) = a, b
    assert da['num_points'] == db['num_points']
    assert torch.equal(da['sample_vid'], db['sample_vid']), 'knn #1 / cull mask'
    assert torch.equal(da['point_sample'], db['point_sample'])
    assert torch.equal(da['point_vid3'], db['point_vid3']), 'knn #3'
    for k in ('fine_sample_vid',):
        if k in da:
            assert torch.equal(da[k], db[k]), k
    for x, y in zip(oa, ob):
        assert torch.equal(x, y)


def modules(smpl_model, precision):
    from sherf_b200.triplane import hot_path_modules
    ren, dec = hot_path_modules(smpl_model, seed=0, mlp_precision=precision, dense_sigma=True)
    return ren.cuda(), dec.cuda()


def test_bench_view_lists_equal_legacy(monkeypatch, smpl_model):
    """bench.py's 512x512x64 view (bf16x3): identical ids and images; the lists are in use (few overflows, candidates queued)."""
    ren, dec = modules(smpl_model, 'bf16x3')
    scene = scene_to(S.make_scene(S.SceneSpec(H=512, W=512, samples=64, seed=0, cam_azim_deg=25.0), smpl_model), 'cuda')
    a, b = both_paths(monkeypatch, ren, dec, scene)
    assert_same(a, b)
    st = a[2]
    print('\n[512x512x64] list statistics', st)
    assert st['candidates'] > 0 and st['cull_subcells'] > 0 and st['canon_subcells'] > 0
    assert st['cull_overflow'] < 0.05 and st['canon_overflow'] < 0.5


@pytest.mark.parametrize('precision', ['bf16x3', 'fp32'])
@pytest.mark.parametrize('seed,azim,rgr,n_imp', [(1, 90.0, False, 0), (2, 200.0, True, 0), (3, -30.0, False, 32), (4, 140.0, True, 24)])
def test_other_views_lists_equal_legacy(monkeypatch, smpl_model, precision, seed, azim, rgr, n_imp):
    ren, dec = modules(smpl_model, precision)
    scene = scene_to(S.make_scene(S.SceneSpec(H=160, W=128, samples=48, seed=seed, cam_azim_deg=azim, random_global_R=rgr), smpl_model), 'cuda')
    scene['rendering_options']['depth_resolution_importance'] = n_imp
    a, b = both_paths(monkeypatch, ren, dec, scene)
    assert a[1]['num_points'] > 0
    assert_same(a, b)


@pytest.mark.parametrize('n_imp', [0, 32])
def test_capacity_one_overflows_to_grid_search(monkeypatch, smpl_model, n_imp):
    """SHERF_NN_LIST_CAP=1: (almost) every sub-cell overflows and its queries take the grid searches; results unchanged."""
    ren, dec = modules(smpl_model, 'bf16x3')
    scene = scene_to(S.make_scene(S.SceneSpec(H=160, W=128, samples=48, seed=5, cam_azim_deg=60.0), smpl_model), 'cuda')
    scene['rendering_options']['depth_resolution_importance'] = n_imp
    a, b = both_paths(monkeypatch, ren, dec, scene, cap=1)
    assert a[2]['cap'] == 1 and a[2]['cull_overflow'] > 0.3 and a[2]['canon_overflow'] > 0.3
    assert_same(a, b)


def test_exact_ties_smallest_id_wins(monkeypatch, smpl_model):
    """Vertex b = a + 1 gets every per-vertex row of vertex a (template, shape and pose blend shapes, skinning weights), for every 5th a:
    the two coincide in every pose, and both searches must return a, never b."""
    V = smpl_model['weights'].shape[0]
    m = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in smpl_model.items()}
    src = np.arange(0, V - 1, 5)
    dst = src + 1
    for k in ('v_template', 'shapedirs', 'posedirs', 'weights'):
        m[k][dst] = m[k][src]
    ren, dec = modules(m, 'bf16x3')
    cpu = S.make_scene(S.SceneSpec(H=192, W=192, samples=64, seed=0, cam_azim_deg=25.0), m)
    scene = scene_to(cpu, 'cuda')
    tv = cpu['input_data']['t_vertices'][0].numpy()
    pv = cpu['input_data']['vertices'][0].numpy()
    tied = dst[np.all(tv[dst] == tv[src], 1) & np.all(pv[dst] == pv[src], 1)]
    assert tied.size > 0.9 * dst.size
    a, b = both_paths(monkeypatch, ren, dec, scene)
    assert_same(a, b)
    dbg = a[1]
    vid1 = dbg['sample_vid'].cpu().numpy()
    vid3 = dbg['point_vid3'].cpu().numpy()
    srcs = src[np.isin(dst, tied)]
    assert np.isin(vid1[vid1 >= 0], srcs).any() and np.isin(vid3, srcs).any(), 'no tied vertex was chosen: the test would not test ties'
    assert not np.isin(vid1, tied).any() and not np.isin(vid3, tied).any()
