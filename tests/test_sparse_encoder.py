"""Sparse 3-D encoder (SURVEY.md 8f rank 1).  "Parity unpinned" for the per-convolution rules: spconv 2.3.3 is absent, so the oracle states
its semantics (oracle/sparse_encoder.py, oracle/spconv_shim.py headers).  CPU: the gather-form oracle == the dense conv3d + activity-mask
formulation of the same network == the reference's OWN SparseConvNet.forward run on functional spconv stand-ins (its answers stored in
tests/golden/reference_sparse_encoder.npz by oracle/gen_golden_reference_calls.py).
GPU: sherf_sparse_encode (through SparseConvNet.forward) == the oracle; then the render path fed with a SparseConvTensor == the
render path fed with the oracle's dense volumes.  Tolerance: 2e-4 relative to each level's maximum (fp32, different summation order)."""
import json
import os

import numpy as np
import pytest
import torch

from sherf_b200 import synthetic as S
from oracle import sparse_encoder as SE
from oracle.gen_golden_reference_calls import sample_index


def reference_calls():
    from conftest import GOLDEN_DIR
    return np.load(os.path.join(GOLDEN_DIR, 'reference_sparse_encoder.npz'))


def _shell(n, shape, seed, dup=20):
    """Voxel coordinates on an ellipsoid shell (like SMPL vertices at 5 mm) with `dup` duplicated rows."""
    g = torch.Generator().manual_seed(seed)
    p = torch.randn(n, 3, generator=g)
    p = p / p.norm(dim=1, keepdim=True)
    half = torch.tensor([(s - 1) / 2.0 for s in shape])
    coord = torch.round(p * (half * 0.8) + half).int()
    coord = torch.cat([coord, coord[:dup]])
    feat = torch.randn(coord.shape[0], 32, generator=g)
    return coord, feat


def test_oracle_sparse_equals_dense_formulation():
    from sherf_b200.renderer import SparseConvNet
    torch.manual_seed(0)
    sd = SE.random_state_dict(SparseConvNet(4), 1)
    coord, feat = _shell(200, (32, 64, 64), 2)
    a = SE.encode_sparse(sd, coord, feat, (32, 64, 64))
    b = SE.encode_dense(sd, coord, feat, (32, 64, 64))
    assert [tuple(v.shape) for v in a] == [(1, 32, 16, 32, 32), (1, 64, 8, 16, 16), (1, 96, 4, 8, 8)]
    for x, y in zip(a, b):
        assert float((x - y).abs().max()) <= 2e-5 * float(x.abs().max())
        assert int((x != 0).any(1).sum()) > 20
    assert len(SE.conv_list()) == 13 and SE.conv_list()[2][2] == 'down'


FORWARD_CASES = [((32, 64, 64), 200, 2), ((32, 32, 96), 60, 9)]        # (spatial shape, voxels, seed)
FORWARD_ROWS = 16                                                      # grid points of each case whose reference output is stored


def forward_grid(seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(1, 1, 1, 700, 3, generator=g) * 2 - 1) * 0.95                   # renderer.py:336 hands [1,1,1,P,3]


def test_reference_sparse_conv_net_forward_under_the_functional_spconv_stand_ins():
    """The reference's OWN SparseConvNet (renderer.py:707-797: layer order, the `.dense()` taps, grid_sample, concatenation) runs on the
    spconv stand-ins of oracle/spconv_shim.py (dense conv3d formulation of the three spconv rules) and must agree with the gather-form oracle
    that the CUDA kernels are checked against.  Pins the network topology and the weight / BatchNorm bookkeeping on the reference's code; the
    per-convolution rules remain restated (spconv itself is absent): parity of f1 stays "unpinned" for them.  The reference's state-dict
    layout and its output features at FORWARD_ROWS grid points are stored."""
    import torch.nn.functional as F
    from sherf_b200.renderer import SparseConvNet
    g = reference_calls()
    ours = SparseConvNet(4)
    assert json.loads(str(g['state_dict_shapes'])) == [[k, list(v.shape)] for k, v in ours.state_dict().items()]
    sd = SE.random_state_dict(ours, 1)
    for i, (shape, n, seed) in enumerate(FORWARD_CASES):
        coord, feat = _shell(n, shape, seed)
        grid = forward_grid(seed)
        got = torch.from_numpy(g[f'forward{i}/rows'])                                     # [FORWARD_ROWS, 32 + 64 + 96]
        dense = SE.encode_sparse(sd, coord, feat, shape)
        feats = torch.cat([F.grid_sample(v, grid, padding_mode='zeros', align_corners=True) for v in dense], dim=1)
        want = feats.view(1, -1, feats.size(4)).transpose(1, 2)
        assert tuple(want.shape) == (1, 700, 192)
        assert int((want != 0).sum()) > 1000
        assert float((got - want[0, sample_index(700, FORWARD_ROWS, seed)]).abs().max()) <= 2e-5 * float(want.abs().max())


def test_duplicate_voxels_first_row_wins():
    coord = torch.tensor([[1, 2, 3], [4, 4, 4], [1, 2, 3]], dtype=torch.int32)
    feat = torch.arange(3 * 32, dtype=torch.float32).reshape(3, 32)
    c, f = SE.unique_voxels(coord, feat)
    assert c.tolist() == [[1, 2, 3], [4, 4, 4]] and torch.equal(f, feat[:2])


@pytest.mark.gpu
@pytest.mark.parametrize('shape,n,graph', [((32, 64, 64), 300, False), ((32, 32, 96), 40, False), ((16, 32, 32), 1500, False), ((32, 64, 64), 300, True)])
def test_cuda_encoder_against_oracle(shape, n, graph):
    """graph = False: the evaluation forward (torch.no_grad: convolutions as gathered linear layers on tcgen05, 3xTF32 split products).
    graph = True: eval() under autograd (parameters require grad): the differentiable kernels on the running statistics, fp32 FMA convolutions."""
    from sherf_b200.renderer import SparseConvNet, SparseConvTensor
    with torch.set_grad_enabled(graph):
        _encoder_against_oracle(shape, n, graph, SparseConvNet, SparseConvTensor)


def _encoder_against_oracle(shape, n, graph, SparseConvNet, SparseConvTensor):
    dev = torch.device('cuda:0')
    torch.manual_seed(0)
    enc = SparseConvNet(4)
    sd = SE.random_state_dict(enc, 3)
    enc.load_state_dict(sd)
    coord, feat = _shell(n, shape, 5)
    want = SE.encode_sparse(sd, coord, feat, shape)
    idx = torch.cat([torch.zeros(coord.shape[0], 1, dtype=torch.int32), coord], 1)
    got = enc.to(dev).eval()(SparseConvTensor(feat.to(dev), idx.to(dev), list(shape), 1))
    torch.cuda.synchronize()
    for lvl, (g, w) in enumerate(zip([v.detach() for v in got], want)):
        assert g.shape == w.shape
        err = float((g.cpu() - w).abs().max()) / float(w.abs().max())
        same_sites = bool(torch.equal((g.cpu() != 0).any(1), (w != 0).any(1)))
        print(f'\\n[sparse encoder {shape} level {lvl + 1}] active sites {int((w != 0).any(1).sum())}, max err / max = {err:.2e}, same sites {same_sites}')
        assert err <= 2e-4
    again = enc(SparseConvTensor(feat.to(dev), idx.to(dev), list(shape), 1))
    assert all(v.requires_grad == graph for v in got)
    assert all(torch.equal(a, b) for a, b in zip(got, again)), 'the encoder must be deterministic'


@pytest.mark.gpu
def test_render_from_sparse_tensor(smpl_model):
    """The reference's own call: ImportanceRenderer.forward(..., canonical_sp_conv_volume = SparseConvTensor, ...) (triplane.py:137,156).
    The sparse tensor is made like prepare_sp_input does (triplane.py:174-217) from the canonical vertices."""
    from conftest import scene_to
    from sherf_b200.renderer import SparseConvTensor
    from sherf_b200.triplane import hot_path_modules
    dev = torch.device('cuda:0')
    cpu_scene = S.make_scene(S.SceneSpec(H=32, W=32, samples=24, seed=3), smpl_model)
    scene = scene_to(cpu_scene, dev)
    ren, dec = hot_path_modules(smpl_model, seed=0, dense_sigma=True)
    sd = SE.random_state_dict(ren.encoder_3d, 7)
    ren.encoder_3d.load_state_dict(sd)
    tv = cpu_scene['input_data']['t_vertices'][0]
    bounds = cpu_scene['obs_sp_input']['bounds'][0]
    out_sh = cpu_scene['obs_sp_input']['out_sh']
    coord = torch.round((tv[:, [2, 1, 0]] - bounds[0][[2, 1, 0]]) / 0.005).to(torch.int32)          # triplane.py:193
    feat = torch.randn(coord.shape[0], 32, generator=torch.Generator().manual_seed(1))
    idx = torch.cat([torch.zeros(coord.shape[0], 1, dtype=torch.int32), coord], 1)
    ren, dec = ren.to(dev).eval(), dec.to(dev)
    sp = SparseConvTensor(feat.to(dev), idx.to(dev), out_sh, 1)

    def render(vol):
        return ren(scene['planes'], scene['obs_input_img'], scene['obs_input_feature'], vol, None, scene['obs_sp_input'], dec,
                   scene['ray_origins'], scene['ray_directions'], scene['near'], scene['far'], scene['input_data'], scene['rendering_options'])
    a = render(sp)
    vols = ren.encoder_3d(sp)
    assert [tuple(v.shape[1:]) for v in vols] == [(32, out_sh[0] // 2, out_sh[1] // 2, out_sh[2] // 2),
                                                 (64, out_sh[0] // 4, out_sh[1] // 4, out_sh[2] // 4), (96, out_sh[0] // 8, out_sh[1] // 8, out_sh[2] // 8)]
    b = render(vols)
    assert all(torch.equal(x, y) for x, y in zip(a, b))
    assert float(a[2].max()) > 0.2 and float(vols[0].abs().max()) > 0
    print(f'\\n[render from SparseConvTensor] {coord.shape[0]} vertices -> active level-1 sites {int((vols[0][0] != 0).any(0).sum())}')


# the third case is DENSE (every voxel has active neighbours on all sides, strided convolutions merge several inputs per output): the shells of
# the other cases mostly exercise the centre tap
TRAINING_CASES = [((32, 64, 64), 300, 20, True), ((32, 32, 96), 60, 0, True), ((16, 32, 32), 4000, 60, True), ((32, 64, 64), 260, 10, False)]
STRICT, GATE_FLIP_BOUND = 2e-4, 2e-2


@pytest.mark.gpu
def test_cuda_encoder_training_step_against_the_reference_module():
    """Four voxel sets (see _training_step_case).  Every gradient must be within STRICT = 2e-4 relative L2 (on B200: <= 4e-6 over whole gradients, <= 3.3e-5 over the stored samples) -- except that ONE
    case may sit in the gate-flip regime (<= 2e-2): among the ~ 1e5-1e6 ReLU units of a case the smallest |pre-activation| is ~ 1e-6 (computed
    on the reference), the same size as the fp32 summation-order differences between the two implementations; a unit that opens on one side
    only moves the gradients below it by ~ 1 / rows-per-channel (5.6e-3 seen with a fifth voxel set, n = 200 in eval(); tests/helpers/sparse_gate_counts.py prints
    both sides' per-layer gate counts).  The four sets below are flip-free on B200 with this build; the allowance covers a toolchain whose
    rounding differs."""
    worst = [_training_step_case(i, *case) for i, case in enumerate(TRAINING_CASES)]
    print('   worst gradient error per case: ' + '  '.join(f'{w:.1e}' for w in worst))
    assert all(w <= GATE_FLIP_BOUND for w in worst), worst
    assert sum(w > STRICT for w in worst) <= 1, worst


TRAINING_GRAD_SAMPLE = 128       # entries of each reference gradient that are stored (all of the smaller ones)
TRAINING_OUTPUT_ROWS = 8          # grid points of each case whose reference output features are stored


def training_inputs(shape, n, dup):
    coord, feat = _shell(n, shape, 13, dup=dup)
    idx = torch.cat([torch.zeros(coord.shape[0], 1, dtype=torch.int32), coord], 1)
    g = torch.Generator().manual_seed(17)
    grid = (torch.rand(1, 1, 1, 900, 3, generator=g) * 2 - 1) * 0.95
    cot = torch.randn(1, 900, 192, generator=g)
    return coord, feat, idx, grid, cot


def _training_step_case(i, shape, n, dup, train):
    """train(): batch-statistics BatchNorm, running-statistics update and the backward pass (sherf_sparse_encode_train / _backward) against
    torch autograd through the REFERENCE's own SparseConvNet (renderer.py:707-797) in train() on the functional spconv stand-ins
    (oracle/spconv_shim.py; duplicate rows stay rows of the level-0 BatchNorms like in spconv).  Loss = <the features the reference forward
    returns (grid_sample of the three dense levels, renderer.py:764-785), a fixed random cotangent>.  Gradients: 13 conv weights, 26
    BatchNorm parameters, the input features.  Tolerance 2e-4 relative L2 (fp32, different summation orders; measured in the log).
    train = False: the same gradients in eval() (BatchNorm on its running statistics, which then do not move).
    The reference's answers are stored (oracle/gen_golden_reference_calls.py): the output features of TRAINING_OUTPUT_ROWS grid points and the
    norm of the whole output, TRAINING_GRAD_SAMPLE entries of each gradient, the running statistics after the step.
    (A ReLU unit whose pre-activation is zero to rounding can open on one side and stay shut on the other: with ~ 200 rows per level-3
    channel ONE such gate moves the gradients below it by ~ 5e-3 -- observed with n = 200, tests/helpers/sparse_gate_counts.py prints the per-layer gate counts.)"""
    import torch.nn.functional as F
    from sherf_b200.renderer import SparseConvNet, SparseConvTensor
    ref = reference_calls()
    dev = torch.device('cuda:0')
    torch.manual_seed(0)
    ours = SparseConvNet(4)
    ours.load_state_dict(SE.random_state_dict(ours, 7))
    coord, feat, idx, grid, cot = training_inputs(shape, n, dup)

    # ---- the CUDA path, train() ----
    ours = ours.to(dev).train(train).requires_grad_(True)
    f_our = feat.to(dev).requires_grad_(True)
    vols = ours(SparseConvTensor(f_our, idx.to(dev), list(shape), 1))
    assert all(v.requires_grad for v in vols)
    feats = torch.cat([F.grid_sample(v, grid.to(dev), padding_mode='zeros', align_corners=True) for v in vols], dim=1)
    out_our = feats.view(1, -1, feats.size(4)).transpose(1, 2)
    (out_our * cot.to(dev)).sum().backward()
    torch.cuda.synchronize()

    def rel(a, b):
        a, b = a.detach().double().cpu().reshape(-1), b.detach().double().cpu().reshape(-1)
        return float((a - b).norm() / (b.norm() + 1e-30))
    rows = sample_index(out_our.shape[1], TRAINING_OUTPUT_ROWS, 100 + i)
    e_out = rel(out_our[0, rows.to(dev)], torch.from_numpy(ref[f'train{i}/output_rows']))
    norm_ref = float(ref[f'train{i}/output_norm'])
    print(f'\n[sparse encoder {"train" if train else "eval"}() {shape} n={n} dup={dup}] output rel L2 {e_out:.2e}')
    assert e_out <= 2e-5
    assert abs(float(out_our.detach().double().norm()) - norm_ref) <= 2e-5 * norm_ref
    got = {k: p for k, p in ours.named_parameters() if not (k.startswith('down3') or k.startswith('conv4'))}
    assert json.loads(str(ref[f'train{i}/grad_names'])) == list(got) + ['input_features'] and len(got) == 39
    grads = {k: p.grad for k, p in got.items()}
    grads['input_features'] = f_our.grad
    want = torch.from_numpy(ref[f'train{i}/grads'])
    worst = 0.0
    errs = {}
    at = 0
    for j, (k, gr) in enumerate(grads.items()):
        assert gr is not None, k
        sel = sample_index(gr.numel(), TRAINING_GRAD_SAMPLE, 1000 * i + j)
        errs[k] = rel(gr.reshape(-1)[sel.to(dev)], want[at:at + sel.numel()])
        at += sel.numel()
        worst = max(worst, errs[k])
    assert at == want.numel()
    print('   ' + '  '.join(f'{k} {v:.1e}' for k, v in errs.items()))
    print(f'   worst gradient rel L2 (39 parameters + input features) {worst:.2e}')
    # running statistics after one step (momentum 0.01, unbiased variance) and the batch counter
    osd = ours.state_dict()
    names, flat = json.loads(str(ref[f'train{i}/stat_names'])), torch.from_numpy(ref[f'train{i}/stats'])
    assert len(names) == 13 * 3
    at = 0
    for k in names:
        v = flat[at:at + osd[k].numel()]
        at += osd[k].numel()
        if 'num_batches' in k:
            assert int(osd[k]) == int(v) == (1 if train else 0), k
        else:
            assert float((osd[k].cpu().reshape(-1) - v).abs().max()) <= 1e-5 * max(1.0, float(v.abs().max())), k
    assert at == flat.numel()
    # the layers the reference never evaluates for num_layers = 4 stay untouched
    assert all(p.grad is None for k, p in ours.named_parameters() if k.startswith('down3') or k.startswith('conv4'))
    return worst


def test_strided_sparse_conv_output_sites_known_answers():
    """Hand-derived output sites of SparseConv3d(k=3, stride=2, padding=1) -- the rule of a regular strided convolution restricted to active
    inputs (spconv `ops.get_conv_output_size` / `get_indice_pairs`): output o is active iff 2 o - 1 + k = p for an active input p, k in {0,1,2}.
      p = (0,0,0): only k = 1, o = 0                      -> 1 site
      p = (1,1,1): per axis (o, k) in {(0,2), (1,0)}      -> the 8 sites {0,1}^3
      p = (2,0,1): axis values 2 -> o = 1 (k = 1); 0 -> o = 0; 1 -> o in {0,1}   -> (1,0,0), (1,0,1)
    Both statements of the rule (the gather-form oracle and the functional spconv stand-in the reference module runs on) must produce them, with
    out[o] = sum of W[:, k] . in[p] over exactly those pairs."""
    from oracle import spconv_shim as SP
    shape = (4, 4, 4)
    cases = {(0, 0, 0): {(0, 0, 0)}, (1, 1, 1): {(a, b, c) for a in (0, 1) for b in (0, 1) for c in (0, 1)}, (2, 0, 1): {(1, 0, 0), (1, 0, 1)}}
    torch.manual_seed(0)
    conv = SP.SparseConv3d(2, 3, 3, 2, padding=1, bias=False)
    with torch.no_grad():
        conv.weight.copy_(torch.randn_like(conv.weight))
    for p, want_sites in cases.items():
        feat = torch.tensor([[1.0, -2.0]])
        x = SP.SparseConvTensor(feat, torch.tensor([[0, *p]]), list(shape), 1)
        with torch.no_grad():
            y = conv(x)
        got_sites = {tuple(r[1:]) for r in y.indices.tolist()}
        assert got_sites == want_sites, (p, got_sites)
        assert y.spatial_shape == [2, 2, 2]                              # floor((4 + 2 - 3) / 2) + 1
        for row, o in zip(y.features, [tuple(r[1:]) for r in y.indices.tolist()]):
            k = tuple(p[a] - 2 * o[a] + 1 for a in range(3))             # the one offset that links p to o
            assert all(0 <= kk <= 2 for kk in k)
            assert torch.allclose(row, conv.weight[:, k[0], k[1], k[2]] @ feat[0], atol=1e-6)
    # the same three inputs together through the gather-form oracle's site rule (first strided layer of the encoder: down0)
    from sherf_b200.renderer import SparseConvNet
    sd = SE.random_state_dict(SparseConvNet(4), 1)
    coord = torch.tensor(list(cases), dtype=torch.int32)
    vols = SE.encode_sparse(sd, coord, torch.randn(3, 32), (32, 32, 32))
    active = {tuple(i) for i in torch.nonzero((vols[0][0] != 0).any(0)).tolist()}
    assert active == set().union(*cases.values())
