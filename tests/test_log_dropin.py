"""CPU: LoG's own code against this repository's drop-in modules, replayed from tests/golden/reference_log_dropin.npz.

The golden file records what LoG's `LoG/render/renderer.py` and `LoG/model/*`, run UNMODIFIED with `dropin/` on the path
and this repository's kernels on the CPU SIMT emulation, did with the drop-in: the class each module name LoG imports
binds to (renderer.py:1, 99-105), the settings `BaseRender.prepare` builds (:57-78), every keyword set `render()`
(:117-153) passes to `GaussianRasterizer.forward`, the image cotangent LoG's loss sent back, LoG's own
`TensorTree.traverse` results and LoG's own `SparseOptimizer.step` results (generator: tests/golden/make_dropin_golden.py,
which needs a LoG checkout).  Here the recorded calls are replayed against the current code: the rasteriser against the
fp64 oracle, the fused tree walk and the fused sparse Adam against LoG's recorded results."""
import importlib
import os
import types

import numpy as np
import pytest
import torch

from oracle import c_oracle, torch_dense as O
from util import device, rel

GOLD = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'reference_log_dropin.npz'))
TENSOR_FIELDS = ('bg', 'viewmatrix', 'projmatrix', 'campos')


def settings(p, dev):
    from log_b200 import GaussianRasterizationSettings
    s = {}
    for f in GaussianRasterizationSettings._fields:
        v = GOLD[f'{p}settings/{f}']
        s[f] = torch.from_numpy(v).to(dev) if f in TENSOR_FIELDS else v.item()
    return GaussianRasterizationSettings(**s)


def oracle_camera(p):
    s = settings(p, 'cpu')
    cam = O.make_camera(s.image_width, s.image_height)
    return cam._replace(tanfovx=s.tanfovx, tanfovy=s.tanfovy, scale_modifier=s.scale_modifier, sh_degree=s.sh_degree,
                        **{f: getattr(s, f).double() for f in TENSOR_FIELDS})


def call_names(p, kind):
    return sorted(k[len(p + kind) + 1:] for k in GOLD.files if k.startswith(p + kind + '/'))


def replay(p, dev, tensors=None):
    """Call the recorded class with the recorded keyword set; `tensors` replaces the recorded tensor values."""
    import log_b200.rasterizer as ours
    tensors = tensors or {k: torch.from_numpy(GOLD[f'{p}kw/{k}']) for k in call_names(p, 'kw')}
    kw = {k: v.to(dev).requires_grad_(bool(GOLD[f'{p}requires_grad/{k}'])) for k, v in tensors.items()}
    call = dict(kw, **{k: None for k in GOLD[p + 'none']}, **{k: GOLD[f'{p}flag/{k}'].item() for k in call_names(p, 'flag')})
    rast = getattr(ours, str(GOLD[p + 'class']))(settings(p, dev))
    out = rast(**call)
    assert len(out) == int(GOLD[p + 'num_out'])
    return out, kw


def filter_mode(p):
    if str(GOLD[p + 'class']) == 'StockGaussianRasterizer':
        return c_oracle.FILTER_ADD
    return c_oracle.FILTER_NONE if (p + 'flag/use_filter' in GOLD.files and not GOLD[p + 'flag/use_filter']) else c_oracle.FILTER_MAX


def check_against_oracle(p, out, kw, G, image_bound=1e-4, grad_bound=2e-4):
    """The replayed call's outputs and (with cotangent G) the gradients returned into LoG's tensors vs the fp64 oracle."""
    d = {k: v.detach().cpu().double() for k, v in kw.items()}
    ref = c_oracle.render(oracle_camera(p), d['means3D'], d['opacities'], d['scales'], d['rotations'], colors_precomp=d['colors_precomp'],
                          filter_mode=filter_mode(p), dL_dimage=None if G is None else G.double(), dtype=np.float64)
    assert rel(out[0], ref['image']) < image_bound
    assert (out[1].cpu().numpy() != ref['radii']).sum() <= 1
    if len(out) == 5:
        assert (out[2].cpu().numpy() != ref['point_id_pixel']).sum() <= 2
        assert rel(out[4], ref['point_weight']) < 1e-4
    if G is not None:
        (out[0] * G.to(out[0].device)).sum().backward()
        pairs = [(n_, g_) for n_, g_ in (('means2D', 'dmeans2D'), ('means3D', 'dmeans3D'), ('colors_precomp', 'dcolors'),
                                         ('opacities', 'dopacities'), ('scales', 'dscales'), ('rotations', 'drotations')) if kw[n_].requires_grad]
        # LoG initialises isotropic scales, for which d loss / d rotation is exactly zero, and stays near-isotropic: there
        # fp32 arithmetic itself cannot reach the bound, which becomes twice the fp32 oracle's own error
        ref32 = c_oracle.render(oracle_camera(p), d['means3D'], d['opacities'], d['scales'], d['rotations'], colors_precomp=d['colors_precomp'],
                                filter_mode=filter_mode(p), dL_dimage=G.double(), dtype=np.float32)
        for name, grad in pairs:
            assert rel(kw[name].grad.reshape(ref[grad].shape), ref[grad]) < max(grad_bound, 2 * rel(ref32[grad], ref[grad])), name
    return ref


def test_reference_renderer_binds_to_dropin():
    import log_b200.rasterizer as ours
    for module, cls in zip(GOLD['bind/modules'], GOLD['bind/classes']):
        m = importlib.import_module(str(module))
        assert m.GaussianRasterizer is getattr(ours, str(cls))
        assert m.GaussianRasterizationSettings is ours.GaussianRasterizationSettings
    assert list(GOLD['bind/classes']) == ['GaussianRasterizer', 'StockGaussianRasterizer']
    s = settings('bind/', 'cpu')
    assert (s.image_width, s.image_height, s.sh_degree, s.prefiltered, s.debug) == (64, 48, 0, False, False)
    assert abs(s.tanfovx - 0.5463024898) < 1e-6
    assert ours.GaussianRasterizer(s).raster_settings is s


def test_reference_render_reaches_our_forward_with_its_own_kwargs(built):
    """CPU tensors: our forward must be reached (no TypeError on the keyword set, including use_filter=False for the
    fork in eval mode, renderer.py:151-152) and must refuse loudly instead of computing on the CPU."""
    from log_b200._capi import LgrError
    p = 'cpu_refusal/call0/'
    assert GOLD[p + 'flag/use_filter'].item() is False and str(GOLD[p + 'class']) == 'GaussianRasterizer'
    with pytest.raises(LgrError, match='no CPU fallback'):
        replay(p, 'cpu')


@pytest.mark.parametrize('origin,training', [(False, True), (False, False), (True, True)])
def test_reference_render_end_to_end_on_the_emulated_backend(emulated_backend, origin, training):
    """LoG's render() with this repo's rasteriser behind it, replayed on the CPU SIMT emulation: the flavour and filter it
    selected (fork + filter in training, fork without filter in eval :151-152, stock with use_origin_render), the image,
    radii, point_id / point_count (as LoG's renderer derived them) and point_weight equal the oracle's, and the gradient
    into viewspace_points (read at counter.py:40) is filled."""
    name = f'render_origin{int(origin)}_training{int(training)}'
    p = f'{name}/call0/'
    W, H, n = 64, 48, 300
    sc = {k: v.to(torch.float32) for k, v in O.make_scene(n, W, H, 4.0, seed=12).items()}
    tensors = {'means3D': sc['means3D'], 'means2D': torch.zeros(n, 3), 'colors_precomp': sc['colors'], 'opacities': sc['opacities'],
               'scales': sc['scales'], 'rotations': sc['rotations']}
    assert sorted(tensors) == call_names(p, 'kw_sum')
    for k, v in tensors.items():      # the scene LoG was given is the one regenerated here
        assert tuple(v.shape) == tuple(GOLD[f'{p}kw_shape/{k}']) and abs(float(v.double().sum()) - float(GOLD[f'{p}kw_sum/{k}'])) < 1e-9
    assert str(GOLD[p + 'class']) == ('StockGaussianRasterizer' if origin else 'GaussianRasterizer')
    assert filter_mode(p) == (c_oracle.FILTER_ADD if origin else c_oracle.FILTER_MAX if training else c_oracle.FILTER_NONE)
    G = O.make_cotangent(3, H, W).to(torch.float32)
    out, kw = replay(p, device(), tensors)
    ref = check_against_oracle(p, out, kw, G)
    if not origin:
        ids, cnt = np.unique(ref['point_id_pixel'], return_counts=True)
        keep = ids >= 0
        pid, pcount = GOLD[f'{name}/ret/point_id'], GOLD[f'{name}/ret/point_count']
        assert (pid != ids[keep]).sum() <= 2 if len(pid) == keep.sum() else False
        assert abs(int(pcount.sum()) - int(cnt[keep].sum())) <= 3
        got_ids, got_cnt = np.unique(out[2].cpu().numpy(), return_counts=True)
        assert np.array_equal(got_ids[got_ids >= 0], pid) and np.array_equal(got_cnt[got_ids >= 0], pcount)
    assert float(kw['means2D'].grad.abs().sum()) > 0


def walk_objects(p, dev):
    """Stand-ins for LoG's TensorTree / Gaussian / rasteriser: the attributes log_b200.tree.traverse reads."""
    max_child, max_level = (int(x) for x in GOLD[p + 'tree_args'])
    t = lambda k: torch.from_numpy(GOLD[p + k]).to(dev)
    tree = types.SimpleNamespace(node_index=t('node_index'), tree=t('tree'), max_child=max_child, max_level=max_level)
    model = types.SimpleNamespace(xyz=t('xyz'), scaling=t('scaling'), rotation=t('rotation'),
                                  activation=types.SimpleNamespace(scaling_activation=torch.exp))
    return tree, model, types.SimpleNamespace(raster_settings=settings(p, dev))


def check_walk(p_tree, p_query):
    from log_b200.tree import traverse
    dev = device()
    tree, model, rast = walk_objects(p_tree, dev)
    tree.min_resolution_pixel, max_depth = GOLD[p_query + 'args']
    got = traverse(tree, model, torch.from_numpy(GOLD[p_query + 'roots']).long().to(dev), rast, max_depth=int(max_depth))
    assert got.dtype == torch.int64
    assert np.array_equal(got.cpu().numpy(), GOLD[p_query + 'want']), p_query
    return got


def test_fused_tree_walk_equals_the_reference_traverse_call_path(emulated_backend):
    """LoG's own `TensorTree.traverse` driving its own `Gaussian.compute_radius` (level_of_gaussian.py:64-93, with
    dropin/LoG_cuda/compute_radius.py underneath) against `log_b200.tree.traverse` on the same objects: identical index
    tensors, also when many nodes are culled (radius 0)."""
    nq = GOLD['walk/num_queries']
    assert len(nq) == 2 and nq.sum() >= 4
    for t, q in ((t, q) for t in range(len(nq)) for q in range(int(nq[t]))):
        check_walk(f'walk/tree{t}/', f'walk/tree{t}/q{q}/')


def check_loop_calls(scenario):
    """Every kept rasteriser call of a LoG training loop, with the cotangent LoG's loss sent back, against the oracle."""
    for i in GOLD[f'{scenario}/calls_kept']:
        p = f'{scenario}/call{i}/'
        assert str(GOLD[p + 'class']) == 'GaussianRasterizer' and filter_mode(p) == c_oracle.FILTER_MAX
        out, kw = replay(p, device())
        check_against_oracle(p, out, kw, torch.from_numpy(GOLD[p + 'grad_image']).float())


def test_log_training_loop_in_miniature(emulated_backend):
    """BASELINE config 3 in miniature: LoG's OWN classes -- `LoG` / `GaussianPoint` / `TensorTree` / `Counter` /
    `SparseOptimizer` (LoG/model/level_of_gaussian.py) and `NaiveRendererAndLoss` (LoG/render/renderer.py) -- drove five
    training iterations as `Trainer.training_step` does (LoG/utils/trainer.py:144-166: render, loss.backward(),
    update_by_output, step) with this repo's rasteriser behind them; when recorded, the loss fell at every step and the
    first loss equalled LoG's loss of the ORACLE's image.  Replayed: the last iteration's rasteriser call, image and every
    gradient LoG received (with the cotangent LoG's loss sent back, stored at half precision), against the oracle."""
    assert list(GOLD['loop/calls_kept']) == [4] and int(GOLD['loop/num_calls']) == 5
    check_loop_calls('loop')


def test_log_training_loop_with_tree_nodes_and_the_fused_walk(emulated_backend):
    """The same loop taken into LoG's depth stage: `upgrade_tree`, `update_depth_stage` (LoG's own Splitter creates child
    nodes), then training continues through `LoG.prepare` -> `render_to_check` -> `TensorTree.traverse`
    (level_of_gaussian.py:223-257).  `log_b200.tree.traverse` returns exactly the tensor LoG's own traverse returned
    (first and last walk), and the last rasteriser call matches the oracle."""
    walks = GOLD['deep/walks_kept']
    assert int(GOLD['deep/num_walks']) == 4 and list(walks) == [0, 3]
    for w in walks:
        got = check_walk(f'deep/walk{w}/', f'deep/walk{w}/')
        assert got.numel() > 0 and int(GOLD[f'deep/walk{w}/node_index'].shape[0]) > 300
    check_loop_calls('deep')


def test_log_training_loop_with_the_fused_sparse_adam(emulated_backend):
    """`SparseOptimizer.step` (LoG/model/sparse_optimizer.py:163-196: gather state, `_single_tensor_adam`, scatter back)
    replaced by one `sparse_adam_step_` per parameter, as INTEGRATION.md describes: for each of LoG's five steps and each
    parameter group, the rows of the parameter and both Adam moments equal LoG's own optimiser's (a seeded sample of the
    visible rows is stored; the rows left out are zero and must stay zero)."""
    from log_b200.optim import sparse_adam_step_
    dev = device()
    assert int(GOLD['loop/num_steps']) == 5
    for s in range(5):
        keys = list(GOLD[f'loop/step{s}/keys'])
        assert {'xyz', 'scaling', 'opacity', 'rotation', 'colors'} <= set(keys)
        for key in keys:
            p = f'loop/step{s}/{key}/'
            step, lr, n = GOLD[p + 'hyper']
            rows = torch.from_numpy(GOLD[p + 'rows']).to(dev)
            full = {}
            for k in ('param', 'm', 'v'):
                a = GOLD[f'{p}{k}_in']
                full[k] = torch.zeros((int(n),) + a.shape[1:], dtype=torch.float32, device=dev)
                full[k][rows] = torch.from_numpy(a).to(dev)
            sparse_adam_step_(full['param'], torch.from_numpy(GOLD[p + 'grad']).to(dev), full['m'], full['v'], rows,
                              step=int(step), lr=float(lr), eps=1e-15)
            rest = torch.ones(int(n), dtype=torch.bool, device=dev)
            rest[rows] = False
            for k in ('param', 'm', 'v'):
                assert rel(full[k][rows], GOLD[f'{p}{k}_out']) < 2e-6, (s, key, k)
                assert not full[k][rest].any(), (s, key, k)
