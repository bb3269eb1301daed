"""Record how LoG's own code drives this repository's drop-in modules, as golden data for tests/test_log_dropin.py.

Usage:  python tests/golden/make_dropin_golden.py <root of a LoG checkout (the directory that contains LoG/)>

LoG's `LoG/render/renderer.py` and `LoG/model/*` run UNMODIFIED with `dropin/` on the path and this repository's kernels on
the CPU SIMT emulation (tests/emu), in the scenarios listed in `main()`.  Every call LoG makes into this repository is
recorded -- `GaussianRasterizer.forward` (settings, keyword arguments, outputs, the image cotangent that came back and the
gradients returned into LoG's tensors), `TensorTree.traverse` (LoG's own walk, beside which `log_b200.tree.traverse` is
checked) and `SparseOptimizer.step` (LoG's own optimiser, which `log_b200.optim.sparse_adam_step_` replaces) -- together
with what LoG's code made of the results.  The test replays the calls against the current code, so LoG's checkout is
needed only here.  Writes tests/golden/reference_log_dropin.npz.
"""
import importlib
import importlib.util
import os
import sys
import types

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, 'tests', 'emu'), os.path.join(ROOT, 'tests'), os.path.join(ROOT, 'dropin'), ROOT):
    if p not in sys.path:
        sys.path.insert(0, p)

SETTINGS_FIELDS = ('image_height', 'image_width', 'tanfovx', 'tanfovy', 'bg', 'scale_modifier', 'viewmatrix', 'projmatrix',
                   'sh_degree', 'campos', 'prefiltered', 'debug')
OUT = {}


def arr(t):
    return t.detach().cpu().numpy().copy() if torch.is_tensor(t) else np.asarray(t)


def put_settings(p, s):
    for f in SETTINGS_FIELDS:
        OUT[f'{p}settings/{f}'] = arr(getattr(s, f))


class RasterRecorder:
    """Wraps GaussianRasterizer.forward (both flavours): records every call under `<scenario>/call<i>/`."""

    def __init__(self):
        from log_b200.rasterizer import GaussianRasterizer
        self.cls, self.orig, self.scenario, self.n = GaussianRasterizer, GaussianRasterizer.forward, None, {}
        self.fingerprint_only = False      # inputs regenerated from seeds by the test: store sum and shape only
        rec = self

        def forward(self_, **kw):
            return rec.record(self_, kw)
        GaussianRasterizer.forward = forward

    def close(self):
        self.cls.forward = self.orig

    def record(self, rast, kw):
        if self.scenario is None:
            return self.orig(rast, **kw)
        i = self.n.get(self.scenario, 0)
        self.n[self.scenario] = i + 1
        p = f'{self.scenario}/call{i}/'
        OUT[p + 'class'] = np.array(type(rast).__name__)
        put_settings(p, rast.raster_settings)
        none, flags = [], {}
        for k, v in kw.items():
            if v is None:
                none.append(k)
            elif torch.is_tensor(v):
                if self.fingerprint_only:
                    OUT[p + f'kw_sum/{k}'] = np.array(float(v.detach().double().sum()))
                    OUT[p + f'kw_shape/{k}'] = np.array(v.shape)
                else:
                    OUT[p + f'kw/{k}'] = arr(v)
                OUT[p + f'requires_grad/{k}'] = np.array(v.requires_grad)
            else:
                flags[k] = v
        OUT[p + 'none'] = np.array(sorted(none), dtype=str)
        for k, v in flags.items():
            OUT[p + f'flag/{k}'] = np.array(v)
        out = self.orig(rast, **kw)
        OUT[p + 'num_out'] = np.array(len(out))
        if out[0].requires_grad and not self.fingerprint_only:      # the cotangent LoG's loss sends back (half precision:
            out[0].register_hook(lambda g: OUT.__setitem__(p + 'grad_image', arr(g).astype(np.float16)))      # an input to both sides)
        return out


def emulated(mp):
    """What tests/conftest.py:emulated_backend does."""
    import ctypes
    import build_emu
    import util
    from log_b200 import _capi
    mp.setattr(_capi, '_lib', _capi.bind(ctypes.CDLL(build_emu.build())))
    mp.setattr(_capi, 'current_stream', lambda device=None: None)
    mp.setattr(_capi, 'require_cuda', lambda t, name: None)
    mp.setattr(util, 'DEVICE', ['cpu'])


def load_log(mp, ref):
    """LoG's modules, with dropin/LoG_cuda/compute_radius.py in place of LoG's JIT-compiled module."""
    spec = importlib.util.spec_from_file_location('LoG.cuda.compute_radius', os.path.join(ROOT, 'dropin', 'LoG_cuda', 'compute_radius.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    mp.setitem(sys.modules, 'LoG.cuda.compute_radius', mod)
    mp.syspath_prepend(ref)
    return importlib.import_module('LoG.render.renderer'), importlib.import_module('LoG.model.level_of_gaussian')


def camera_dict():
    return {'FoVx': 1.0, 'FoVy': 0.8, 'image_height': 48, 'image_width': 64, 'world_view_transform': torch.eye(4),
            'full_proj_transform': torch.eye(4), 'camera_center': torch.zeros(3), 'K': torch.eye(3)}


def scenario_bind(R):
    """Which class each module name LoG imports resolves to (renderer.py:1, 99-105), and the settings prepare() builds."""
    mods, classes = [], []
    for origin in (False, True):
        R.NaiveRendererAndLoss(use_origin_render=origin)
        mods.append('diff_gaussian_rasterization' if origin else 'diff_gaussian_rasterization_wodilate')
        classes.append(R.BaseRender.GaussianRasterizer.__name__)
    OUT['bind/modules'], OUT['bind/classes'] = np.array(mods), np.array(classes)
    put_settings('bind/', R.BaseRender.prepare(camera_dict(), torch.zeros(3)).raster_settings)


def scenario_cpu_refusal(R, rec):
    """The fork in eval mode with CPU tensors: the keyword set LoG passes (renderer.py:141-153, use_filter=False)."""
    class Model:
        training = False
        visibility_flag = None
        empty_xyz = torch.zeros((0, 3))

        def get_all(self, camera, rasterizer, **kw):
            n = 5
            return {'xyz': torch.rand(n, 3), 'opacity': torch.rand(n, 1), 'colors': torch.rand(n, 3),
                    'scaling': torch.rand(n, 3), 'rotation': torch.nn.functional.normalize(torch.rand(n, 4))}
    from log_b200._capi import LgrError
    rr = R.NaiveRendererAndLoss(use_origin_render=False)
    rec.scenario = 'cpu_refusal'
    try:
        rr.render(camera_dict(), R.BaseRender.prepare(camera_dict(), torch.zeros(3)), Model())
        raise AssertionError('the CPU call was not refused')
    except LgrError as e:
        assert 'no CPU fallback' in str(e)
    rec.scenario = None


def scenario_render(R, rec, origin, training):
    """LoG's render() (renderer.py:117-205) on a 64x48 view of 300 points, then loss.backward() with a fixed cotangent."""
    from oracle import torch_dense as O
    from util import f32_camera
    W, H, n = 64, 48, 300
    cam = f32_camera(O.make_camera(W, H, bg=(0.0, 0.0, 0.0)))
    sc = {k: v.to(torch.float32) for k, v in O.make_scene(n, W, H, 4.0, seed=12).items()}
    camera = {'FoVx': 2 * np.arctan(cam.tanfovx), 'FoVy': 2 * np.arctan(cam.tanfovy), 'image_height': H, 'image_width': W,
              'world_view_transform': cam.viewmatrix.float(), 'full_proj_transform': cam.projmatrix.float(),
              'camera_center': cam.campos.float(), 'K': torch.eye(3)}

    class Model:
        visibility_flag = None
        empty_xyz = torch.zeros((0, 3))

        def get_all(self, camera, rasterizer, **kw):
            self.leaves = {k: v.clone().requires_grad_(True) for k, v in sc.items()}
            return {'xyz': self.leaves['means3D'], 'opacity': self.leaves['opacities'], 'colors': self.leaves['colors'],
                    'scaling': self.leaves['scales'], 'rotation': self.leaves['rotations']}
    model = Model()
    model.training = training
    rr = R.NaiveRendererAndLoss(use_origin_render=origin)
    rast = R.BaseRender.prepare(camera, torch.zeros(3))
    name = f'render_origin{int(origin)}_training{int(training)}'
    rec.scenario, rec.fingerprint_only = name, True
    ret, _ = rr.render(camera, rast, model)
    G = O.make_cotangent(3, H, W).to(torch.float32)
    (ret['render'] * G).sum().backward()
    rec.scenario, rec.fingerprint_only = None, False
    # what LoG's renderer derives from the 5-tuple (renderer.py:154-159); the rest of `ret` is the rasteriser's own output
    for k in ('point_id', 'point_count'):
        OUT[f'{name}/ret/{k}'] = arr(ret[k]).astype(np.int32)
    assert ret['viewspace_points'].grad is not None and float(ret['viewspace_points'].grad.abs().sum()) > 0


def put_tree(p, tree, g, rast):
    """What log_b200.tree.traverse reads of LoG's TensorTree, Gaussian and rasteriser."""
    OUT[p + 'node_index'], OUT[p + 'tree'] = arr(tree.node_index), arr(tree.tree)
    OUT[p + 'tree_args'] = np.array([tree.max_child, tree.max_level], dtype=np.int64)
    OUT[p + 'xyz'], OUT[p + 'scaling'], OUT[p + 'rotation'] = arr(g.xyz), arr(g.scaling), arr(g.rotation)
    put_settings(p, rast.raster_settings)


def put_query(p, min_px, max_depth, roots, want):
    OUT[p + 'args'] = np.array([min_px, max_depth], dtype=np.float64)
    OUT[p + 'roots'], OUT[p + 'want'] = arr(roots).astype(np.int32), arr(want).astype(np.int32)


def scenario_walk(L):
    """LoG's TensorTree.traverse driving its own Gaussian.compute_radius (level_of_gaussian.py:64-93), on trees built with
    its own initialize / split, including many culled nodes; queries whose radius sits within fp32 noise of the
    threshold are not recorded."""
    from log_b200 import GaussianRasterizationSettings, GaussianRasterizer
    from oracle import torch_dense as O
    TensorTree = importlib.import_module('LoG.model.tensor_tree').TensorTree
    rng = np.random.default_rng(3)
    cam = O.make_camera(160, 96)
    settings = GaussianRasterizationSettings(
        image_height=96, image_width=160, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=torch.zeros(3), scale_modifier=1.0,
        viewmatrix=cam.viewmatrix.float(), projmatrix=cam.projmatrix.float(), sh_degree=0, campos=cam.campos.float(),
        prefiltered=False, debug=False)
    rast = GaussianRasterizer(settings)
    num_queries = []
    for t, (max_child, n_root) in enumerate(((2, 120), (4, 15))):
        tree = TensorTree(max_child=max_child, max_level=20)
        tree.initialize(torch.zeros(n_root, 3))
        for rd in range(4):
            leaves = torch.where(tree.is_leaf & (tree.depth == rd))[0]
            tree.split(leaves[torch.from_numpy(rng.random(len(leaves)) < 0.6)])
        P = tree.num_points
        depth = tree.depth.numpy().astype(np.float64)
        z = rng.uniform(0.5, 10.0, P)
        g = L.Gaussian()
        g.xyz = torch.from_numpy(np.stack([rng.uniform(-2.0, 2.0, P) * cam.tanfovx * z, rng.uniform(-2.0, 2.0, P) * cam.tanfovy * z, z], -1)).float()
        sig = np.exp(rng.normal(np.log(12.0) - 1.0 * depth, 1.0)) / 3.0 * z / (160 / (2 * cam.tanfovx))
        g.scaling = torch.from_numpy(np.log(sig[:, None] * rng.uniform(0.3, 1.0, (P, 3)))).float()
        g.rotation = torch.from_numpy(rng.normal(size=(P, 4))).float()
        roots = torch.where(tree.is_root)[0]
        put_tree(f'walk/tree{t}/', tree, g, rast)
        q = 0
        for min_px, max_depth in ((3.0, 1000), (6.0, 2), (1.5, 1000)):
            tree.min_resolution_pixel = min_px
            want = tree.traverse(g, roots.long(), rast, max_depth=max_depth)
            r2d = g.compute_radius(want, rast)[1]
            assert (r2d == 0).sum() > 10                               # culled nodes are part of the case
            if (torch.abs(r2d[r2d > 0] / min_px - 1) < 1e-4).any():
                continue
            put_query(f'walk/tree{t}/q{q}/', min_px, max_depth, roots, want)
            q += 1
        num_queries.append(q)
    OUT['walk/num_queries'] = np.array(num_queries)


def miniature_log(mp, R, L, densify=None):
    """LoG's own model / renderer / batch for a 64x48 view of 300 points, as LoG's Trainer.training_step runs them
    (LoG/utils/trainer.py:144-166).  Stand-ins: simple_knn.distCUDA2 (CUDA-only, used once for the initial scales) and
    Tensor.cuda()."""
    from oracle import torch_dense as O

    def dist2(x):                                  # mean squared distance to the 3 nearest neighbours, as distCUDA2
        d = torch.cdist(x, x)
        d.fill_diagonal_(float('inf'))
        return (d.topk(3, largest=False).values ** 2).mean(-1)
    knn, knn_c = types.ModuleType('simple_knn'), types.ModuleType('simple_knn._C')
    knn_c.distCUDA2, knn._C = dist2, knn_c
    mp.setitem(sys.modules, 'simple_knn', knn)
    mp.setitem(sys.modules, 'simple_knn._C', knn_c)
    mp.setattr(torch.Tensor, 'cuda', lambda self, *a, **k: self)

    class AD(dict):
        __getattr__ = dict.__getitem__

    rng = np.random.default_rng(0)
    W, H, n = 64, 48, 300
    cam = O.make_camera(W, H)
    z = rng.uniform(2, 6, n)
    xyz = np.stack([rng.uniform(-1, 1, n) * cam.tanfovx * z, rng.uniform(-1, 1, n) * cam.tanfovy * z, z], -1).astype(np.float32)
    colors = rng.uniform(0, 1, (n, 3)).astype(np.float32)
    model = L.LoG(gaussian=dict(init_ply=dict(filename={'xyz': xyz, 'colors': colors}, scale3d=1., init_opacity=0.5), sh_degree=1, xyz_scale=1.),
                  tree=AD(max_child=2, max_level=5),
                  optimizer=AD(optimize_keys=['xyz', 'colors', 'scaling', 'opacity', 'rotation', 'shs'], opt_all_levels=True,
                               lr_dict=dict(xyz=0.00016, xyz_final=0.0000016, xyz_scale=1., colors=0.0025, shs=0.000125, scaling=0.005,
                                            opacity=0.05, rotation=0.001, max_steps=100)),
                  densify_and_remove=AD(dict(upgrade_sh_iter=10, densify_from_iter=1, densify_every_iter=1, upgrade_repeat=50), **(densify or {})),
                  use_view_correction=False)
    model.base_iter = 1
    model.training_setup()
    model.train()
    rend = R.NaiveRendererAndLoss(split='train')
    batch = {'camera': {'camera_center': cam.campos.float()[None], 'world_view_transform': cam.viewmatrix.float()[None],
                        'full_proj_transform': cam.projmatrix.float()[None], 'image_width': torch.tensor([W]), 'image_height': torch.tensor([H]),
                        'FoVx': torch.tensor([2 * np.arctan(cam.tanfovx)]), 'FoVy': torch.tensor([2 * np.arctan(cam.tanfovy)]),
                        'K': torch.eye(3)[None], 'R': torch.eye(3)[None], 'T': torch.zeros(1, 3, 1)},
             'image': torch.rand(1, H, W, 3, generator=torch.Generator().manual_seed(1)), 'index': torch.tensor([0])}
    return model, rend, batch


def train(model, rend, batch, iters):
    """Trainer.training_step (trainer.py:144-166): render, loss.backward(), update_by_output, step."""
    losses = []
    for _ in range(iters):
        model.clear()
        out = rend(batch, model)
        out['loss'].backward()
        model.update_by_output(out)
        model.step()
        losses.append(float(out['loss'].detach()))
    return losses, out


def scenario_loop(mp, R, L, rec):
    """BASELINE config 3 in miniature: five training iterations of LoG's own classes.  Kept: the rasteriser call of the
    last iteration, and every SparseOptimizer.step (sparse_optimizer.py:163-196) per parameter group on a
    seeded sample of the visible rows -- parameter, exp_avg and exp_avg_sq before and after, the gradient rows, the step
    count and the learning rate."""
    from oracle import c_oracle, torch_dense as O
    model, rend, batch = miniature_log(mp, R, L)
    opt, g = model.optimizer, model.gaussian
    orig_step, n_step = opt.step, [0]
    rng = np.random.default_rng(5)

    def step(gaussian, index, params, flag_vis):
        p = f'loop/step{n_step[0]}/'
        n_step[0] += 1
        before = {}
        for key, param in params.items():
            if param.grad is not None:
                before[key] = (arr(getattr(gaussian, key).data), arr(param.grad[flag_vis]), arr(opt.exp_avg[key]), arr(opt.exp_avg_sq[key]))
        orig_step(gaussian, index, params, flag_vis)
        steps, rows = int(opt.global_steps.item()), arr(index[flag_vis]).astype(np.int64)
        for key, (p_in, grad, m_in, v_in) in before.items():
            lr = opt.xyz_lr if key == 'xyz' else opt.scaling_scheduler_args(steps) if key == 'scaling' else opt.lr_dict[key]
            p_out, m_out, v_out = arr(getattr(gaussian, key).data), arr(opt.exp_avg[key]), arr(opt.exp_avg_sq[key])
            untouched = np.setdiff1d(np.arange(p_in.shape[0]), rows)
            assert np.array_equal(p_out[untouched], p_in[untouched]) and np.array_equal(m_out[untouched], m_in[untouched])
            s_ = np.sort(rng.choice(len(rows), min(16, len(rows)), replace=False))
            r_ = rows[s_]
            q = p + f'{key}/'
            OUT[q + 'rows'], OUT[q + 'grad'] = r_, grad[s_]
            OUT[q + 'hyper'] = np.array([steps, lr, p_in.shape[0]], dtype=np.float64)
            for k_, a_ in (('param_in', p_in), ('m_in', m_in), ('v_in', v_in), ('param_out', p_out), ('m_out', m_out), ('v_out', v_out)):
                OUT[q + k_] = a_[r_]
        OUT[p + 'keys'] = np.array(sorted(before), dtype=str)
    opt.step = step
    rec.scenario = 'loop'
    losses, _ = train(model, rend, batch, 5)
    rec.scenario = None
    assert all(b < a for a, b in zip(losses, losses[1:])), losses
    assert int(opt.global_steps.item()) == 5
    OUT['loop/num_steps'] = np.array(n_step[0])
    # the first loss is LoG's own loss (renderer.py:253-266) of the ORACLE's image of the same inputs
    kw = {k: torch.from_numpy(OUT[f'loop/call0/kw/{k}']).double() for k in ('means3D', 'opacities', 'scales', 'rotations', 'colors_precomp')}
    s0 = {f: torch.from_numpy(np.asarray(OUT[f'loop/call0/settings/{f}'])).double() for f in ('viewmatrix', 'projmatrix', 'campos', 'bg')}
    cam = O.make_camera(int(OUT['loop/call0/settings/image_width']), int(OUT['loop/call0/settings/image_height']))._replace(
        tanfovx=float(OUT['loop/call0/settings/tanfovx']), tanfovy=float(OUT['loop/call0/settings/tanfovy']), **s0)
    ref = c_oracle.render(cam, kw['means3D'], kw['opacities'], kw['scales'], kw['rotations'], colors_precomp=kw['colors_precomp'],
                          filter_mode=c_oracle.FILTER_MAX, dtype=np.float64)
    first = {}
    rend.calculate_loss(batch['image'].permute(0, 3, 1, 2), torch.from_numpy(ref['image']).float()[None], first)
    assert abs(losses[0] - float(first['loss'])) < 1e-5 * max(1.0, abs(losses[0])), (losses[0], float(first['loss']))
    keep_calls(rec, 'loop', (rec.n['loop'] - 1,))


def keep_calls(rec, scenario, keep, what='call'):
    """Drop the recorded calls of `scenario` other than `keep` (the golden file stays small)."""
    n = rec.n[scenario] if what == 'call' else int(OUT[f'{scenario}/num_walks'])
    for i in range(n):
        if i not in keep:
            for k in [k for k in OUT if k.startswith(f'{scenario}/{what}{i}/')]:
                del OUT[k]
    OUT[f'{scenario}/{what}s_kept'] = np.array(sorted(keep))


def scenario_deep(mp, R, L, rec):
    """The same loop taken into LoG's depth stage (upgrade_tree, update_depth_stage: LoG's Splitter creates child nodes),
    then four more iterations through LoG.prepare -> TensorTree.traverse (level_of_gaussian.py:223-257); every traverse
    call is recorded with LoG's own result."""
    model, rend, batch = miniature_log(mp, R, L, densify=dict(
        split_grad_thres=0.0, radius2d_thres=0, min_steps_split=0, remove_weights_thres=0.005, max_split_points=20000,
        sort_method='radii', scaling_decay=0.9))
    rec.scenario = 'deep'
    train(model, rend, batch, 3)
    model.set_stage('depth')
    model.upgrade_tree()
    train(model, rend, batch, 3)
    model.update_depth_stage(10)
    assert model.tree.num_nodes > 0 and model.num_points > 300
    orig, n_walk = model.tree.traverse, [0]

    def walk(g, root_index, rasterizer, max_depth=1000):
        want = orig(g, root_index, rasterizer, max_depth=max_depth)
        put_tree(f'deep/walk{n_walk[0]}/', model.tree, g, rasterizer)
        put_query(f'deep/walk{n_walk[0]}/', model.tree.min_resolution_pixel, max_depth, root_index, want)
        n_walk[0] += 1
        return want
    model.tree.traverse = walk
    losses, out = train(model, rend, batch, 4)
    rec.scenario = None
    assert losses[-1] < losses[0], losses
    assert out['visibility_flag'][0]['index_node'].numel() > 0       # parents and leaves are both in play
    OUT['deep/num_walks'] = np.array(n_walk[0])
    keep_calls(rec, 'deep', (rec.n['deep'] - 1,))
    keep_calls(rec, 'deep', (0, n_walk[0] - 1), what='walk')


def main(ref):
    assert os.path.isdir(os.path.join(ref, 'LoG')), f'{ref} holds no LoG/ directory'
    torch.manual_seed(0)
    rec = RasterRecorder()
    try:
        with pytest.MonkeyPatch.context() as mp:
            R, _ = load_log(mp, ref)
            scenario_bind(R)
            scenario_cpu_refusal(R, rec)
            emulated(mp)
            for origin, training in ((False, True), (False, False), (True, True)):
                scenario_render(R, rec, origin, training)
        for scenario in (scenario_walk, scenario_loop, scenario_deep):
            with pytest.MonkeyPatch.context() as mp:
                R, L = load_log(mp, ref)
                emulated(mp)
                if scenario is scenario_walk:
                    scenario(L)
                else:
                    scenario(mp, R, L, rec)
    finally:
        rec.close()
    for s, n in rec.n.items():
        OUT[f'{s}/num_calls'] = np.array(n)
    path = os.path.join(HERE, 'reference_log_dropin.npz')
    np.savez_compressed(path, **OUT)
    print('wrote', path, len(OUT), 'arrays,', os.path.getsize(path), 'bytes;', 'calls', rec.n)


if __name__ == '__main__':
    main(os.path.abspath(sys.argv[1]))
