"""GPU parity: the CUDA path, called through the public GaussianRasterizer API (ctypes -> C ABI), against the oracle.

Tolerances (BASELINE.json north_star: "RGB and gradients within 1e-4 relative"):
  * float outputs: norm-wise relative error ||gpu - oracle|| / ||oracle|| <= 1e-4 against the float64 C oracle fed
    the same float32-rounded inputs.  (fp32 atomics make gradients non-bit-reproducible; element-wise relative error
    is meaningless on near-zero entries.)  The path computes in fp32 like the reference; where fp32 arithmetic itself
    cannot reach 1e-4 (e.g. d/d rotation of a nearly isotropic Gaussian under a white-noise cotangent cancels
    catastrophically) the bound is 4x the error of the SAME algorithm evaluated in plain fp32 on the CPU
    (the float32 build of the C oracle): tol = max(1e-4, 4 * err_fp32_oracle).
  * integer outputs (radii, point_id_pixel): exact, except where the deciding float lies on a rounding boundary
    (ceil of the radius / two almost equal weights); those cases are detected with the oracle and bounded.
The blend semantics themselves are this repo's restatement of the published algorithm (parity unpinned against
LoG's un-vendored binaries, see oracle/lgr_oracle.c header).
"""
import math
import os

import numpy as np
import pytest
import torch

from oracle import c_oracle, torch_dense as O
from util import device, f32_camera, rel, run_gpu

pytestmark = pytest.mark.gpu
TOL = 1e-4
GOLD = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'reference_geometry_sh.npz'))


def f32_scene(sc):
    return {k: v.to(torch.float32).to(torch.float64) for k, v in sc.items()}


def oracle(cam, sc, G, fm, deg, dtype=np.float64):
    kw = dict(colors_precomp=sc['colors']) if deg == 0 else dict(shs=sc['shs'])
    return c_oracle.render(cam, sc['means3D'], sc['opacities'], sc['scales'], sc['rotations'], filter_mode=fm,
                           dL_dimage=G, dtype=dtype, **kw)


def check_all(got, ref, deg, fork, n_pix, ref32=None, case=None, filter_on=True):
    """north_star's bound is 1e-4 relative (norm-wise) for RGB and every gradient, and it is what is enforced -- except
    where fp32 arithmetic itself cannot reach it: the oracle is also built in fp32 (same algorithm, plain C, no atomics),
    and where THAT build is further than 1e-4 from its own fp64 build (big splats: sigma 8 px and more; sub-pixel splats with
    the filter off), the bound is the fp32 oracle's own error -- i.e. the CUDA path must be at least as accurate as a
    straight fp32 restatement.  (Round 1 allowed 4 x that error.)  Every achieved error, the fp32 floor and the bound used
    are recorded (util.record_parity -> profiles/parity_rNN.json)."""
    def tol(k):      # 1.05: where one borderline fp32 decision dominates BOTH fp32 results, the two errors agree to 5 digits
        return TOL if ref32 is None else max(TOL, 1.05 * rel(ref32[k], ref[k]))
    errs = {}
    keys = ['image', 'dmeans3D', 'dmeans2D', 'dopacities', 'dscales', 'drotations'] + (['dcolors'] if deg == 0 else ['dshs'])
    if fork:
        keys += ['point_weight', 'point_weight_pixel']
    for k in keys:
        if k in got:
            errs[k] = (rel(got[k], ref[k]), None if ref32 is None else rel(ref32[k], ref[k]))
    if case is not None:
        from util import record_parity
        record_parity(case, errs, TOL, filter_on)
    rg, rr = np.asarray(got['radii'].cpu().numpy() if hasattr(got['radii'], 'cpu') else got['radii']), ref['radii']
    assert (rg != rr).sum() <= max(2, int(2e-4 * rr.size)), ((rg != rr).sum(), rr.size)
    assert np.abs(rg - rr).max() <= 1
    for k, (e, _) in errs.items():
        assert e < tol(k), (k, e, tol(k))
    if fork:
        pg = got['point_id_pixel']
        pg, pr = (pg.cpu().numpy() if hasattr(pg, 'cpu') else pg), ref['point_id_pixel']
        bad = pg != pr
        assert bad.sum() <= max(3, int(1e-3 * n_pix)), bad.sum()
        assert ((pg == -1) == (pr == -1)).mean() > 0.999


def borderline_decisions(cam, sc, fm, thr=1e-6):
    """(Gaussian ids, pixel ids) of the pairs with |alpha * 255 - 1| < thr in float64.  The rule
    `alpha < 1/255 -> skip` is a discontinuity: a pair sitting within fp32 round-off of it can legitimately be decided
    either way by two fp32 implementations, which moves that Gaussian's gradient by O(1%) and that pixel by O(0.004).
    Scenes with millions of low-opacity pairs always contain a few; they are excluded from the comparison by name."""
    pr = O.project(sc['means3D'], sc['scales'], sc['rotations'], cam, fm)
    H, W = cam.image_height, cam.image_width
    ys, xs = np.meshgrid(np.arange(H), np.arange(W), indexing='ij')
    xy, con, op = pr['xy'].numpy(), pr['conic'].numpy(), sc['opacities'].numpy().reshape(-1)
    gs, ps = [], []
    for i in np.nonzero(pr['valid'].numpy())[0]:
        dx, dy = xy[i, 0] - xs, xy[i, 1] - ys
        power = -0.5 * (con[i, 0] * dx * dx + con[i, 2] * dy * dy) - con[i, 1] * dx * dy
        near = np.abs(op[i] * np.exp(np.minimum(power, 0)) * 255 - 1) < thr
        if near.any():
            gs.append(int(i))
            ps.extend(np.nonzero(near.reshape(-1))[0].tolist())
    return np.array(gs, dtype=np.int64), np.array(sorted(set(ps)), dtype=np.int64)


def drop(d, gs, ps):
    """Copy of a result dict with the named Gaussian rows / pixels zeroed (numpy)."""
    out = {}
    for k, v in d.items():
        if v is None or np.isscalar(v):
            out[k] = v
            continue
        a = np.array(v.detach().cpu().numpy() if hasattr(v, 'detach') else v, copy=True)
        if k == 'image':
            a.reshape(3, -1)[:, ps] = 0
        elif k in ('point_weight_pixel', 'point_id_pixel', 'final_T'):
            a.reshape(-1)[ps] = 0
        elif a.ndim >= 1 and a.shape[0] == sc_n[0]:
            a[gs] = 0
        out[k] = a
    return out


sc_n = [0]


CASES = [
    # W, H, n, median sigma px, sh degree, flavour, use_filter, rotated camera
    (256, 256, 1000, 3.0, 0, 'fork', True, False),      # BASELINE config 0 shape
    (200, 120, 3000, 6.0, 0, 'stock', True, True),
    (333, 211, 5000, 2.0, 3, 'stock', True, True),      # non-multiple-of-16 image, SH degree 3
    (160, 96, 2000, 1.5, 2, 'fork', False, False),      # fork with use_filter=False
    (128, 128, 1500, 4.0, 1, 'fork', True, True),
    (96, 64, 400, 20.0, 0, 'fork', True, False),        # big splats: many tiles per Gaussian
]


@pytest.mark.parametrize('W,H,n,r,deg,flavour,use_filter,rot', CASES)
def test_forward_backward_parity(built, W, H, n, r, deg, flavour, use_filter, rot):
    kwc = dict(R=[[0.98, 0.0, 0.199], [0, 1, 0], [-0.199, 0, 0.98]], T=[0.1, -0.05, 0.3]) if rot else {}
    cam = f32_camera(O.make_camera(W, H, bg=(0.2, 0.5, 0.7), sh_degree=deg, **kwc))
    sc = f32_scene(O.make_scene(n, W, H, r, sh_degree=deg, seed=11))
    sc['means3D'][:5, 2] = -1.0
    sc['means3D'][5:10, 0] += 50
    sc['opacities'][10:14] = 0.001
    sc['opacities'][14:18] = 1.0
    G = O.make_cotangent(3, H, W).to(torch.float32).to(torch.float64)
    fm = O.FILTER_ADD if flavour == 'stock' else (O.FILTER_MAX if use_filter else O.FILTER_NONE)
    ref = oracle(cam, sc, G, fm, deg)
    ref32 = oracle(cam, sc, G, fm, deg, dtype=np.float32)
    got = run_gpu(cam, sc, G, flavour=flavour, use_filter=use_filter, sh_degree=deg)
    check_all(got, ref, deg, flavour == 'fork', H * W, ref32, case=f'parity[{W}x{H},n={n},sigma={r},sh={deg},{flavour},filter={use_filter},rot={rot}]',
              filter_on=use_filter)


def test_scale_modifier_and_background(built, size=(128, 80, 800)):
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(1.0, 1.0, 1.0)))._replace(scale_modifier=1.5)
    sc = f32_scene(O.make_scene(n, W, H, 3.0, seed=5))
    G = O.make_cotangent(3, H, W)
    ref = oracle(cam, sc, G, O.FILTER_ADD, 0)
    got = run_gpu(cam, sc, G, flavour='stock')
    check_all(got, ref, 0, False, H * W, oracle(cam, sc, G, O.FILTER_ADD, 0, dtype=np.float32))


def test_empty_input(built):
    """N = 0 must work (renderer.py:119-127)."""
    cam = O.make_camera(48, 40, bg=(0.3, 0.6, 0.9))
    z = lambda *s: torch.zeros(*s)
    sc = dict(means3D=z(0, 3), scales=z(0, 3), rotations=z(0, 4), opacities=z(0, 1), colors=z(0, 3))
    got = run_gpu(cam, sc, None)
    img = got['image'].cpu().numpy()
    np.testing.assert_allclose(img, np.broadcast_to(np.array([0.3, 0.6, 0.9], np.float32)[:, None, None], img.shape))
    assert got['radii'].numel() == 0 and (got['point_id_pixel'] == -1).all() and got['point_weight'].numel() == 0
    got = run_gpu(cam, sc, O.make_cotangent(3, 40, 48))      # backward with N = 0
    assert got['dmeans3D'].shape == (0, 3)


def test_all_culled_and_single(built):
    W, H = 64, 64
    cam = f32_camera(O.make_camera(W, H, bg=(0.1, 0.1, 0.1)))
    sc = f32_scene(O.make_scene(20, W, H, 3.0, seed=2))
    sc['means3D'][:, 2] = -3.0
    G = O.make_cotangent(3, H, W)
    got = run_gpu(cam, sc, G)
    assert (got['radii'] == 0).all() and float(got['dmeans3D'].abs().max()) == 0.0
    assert (got['point_id_pixel'] == -1).all()
    sc = f32_scene(O.make_scene(1, W, H, 5.0, seed=4))
    ref = oracle(cam, sc, G, O.FILTER_MAX, 0)
    got = run_gpu(cam, sc, G)
    check_all(got, ref, 0, True, H * W, oracle(cam, sc, G, O.FILTER_MAX, 0, dtype=np.float32))


def test_depth_ties_are_broken_by_index(built, size=(96, 64, 1200)):
    """All Gaussians on one plane z = const seen by an identity camera: every depth key is identical, so the order
    inside a tile must fall back to the Gaussian index (stable sort of index-ordered duplicates)."""
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H))
    sc = f32_scene(O.make_scene(n, W, H, 4.0, seed=9))
    z = 5.0
    sc['means3D'][:, :2] *= (z / sc['means3D'][:, 2:3])
    sc['means3D'][:, 2] = z
    sc['opacities'][:] = sc['opacities'].clamp(0.3, 0.9)
    G = O.make_cotangent(3, H, W)
    ref = oracle(cam, sc, G, O.FILTER_MAX, 0)
    got = run_gpu(cam, sc, G)
    check_all(got, ref, 0, True, H * W, oracle(cam, sc, G, O.FILTER_MAX, 0, dtype=np.float32))
    # and invariance: a second run gives the bit-identical image (deterministic order)
    got2 = run_gpu(cam, sc, None)
    assert torch.equal(got['image'].detach(), got2['image'])


@pytest.mark.parametrize('n', [3500, 15000])
def test_long_tile_lists(built, n):
    """Tile lists longer than the small (2560) and the large (13312) shared-memory sort capacity."""
    W, H = 32, 32
    cam = f32_camera(O.make_camera(W, H, bg=(0.5, 0.5, 0.5)))
    sc = O.make_scene(n, W, H, 8.0, seed=13)
    sc['opacities'][:] *= 0.05        # keep the transmittance alive through thousands of splats
    sc['opacities'][:] += 0.004
    sc = f32_scene(sc)
    G = O.make_cotangent(3, H, W)
    ref = oracle(cam, sc, G, O.FILTER_MAX, 0)
    ref32 = oracle(cam, sc, G, O.FILTER_MAX, 0, dtype=np.float32)
    got = run_gpu(cam, sc, G)
    # millions of pairs hover around alpha = 1/255 here (seed 13 has one at 1.3e-7): exclude the borderline ones
    gs, ps = borderline_decisions(cam, sc, O.FILTER_MAX)
    assert len(gs) <= 40
    sc_n[0] = n
    check_all(drop(got, gs, ps), drop(ref, gs, ps), 0, True, H * W, drop(ref32, gs, ps))


def test_tile_row_shards_sum_to_full(built, size=(160, 112, 3000)):
    """Multi-GPU sharding primitive: rendering tile rows [0,k) and [k,gy) separately and adding the results
    reproduces the un-sharded image and gradients."""
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.2, 0.3, 0.4)))
    sc = f32_scene(O.make_scene(n, W, H, 5.0, seed=21))
    G = O.make_cotangent(3, H, W)
    full = run_gpu(cam, sc, G)
    gy = (H + 15) // 16
    a = run_gpu(cam, sc, G, tile_rows=(0, 3))
    b = run_gpu(cam, sc, G, tile_rows=(3, gy))
    assert torch.equal(full['image'].detach(), (a['image'] + b['image']).detach())
    for k in ['dmeans3D', 'dmeans2D', 'dopacities', 'dscales', 'drotations', 'dcolors']:
        assert rel(a[k] + b[k], full[k]) < 1e-5, k
    assert torch.equal(torch.maximum(a['point_weight'], b['point_weight']), full['point_weight'])


@pytest.mark.parametrize('ci', [0, 1, 2])
def test_compute_radius_matches_reference_golden(built, ci):
    """lgr_compute_radius vs the golden radii produced by the reference's geometry.compute_radius."""
    from log_b200 import compute_radius
    p = f'cam{ci}_'
    dev = device()
    W, H = GOLD[p + 'spec'][0], GOLD[p + 'spec'][1]
    fovx, fovy = GOLD[p + 'FoV']
    tx, ty = math.tan(fovx / 2), math.tan(fovy / 2)
    t = lambda k: torch.from_numpy(GOLD[p + k]).to(device=dev, dtype=torch.float32)
    got = compute_radius(t('xyz'), t('scaling'), t('rotation'), t('full_proj_transform'), t('world_view_transform'),
                         W / (2 * tx), H / (2 * ty), tx, ty).cpu().numpy()
    P = GOLD[p + 'full_proj_transform']
    hom = GOLD[p + 'xyz'] @ P[:3] + P[3]
    ndc = hom[:, :2] / (hom[:, 3:4] + 1e-7)
    keep = (np.abs(ndc) <= 1.3).all(-1)
    margin = np.abs(np.abs(ndc) - 1.3).min(-1) > 1e-4
    np.testing.assert_allclose(got[keep & margin], GOLD[p + 'radius'][keep & margin], rtol=3e-4)
    assert (got[~keep & margin] == 0).all()


def test_fork_rasterizer_compute_radius_method(built, size=(320, 200, 4000)):
    """rasterizer.compute_radius(xyz, scaling, rotation) -- level_of_gaussian.py:59."""
    from log_b200 import GaussianRasterizer
    from util import settings_from_camera
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H))
    sc = f32_scene(O.make_scene(n, W, H, 3.0, seed=3))
    dev = device()
    r = GaussianRasterizer(settings_from_camera(cam, dev))
    got = r.compute_radius(*(sc[k].to(device=dev, dtype=torch.float32) for k in ('means3D', 'scales', 'rotations')))
    want = c_oracle.compute_radius(cam, sc['means3D'], sc['scales'], sc['rotations'])
    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=3e-4, atol=1e-5)


def test_backward_is_linear_in_the_cotangent(built, size=(192, 128, 4000)):
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.3, 0.3, 0.3)))
    sc = f32_scene(O.make_scene(n, W, H, 4.0, seed=17))
    G1, G2 = O.make_cotangent(3, H, W, seed=1), O.make_cotangent(3, H, W, seed=2)
    a, b, c = run_gpu(cam, sc, G1), run_gpu(cam, sc, G2), run_gpu(cam, sc, 2.0 * G1 - 0.5 * G2)
    for k in ['dmeans3D', 'dmeans2D', 'dopacities', 'dscales', 'drotations', 'dcolors']:
        assert rel(2.0 * a[k] - 0.5 * b[k], c[k]) < 1e-4, k


@pytest.mark.parametrize('world', [2, 3])
def test_band_mode_rows_reproduce_dense_gradients(built, world, size=(208, 144, 4001)):
    """Multi-GPU band mode, emulated on one GPU: every "rank" renders its tile band with the owner-grouped id lists,
    returns packed gradient rows; adding every rank's rows into the owner shards reproduces the dense gradients of the
    un-sharded run, and the bands add up to the full image."""
    from log_b200 import rasterize_backward, rasterize_forward, sharded
    from log_b200._capi import LGR_FILTER_MAX
    from util import settings_from_camera
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.2, 0.3, 0.4)))
    sc = f32_scene(O.make_scene(n, W, H, 5.0, seed=33))
    G = O.make_cotangent(3, H, W)
    full = run_gpu(cam, sc, G)
    dense = sharded.pack_grads((full['dmeans3D'], full['dmeans2D'], full['dopacities'], full['dscales'], full['drotations'],
                                full['dcolors']))
    dev = device()
    s = settings_from_camera(cam, dev)
    t = {k: v.to(device=dev, dtype=torch.float32).contiguous() for k, v in sc.items()}
    Gd = G.to(device=dev, dtype=torch.float32)
    op = t['opacities'].reshape(-1)
    rows_all, image = [], torch.zeros(3, H, W, device=dev)
    for r, band in enumerate(sharded.tile_row_partition(H, world)):
        img, radii, pid, pwp, pw, st = rasterize_forward(s, t['means3D'], op, t['scales'], t['rotations'], t['colors'], None,
                                                         LGR_FILTER_MAX, True, band, num_owners=world)
        assert sum(st.band_counts_host) <= n and len(st.band_counts_host) == world
        assert ((radii == full['radii']) | (radii == 0)).all()     # band mode: radii only near the band
        image += img
        rows_all.append(rasterize_backward(st, Gd, t['means3D'], op, t['scales'], t['rotations'], t['colors'], None))
    assert torch.equal(image, full['image'].detach())
    rows_all = torch.cat(rows_all)
    ids = rows_all[:, 17].contiguous().view(torch.int32)
    assert int(ids.min()) >= 0 and int(ids.max()) < n
    shards = [sharded.rows_to_shard(rows_all, lo, hi) for lo, hi in sharded.owner_partition(n, world)]
    assert torch.equal(torch.cat(shards)[:, 18].int(), full['radii'])    # owners recover every radius (max over bands)
    got = torch.cat(shards)[:, :17]
    assert got.shape == dense.shape
    assert rel(got, dense) < 2e-5
    for a, b in zip(sharded.unpack_grads(got), sharded.unpack_grads(dense)):
        assert rel(a, b) < 5e-5


@pytest.mark.gpu
@pytest.mark.parametrize('size', [(48, 32, 3000, 2.0), (96, 64, 2500, 5.0)])
def test_recorded_subtile_bits_do_not_change_the_backward(built, monkeypatch, size):
    """lgr_view.contrib_d: the forward records, per tile-list entry, which sub-tiles composited it (or stopped a pixel at
    it), and the backward walks only those pairs.  Same contributions, so the gradients must equal the backward that
    re-tests the boxes itself -- on tile lists of several staged batches (> 256 entries), where the record crosses batches."""
    import log_b200.rasterizer as R
    W, H, n, r = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.1, 0.2, 0.3)))
    sc = f32_scene(O.make_scene(n, W, H, r, seed=41))
    G = O.make_cotangent(3, H, W)
    monkeypatch.setattr(R, 'CONTRIB_BITS', False)
    a, a2 = run_gpu(cam, sc, G), run_gpu(cam, sc, G)
    monkeypatch.setattr(R, 'CONTRIB_BITS', True)
    b, b2 = run_gpu(cam, sc, G), run_gpu(cam, sc, G)
    assert torch.equal(a['image'], b['image'])
    for k in ['dmeans3D', 'dmeans2D', 'dopacities', 'dscales', 'drotations', 'dcolors']:
        # the blend backward accumulates per-Gaussian gradients with float atomics, so two runs of the SAME path differ in
        # the last bits (most in dscales, where the chain rule cancels): the bound also covers twice that measured spread
        spread = max(rel(a2[k], a[k]), rel(b2[k], b[k]))
        assert rel(b[k], a[k]) < max(2e-6, 2 * spread), (k, rel(b[k], a[k]), spread)


@pytest.mark.gpu
def test_device_sized_forward_equals_host_sized(built, size=(160, 112, 3000)):
    """lgr_forward_render_device_sized (no read-back of D, launch shapes independent of the data: CUDA-graph capturable) must
    produce exactly what the host-sized call produces, forward and backward; and when the view needs more instances than
    the caller's capacity it must say so (overflow flag) without touching memory out of bounds."""
    from log_b200 import GaussianRasterizer
    from util import settings_from_camera
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.1, 0.2, 0.3)))
    sc = f32_scene(O.make_scene(n, W, H, 5.0, seed=21))
    dev = device()
    G = O.make_cotangent(3, H, W).to(device=dev, dtype=torch.float32)

    def run(capacity):
        rast = GaussianRasterizer(settings_from_camera(cam, dev))
        rast.instance_capacity = capacity
        t = {k: v.to(device=dev, dtype=torch.float32).requires_grad_(True) for k, v in sc.items()}
        m2d = torch.zeros(n, 3, device=dev, requires_grad=True)
        out = rast(means3D=t['means3D'], means2D=m2d, shs=None, colors_precomp=t['colors'], opacities=t['opacities'], scales=t['scales'],
                   rotations=t['rotations'], cov3D_precomp=None)
        (out[0] * G).sum().backward()
        return out, {k: v.grad for k, v in t.items()}, m2d.grad, rast.last_state
    out_h, g_h, m_h, st_h = run(None)
    D = st_h.num_instances
    out_d, g_d, m_d, st_d = run(D + D // 4 + 64)
    stats = st_d.read_stats()
    assert stats['overflow'] == 0 and stats['num_instances'] == D and stats['max_tile_len'] == st_h.max_tile_len
    for a, b in zip(out_h, out_d):
        assert torch.equal(a, b)
    assert rel(m_d, m_h) < 2e-6                  # float atomics: accumulation order differs from run to run
    for k in g_h:
        assert rel(g_d[k], g_h[k]) < 2e-6, k
    # capacity too small: flagged, nothing out of bounds, image = background
    out_o, _, _, st_o = run(max(D // 3, 1))
    assert st_o.read_stats()['overflow'] & 1
    assert torch.isfinite(out_o[0]).all()


@pytest.mark.gpu
def test_band_mode_with_no_binned_instance(built, size=(64, 48, 300)):
    """Band mode when the band lists are non-empty (they follow the stock rectangle) but no splat reaches alpha >= 1/255
    anywhere (D == 0): the scatter kernel must still write the row -> id map and zero the listed accumulator rows, so the
    backward returns all-zero gradient rows carrying valid ids (round-1 advisor finding: it read an unwritten map)."""
    from log_b200 import rasterize_backward, rasterize_forward, sharded
    from log_b200._capi import LGR_FILTER_MAX
    from util import settings_from_camera
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.2, 0.3, 0.4)))
    sc = f32_scene(O.make_scene(n, W, H, 5.0, seed=5))
    sc['opacities'][:] = 0.001                      # below 1/255 everywhere
    dev = device()
    s = settings_from_camera(cam, dev)
    t = {k: v.to(device=dev, dtype=torch.float32).contiguous() for k, v in sc.items()}
    Gd = O.make_cotangent(3, H, W).to(device=dev, dtype=torch.float32)
    op = t['opacities'].reshape(-1)
    for band in sharded.tile_row_partition(H, 2):
        img, radii, pid, pwp, pw, st = rasterize_forward(s, t['means3D'], op, t['scales'], t['rotations'], t['colors'], None,
                                                         LGR_FILTER_MAX, True, band, num_owners=2)
        assert st.num_instances == 0 and sum(st.band_counts_host) > 0
        rows = rasterize_backward(st, Gd, t['means3D'], op, t['scales'], t['rotations'], t['colors'], None)
        ids = rows[:, 17].contiguous().view(torch.int32)
        assert int(ids.min()) >= 0 and int(ids.max()) < n
        assert float(rows[:, :17].abs().max()) == 0.0


@pytest.mark.parametrize('W,H,n,r', [(200, 120, 3000, 6.0), (64, 64, 0, 3.0), (333, 211, 20000, 2.0)])
def test_point_id_count_equals_torch_unique(built, W, H, n, r):
    """SURVEY 8(f) row 1: (point_id, point_count) from the blend kernel's winner histogram equals what LoG computes with
    torch.unique over the H x W id map (renderer.py:156-159)."""
    from log_b200 import GaussianRasterizer, point_id_count
    from util import settings_from_camera
    dev = device()
    cam = f32_camera(O.make_camera(W, H))
    sc = O.make_scene(max(n, 1), W, H, r, seed=8, dtype=torch.float32)
    t = {k: v[:n].to(dev) for k, v in sc.items()}
    rast = GaussianRasterizer(settings_from_camera(cam, dev))
    out = rast(means3D=t['means3D'], means2D=torch.zeros(n, 3, device=dev), shs=None, colors_precomp=t['colors'],
               opacities=t['opacities'], scales=t['scales'], rotations=t['rotations'], cov3D_precomp=None)
    pid_pixel = out[2]
    want_id, want_cnt = torch.unique(pid_pixel, sorted=True, return_counts=True)
    if want_id.numel() and want_id[0] == -1:
        want_id, want_cnt = want_id[1:], want_cnt[1:]
    got_id, got_cnt = point_id_count(rast.last_point_count)
    assert torch.equal(got_id.long(), want_id.long()) and torch.equal(got_cnt.long(), want_cnt.long())
    assert int(rast.last_point_count.sum()) == int((pid_pixel >= 0).sum())


@pytest.mark.parametrize('world', [2, 5])
def test_fused_push_route_emulated_on_one_gpu(built, world, size=(224, 160, 6001)):
    """The fused exchange (project_bwd stores packed rows straight into the owners' staging buffers, then
    lgr_grad_scatter_add_staged) exercised on ONE GPU: the "peer" pointers are local buffers, one per virtual rank."""
    import ctypes
    from log_b200 import _capi, rasterize_backward, rasterize_forward, sharded
    from log_b200._capi import LGR_FILTER_MAX
    from util import settings_from_camera
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.1, 0.2, 0.3)))
    sc = f32_scene(O.make_scene(n, W, H, 4.0, seed=41))
    G = O.make_cotangent(3, H, W)
    full = run_gpu(cam, sc, G)
    dense = sharded.pack_grads((full['dmeans3D'], full['dmeans2D'], full['dopacities'], full['dscales'], full['drotations'],
                                full['dcolors']))
    dev = device()
    s = settings_from_camera(cam, dev)
    t = {k: v.to(device=dev, dtype=torch.float32).contiguous() for k, v in sc.items()}
    Gd, op = G.to(device=dev, dtype=torch.float32), t['opacities'].reshape(-1)
    chunk = sharded.owner_chunk(n, world)
    floats = _capi.LGR_STAGE_HEADER_FLOATS + world * chunk * _capi.LGR_ROW_FLOATS
    stages = [torch.full((floats,), float('nan'), device=dev) for _ in range(world)]     # garbage where nothing is written
    for st_ in stages:
        st_[:_capi.LGR_STAGE_HEADER_FLOATS].view(torch.int32).fill_(12345)              # stale counts must be overwritten
    ptrs = torch.tensor([st_.data_ptr() for st_ in stages], dtype=torch.int64, device=dev)
    for r, band in enumerate(sharded.tile_row_partition(H, world)):
        *_, st = rasterize_forward(s, t['means3D'], op, t['scales'], t['rotations'], t['colors'], None, LGR_FILTER_MAX, True,
                                   band, num_owners=world)
        assert rasterize_backward(st, Gd, t['means3D'], op, t['scales'], t['rotations'], t['colors'], None,
                                  peer_stage=ptrs, my_rank=r) is None
    lib = _capi.load()
    shards = []
    for o, (lo, hi) in enumerate(sharded.owner_partition(n, world)):
        shard = torch.zeros((chunk, _capi.LGR_ROW_FLOATS), device=dev)
        _capi.check(lib.lgr_grad_scatter_add_staged(ctypes.c_void_p(stages[o].data_ptr()), world, chunk, lo, hi,
                                                    ctypes.c_void_p(shard.data_ptr()),
                                                    _capi.current_stream()), 'staged')
        shards.append(shard[:hi - lo])
    got = torch.cat(shards)
    assert torch.isfinite(got).all()
    assert rel(got[:, :17], dense) < 2e-5
    assert torch.equal(got[:, 18].int(), full['radii'])


def test_fused_activations_match_torch_activations(built, size=(176, 112, 2500)):
    """SURVEY 8(f) row 3: with raw_params=True the kernels apply LoG's activations (activation.py:36-44: exp, sigmoid,
    F.normalize, SH2RGB) themselves; image and gradients w.r.t. the RAW parameters equal torch activations followed by
    the ordinary call, and the fp64 oracle differentiated through the same activations."""
    from log_b200 import GaussianRasterizer
    from util import settings_from_camera
    W, H, n = size
    cam = f32_camera(O.make_camera(W, H, bg=(0.3, 0.2, 0.1)))
    sc = f32_scene(O.make_scene(n, W, H, 4.0, seed=55))
    g = torch.Generator().manual_seed(1)
    raw64 = dict(means3D=sc['means3D'], scales=torch.log(sc['scales']), opacities=torch.logit(sc['opacities'].clamp(0.02, 0.98)),
                 rotations=sc['rotations'] * (0.5 + torch.rand(n, 1, generator=g, dtype=torch.float64) * 2.0),   # un-normalised
                 colors=(sc['colors'] - 0.5) / O.C0)
    raw64 = {k: v.to(torch.float32).to(torch.float64) for k, v in raw64.items()}
    G = O.make_cotangent(3, H, W).to(torch.float32)
    dev = device()
    rast = GaussianRasterizer(settings_from_camera(cam, dev))

    def run(fused):
        t = {k: v.to(device=dev, dtype=torch.float32).requires_grad_(True) for k, v in raw64.items()}
        m2d = torch.zeros(n, 3, device=dev, requires_grad=True)
        if fused:
            out = rast(means3D=t['means3D'], means2D=m2d, shs=None, colors_precomp=t['colors'], opacities=t['opacities'],
                       scales=t['scales'], rotations=t['rotations'], cov3D_precomp=None, raw_params=True)
        else:
            out = rast(means3D=t['means3D'], means2D=m2d, shs=None, colors_precomp=t['colors'] * O.C0 + 0.5,
                       opacities=torch.sigmoid(t['opacities']), scales=torch.exp(t['scales']),
                       rotations=torch.nn.functional.normalize(t['rotations']), cov3D_precomp=None)
        (out[0] * G.to(dev)).sum().backward()
        return out[0].detach(), {k: v.grad for k, v in t.items()}, m2d.grad

    img_f, g_f, m2_f = run(True)
    img_t, g_t, m2_t = run(False)
    assert rel(img_f, img_t) < 1e-5
    assert rel(m2_f, m2_t) < 1e-4
    for k in g_t:
        assert rel(g_f[k], g_t[k]) < 1e-4, (k, rel(g_f[k], g_t[k]))
    # and against the oracle, differentiated through the same activations in float64
    leaves = {k: v.clone().requires_grad_(True) for k, v in raw64.items()}
    out = O.render(leaves['means3D'], torch.sigmoid(leaves['opacities']), torch.exp(leaves['scales']),
                   torch.nn.functional.normalize(leaves['rotations']), cam, colors_precomp=leaves['colors'] * O.C0 + 0.5,
                   filter_mode=O.FILTER_MAX)
    (out['image'] * G.to(torch.float64)).sum().backward()
    assert rel(img_f, out['image'].detach()) < 1e-4
    for k in g_t:
        assert rel(g_f[k], leaves[k].grad) < TOL, (k, rel(g_f[k], leaves[k].grad))


@pytest.mark.gpu
@pytest.mark.parametrize('deg', [0, 2])
def test_gather_fused_render_equals_log_get_all(built, deg, size=(160, 96, 3000, 1700)):
    """SURVEY 8(f) row 3, the gather half: `render_gathered` reads LoG's raw parameter TABLES through an index and applies
    the activations in the projection kernel.  It must equal what LoG does (level_of_gaussian.py:262-296,
    activation.py:27-44): gathered `nn.Parameter` copies -> torch activations (+ eval_sh_wobase) -> the ordinary rasteriser
    call -> autograd; image, aux outputs, the `screenspace_points` gradient and the COMPACT raw-parameter gradients (the
    rows SparseOptimizer reads) are compared.  The index is unsorted and the tables hold rows the view never touches."""
    from log_b200 import GaussianRasterizer
    from log_b200.gathered import render_gathered
    from util import settings_from_camera
    W, H, n_table, m = size
    K = 15
    cam = f32_camera(O.make_camera(W, H, bg=(0.3, 0.2, 0.1), sh_degree=deg, R=[[0.98, 0.0, 0.199], [0, 1, 0], [-0.199, 0, 0.98]],
                                   T=[0.1, -0.05, 0.3]))
    sc = f32_scene(O.make_scene(n_table, W, H, 4.0, seed=57, sh_degree=3))
    g = torch.Generator().manual_seed(3)
    dev = device()
    tables = {'xyz': sc['means3D'], 'scaling': torch.log(sc['scales']), 'opacity': torch.logit(sc['opacities'].clamp(0.02, 0.98)).reshape(-1, 1),
              'rotation': sc['rotations'] * (0.5 + torch.rand(n_table, 1, generator=g, dtype=torch.float64) * 2.0),
              'colors': (sc['colors'] - 0.5) / O.C0, 'shs': sc['shs'][:, 1:1 + K].contiguous()}
    tables = {k: v.to(device=dev, dtype=torch.float32).contiguous() for k, v in tables.items()}
    index = torch.randperm(n_table, generator=g)[:m].to(dev)
    G = O.make_cotangent(3, H, W).to(device=dev, dtype=torch.float32)
    settings = settings_from_camera(cam, dev)
    # LoG's path
    ret = {k: torch.nn.Parameter(v[index]) for k, v in tables.items()}
    colors = ret['colors'] * O.C0 + 0.5
    if deg > 0:
        d = ret['xyz'].detach() - settings.campos[None]
        d = d / torch.norm(d, dim=-1, keepdim=True)
        colors = colors + _eval_sh_wobase(deg, ret['shs'], d)
    m2d_t = torch.zeros(m, 3, device=dev, requires_grad=True)
    out_t = GaussianRasterizer(settings)(means3D=ret['xyz'], means2D=m2d_t, shs=None, colors_precomp=colors, opacities=torch.sigmoid(ret['opacity']),
                                         scales=torch.exp(ret['scaling']), rotations=torch.nn.functional.normalize(ret['rotation']),
                                         cov3D_precomp=None)
    (out_t[0] * G).sum().backward()
    # fused
    m2d_f = torch.zeros(m, 3, device=dev, requires_grad=True)
    use = dict(tables) if deg > 0 else {k: v for k, v in tables.items() if k != 'shs'}
    out_f, pcount, params = render_gathered(settings, use, index, m2d_f)
    (out_f[0] * G).sum().backward()
    assert rel(out_f[0], out_t[0]) < 1e-5
    assert torch.equal(out_f[1], out_t[1]) and torch.equal(out_f[2], out_t[2])
    assert rel(out_f[4], out_t[4]) < 1e-5
    assert rel(m2d_f.grad, m2d_t.grad) < 1e-4
    for k in use:
        if k == 'shs' and deg == 0:
            continue
        assert params[k].grad.shape == ret[k].grad.shape, k
        # two fp32 paths against each other (each is checked against the fp64 oracle to 1e-4 elsewhere): twice the bound
        assert rel(params[k].grad, ret[k].grad) < 2e-4, (k, rel(params[k].grad, ret[k].grad))


def _eval_sh_wobase(deg, sh, dirs):
    """eval_sh_wobase (LoG/model/sh_utils.py:31-58) through the oracle's eval_sh: a zero DC coefficient in front of the rest
    coefficients, minus the 0.5 offset eval_sh adds (its basis is pinned to the reference by tests/test_oracle_golden.py)."""
    full = torch.cat([torch.zeros_like(sh[:, :1]), sh], dim=1)
    return O.eval_sh(deg, full, dirs) - 0.5


def check_fused_log_colour_activation_with_sh(deg, size=(160, 96, 1800)):
    """SURVEY 8(f) row 3, colour part: LoG computes colours as SH2RGB(dc) + eval_sh_wobase(normalize(xyz.detach() - campos),
    shs, degree) with NO clamp (LoG/model/activation.py:27-34, sh_utils.py:31-73).  With raw_params and both raw DC colours
    and rest coefficients the kernels do that themselves; image and every gradient (incl. d/d rest, and NO colour
    gradient into the positions) equal torch activations + the ordinary call and the fp64 oracle."""
    from log_b200 import GaussianRasterizer
    from util import settings_from_camera
    W, H, n = size
    K = 15                                                     # LoG allocates (max_sh_degree+1)^2 - 1 = 15 rest coefficients
    cam = f32_camera(O.make_camera(W, H, bg=(0.3, 0.2, 0.1), sh_degree=deg, R=[[0.98, 0.0, 0.199], [0, 1, 0], [-0.199, 0, 0.98]],
                                   T=[0.1, -0.05, 0.3]))
    sc = f32_scene(O.make_scene(n, W, H, 4.0, seed=56, sh_degree=3))
    raw64 = dict(means3D=sc['means3D'], scales=torch.log(sc['scales']), opacities=torch.logit(sc['opacities'].clamp(0.02, 0.98)),
                 rotations=sc['rotations'] * 1.7, colors=(sc['colors'] - 0.5) / O.C0, shs=sc['shs'][:, 1:1 + K] * 3.0)
    raw64 = {k: v.to(torch.float32).to(torch.float64).contiguous() for k, v in raw64.items()}
    G = O.make_cotangent(3, H, W).to(torch.float32)
    dev = device()
    rast = GaussianRasterizer(settings_from_camera(cam, dev, deg))
    campos = cam.campos

    def log_colours(t, cp):      # activation.py:27-34 (eval_sh on [dc | rest] is SH2RGB(dc) + eval_sh_wobase(rest), unclamped)
        d = t['means3D'].detach() - cp[None]
        d = d / torch.norm(d, dim=-1, keepdim=True)
        return O.eval_sh(deg, torch.cat([t['colors'][:, None], t['shs']], dim=1), d)

    def run(fused):
        t = {k: v.to(device=dev, dtype=torch.float32).requires_grad_(True) for k, v in raw64.items()}
        m2d = torch.zeros(n, 3, device=dev, requires_grad=True)
        if fused:
            out = rast(means3D=t['means3D'], means2D=m2d, shs=t['shs'], colors_precomp=t['colors'], opacities=t['opacities'],
                       scales=t['scales'], rotations=t['rotations'], cov3D_precomp=None, raw_params=True)
        else:
            out = rast(means3D=t['means3D'], means2D=m2d, shs=None, colors_precomp=log_colours(t, campos.to(device=dev, dtype=torch.float32)),
                       opacities=torch.sigmoid(t['opacities']), scales=torch.exp(t['scales']),
                       rotations=torch.nn.functional.normalize(t['rotations']), cov3D_precomp=None)
        (out[0] * G.to(dev)).sum().backward()
        return out[0].detach(), {k: v.grad for k, v in t.items()}, m2d.grad

    img_f, g_f, m2_f = run(True)
    img_t, g_t, m2_t = run(False)
    assert rel(img_f, img_t) < 1e-5
    assert rel(m2_f, m2_t) < 1e-4
    for k in g_t:
        assert rel(g_f[k], g_t[k]) < 1e-4, (k, rel(g_f[k], g_t[k]))
    nb = (deg + 1) ** 2 - 1
    assert float(g_f['shs'][:, :nb].abs().max()) > 0.0 and (nb == K or float(g_f['shs'][:, nb:].abs().max()) == 0.0)
    leaves = {k: v.clone().requires_grad_(True) for k, v in raw64.items()}
    out = O.render(leaves['means3D'], torch.sigmoid(leaves['opacities']), torch.exp(leaves['scales']),
                   torch.nn.functional.normalize(leaves['rotations']), cam, colors_precomp=log_colours(leaves, campos),
                   filter_mode=O.FILTER_MAX)
    (out['image'] * G.to(torch.float64)).sum().backward()
    assert rel(img_f, out['image'].detach()) < 1e-4
    for k in g_t:
        assert rel(g_f[k], leaves[k].grad) < TOL, (k, rel(g_f[k], leaves[k].grad))


def check_cov3D_precomp(size=(96, 64, 600, 3.0), flavour='stock'):
    """The stock API's cov3D_precomp (a precomputed world-space covariance instead of scales / rotations; LoG always passes
    None, renderer.py:133,149, but diff_gaussian_rasterization's public signature has it):
      * against the fp64 torch oracle given the same (N,6) covariances: image, radii, every gradient incl. dL/dcov3D;
      * against the scale / rotation path of the same library: same image; dL/dcov3D chain-ruled through
        Sigma = R S S^T R^T reproduces that path's dscales / drotations;
      * scale_modifier does not touch a precomputed covariance (stock behaviour)."""
    W, H, n, r = size
    fork = flavour == 'fork'
    cam = f32_camera(O.make_camera(W, H, bg=(0.1, 0.3, 0.2)))
    sc = f32_scene(O.make_scene(n, W, H, r, seed=23))
    sc['means3D'][:4, 2] = -1.0                  # behind the camera
    sc['opacities'][4:8] = 0.001                 # below 1/255
    G = O.make_cotangent(3, H, W).to(torch.float32).to(torch.float64)
    fm = O.FILTER_MAX if fork else O.FILTER_ADD

    def sigma6(scales, rotations):
        S = O.cov3d(scales, rotations, 1.0)
        return torch.stack([S[:, 0, 0], S[:, 0, 1], S[:, 0, 2], S[:, 1, 1], S[:, 1, 2], S[:, 2, 2]], dim=-1)
    cov6 = sigma6(sc['scales'], sc['rotations']).to(torch.float32).to(torch.float64)      # what the kernels are given
    # ---- fp64 oracle with the same covariances
    leaf = {k: sc[k].clone().requires_grad_(True) for k in ('means3D', 'opacities', 'colors')}
    c6 = cov6.clone().requires_grad_(True)
    m2d = torch.zeros(n, 3, dtype=torch.float64, requires_grad=True)
    out = O.render(leaf['means3D'], leaf['opacities'], None, None, cam, colors_precomp=leaf['colors'], filter_mode=fm,
                   means2D=m2d, cov3D_precomp=c6)
    (out['image'] * G).sum().backward()
    got = run_gpu(cam, sc, G, flavour=flavour, cov3D=cov6)
    errs = {'image': rel(got['image'], out['image']), 'dmeans3D': rel(got['dmeans3D'], leaf['means3D'].grad),
            'dmeans2D': rel(got['dmeans2D'][:, :2], m2d.grad[:, :2]), 'dopacities': rel(got['dopacities'], leaf['opacities'].grad.reshape(-1)),
            'dcolors': rel(got['dcolors'], leaf['colors'].grad), 'dcov3D': rel(got['dcov3D'], c6.grad)}
    from util import record_parity
    record_parity(f'cov3D_precomp[{W}x{H},n={n},sigma={r},{flavour}]', {k: (v, None) for k, v in errs.items()}, TOL)
    for k, e in errs.items():
        assert e < TOL, (k, e)
    rg = got['radii'].cpu().numpy()
    assert (rg != out['radii'].numpy()).sum() <= 2
    dead = rg == 0
    assert dead[:8].all() or (rg[:4] == 0).all()
    assert not got['dcov3D'].cpu().numpy()[dead].any()                      # culled rows: zero gradient, not garbage
    # ---- against the scale / rotation path of the library itself
    base = run_gpu(cam, sc, G, flavour=flavour)
    assert rel(got['image'], base['image']) < 2e-5                           # Sigma rounded to fp32 once vs built in registers
    sl = sc['scales'].clone().requires_grad_(True)
    rl = sc['rotations'].clone().requires_grad_(True)
    (sigma6(sl, rl) * got['dcov3D'].detach().cpu().to(torch.float64)).sum().backward()
    assert rel(sl.grad, base['dscales']) < TOL and rel(rl.grad, base['drotations']) < TOL
    # ---- scale_modifier leaves a precomputed covariance alone
    mod = run_gpu(cam._replace(scale_modifier=1.7), sc, None, flavour=flavour, cov3D=cov6)
    assert torch.equal(mod['image'], run_gpu(cam, sc, None, flavour=flavour, cov3D=cov6)['image'])
    # ---- the stock argument rule
    from log_b200 import StockGaussianRasterizer
    from util import settings_from_camera
    rast = StockGaussianRasterizer(settings_from_camera(cam, device()))
    t = lambda x: x.to(device=device(), dtype=torch.float32)
    with pytest.raises(Exception, match='exactly one'):
        rast(means3D=t(sc['means3D']), means2D=None, opacities=t(sc['opacities']), colors_precomp=t(sc['colors']),
             scales=t(sc['scales']), rotations=t(sc['rotations']), cov3D_precomp=t(cov6))
    with pytest.raises(Exception, match='exactly one'):
        rast(means3D=t(sc['means3D']), means2D=None, opacities=t(sc['opacities']), colors_precomp=t(sc['colors']))


def check_mark_visible(n=3000):
    """GaussianRasterizer.markVisible(positions) of the stock module: view-space z > 0.2 (the projection's near cull)."""
    from log_b200 import GaussianRasterizer
    from util import settings_from_camera
    cam = f32_camera(O.make_camera(128, 96, R=[[0.98, 0.0, 0.199], [0, 1, 0], [-0.199, 0, 0.98]], T=[0.1, -0.05, 0.3]))
    g = torch.Generator().manual_seed(3)
    pos = (torch.rand(n, 3, generator=g, dtype=torch.float64) * 8 - 4).to(torch.float32)
    pos[:7, 2] = torch.tensor([0.2, 0.19999, 0.20001, -5.0, 0.0, 100.0, 0.3]) - 0.3      # around the plane (T_z = 0.3 for x = y = 0)
    pos[:7, :2] = 0.0
    rast = GaussianRasterizer(settings_from_camera(cam, device()))
    got = rast.markVisible(pos.to(device()))
    assert got.dtype == torch.bool and got.shape == (n,)
    V = cam.viewmatrix.to(torch.float32)
    z = pos[:, 0] * V[0, 2] + pos[:, 1] * V[1, 2] + pos[:, 2] * V[2, 2] + V[3, 2]
    want = z > 0.2
    sure = (z - 0.2).abs() > 1e-5                 # fp32 summation order may flip a point sitting on the plane
    assert torch.equal(got.cpu()[sure], want[sure]) and sure.sum() > n - 10
    assert rast.markVisible(pos[:0].to(device())).shape == (0,)
    # consistent with the rasteriser's own cull: every point with a radius is marked visible
    sc = f32_scene(O.make_scene(500, 128, 96, 3.0, seed=8))
    sc['means3D'][:20, 2] = -1.0
    res = run_gpu(cam, sc, None)
    vis = rast.markVisible(sc['means3D'].to(device=device(), dtype=torch.float32))
    assert bool((vis | (res['radii'] == 0)).all()) and not bool(vis.all())
