#!/usr/bin/env python
"""bench.py -- the headline benchmark of the hot path (BASELINE.json):
forward + backward of the differentiable Gaussian-splatting rasteriser on synthetic Gaussians at 1080p.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 10m|100k|1k] [--impl ours|reference]

A "step" is one pass of the hot path over one view: project -> bin/sort -> blend -> backward sweep -> per-Gaussian
backward.  `value` = Gaussians processed per second by the whole job with inputs resident in HBM; `e2e` = the same
through the public GaussianRasterizer autograd API with HOST (pinned) inputs copied in and the loss read back every
step.  N > 1: tile rows are sharded over ranks (strong scaling of ONE view), per-Gaussian gradients are reduced to
owner ranks with NCCL; time = max over ranks.

N > 1 default: shard mode (log_b200/sharded.py:SplatExchange: Gaussians AND tile-row bands sharded, splat records pushed to
the band owners over NVLink peer memory, 2D gradients returned, no reduction); `LGR_MULTI=band` selects the round-1
layout (Gaussians replicated, gradient rows reduced to owner ranks).  Every N > 1 line carries `parity`: outside the timed
region each rank repeats the step on ONE GPU and compares its band of the image and its own Gaussians' gradients.

`--impl reference` times the CPU implementation of the same path (the oracle port: the reference's rasteriser is an
un-vendored CUDA package that cannot be built or run on a CPU, see DESIGN.md) on the box's host cores.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (N, W, H, median sigma px, sh_degree)   -- SURVEY.md 8(d) / BASELINE.json configs
    '10m': (10_000_000, 1920, 1080, 1.5, 0),     # config 3 (the metric's configuration): precomputed colour, as LoG feeds
    '100k': (100_000, 1920, 1080, 8.0, 3),       # config 1: SH degree 3 in-kernel
    '1k': (1_000, 256, 256, 3.0, 0),             # config 0 (plumbing)
    'big300k': (300_000, 1920, 1080, 35.0, 0),   # diagnostic: LoG-at-initialisation regime (kNN-sized splats, sigma ~35 px, tile lists > 4096)
    '50m4k': (50_000_000, 3840, 2160, 1.5, 0),   # config 4 (city scale, 4K): meant for `LGR_MULTI=shard` on 8 GPUs; not yet run
}
CPU_SAMPLE = {'10m': 1_000_000, '100k': 100_000, '1k': 1_000, '50m4k': 1_000_000, 'big300k': 20_000}   # Gaussians in the bounded CPU sample
DUMP_SAMPLE = 1 << 16      # --dump-outputs: Gaussians and pixels kept per array (at most ~25 MB in all, SH degree 3 included)
GRAD_NAMES = ('dmeans3D', 'dmeans2D', 'dopacities', 'dscales', 'drotations', 'dcolors', 'dshs')


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line)

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def algorithmic_bytes(n, H, W, D, sh_degree):
    """SURVEY.md 8(d): per-kernel split of B_model = B_min + 112 D  (fp32)."""
    b_in = 56 if sh_degree == 0 else 56 - 12 + 4 * 3 * (sh_degree + 1) ** 2
    b_grad = 68 if sh_degree == 0 else 68 - 12 + 4 * 3 * (sh_degree + 1) ** 2
    HW = H * W
    k = {'project_fwd': n * b_in + n * 8, 'bin_sort': D * 32, 'blend_fwd': D * 40 + HW * 20,
         'blend_bwd': D * 40 + HW * 12, 'project_bwd': n * b_in + n * b_grad}
    b_min = n * b_in + n * 8 + HW * 20 + n * b_in + HW * 12 + n * b_grad
    return k, b_min, b_min + 112 * D


def workload_name(w):
    n, W, H, r, deg = WORKLOADS[w]
    return (f'{w}: {n} synthetic Gaussians (median sigma {r} px), {W}x{H}, sh_degree {deg}, forward+backward, '
            'fork flavour (max(cov,0.3) filter, 5-tuple aux outputs)')


def make_inputs(workload, dtype=torch.float32):
    from log_b200.synthetic import make_camera, make_cotangent, make_scene
    n, W, H, r, deg = WORKLOADS[workload]
    cam = make_camera(W, H, dtype=dtype, sh_degree=deg)
    sc = make_scene(n, W, H, r, seed=0, sh_degree=deg, dtype=dtype)
    G = make_cotangent(3, H, W, seed=1, dtype=dtype)
    return cam, sc, G


def morton_order(cam, sc, W, H):
    """Permute the scene so that neighbours in memory are neighbours on screen (Morton order of the projected centre, 4-pixel
    cells): a diagnostic for the same-address atomics of binning, which a spatially random order never stresses."""
    m = sc['means3D'].double()
    P = cam.projmatrix.double()
    hom = m @ P[:3] + P[3]
    ndc = hom[:, :2] / (hom[:, 3:4] + 1e-7)
    px = (((ndc[:, 0] + 1) * W - 1) * 0.5).clamp(0, W - 1).long() >> 2
    py = (((ndc[:, 1] + 1) * H - 1) * 0.5).clamp(0, H - 1).long() >> 2

    def spread(v):
        v = (v | (v << 8)) & 0x00FF00FF
        v = (v | (v << 4)) & 0x0F0F0F0F
        v = (v | (v << 2)) & 0x33333333
        return (v | (v << 1)) & 0x55555555
    perm = torch.argsort(spread(px) | (spread(py) << 1))
    return {k: v[perm].contiguous() for k, v in sc.items()}


def dump_outputs(path, out):
    """--dump-outputs: the arrays the timed path returned in its last step, one DIR/<name>.npy each (float32 as computed,
    integer arrays as float64).  Per-Gaussian arrays keep the rows listed in gaussian_index.npy, per-pixel arrays the
    pixels (row-major) listed in pixel_index.npy: fixed seeded samples of DUMP_SAMPLE each, the same in every run, so that
    two builds can be compared file by file."""
    os.makedirs(path, exist_ok=True)
    rng = np.random.default_rng(0)
    n, (H, W) = out['radii'].shape[0], out['image'].shape[1:]
    gi = np.sort(rng.choice(n, min(n, DUMP_SAMPLE), replace=False))
    pi = np.sort(rng.choice(H * W, min(H * W, DUMP_SAMPLE), replace=False))
    arrays = {'gaussian_index': gi.astype(np.float64), 'pixel_index': pi.astype(np.float64)}
    gi_d, pi_d = (torch.from_numpy(a).to(out['image'].device) for a in (gi, pi))
    for name, t in out.items():
        if t is None:
            continue
        per_pixel = name in ('image', 'point_id_pixel', 'point_weight_pixel')
        t = t.detach().reshape(-1, H * W)[:, pi_d].squeeze(0) if per_pixel else t.detach()[gi_d]
        a = t.cpu().numpy()
        arrays[name] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
    assert sum(a.nbytes for a in arrays.values()) <= 64 << 20
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def pick_cpu_threads(c_oracle, step):
    """The CPU arm gets the team size that is FASTEST on this box: all logical CPUs or one thread per physical core
    (half of them) -- the port is bound by memory and atomics, and SMT siblings slow it down on some hosts.  torchrun
    exports OMP_NUM_THREADS=1 to its children, so the team is always sized explicitly.  Returns (threads, {threads: seconds})."""
    ncpu = os.cpu_count() or 1
    tried = {}
    for nt in sorted({ncpu, max(1, ncpu // 2)}, reverse=True):
        c_oracle.set_num_threads(nt)
        step()                                     # warm-up at this team size
        t0 = time.perf_counter()
        step()
        tried[nt] = time.perf_counter() - t0
    best = min(tried, key=tried.get)
    c_oracle.set_num_threads(best)
    return best, tried


def run_reference(args, rank, world):
    """CPU arm: the oracle port (C, OpenMP, all host threads) on a bounded sample of the workload."""
    if rank != 0:
        return
    from oracle import c_oracle
    n, W, H, r, deg = WORKLOADS[args.workload]
    ns = min(n, CPU_SAMPLE[args.workload])
    cam, sc, G = make_inputs(args.workload)
    sub = {k: v[:ns].numpy() for k, v in sc.items()}
    kw = dict(colors_precomp=sub['colors']) if deg == 0 else dict(shs=sub['shs'])
    def step():
        c_oracle.render(cam, sub['means3D'], sub['opacities'], sub['scales'], sub['rotations'],
                        filter_mode=c_oracle.FILTER_MAX, dL_dimage=G.numpy(), dtype=np.float32, want_aux=True, **kw)
    cores, tried = pick_cpu_threads(c_oracle, step)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = ns / dt
    sample = (f'first {ns} of {n} Gaussians, {W}x{H}, fwd+bwd, fp32, {cores} OpenMP threads (fastest of ' +
              ', '.join(f'{k}: {v:.2f} s' for k, v in sorted(tried.items())) + ')')
    print(json.dumps({
        'impl': 'reference', 'metric': 'gaussians_per_s_fwd_bwd', 'value': val, 'unit': 'Gaussians/s', 'n_gpus': 0,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'mpix_per_s': W * H / dt / 1e6,
        'config': {'workload': workload_name(args.workload), 'sample': sample},
        'cpu_baseline': {'value': val, 'unit': 'Gaussians/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': val, 'unit': 'Gaussians/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default='10m', choices=sorted(WORKLOADS))
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed as DIR/<name>.npy (rank 0: the image and '
                         'gradients of its band and Gaussians under N > 1; seeded samples of large arrays)')
    ap.add_argument('--order', default='random', choices=['random', 'morton'],
                    help='order of the synthetic Gaussians in memory: random (SURVEY 8d, the default and the reported metric) or '
                         'sorted along a Morton curve of their screen position (spatially coherent, like tree-ordered LoG data)')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    from log_b200 import GaussianRasterizationSettings, GaussianRasterizer, _capi, rasterize_backward, rasterize_forward
    from log_b200 import sharded
    from log_b200._capi import LGR_FILTER_MAX
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; log_b200 has no CPU fallback (use --impl reference for the CPU arm)')
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    assert world == args.gpus or world == 1, (world, args.gpus)
    if args.dump_outputs and world > 1 and os.environ.get('LGR_MULTI', 'shard') != 'shard':
        raise SystemExit('bench.py: --dump-outputs covers one GPU and shard mode; band mode returns packed gradient rows')

    n, W, H, r, deg = WORKLOADS[args.workload]
    cam, sc, G = make_inputs(args.workload)
    if args.order == 'morton':
        sc = morton_order(cam, sc, W, H)
    host = {k: v.pin_memory() for k, v in sc.items()}
    host_G = G.pin_memory()
    settings = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=cam.bg.to(dev), scale_modifier=1.0,
        viewmatrix=cam.viewmatrix.to(dev), projmatrix=cam.projmatrix.to(dev), sh_degree=deg, campos=cam.campos.to(dev),
        prefiltered=False, debug=False)
    tile_rows = sharded.tile_row_partition(H, world)[rank] if world > 1 else None
    d = {k: v.to(dev) for k, v in host.items()}
    dG = host_G.to(dev)
    col = d['colors'] if deg == 0 else None
    shs = d['shs'] if deg > 0 else None
    opac = d['opacities'].reshape(-1)
    stats = {}

    phase_ev = []
    peer = None
    # gradient exchange route: measured on this pool (10 M workload, ms/step) -- 2 GPUs: peer 3.56 / nccl 4.10; 4 GPUs: peer
    # 2.55; 8 GPUs: peer 2.68 / nccl 1.85.  The fused NVLink push wins while few ranks write into each owner; at 8 ranks
    # all ranks push their owner-grouped rows in the same owner order (incast) and NCCL's staggered all-to-all is faster.
    route = os.environ.get('LGR_EXCHANGE', 'peer' if world <= 4 else 'nccl')
    # LGR_MULTI=shard: Gaussian-sharded ranks exchanging splat records / 2D gradients (log_b200/sharded.py:SplatExchange)
    # instead of replicated Gaussians + gradient rows.  Opt-in until its first hardware run has been checked in.
    shard = None
    if world > 1 and os.environ.get('LGR_MULTI', 'shard') == 'shard':
        shard = sharded.SplatExchange.over_symmetric_memory(n, H)
        lo_, hi_ = shard.lo, shard.hi
        loc = {k: v[lo_:hi_].contiguous() for k, v in d.items()}
        loc_op = loc['opacities'].reshape(-1)
    if world > 1 and route == 'peer' and shard is None:
        try:
            peer = sharded.PeerExchange(n)
        except Exception as e:      # symmetric memory unavailable: NCCL all-to-all route
            peer = None
            if rank == 0:
                print(f'bench.py: peer exchange unavailable ({e!r}); using NCCL all-to-all', file=sys.stderr)

    inst_cap = [None]          # N = 1: instance capacity of the device-sized call, learned from the warm-up steps

    def step_resident(record=False):
        if shard is not None:
            if record:
                ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                ev[0].record()
            img, radii, pid, pwp, st = shard.forward(settings, loc['means3D'], loc_op, loc['scales'], loc['rotations'],
                                                     loc['colors'] if deg == 0 else None, loc['shs'] if deg > 0 else None,
                                                     filter_mode=LGR_FILTER_MAX, want_aux=True)
            if record:
                ev[1].record()
            g, pw, _ = shard.backward(st, dG)          # sweep + return, barrier, gather + per-Gaussian backward
            if record:
                ev[2].record()
                ev[3].record()
                phase_ev.append(ev)
            return dict(image=img, radii=radii, point_id_pixel=pid, point_weight_pixel=pwp, point_weight=pw, **dict(zip(GRAD_NAMES, g)))
        if world > 1:      # band mode: owner-grouped id lists, packed gradient rows, one all-to-all to the owner ranks
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            ev[0].record()
            img, radii, pid, pwp, pw, st = rasterize_forward(settings, d['means3D'], opac, d['scales'], d['rotations'], col, shs,
                                                             LGR_FILTER_MAX, True, tile_rows, num_owners=world)
            ev[1].record()
            if peer is not None:
                g = peer.backward(st, dG, d['means3D'], opac, d['scales'], d['rotations'], col)
                ev[2].record()
            else:
                rows = rasterize_backward(st, dG, d['means3D'], opac, d['scales'], d['rotations'], col, shs)
                ev[2].record()
                g = sharded.exchange_rows_to_owners(rows, st.band_counts_host, n)
            ev[3].record()
            if record:
                phase_ev.append(ev)
            stats['rows'] = sum(st.band_counts_host)
        else:
            img, radii, pid, pwp, pw, st = rasterize_forward(settings, d['means3D'], opac, d['scales'], d['rotations'], col, shs,
                                                             LGR_FILTER_MAX, True, tile_rows, instance_capacity=inst_cap[0])
            g = rasterize_backward(st, dG, d['means3D'], opac, d['scales'], d['rotations'], col, shs)
            stats['state'] = st
        if st.max_tile_len is not None:
            stats['D'], stats['D_stock'], stats['maxlen'], stats['visible'] = st.num_instances, st.stock_instances, st.max_tile_len, st.num_visible
        return dict(image=img, radii=radii, point_id_pixel=pid, point_weight_pixel=pwp, point_weight=pw, **dict(zip(GRAD_NAMES, g)))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sync_free = bool(int(os.environ.get('LGR_SYNC_FREE', '1'))) and (world == 1 or shard is not None)
    if shard is not None:
        shard.sync_free = sync_free      # the view is static here and check_overflow() follows the timed loop
    use_graph = sync_free and bool(int(os.environ.get('LGR_GRAPH', '1')))
    for _ in range(args.warmup):
        step_resident()
        if world == 1 and sync_free and inst_cap[0] is None and stats['maxlen'] <= _capi.load().lgr_sort_smem_capacity():
            inst_cap[0] = stats['D'] + stats['D'] // 4 + 4096      # later steps: device-sized, nothing read back
    barrier()
    # The timed steps: no profiling events, no per-step host reads.  With device-sized calls a step contains no host
    # synchronisation, so one step is captured in a CUDA graph and replayed (inputs and scratch are static buffers).
    graph, graph_note = None, 'off'
    if use_graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                step_resident()
            torch.cuda.current_stream().wait_stream(side)
            barrier()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                g_static = step_resident()
            graph_note = 'one step (forward + backward' + (', both exchanges and barriers' if shard is not None else '') + ') captured once, replayed per step'
        except Exception as e:      # capture is an optimisation: fall back to plain launches and say so
            graph = None
            graph_note = f'capture failed ({type(e).__name__}: {str(e)[:120]}); plain launches'
            torch.cuda.synchronize()
    flags = torch.tensor([0 if graph is not None else 1], device=dev)
    if world > 1:      # all ranks replay, or none does
        dist.all_reduce(flags, op=dist.ReduceOp.MAX)
        if int(flags.item()) and graph is not None:
            graph, graph_note = None, 'capture failed on another rank; plain launches'
    barrier()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        if graph is not None:
            graph.replay()
        else:
            last = step_resident()
    e1.record()
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, g_static if graph is not None else last)
    clk = clocks.stop() if rank == 0 else None
    ms_total = e0.elapsed_time(e1)
    t = torch.tensor([ms_total], device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    # did every device-sized step fit its buffers?  (one read-back, after the timed region)
    if shard is not None:
        sst = shard.check_overflow()
        stats['rows'] = sst['num_rows']
        stats['D'], stats['D_stock'], stats['maxlen'], stats['visible'] = sst['num_instances'], sst['stock_instances'], sst['max_tile_len'], sst['num_rows']
    elif world == 1 and inst_cap[0] is not None:
        sst = stats['state'].read_stats()
        if sst['overflow']:
            raise SystemExit(f'bench.py: device-sized step outgrew its buffers: {sst}')
        stats['D'], stats['D_stock'], stats['maxlen'], stats['visible'] = sst['num_instances'], sst['stock_instances'], sst['max_tile_len'], sst['num_visible']
    # ---- a second, PROFILED pass (per-kernel CUDA events, phase events): explains the step, is not the step time ----
    prof_steps = max(3, min(args.steps, 10))
    _capi.profile_enable(True)
    phase_ev.clear()
    for _ in range(prof_steps):
        step_resident(record=True)
    barrier()
    phases = None
    if phase_ev:
        phases = {k: sum(ev[i].elapsed_time(ev[i + 1]) for ev in phase_ev) / len(phase_ev)
                  for i, k in enumerate(('forward', 'backward', 'exchange'))}
        phases['rows_sent_per_rank'] = stats.get('rows')
    prof = _capi.profile_collect()
    _capi.profile_enable(False)
    prof = {k: (v[0] * args.steps / prof_steps, v[1]) for k, v in prof.items()}      # scaled to the K timed steps (reported per step below)

    # ---- parity of the multi-GPU result (outside the timed region): the same step on ONE GPU, compared on every rank ----
    parity = None
    if world > 1:
        def relerr(got, want):
            d = (got.double() - want.double()).norm()
            return float(d / want.double().norm().clamp_min(1e-30))
        img1, rad1, pid1, pwp1, pw1, st1 = rasterize_forward(settings, d['means3D'], opac, d['scales'], d['rotations'], col, shs, LGR_FILTER_MAX, True, None)
        g1 = rasterize_backward(st1, dG, d['means3D'], opac, d['scales'], d['rotations'], col, shs)
        names = ('dmeans3D', 'dmeans2D', 'dopacities', 'dscales', 'drotations', 'dcolors')
        errs = {}
        if shard is not None:
            imgN, radN, pidN, pwpN, stN = shard.forward(settings, loc['means3D'], loc_op, loc['scales'], loc['rotations'],
                                                        loc['colors'] if deg == 0 else None, loc['shs'] if deg > 0 else None,
                                                        filter_mode=LGR_FILTER_MAX, want_aux=True)
            gN, pwN, pcN = shard.backward(stN, dG)
            y0, y1 = shard.band[0] * 16, min(shard.band[1] * 16, H)
            errs['image'] = relerr(imgN[:, y0:y1], img1[:, y0:y1]) if y1 > y0 else 0.0
            errs['point_id_pixel_mismatch'] = float((pidN[y0:y1] != pid1[y0:y1]).float().mean()) if y1 > y0 else 0.0
            for k, name in enumerate(names):
                errs[name] = relerr(gN[k].reshape(hi_ - lo_, -1), g1[k][lo_:hi_].reshape(hi_ - lo_, -1)) if hi_ > lo_ else 0.0
            errs['radii_mismatch'] = float((radN != rad1[lo_:hi_]).float().mean()) if hi_ > lo_ else 0.0
            errs['point_weight'] = relerr(pwN, pw1[lo_:hi_]) if hi_ > lo_ else 0.0
        else:
            imgN, radN, pidN, pwpN, pwN, stN = rasterize_forward(settings, d['means3D'], opac, d['scales'], d['rotations'], col, shs,
                                                                 LGR_FILTER_MAX, True, tile_rows, num_owners=world)
            if peer is not None:
                gsh = peer.backward(stN, dG, d['means3D'], opac, d['scales'], d['rotations'], col)
            else:
                gsh = sharded.exchange_rows_to_owners(rasterize_backward(stN, dG, d['means3D'], opac, d['scales'], d['rotations'], col, shs),
                                                      stN.band_counts_host, n)
            lo_b, hi_b = sharded.owner_partition(n, world)[rank]
            y0, y1 = tile_rows[0] * 16, min(tile_rows[1] * 16, H)
            errs['image'] = relerr(imgN[:, y0:y1], img1[:, y0:y1]) if y1 > y0 else 0.0
            want = sharded.pack_grads((g1[0], g1[1], g1[2], g1[3], g1[4], g1[5]))[lo_b:hi_b]
            for k, name in enumerate(names):
                sl = sharded.unpack_grads(gsh[:hi_b - lo_b, :17])[k], sharded.unpack_grads(want)[k]
                errs[name] = relerr(sl[0].reshape(hi_b - lo_b, -1), sl[1].reshape(hi_b - lo_b, -1)) if hi_b > lo_b else 0.0
        keys = sorted(errs)
        te = torch.tensor([errs[k] for k in keys], device=dev, dtype=torch.float64)
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        parity = {k: float(v) for k, v in zip(keys, te.tolist())}
        parity['bound'] = 2e-5
        parity['what'] = ('max over ranks of the norm-wise relative error between the N-rank result (each rank: its band of the image, '
                          'the gradients of the Gaussians it owns) and the same step on one GPU')
        parity['ok'] = all(v <= 2e-5 for k, v in parity.items() if k not in ('bound', 'what', 'point_id_pixel_mismatch', 'radii_mismatch')) and \
            parity.get('radii_mismatch', 0.0) == 0.0 and parity.get('point_id_pixel_mismatch', 0.0) <= 1e-5
        del img1, rad1, pid1, pwp1, pw1, st1, g1, imgN, stN
        torch.cuda.empty_cache()

    # ---- end to end through the public API: pinned host inputs in, loss out, every step ----
    # Two preallocated device input sets; every step copies ALL of its inputs from pinned host memory into one of them
    # (copy stream, no allocation and no record_stream inside the timed loop) and reads its loss back.  N = 1: the
    # reference-facing GaussianRasterizer + autograd.  N > 1 (shard mode): SplatExchange.rasterize + autograd, and a rank
    # copies only the Gaussians it owns.
    e2e = None
    if not args.no_e2e:
        use_sh = deg > 0
        if shard is not None:
            host = {k: v[shard.lo:shard.hi].contiguous().pin_memory() for k, v in sc.items()}
        in_keys = [k for k in host if not (k == 'colors' and use_sh)]
        # the cotangent image: a rank of the shard mode needs only the rows of its band (the rest of its image is zero)
        gy0, gy1 = (shard.band[0] * 16, min(shard.band[1] * 16, H)) if shard is not None else (0, H)
        host_Gb = host_G[:, gy0:gy1].contiguous().pin_memory()
        h2d_bytes = sum(host[k].numel() * 4 for k in in_keys) + host_Gb.numel() * 4
        sets = []
        for _ in range(2):
            t_ = {k: torch.empty_like(host[k], device=dev).requires_grad_(True) for k in in_keys}
            sets.append((t_, torch.zeros_like(host_G, device=dev), torch.zeros(host['means3D'].shape[0], 3, device=dev, requires_grad=True),
                         torch.empty_like(host_Gb, device=dev)))
        copy_stream = torch.cuda.Stream(device=dev)
        rast = GaussianRasterizer(settings)

        def h2d(which):
            """Issue one step's host->device copies into input set `which` on the copy stream; returns the event that follows them."""
            t_, Gd, _, Gb = sets[which]
            with torch.cuda.stream(copy_stream), torch.no_grad():
                for k in in_keys:
                    t_[k].copy_(host[k], non_blocking=True)
                Gb.copy_(host_Gb, non_blocking=True)
                Gd[:, gy0:gy1].copy_(Gb)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return ev

        def compute(which, ev):
            t_, Gd, m2d, _ = sets[which]
            torch.cuda.current_stream().wait_event(ev)
            for v_ in list(t_.values()) + [m2d]:
                v_.grad = None
            if shard is not None:
                out = shard.rasterize(settings, t_['means3D'], m2d, t_['opacities'], t_['scales'], t_['rotations'],
                                      t_['colors'] if not use_sh else None, t_.get('shs') if use_sh else None,
                                      filter_mode=LGR_FILTER_MAX, want_aux=True)
            elif world > 1:      # band mode has no autograd front end: the C-ABI wrappers directly (round-1 path)
                o_ = t_['opacities'].detach().reshape(-1)
                dt = {k: v.detach() for k, v in t_.items()}
                img, radii, pid, pwp, pw, st = rasterize_forward(settings, dt['means3D'], o_, dt['scales'], dt['rotations'],
                                                                 dt['colors'], None, LGR_FILTER_MAX, True, tile_rows, num_owners=world)
                loss = (img * Gd).sum()
                if peer is not None:
                    peer.backward(st, Gd, dt['means3D'], o_, dt['scales'], dt['rotations'], dt['colors'])
                else:
                    rows = rasterize_backward(st, Gd, dt['means3D'], o_, dt['scales'], dt['rotations'], dt['colors'], None)
                    sharded.exchange_rows_to_owners(rows, st.band_counts_host, n)
                return loss
            else:
                out = rast(means3D=t_['means3D'], means2D=m2d, shs=t_.get('shs') if use_sh else None,
                           colors_precomp=t_['colors'] if not use_sh else None, opacities=t_['opacities'], scales=t_['scales'],
                           rotations=t_['rotations'], cov3D_precomp=None)
            loss = (out[0] * Gd).sum()
            loss.backward()
            return loss

        def run_e2e(steps, prefetch):
            """prefetch=True: the copies of step k+1 (other input set) are issued before step k's loss is read (double buffering);
            False: copy, compute, read back, strictly in turn."""
            ev, val = h2d(0), 0.0
            for k in range(steps):
                cur = k & 1
                nxt = None
                if prefetch and k + 1 < steps:
                    nxt = h2d(cur ^ 1)          # set cur^1 was last used by step k-1, whose loss has been read: free
                loss = compute(cur, ev)
                val = float(loss.item())        # D2H read of the step's result
                if not prefetch and k + 1 < steps:
                    nxt = h2d(cur ^ 1)
                ev = nxt
            return val

        ne = max(3, min(args.steps, 10))
        res = {}
        for mode in (False, True):
            run_e2e(4, mode)                        # warm-up (the caching allocator reaches its steady state)
            barrier()
            t0 = time.perf_counter()
            run_e2e(ne, mode)
            barrier()
            te = torch.tensor([(time.perf_counter() - t0) / ne], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            res[mode] = float(te.item())
        # Both schedules are end to end (every step's copies and its read-back are inside the timed region); which one wins
        # depends on the box (host memory placement, PCIe contention with the peer traffic of the other ranks), so the
        # headline is the better of the two and both are reported.
        best = min(res, key=res.get)
        e2e = {'value': n / res[best], 'unit': 'Gaussians/s', 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': 4,
               'ms_per_step': res[best] * 1e3, 'steps': ne,
               'api': ('SplatExchange.rasterize + autograd (each rank copies the Gaussians it owns)' if shard is not None else
                       'rasterize_forward / rasterize_backward (band mode has no autograd front end)' if world > 1 else
                       'GaussianRasterizer(...) + loss.backward()'),
               'h2d': 'every step copies all of its inputs from pinned host memory into one of two preallocated device sets on a copy '
                      'stream and reads the loss back; max over ranks, wall clock.  Two schedules are timed: pipelined (the copies of '
                      'step k+1 are issued before step k is read back) and serial (copy, compute, read back in turn); '
                      'ms_per_step is the faster one (`schedule`)',
               'schedule': 'pipelined' if best else 'serial',
               'ms_per_step_pipelined': res[True] * 1e3, 'ms_per_step_serial_copy': res[False] * 1e3}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = peaks()
    D_stock, D_bin = stats['D_stock'], stats['D']
    kb, b_min, b_model = algorithmic_bytes(n, H, W, D_bin, deg)             # what the launches actually process
    kb_stock, _, b_model_stock = algorithmic_bytes(n, H, W, D_stock, deg)   # SURVEY 8(d)'s stock radius-square rule, beside it
    kms = {'project_fwd': prof['project_fwd'][0], 'bin_sort': prof['tile_scan'][0] + prof['bin_scatter'][0] + prof['tile_sort'][0],
           'blend_fwd': prof['blend_fwd'][0], 'blend_bwd': prof['blend_bwd'][0], 'project_bwd': prof['project_bwd'][0]}
    kms = {k: v / args.steps for k, v in kms.items()}
    kms_bin = {k: prof[k][0] / args.steps for k in ('tile_scan', 'bin_scatter', 'tile_sort')}
    dom = max(kms, key=kms.get)
    ach = kb[dom] / (kms[dom] * 1e-3) / 1e9 if kms[dom] > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, 'profiles', 'traffic.json')
    if os.path.exists(tp) and world == 1:      # the ncu capture is of the single-GPU full-image launch
        traffic = json.load(open(tp)).get(args.workload, {}).get(dom)
    launches = int(round(sum(v[1] for v in prof.values()) * args.steps / prof_steps))      # of the K timed steps (counted in the profiled pass)
    line = {
        'metric': 'gaussians_per_s_fwd_bwd', 'value': n / (ms_step * 1e-3), 'unit': 'Gaussians/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'strong',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'mpix_per_s': W * H / (ms_step * 1e-3) / 1e6,
        'config': {'workload': workload_name(args.workload) + ('' if args.order == 'random' else f' [memory order: {args.order}]'),
                   'parallelism': (f'Gaussians sharded x{world} + tile-row bands x{world}: splat records pushed to the band owners, 2D gradients returned, over NVLink peer memory (shard mode)') if shard is not None else (f'tile-row bands x{world}, gradient rows ' + ('pushed to owner ranks over NVLink peer memory (fused in the backward kernel)' if peer is not None else 'NCCL all-to-all to owner ranks')) if world > 1 else 'single GPU', 'l2': 'inputs+intermediates > L2 (126 MB)' if n >= 1_000_000 else 'working set fits L2; not flushed',
                   'instances_stock_rule': D_stock, 'instances_binned': D_bin, 'longest_tile_list': stats['maxlen'], 'visible': stats['visible'],
                   'launch': ('device-sized calls (no host read-back inside a step); ' if sync_free else 'host-sized calls (one 32-byte read-back per forward); ') + 'CUDA graph: ' + graph_note,
                   'kernel_split': f'kernel_ms / phase_ms_rank0 come from a separate profiled pass of {prof_steps} steps (per-kernel CUDA events, plain launches)'},
        'roofline': {'bound': 'hbm', 'kernel': dom, 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak,
                     'traffic': traffic, 'peak_source': peak_src, 'algorithmic_bytes': kb[dom], 'kernel_ms': kms[dom],
                     'instances': 'binned (instances_binned): the (Gaussian, tile) pairs the launch processes',
                     'frac_stock_rule_instances': (kb_stock[dom] / (kms[dom] * 1e-3) / 1e9 / peak) if kms[dom] > 0 else 0.0},
        'roofline_step': {'b_model_bytes': b_model, 'b_min_bytes': b_min, 'achieved': b_model / (ms_step * 1e-3) / 1e9,
                          'frac': b_model / (ms_step * 1e-3) / 1e9 / peak, 'b_min_frac': b_min / (ms_step * 1e-3) / 1e9 / peak,
                          'frac_stock_rule_instances': b_model_stock / (ms_step * 1e-3) / 1e9 / peak},
        'kernel_ms': kms, 'kernel_ms_bin_sort': kms_bin, 'phase_ms_rank0': phases, 'gpu_launches': launches, 'clocks': clk, 'e2e': e2e,
    }
    if world > 1:
        line['parity'] = parity
        line['kernel_ms_exchange'] = {k: prof[k][0] / args.steps for k in ('shard_send', 'shard_recv', 'shard_return', 'shard_gather') if k in prof}
    if world == 1 and not args.no_cpu_baseline:
        from oracle import c_oracle          # the checker, timed as the CPU baseline (bounded sample)
        ns = min(n, CPU_SAMPLE[args.workload])
        sub = {k: v[:ns].numpy() for k, v in sc.items()}
        kw = dict(colors_precomp=sub['colors']) if deg == 0 else dict(shs=sub['shs'])
        def cpu_step():
            c_oracle.render(cam, sub['means3D'], sub['opacities'], sub['scales'], sub['rotations'], filter_mode=c_oracle.FILTER_MAX,
                            dL_dimage=G.numpy(), dtype=np.float32, want_aux=True, **kw)
        nthreads, tried = pick_cpu_threads(c_oracle, cpu_step)          # includes the warm-up
        times = []
        for rep in range(3):
            t0 = time.perf_counter()
            cpu_step()
            times.append(time.perf_counter() - t0)
        dt = float(np.median(times))
        line['cpu_baseline'] = {'value': ns / dt, 'unit': 'Gaussians/s', 'cores': c_oracle.num_threads(), 'kind': 'port',
                                'sample': f'first {ns} of {n} Gaussians, {W}x{H}, fwd+bwd, fp32 C oracle, {nthreads} OpenMP threads (fastest of '
                                          + ', '.join(f'{k}: {v:.2f} s' for k, v in sorted(tried.items())) + '), median of 3 repetitions after warm-up',
                                'seconds': dt, 'seconds_all': times}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
