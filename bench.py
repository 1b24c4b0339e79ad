#!/usr/bin/env python
"""bench.py -- headline benchmark of the FourierGrid / DVGO rendering hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference|reference-gpu] [--workload truck|bicycle]
                    [--dump-outputs DIR]

Metric (BASELINE.json): ray-samples/sec, 8192 rays x 512 samples, one training iteration per step
(forward + loss + backward + total-variation + MaskedAdam, i.e. run_train.py:251-288 of the reference).
Workload `truck` = BASELINE config[1]: FourierGridModel, 153^3 grids (S = 512 at stepsize 0.5), F = 4 => 9 slabs,
12-channel k0 + 39->128->128->3 rgbnet, dense mode (fast_color_thres = 0, density ~ N(0,1), alpha_init 1e-4: every
nominal sample is live -- the roofline configuration of SURVEY.md 8d), synthetic seeded rays / grids (seed 777).
`bicycle` = config[2]: DirectContractedVoxGO 320^3 DenseGrid, stepsize 1.045 (S = 512).

One JSON line on stdout (rank 0).  `value` = device-timed throughput with the ray batch resident in HBM; `e2e` = same
step through the public model API with the batch in pinned HOST memory (H2D of rays + target, D2H of the loss, every
step, inside the timed region).  `roofline` = the dominant hand-written kernel, timed live with CUDA events inside the
timed region.  `cpu_baseline` / `--impl reference` = the reference's algorithm on the host cores (CPU oracle port of
the same step: torch F.grid_sample CPU path + C restatement of the CUDA-only ops) on a bounded ray sample, with the
thread count that is fastest for it.  `psnr_delta_vs_ref` = second half of the metric (oracle/psnr_check.py).
`--impl reference-gpu` (informative, not part of the driver contract) = the reference's GPU path on this B200: its
algorithm op by op with its own CUDA extension from oracle/_ref + ATen / cuBLAS.
A/B switches (env): UBN_BENCH_TAIL=peer|pipelined|sequential (training-step tail), UBN_BENCH_LOSS=fused|torch,
UBN_TV_IMPL=1|0 (streaming / element-per-thread TV; scripts/check_tv_stream.py), UBN_RGBNET_MODE=tc3|tc1|simt,
UBN_RGBNET_BWD_MODE=fused|tc3|simt (every mode is exercised by tests/test_gpu_models.py::test_fused_rgbnet_vs_torch),
UBN_NCCL_HIGH_PRIORITY=1|0, UBN_PEER_MAP=auto|symm|ipc.
`--dump-outputs DIR` (rank 0): after the timed steps, what the last timed step computed -- the returned arrays of the model
forward and the loss (training workloads) or the frame (render workloads), and the parameters after its update -- as
DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs (dump_outputs).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

N_RAYS, N_SAMPLES = 8192, 512
SEED = 777


DUMP_ROWS = 1 << 18      # arrays with more rows (first dimension) are dumped at this many fixed, seeded rows


def dump_outputs(out_dir, arrays):
    """Write each tensor as out_dir/<name>.npy: floating point as float32, integers / bools as float64 (exact).  A tensor with more
    than DUMP_ROWS rows is written at DUMP_ROWS rows drawn with a fixed seed from its row count, so arrays of one length share rows
    and two runs share positions.  Grids are flattened first.  Bounded at ~8 bytes x DUMP_ROWS x columns per array (~15 MB for
    the truck step)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach()
        if t.dim() >= 4:
            t = t.reshape(-1)
        if t.dim() and t.shape[0] > DUMP_ROWS:
            g = torch.Generator().manual_seed(SEED * 1000003 + t.shape[0])
            idx = torch.randint(0, t.shape[0], (DUMP_ROWS,), generator=g).sort().values
            t = t[idx.to(t.device)]
        t = t.float() if t.is_floating_point() else t.double()
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy())


def step_arrays(ret, loss, model):
    """The tensors of a forward's result dict, the loss and the parameters, named for dump_outputs."""
    out = {k: v for k, v in ret.items() if torch.is_tensor(v)}
    if loss is not None:
        out['loss'] = loss
    out.update({'param.' + k: v for k, v in model.named_parameters()})
    return out


def workload_kwargs(name):
    if name == 'truck':
        world = 153
        return 'fouriergrid', dict(xyz_min=[-1.] * 3, xyz_max=[1.] * 3, num_voxels_density=world ** 3,
                                   num_voxels_base_density=world ** 3, num_voxels_rgb=world ** 3,
                                   num_voxels_base_rgb=world ** 3, num_voxels_viewdir=-1, alpha_init=1e-4,
                                   fast_color_thres=0, rgbnet_dim=12, fourier_freq_num=4), 0.5
    if name == 'bicycle':
        world = 320
        return 'dcvgo', dict(xyz_min=[-1.] * 3, xyz_max=[1.] * 3, num_voxels=world ** 3, num_voxels_base=world ** 3,
                             alpha_init=1e-4, fast_color_thres=0, rgbnet_dim=12, contracted_norm='l2'), 1.045
    raise ValueError(name)


def synth_batch(n, seed):
    g = torch.Generator().manual_seed(seed)
    ro = torch.rand(n, 3, generator=g) - 0.5
    rd = torch.randn(n, 3, generator=g)
    vd = rd / rd.norm(dim=-1, keepdim=True)
    target = torch.rand(n, 3, generator=g)
    return ro, rd, vd, target


def step_loss(ret, target, n_rays):
    """The always-on loss terms of run_train.py:254-279: MSE + 1e-3 * entropy_last + 1e-2 * rgbper."""
    loss = torch.nn.functional.mse_loss(ret['rgb_marched'], target)
    pout = ret['alphainv_last'].clamp(1e-6, 1 - 1e-6)
    loss = loss + 1e-3 * (-(pout * torch.log(pout) + (1 - pout) * torch.log(1 - pout)).mean())
    rgbper = (ret['raw_rgb'] - target[ret['ray_id']]).pow(2).sum(-1)
    return loss + 1e-2 * (rgbper * ret['weights'].detach()).sum() / n_rays


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-lms', '50'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')] + [time.time()])

    def mark(self):
        """Timestamp the start of the timed region: only samples taken after it are reported (fallback: all)."""
        self.t0 = time.time()

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        t0 = getattr(self, 't0', 0.0)
        timed = [r for r in self.rows if len(r) >= 8 and r[-1] >= t0]
        if len(timed) >= 2:
            self.rows = timed
        sm = sorted(float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace('.', '').isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace('.', '').isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


def algorithmic_bytes(flavor, kwargs):
    """SURVEY.md 8d gather model, rho = 1: fwd 32*P_d + 32*C*P_k bytes per ray-sample; bwd = 2x (RMW scatter)."""
    P = (1 + 2 * kwargs.get('fourier_freq_num', 0)) if flavor == 'fouriergrid' else 1
    C = 12
    return {'march_density_fwd': 32 * P, 'march_feature_fwd': 32 * C * P,
            'march_density_bwd': 2 * 32 * P, 'march_feature_bwd': 2 * 32 * C * P}


def load_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    except Exception:
        return 6650.0, 'fallback (B200_PROFILING.md)'


def load_tensor_peak():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            return float(json.load(f)['bf16_tflops_sustained']), 'measured sustained bf16 (MEASURED_PEAKS.json)'
    except Exception:
        return 1400.0, 'fallback (B200_PROFILING.md)'


def load_traffic(kernel):
    try:
        with open(os.path.join(ROOT, 'profiles', 'traffic.json')) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


# ----------------------------------------------------------------------------------------------------------
_CPU_SCENE = {}


def cpu_reference_step(flavor, kwargs, stepsize, n_rays, threads, steps, warmup):
    """The reference's algorithm on host cores: oracle port of forward + loss + backward (torch F.grid_sample CPU path +
    C restatement of the CUDA-only ops) on a bounded ray sample of the same workload (same grids).  The TV / Adam sweeps
    are NOT included: the reference has no CPU implementation of them (CUDA-only extension), so the CPU figure covers
    LESS work per step than the GPU arm -- it flatters the baseline, never the GPU.  Returns ray-samples/s."""
    from oracle import cpu_ref
    from unboundednerfpytorch_b200 import models
    torch.set_num_threads(threads)
    p = _CPU_SCENE.get(flavor)
    if p is None:                                          # built once per process (1.7 GB of N(0,1) grids)
        torch.manual_seed(SEED)
        cls = models.FourierGridModel if flavor == 'fouriergrid' else models.DirectContractedVoxGO
        m = cls(**kwargs)                                  # CPU tensors; used only as a shape / init recipe
        g = torch.Generator().manual_seed(SEED)
        with torch.no_grad():
            m.density.grid.copy_(torch.randn(m.density.grid.shape, generator=g))
            m.k0.grid.copy_(torch.randn(m.k0.grid.shape, generator=g))
        state = {k: v.detach().contiguous() for k, v in m.state_dict().items()}
        p = _CPU_SCENE[flavor] = cpu_ref.params_from_state(flavor, kwargs, state, requires_grad=True)
        del m, state
    ro, rd, vd, target = synth_batch(n_rays, SEED)
    leaves = [p['density_grid'], p['k0_grid']] + list(p['rgbnet'].values())
    times = []
    for it in range(1, warmup + steps + 1):
        t0 = time.perf_counter()
        for x in leaves:
            x.grad = None
        ret = cpu_ref.model_forward(flavor, p, ro, rd, vd, stepsize, bg=1, rand_bkgd=False, render_depth=False)
        step_loss(ret, target, n_rays).backward()
        dt = time.perf_counter() - t0
        if it > warmup:
            times.append(dt)
    S = ret['n_max']
    return n_rays * S / (sum(times) / len(times)), sum(times) / len(times)


def gpu_reference_step(flavor, kwargs, stepsize, steps, warmup, dev):
    """SURVEY.md 8(d): "also time the patched reference CUDA path on the same B200 (the real competitor)".
    The reference's GPU training step op for op: its Python algorithm (oracle.cpu_ref.model_forward on CUDA tensors: ATen
    grid_sample, cuBLAS rgbnet, index_add for torch_scatter) + the reference's OWN CUDA extension compiled from
    /root/reference into oracle/_ref (raw2alpha / alpha2weight / maskcache / cumdist / total_variation / masked Adam),
    grids in the reference layout.  A baseline leg like cpu_baseline: nothing of this repo's library runs here.
    Returns (ms_per_step, survivors) or None when oracle/_ref is absent."""
    import importlib.util
    import types
    from oracle import cpu_ref
    from unboundednerfpytorch_b200 import models
    mods = {}
    for name in ('render_utils_cuda', 'total_variation_cuda', 'adam_upd_cuda', 'ub360_utils_cuda'):
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'oracle', '_ref', name + '.so')
        if not os.path.exists(path):
            return None
        spec = importlib.util.spec_from_file_location(name, path)
        mods[name] = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mods[name])
    ru = mods['render_utils_cuda']
    ext = types.SimpleNamespace(raw2alpha=ru.raw2alpha, raw2alpha_backward=ru.raw2alpha_backward, alpha2weight=ru.alpha2weight,
                                alpha2weight_backward=ru.alpha2weight_backward, maskcache_lookup=ru.maskcache_lookup,
                                cumdist_thres=mods['ub360_utils_cuda'].cumdist_thres)
    torch.manual_seed(SEED)
    cls = models.FourierGridModel if flavor == 'fouriergrid' else models.DirectContractedVoxGO
    m = cls(**kwargs)                                  # CPU tensors; shape / init recipe only
    g = torch.Generator().manual_seed(SEED)
    with torch.no_grad():
        m.density.grid.copy_(torch.randn(m.density.grid.shape, generator=g))
        m.k0.grid.copy_(torch.randn(m.k0.grid.shape, generator=g))
    state = {k: v.detach().clone().contiguous() for k, v in m.state_dict().items()}     # reference layout [P,C,X,Y,Z]
    del m
    p = cpu_ref.params_from_state(flavor, kwargs, state, requires_grad=False)
    for k, v in list(p.items()):
        if torch.is_tensor(v):
            p[k] = v.to(dev)
    p['rgbnet'] = {k: v.to(dev).requires_grad_(True) for k, v in p['rgbnet'].items()}
    for k in ('density_grid', 'k0_grid'):
        p[k] = p[k].requires_grad_(True)
    grids = [p['density_grid'], p['k0_grid']]
    leaves = grids + list(p['rgbnet'].values())
    adam = [(torch.zeros_like(x), torch.zeros_like(x)) for x in leaves]
    ro, rd, vd, target = [t.to(dev) for t in synth_batch(N_RAYS, SEED)]
    w_d = 1e-6 / N_RAYS * p['world_len'] / 128
    w_k = 1e-7 / N_RAYS * p['world_len'] / 128
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for it in range(1, warmup + steps + 1):
        if it == warmup + 1:
            torch.cuda.synchronize()
            e0.record()
        for x in leaves:
            x.grad = None
        ret = cpu_ref.model_forward(flavor, p, ro, rd, vd, stepsize, bg=1, rand_bkgd=False, render_depth=False, ext=ext)
        step_loss(ret, target, N_RAYS).backward()
        with torch.no_grad():
            mods['total_variation_cuda'].total_variation_add_grad(grids[0], grids[0].grad, w_d, w_d, w_d, True)
            mods['total_variation_cuda'].total_variation_add_grad(grids[1], grids[1].grad, w_k, w_k, w_k, True)
            for i, (x, (m1, m2)) in enumerate(zip(leaves, adam)):
                fn = mods['adam_upd_cuda'].masked_adam_upd if i < 2 else mods['adam_upd_cuda'].adam_upd
                fn(x, x.grad.contiguous(), m1, m2, it, 0.9, 0.99, 0.1 if i < 2 else 1e-3, 1e-8)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps, int(ret['weights'].numel())


def tune_cpu_reference(flavor, kwargs, stepsize, cores, n_steps, max_rays, budget_s=180.0):
    """(threads, rays) for the CPU legs: the thread count that is actually fastest for the oracle port (torch's CPU kernels on
    these shapes stop scaling long before 128 threads; an oversubscribed baseline would flatter the GPU arm), probed with one
    warm + one timed step on 32 rays each, and as many rays (<= max_rays) as keep n_steps steps within ~budget_s (the
    per-step cost is at most linear in the rays)."""
    probes = {}
    for th in sorted({min(c, cores) for c in (8, 16, 32, 64, cores)}):
        probes[th] = cpu_reference_step(flavor, kwargs, stepsize, 32, th, 1, 1)[1]
    best = min(probes, key=probes.get)
    fit = int(32 * (budget_s / max(n_steps, 1)) / max(probes[best], 1e-3)) // 16 * 16
    return best, max(32, min(max_rays, fit))


# ----------------------------------------------------------------------------------------------------------
FRAME_HW = (1067, 1600)      # Mip-NeRF-360 'garden' at the resolution BASELINE config 4 names


def frame_rays(dev, H, W):
    """One pinhole view (focal = W, SURVEY.md 8d) from inside the unit scene, rays built on the device (ray_gen.cu)."""
    import numpy as np
    from unboundednerfpytorch_b200 import rays as R
    K = np.array([[float(W), 0, W / 2], [0, float(W), H / 2], [0, 0, 1]], dtype=np.float64)
    c2w = torch.tensor([[1., 0., 0., 0.15], [0., 1., 0., -0.10], [0., 0., 1., 0.35]])
    ro, rd, vd = R._rays_of_a_view(H, W, K, c2w, False, False, False, False, 'center', device=dev)
    return ro.view(-1, 3), rd.view(-1, 3), vd.view(-1, 3)


def block_model(seed, dev):
    from unboundednerfpytorch_b200 import models
    flavor, kwargs, stepsize = workload_kwargs('bicycle')
    torch.manual_seed(seed)
    m = models.DirectContractedVoxGO(**kwargs).to(dev)
    g = torch.Generator(device=dev).manual_seed(seed)
    with torch.no_grad():
        m.density.grid.copy_(torch.randn(m.density.grid.shape, generator=g, device=dev))
        m.k0.grid.copy_(torch.randn(m.k0.grid.shape, generator=g, device=dev))
    return m, stepsize


def render_workload(args, emit):
    """BASELINE configs 4 and 5 (forward only, strong scaling: the frame is fixed, the ranks divide it / hold one block each).
    garden:     one 1600x1067 frame = 1 707 200 rays in 8192-ray chunks (run_render.py:56), DCVGO 320^3 + 12-ch k0 + rgbnet
                replicated, contiguous ray shards per rank, one all-gather of [rays, 5] (render.render_frame_sharded).
    missionbay: one block model per rank (seed 777 + rank, centroid on a line through the scene), every rank renders the
                whole frame, visibility gate + inverse-distance-weighted composite in one all-reduce (render.render_blocks_idw;
                eval_block_nerf.py:95-133, :215-216).  Rank 0 afterwards checks the composite against a single-GPU loop over all
                block models (outside the timed region)."""
    from unboundednerfpytorch_b200 import dist as ubdist, render as RD
    rank, world, local = ubdist.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    H, W = FRAME_HW
    ro, rd, vd = frame_rays(dev, H, W)
    n_rays = ro.shape[0]
    rk = dict(near=0., far=1e9, bg=1, rand_bkgd=False, stepsize=1.045, coherent_rays=args.tma)
    if args.workload == 'garden':
        model, _ = block_model(SEED, dev)
        fn = lambda: RD.render_frame_sharded(model, ro, rd, vd, rk)
    else:
        model, _ = block_model(SEED + rank, dev)
        cen = lambda r: [(-0.7 + 1.4 * r / max(world - 1, 1)) if world > 1 else 0.0, 0.0, 0.0]
        fn = lambda: RD.render_blocks_idw(model, ro, rd, vd, rk, centroid=cen(rank), cam_origin=ro[0])
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(max(args.warmup, 1)):
        out = fn()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    clocks.mark()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        torch.distributed.barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_arrays(out if args.workload == 'garden' else {'rgb_marched': out[0]}, None, model))
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
    ms_frame = ms.item() / args.steps
    clk = clocks.stop() if rank == 0 else None
    check = {}
    if args.workload == 'garden':
        frame = out['rgb_marched']
        # rank 0 re-renders three chunks that other ranks produced: the gathered frame must equal a local render bit for bit
        if rank == 0:
            worst = 0.0
            for c in (0, (n_rays // 8192) // 2, n_rays // 8192 - 1):
                sl = slice(c * 8192, min((c + 1) * 8192, n_rays))
                loc = RD.render_rays(model, ro[sl], rd[sl], vd[sl], rk)['rgb_marched']
                worst = max(worst, float((loc - frame[sl]).abs().max()))
            check = {'gathered_vs_local_max_abs': worst, 'frame_mean': float(frame.mean())}
    else:
        frame, info = out
        if world > 1:
            vis = torch.zeros(world, device=dev)
            vis[rank] = info['visible'].float()
            torch.distributed.all_reduce(vis)
        if rank == 0:
            num = torch.zeros(n_rays, 3, device=dev)
            den = torch.zeros((), device=dev)
            for r in range(world):                       # single-GPU restatement: loop over all block models on this GPU
                mb, _ = block_model(SEED + r, dev)
                o = RD.render_rays(mb, ro, rd, vd, rk, keys=('rgb_marched', 'alphainv_last'))
                v = ((1.0 - o['alphainv_last']).mean() > 0.05).float()
                w = (ro[0] - torch.tensor(cen(r), device=dev)).norm().clamp_min(1e-8).pow(-4) * v
                num += o['rgb_marched'] * w
                den += w
                del mb
            want = num / den.clamp_min(1e-30)
            check = {'composite_vs_single_gpu_loop_max_abs': float((frame - want).abs().max()), 'frame_mean': float(frame.mean()),
                     'visible_blocks': int(vis.sum()) if world > 1 else int(info['visible'])}
    if rank == 0:
        rays_total = n_rays * (world if args.workload == 'missionbay' else 1)
        emit({'metric': 'rays/sec (render, fwd only, 512 samples per ray)', 'value': rays_total / (ms_frame * 1e-3), 'unit': 'rays/s',
              'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_frame, 'higher_is_better': True,
              'scaling': 'strong' if args.workload == 'garden' else 'weak (one block model per GPU, same frame)',
              'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
              'config': {'workload': f'{args.workload}: DCVGO 320^3 DenseGrid + 12-ch k0 + rgbnet, one {W}x{H} frame = {n_rays} rays in '
                                     f'8192-ray chunks, 512 samples per ray, dense mode (thres=0)',
                         'step': 'one full frame (render, forward only)' + (' + IDW composite all-reduce' if args.workload == 'missionbay'
                                                                          else ' + frame all-gather'),
                         'parallelism': (f'rays sharded contiguously over {world} GPUs, grids replicated' if args.workload == 'garden'
                                         else f'{world} block models, one per GPU'),
                         'l2_policy': 'inputs larger than L2 (1.7 GB of grids)'},
              'ray_samples_per_s': rays_total * N_SAMPLES / (ms_frame * 1e-3), 'tma_feature_read': args.tma,
              'clocks': clk, 'check': check})
    if world > 1:
        torch.distributed.destroy_process_group()


# ----------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'reference-gpu'])
    ap.add_argument('--workload', default='truck', choices=['truck', 'bicycle', 'garden', 'missionbay'])
    ap.add_argument('--cpu-rays', type=int, default=1024, help='upper bound of the ray sample of the CPU legs (shrunk to fit the time budget)')
    ap.add_argument('--no-reduced-precision', action='store_true', help='skip the labelled TF32x1 rgbnet line')
    ap.add_argument('--feature-kernel', type=int, default=None, choices=[0, 1, 2, 3, 4, 5, 6],
                    help='A/B: pass-B kernel family (0 warp-cooperative, 1 lane-per-sample forward, 2 forward + backward); default = library default')
    ap.add_argument('--tma', action='store_true', help='A/B (render workloads): TMA-staged brick feature read instead of the gather kernel')
    ap.add_argument('--no-tma', action='store_true', help='(default; kept for old scripts)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-reference-gpu', action='store_true', help='skip the reference-GPU baseline leg (oracle/_ref + ATen) of the N = 1 line')
    ap.add_argument('--only-timed', action='store_true', help='warm-up + timed region only (for ncu captures)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed to DIR/<name>.npy (see dump_outputs)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup

    # fd 1 carries exactly one JSON line: native libraries (NCCL's "NCCL version ..." banner) write to stderr instead
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(json_fd, (json.dumps(obj) + '\n').encode())

    if args.workload in ('garden', 'missionbay'):
        if args.impl != 'ours':
            if int(os.environ.get('RANK', '0')) == 0:
                emit({'impl': args.impl, 'unavailable': 'the reference arm is defined for the training workloads (truck / bicycle) only'})
            return
        return render_workload(args, emit)
    from unboundednerfpytorch_b200 import dist as ubdist
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    flavor, kwargs, stepsize = workload_kwargs(args.workload)
    cores = os.cpu_count() or 1
    config = {'workload': f'{args.workload}: {flavor} {"153^3 F=4 (9 slabs)" if args.workload == "truck" else "320^3 DenseGrid"} '
                          f'+ 12-ch k0 + rgbnet, {N_RAYS} rays x {N_SAMPLES} samples per GPU, dense mode (thres=0)',
              'step': 'fwd + loss(mse+entropy_last+rgbper) + bwd + dense TV + MaskedAdam',
              'rays_per_gpu': N_RAYS, 'samples_per_ray': N_SAMPLES, 'parallelism': f'ray-sharded dp{max(world, 1)}, grids replicated',
              'l2_policy': 'inputs larger than L2: 1.7 GB (truck) / 1.7 GB (bicycle) of grid + equally large grad/Adam state'
                           ' touched every step'}

    # ------------------------------------------------------------------ reference arm: CPU, rank 0 only
    if args.impl == 'reference':
        if rank != 0:
            return
        # bounded sample, fastest thread count: see tune_cpu_reference
        cores, args.cpu_rays = tune_cpu_reference(flavor, kwargs, stepsize, cores, max(args.steps, 1) + args.warmup, args.cpu_rays)
        v, sec = cpu_reference_step(flavor, kwargs, stepsize, args.cpu_rays, cores, max(args.steps, 1), args.warmup)
        line = {'impl': 'reference', 'metric': 'ray-samples/sec (fwd+bwd train step) 8192x512', 'value': v, 'unit': 'ray-samples/s',
                'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3 * (N_RAYS / args.cpu_rays),
                'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': config,
                'cpu_baseline': {'value': v, 'unit': 'ray-samples/s', 'cores': cores, 'kind': 'port',
                                 'sample': f'{args.cpu_rays} of {N_RAYS} rays x {N_SAMPLES} samples, same grids, fwd+loss+bwd (no TV/Adam sweeps on CPU)'},
                'e2e': {'value': v, 'unit': 'ray-samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        emit(line)
        return

    # ------------------------------------------------------------------ informative: the reference's GPU path on this B200
    if args.impl == 'reference-gpu':
        if rank != 0:
            return
        dev = torch.device('cuda', 0)
        out = gpu_reference_step(flavor, kwargs, stepsize, max(args.steps, 1), max(args.warmup, 1), dev)
        if out is None:
            emit({'impl': 'reference-gpu', 'unavailable': 'oracle/_ref not built (needs /root/reference at build time)'})
            return
        ms, surv = out
        emit({'impl': 'reference-gpu', 'metric': 'ray-samples/sec (fwd+bwd train step) 8192x512',
              'value': N_RAYS * N_SAMPLES / (ms * 1e-3), 'unit': 'ray-samples/s', 'n_gpus': 1, 'steps': args.steps,
              'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'dtype': 'f32', 'data': 'synthetic',
              'config': config, 'survivors': surv,
              'what': "reference algorithm op by op on CUDA: ATen grid_sample + cuBLAS rgbnet + the reference's own CUDA "
                      "extension (oracle/_ref) for raw2alpha / alpha2weight / TV / masked Adam; none of this repo's kernels"})
        return

    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl ours needs a GPU (no CPU fallback exists)')
    rank, world, local = ubdist.init_from_env()
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    from unboundednerfpytorch_b200 import _cabi, models
    from unboundednerfpytorch_b200.functional import render_loss
    from unboundednerfpytorch_b200.masked_adam import create_optimizer_or_freeze_model
    _cabi.load()
    if args.feature_kernel is not None:
        from unboundednerfpytorch_b200 import ops as _ops
        _ops.set_feature_kernel(args.feature_kernel)
    torch.manual_seed(SEED)
    cls = models.FourierGridModel if flavor == 'fouriergrid' else models.DirectContractedVoxGO
    model = cls(**kwargs).to(dev)
    g = torch.Generator(device=dev).manual_seed(SEED)
    with torch.no_grad():
        model.density.grid.copy_(torch.randn(model.density.grid.shape, generator=g, device=dev))
        model.k0.grid.copy_(torch.randn(model.k0.grid.shape, generator=g, device=dev))
    cfg_train = dict(lrate_density=1e-1, lrate_k0=1e-1, lrate_rgbnet=1e-3, lrate_decay=20, skip_zero_grad_fields=['density', 'k0'])
    opt = create_optimizer_or_freeze_model(model, cfg_train, global_step=0)
    rk = dict(near=0., far=1e9, bg=1, rand_bkgd=False, stepsize=stepsize)
    params = [p for p in model.parameters() if p.requires_grad]
    # TV weight / (global ray count): with the mean-over-ranks gradient exchange the N-GPU step equals the 1-GPU step on the
    # concatenated batch of world x 8192 rays (run_train.py:283-287 divides by len(rays_o))
    n_global = N_RAYS * world
    tv_terms = model.tv_terms(1e-6 / n_global, 1e-7 / n_global, True)
    tail_mode = os.environ.get('UBN_BENCH_TAIL', 'peer')
    peer_tail = None
    if tail_mode == 'peer':
        try:
            peer_tail = ubdist.PeerTail(opt)
        except Exception as e:        # peer mapping unavailable on this box (no P2P / IPC): fall back to the NCCL-pipelined tail on ALL ranks
            sys.stderr.write(f'[bench] PeerTail unavailable on rank {rank} ({e!r}); using the pipelined NCCL tail\n')
            peer_tail = None
        if world > 1:                 # every rank must take the same route
            ok = torch.tensor([1 if peer_tail is not None else 0], device=dev)
            torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
            if int(ok.item()) == 0:
                if peer_tail is not None:
                    raise SystemExit('PeerTail came up on some ranks only; set UBN_BENCH_TAIL=pipelined')
                tail_mode = 'pipelined'
        elif peer_tail is None:
            tail_mode = 'pipelined'

    # every rank gets its own 8192-ray batch (weak scaling); host copies are pinned for the e2e leg
    host = [t.pin_memory() for t in synth_batch(N_RAYS, SEED + rank)]
    dev_batch = [t.to(dev) for t in host]

    tail_events = []
    survivors = [N_RAYS * N_SAMPLES]
    last_step = []                    # (ret, loss) of the latest step, kept only for --dump-outputs

    def train_step(ro, rd, vd, target, it):
        ret = model(ro, rd, vd, global_step=it, is_train=True, **rk)
        survivors[0] = int(ret['weights'].numel())        # M: samples that reach the feature grid / rgbnet (no sync: a shape)
        opt.zero_grad(set_to_none=True)
        if os.environ.get('UBN_BENCH_LOSS', 'fused') == 'torch':     # A/B switch: the reference's torch composition
            loss = step_loss(ret, target, N_RAYS)
        else:                                                        # same three terms, value + gradients in two launches
            loss, _ = render_loss(ret, target, 1.0, 1e-3, 1e-2)
        loss.backward()
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        ev[0].record()
        if peer_tail is not None:         # default: ONE sweep per grid over NVLink peer memory (reduce-scatter -> TV -> Adam -> all-gather)
            peer_tail.step(tv_terms)
        elif tail_mode == 'pingpong' and world == 1:      # A/B: single-sweep TV + Adam without the persistent gradient buffers
            opt.step_fused_tv(tv_terms, write_grad=False)
        elif tail_mode == 'sequential':   # A/B: whole-tensor all-reduce first, then the two sweeps
            if world > 1:
                ubdist.allreduce_grads(params)
            model.density_total_variation_add_grad(1e-6 / n_global, True)
            model.k0_total_variation_add_grad(1e-7 / n_global, True)
            opt.step()
        else:                             # A/B: slab-pipelined NCCL all-reduce || TV || Adam
            ubdist.reduce_tv_step(opt, tv_terms)
        ev[1].record()
        tail_events.append(ev)
        if args.dump_outputs:
            last_step[:] = [ret, loss]
        return loss

    def sync_all():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed_region(fn, steps):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)
        return ms.item()

    it = [0]

    def dev_step(_):
        it[0] += 1
        train_step(*dev_batch, it[0])

    def e2e_step(_):
        it[0] += 1
        ro, rd, vd, target = [t.to(dev, non_blocking=True) for t in host]
        loss = train_step(ro, rd, vd, target, it[0])
        return loss.item()                                   # D2H read of the step's result

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()                 # started before the warm-up (nvidia-smi needs ~1 s to produce its first row)
    for i in range(args.warmup):
        dev_step(i)
    torch.cuda.synchronize()
    clocks.mark()
    _cabi.TIMER = _cabi.KernelTimer()
    _cabi.reset_launch_count()
    del tail_events[:]
    ms_total = timed_region(dev_step, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, step_arrays(last_step[0], last_step[1], model))
    del last_step[:]
    tail_ms = sum(a.elapsed_time(b) for a, b in tail_events) / max(len(tail_events), 1)   # all-reduce + TV + Adam per step
    launches = _cabi.launch_count()
    ktimes = _cabi.TIMER.summary()
    _cabi.TIMER = None
    clk = clocks.stop() if rank == 0 else None
    if args.only_timed:
        if rank == 0:
            emit({'only_timed': True, 'ms_per_step': ms_total / args.steps, 'gpu_launches': launches,
                  'kernels_ms': {k: round(v[0], 4) for k, v in ktimes.items()}})
        if world > 1:
            torch.distributed.destroy_process_group()
        return
    for i in range(2):
        e2e_step(i)
    ms_e2e = timed_region(e2e_step, args.steps)

    # forward-only (render) throughput, for context
    def fwd_only(_):
        with torch.no_grad():
            model(*dev_batch[:3], global_step=None, is_train=False, **rk)
    fwd_only(0)
    ms_fwd = timed_region(fwd_only, args.steps)

    # second, clearly labelled line: the same step with the rgbnet at ONE TF32 pass per product (the opt-in reduced-precision
    # training mode, UBN_RGBNET_MODE=tc1; ~1e-3 relative error inside the MLP, gated at |PSNR delta| <= 0.01 dB by
    # tests/test_gpu_models.py).  Not the headline: the headline computes at fp32 grade (3xTF32), the reference's own precision.
    ms_tc1 = None
    if world == 1 and not args.no_reduced_precision:
        from unboundednerfpytorch_b200 import shade as _shade
        mode0, _shade.MODE = _shade.MODE, 'tc1'
        try:
            for i in range(3):
                dev_step(i)
            ms_tc1 = timed_region(dev_step, args.steps)
        finally:
            _shade.MODE = mode0

    if rank != 0:
        if world > 1:
            torch.distributed.destroy_process_group()
        return

    samples_per_step = N_RAYS * N_SAMPLES * world
    ms_per_step = ms_total / args.steps
    value = samples_per_step / (ms_per_step * 1e-3)
    peak, peak_src = load_peaks()
    abytes = algorithmic_bytes(flavor, kwargs)
    tpeak, tsrc = load_tensor_peak()
    # rgbnet kernels are FLOP-bound: 2*(12*128 + 128*128 + 128*3) FLOP/sample forward, 2x that backward (dX and dW GEMMs)
    aflops = {'rgbnet_fwd': 2 * (12 * 128 + 128 * 128 + 128 * 3), 'rgbnet_bwd': 4 * (128 * 128)}   # bwd: dH1 + dW2 GEMMs
    abytes['rgbnet_bwd_small'] = 128 * 4 * 2 + 12 * 4 * 2 + 3 * 4 * 2   # streams dZ1 + H2 rows, X, rgb/grad_rgb, writes dX
    # SURVEY.md 8d: B = 32 P_d per NOMINAL sample + rho * 32 C P_k per nominal sample, rho = M / (N S): the density pass touches
    # every nominal sample, the feature / rgbnet kernels only the M survivors of cumdist + mask cache + thresholds
    M = survivors[0]
    units = {k: (N_RAYS * N_SAMPLES if k.startswith('march_density') else M) for k in list(abytes) + list(aflops)}
    traffic_src = 'profiles/traffic.json (static: dram__bytes_read.sum + dram__bytes_write.sum of the committed ncu --set full capture of this kernel on the truck workload, not re-measured in this run)'

    def kernel_roof(name, kms):
        if name in abytes:
            ach = abytes[name] * units[name] / (kms * 1e-3) / 1e9
            traffic = load_traffic(name) if args.workload == 'truck' else None
            out = {'kernel': name, 'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s', 'frac': ach / peak,
                   'traffic': traffic, 'traffic_source': traffic_src, 'kernel_ms': kms,
                   'algorithmic_bytes_per_sample': abytes[name], 'samples_per_launch': units[name], 'peak_source': peak_src}
            if traffic:
                # the physical side of the same launch: DRAM bytes of the committed ncu capture over this run's kernel time
                out['dram_achieved'] = traffic / (kms * 1e-3) / 1e9
                out['dram_frac'] = out['dram_achieved'] / peak
            if out['frac'] > 1.0:
                out['note'] = ('frac > 1: SURVEY 8d counts every corner record of every sample as HBM traffic; neighbouring samples share '
                               'corners in L1 / L2 (and the scatter merges equal cells in registers), so the kernel moves fewer DRAM bytes '
                               'than the model -- dram_frac is the physical utilisation')
            return out
        ach = aflops[name] * units[name] / (kms * 1e-3) / 1e12
        return {'kernel': name, 'bound': 'tensor', 'achieved': ach, 'peak': tpeak, 'unit': 'TFLOP/s', 'frac': ach / tpeak,
                'traffic': load_traffic(name) if args.workload == 'truck' else None, 'traffic_source': traffic_src, 'kernel_ms': kms,
                'algorithmic_flops_per_sample': aflops[name], 'samples_per_launch': units[name],
                'peak_source': tsrc, 'note': 'tcgen05 kind::tf32 with 3-pass split accumulation (fp32-grade, needed for the 1e-5 parity gate): useful FLOPs are '
                                             'counted once, the tensor pipe executes 3x that at half the bf16 rate; measured against the bf16 peak'}

    dom = max(ktimes, key=lambda k: ktimes[k][0]) if ktimes else None
    roof = None
    if dom:
        roof = kernel_roof(dom, ktimes[dom][0])
        roof['all_kernels_ms'] = {k: round(v[0], 4) for k, v in ktimes.items()}
        roof['all_kernels_frac'] = {k: round(kernel_roof(k, v[0])['frac'], 4) for k, v in ktimes.items()}
        hbm_k = [k for k in ktimes if k in abytes]
        if hbm_k:
            kd = max(hbm_k, key=lambda k: ktimes[k][0])
            roof['dominant_hbm_kernel'] = kernel_roof(kd, ktimes[kd][0])
    h2d = sum(t.numel() * t.element_size() for t in host)
    line = {'metric': 'ray-samples/sec (fwd+bwd train step) 8192x512', 'value': value, 'unit': 'ray-samples/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config, 'clocks': clk,
            'e2e': {'value': samples_per_step / (ms_e2e / args.steps * 1e-3), 'unit': 'ray-samples/s',
                    'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': 4, 'ms_per_step': ms_e2e / args.steps},
            'gpu_launches': launches, 'survivors_per_step': M, 'rho': M / (N_RAYS * N_SAMPLES), 'roofline': roof,
            'tail_ms': {'value': tail_ms, 'what': 'gradient all-reduce (N>1) + dense TV + MaskedAdam, per step',
                        'mode': tail_mode},
            'fwd_only': {'value': samples_per_step / (ms_fwd / args.steps * 1e-3), 'unit': 'ray-samples/s',
                         'ms_per_step': ms_fwd / args.steps}}
    # north_star's target is stated on the fused sample + interpolate + composite forward: SURVEY 8d forward bytes of the whole render
    # pass (density read for every nominal sample + feature read for the survivors) over its measured time, against the HBM peak
    fwd_bytes = (abytes['march_density_fwd'] * N_RAYS * N_SAMPLES + abytes['march_feature_fwd'] * M) * world
    fwd_gbs = fwd_bytes / (ms_fwd / args.steps * 1e-3) / 1e9
    line['fwd_only'].update({'algorithmic_bytes': fwd_bytes, 'achieved_gbs': fwd_gbs, 'frac_of_hbm_peak': fwd_gbs / (peak * world),
                             'what': 'whole forward / render pass (march + rgbnet + composite, no backward)'})
    if ms_tc1 is not None:
        line['reduced_precision_tf32x1'] = {
            'ms_per_step': ms_tc1 / args.steps, 'value': samples_per_step / (ms_tc1 / args.steps * 1e-3), 'unit': 'ray-samples/s',
            'dtype': 'tf32 x1 inside the rgbnet (fp32 everywhere else)',
            'note': 'NOT the headline: same step with one TF32 pass per product in the rgbnet forward and backward (opt-in training mode, '
                    'PSNR delta gated <= 0.01 dB in tests/test_gpu_models.py); the headline value computes at fp32 grade (3xTF32)'}
    if world == 1 and not args.no_reference_gpu:
        # the real competitor (SURVEY.md 8d): the reference's GPU path on this same B200 -- its algorithm op by op with its own CUDA
        # extension (oracle/_ref) + ATen grid_sample + cuBLAS; a baseline leg like cpu_baseline, outside every timed region above
        try:
            torch.cuda.empty_cache()
            out = gpu_reference_step(flavor, kwargs, stepsize, 5, 2, dev)
            line['reference_gpu'] = ({'ms_per_step': out[0], 'value': N_RAYS * N_SAMPLES / (out[0] * 1e-3), 'unit': 'ray-samples/s',
                                      'survivors': out[1], 'speedup_vs_reference_gpu': out[0] / ms_per_step,
                                      'what': "reference algorithm op by op on this GPU: ATen grid_sample + cuBLAS rgbnet + the reference's own "
                                              "CUDA extension (oracle/_ref) for raw2alpha / alpha2weight / TV / masked Adam; same step, same grids"}
                                     if out is not None else {'unavailable': 'oracle/_ref not built'})
        except Exception as e:
            line['reference_gpu'] = {'unavailable': f'failed: {e}'}
    if not args.no_cpu_baseline and world == 1:              # rank 0 at N = 1 only
        try:
            cores, args.cpu_rays = tune_cpu_reference(flavor, kwargs, stepsize, cores, 2, args.cpu_rays, budget_s=30.0)
            v, sec = cpu_reference_step(flavor, kwargs, stepsize, args.cpu_rays, cores, 1, 1)
            line['cpu_baseline'] = {'value': v, 'unit': 'ray-samples/s', 'cores': cores, 'kind': 'port',
                                    'sample': f'{args.cpu_rays} of {N_RAYS} rays x {N_SAMPLES} samples, same grids, fwd+loss+bwd (no TV/Adam sweeps on CPU), '
                                              f'{sec:.1f} s/step'}
        except Exception as e:                                           # never lose the GPU numbers to a CPU-side problem
            line['cpu_baseline'] = {'value': None, 'unit': 'ray-samples/s', 'cores': cores, 'kind': 'port', 'sample': f'failed: {e}'}
        try:
            # second half of BASELINE.json's metric: PSNR delta vs ref on the procedural teacher / student scene, the oracle as
            # the checker (oracle/psnr_check.py; same protocol as tests/test_gpu_models.py::test_psnr_delta_vs_oracle)
            from oracle.psnr_check import psnr_delta
            torch.set_num_threads(cores)
            pd = psnr_delta(flavor, 3 if flavor == 'fouriergrid' else 0, dev)
            line['psnr_delta_vs_ref'] = {'delta_db': pd['delta_db'], 'psnr_ref_db': pd['psnr_oracle'], 'psnr_ours_db': pd['psnr_cuda'],
                                         'ours_vs_ref_image_db': pd['psnr_cuda_vs_oracle'],
                                         'scene': 'procedural teacher / noisy student, 2 views 24x24, 32^3 grids (no datasets offline)'}
        except Exception as e:
            line['psnr_delta_vs_ref'] = {'delta_db': None, 'failed': str(e)}
    emit(line)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == '__main__':
    main()
