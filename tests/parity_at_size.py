"""Shared machinery of the at-size parity tests (tests/test_gpu_parity_at_size.py) and of the diagnostic script
scripts/parity_at_size_report.py: run the BENCHMARKED configurations (bench.py's workloads, 8192 rays x 512 samples) through

  (a) this library's fused CUDA path (models.*.forward + loss + backward), and
  (b) the reference's GPU path op for op: oracle.cpu_ref.model_forward on CUDA tensors with ext = the reference's OWN CUDA
      extension compiled into oracle/_ref (ATen grid_sample, cuBLAS rgbnet, index_add for torch_scatter) -- i.e. what
      FourierGrid_model.py:554-672 / dcvgo.py:264-384 execute on a GPU,

on identical seeded grids, rays and targets, and reduce the differences to a small dict of statistics.

north_star tolerance: sample indices / hit masks bit-exact; fp32 rgb / depth / weights within 1e-5 relative.  "Relative" is
taken against the larger of |reference value| and the tensor's scale (max |reference|): a per-element relative error of a
quantity that passes through zero (raw_density, gradients) is not meaningful, the usual rtol + atol = rtol * scale form is.
Gradients that pass through the ReLU MLP are additionally judged against an fp64 evaluation (colour_branch_fp64).
"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

RTOL = 1e-5
FLOAT_KEYS = ('rgb_marched', 'alphainv_last', 'depth', 'weights', 'raw_alpha', 'raw_density', 'raw_rgb', 't', 's', 'wsum_mid')

# name -> (bench workload, density N(mean, std), fast_color_thres, mask-cache keep probability)
CONFIGS = {
    'truck_dense': dict(workload='truck', mean=0.0, std=1.0, thres=0.0),             # the headline bench line (rho = 1)
    'truck_realistic': dict(workload='truck', mean=6.0, std=4.0, thres=1e-4),        # SURVEY 8d realistic mode: rays terminate
    'bicycle_dense': dict(workload='bicycle', mean=0.0, std=1.0, thres=0.0, mask_keep=0.9),   # DCVGO 320^3 + cumdist + mask cache
}


def build_pair(name, dev, n_rays=8192, seed=777):
    """-> (ours: nn.Module on dev, p: oracle parameter dict on dev, (ro, rd, vd, target) on dev, stepsize, flavor)."""
    import bench
    from oracle import cpu_ref
    from unboundednerfpytorch_b200 import models
    c = CONFIGS[name]
    flavor, kw, stepsize = bench.workload_kwargs(c['workload'])
    kw = dict(kw, fast_color_thres=c['thres'])
    torch.manual_seed(seed)
    cls = models.FourierGridModel if flavor == 'fouriergrid' else models.DirectContractedVoxGO
    m = cls(**kw)
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        m.density.grid.copy_(torch.randn(m.density.grid.shape, generator=g) * c['std'] + c['mean'])
        m.k0.grid.copy_(torch.randn(m.k0.grid.shape, generator=g))
        if flavor == 'dcvgo':
            m.mask_cache.mask.copy_(torch.rand(m.mask_cache.mask.shape, generator=g) < c.get('mask_keep', 1.0))
    state = {k: v.detach().clone().contiguous() for k, v in m.state_dict().items()}        # reference layout [P,C,X,Y,Z]
    p = cpu_ref.params_from_state(flavor, kw, state, requires_grad=False)
    for k, v in list(p.items()):
        if torch.is_tensor(v):
            p[k] = v.to(dev)
    p['rgbnet'] = {k: v.to(dev).requires_grad_(True) for k, v in p['rgbnet'].items()}
    for k in ('density_grid', 'k0_grid'):
        p[k] = p[k].requires_grad_(True)
    del state
    ours = m.to(dev)
    batch = [t.to(dev) for t in bench.synth_batch(n_rays, seed)]
    return ours, p, batch, stepsize, flavor


def _stat(a, b, scale=None, n=None):
    """Error statistics of a (ours) against b (reference GPU path):
    rel_scale = max |a-b| / max|b|                       (rtol * scale criterion)
    rel_elem  = max |a-b| / |b| over elements with |b| >= 1 % of the scale     (per-element relative error away from zero)
    frac_gt   = fraction of elements with |a-b| > 1e-5 * max(|b|, 1 % scale).
    scale, n: max |b| and the element count of the whole tensor when a and b are samples of it (n_sample elements)."""
    a, b = a.detach().float(), b.detach().float().reshape(a.shape)
    if a.numel() == 0:
        return dict(n=0, max_abs=0.0, scale=0.0, rel_scale=0.0, rel_elem=0.0, frac_gt=0.0)
    scale = b.abs().max().item() if scale is None else scale
    err = (a - b).abs()
    floor = 0.01 * scale if scale > 0 else 1.0
    big = b.abs() >= floor
    rel_elem = (err[big] / b.abs()[big]).max().item() if bool(big.any()) else 0.0
    frac = (err > RTOL * b.abs().clamp_min(floor)).float().mean().item()
    return dict(n=a.numel() if n is None else n, n_sample=a.numel(), max_abs=err.max().item(), scale=scale,
                rel_scale=err.max().item() / (scale if scale > 0 else 1.0), rel_elem=rel_elem, frac_gt=frac)


def colour_branch_fp64(flavor, p, ref, vd, target, n_rays, chunk=1 << 19):
    """fp64 re-evaluation of the colour branch of the reference's algorithm (feature-grid interpolation -> rgbnet -> composite ->
    the rgb-dependent loss terms of bench.step_loss) on the fp32 run's own sample set, sample positions, weights and targets:
    the yardstick for the gradients that flow through the ReLU MLP.

    Two fp32 implementations of a ReLU MLP cannot agree to 1e-5 on such gradients element by element: a pre-activation within
    rounding distance (~1e-7) of zero gets a different ReLU mask in cuBLAS, in this library and in exact arithmetic, which
    changes that sample's whole contribution (observed: ~40 of 1.3 M samples).  So gradient parity is stated against this fp64
    evaluation: this library must deviate from it no more (in size and in number of affected elements) than the reference's own
    fp32 GPU path does.  Returns ({name: fp64 grad}, n_ambiguous) -- n_ambiguous = samples with a pre-activation within 1e-6
    of zero."""
    from oracle import cpu_ref
    dev = vd.device
    dd = lambda t: t.detach().double()
    kg = dd(p['k0_grid']).requires_grad_(True)
    W = {k: dd(v).requires_grad_(True) for k, v in p['rgbnet'].items()}
    gmin = torch.tensor([-1., -1., -1.], device=dev, dtype=torch.float64) - p['bg_len']
    gmax = torch.tensor([1., 1., 1.], device=dev, dtype=torch.float64) + p['bg_len']
    ray_id, w = ref['ray_id'], dd(ref['weights'])
    emb_rays = cpu_ref.view_embedding(dd(vd), dd(p['viewfreq'])).flatten(0, -2)
    tgt = dd(target)
    M = ray_id.numel()
    marched = torch.zeros(n_rays, 3, device=dev, dtype=torch.float64)
    per_sum = torch.zeros((), device=dev, dtype=torch.float64)
    n_amb = 0
    # two passes would be needed for a chunked mse; instead accumulate rgb_marched with grad across chunks (graph kept per chunk)
    for lo in range(0, M, chunk):
        sl = slice(lo, min(lo + chunk, M))
        k0 = cpu_ref.fourier_grid_forward(kg, dd(ref['_ray_pts'][sl]), gmin, gmax, p['freq_k0'])
        x = torch.cat([k0, emb_rays[ray_id[sl]]], -1)
        z1 = torch.nn.functional.linear(x, W['W1'], W['b1'])
        z2 = torch.nn.functional.linear(torch.relu(z1), W['W2'], W['b2'])
        rgb = torch.sigmoid(torch.nn.functional.linear(torch.relu(z2), W['W3'], W['b3']))
        with torch.no_grad():
            n_amb += int(((z1.abs().amin(1) < 1e-6) | (z2.abs().amin(1) < 1e-6)).sum())
        marched = marched.index_add(0, ray_id[sl], w[sl, None] * rgb)
        per_sum = per_sum + (((rgb - tgt[ray_id[sl]]).pow(2).sum(-1)) * w[sl]).sum()
    marched = marched + (dd(ref['alphainv_last'])[:, None] * 1.0 if flavor == 'dcvgo' else 0.0)      # bg = 1 (dcvgo.py:350)
    loss = torch.nn.functional.mse_loss(marched, tgt) + 1e-2 * per_sum / n_rays
    loss.backward()
    grads = {'k0.grid': kg.grad}
    grads.update({'rgbnet.' + k: v.grad for k, v in W.items()})
    return grads, n_amb


def density_scatter_fp64(p, pts_q, g_density_q, chunk=1 << 20):
    """fp64 evaluation of the density-grid scatter: the adjoint of the reference's grid read (F.grid_sample over the slabs + mean)
    applied to the reference run's own per-sample gradients d loss / d raw_density.  The fp32 implementations (ATen's atomicAdd
    scatter in the reference, the vector reductions here) differ from each other only by the order -- and, in this library, the
    in-register merging -- of fp32 additions; this is what both are judged against."""
    from oracle import cpu_ref
    dev = pts_q.device
    kg = torch.zeros_like(p['density_grid'], dtype=torch.float64).requires_grad_(True)
    gmin = torch.tensor([-1., -1., -1.], device=dev, dtype=torch.float64) - p['bg_len']
    gmax = torch.tensor([1., 1., 1.], device=dev, dtype=torch.float64) + p['bg_len']
    for lo in range(0, pts_q.shape[0], chunk):
        sl = slice(lo, min(lo + chunk, pts_q.shape[0]))
        d = cpu_ref.fourier_grid_forward(kg, pts_q[sl].double(), gmin, gmax, p['freq_density'])
        (d.reshape(-1) * g_density_q[sl].double().reshape(-1)).sum().backward()
    return kg.grad


def _vs_truth(a, b, truth, scale=None, n=None):
    """Deviation of ours (a) and of the reference GPU path (b) from the fp64 yardstick, relative to max |truth| (scale and n: of
    the whole tensor, when a, b and truth are samples of it)."""
    t = truth.reshape(b.shape)
    scale = (t.abs().max().item() if scale is None else scale) or 1.0
    ea, eb = (a.detach().double() - t).abs(), (b.detach().double() - t).abs()
    tol = RTOL * scale
    return dict(scale=scale, ours_max=ea.max().item() / scale, ref_max=eb.max().item() / scale,
                ours_n_bad=int((ea > tol).sum()), ref_n_bad=int((eb > tol).sum()), n=a.numel() if n is None else n,
                n_sample=a.numel())


def compare(name, dev, n_rays=8192, backward=True, ext=None, truth=True):
    """Run both paths, return {'ids_equal', 'M', 'M_ref', key: stat..., 'grad <param>': stat..., 'truth <param>': ...}."""
    import bench
    from oracle import cpu_ref
    ours, p, (ro, rd, vd, target), stepsize, flavor = build_pair(name, dev, n_rays)
    out = {'config': name, 'flavor': flavor}
    rk = dict(near=0., far=1e9, bg=1, rand_bkgd=False, stepsize=stepsize, render_depth=True)
    ref = cpu_ref.model_forward(flavor, p, ro, rd, vd, stepsize, bg=1, rand_bkgd=False, render_depth=True, ext=ext,
                                keep_intermediates=True)
    ret = ours(ro, rd, vd, global_step=None, is_train=False, **rk)
    out['M'], out['M_ref'], out['n_max'] = int(ret['ray_id'].numel()), int(ref['ray_id'].numel()), int(ret['n_max'])
    same_shape = ret['ray_id'].shape == ref['ray_id'].shape
    out['ray_id_equal'] = bool(same_shape and torch.equal(ret['ray_id'], ref['ray_id']))
    out['step_id_equal'] = bool(same_shape and torch.equal(ret['step_id'], ref['step_id']))
    if not same_shape or not (out['ray_id_equal'] and out['step_id_equal']):
        ka = ret['ray_id'] * 65536 + ret['step_id']
        kb = ref['ray_id'] * 65536 + ref['step_id']
        in_b, in_a = torch.isin(ka, kb), torch.isin(kb, ka)
        out['flips'] = int((~in_b).sum() + (~in_a).sum())
        for k in FLOAT_KEYS:                       # diagnostics on the common samples / all rays (the test fails on flips anyway)
            if k in ref and k in ret:
                if ret[k].shape[0] == ret['ray_id'].shape[0] and ret[k].dim() >= 1 and k not in ('rgb_marched', 'alphainv_last', 'depth', 'wsum_mid'):
                    out[k] = _stat(ret[k][in_b], ref[k].reshape(ref['ray_id'].shape[0], *ret[k].shape[1:])[in_a])
                else:
                    out[k] = _stat(ret[k], ref[k])
        return out, ours, p
    out['flips'] = 0
    for k in FLOAT_KEYS:
        if k in ref and k in ret:
            out[k] = _stat(ret[k], ref[k])
    if backward:
        ours.zero_grad(set_to_none=True)
        bench.step_loss(ret, target, n_rays).backward()
        loss_ref = bench.step_loss(ref, target, n_rays)
        g_dq = torch.autograd.grad(loss_ref, ref['_density_q'], retain_graph=True)[0] if truth else None
        loss_ref.backward()
        pairs = [('density.grid', ours.density.grid.grad, p['density_grid'].grad), ('k0.grid', ours.k0.grid.grad, p['k0_grid'].grad)]
        names = {'W1': ours.rgbnet[0].weight, 'b1': ours.rgbnet[0].bias, 'W2': ours.rgbnet[2][0].weight,
                 'b2': ours.rgbnet[2][0].bias, 'W3': ours.rgbnet[3].weight, 'b3': ours.rgbnet[3].bias}
        pairs += [('rgbnet.' + k, v.grad, p['rgbnet'][k].grad) for k, v in names.items()]
        for nm, a, b in pairs:
            out['grad ' + nm] = _stat(a, b)
        if truth:
            grads64, out['n_relu_ambiguous'] = colour_branch_fp64(flavor, p, ref, vd, target, n_rays)
            for nm, a, b in pairs:
                if nm in grads64:
                    out['truth ' + nm] = _vs_truth(a, b, grads64[nm])
            out['truth density.grid'] = _vs_truth(pairs[0][1], pairs[0][2], density_scatter_fp64(p, ref['_pts_q'], g_dq))
            del g_dq
        # the reference against ITSELF: its grid scatters are fp32 atomicAdds (ATen grid_sampler_3d_backward), so two runs of the
        # reference differ by the summation order alone -- the floor any other implementation can be asked to reach
        first = {nm: b.detach().clone() for nm, a, b in pairs[:2]}
        for k in ('density_grid', 'k0_grid'):
            p[k].grad = None
        ref2 = cpu_ref.model_forward(flavor, p, ro, rd, vd, stepsize, bg=1, rand_bkgd=False, render_depth=False, ext=ext)
        bench.step_loss(ref2, target, n_rays).backward()
        out['refself density.grid'] = _stat(p['density_grid'].grad, first['density.grid'])
        out['refself k0.grid'] = _stat(p['k0_grid'].grad, first['k0.grid'])
        del ref2, first
    return out, ours, p


# ---------------------------------------------------------------------------------------------------------------------------
# The same comparison without the reference: record() keeps, per configuration, what compare() judges this library against --
# the sample set (digests); every reference output and gradient at SAMPLE fixed positions (k0.grid at K0_SAMPLE) with the scale
# of the whole tensor; the fp64 gradients at the first TRUTH_SAMPLE of those positions (as float32 differences from the
# reference's value: fp64-exact to ~1e-15 at float32 size) with the reference's deviation from them on those positions and on
# the whole tensor; the reference's run-to-run statistics on the whole tensors -- and compare_recorded() judges a run of this
# library against that record with the statistics above, taken on the stored positions against whole-tensor scales and counts.
SAMPLE = 256
K0_SAMPLE = 16384         # resolves the k0.grid bar frac_gt <= 1e-3 (16 elements); at 1.3e-4 (measured, full tensor) ~2 are expected
TRUTH_SAMPLE = 4096


def _index(nm, shape):
    from tests.util import sample_index
    return sample_index(shape, K0_SAMPLE if nm == 'k0.grid' else SAMPLE)


def _numel(shape):
    n = 1
    for s in shape:
        n *= int(s)
    return n


def count_bar(st):
    """Largest count of elements beyond 1e-5 of scale against fp64 (ours_n_bad) that passes the whole-tensor bar
    `ours_n_bad <= max(16, 3 x the reference's count)`.  On n_sample uniformly drawn positions of n, a tensor with N such elements
    shows a count of about Poisson(n_sample N / n): the bar is that mean for N = max(16, 3 x the reference's whole-tensor count)
    plus four of its standard deviations plus one, so a library within the whole-tensor bar passes on all but ~1e-4 of position
    draws, and one several times over it fails.  On a whole tensor (n_sample = n) it is the whole-tensor bar itself."""
    n, k = st['n'], st.get('n_sample', st['n'])
    lam = k / n * max(16, 3 * st.get('ref_n_bad_full', st['ref_n_bad']))
    return lam if k >= n else lam + 4 * lam ** 0.5 + 1


def record(name, dev, ext, n_rays=8192):
    """Run the reference GPU path (ext = its CUDA extension) once and reduce it to a record for compare_recorded()."""
    import bench
    from oracle import cpu_ref
    from tests.util import digest, sample_index, take
    _, p, (ro, rd, vd, target), stepsize, flavor = build_pair(name, dev, n_rays)
    ref = cpu_ref.model_forward(flavor, p, ro, rd, vd, stepsize, bg=1, rand_bkgd=False, render_depth=True, ext=ext,
                                keep_intermediates=True)
    rec = {'M_ref': int(ref['ray_id'].numel()), 'ray_id': digest(ref['ray_id']), 'step_id': digest(ref['step_id']), 'out': {},
           'grad': {}, 'truth': {}}
    for k in FLOAT_KEYS:
        if k in ref:
            t = ref[k].detach()
            rec['out'][k] = dict(shape=tuple(t.shape), scale=t.abs().max().item(), sample=take(t, sample_index(t.shape, SAMPLE)))
    loss_ref = bench.step_loss(ref, target, n_rays)
    g_dq = torch.autograd.grad(loss_ref, ref['_density_q'], retain_graph=True)[0]
    loss_ref.backward()
    grads = {'density.grid': p['density_grid'].grad, 'k0.grid': p['k0_grid'].grad}
    grads.update({'rgbnet.' + k: v.grad for k, v in p['rgbnet'].items()})
    for nm, g in grads.items():
        rec['grad'][nm] = dict(shape=tuple(g.shape), scale=g.abs().max().item(), sample=take(g, _index(nm, g.shape)))
    grads64, rec['n_relu_ambiguous'] = colour_branch_fp64(flavor, p, ref, vd, target, n_rays)
    grads64['density.grid'] = density_scatter_fp64(p, ref['_pts_q'], g_dq)
    del g_dq
    for nm, t in grads64.items():
        idx = _index(nm, t.shape)[:TRUTH_SAMPLE]
        b, tt = take(grads[nm], idx), take(t, idx)
        st = _vs_truth(b, b, tt, t.abs().max().item())
        full = _vs_truth(grads[nm], grads[nm], t)
        rec['truth'][nm] = dict(scale=full['scale'], delta=(tt - b.double()).float(), ref_max=st['ref_max'], ref_n_bad=st['ref_n_bad'],
                                ref_max_full=full['ref_max'], ref_n_bad_full=full['ref_n_bad'])
    del grads64
    first = {nm: grads[nm].detach().clone() for nm in ('density.grid', 'k0.grid')}
    for k in ('density_grid', 'k0_grid'):
        p[k].grad = None
    ref2 = cpu_ref.model_forward(flavor, p, ro, rd, vd, stepsize, bg=1, rand_bkgd=False, render_depth=False, ext=ext)
    bench.step_loss(ref2, target, n_rays).backward()
    rec['refself density.grid'] = _stat(p['density_grid'].grad, first['density.grid'])
    rec['refself k0.grid'] = _stat(p['k0_grid'].grad, first['k0.grid'])
    return rec


def compare_recorded(name, dev, rec, n_rays=8192):
    """compare() of this library's fused path against a record(): the same keys, the statistics taken on the stored positions
    ('n' = element count of the whole tensor, 'n_sample' = positions compared; 'truth' entries carry the reference's
    whole-tensor ref_max_full / ref_n_bad_full for count_bar).  'flips' is None when the sample set differs (the record holds
    its digest, not the samples)."""
    import bench
    from tests.util import digest, sample_index, take
    ours, p, (ro, rd, vd, target), stepsize, flavor = build_pair(name, dev, n_rays)
    del p
    out = {'config': name, 'flavor': flavor}
    rk = dict(near=0., far=1e9, bg=1, rand_bkgd=False, stepsize=stepsize, render_depth=True)
    ret = ours(ro, rd, vd, global_step=None, is_train=False, **rk)
    out['M'], out['M_ref'], out['n_max'] = int(ret['ray_id'].numel()), rec['M_ref'], int(ret['n_max'])
    out['ray_id_equal'] = digest(ret['ray_id']) == rec['ray_id']
    out['step_id_equal'] = digest(ret['step_id']) == rec['step_id']
    out['flips'] = 0 if out['ray_id_equal'] and out['step_id_equal'] else None
    for k, r in rec['out'].items():
        if k in ret:
            assert tuple(ret[k].shape) == r['shape'], f'{name} {k}: shape {tuple(ret[k].shape)} vs {r["shape"]}'
            out[k] = _stat(take(ret[k], sample_index(r['shape'], SAMPLE)), r['sample'], r['scale'], _numel(r['shape']))
    if out['flips'] is None:
        return out, ours
    ours.zero_grad(set_to_none=True)
    bench.step_loss(ret, target, n_rays).backward()
    names = {'density.grid': ours.density.grid, 'k0.grid': ours.k0.grid, 'rgbnet.W1': ours.rgbnet[0].weight,
             'rgbnet.b1': ours.rgbnet[0].bias, 'rgbnet.W2': ours.rgbnet[2][0].weight, 'rgbnet.b2': ours.rgbnet[2][0].bias,
             'rgbnet.W3': ours.rgbnet[3].weight, 'rgbnet.b3': ours.rgbnet[3].bias}
    for nm, v in names.items():
        r = rec['grad'][nm]
        assert tuple(v.grad.shape) == r['shape'], f'{name} grad {nm}: shape {tuple(v.grad.shape)} vs {r["shape"]}'
        n = _numel(r['shape'])
        a = take(v.grad, _index(nm, r['shape']))
        out['grad ' + nm] = _stat(a, r['sample'], r['scale'], n)
        if nm in rec['truth']:
            t = rec['truth'][nm]
            k = t['delta'].numel()
            b = r['sample'][:k]
            st = _vs_truth(a[:k], b, b.double() + t['delta'].double(), t['scale'], n)
            out['truth ' + nm] = dict(st, ref_max=t['ref_max'], ref_n_bad=t['ref_n_bad'], ref_max_full=t['ref_max_full'],
                                      ref_n_bad_full=t['ref_n_bad_full'])
    out['n_relu_ambiguous'] = rec['n_relu_ambiguous']
    out['refself density.grid'], out['refself k0.grid'] = rec['refself density.grid'], rec['refself k0.grid']
    return out, ours
