"""GPU parity tests of the drop-in ops (through the C ABI) against
  (1) the CPU oracle on identical seeded inputs,
  (2) the reference's OWN CUDA extension on the same inputs (bit-exact), as recorded in tests/golden/ref_gpu.pkl.xz,
  (3) the golden fixtures recorded from the reference's Python.
Tolerance: bit-exact for int / bool outputs; 1e-5 relative for fp32 (BASELINE.json north_star)."""
import pytest
import torch

from tests.util import assert_close, assert_equal, assert_equal_ref, load_golden

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


@pytest.fixture(scope='module')
def ops():
    from unboundednerfpytorch_b200 import ops as _ops
    return _ops


def _rays(n, seed, kind='aabb'):
    g = torch.Generator().manual_seed(seed)
    if kind == 'aabb':
        ro = torch.randn(n, 3, generator=g) * 0.3 + torch.tensor([0., 0., -2.5])
        rd = torch.randn(n, 3, generator=g) * 0.3 + torch.tensor([0., 0., 1.])
        rd[::17, 0] = 0.0           # exercise the zero-component branch
        rd[5::23, 1] = 0.0
    else:
        ro = torch.rand(n, 3, generator=g) - 0.5
        rd = torch.randn(n, 3, generator=g)
    return ro.contiguous(), rd.contiguous()


BOX = (torch.tensor([-1., -1.1, -0.9]), torch.tensor([1.05, 1., 1.2]))


@pytest.mark.parametrize('n', [1, 7, 1000, 8192])
def test_ray_aabb_and_counts(ops, oracle, n):
    ro, rd = _rays(n, 777 + n)
    mn, mx = BOX
    args_c = (ro, rd, mn, mx)
    args_g = tuple(t.to(DEV) for t in args_c)
    tmin_c, tmax_c = oracle.infer_t_minmax(*args_c, 0.2, 1e9)
    tmin_g, tmax_g = ops.infer_t_minmax(*args_g, 0.2, 1e9)
    assert_close(tmin_g, tmin_c, what='t_min'); assert_close(tmax_g, tmax_c, what='t_max')
    ns_c = oracle.infer_n_samples(rd, tmin_c, tmax_c, 0.03)
    ns_g = ops.infer_n_samples(args_g[1], tmin_g, tmax_g, 0.03)
    # counts may differ only where (t_max-t_min)*|d|/stepdist sits within float rounding of an integer
    assert (ns_g.cpu() - ns_c).abs().max() <= 1 and (ns_g.cpu() != ns_c).float().mean() < 1e-3
    st_c, dr_c = oracle.infer_ray_start_dir(ro, rd, tmin_c)
    st_g, dr_g = ops.infer_ray_start_dir(args_g[0], args_g[1], tmin_g)
    assert_close(st_g, st_c, what='start'); assert_close(dr_g, dr_c, what='dir')
    ru = lambda ref: ref('render_utils_cuda')
    assert_equal_ref(f'infer_t_minmax/{n}', (tmin_g, tmax_g), lambda ref: ru(ref).infer_t_minmax(*args_g, 0.2, 1e9))
    assert_equal_ref(f'infer_n_samples/{n}', ns_g,
                     lambda ref: ru(ref).infer_n_samples(args_g[1], *ru(ref).infer_t_minmax(*args_g, 0.2, 1e9), 0.03))
    assert_equal_ref(f'infer_ray_start_dir/{n}', (st_g, dr_g), lambda ref: ru(ref).infer_ray_start_dir(args_g[0], args_g[1], tmin_g))


@pytest.mark.parametrize('n', [1, 33, 1024, 8192])
def test_sample_pts_on_rays(ops, oracle, n):
    ro, rd = _rays(n, 100 + n)
    mn, mx = BOX
    stepdist = 0.5 * 2 / 64
    out_g = ops.sample_pts_on_rays(ro.to(DEV), rd.to(DEV), mn.to(DEV), mx.to(DEV), 0.2, 1e9, stepdist)
    # floats too: same arithmetic, same compiler
    assert_equal_ref(f'sample_pts_on_rays/{n}', out_g, lambda ref: ref('render_utils_cuda').sample_pts_on_rays(
        ro.to(DEV), rd.to(DEV), mn.to(DEV), mx.to(DEV), 0.2, 1e9, stepdist))
    out_c = oracle.sample_pts_on_rays(ro, rd, mn, mx, 0.2, 1e9, stepdist)
    if torch.equal(out_g[4].cpu(), out_c[4]):
        for a, b, nm in zip(out_g, out_c, ('pts', 'mask_outbbox', 'ray_id', 'step_id', 'N_steps', 't_min', 't_max')):
            if a.dtype == torch.float32:
                assert_close(a, b, what=nm)
            elif nm == 'mask_outbbox':
                assert (a.cpu() != b).float().mean() < 1e-4      # points within an ulp of a bbox face
            else:
                assert_equal(a, b, nm)
    # structural properties (size independent)
    pts, mask, ray_id, step_id, n_steps, t_min, t_max = out_g
    assert int(n_steps.sum()) == pts.shape[0]
    assert (ray_id[1:] >= ray_id[:-1]).all()
    assert_equal(torch.bincount(ray_id, minlength=n), n_steps, 'ray_id histogram')
    first = torch.ones_like(ray_id, dtype=torch.bool); first[1:] = ray_id[1:] != ray_id[:-1]
    assert (step_id[first] == 0).all() and ((step_id[1:] - step_id[:-1])[~first[1:]] == 1).all()


def test_sample_ndc_and_bg(ops, oracle):
    ro, rd = _rays(257, 5, 'free')
    mn, mx = BOX
    pg, mg = ops.sample_ndc_pts_on_rays(ro.to(DEV), rd.to(DEV), mn.to(DEV), mx.to(DEV), 65)
    pc, mc = oracle.sample_ndc_pts_on_rays(ro, rd, mn, mx, 65)
    assert_close(pg, pc, what='ndc pts'); assert (mg.cpu() != mc).float().mean() < 1e-4
    tmax = torch.rand(257, generator=torch.Generator().manual_seed(6)) + 1
    bg = ops.sample_bg_pts_on_rays(ro.to(DEV), rd.to(DEV), tmax.to(DEV), 0.5, 32)
    bc = oracle.sample_bg_pts_on_rays(ro, rd, tmax, 0.5, 32)
    assert_close(bg, bc, rtol=2e-5, what='bg pts')
    assert_equal_ref('sample_ndc_pts_on_rays', (pg, mg), lambda ref: ref('render_utils_cuda').sample_ndc_pts_on_rays(
        ro.to(DEV), rd.to(DEV), mn.to(DEV), mx.to(DEV), 65))
    assert_equal_ref('sample_bg_pts_on_rays', bg, lambda ref: ref('render_utils_cuda').sample_bg_pts_on_rays(
        ro.to(DEV), rd.to(DEV), tmax.to(DEV), 0.5, 32))


@pytest.mark.parametrize('n', [0, 1, 999, 300000])
def test_maskcache_lookup(ops, oracle, n):
    g = torch.Generator().manual_seed(n)
    mask = torch.rand(33, 20, 41, generator=g) > 0.5
    xyz = torch.rand(n, 3, generator=g) * 3 - 1.5
    mn, mx = BOX
    scale = (torch.tensor(mask.shape).float() - 1) / (mx - mn)
    shift = -mn * scale
    out_g = ops.maskcache_lookup(mask.to(DEV), xyz.to(DEV), scale.to(DEV), shift.to(DEV))
    out_c = oracle.maskcache_lookup(mask, xyz, scale, shift)
    assert out_g.dtype == torch.bool and out_g.shape == (n,)
    assert_equal(out_g, out_c, 'maskcache vs oracle')           # same fma + round-half-away => bit exact
    if n > 0:
        assert_equal_ref(f'maskcache_lookup/{n}', out_g, lambda ref: ref('render_utils_cuda').maskcache_lookup(
            mask.to(DEV), xyz.to(DEV), scale.to(DEV), shift.to(DEV)))


def test_maskgrid_golden():
    from unboundednerfpytorch_b200 import grid as G
    r = load_golden('l1_grids.pt')['maskgrid']
    mg = G.MaskGrid(path=None, mask=r['mask'], xyz_min=r['xyz_min'], xyz_max=r['xyz_max']).to(DEV)
    assert_equal(mg(r['xyz'].to(DEV)), r['out'], 'MaskGrid.forward vs reference python')
    assert_close(mg.xyz2ijk_scale, r['scale']); assert_close(mg.xyz2ijk_shift, r['shift'])


@pytest.mark.parametrize('n', [0, 5, 4097, 1 << 20])
def test_raw2alpha(ops, oracle, n):
    g = torch.Generator().manual_seed(n + 1)
    d = torch.randn(n, generator=g) * 6
    if n > 4:
        d[:2] = torch.tensor([90., -90.])        # exp overflow -> inf, underflow -> 0
    gb = torch.randn(n, generator=g)
    e_g, a_g = ops.raw2alpha(d.to(DEV), -2.0, 0.5)
    e_c, a_c = oracle.raw2alpha(d, -2.0, 0.5)
    assert_close(a_g, a_c, what='alpha')
    fin = torch.isfinite(e_c)
    assert_close(e_g.cpu()[fin], e_c[fin], what='exp')
    assert torch.equal(torch.isinf(e_g.cpu()), torch.isinf(e_c))
    g_g = ops.raw2alpha_backward(e_g, gb.to(DEV), 0.5)
    g_c = oracle.raw2alpha_backward(e_c, gb, 0.5)
    assert_close(g_g, g_c, what='raw2alpha grad')
    itv = torch.rand(n, generator=g) + 0.1
    e2, a2 = ops.raw2alpha_nonuni(d.to(DEV), 0.3, itv.to(DEV))
    e2c, a2c = oracle.raw2alpha_nonuni(d, 0.3, itv)
    assert_close(a2, a2c, what='alpha nonuni')
    assert_close(ops.raw2alpha_nonuni_backward(e2, gb.to(DEV), itv.to(DEV))[fin.to(DEV)],
                 oracle.raw2alpha_nonuni_backward(e2c, gb, itv)[fin], what='nonuni grad')
    if n > 0:
        ru = lambda ref: ref('render_utils_cuda')
        assert_equal_ref(f'raw2alpha/{n}', (e_g, a_g), lambda ref: ru(ref).raw2alpha(d.to(DEV), -2.0, 0.5))
        assert_equal_ref(f'raw2alpha_backward/{n}', g_g,
                         lambda ref: ru(ref).raw2alpha_backward(ru(ref).raw2alpha(d.to(DEV), -2.0, 0.5)[0], gb.to(DEV), 0.5))


def _ragged(n_rays, max_len, seed, opaque_frac=0.3):
    g = torch.Generator().manual_seed(seed)
    lens = torch.randint(0, max_len + 1, (n_rays,), generator=g)
    lens[torch.rand(n_rays, generator=g) < 0.1] = 0
    ray_id = torch.repeat_interleave(torch.arange(n_rays), lens)
    alpha = torch.rand(len(ray_id), generator=g) * 0.05
    opaque = torch.rand(n_rays, generator=g) < opaque_frac
    alpha[opaque[ray_id]] = torch.rand(int(opaque[ray_id].sum()), generator=g) * 0.6
    return alpha, ray_id, lens


@pytest.mark.parametrize('n_rays,max_len', [(1, 5), (7, 9), (100, 70), (1000, 300), (8192, 64)])
def test_alpha2weight_ragged(ops, oracle, n_rays, max_len):
    alpha, ray_id, lens = _ragged(n_rays, max_len, n_rays * 31 + max_len)
    out_g = ops.alpha2weight(alpha.to(DEV), ray_id.to(DEV), n_rays)
    out_c = oracle.alpha2weight(alpha, ray_id, n_rays)
    names = ('weight', 'T', 'alphainv_last', 'i_start', 'i_end')
    for a, b, nm in zip(out_g, out_c, names):
        (assert_equal if a.dtype == torch.int64 else assert_close)(a, b, nm)     # identical double/float chain => i_end exact
    g = torch.Generator().manual_seed(3)
    gw, gl = torch.randn(len(alpha), generator=g), torch.randn(n_rays, generator=g)
    gg = ops.alpha2weight_backward(alpha.to(DEV), *out_g, n_rays, gw.to(DEV), gl.to(DEV))
    gc = oracle.alpha2weight_backward(alpha, *out_c, n_rays, gw, gl)
    assert_close(gg, gc, rtol=2e-5, atol=1e-6, what='alpha2weight grad')
    if len(alpha) > 0:
        ru = lambda ref: ref('render_utils_cuda')
        key = f'alpha2weight/{n_rays}-{max_len}'
        assert_equal_ref(key, out_g, lambda ref: ru(ref).alpha2weight(alpha.to(DEV), ray_id.to(DEV), n_rays))
        assert_equal_ref(key + '/backward', gg, lambda ref: ru(ref).alpha2weight_backward(
            alpha.to(DEV), *ru(ref).alpha2weight(alpha.to(DEV), ray_id.to(DEV), n_rays), n_rays, gw.to(DEV), gl.to(DEV)))


def test_alpha2weight_full_size_properties(ops):
    """BASELINE size 8192 x 512 (dense, no early stop) + an opaque variant: size-independent properties."""
    n_rays, S = 8192, 512
    g = torch.Generator().manual_seed(777)
    ray_id = torch.arange(n_rays).repeat_interleave(S).to(DEV)
    for scale in (1e-4, 0.2):
        alpha = (torch.rand(n_rays * S, generator=g) * scale).to(DEV)
        w, T, last, i_s, i_e = ops.alpha2weight(alpha, ray_id, n_rays)
        # telescoping identity: sum_i w_i + T_last == 1 per ray
        tot = w.view(n_rays, S).double().sum(1) + last.double()
        assert (tot - 1).abs().max() < 5e-5
        assert_equal(i_s, torch.arange(n_rays, device=DEV) * S, 'i_start')
        if scale < 1e-3:
            assert_equal(i_e, (torch.arange(n_rays, device=DEV) + 1) * S, 'i_end (no early stop)')
            ref64 = torch.cumprod(1 - alpha.view(n_rays, S).double(), 1)[:, -1]
            assert_close(last, ref64.float(), rtol=1e-5, what='T_last vs float64 cumprod')
        else:
            stopped = (i_e - i_s) < S
            assert stopped.all() and (last < 1e-3).all()
            idx = (i_e - 1).clamp(min=0)
            assert (T[idx] >= 1e-3).all()                     # the stop element itself still saw T >= 1e-3
            tail = torch.arange(S, device=DEV)[None] >= (i_e - i_s)[:, None]
            assert (w.view(n_rays, S)[tail] == 0).all() and (T.view(n_rays, S)[tail] == 1).all()


def test_autograd_functions_golden():
    """Raw2Alpha / Alphas2Weights autograd.Functions reproduce the reference's Functions (dvgo.py:430-488)."""
    from unboundednerfpytorch_b200.functional import Alphas2Weights, Raw2Alpha, Raw2Alpha_nonuni
    g = load_golden('l1_autograd_fns.pt')
    r = g['chain']
    dens = r['density'].to(DEV).requires_grad_(True)
    alpha = Raw2Alpha.apply(dens, torch.tensor([r['shift']], device=DEV), r['interval'])
    w, last = Alphas2Weights.apply(alpha, r['ray_id'].to(DEV), r['n_rays'])
    assert_close(alpha, r['alpha']); assert_close(w, r['weights']); assert_close(last, r['alphainv_last'])
    ((w * r['gw'].to(DEV)).sum() + (last * r['gl'].to(DEV)).sum()).backward()
    assert_close(dens.grad, r['grad_density'], rtol=2e-5, what='chain grad')
    n = g['nonuni']
    d2 = n['density'].to(DEV).requires_grad_(True)
    a2 = Raw2Alpha_nonuni.apply(d2, n['shift'], n['interval'].to(DEV))
    assert_close(a2, n['alpha'])
    (a2 * n['g'].to(DEV)).sum().backward()
    assert_close(d2.grad, n['grad_density'], what='nonuni grad')


@pytest.mark.parametrize('n_rays,n_pts', [(1, 1), (5, 8), (100, 133), (8192, 511)])
def test_cumdist_thres(ops, oracle, n_rays, n_pts):
    g = torch.Generator().manual_seed(n_rays + n_pts)
    dist = torch.rand(n_rays, n_pts, generator=g) * 0.02
    out_g = ops.cumdist_thres(dist.to(DEV), 0.0149)
    assert_equal(out_g, oracle.cumdist_thres(dist, 0.0149), 'cumdist vs oracle')     # same sequential float adds
    assert_equal_ref(f'cumdist_thres/{n_rays}-{n_pts}', out_g,
                     lambda ref: ref('ub360_utils_cuda').cumdist_thres(dist.to(DEV), 0.0149))


@pytest.mark.parametrize('shape,layout', [((1, 1, 5, 6, 7), 'ref'), ((1, 12, 9, 8, 10), 'ref'), ((9, 12, 6, 5, 7), 'cl'),
                                          ((1, 3, 33, 20, 41), 'cl'), ((2, 12, 20, 9, 11), 'cl'),
                                          ((1, 12, 40, 70, 11), 'cl'), ((3, 4, 17, 33, 40), 'cl')])
def test_total_variation(ops, oracle, shape, layout):
    from unboundednerfpytorch_b200 import grid as G
    g = torch.Generator().manual_seed(sum(shape))
    param = torch.randn(shape, generator=g) * 2
    for dense in (True, False):
        grad = torch.randn(shape, generator=g) * (torch.rand(shape, generator=g) > 0.6)
        grad_c = grad.clone()
        oracle.total_variation_add_grad(param, grad_c, 0.3, 0.2, 0.1, dense)
        p_g, g_g = param.to(DEV), grad.to(DEV)
        if layout == 'cl':
            p_g, g_g = G._as_cl3d(p_g), G._as_cl3d(g_g)
        ops.total_variation_add_grad(p_g, g_g, 0.3, 0.2, 0.1, dense)
        assert_close(g_g, grad_c, what=f'tv dense={dense}')
        if not dense:
            assert torch.equal(g_g.cpu()[grad == 0], grad[grad == 0])        # untouched where grad was 0

        def tv_ref(ref):
            g_r = grad.to(DEV)
            ref('total_variation_cuda').total_variation_add_grad(param.to(DEV), g_r, 0.3, 0.2, 0.1, dense)
            return g_r
        assert_equal_ref(f'total_variation_add_grad/{"x".join(map(str, shape))}/{layout}/{int(dense)}', g_g.contiguous(), tv_ref)
    tv = load_golden('l1_grids.pt')['tv']
    for k in ('dense1', 'dense0'):
        gg = tv[k]['grad_in'].to(DEV)
        ops.total_variation_add_grad(tv['param'].to(DEV), gg, tv['wx'], tv['wy'], tv['wz'], k == 'dense1')
        assert_close(gg, tv[k]['grad_out'], what='tv golden')


@pytest.mark.parametrize('n', [1, 7, 4096, 1000003])
def test_adam_variants(ops, oracle, n):
    g = torch.Generator().manual_seed(n)
    for mode in (0, 1, 2):
        p = torch.randn(n, generator=g); m = torch.zeros(n); v = torch.zeros(n)
        perlr = torch.rand(n, generator=g)
        pg, mg, vg, lg = p.to(DEV), m.to(DEV), v.to(DEV), perlr.to(DEV)
        pr, mr, vr = pg.clone(), mg.clone(), vg.clone()          # the reference's state (advanced while recording)
        for step in (1, 2, 3):
            grad = torch.randn(n, generator=g) * (torch.rand(n, generator=g) > 0.5)
            gg = grad.to(DEV)
            if mode == 0:
                oracle.adam_upd(p, grad, m, v, step, 0.9, 0.99, 0.1, 1e-8); ops.adam_upd(pg, gg, mg, vg, step, 0.9, 0.99, 0.1, 1e-8)
            elif mode == 1:
                oracle.masked_adam_upd(p, grad, m, v, step, 0.9, 0.99, 0.1, 1e-8); ops.masked_adam_upd(pg, gg, mg, vg, step, 0.9, 0.99, 0.1, 1e-8)
            else:
                oracle.adam_upd_with_perlr(p, grad, m, v, perlr, step, 0.9, 0.99, 0.1, 1e-8)
                ops.adam_upd_with_perlr(pg, gg, mg, vg, lg, step, 0.9, 0.99, 0.1, 1e-8)
            assert_close(pg, p, what=f'adam mode {mode} p'); assert_close(mg, m, what='m'); assert_close(vg, v, what='v')

            def adam_ref(ref, gg=gg, step=step):
                refm = ref('adam_upd_cuda')
                if mode == 0:
                    refm.adam_upd(pr, gg, mr, vr, step, 0.9, 0.99, 0.1, 1e-8)
                elif mode == 1:
                    refm.masked_adam_upd(pr, gg, mr, vr, step, 0.9, 0.99, 0.1, 1e-8)
                else:
                    refm.adam_upd_with_perlr(pr, gg, mr, vr, lg, step, 0.9, 0.99, 0.1, 1e-8)
                return pr, mr, vr
            assert_equal_ref(f'adam/{n}/mode{mode}/step{step}', (pg, mg, vg), adam_ref)


def test_masked_adam_golden_and_fused_tail(ops):
    from unboundednerfpytorch_b200.masked_adam import MaskedAdam
    g = load_golden('l1_masked_adam.pt')
    for mode in ('plain', 'masked', 'perlr'):
        r = g[mode]
        p = torch.nn.Parameter(r['p0'].to(DEV)); q = torch.nn.Parameter(r['q0'].to(DEV))
        opt = MaskedAdam([{'params': [p], 'lr': 0.1, 'skip_zero_grad': mode == 'masked'},
                          {'params': [q], 'lr': 1e-3, 'skip_zero_grad': False}])
        if mode == 'perlr':
            opt.per_lr = r['per_lr'].to(DEV)
        for (gp, gq), p_ref, q_ref in zip(r['grads'], r['ps'], r['qs']):
            p.grad, q.grad = gp.to(DEV), gq.to(DEV)
            opt.step()
            assert_close(p, p_ref, what=mode + ' p'); assert_close(q, q_ref, what=mode + ' q')
    # fused tail == TV followed by masked Adam, and it clears the consumed gradients
    gen = torch.Generator().manual_seed(9)
    shape = (3, 4, 7, 6, 9)
    for tv_mode in (0, 1, 2):
        param = torch.randn(shape, generator=gen).to(DEV)
        grad = (torch.randn(shape, generator=gen) * (torch.rand(shape, generator=gen) > 0.7)).to(DEV)
        m = torch.rand(shape, generator=gen).to(DEV) * 0.1; v = torch.rand(shape, generator=gen).to(DEV) * 0.1
        p2, g2, m2, v2 = param.clone(), grad.clone(), m.clone(), v.clone()
        if tv_mode:
            ops.total_variation_add_grad(p2, g2, 0.2, 0.2, 0.2, tv_mode == 1)
        ops.masked_adam_upd(p2, g2, m2, v2, 4, 0.9, 0.99, 0.1, 1e-8)
        ops.tv_adam_fused(param, grad, m, v, 0.2, 0.2, 0.2, tv_mode, 4, 0.9, 0.99, 0.1, 1e-8, skip_zero_grad=True, zero_grad=True)
        assert_equal(param, p2, 'fused tail param'); assert_equal(m, m2, 'fused tail m'); assert_equal(v, v2, 'fused tail v')
        assert (grad == 0).all()


@pytest.mark.parametrize('key', ['dense_C1', 'dense_C3', 'dense_C12', 'fourier_C1_F2', 'fourier_C12_F4', 'fourier_C3_F1'])
@pytest.mark.parametrize('layout', ['cl', 'ref'])
def test_grid_modules_golden(key, layout):
    """DenseGrid / FourierGrid forward + backward vs the reference modules (F.grid_sample) on the golden inputs."""
    from unboundednerfpytorch_b200 import grid as G
    r = load_golden('l1_grids.pt')[key]
    grid = r['grid'].to(DEV)
    grid = (G._as_cl3d(grid) if layout == 'cl' else grid.contiguous()).requires_grad_(True)
    out = G.grid_sample(grid, r['xyz'].to(DEV), r['xyz_min'], r['xyz_max'], r.get('num_freqs', 0))
    assert out.shape == r['out'].shape
    assert_close(out, r['out'], rtol=2e-5, atol=2e-6, what=key + ' fwd')
    (out * r['w'].to(DEV)).sum().backward()
    assert grid.grad.stride() == grid.stride()
    assert_close(grid.grad, r['grad_grid'], rtol=2e-5, atol=2e-6, what=key + ' bwd')


@pytest.mark.parametrize('C,F_,n', [(1, 0, 100000), (12, 0, 50000), (12, 4, 20000), (1, 4, 20000), (4, 2, 1000), (16, 0, 999)])
def test_grid_sample_vs_torch_and_adjoint(oracle, C, F_, n):
    """Seeded larger case vs the CPU oracle (torch F.grid_sample), plus the adjoint identity
    <A x, y> == <x, A^T y> that ties the scatter kernel to the gather kernel at any size."""
    from unboundednerfpytorch_b200 import grid as G
    g = torch.Generator().manual_seed(C * 100 + F_)
    P = 1 + 2 * F_ if F_ else 1
    grid = torch.randn(P, C, 23, 17, 29, generator=g)
    xyz = (torch.rand(n, 3, generator=g) * 2 - 1) * 1.25             # a few points outside [-1.2, 1.2]
    mn, mx = [-1.2] * 3, [1.2] * 3
    ref = oracle.fourier_grid_forward(grid, xyz, torch.tensor(mn), torch.tensor(mx), F_)
    gg = G._as_cl3d(grid.to(DEV)).requires_grad_(True)
    out = G.grid_sample(gg, xyz.to(DEV), mn, mx, F_)
    assert_close(out, ref, rtol=2e-5, atol=2e-6, what='gather')
    y = torch.randn(out.shape, generator=g).to(DEV)
    (out * y).sum().backward()
    lhs = (out.detach().double() * y.double()).sum()
    rhs = (gg.detach().double() * gg.grad.double()).sum()
    assert abs(lhs - rhs) <= 1e-4 * max(1.0, abs(lhs)), (lhs, rhs)


def test_host_scalar_cache_is_per_tensor_object():
    """The cached `.item()` of act_shift must not leak to a new tensor that reuses the freed address."""
    from unboundednerfpytorch_b200.functional import host_scalar
    for k in range(8):
        t = torch.tensor([float(k)], device=DEV)
        assert host_scalar(t) == float(k)
        t.add_(0.5)                                  # in-place update bumps the version
        assert host_scalar(t) == float(k) + 0.5
        del t


def test_rays_of_a_view_golden():
    """ubn_get_rays_of_a_view (one launch per view) vs the reference's dvgo.get_rays_of_a_view on every flag combination,
    and get_training_rays_flatten vs dvgo.get_training_rays_flatten (dvgo.py:492-612)."""
    from unboundednerfpytorch_b200 import rays as R
    rec = load_golden('l1_rays.pt')
    for v in rec['views']:
        o, d, vd = R.get_rays_of_a_view(v['H'], v['W'], v['K'].numpy(), v['c2w'], v['ndc'], v['inverse_y'], v['flip_x'],
                                        v['flip_y'], mode=v['mode'])
        tag = f"ndc={v['ndc']} inv={v['inverse_y']} fx={v['flip_x']} fy={v['flip_y']} {v['mode']}"
        assert o.is_cuda and o.shape == (v['H'], v['W'], 3)
        assert_close(o, v['rays_o'], rtol=2e-6, what='rays_o ' + tag)
        assert_close(d, v['rays_d'], rtol=2e-6, what='rays_d ' + tag)
        assert_close(vd, v['viewdirs'], rtol=2e-6, what='viewdirs ' + tag)
    o2, d2 = R.get_rays(5, 7, rec['views'][0]['K'].numpy(), rec['views'][0]['c2w'].to(DEV), False, False, False)
    assert_close(o2, rec['views'][0]['rays_o']); assert_close(d2, rec['views'][0]['rays_d'])
    f = rec['flatten']
    out = R.get_training_rays_flatten([im.to(DEV) for im in f['imgs']], f['poses'], f['HW'].numpy(), f['Ks'].numpy(),
                                      ndc=False, inverse_y=False, flip_x=False, flip_y=False)
    for a, k in zip(out[:4], ('rgb_tr', 'rays_o_tr', 'rays_d_tr', 'viewdirs_tr')):
        assert_close(a, f[k], rtol=2e-6, what=k)
    assert list(out[4]) == list(f['imsz'])
    # mode 'random': offsets in [0,1) of the pixel, statistically centred
    o3, d3, _ = R.get_rays_of_a_view(64, 64, rec['views'][0]['K'].numpy(), rec['views'][0]['c2w'], False, False, False, False,
                                     mode='random')
    _, dl, _ = R.get_rays_of_a_view(64, 64, rec['views'][0]['K'].numpy(), rec['views'][0]['c2w'], False, False, False, False,
                                    mode='lefttop')
    _, dc, _ = R.get_rays_of_a_view(64, 64, rec['views'][0]['K'].numpy(), rec['views'][0]['c2w'], False, False, False, False,
                                    mode='center')
    assert ((d3 - dl).abs().max() <= (1 / 9.1) * 1.8) and ((d3 - dc).mean().abs() < 5e-3)


def test_gather_ray_batch():
    """One-launch batch assembly == four index ops (run_train.py:204-212); negative indices wrap, bad ones raise."""
    from unboundednerfpytorch_b200 import rays as R
    g = torch.Generator().manual_seed(3)
    arrs = [torch.randn(1000, 3, generator=g).to(DEV) for _ in range(4)]
    sel = torch.randint(0, 1000, (4096,), generator=g)
    sel[:3] = torch.tensor([-1, -1000, 999])
    outs = R.gather_ray_batch(sel, *arrs)
    for o, a in zip(outs, arrs):
        assert_equal(o, a[sel.to(DEV)], 'gather')
    assert R.gather_ray_batch(sel[:0], arrs[0])[0].shape == (0, 3)
    with pytest.raises(IndexError):
        R.gather_ray_batch(torch.tensor([5, 1000]), arrs[0], arrs[1])


@pytest.mark.parametrize('n_rays,n_pts', [(1, 1), (37, 500), (8192, 300000), (64, 0)])
def test_render_loss_vs_torch(n_rays, n_pts):
    """ubn_render_loss (value + gradients in two launches) vs the reference's torch composition, run_train.py:254-279."""
    from unboundednerfpytorch_b200.functional import render_loss
    g = torch.Generator().manual_seed(n_rays + n_pts)
    rgbm = torch.rand(n_rays, 3, generator=g)
    last = torch.rand(n_rays, generator=g)
    last[::5] = 0.0                     # below the clamp: no gradient
    if n_rays > 3:
        last[1], last[2] = 1.0, 2e-6    # above the clamp (no gradient) / just inside it
    raw = torch.rand(n_pts, 3, generator=g)
    w = torch.rand(n_pts, generator=g)
    rid = torch.sort(torch.randint(0, n_rays, (n_pts,), generator=g)).values
    tgt = torch.rand(n_rays, 3, generator=g)

    def torch_loss(rgbm, last, raw, w, rid, tgt):
        loss = 1.0 * torch.nn.functional.mse_loss(rgbm, tgt)
        pout = last.clamp(1e-6, 1 - 1e-6)
        ent = -(pout * torch.log(pout) + (1 - pout) * torch.log(1 - pout)).mean()
        per = ((raw - tgt[rid]).pow(2).sum(-1) * w.detach()).sum() / len(rgbm)
        return loss + 1e-3 * ent + 1e-2 * per, (loss, ent, per)

    a = [t.clone().double().requires_grad_(t.dtype.is_floating_point and i < 3) for i, t in enumerate((rgbm, last, raw))]
    ref, terms = torch_loss(a[0], a[1], a[2], w.double(), rid, tgt.double())          # fp64 torch as the yardstick
    ref.backward()
    b = [t.clone().to(DEV).requires_grad_(True) for t in (rgbm, last, raw)]
    ret = dict(rgb_marched=b[0], alphainv_last=b[1], raw_rgb=b[2], weights=w.to(DEV), ray_id=rid.to(DEV))
    loss, t3 = render_loss(ret, tgt.to(DEV), 1.0, 1e-3, 1e-2)
    loss.backward()
    assert_close(loss.detach().cpu().double(), ref.detach(), rtol=2e-6, what='loss')
    for k, v in zip(('mse', 'entropy_last', 'rgbper'), terms):
        assert_close(t3[k].cpu().double(), v.detach(), rtol=2e-6, what=k)
    for mine, theirs, nm in zip(b, a, ('rgb_marched', 'alphainv_last', 'raw_rgb')):
        if n_pts == 0 and nm == 'raw_rgb':
            assert mine.grad is None or mine.grad.numel() == 0
            continue
        assert_close(mine.grad.cpu().double(), theirs.grad, rtol=2e-5, atol=1e-10, what='grad ' + nm)
    # terms switched off: no gradient to alphainv_last / raw_rgb, value = mse
    b2 = [t.clone().to(DEV).requires_grad_(True) for t in (rgbm, last, raw)]
    l2, _ = render_loss(dict(rgb_marched=b2[0], alphainv_last=b2[1], raw_rgb=b2[2], weights=w.to(DEV), ray_id=rid.to(DEV)),
                        tgt.to(DEV), 1.0, 0.0, 0.0)
    l2.backward()
    assert_close(l2.detach().cpu().double(), terms[0].detach(), rtol=2e-6, what='mse only')
    assert b2[1].grad is None and b2[2].grad is None


@pytest.mark.parametrize('n_rays,n_pts', [(3, 40), (64, 5000), (8192, 300000)])
def test_full_loss_set_vs_reference_composition(oracle, n_rays, n_pts):
    """The loss set the unbounded configs actually use (bicycle_single.py:25,48-57: weight_main, weight_freq = 5, weight_entropy_last,
    weight_nearclip = 1, weight_distortion = 0.05, weight_rgbper): render_loss (two launches + the distortion kernel) vs the
    reference's torch composition run_train.py:253-279 in fp64, with FourierMSELoss (FourierGrid_model.py:114-130) as written
    there (torch.fft.fft over the colour axis) and flatten_eff_distloss restated by the oracle (dcvgo.py:387-409 maths)."""
    from unboundednerfpytorch_b200.functional import render_loss
    g = torch.Generator().manual_seed(3 * n_rays + n_pts)
    rgbm, last = torch.rand(n_rays, 3, generator=g), torch.rand(n_rays, generator=g) * 0.98 + 0.01
    raw, w = torch.rand(n_pts, 3, generator=g), torch.rand(n_pts, generator=g) * 0.1
    dens = torch.randn(n_pts, generator=g)
    rid = torch.sort(torch.randint(0, n_rays, (n_pts,), generator=g)).values
    rid[-1] = n_rays - 1
    t = torch.rand(n_pts, generator=g) * 4
    s_ = 1 - 1 / (1 + t)
    tgt = torch.rand(n_rays, 3, generator=g)
    W = dict(main=1.0, freq=5.0, ent=1e-3, clip=1.0, dist=0.05, per=1e-2)
    near_thres, n_max = 0.7, 512

    def ref_loss(rgbm, last, raw, w, dens):
        mse = torch.nn.functional.mse_loss(rgbm, tgt.double())
        freq = torch.nn.functional.mse_loss(torch.fft.fft(rgbm, dim=-1).real, torch.fft.fft(tgt.double(), dim=-1).real)
        loss = W['main'] * mse + W['freq'] * freq
        pout = last.clamp(1e-6, 1 - 1e-6)
        loss = loss + W['ent'] * (-(pout * torch.log(pout) + (1 - pout) * torch.log(1 - pout)).mean())
        d = dens[t.double() < near_thres]
        loss = loss + W['clip'] * (d - d.detach()).sum()
        dist_l = oracle.flatten_eff_distloss(w, s_.double(), 1 / n_max, rid)
        loss = loss + W['dist'] * dist_l
        per = ((raw - tgt.double()[rid]).pow(2).sum(-1) * w.detach()).sum() / n_rays
        return loss + W['per'] * per, freq, dist_l

    a = [x.clone().double().requires_grad_(True) for x in (rgbm, last, raw, w, dens)]
    ref, freq, dist_l = ref_loss(*a)
    ref.backward()
    b = [x.clone().to(DEV).requires_grad_(True) for x in (rgbm, last, raw, w, dens)]
    ret = dict(rgb_marched=b[0], alphainv_last=b[1], raw_rgb=b[2], weights=b[3], raw_density=b[4], ray_id=rid.to(DEV), t=t.to(DEV),
               s=s_.to(DEV), n_max=n_max)
    loss, terms = render_loss(ret, tgt.to(DEV), W['main'], W['ent'], W['per'], weight_freq=W['freq'], weight_nearclip=W['clip'],
                              near_thres=near_thres, weight_distortion=W['dist'])
    loss.backward()
    assert_close(loss.detach().cpu().double(), ref.detach(), rtol=5e-6, what='loss')
    assert_close(terms['freq'].cpu().double(), freq.detach(), rtol=5e-6, what='freq term')
    assert_close(terms['distortion'].cpu().double(), dist_l.detach(), rtol=2e-5, what='distortion term')
    for mine, theirs, nm in zip(b, a, ('rgb_marched', 'alphainv_last', 'raw_rgb', 'weights', 'raw_density')):
        scale = float(theirs.grad.abs().max()) + 1e-30
        assert_close(mine.grad.cpu().double(), theirs.grad, rtol=2e-5, atol=1e-6 * scale, what='grad ' + nm)
    assert int((b[4].grad != 0).sum()) == int((t < near_thres).sum())


@pytest.mark.parametrize('n_rays,n_pts', [(1, 1), (50, 777), (8192, 200000), (9, 0)])
def test_composite_rgb_vs_torch(n_rays, n_pts):
    """ubn_composite_fwd/bwd == segment_coo(weights[:,None] * rgb, ray_id, zeros, 'sum') and its autograd (bit-exact forward
    against the two-op form through the same kernel family; gradients against torch index_add autograd)."""
    from unboundednerfpytorch_b200.functional import composite_rgb, segment_sum
    g = torch.Generator().manual_seed(n_rays * 7 + n_pts)
    w = torch.rand(n_pts, generator=g)
    rgb = torch.rand(n_pts, 3, generator=g)
    rid = torch.sort(torch.randint(0, n_rays, (n_pts,), generator=g)).values
    if n_pts > 10:
        rid[rid == 3] = 4                                   # an empty ray in the middle
    gout = torch.randn(n_rays, 3, generator=g)
    a = [t.clone().to(DEV).requires_grad_(True) for t in (w, rgb)]
    out = composite_rgb(a[0], a[1], rid.to(DEV), n_rays)
    out.backward(gout.to(DEV))
    b = [t.clone().to(DEV).requires_grad_(True) for t in (w, rgb)]
    two_op = segment_sum(b[0].unsqueeze(-1) * b[1], rid.to(DEV), n_rays)
    assert_equal(out, two_op, 'fused composite vs mul + segment_sum')
    c = [t.clone().double().requires_grad_(True) for t in (w, rgb)]
    ref = torch.zeros(n_rays, 3, dtype=torch.float64).index_add_(0, rid, c[0].unsqueeze(-1) * c[1])
    ref.backward(gout.double())
    assert_close(out.detach().cpu().double(), ref.detach(), rtol=1e-5, what='composite')
    if n_pts:
        assert_close(a[0].grad.cpu().double(), c[0].grad, rtol=1e-5, atol=1e-6, what='grad weights')
        assert_close(a[1].grad.cpu().double(), c[1].grad, rtol=1e-6, what='grad rgb')


@pytest.mark.parametrize('n_rays,n_pts', [(1, 1), (7, 40), (300, 20000), (8192, 400000)])
def test_distortion_loss_vs_oracle(oracle, n_rays, n_pts):
    """ubn_distortion_loss vs the oracle's restatement of flatten_eff_distloss (dcvgo.py:387-409 maths), value + grad."""
    from unboundednerfpytorch_b200.functional import flatten_eff_distloss
    g = torch.Generator().manual_seed(n_rays + 3 * n_pts)
    w = torch.rand(n_pts, generator=g) * 0.1
    s = torch.sort(torch.rand(n_pts, generator=g)).values
    rid = torch.sort(torch.randint(0, n_rays, (n_pts,), generator=g)).values
    rid[-1] = n_rays - 1
    wd = w.clone().double().requires_grad_(True)
    ref = oracle.flatten_eff_distloss(wd, s.double(), 1 / 64, rid)
    ref.backward()
    wg = w.clone().to(DEV).requires_grad_(True)
    out = flatten_eff_distloss(wg, s.to(DEV), 1 / 64, rid.to(DEV))
    out.backward()
    assert_close(out.detach().cpu().double(), ref.detach(), rtol=2e-5, what='distortion loss')
    # the gradient is a difference of prefix / suffix sums of size ~ 2 * s * sum(w) / R that nearly cancel: fp32 rounding is
    # relative to those terms, not to the (much smaller) result
    term = 2.0 * float(torch.zeros(n_rays, dtype=torch.float64).index_add_(0, rid, w.double()).max()) / n_rays
    assert_close(wg.grad.cpu().double(), wd.grad, rtol=1e-4, atol=2e-6 * term + 1e-12, what='grad w')

@pytest.mark.parametrize('shape', [(2, 12, 20, 9, 11), (1, 12, 40, 70, 11), (3, 4, 17, 33, 40)])
def test_tv_adam_pingpong_matches_two_sweeps(shape):
    """MaskedAdam.step_fused_tv (one ping-pong sweep) == total_variation_add_grad + step(), bit for bit, over 3 steps,
    dense and sparse TV, masked and plain Adam."""
    from unboundednerfpytorch_b200 import grid as G, ops
    from unboundednerfpytorch_b200.masked_adam import MaskedAdam
    for skip in (True, False):
        g = torch.Generator().manual_seed(sum(shape) + skip)
        init = torch.randn(shape, generator=g)
        pa = torch.nn.Parameter(G._as_cl3d(init.clone().to(DEV)))
        pb = torch.nn.Parameter(G._as_cl3d(init.clone().to(DEV)))
        oa = MaskedAdam([dict(params=[pa], lr=0.1, skip_zero_grad=skip)])
        ob = MaskedAdam([dict(params=[pb], lr=0.1, skip_zero_grad=skip)])
        for it in range(3):
            grad = (torch.randn(shape, generator=g) * (torch.rand(shape, generator=g) > 0.6)).to(DEV)
            pa.grad = torch.empty_like(pa, memory_format=torch.preserve_format).copy_(grad)
            pb.grad = torch.empty_like(pb, memory_format=torch.preserve_format).copy_(grad)
            dense = it != 1
            oa.step_fused_tv({pa: (0.3, 0.2, 0.1, dense)})
            ops.total_variation_add_grad(pb, pb.grad, 0.3, 0.2, 0.1, dense)
            ob.step()
            assert pa.stride() == pb.stride()
            assert_equal(pa.data, pb.data, f'param step {it} skip={skip}')
            assert_equal(pa.grad, pb.grad, 'grad after TV')
            assert_equal(oa.state[pa]['exp_avg'], ob.state[pb]['exp_avg'], 'exp_avg')
            assert_equal(oa.state[pa]['exp_avg_sq'], ob.state[pb]['exp_avg_sq'], 'exp_avg_sq')
