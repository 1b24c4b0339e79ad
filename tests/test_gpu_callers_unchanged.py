""""Callers unchanged" (BASELINE.json north_star, SURVEY.md 8b), checked against a stored run.  When recording
(UBN_RECORD_REF_GOLDEN, see tests/util.py) the reference's OWN Python files -- FourierGrid_model.py, dcvgo.py, dvgo.py, grid.py,
FourierGrid_grid.py, masked_adam.py, staged UNMODIFIED by __graft_entry__.build() into git-ignored oracle/_ref/py/ where the
reference checkout is readable -- are imported over ``legacy.install()`` (this library behind the four bare-name extension
modules render_utils_cuda / total_variation_cuda / adam_upd_cuda / ub360_utils_cuda) and run on the GPU exactly as run_train.py
drives them: model.forward, loss.backward, *_total_variation_add_grad, MaskedAdam.step.  What they return is stored in
tests/golden/ref_gpu.pkl.xz (digests, scales and 256 fixed positions per tensor).  Otherwise the reference's files and the
legacy shim are NOT run: the test checks that this library's own model classes (fused path) match that stored run on the same
state dict: sample ids bit-exact, floats within 1e-5 of the scale, parameters after one MaskedAdam step bit-exact.

This doubles as the cleanest reference-GPU oracle: every torch op in the staged files is the reference's, only the four
extension modules (and the un-vendored torch_scatter / torch_efficient_distloss packages) are ours."""
import os
import sys
import types

import pytest
import torch

from tests.util import RECORD, ROOT, assert_equal_summary, record_golden, ref_golden, sample_index, summarize, take

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
PY = os.path.join(ROOT, 'oracle', '_ref', 'py')
SAMPLE = 256
OUT_KEYS = ('rgb_marched', 'alphainv_last', 'weights', 'raw_alpha', 'raw_density', 'raw_rgb', 'depth')


@pytest.fixture(scope='module')
def ref_modules():
    """The reference's staged model / optimizer modules over this library: needed only while recording."""
    if not RECORD:
        return None
    from unboundednerfpytorch_b200 import functional as F_, legacy
    legacy.install()
    ts = types.ModuleType('torch_scatter')               # un-vendored third-party packages on the path (SURVEY 8c)
    ts.segment_coo = F_.segment_coo

    def scatter_add(src, index, dim=0, out=None, dim_size=None):   # imported by dmpigo.py:11, never called on this path
        raise NotImplementedError
    ts.scatter_add = scatter_add
    sys.modules['torch_scatter'] = ts
    td = types.ModuleType('torch_efficient_distloss')
    td.flatten_eff_distloss = F_.flatten_eff_distloss
    sys.modules['torch_efficient_distloss'] = td
    sys.path.insert(0, PY)
    try:
        from FourierGrid import FourierGrid_model, dcvgo, masked_adam
    finally:
        sys.path.remove(PY)
    return types.SimpleNamespace(fg=FourierGrid_model, dcvgo=dcvgo, adam=masked_adam)


def _default_cuda(on):
    """run_FourierGrid.py:87 `torch.set_default_tensor_type('torch.cuda.FloatTensor')` (deprecated in torch 2.x, still there);
    falls back to torch.set_default_device."""
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        try:
            torch.set_default_tensor_type('torch.cuda.FloatTensor' if on else 'torch.FloatTensor')
        except Exception:
            torch.set_default_device(DEV if on else 'cpu')


def _stat(a, rec):
    """max |a - reference| / max |reference| on the recorded positions (a is all of ours)."""
    a = take(a.detach().float(), sample_index(a.shape, rec['sample'].numel())) if 'sample' in rec else a.detach().float().cpu()
    b = (rec['sample'] if 'sample' in rec else rec['full']).float()
    return (a - b.reshape(a.shape)).abs().max().item() / (rec['scale'] + 1e-30)


CASES = {
    'fouriergrid': dict(cls='FourierGridModel', kw=dict(
        xyz_min=[-1.] * 3, xyz_max=[1.] * 3, num_voxels_density=48 ** 3, num_voxels_base_density=48 ** 3, num_voxels_rgb=48 ** 3,
        num_voxels_base_rgb=48 ** 3, num_voxels_viewdir=-1, alpha_init=1e-4, fast_color_thres=1e-4, rgbnet_dim=12,
        fourier_freq_num=3), mean=5.0, std=4.0, stepsize=0.5),
    'dcvgo': dict(cls='DirectContractedVoxGO', kw=dict(
        xyz_min=[-1.] * 3, xyz_max=[1.] * 3, num_voxels=64 ** 3, num_voxels_base=64 ** 3, alpha_init=1e-4, fast_color_thres=1e-4,
        rgbnet_dim=12, contracted_norm='l2'), mean=5.0, std=4.0, stepsize=0.5),
}


RK = dict(near=0., far=1e9, bg=1, rand_bkgd=False, inverse_y=False, flip_x=False, flip_y=False, render_depth=True)
CFG = dict(lrate_density=1e-1, lrate_k0=1e-1, lrate_rgbnet=1e-3, lrate_decay=20, skip_zero_grad_fields=['density', 'k0'])


def _train_iteration(m, opt, ro, rd, vd, target, stepsize):
    """One training iteration the way run_train.py:251-289 drives it: forward, the always-on losses, backward, TV."""
    n = ro.shape[0]
    out = m(ro, rd, vd, global_step=1, is_train=True, stepsize=stepsize, **RK)
    opt.zero_grad(set_to_none=True)
    loss = torch.nn.functional.mse_loss(out['rgb_marched'], target)
    pout = out['alphainv_last'].clamp(1e-6, 1 - 1e-6)
    loss = loss + 1e-3 * (-(pout * torch.log(pout) + (1 - pout) * torch.log(1 - pout)).mean())
    rgbper = (out['raw_rgb'] - target[out['ray_id']]).pow(2).sum(-1)
    loss = loss + 1e-2 * (rgbper * out['weights'].detach()).sum() / n
    loss.backward()
    m.density_total_variation_add_grad(1e-6 / n, True)
    m.k0_total_variation_add_grad(1e-7 / n, True)


def _trained(named):
    return sorted(k for k in named if k in ('density.grid', 'k0.grid') or k.startswith('rgbnet'))


def _step_grads(named, seed=5):
    """Seeded gradients (half of the grid entries zero, for skip_zero_grad) fed to both optimisers: Adam's m / (sqrt(v) + eps)
    ~ sign(g) at step 1 turns a last-bit gradient difference into a 2 lr parameter difference, so the step is compared on
    identical gradients."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k in _trained(named):
        shape = named[k].shape
        grad = torch.randn(shape, generator=g, device='cpu')
        if k in ('density.grid', 'k0.grid'):
            grad = grad * (torch.rand(shape, generator=g, device='cpu') > 0.5)
        out[k] = grad.to(DEV)
    return out


def _reference_record(ref_modules, flavor, state, ro, rd, vd, target):
    """Run the reference's unmodified classes (over this library) on the state dict; summaries of what the test compares."""
    import numpy as np
    c = CASES[flavor]
    ref_cls = getattr(ref_modules.fg if flavor == 'fouriergrid' else ref_modules.dcvgo, c['cls'])
    kw = dict(c['kw'], xyz_min=np.array(c['kw']['xyz_min'], dtype=np.float32), xyz_max=np.array(c['kw']['xyz_max'], dtype=np.float32))
    # the reference model, built the way run_train.py builds it: default tensor type = CUDA (run_FourierGrid.py:87; the
    # model code relies on it: torch.zeros([N,3]) without a device at FourierGrid_model.py:643, dcvgo.py:348)
    _default_cuda(True)
    try:
        ref = ref_cls(**kw)
        missing, unexpected = ref.load_state_dict(state, strict=False)
        assert not unexpected, unexpected
        ref = ref.to(DEV)
        a = ref(ro, rd, vd, global_step=None, is_train=False, stepsize=c['stepsize'], **RK)
        rec = {'out ' + k: summarize(a[k], SAMPLE) for k in ('ray_id', 'step_id') + OUT_KEYS}
        groups = [{'params': [ref.density.grid] if hasattr(ref.density, 'grid') else list(ref.density.parameters()), 'lr': 0.1, 'skip_zero_grad': True},
                  {'params': [ref.k0.grid], 'lr': 0.1, 'skip_zero_grad': True},
                  {'params': list(ref.rgbnet.parameters()), 'lr': 1e-3, 'skip_zero_grad': False}]
        opt = ref_modules.adam.MaskedAdam(groups)
        _train_iteration(ref, opt, ro, rd, vd, target, c['stepsize'])
        named = dict(ref.named_parameters())
        rec.update({'grad ' + k: summarize(named[k].grad, SAMPLE) for k in _trained(named)})
        for k, g in _step_grads(named).items():
            named[k].grad = g
        opt.step()
        sd = ref.state_dict()
        rec.update({'param ' + k: summarize(sd[k], SAMPLE) for k in _trained(named)})
        return rec
    finally:
        _default_cuda(False)


@pytest.mark.parametrize('flavor', list(CASES))
def test_library_matches_recorded_run_of_unmodified_reference_callers(ref_modules, flavor):
    from unboundednerfpytorch_b200 import grid as G
    from unboundednerfpytorch_b200 import models
    from unboundednerfpytorch_b200.masked_adam import create_optimizer_or_freeze_model
    c = CASES[flavor]
    N = 2048
    g = torch.Generator().manual_seed(11)
    ro = (torch.rand(N, 3, generator=g) - 0.5).to(DEV)
    rd = torch.randn(N, 3, generator=g).to(DEV)
    vd = rd / rd.norm(dim=-1, keepdim=True)
    target = torch.rand(N, 3, generator=g).to(DEV)

    torch.manual_seed(777)
    ours = getattr(models, c['cls'])(**c['kw'])
    with torch.no_grad():
        ours.density.grid.copy_(torch.randn(ours.density.grid.shape, generator=g) * c['std'] + c['mean'])
        ours.k0.grid.copy_(torch.randn(ours.k0.grid.shape, generator=g))
        if flavor == 'dcvgo':
            ours.mask_cache.mask.copy_(torch.rand(ours.mask_cache.mask.shape, generator=g) < 0.9)
    state = {k: v.detach().clone().contiguous() for k, v in ours.state_dict().items()}
    ours = ours.to(DEV)
    key = f'callers_unchanged/{flavor}'
    if RECORD:
        record_golden(key, _reference_record(ref_modules, flavor, state, ro, rd, vd, target))
    rec = ref_golden(key)

    b = ours(ro, rd, vd, global_step=None, is_train=False, stepsize=c['stepsize'], **RK)
    assert_equal_summary(b['ray_id'], rec['out ray_id'], f'{flavor} ray_id (survivor set)')
    assert_equal_summary(b['step_id'], rec['out step_id'], f'{flavor} step_id (survivor set)')
    assert b['ray_id'].numel() > 1000
    for k in OUT_KEYS:
        e = _stat(b[k], rec['out ' + k])
        assert e <= 1e-5, f'{flavor} {k}: {e:.2e} of scale'

    # gradients (incl. the TV term) before the optimiser.  density.grid does not pass through the ReLU MLP: tight.  k0.grid and
    # the rgbnet do: a pre-activation within fp32 rounding of zero flips its ReLU mask between cuBLAS (reference) and the
    # tcgen05 kernels (ours), which changes that sample's contribution (tests/parity_at_size.py quantifies this against fp64)
    opt = create_optimizer_or_freeze_model(ours, CFG, global_step=0)
    _train_iteration(ours, opt, ro, rd, vd, target, c['stepsize'])
    named = dict(ours.named_parameters())
    assert _stat(named['density.grid'].grad, rec['grad density.grid']) <= 2e-5
    r = rec['grad k0.grid']
    gk = take(named['k0.grid'].grad, sample_index(named['k0.grid'].shape, r['sample'].numel()))
    beyond = ((gk - r['sample']).abs() > 1e-5 * r['scale']).float().mean().item()
    assert beyond <= 1e-3, f'{flavor} k0.grid grad: {beyond:.2e} of the elements beyond 1e-5 of scale'
    for k in _trained(named):
        if k.startswith('rgbnet'):
            assert _stat(named[k].grad, rec['grad ' + k]) <= 5e-4, f'{flavor} grad {k}'
    # the optimiser step itself: the reference's unmodified MaskedAdam (over legacy adam_upd_cuda) and this library's
    # MaskedAdam must agree BIT FOR BIT when fed the same gradients
    for k, grad in _step_grads(named).items():
        named[k].grad = G._as_cl3d(grad) if grad.dim() == 5 else grad
    opt.step()
    sd = ours.state_dict()
    for k in _trained(named):
        assert_equal_summary(sd[k], rec['param ' + k], f'{flavor} parameter {k} after MaskedAdam.step')
