"""Shared helpers for the parity tests."""
import importlib.util
import os

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-5          # north-star tolerance for fp32 RGB / depth / weights (BASELINE.json)


def load_golden(name):
    return torch.load(os.path.join(ROOT, 'tests', 'golden', name), map_location='cpu', weights_only=False)


def assert_close(a, b, rtol=RTOL, atol=1e-6, what=''):
    if isinstance(rtol, str):              # allow assert_close(a, b, 'name') like assert_equal
        rtol, what = RTOL, rtol
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    assert a.shape == b.shape, f'{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}'
    if a.numel() == 0:
        return
    err = (a - b).abs()
    tol = atol + rtol * b.abs()
    bad = err > tol
    assert not bad.any(), (f'{what}: {int(bad.sum())}/{a.numel()} elements off; max abs err {err.max().item():.3e}, '
                           f'max rel err {(err / b.abs().clamp_min(1e-12)).max().item():.3e}')


def assert_equal(a, b, what=''):
    a, b = a.detach().cpu(), b.detach().cpu()
    assert a.shape == b.shape, f'{what}: shape {tuple(a.shape)} vs {tuple(b.shape)}'
    assert torch.equal(a, b), f'{what}: {int((a != b).sum())}/{a.numel()} elements differ (bit-exact target)'


_ref_cache = {}


def ref_cuda(name):
    """The reference's OWN CUDA extension module built into oracle/_ref by `make -C oracle ref` (only possible where the
    reference checkout is readable).  Used only while recording REF_GOLDEN; the tests compare against the record."""
    if name in _ref_cache:
        return _ref_cache[name]
    path = os.path.join(ROOT, 'oracle', '_ref', f'{name}.so')
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    _ref_cache[name] = mod
    return mod


def ref_ext():
    """Namespace of the reference's own CUDA functions in the shape oracle.cpu_ref.model_forward(ext=...) expects: with CUDA
    tensors that call IS the reference's GPU path op for op (ATen grid_sample, cuBLAS rgbnet, index_add for torch_scatter,
    the reference's .cu kernels for everything else)."""
    import types
    ru, ub = ref_cuda('render_utils_cuda'), ref_cuda('ub360_utils_cuda')
    return types.SimpleNamespace(raw2alpha=ru.raw2alpha, raw2alpha_backward=ru.raw2alpha_backward, alpha2weight=ru.alpha2weight,
                                 alpha2weight_backward=ru.alpha2weight_backward, maskcache_lookup=ru.maskcache_lookup,
                                 cumdist_thres=ub.cumdist_thres)


# What the reference's own GPU code returned for the tests' seeded inputs, so that the comparisons run without the reference:
# tests/golden/ref_gpu.pkl.xz maps a key to a list of summaries (summarize()), tensors stored as numpy arrays, lzma-compressed.  Setting UBN_RECORD_REF_GOLDEN=<file> on a GPU box
# where oracle/_ref is built makes the tests run the reference instead, check against it directly and write the records there.
REF_GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'ref_gpu.pkl.xz')
RECORD = os.environ.get('UBN_RECORD_REF_GOLDEN')
N_SAMPLE = 32          # bit-exact records: the digest decides, the sample makes a failure readable
_golden = {}


def sample_index(shape, k, seed=0):
    """k fixed pseudo-random flat positions of a tensor of this shape (the same on every machine); all of them when k >= size."""
    n = 1
    for s in shape:
        n *= int(s)
    if k >= n:
        return torch.arange(n)
    g = torch.Generator().manual_seed(n * 1000003 + seed)
    return torch.randint(0, max(n, 1), (min(k, n),), generator=g, device='cpu')


def take(t, idx):
    """t at flat positions idx, without copying t when it is not contiguous."""
    return t.detach()[torch.unravel_index(idx.to(t.device), t.shape)].cpu() if t.numel() else t.detach().reshape(-1).cpu()


def digest(t):
    import hashlib
    return hashlib.sha256(t.detach().contiguous().cpu().numpy().tobytes()).hexdigest()


def summarize(t, k=N_SAMPLE):
    """shape, dtype, SHA-256 of the bytes, max |t| and t at sample_index (all of t when it is that small)."""
    t = t.detach()
    rec = dict(shape=tuple(t.shape), dtype=str(t.dtype), sha256=digest(t))
    if t.is_floating_point() and t.numel():
        rec['scale'] = t.abs().max().item()
    if t.numel() <= k:
        rec['full'] = t.cpu().clone()
    else:
        rec['sample'] = take(t, sample_index(t.shape, k)).clone()
    return rec


def _convert(o, fn):
    if isinstance(o, dict):
        return {k: _convert(v, fn) for k, v in o.items()}
    if isinstance(o, (list, tuple)):
        return type(o)(_convert(v, fn) for v in o)
    return fn(o)


def _load(path):
    import lzma
    import pickle
    import numpy as np
    with lzma.open(path, 'rb') as f:
        return _convert(pickle.load(f), lambda v: torch.from_numpy(v) if isinstance(v, np.ndarray) else v)


def ref_golden(key):
    """The recorded summaries under key (replay), loaded once."""
    if not _golden:
        _golden.update(_load(REF_GOLDEN))
    assert key in _golden, f'{key} is not recorded in {REF_GOLDEN}'
    return _golden[key]


def record_golden(key, recs):
    import lzma
    import pickle
    if not _golden and os.path.exists(RECORD):
        _golden.update(_load(RECORD))
    _golden[key] = recs
    with lzma.open(RECORD, 'wb', preset=9) as f:
        pickle.dump(_convert(_golden, lambda v: v.detach().cpu().numpy() if torch.is_tensor(v) else v), f, protocol=4)


def assert_equal_summary(a, rec, what=''):
    """Bit-exact comparison of a with a recorded summary: shape, dtype, the sample (for a readable failure), then the digest."""
    assert tuple(a.shape) == tuple(rec['shape']), f'{what}: shape {tuple(a.shape)} vs {rec["shape"]}'
    assert str(a.dtype) == rec['dtype'], f'{what}: dtype {a.dtype} vs {rec["dtype"]}'
    if 'full' in rec:
        assert_equal(a, rec['full'], what)
        return
    assert_equal(take(a, sample_index(a.shape, rec['sample'].numel())), rec['sample'], what + ' (sample)')
    assert digest(a) == rec['sha256'], f'{what}: equal on the sample, but the SHA-256 of the whole tensor differs'


def assert_equal_ref(key, ours, compute):
    """ours (a tensor or a sequence) must equal, bit for bit, what the reference's own CUDA extension returns for the same
    inputs: compute(ref_cuda) while recording, the record under key otherwise."""
    ours = [ours] if torch.is_tensor(ours) else list(ours)
    if RECORD:
        theirs = compute(ref_cuda)
        theirs = [theirs] if torch.is_tensor(theirs) else list(theirs)
        assert len(theirs) == len(ours)
        for i, (a, b) in enumerate(zip(ours, theirs)):
            assert_equal(a, b, f'{key}[{i}] vs ref-cuda')
        record_golden(key, [summarize(b) for b in theirs])
        return
    recs = ref_golden(key)
    assert len(recs) == len(ours)
    for i, (a, rec) in enumerate(zip(ours, recs)):
        assert_equal_summary(a, rec, f'{key}[{i}] vs ref-cuda')


def seeded_rays(n, seed, device='cpu', spread=0.5):
    g = torch.Generator().manual_seed(seed)
    ro = (torch.rand(n, 3, generator=g) - 0.5) * 2 * spread
    rd = torch.randn(n, 3, generator=g)
    vd = rd / rd.norm(dim=-1, keepdim=True)
    return ro.to(device), rd.to(device), vd.to(device)


def cfg1_scene(seed=777 + 64):
    """BASELINE config 1 (SURVEY.md 8d): DVGO 64^3 DenseGrid, 1024 rays, stepsize 0.5.  Seeded, so the 13 MB of grids are
    regenerated by the test instead of being stored: returns (kwargs, density grid, k0 grid, rgbnet state, rays_o, rays_d, viewdirs)."""
    gen = torch.Generator().manual_seed(seed)
    kw = dict(xyz_min=[-1., -1., -1.], xyz_max=[1., 1., 1.], num_voxels=64 ** 3, num_voxels_base=64 ** 3, alpha_init=1e-2,
              fast_color_thres=1e-4, rgbnet_dim=12, rgbnet_direct=True, mask_cache_world_size=[64, 64, 64])
    dens = torch.randn(1, 1, 64, 64, 64, generator=gen) * 3
    k0 = torch.randn(1, 12, 64, 64, 64, generator=gen)
    net = {f'rgbnet.{k}': v for k, v in
           zip(('0.weight', '0.bias', '2.0.weight', '2.0.bias', '3.weight', '3.bias'),
               (torch.randn(128, 39, generator=gen) * 0.16, torch.randn(128, generator=gen) * 0.1,
                torch.randn(128, 128, generator=gen) * 0.09, torch.randn(128, generator=gen) * 0.1,
                torch.randn(3, 128, generator=gen) * 0.09, torch.zeros(3)))}
    N = 1024
    ro = torch.randn(N, 3, generator=gen) * 0.2 + torch.tensor([0., 0., -2.5])
    rd = torch.randn(N, 3, generator=gen) * 0.25 + torch.tensor([0., 0., 1.])
    vd = rd / rd.norm(dim=-1, keepdim=True)
    return kw, dens, k0, net, ro, rd, vd
