"""Parity of the BENCHMARKED configurations at the benchmarked size (8192 rays x 512 samples) against the reference's own GPU
path: oracle.cpu_ref.model_forward on CUDA tensors with the reference's CUDA extension (machinery and the tolerance definition:
tests/parity_at_size.py), as recorded in tests/golden/ref_gpu.pkl.xz.  The record holds the sample set by digest; every output and
gradient by its whole-tensor scale and 256 fixed positions (k0.grid: 16384); the fp64 gradients at up to 4096 of those
positions; the reference's deviation from fp64 on those positions and on the whole tensor; and its run-to-run statistics on
the whole tensors.  Every statistic of this library is therefore taken on the stored positions (see 'Bars on the stored
positions' below).  Replaces the 40^3 / 96-ray CPU-oracle comparison with loose absolute
tolerances as the evidence for the headline workload.

  truck_dense      FourierGridModel 153^3, F = 4 (9 slabs), thres 0 -- the line bench.py reports
  truck_realistic  same grids ~ N(6, 4), fast_color_thres 1e-4: both threshold compactions, early ray termination
  bicycle_dense    DirectContractedVoxGO 320^3, l2 contraction, cumdist filter + 90 % mask cache

Bar (BASELINE.json north_star): ray_id / step_id bit-exact (zero membership flips); fp32 outputs within 1e-5 of the reference
relative to the tensor scale.  Three places where "1e-5 of the reference, element by element" is not a meaningful bar, and what is
asserted instead (each measured, see tests/parity_at_size.py and DESIGN.md section 2):

* alpha = 1 - (1 + e)^-interval (render_utils_kernel.cu:439-441) is quantised at ulp(1) = 6e-8 whatever its size; in dense mode
  (alpha ~ 5e-5) one ulp of 1 is 1e-3 of alpha.  weights / raw_alpha: 1e-5 of scale OR one ulp of 1.0 absolute.
* the grid scatters are fp32 atomics in the reference too (ATen grid_sampler_3d_backward): the reference differs from ITSELF from
  run to run.  density.grid grad: within max(1e-5 of scale, 3 x the reference's own run-to-run difference).
* gradients through the ReLU MLP (k0.grid, rgbnet.*): a pre-activation within rounding distance of zero flips its ReLU mask
  between ANY two fp32 implementations (cuBLAS vs tcgen05 vs exact), changing that sample's whole contribution.  Judged against
  an fp64 evaluation of the reference's algorithm: this library deviates from it no more than the reference's fp32 GPU path
  does (max error within 3x, count of elements beyond 1e-5 of scale within 3x), and beyond-tolerance elements vs the reference
  stay below 1e-3 of the tensor.

Bars on the stored positions: maxima are compared position for position against whole-tensor scales, with the reference's
maximum taken on the same positions.  The share of k0.grid gradient elements beyond 1e-5 (<= 1e-3, tensors above 16384 elements)
is measured on 16384 positions, where 1e-3 is 16 elements (measured on the whole tensor: 1.2e-5 .. 1.3e-4, i.e. ~0.2 .. 2).  The
count of elements beyond 1e-5 of scale against fp64 (whole tensor: <= max(16, 3 x the reference's count)) is judged by
parity_at_size.count_bar: that bar scaled to the stored positions from the reference's whole-tensor count, plus the sampling
spread of such a count."""
import pytest
import torch

from tests import parity_at_size as P
from tests.util import RECORD, record_golden, ref_ext, ref_golden

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ULP1 = 2.0 ** -23            # fp32 spacing at 1.0 (alpha = 1 - x is quantised at half of it)


@pytest.mark.parametrize('name', list(P.CONFIGS))
def test_benchmarked_config_vs_reference_gpu_path(name):
    if RECORD:
        record_golden(f'parity_at_size/{name}', P.record(name, torch.device(DEV), ref_ext()))
        torch.cuda.empty_cache()
    out, _ = P.compare_recorded(name, torch.device(DEV), ref_golden(f'parity_at_size/{name}'))
    print(f'[parity-at-size] {out}')
    assert out['n_max'] == 512
    assert out['M'] == out['M_ref'] and out['flips'] == 0, f"sample set differs from the reference's (M {out['M']} vs {out['M_ref']})"
    assert out['ray_id_equal'] and out['step_id_equal']
    if name == 'truck_dense':
        assert out['M'] == 8192 * 512
    for k in ('rgb_marched', 'alphainv_last', 'depth', 'raw_density', 'raw_rgb', 't', 's', 'wsum_mid'):
        if k in out:
            assert out[k]['rel_scale'] <= P.RTOL, f'{name} {k}: {out[k]}'
    for k in ('weights', 'raw_alpha'):
        assert out[k]['rel_scale'] <= P.RTOL or out[k]['max_abs'] <= ULP1, f'{name} {k}: {out[k]}'
    # density-grid gradient: close to the reference's (within its own run-to-run variation), or -- the scatter merges samples of a
    # cell in registers before they reach the L2 reductions, which changes the fp32 summation order more than two runs of the
    # reference differ -- at least as close to the fp64 scatter of the reference's own per-sample gradients as the reference is
    g, tr = out['grad density.grid'], out['truth density.grid']
    near_ref = g['rel_scale'] <= max(P.RTOL, 3 * out['refself density.grid']['rel_scale'])
    near_truth = tr['ours_max'] <= max(P.RTOL, 3 * tr['ref_max']) and tr['ours_n_bad'] <= P.count_bar(tr)
    assert near_ref or near_truth, f"{name} density.grid grad: vs ref {g} (ref vs itself {out['refself density.grid']}), vs fp64 {tr}"
    for k, st in out.items():
        if not k.startswith('truth ') or k == 'truth density.grid':
            continue
        assert st['ours_max'] <= max(P.RTOL, 3 * st['ref_max']), f'{name} {k}: {st}'
        assert st['ours_n_bad'] <= P.count_bar(st), f'{name} {k}: {st} (bar {P.count_bar(st):.2f})'
        vs_ref = out['grad ' + k[len('truth '):]]
        assert vs_ref['frac_gt'] <= 1e-3 or vs_ref['n'] <= 16384, f'{name} grad {k}: {vs_ref}'
