"""GPU parity of the contracted-space front-end (DirectContractedVoxGO, SURVEY.md section 8(f-3)):
fused kernel vs the CPU oracle (oracle/pipeline.dcvgo_forward) and vs the same forward structure
running on the reference's own CUDA kernels (render_utils_cuda + ub360_utils_cuda, replayed from their
stored results: tests/ref_calls.py)."""
import os

import pytest
import torch

from helpers import make_state, model_from_state, rays_for, compare
from oracle import ops, pipeline
from ref_calls import RefCalls

pytestmark = pytest.mark.gpu


@pytest.fixture
def ref_ops(request, cuda_device):
    rc = RefCalls.for_test(request)
    yield rc.ops()
    rc.finish()


def test_cumdist_thres_oracle_vs_reference_kernel(ref_ops, cuda_device):
    g = torch.Generator().manual_seed(5)
    dist = torch.rand(257, 83, generator=g) * 0.02
    for thres in (0.0, 0.0123, 0.05, 10.0):
        a = ops.CpuOps.cumdist_thres(dist, thres)
        b = ref_ops.cumdist_thres(dist.to(cuda_device), thres)
        assert torch.equal(a, b.cpu()), thres


def _check(ours, ref, stats, n, mode, bar):
    c = ours['counters'].cpu().tolist()
    rs = ours['ray_stats'].cpu().long()
    ors = ref['_ray_stats'].cpu()
    bad = (rs[:, 1] != ors[:, 0]) | (rs[:, 2] != ors[:, 1])
    assert int(bad.sum()) <= max(1, int(1e-4 * n)), (mode, int(bad.sum()), c, stats)
    assert abs(c[2] - stats['S_c']) <= max(2, 1e-4 * stats['S_c']), (mode, c, stats)
    cmp = compare(ours, ref, n)
    assert cmp['rgb_marched_psnr'] >= bar, (mode, cmp)
    assert cmp['depth_psnr'] >= bar, (mode, cmp)
    assert cmp['alphainv_last_maxabs'] <= 1e-5, (mode, cmp)
    return cmp


@pytest.mark.parametrize('regime', ['fog', 'shell'])
@pytest.mark.parametrize('radius', [4.0, 0.6])           # camera outside / inside the inner unit cube
def test_dcvgo_fused_vs_cpu_oracle(cuda_device, regime, radius):
    dev = cuda_device
    st = make_state('cfgC', res=48, regime=regime)
    (ro, rd, vd), kw = rays_for(st, 48, 64, radius=radius)
    stats = {}
    ref = pipeline.forward(st, ro, rd, vd, ops.CpuOps, stats=stats, **kw)
    assert stats['S_m'] > 0
    m = model_from_state(st, dev)
    for mode, bar in (('fp32', 80.0), ('f16x3', 70.0), ('f16', 70.0), ('ws', 70.0), ('auto', 70.0)):
        ours = m.render_rays(ro.to(dev), rd.to(dev), vd.to(dev), kw, image_hw=(48, 64), mlp_mode=mode, debug=True)
        _check(ours, ref, stats, ro.shape[0], mode, bar)
    with torch.no_grad():
        out = m(ro.to(dev), rd.to(dev), vd.to(dev), **kw)
    assert out['rgb_feature'] is out['rgb_marched'] and out['depth'].shape == (ro.shape[0],)


@pytest.mark.parametrize('regime', ['fog', 'shell'])
def test_dcvgo_fused_vs_reference_kernels_pipeline(ref_ops, cuda_device, regime):
    dev = cuda_device
    st = make_state('cfgC', res=48, regime=regime)
    (ro, rd, vd), kw = rays_for(st, 48, 64, radius=0.6)
    torch.backends.cuda.matmul.allow_tf32 = False
    stats = {}
    ref = pipeline.forward(pipeline.state_to(st, dev), ro.to(dev), rd.to(dev), vd.to(dev), ref_ops, stats=stats, **kw)
    m = model_from_state(st, dev)
    for mode, bar in (('fp32', 80.0), ('f16x3', 70.0)):
        ours = m.render_rays(ro.to(dev), rd.to(dev), vd.to(dev), kw, mlp_mode=mode, debug=True)
        _check(ours, ref, stats, ro.shape[0], mode, bar)


def test_dcvgo_no_rgbnet_and_ragged(cuda_device):
    """k0 as direct colour (rgbnet_dim=0) and a ray count that is not a multiple of the tile."""
    dev = cuda_device
    st = make_state('cfgC', res=32, regime='fog', k0_dim=0)
    (ro, rd, vd), kw = rays_for(st, 19, 23, radius=0.6)
    stats = {}
    ref = pipeline.forward(st, ro, rd, vd, ops.CpuOps, stats=stats, **kw)
    m = model_from_state(st, dev)
    ours = m.render_rays(ro.to(dev), rd.to(dev), vd.to(dev), kw, mlp_mode='fp32', debug=True)
    _check(ours, ref, stats, ro.shape[0], 'fp32', 80.0)


@pytest.mark.parametrize('regime', ['fog', 'shell'])
def test_dcvgo_fused_vs_committed_golden(cuda_device, regime):
    """tests/golden/marcher_cfgC_*.pt (oracle outputs, tests/golden/make_golden.py) -- no oracle run needed."""
    gold = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', f'marcher_cfgC_{regime}.pt'),
                      map_location='cpu', weights_only=False)
    st = make_state('cfgC', res=24, regime=regime)
    (ro, rd, vd), kw = rays_for(st, 12, 16, radius=0.6)
    m = model_from_state(st, cuda_device)
    ours = m.render_rays(ro.to(cuda_device), rd.to(cuda_device), vd.to(cuda_device), kw, mlp_mode='fp32', debug=True)
    c = ours['counters'].cpu().tolist()
    assert abs(c[0] - gold['stats']['S_m']) <= 2 and abs(c[2] - gold['stats']['S_c']) <= 2, (c, gold['stats'])
    cmp = compare(ours, gold, ro.shape[0])
    assert cmp['rgb_marched_psnr'] >= 80.0 and cmp['depth_psnr'] >= 80.0 and cmp['alphainv_last_maxabs'] <= 1e-5, cmp
