"""GPU: pin the oracle against the REFERENCE'S OWN KERNELS.

The reference extension (lib/cuda/render_utils*.{cpp,cu}) is replayed from the digests of what it
returned (tests/ref_calls.py).  Here every forward op of the C restatement (oracle/render_utils_ref.c)
is compared with it on seeded inputs, and the whole reference pipeline run on the reference kernels
(oracle/pipeline.py + the reference ops) is compared with the fused kernel.
"""
import pytest
import torch

from oracle import ops, pipeline, scenes
from helpers import compare, make_state, model_from_state, rays_for
from ref_calls import RefCalls

pytestmark = pytest.mark.gpu


@pytest.fixture
def ref_ops(request, cuda_device):
    rc = RefCalls.for_test(request)
    yield rc.ops()
    rc.finish()


def _rays(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    ro = torch.randn(n, 3, generator=g) * 0.3 + torch.tensor([0., 0., 3.5])
    rd = torch.randn(n, 3, generator=g) * 0.25 + torch.tensor([0., 0., -1.])
    rd[::17, 0] = 0.0          # exercise the d == 0 -> 1e-6 substitution
    rd[::29, 1] = 0.0
    return ro.contiguous(), rd.contiguous()


def test_sample_pts_on_rays_bit_exact(ref_ops, cuda_device):
    dev = cuda_device
    ro, rd = _rays(4099)
    mn, mx = torch.tensor([-1., -1., -1.]), torch.tensor([1., 1., 1.])
    stepdist = 0.5 * 2.0 / 160
    c = ops.CpuOps.sample_pts_on_rays(ro, rd, mn, mx, 0.2, 1e9, stepdist)
    g = ref_ops.sample_pts_on_rays(ro.to(dev), rd.to(dev), mn.to(dev), mx.to(dev), 0.2, 1e9, stepdist)
    names = ['ray_pts', 'mask_outbbox', 'ray_id', 'step_id', 'N_steps', 't_min', 't_max']
    for name, a, b in zip(names, c, g):
        assert torch.equal(a, b.cpu()), f'{name} differs from the reference kernel'


def test_sample_ndc_pts_bit_exact(ref_ops, cuda_device):
    dev = cuda_device
    ro, rd, _ = scenes.llff_rays(24, 32)
    mn, mx = torch.tensor([-1.5, -1.67, -1.]), torch.tensor([1.5, 1.67, 1.])
    c = ops.CpuOps.sample_ndc_pts_on_rays(ro, rd, mn, mx, 64)
    g = ref_ops.sample_ndc_pts_on_rays(ro.to(dev), rd.to(dev), mn.to(dev), mx.to(dev), 64)
    assert torch.equal(c[0], g[0].cpu()) and torch.equal(c[1], g[1].cpu())


def test_maskcache_lookup_bit_exact(ref_ops, cuda_device):
    dev = cuda_device
    g = torch.Generator().manual_seed(3)
    world = torch.rand(40, 37, 45, generator=g) > 0.5
    xyz = (torch.rand(200000, 3, generator=g) * 2.4 - 1.2).contiguous()
    mg = pipeline.mask_grid_state(world, [-1, -1, -1], [1, 1, 1])
    c = ops.CpuOps.maskcache_lookup(world, xyz, mg['xyz2ijk_scale'], mg['xyz2ijk_shift'])
    r = ref_ops.maskcache_lookup(world.to(dev), xyz.to(dev), mg['xyz2ijk_scale'].to(dev), mg['xyz2ijk_shift'].to(dev))
    assert torch.equal(c, r.cpu())


def test_raw2alpha_and_alpha2weight(ref_ops, cuda_device):
    dev = cuda_device
    g = torch.Generator().manual_seed(4)
    dens = (torch.randn(100000, generator=g) * 4).contiguous()
    ce, ca = ops.CpuOps.raw2alpha(dens, -4.595, 0.5)
    ge, ga = ref_ops.raw2alpha(dens.to(dev), -4.595, 0.5)
    # expf/powf: CUDA math library vs glibc, <= 2 ulp each
    assert (ca - ga.cpu()).abs().max().item() <= 3e-7
    assert ((ce - ge.cpu()).abs() / ce.abs().clamp_min(1e-30)).max().item() <= 5e-7
    # alpha2weight is exact arithmetic (float*float, double product): feed both the SAME alphas
    n_rays = 777
    ray_id = torch.sort(torch.randint(0, n_rays, (100000,), generator=g))[0]
    alpha = ga.cpu().clamp(0, 1).contiguous()
    cw = ops.CpuOps.alpha2weight(alpha, ray_id, n_rays)
    gw = ref_ops.alpha2weight(alpha.to(dev), ray_id.to(dev), n_rays)
    for name, a, b in zip(['weights', 'T', 'alphainv_last', 'i_start', 'i_end'], cw, gw):
        assert torch.equal(a, b.cpu()), name


@pytest.mark.parametrize('name,regime', [('cfgA', 'fog'), ('cfgA', 'shell'), ('cfgB', 'fog'), ('cfgB', 'shell')])
def test_fused_kernel_vs_reference_kernels_pipeline(ref_ops, cuda_device, name, regime):
    """The reference's forward structure running on the reference's own CUDA kernels + ATen CUDA
    grid_sample / Linear (the closest thing to `run_sr.py` on this box) vs the fused kernel."""
    dev = cuda_device
    st = make_state(name, regime=regime) if name == 'cfgA' else make_state(name, xy=48, depth=32, regime=regime)
    (ro, rd, vd), kw = rays_for(st, 48, 64)
    torch.backends.cuda.matmul.allow_tf32 = False
    st_dev = pipeline.state_to(st, dev)
    stats = {}
    ref = pipeline.forward(st_dev, ro.to(dev), rd.to(dev), vd.to(dev), ref_ops, stats=stats, **kw)
    m = model_from_state(st, dev)
    for mode, bar in (('fp32', 80.0), ('f16x3', 70.0)):
        ours = m.render_rays(ro.to(dev), rd.to(dev), vd.to(dev), kw, mlp_mode=mode, debug=True)
        c = ours['counters'].cpu().tolist()
        rs = ours['ray_stats'].cpu().long()
        ors = ref['_ray_stats'].cpu()
        # same device math library on both sides: the early-out and the survivors must agree except
        # for FMA-order differences inside ATen's trilinear kernel (<= 1e-4 of the rays)
        bad = (rs[:, 1] != ors[:, 0]) | (rs[:, 2] != ors[:, 1])
        assert int(bad.sum()) <= max(1, int(1e-4 * ro.shape[0])), (int(bad.sum()), c, stats)
        assert abs(c[2] - stats['S_c']) <= max(2, 1e-4 * stats['S_c']), (c, stats)
        cmp = compare(ours, ref, ro.shape[0])
        assert cmp['rgb_marched_psnr'] >= bar, (mode, cmp)
        assert cmp['alphainv_last_maxabs'] <= 1e-5, (mode, cmp)
