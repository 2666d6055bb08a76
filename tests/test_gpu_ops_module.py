"""GPU: k4nerf.render_utils_cuda (the 13-function op-level drop-in, csrc/k4_ops.cu) against the
REFERENCE'S OWN compiled extension (replayed from its stored results, tests/ref_calls.py): every output
bit-identical."""
import pytest
import torch

from oracle import scenes
from ref_calls import RefCalls

pytestmark = pytest.mark.gpu


@pytest.fixture
def mods(request, cuda_device):
    from k4nerf import render_utils_cuda as ours
    rc = RefCalls.for_test(request)
    yield ours, rc.module('render_utils_cuda')
    rc.finish()


def _rays(n, dev, seed=0):
    g = torch.Generator().manual_seed(seed)
    ro = torch.randn(n, 3, generator=g) * 0.3 + torch.tensor([0., 0., 3.5])
    rd = torch.randn(n, 3, generator=g) * 0.25 + torch.tensor([0., 0., -1.])
    rd[::17, 0] = 0.0
    rd[::29, 1] = 0.0
    return ro.to(dev).contiguous(), rd.to(dev).contiguous()


def _eq(a, b, name):
    assert a.dtype == b.dtype and a.shape == b.shape, (name, a.dtype, b.dtype, a.shape, b.shape)
    assert torch.equal(a, b), f'{name}: {(a != b).sum().item()} of {a.numel()} elements differ'


def test_sampling_ops_bit_exact(mods, cuda_device):
    ours, ref = mods
    dev = cuda_device
    ro, rd = _rays(5003, dev)
    mn, mx = torch.tensor([-1., -1., -1.], device=dev), torch.tensor([1., 1., 1.], device=dev)
    stepdist = 0.5 * 2.0 / 160
    for name, a, b in zip(('t_min', 't_max'), ours.infer_t_minmax(ro, rd, mn, mx, 0.2, 1e9), ref.infer_t_minmax(ro, rd, mn, mx, 0.2, 1e9)):
        _eq(a, b, name)
    t_min, t_max = ref.infer_t_minmax(ro, rd, mn, mx, 0.2, 1e9)
    _eq(ours.infer_n_samples(rd, t_min, t_max, stepdist), ref.infer_n_samples(rd, t_min, t_max, stepdist), 'n_samples')
    for name, a, b in zip(('start', 'dir'), ours.infer_ray_start_dir(ro, rd, t_min), ref.infer_ray_start_dir(ro, rd, t_min)):
        _eq(a, b, name)
    names = ['ray_pts', 'mask_outbbox', 'ray_id', 'step_id', 'N_steps', 't_min', 't_max']
    for name, a, b in zip(names, ours.sample_pts_on_rays(ro, rd, mn, mx, 0.2, 1e9, stepdist), ref.sample_pts_on_rays(ro, rd, mn, mx, 0.2, 1e9, stepdist)):
        _eq(a, b, name)
    o, d, _ = scenes.llff_rays(24, 32)
    o, d = o.to(dev), d.to(dev)
    mn2, mx2 = torch.tensor([-1.5, -1.67, -1.], device=dev), torch.tensor([1.5, 1.67, 1.], device=dev)
    for name, a, b in zip(('ndc_pts', 'ndc_mask'), ours.sample_ndc_pts_on_rays(o, d, mn2, mx2, 64), ref.sample_ndc_pts_on_rays(o, d, mn2, mx2, 64)):
        _eq(a, b, name)
    tm = (torch.rand(ro.shape[0], generator=torch.Generator().manual_seed(1)) * 2 + 1).to(dev).contiguous()
    _eq(ours.sample_bg_pts_on_rays(ro, rd, tm, 0.5, 32), ref.sample_bg_pts_on_rays(ro, rd, tm, 0.5, 32), 'bg_pts')


def test_maskcache_and_activation_ops_bit_exact(mods, cuda_device):
    ours, ref = mods
    dev = cuda_device
    g = torch.Generator().manual_seed(3)
    world = (torch.rand(40, 37, 45, generator=g) > 0.5).to(dev)
    xyz = (torch.rand(200000, 3, generator=g) * 2.4 - 1.2).to(dev).contiguous()
    scale = ((torch.tensor([40., 37., 45.]) - 1) / 2).to(dev)
    shift = (scale * 1.0).contiguous()
    _eq(ours.maskcache_lookup(world, xyz, scale, shift), ref.maskcache_lookup(world, xyz, scale, shift), 'maskcache')
    dens = (torch.randn(100001, generator=g) * 4).to(dev).contiguous()
    for name, a, b in zip(('exp', 'alpha'), ours.raw2alpha(dens, -4.595, 0.5), ref.raw2alpha(dens, -4.595, 0.5)):
        _eq(a, b, name)
    iv = (torch.rand(100001, generator=g) + 0.1).to(dev).contiguous()
    for name, a, b in zip(('exp_nu', 'alpha_nu'), ours.raw2alpha_nonuni(dens, -4.595, iv), ref.raw2alpha_nonuni(dens, -4.595, iv)):
        _eq(a, b, name)
    e, _ = ref.raw2alpha(dens, -4.595, 0.5)
    gb = torch.randn(100001, generator=g).to(dev).contiguous()
    _eq(ours.raw2alpha_backward(e, gb, 0.5), ref.raw2alpha_backward(e, gb, 0.5), 'raw2alpha_backward')
    _eq(ours.raw2alpha_nonuni_backward(e, gb, iv), ref.raw2alpha_nonuni_backward(e, gb, iv), 'raw2alpha_nonuni_backward')


def test_alpha2weight_forward_backward_bit_exact(mods, cuda_device):
    ours, ref = mods
    dev = cuda_device
    g = torch.Generator().manual_seed(4)
    n_rays, n_pts = 777, 100000
    ray_id = torch.sort(torch.randint(0, n_rays, (n_pts,), generator=g))[0].to(dev)
    alpha = (torch.rand(n_pts, generator=g) ** 3).to(dev).contiguous()
    a = ours.alpha2weight(alpha, ray_id, n_rays)
    b = ref.alpha2weight(alpha, ray_id, n_rays)
    for name, x, y in zip(('weights', 'T', 'alphainv_last', 'i_start', 'i_end'), a, b):
        _eq(x, y, name)
    gw = torch.randn(n_pts, generator=g).to(dev).contiguous()
    gl = torch.randn(n_rays, generator=g).to(dev).contiguous()
    _eq(ours.alpha2weight_backward(alpha, *b, n_rays, gw, gl), ref.alpha2weight_backward(alpha, *b, n_rays, gw, gl), 'alpha2weight_backward')
    # empty inputs (render_utils_kernel.cu:406,465,629)
    e = torch.zeros(0, device=dev)
    assert ours.raw2alpha(e, 0.0, 0.5)[1].numel() == 0
    w0 = ours.alpha2weight(e, torch.zeros(0, dtype=torch.int64, device=dev), 5)
    assert torch.equal(w0[2], torch.ones(5, device=dev))


def test_contract_errors(mods, cuda_device):
    ours, _ = mods
    with pytest.raises(RuntimeError, match='CUDA'):
        ours.raw2alpha(torch.zeros(4), 0.0, 0.5)
    x = torch.zeros(8, 2, device=cuda_device)[:, 0]
    with pytest.raises(RuntimeError, match='contiguous'):
        ours.raw2alpha(x, 0.0, 0.5)
