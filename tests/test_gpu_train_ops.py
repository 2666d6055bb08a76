"""GPU: grid-maintenance and optimiser kernels (SURVEY.md section 8 f-4, csrc/k4_train.cu).

total_variation_add_grad and the three Adam updates are compared BIT FOR BIT with the reference's own
extensions (total_variation_cuda, adam_upd_cuda; replayed from their stored results, tests/ref_calls.py);
update_occupancy_cache / scale_volume_grid are compared with the reference's torch composition
(F.grid_sample + Raw2Alpha formula + F.max_pool3d, F.interpolate) run on the same GPU."""
import pytest
import torch
import torch.nn.functional as F

import k4nerf
from k4nerf import adam_upd_cuda, total_variation_cuda
from helpers import make_state, model_from_state
from oracle import ops
from ref_calls import RefCalls

pytestmark = pytest.mark.gpu


@pytest.fixture
def ref_calls(request, cuda_device):
    rc = RefCalls.for_test(request)
    yield rc
    rc.finish()


@pytest.mark.parametrize('shape', [(1, 1, 17, 9, 33), (1, 12, 20, 24, 16), (1, 3, 1, 5, 2)])
@pytest.mark.parametrize('dense', [True, False])
def test_total_variation_add_grad_bit_exact(cuda_device, ref_calls, shape, dense):
    ref = ref_calls.module('total_variation_cuda')
    g = torch.Generator().manual_seed(3)
    param = (torch.randn(shape, generator=g) * 1.5).to(cuda_device)
    grad = torch.randn(shape, generator=g)
    grad[torch.rand(shape, generator=g) < 0.6] = 0            # sparse gradients: the non-dense mode skips zeros
    grad = grad.to(cuda_device)
    ga, gb = grad.clone(), grad.clone()
    total_variation_cuda.total_variation_add_grad(param, ga, 0.37, 1.1, 2.3e-3, dense)
    ref.total_variation_add_grad(param, gb, 0.37, 1.1, 2.3e-3, dense)
    torch.cuda.synchronize()
    assert torch.equal(ga, gb)
    assert not torch.equal(ga, grad)
    if not dense:
        assert torch.equal(ga[grad == 0], grad[grad == 0])


@pytest.mark.parametrize('n', [4096 * 3, 1001])               # float4 path and the scalar tail path
@pytest.mark.parametrize('variant', ['plain', 'masked', 'perlr'])
def test_adam_updates_bit_exact(cuda_device, ref_calls, n, variant):
    ref = ref_calls.module('adam_upd_cuda')
    g = torch.Generator().manual_seed(7)
    mk = lambda s=1.0: (torch.randn(n, generator=g) * s).to(cuda_device)
    p0, m0, v0 = mk(), mk(0.1), (mk(0.1) ** 2)
    perlr = torch.rand(n, generator=g).to(cuda_device)
    ours, theirs = [p0.clone(), m0.clone(), v0.clone()], [p0.clone(), m0.clone(), v0.clone()]
    for step in (1, 2, 7, 1000):
        grad = torch.randn(n, generator=g)
        grad[torch.rand(n, generator=g) < 0.7] = 0
        grad = grad.to(cuda_device)
        for mod, (p, m, v) in ((adam_upd_cuda, ours), (ref, theirs)):
            if variant == 'plain':
                mod.adam_upd(p, grad, m, v, step, 0.9, 0.99, 0.1, 1e-8)
            elif variant == 'masked':
                mod.masked_adam_upd(p, grad, m, v, step, 0.9, 0.99, 0.1, 1e-8)
            else:
                mod.adam_upd_with_perlr(p, grad, m, v, perlr, step, 0.9, 0.99, 0.1, 1e-8)
        torch.cuda.synchronize()
        for a, b, name in zip(ours, theirs, ('param', 'exp_avg', 'exp_avg_sq')):
            assert torch.equal(a, b), (variant, step, name, (a - b).abs().max().item())
    assert not torch.equal(ours[0], p0)


def test_masked_adam_optimizer_matches_manual_updates(cuda_device):
    """MaskedAdam.step dispatch (lib/masked_adam.py:41-73): per-voxel lr wins for the matching shape,
    skip_zero_grad selects the masked kernel, state keys as the reference."""
    g = torch.Generator().manual_seed(1)
    a = torch.nn.Parameter(torch.randn(1, 1, 6, 5, 4, generator=g).to(cuda_device))
    b = torch.nn.Parameter(torch.randn(33, generator=g).to(cuda_device))
    opt = k4nerf.MaskedAdam([{'params': [a], 'lr': 0.1, 'skip_zero_grad': True}, {'params': [b], 'lr': 0.01, 'skip_zero_grad': False}])
    a.grad = torch.zeros_like(a)
    a.grad[0, 0, 1, 2, 3] = 2.0
    b.grad = torch.ones_like(b)
    a0, b0 = a.detach().clone(), b.detach().clone()
    opt.step()
    assert set(opt.state[a].keys()) == {'step', 'exp_avg', 'exp_avg_sq'} and opt.state[a]['step'] == 1
    changed = (a.detach() != a0)
    assert int(changed.sum()) == 1 and bool(changed[0, 0, 1, 2, 3])
    assert torch.allclose(b.detach(), b0 - 0.01, atol=1e-6)           # first Adam step moves by lr * sign(g)
    count = torch.zeros_like(a)
    count[0, 0, 1, 2, 3] = 4.0
    count[0, 0, 0, 0, 0] = 2.0
    opt.set_pervoxel_lr(count)
    a.grad = torch.ones_like(a)
    a1 = a.detach().clone()
    opt.step()
    moved = (a.detach() != a1)
    assert int(moved.sum()) == 2                                          # per-voxel lr 0 elsewhere


def _torch_alpha(density, shift, interval):
    return 1 - torch.pow(1 + torch.exp(density + shift), -interval)


@pytest.mark.parametrize('name', ['cfgA', 'cfgB', 'cfgC'])
def test_update_occupancy_cache_vs_torch_composition(cuda_device, name):
    dev = cuda_device
    st = make_state(name, regime='fog') if name != 'cfgB' else make_state(name, xy=40, depth=24, regime='fog')
    m = model_from_state(st, dev)
    with torch.no_grad():                              # a spread of alphas, none saturated at 1
        if name == 'cfgB':
            m.density.grid.sub_(8.0)                   # interval = 256/24: keep exp(d) small
        else:
            m.density.grid.mul_(4.0).sub_(2.0)
    mask0 = m.mask_cache.mask.clone()
    # reference composition (lib/dvgo.py:224-233) with ATen ops on the same device
    shp = mask0.shape
    xyz = torch.stack(torch.meshgrid(*[torch.linspace(float(m.xyz_min[a]), float(m.xyz_max[a]), shp[a], device=dev) for a in range(3)],
                                     indexing='ij'), -1)
    ind = ((xyz.reshape(1, 1, 1, -1, 3) - m.xyz_min) / (m.xyz_max - m.xyz_min)).flip((-1,)) * 2 - 1
    den = F.grid_sample(m.density.grid, ind, mode='bilinear', align_corners=True).reshape(shp)
    shift = 0.0 if name == 'cfgB' else float(m.act_shift)
    alpha = _torch_alpha(den, shift, float(m.voxel_size_ratio))
    # threshold at the 98.5th percentile of the voxel alphas: after the 3x3x3 max-pool about a third stays occupied
    thres = float(torch.quantile(alpha.flatten()[:1 << 20], 0.985))
    assert 0 < thres < 0.999
    m.fast_color_thres = thres
    want = mask0 & (F.max_pool3d(alpha[None, None], kernel_size=3, padding=1, stride=1)[0, 0] > thres)
    m.update_occupancy_cache()
    got = m.mask_cache.mask
    flips = int((got != want).sum())
    assert flips <= max(1, int(1e-4 * got.numel())), (flips, got.numel())
    assert 0 < int(got.sum()) < got.numel()            # the update really decided something both ways
    # the next render sees the new mask
    from helpers import rays_for
    (ro, rd, vd), kw = rays_for(st, 16, 16)
    out = m.render_rays(ro.to(dev), rd.to(dev), vd.to(dev), kw, debug=True)
    assert out['rgb_marched'].isfinite().all()


def test_resample_trilinear_vs_aten(cuda_device):
    g = torch.Generator().manual_seed(4)
    src = torch.randn(1, 5, 13, 9, 21, generator=g).to(cuda_device)
    for size in ((20, 17, 33), (13, 9, 21), (7, 4, 11), (1, 1, 1)):
        grid_ = k4nerf.grid.DenseGrid(5, list(src.shape[2:]), [-1, -1, -1], [1, 1, 1]).to(cuda_device)
        grid_.grid.data.copy_(src)
        grid_.scale_volume_grid(torch.tensor(size))
        want = F.interpolate(src, size=size, mode='trilinear', align_corners=True)
        assert grid_.grid.shape == want.shape
        assert torch.allclose(grid_.grid.data, want, atol=2e-6, rtol=1e-6), (size, (grid_.grid.data - want).abs().max().item())


def test_scale_volume_grid_end_to_end(cuda_device):
    """DirectVoxGO.scale_volume_grid (lib/dvgo.py:200-221): new world size, resampled grids, rebuilt mask."""
    dev = cuda_device
    st = make_state('cfgA', res=24, regime='fog')
    m = model_from_state(st, dev)
    with torch.no_grad():
        m.density.grid.mul_(4.0).sub_(2.0)
    den0, k00, mask0 = m.density.grid.data.clone(), m.k0.grid.data.clone(), m.mask_cache.mask.clone()
    m.scale_volume_grid(32 ** 3)
    ws = m.world_size.tolist()
    assert ws == [32, 32, 32] and list(m.density.grid.shape[2:]) == ws and list(m.k0.grid.shape[1:]) == [12] + ws
    want_den = F.interpolate(den0, size=tuple(ws), mode='trilinear', align_corners=True)
    assert torch.allclose(m.density.grid.data, want_den, atol=2e-6, rtol=1e-6)
    assert torch.allclose(m.k0.grid.data, F.interpolate(k00, size=tuple(ws), mode='trilinear', align_corners=True), atol=2e-6, rtol=1e-6)
    alpha = _torch_alpha(want_den, float(m.act_shift), float(m.voxel_size_ratio))
    want_mask = F.max_pool3d(alpha, kernel_size=3, padding=1, stride=1)[0, 0] > float(m.fast_color_thres)   # old mask was all true
    assert bool(mask0.all())
    flips = int((m.mask_cache.mask != want_mask).sum())
    assert flips <= max(1, int(1e-4 * want_mask.numel())), flips
    assert list(m.mask_cache.mask.shape) == ws
    from helpers import rays_for
    (ro, rd, vd), kw = rays_for(st, 16, 16)
    out = m.render_rays(ro.to(dev), rd.to(dev), vd.to(dev), kw)
    assert out['rgb_marched'].isfinite().all()


def test_total_variation_hooks(cuda_device):
    dev = cuda_device
    st = make_state('cfgA', res=16, regime='fog')
    m = model_from_state(st, dev)
    m.density.grid.grad = torch.zeros_like(m.density.grid)
    m.k0.grid.grad = torch.zeros_like(m.k0.grid)
    m.density_total_variation_add_grad(1e-3, True)
    m.k0_total_variation_add_grad(1e-3, False)             # sparse mode with an all-zero grad: untouched
    assert float(m.density.grid.grad.abs().sum()) > 0 and float(m.k0.grid.grad.abs().sum()) == 0
    # dense TV gradient == autograd of the reference's loss definition: sum over neighbour pairs of
    # huber(delta=1)(difference) * w/6 * 2 directions ... checked through the analytic form instead:
    p = m.density.grid.data
    w = float(1e-3 * m.world_size.max() / 128) / 6
    want = torch.zeros_like(p)
    for dim in (2, 3, 4):
        d = (p.narrow(dim, 1, p.shape[dim] - 1) - p.narrow(dim, 0, p.shape[dim] - 1)).clamp(-1, 1) * w
        want.narrow(dim, 1, p.shape[dim] - 1).add_(d)
        want.narrow(dim, 0, p.shape[dim] - 1).sub_(d)
    assert torch.allclose(m.density.grid.grad, want, atol=1e-7, rtol=1e-5)


def test_mask_cache_path_constructor_branch(cuda_device, tmp_path):
    """Fine-stage constructor with a coarse checkpoint (lib/dvgo.py:134-145, lib/grid.py:277-285): the mask is
    the coarse occupancy (max-pooled density, softplus alpha >= thres) looked up at the fine mask grid."""
    g = torch.Generator().manual_seed(8)
    dens = torch.randn(1, 1, 10, 12, 9, generator=g) * 4 - 2
    coarse = {'model_state_dict': {'density.grid': dens, 'act_shift': torch.tensor([-4.5951])},
              'model_kwargs': {'voxel_size_ratio': 1.0, 'xyz_min': [-1.0, -1.0, -1.0], 'xyz_max': [1.0, 1.0, 1.0]}}
    path = str(tmp_path / 'coarse_last.tar')
    torch.save(coarse, path)
    mg = k4nerf.grid.MaskGrid(path=path, mask_cache_thres=0.5)
    d = F.max_pool3d(dens, kernel_size=3, padding=1, stride=1)
    want = (1 - torch.exp(-F.softplus(d - 4.5951) * 1.0) >= 0.5)[0, 0]
    assert torch.equal(mg.mask, want) and 0 < int(want.sum()) < want.numel()
    m = k4nerf.DirectVoxGO(xyz_min=[-0.8, -0.8, -0.8], xyz_max=[0.8, 0.8, 0.8], num_voxels=16 ** 3, num_voxels_base=16 ** 3,
                           alpha_init=1e-2, mask_cache_path=path, mask_cache_thres=0.5, fast_color_thres=1e-4, rgbnet_dim=0)
    ws = m.world_size.tolist()
    assert list(m.mask_cache.mask.shape) == ws and m.get_kwargs()['mask_cache_path'] == path
    # nearest-voxel lookup of the coarse mask at the fine grid's points (lib/grid.py:295-304)
    pts = torch.stack(torch.meshgrid(*[torch.linspace(-0.8, 0.8, w) for w in ws], indexing='ij'), -1)
    ijk = torch.round(pts * mg.xyz2ijk_scale + mg.xyz2ijk_shift).long()
    assert torch.equal(m.mask_cache.mask, want[ijk[..., 0], ijk[..., 1], ijk[..., 2]])


@pytest.mark.parametrize('dense', [True, False])
def test_total_variation_matches_c_oracle(cuda_device, dense):
    """The same kernel against the CPU restatement (oracle/render_utils_ref.c) -- parity without oracle/_ref."""
    g = torch.Generator().manual_seed(13)
    param = torch.randn(1, 3, 9, 11, 7, generator=g) * 1.5
    grad = torch.randn(param.shape, generator=g)
    grad[torch.rand(param.shape, generator=g) < 0.5] = 0
    want = grad.clone()
    ops.CpuOps.total_variation_add_grad(param, want, 0.37, 1.1, 2.3e-3, dense)
    got = grad.clone().to(cuda_device)
    total_variation_cuda.total_variation_add_grad(param.to(cuda_device), got, 0.37, 1.1, 2.3e-3, dense)
    assert torch.equal(got.cpu(), want)


@pytest.mark.parametrize('variant', ['plain', 'masked', 'perlr'])
def test_adam_matches_c_oracle(cuda_device, variant):
    g = torch.Generator().manual_seed(17)
    n = 4096 + 3
    p, m, v = torch.randn(n, generator=g), torch.randn(n, generator=g) * 0.1, (torch.randn(n, generator=g) * 0.1) ** 2
    perlr = torch.rand(n, generator=g)
    gp, gm, gv, gl = p.to(cuda_device), m.to(cuda_device), v.to(cuda_device), perlr.to(cuda_device)
    for step in (1, 5, 200):
        grad = torch.randn(n, generator=g)
        grad[torch.rand(n, generator=g) < 0.7] = 0
        gg = grad.to(cuda_device)
        if variant == 'plain':
            ops.CpuOps.adam_upd(p, grad, m, v, step, 0.9, 0.99, 0.1, 1e-8)
            adam_upd_cuda.adam_upd(gp, gg, gm, gv, step, 0.9, 0.99, 0.1, 1e-8)
        elif variant == 'masked':
            ops.CpuOps.masked_adam_upd(p, grad, m, v, step, 0.9, 0.99, 0.1, 1e-8)
            adam_upd_cuda.masked_adam_upd(gp, gg, gm, gv, step, 0.9, 0.99, 0.1, 1e-8)
        else:
            ops.CpuOps.adam_upd_with_perlr(p, grad, m, v, perlr, step, 0.9, 0.99, 0.1, 1e-8)
            adam_upd_cuda.adam_upd_with_perlr(gp, gg, gm, gv, gl, step, 0.9, 0.99, 0.1, 1e-8)
        for a, b, name in ((p, gp, 'param'), (m, gm, 'exp_avg'), (v, gv, 'exp_avg_sq')):
            assert torch.equal(a, b.cpu()), (variant, step, name)


# ---- DenseGrid.forward on the fused kernels (k4_op_grid_sample / _backward) vs ATen grid_sample + autograd -------------
@pytest.mark.parametrize('shape,C', [((37, 29, 41), 12), ((24, 24, 24), 1), ((1, 1, 33), 1), ((19, 45, 8), 5)])
def test_dense_grid_forward_and_gradient_scatter_vs_aten(cuda_device, shape, C):
    import torch.nn.functional as F
    from k4nerf import grid as kgrid
    dev = cuda_device
    g = torch.Generator().manual_seed(7)
    lo, hi = torch.tensor([-1.0, -1.3, -0.7]), torch.tensor([1.1, 0.9, 1.4])
    dg = kgrid.DenseGrid(C, shape, lo, hi).to(dev)
    with torch.no_grad():
        dg.grid.copy_(torch.randn(dg.grid.shape, generator=g))
    M = 50000
    xyz = (lo + (hi - lo) * (torch.rand(M, 3, generator=g) * 1.1 - 0.05)).to(dev)      # 5 % of the points outside the box
    xyz[:64] = lo.to(dev)                                                              # exact corners / faces
    xyz[64:128] = hi.to(dev)

    def aten(grid_t, pts):
        ind = ((pts.reshape(1, 1, 1, -1, 3) - lo.to(dev).to(grid_t.dtype)) / (hi - lo).to(dev).to(grid_t.dtype)).flip((-1,)) * 2 - 1
        o = F.grid_sample(grid_t, ind, mode='bilinear', align_corners=True)
        return o.reshape(C, -1).T
    ours = dg(xyz).reshape(M, C)
    ref = aten(dg.grid.detach(), xyz)
    assert torch.equal(ours, ref), (ours - ref).abs().max().item()                     # same corner order and FMA chain as ATen
    w = torch.randn(M, C, generator=g).to(dev)
    (ours * w).sum().backward()
    g64 = dg.grid.detach().double().requires_grad_(True)
    (aten(g64, xyz.double()) * w.double()).sum().backward()
    scale = g64.grad.abs().max().item()
    assert (dg.grid.grad.double() - g64.grad).abs().max().item() <= 2e-5 * scale
    # positions that carry a gradient fall back to the ATen path (not used by the reference, kept for generality)
    xr = xyz[:100].clone().requires_grad_(True)
    dg(xr).sum().backward()
    assert xr.grad is not None and torch.isfinite(xr.grad).all()


def test_coarse_stage_helpers(cuda_device):
    """voxel_count_views / hit_coarse_geo / maskout_near_cam_vox / update_occupancy_cache_lt_nviews (k4nerf/coarse.py) against
    plain-torch restatements of lib/dvgo.py:185-198,235-266,281-293."""
    import torch.nn.functional as F
    import k4nerf
    from helpers import make_state, model_from_state
    from oracle import scenes
    dev = cuda_device
    st = make_state('cfgA', res=32, regime='shell')
    m = model_from_state(st, dev)
    H, W = 24, 32
    views = []
    for th in (20.0, 140.0, 260.0):
        K, c2w = scenes.blender_camera(H, W, theta=th, phi=-25.0)
        views.append(k4nerf.get_rays_of_a_view(H, W, K, c2w, False, False, False, False, device=dev))
    ro = torch.stack([v[0] for v in views]); rd = torch.stack([v[1] for v in views])
    cnt = m.voxel_count_views(ro, rd, [1, 1, 1], near=2.0, far=6.0, stepsize=0.5)
    # restatement: autograd through ATen grid_sample of a grid of ones
    ref = torch.zeros_like(cnt)
    n_samples = int(float(torch.linalg.norm(m.world_size.float() + 1)) / 0.5) + 1
    rng = torch.arange(n_samples, device=dev)[None].float()
    lo, hi = m.xyz_min, m.xyz_max
    for o, d in zip(ro, rd):
        g = torch.ones_like(ref, requires_grad=True)
        o, d = o.reshape(-1, 3), d.reshape(-1, 3)
        v = torch.where(d == 0, torch.full_like(d, 1e-6), d)
        a, b = (hi - o) / v, (lo - o) / v
        t0 = torch.minimum(a, b).amax(-1).clamp(min=2.0, max=1e9)
        t = t0[:, None] + 0.5 * m.voxel_size.to(dev) * rng / d.norm(dim=-1, keepdim=True)
        pts = o[:, None] + d[:, None] * t[..., None]
        ind = ((pts.reshape(1, 1, 1, -1, 3) - lo) / (hi - lo)).flip((-1,)) * 2 - 1
        F.grid_sample(g, ind, mode='bilinear', align_corners=True).sum().backward()
        ref += (g.grad > 1)
    assert (cnt != ref).float().mean().item() < 1e-3 and float(cnt.max()) == 3.0          # sums differ by rounding order only
    # hit_coarse_geo == "some in-box sample of the ray falls into an occupied voxel"
    o, d = ro[0], rd[0]
    hit = m.hit_coarse_geo(o, d, near=2.0, far=6.0, stepsize=0.5)
    pts, ray_id, _ = m.sample_ray(o.reshape(-1, 3), d.reshape(-1, 3), 2.0, 6.0, 0.5)
    ref_hit = torch.zeros(H * W, dtype=torch.bool, device=dev)
    ref_hit.index_put_((ray_id[m.mask_cache(pts)],), torch.tensor(True, device=dev))
    assert hit.shape == (H, W) and torch.equal(hit.reshape(-1), ref_hit) and 0 < int(hit.sum()) < H * W
    # maskout_near_cam_vox
    cam = torch.tensor([[0.9, 0.9, 0.9]], device=dev)
    before = int((m.density.grid == -100).sum())
    m.maskout_near_cam_vox(cam, 0.3)
    assert int((m.density.grid == -100).sum()) > before
    # lt_nviews on the MPI model: voxels seen by fewer than 2 of 2 identical views stay as they are, unseen ones go
    stb = make_state('cfgB', xy=32, depth=16, regime='fog')
    mb = model_from_state(stb, dev)
    rays, kwb = scenes.llff_rays(16, 20), dict(scenes.RENDER_KW_MPI)
    ob, db = rays[0].to(dev), rays[1].to(dev)
    n0 = int(mb.mask_cache.mask.sum())
    mb.update_occupancy_cache_lt_nviews(torch.cat([ob, ob]), torch.cat([db, db]), [ob.shape[0]] * 2, kwb, 2)
    n1 = int(mb.mask_cache.mask.sum())
    assert 0 < n1 < n0
