"""GPU: the training-side forward (k4nerf/train_forward.py, SURVEY.md section 8 f-2).

(i) values: the per-sample lists and per-ray outputs against the oracle pipeline running on the
reference's own kernels (replayed from their stored results, tests/ref_calls.py) on the same device; (ii) gradients: against a float64 pure-torch
restatement of alpha / transmittance / compositing with autograd (no custom backward anywhere);
(iii) a few MaskedAdam steps reduce the loss."""
import pytest
import torch

import k4nerf
from k4nerf import train_forward
from helpers import make_state, model_from_state, rays_for
from oracle import pipeline
from ref_calls import RefCalls

pytestmark = pytest.mark.gpu


@pytest.fixture
def ref_ops(request, cuda_device):
    rc = RefCalls.for_test(request)
    yield rc.ops()
    rc.finish()


def _state(name, regime):
    if name == 'cfgB':
        return make_state(name, xy=40, depth=24, regime=regime)
    return make_state(name, res=32, regime=regime)


@pytest.mark.parametrize('name', ['cfgA', 'cfgB', 'cfgC'])
@pytest.mark.parametrize('regime', ['fog', 'shell'])
def test_sample_lists_match_reference_kernel_pipeline(ref_ops, cuda_device, name, regime):
    dev = cuda_device
    torch.backends.cuda.matmul.allow_tf32 = False
    st = _state(name, regime)
    (ro, rd, vd), kw = rays_for(st, 24, 32, **({'radius': 0.6} if name == 'cfgC' else {}))
    ro, rd, vd = ro.to(dev), rd.to(dev), vd.to(dev)
    ref = pipeline.forward(pipeline.state_to(st, dev), ro, rd, vd, ref_ops, **kw)
    m = model_from_state(st, dev)
    with torch.no_grad():
        ours = train_forward.forward_samples(m, ro, rd, vd, **kw)
    assert ours['ray_id'].shape == ref['ray_id'].shape and torch.equal(ours['ray_id'], ref['ray_id'])
    assert torch.equal(ours['alphainv_last'], ref['alphainv_last'])
    assert torch.equal(ours['weights'], ref['weights']) and torch.equal(ours['raw_alpha'], ref['raw_alpha'])
    assert torch.allclose(ours['raw_rgb'], ref['raw_rgb'], atol=1e-6)
    assert torch.allclose(ours['rgb_marched'], ref['rgb_marched'], atol=1e-5)
    assert torch.allclose(ours['depth'], ref['depth'], atol=1e-5)
    assert ours['rgb_feature'] is ours['rgb_marched']
    if name != 'cfgA':
        assert ours['n_max'] == ref['n_max'] and torch.allclose(ours['s'], ref['s'], atol=1e-7)
    # and the fused inference kernel agrees with its un-fused restatement
    with torch.no_grad():
        fused = m(ro, rd, vd, **kw)
    assert pipeline.psnr(fused['rgb_marched'].cpu(), ours['rgb_marched'].cpu()) > 60


def _float64_restatement(m, ro, rd, vd, kw):
    """alpha / transmittance / compositing in float64 torch ops with plain autograd (DirectVoxGO)."""
    from k4nerf import render_utils_cuda as rops
    n = ro.shape[0]
    stepdist = kw['stepsize'] * m.voxel_size
    pts, outside, ray_id, step_id, *_ = rops.sample_pts_on_rays(ro, rd, m.xyz_min, m.xyz_max, kw['near'], 1e9, stepdist)
    pts, ray_id = pts[~outside], ray_id[~outside]
    occ = m.mask_cache(pts)
    pts, ray_id = pts[occ], ray_id[occ]
    interval = float(kw['stepsize'] * m.voxel_size_ratio)
    den = m.density(pts).double()
    alpha = 1 - (1 + torch.exp(den + float(m.act_shift))) ** (-interval)
    sel = alpha.float() > m.fast_color_thres
    pts, ray_id, alpha = pts[sel], ray_id[sel], alpha[sel]
    log1m = torch.log1p(-alpha)
    cs = torch.cumsum(log1m, 0)
    excl = cs - log1m
    first = torch.ones_like(ray_id, dtype=torch.bool)
    first[1:] = ray_id[1:] != ray_id[:-1]
    seg = torch.cumsum(first.long(), 0) - 1
    T = torch.exp(excl - excl[first][seg])
    live = (T.detach() >= 1e-3)
    T_incl = T * (1 - alpha)
    last_live = live.clone()
    last_live[:-1] &= ~(live[1:] & ~first[1:])
    alphainv_last = torch.ones(n, device=ro.device, dtype=torch.float64).index_put((ray_id[last_live],), T_incl[last_live])
    weights = T * alpha * live
    sel = weights.float() > m.fast_color_thres
    pts, ray_id, weights = pts[sel], ray_id[sel], weights[sel]
    k0 = m.k0(pts)
    e = (vd.unsqueeze(-1) * m.viewfreq).flatten(-2)
    vemb = torch.cat([vd, e.sin(), e.cos()], -1)[ray_id]
    rgb = torch.sigmoid(m.rgbnet(torch.cat([k0, vemb], -1))).double()
    rgb_marched = torch.zeros(n, 3, device=ro.device, dtype=torch.float64).index_add(0, ray_id, weights.unsqueeze(-1) * rgb)
    return rgb_marched + alphainv_last.unsqueeze(-1) * kw['bg'], alphainv_last


@pytest.mark.parametrize('regime', ['fog', 'shell'])
def test_gradients_match_float64_autograd_restatement(cuda_device, regime):
    dev = cuda_device
    torch.backends.cuda.matmul.allow_tf32 = False
    st = make_state('cfgA', res=24, regime=regime)
    (ro, rd, vd), kw = rays_for(st, 20, 24)
    ro, rd, vd = ro.to(dev), rd.to(dev), vd.to(dev)
    g = torch.Generator().manual_seed(0)
    target = torch.rand(ro.shape[0], 3, generator=g).to(dev)
    grads = []
    for which in ('ours', 'restatement'):
        m = model_from_state(st, dev)
        if which == 'ours':
            out = m(ro, rd, vd, global_step=1, **kw)             # autograd enabled -> train_forward
            assert 'weights' in out and out['rgb_marched'].requires_grad
            rgb, last = out['rgb_marched'], out['alphainv_last']
        else:
            rgb, last = _float64_restatement(m, ro, rd, vd, kw)
        loss = ((rgb - target) ** 2).mean() + 0.01 * (last ** 2).mean()
        loss.backward()
        grads.append({k: p.grad.detach().double().clone() for k, p in m.named_parameters() if p.grad is not None} | {'_loss': loss.detach().double()})
    a, b = grads
    assert abs(float(a['_loss'] - b['_loss'])) <= 1e-5 * max(1.0, abs(float(b['_loss'])))
    assert set(a) == set(b) and {'density.grid', 'k0.grid', 'rgbnet.0.weight'} <= set(a)
    for k in a:
        if k == '_loss':
            continue
        scale = b[k].abs().max().item()
        assert scale > 0, k
        err = (a[k] - b[k]).abs().max().item()
        assert err <= 2e-3 * scale, (k, err, scale)


def test_masked_adam_training_steps_reduce_the_loss(cuda_device):
    dev = cuda_device
    st = make_state('cfgA', res=24, regime='fog')
    (ro, rd, vd), kw = rays_for(st, 16, 16)
    ro, rd, vd = ro.to(dev), rd.to(dev), vd.to(dev)
    m = model_from_state(st, dev)
    target = torch.full((ro.shape[0], 3), 0.25, device=dev)
    opt = k4nerf.MaskedAdam([
        {'params': [m.density.grid], 'lr': 0.1, 'skip_zero_grad': True},
        {'params': [m.k0.grid], 'lr': 0.1, 'skip_zero_grad': True},
        {'params': list(m.rgbnet.parameters()), 'lr': 1e-3, 'skip_zero_grad': False}])
    losses = []
    for step in range(8):
        opt.zero_grad(set_to_none=True)
        out = m(ro, rd, vd, global_step=step, **kw)
        loss = ((out['rgb_marched'] - target) ** 2).mean()
        loss.backward()
        m.density_total_variation_add_grad(1e-5, False)
        opt.step()
        losses.append(float(loss.detach()))
        if step in (2, 5):
            # mid-training validation as the reference loop does it (run_sr.py:586-599): NO manual invalidate --
            # the optimiser kernels bump the parameters' versions, so the fused render sees the new weights
            with torch.no_grad():
                fused = m(ro, rd, vd, **kw)['rgb_marched'].clone()
                again = m(ro, rd, vd, **kw)['rgb_marched']
                unfused = train_forward.forward_samples(m, ro, rd, vd, **kw)['rgb_marched']
            assert pipeline.psnr(fused.cpu(), unfused.cpu()) > 55, step
            assert pipeline.psnr(fused.cpu(), again.cpu()) > 90
    assert losses[-1] < 0.9 * losses[0] and all(b < a for a, b in zip(losses, losses[1:])), losses
    with torch.no_grad():                                         # the fused kernel renders the trained scene
        fused = m(ro, rd, vd, **kw)
        unfused = train_forward.forward_samples(m, ro, rd, vd, **kw)
    assert pipeline.psnr(fused['rgb_marched'].cpu(), unfused['rgb_marched'].cpu()) > 55


def test_scene_rebuilds_when_a_baked_scalar_changes(cuda_device):
    """fast_color_thres is baked into the device scene: changing it must change the render."""
    dev = cuda_device
    st = make_state('cfgA', res=24, regime='fog')
    (ro, rd, vd), kw = rays_for(st, 16, 16)
    ro, rd, vd = ro.to(dev), rd.to(dev), vd.to(dev)
    m = model_from_state(st, dev)
    a = m.render_rays(ro, rd, vd, kw, debug=True)['counters'].clone()
    m.fast_color_thres = 0.05
    b = m.render_rays(ro, rd, vd, kw, debug=True)['counters'].clone()
    assert int(b[2]) < int(a[2]), (a, b)                      # fewer shaded samples at the higher threshold


def test_dcvgo_training_keys_and_threshold_schedule(cuda_device):
    """lib/dcvgo.py:358-371 key set (run_sr.py:531-532 reads 't' / 'raw_density') and the dict-valued
    fast_color_thres schedule (lib/dcvgo.py:269-271)."""
    dev = cuda_device
    st = make_state('cfgC', res=24, regime='fog')
    (ro, rd, vd), kw = rays_for(st, 12, 16, radius=0.6)
    ro, rd, vd = ro.to(dev), rd.to(dev), vd.to(dev)
    m = model_from_state(st, dev)
    out = m(ro, rd, vd, global_step=3, is_train=True, **kw)
    n = out['weights'].shape[0]
    for k in ('t', 'raw_density', 'step_id', 's', 'raw_alpha', 'ray_id'):
        assert out[k].shape[0] == n, k
    assert out['wsum_mid'].shape == (ro.shape[0],) and out['n_max'] > 0
    assert torch.allclose(out['s'], 1 - 1 / (1 + out['t']))
    assert (out['wsum_mid'] <= out['weights'].new_zeros(ro.shape[0]).index_add_(0, out['ray_id'], out['weights']) + 1e-6).all()
    # raw_alpha is the activation of raw_density
    interval = float(kw['stepsize'] * m.voxel_size_ratio)
    alpha = 1 - (1 + torch.exp(out['raw_density'].flatten() + float(m.act_shift))) ** (-interval)
    assert torch.allclose(alpha, out['raw_alpha'], atol=1e-6)
    m._fast_color_thres = {0: 1e-4, 5: 0.03}
    m.fast_color_thres = 1e-4
    with torch.no_grad():
        m(ro, rd, vd, global_step=4, **kw)
        assert m.fast_color_thres == 1e-4
        a = m.render_rays(ro, rd, vd, kw, debug=True)['counters'].clone()
        m(ro, rd, vd, global_step=5, **kw)
        assert m.fast_color_thres == 0.03
        b = m.render_rays(ro, rd, vd, kw, debug=True)['counters'].clone()
    assert int(b[2]) < int(a[2])
