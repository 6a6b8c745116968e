"""Pins the CPU oracle (oracle/srn_oracle.py) against fixtures produced by the imported reference
(oracle/gen_golden.py -> tests/golden/*.pt).  CPU only; runs in the `-m "not gpu"` suite."""
import numpy as np
import torch

from oracle import srn_oracle as O


def rel_linf(a, b):
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def test_rrdbnet_forward_backward(golden):
    g = golden('rrdbnet_nb1.pt')
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['w_seed'], g['w_gain'])
    p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    x = O.synth_image(g['x_shape'], g['x_seed']).requires_grad_(True)
    out = O.rrdbnet_forward(x, p, g['nb'])
    assert out.shape == g['out'].shape
    assert rel_linf(out.detach(), g['out']) < 1e-5
    (out * O.synth(tuple(out.shape), g['pat_seed'])).sum().backward()
    assert rel_linf(x.grad, g['dx']) < 1e-4
    for k, ref in g['grads'].items():
        assert rel_linf(p[k].grad, ref) < 1e-4, k
    for k, n in g['grad_norms'].items():
        assert abs(float(p[k].grad.double().norm()) - n) <= 1e-4 * max(n, 1e-12), k


def test_nlayer_discriminator(golden):
    g = golden('nlayer_d.pt')
    sd = O.synth_state_dict(O.nlayer_d_shapes(9, 64, 2), g['w_seed'], 1.0)
    p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    x = O.synth_image(g['x_shape'], g['x_seed']).requires_grad_(True)
    out = O.nlayer_d_forward(x, p, 2)
    assert rel_linf(out.detach(), g['out']) < 1e-5
    (out * O.synth(tuple(out.shape), g['pat_seed'])).sum().backward()
    assert rel_linf(x.grad, g['dx']) < 1e-4
    for k, ref in g['grads'].items():
        assert rel_linf(p[k].grad, ref) < 1e-4, k


def test_vgg19_features(golden):
    g = golden('vgg19.pt')
    sd = O.synth_state_dict(O.vgg19_shapes(34), g['w_seed'], 1.0)
    x = O.synth_image(g['x_shape'], g['x_seed']).requires_grad_(True)
    out = O.vgg19_features(x, sd)
    assert out.shape == g['out'].shape
    assert rel_linf(out.detach(), g['out']) < 1e-5
    (out * O.synth(tuple(out.shape), g['pat_seed'])).sum().backward()
    assert rel_linf(x.grad, g['dx']) < 1e-4


def test_filters_losses_utils(golden):
    g = golden('misc.pt')
    x = O.synth_image(g['x_shape'], g['x_seed'])
    assert torch.allclose(O.filter_low(x, 5, True), g['gau_low_k5'], atol=1e-6)
    assert torch.allclose(O.filter_high(x, 5, True), g['gau_high_k5'], atol=1e-6)
    assert torch.allclose(O.filter_low(x, 5, False, True), g['avg_low_k5_incl'], atol=1e-6)
    assert torch.allclose(O.filter_high(x, 5, False, False), g['avg_high_k5_excl'], atol=1e-6)
    assert torch.allclose(O.filter_high(x, 9, True), g['gau_high_k9'], atol=1e-6)
    w = O.synth_image((2, 1, 4, 3), g['w_seed'])
    up = torch.nn.functional.interpolate(w, size=(16, 12), mode='bilinear', align_corners=False)
    assert torch.equal(up, g['bilinear_x4'])
    p = O.synth((2, 1, 6, 6), g['p_seed'], 3.0)
    for t in ('vanilla', 'lsgan', 'wgan-gp'):
        assert torch.allclose(O.gan_loss(p, True, t), g['gan_%s_real' % t], atol=1e-6)
        assert torch.allclose(O.gan_loss(p, False, t), g['gan_%s_fake' % t], atol=1e-6)
    fa, re = O.b_split(x.repeat(2, 1, 1, 1), [0, 0, 1, 1])
    assert torch.equal(fa, g['b_split_fake']) and torch.equal(re, g['b_split_real'])
    img = O.tensor2img_chw(x[0] * 1.2 - 0.1)
    assert np.array_equal(img, g['tensor2img'].numpy())
    assert abs(O.calculate_psnr(img, O.tensor2img_chw(x[1])) - g['psnr']) < 1e-9


def _check_step(golden, name):
    from helpers import load_train_steps
    g = load_train_steps(golden, name)
    fs = g['fs']
    sdG = O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['wG_seed'], g['gain_G'])
    sdD = O.synth_state_dict(O.nlayer_d_shapes(9 if fs == 'wavelet' else 3, 64, 2), g['wD_seed'], 1.0)
    sdF = O.synth_state_dict(O.vgg19_shapes(34), g['wF_seed'], 1.0)
    optG = O.AdamState(sdG, 5e-5, 0.9)
    optD = O.AdamState(sdD, 5e-5, 0.9)
    B, h, w = g['B'], g['h'], g['w']
    for seed, ref in zip(g['data_seeds'], g['steps']):
        data = {'LR_real': O.synth_image((B, 3, h, w), seed), 'LR_fake': O.synth_image((B, 3, h, w), seed + 1),
                'HR': O.synth_image((B, 3, 4 * h, 4 * w), seed + 2),
                'HR_unpair': O.synth_image((B, 3, 4 * h, 4 * w), seed + 3), 'fake_w': O.synth_image((B, 1, h, w), seed + 4)}
        log, _, _, fake_H = O.dasr_train_step(sdG, sdD, sdF, data, g['nb'], optG, optD, dict(fs=fs))
        assert list(log.keys()) == list(ref['log'].keys())
        for k in log:
            assert abs(log[k] - ref['log'][k]) <= 2e-5 * max(1.0, abs(ref['log'][k])), (k, log[k], ref['log'][k])
        assert rel_linf(fake_H, ref['fake_H']) < 1e-4
        for k, v in ref['G_keep'].items():
            assert rel_linf(sdG[k], v) < 1e-4, k
        for k, v in ref['D_keep'].items():
            assert rel_linf(sdD[k], v) < 1e-4, k
    # Adam moved the weights by ~lr per element per step, like the reference
    sd0 = O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['wG_seed'], g['gain_G'])
    dn = float(sum(((sdG[k] - sd0[k]).double() ** 2).sum() for k in sdG) ** 0.5)
    assert abs(dn - g['steps'][-1]['G_delta_norm']) < 2e-2 * g['steps'][-1]['G_delta_norm']


def test_dasr_train_step_wavelet(golden):
    _check_step(golden, 'dasr_step_wavelet.pt')


def test_dasr_train_step_gau(golden):
    _check_step(golden, 'dasr_step_gau.pt')


def test_sr_test_path(golden):
    g = golden('sr_test.pt')
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['w_seed'], g['gain'])
    lr = O.synth_image(g['lr_shape'], g['lr_seed'])
    with torch.no_grad():
        sr = O.rrdbnet_forward(lr, sd, g['nb'])
    assert rel_linf(sr[0], g['SR']) < 1e-5
    img = O.tensor2img_chw(sr[0] * 8.0 + 0.5)
    hr = O.tensor2img_chw(O.synth_image((1, 3, 40, 56), g['hr_seed'])[0])
    assert abs(O.calculate_psnr(img, hr) - g['psnr']) < 0.05
    assert np.abs(img.astype(int) - g['sr_img'].numpy().astype(int)).max() <= 1
