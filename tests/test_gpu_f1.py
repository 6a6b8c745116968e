"""GPU parity of SURVEY §8f.1: sr_resnet (+ pixelshuffle / BatchNorm 'NAC' variant), Discriminator_VGG_128 / _192 and the
SRRaGAN (ESRGAN) / SRGAN train steps, against fixtures the reference produced (oracle/gen_golden_f1.py)."""
from collections import OrderedDict

import pytest
import torch

from oracle import srn_oracle as O

pytestmark = pytest.mark.gpu
TOL = 1e-3


def rel_linf(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def synth_sd(net, seed, gain=1.0):
    sd = OrderedDict()
    for i, (k, v) in enumerate(net.state_dict().items()):
        if 'running' in k or 'num_batches' in k:
            continue
        shp = tuple(v.shape)
        if v.dim() >= 2:
            fan = 1
            for d in shp[1:]:
                fan *= d
            sd[k] = O.synth(shp, seed * 1000 + i, gain * (2.0 / fan) ** 0.5 * 3 ** 0.5)
        elif '.bn' in k or k.startswith('bn') or (k.endswith('weight') and v.dim() == 1):
            sd[k] = O.synth(shp, seed * 1000 + i, 0.3, 1.0) if k.endswith('weight') else O.synth(shp, seed * 1000 + i, 0.05)
        else:
            sd[k] = O.synth(shp, seed * 1000 + i, 0.05)
    return sd


def check_module(net, g):
    from helpers import as_good_as_reference, truth64
    net.load_state_dict(synth_sd(net, g['w_seed']), strict=False)
    net.train()
    x = O.synth_image(g['x_shape'], g['x_seed'])
    pat = O.synth(tuple(g['out'].shape), g['pat_seed'])
    _, t_dx, t_grads = truth64(net, x, pat)          # float64 result of the same algorithm (fresh running statistics)
    net.cuda()
    xg = x.cuda().requires_grad_(True)
    out = net(xg)
    assert out.shape == g['out'].shape
    e_out = rel_linf(out, g['out'])
    (out * pat.cuda()).sum().backward()
    e_dx = rel_linf(xg.grad, g['dx'])
    named = dict(net.named_parameters())
    big = max(g['grad_norms'].values())
    for k, ref in g['grads'].items():
        if g['grad_norms'][k] >= 1e-4 * big:          # (bias of a conv feeding a BatchNorm: mathematically zero gradient)
            assert as_good_as_reference(named[k].grad, ref, t_grads[k], TOL), k
    for k, n in g['grad_norms'].items():
        if n >= 1e-4 * big:
            got, t = float(named[k].grad.double().norm()), float(t_grads[k].norm())
            assert abs(got - n) <= TOL * n or abs(got - t) <= 3.0 * abs(n - t) + 1e-6 * t, (k, got, n, t)
    state = net.state_dict()
    for k, v in g['running'].items():
        if 'num_batches' in k:
            assert int(state[k]) == int(v), k
        else:
            assert rel_linf(state[k], v) < TOL, k
    print('out %.2e dx %.2e (vs reference fixture)' % (e_out, e_dx))
    assert e_out < TOL
    assert as_good_as_reference(xg.grad, g['dx'], t_dx, TOL)


def test_srresnet_pixelshuffle_vs_reference(golden):
    from dasr_b200.srn.models.modules.architecture import SRResNet
    g = golden('f1_srresnet.pt')
    check_module(SRResNet(3, 3, 64, 2, upscale=4, norm_type=None, act_type='relu', mode='CNA', upsample_mode='pixelshuffle'), g)


def test_srresnet_batchnorm_nac_upconv_vs_reference(golden):
    from dasr_b200.srn.models.modules.architecture import SRResNet
    g = golden('f1_srresnet_bn_nac.pt')
    check_module(SRResNet(3, 3, 32, 1, upscale=2, norm_type='batch', act_type='relu', mode='NAC', res_scale=0.5, upsample_mode='upconv'), g)


def test_discriminator_vgg_128_vs_reference(golden):
    from dasr_b200.srn.models.modules.architecture import Discriminator_VGG_128
    check_module(Discriminator_VGG_128(3, 64), golden('f1_vgg128.pt'))


def test_discriminator_vgg_192_vs_reference(golden):
    from dasr_b200.srn.models.modules.architecture import Discriminator_VGG_192
    check_module(Discriminator_VGG_192(3, 64, norm_type='batch', act_type='leakyrelu', mode='CNA'), golden('f1_vgg192.pt'))


@pytest.mark.parametrize('name', ['srragan', 'srgan'])
def test_srgan_train_steps_vs_reference(golden, name):
    """create_model('srragan' | 'srgan') -> feed_data -> optimize_parameters x2 (train_SRGAN.json's model with a small
    generator): log values, SR output, post-Adam weight norms and D's BatchNorm running statistics."""
    from dasr_b200.srn.models import create_model
    from dasr_b200.srn.options.options import dict_to_nonedict
    from helpers import unwrap
    g = golden('f1_steps_%s.pt' % name)
    opt = dict_to_nonedict({
        'name': 'golden', 'model': name, 'scale': 4, 'gpu_ids': [0], 'is_train': True, 'chop': False, 'val_lpips': False,
        'path': {'pretrain_model_G': None, 'pretrain_model_D': None, 'models': '/tmp', 'training_state': '/tmp'},
        'network_G': {'which_model_G': 'RRDB_net', 'norm_type': None, 'mode': 'CNA', 'nf': 64, 'nb': 1, 'in_nc': 3, 'out_nc': 3,
                      'gc': 32, 'group': 1, 'scale': 4},
        'network_D': {'which_model_D': 'discriminator_vgg_128', 'norm_type': 'batch', 'act_type': 'leakyrelu', 'mode': 'CNA',
                      'nf': 64, 'in_nc': 3},
        'train': {'lr_G': 1e-4, 'weight_decay_G': 0, 'beta1_G': 0.9, 'lr_D': 1e-4, 'weight_decay_D': 0, 'beta1_D': 0.9,
                  'lr_scheme': 'MultiStepLR', 'lr_steps': [50000], 'lr_gamma': 0.5, 'pixel_criterion': 'l1', 'pixel_weight': 1e-2,
                  'feature_criterion': 'l1', 'feature_weight': 1, 'gan_type': 'vanilla', 'gan_weight': 5e-3,
                  'D_update_ratio': 1, 'D_init_iters': 0, 'manual_seed': 0, 'niter': 10, 'val_freq': 10}})
    model = create_model(opt)
    unwrap(model.netG).load_state_dict(O.synth_state_dict(O.rrdbnet_shapes(nb=1), g['wG_seed'], 0.3))
    unwrap(model.netD).load_state_dict(synth_sd(unwrap(model.netD), g['wD_seed']), strict=False)
    unwrap(model.netF).load_state_dict(O.synth_state_dict(O.vgg19_shapes(34), g['wF_seed'], 1.0), strict=False)
    for step, (seed, ref) in enumerate(zip(g['data_seeds'], g['steps']), 1):
        model.feed_data({'LR': O.synth_image((2, 3, 32, 32), seed), 'HR': O.synth_image((2, 3, 128, 128), seed + 1)}, True)
        model.optimize_parameters(step)
        log = model.get_current_log()
        assert list(log.keys()) == list(ref['log'].keys())
        for k in log:
            assert abs(float(log[k]) - ref['log'][k]) <= 2e-3 * max(1.0, abs(ref['log'][k])), (step, k, float(log[k]), ref['log'][k])
        assert rel_linf(model.fake_H, ref['fake_H']) < TOL
        G, D = unwrap(model.netG).state_dict(), unwrap(model.netD).state_dict()
        for k, n in ref['G_norms'].items():       # two Adam steps of lr 1e-4: a handful of sign flips of ~0 gradients move a norm by ~1e-4
            assert abs(float(G[k].double().norm()) - n) <= 1e-3 * max(n, 1e-9), k
        # relativistic losses (srragan) only see score differences: the gradient of the logit bias is mathematically zero,
        # what the backward leaves there is rounding noise and Adam turns noise into a +-lr step -> not comparable
        skip = {'linear2.bias'} if name == 'srragan' else set()
        for k, n in ref['D_norms'].items():
            if k not in skip:
                assert abs(float(D[k].double().norm()) - n) <= 2e-3 * max(n, 1e-9), k
        for k, v in ref['D_running'].items():
            if 'num_batches' in k:
                assert int(D[k]) == int(v), k
