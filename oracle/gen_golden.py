"""Generate tests/golden/*.pt by running the UNMODIFIED reference (/root/reference/codes/SRN) on CPU.

Run here (the container that has /root/reference); the fixtures it writes are committed so the GPU box
(which has no /root/reference) can check against them.  Test infrastructure only.

    python oracle/gen_golden.py

How the reference is made importable (SURVEY.md §8c): `oracle/ref_stubs/` provides empty stand-ins for
lmdb / skimage / IPython / matplotlib / tensorboardX and a functional J=1 Haar `pytorch_wavelets`
(third party, not vendored, version unpinned => the wavelet fixtures are "parity unpinned").
torchvision.models.vgg19 is patched to build the architecture without downloading weights.
All inputs/weights come from oracle.srn_oracle.synth* (hash based, no RNG).
"""
import os
import sys
from collections import OrderedDict

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = '/root/reference/codes'
sys.path.insert(0, os.path.join(HERE, 'ref_stubs'))
sys.path.insert(0, os.path.join(REF, 'SRN'))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torchvision  # noqa: E402

_orig_vgg19 = torchvision.models.vgg19
torchvision.models.vgg19 = lambda pretrained=True, **k: _orig_vgg19(weights=None)

import models.modules.architecture as arch  # noqa: E402  (reference)
import models.modules.loss as ref_loss  # noqa: E402
import utils.util as ref_util  # noqa: E402
from models import create_model  # noqa: E402
from options.options import dict_to_nonedict  # noqa: E402

from oracle import srn_oracle as O  # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
os.makedirs(OUT, exist_ok=True)
torch.set_num_threads(8)


def save(name, obj):
    path = os.path.join(OUT, name)
    torch.save(obj, path)
    print('%-22s %8.1f KB' % (name, os.path.getsize(path) / 1024))


def grad_summary(named_params, keep):
    norms = OrderedDict((k, float(p.grad.double().norm())) for k, p in named_params)
    kept = OrderedDict((k, p.grad.clone()) for k, p in named_params if k in keep)
    return norms, kept


# ---------------------------------------------------------------- G1: RRDBNet (nb=1) fwd + bwd
def gen_rrdbnet():
    nb = 1
    net = arch.RRDBNet(in_nc=3, out_nc=3, nf=64, nb=nb, gc=32, upscale=4, norm_type=None, act_type='leakyrelu',
                       mode='CNA', upsample_mode='upconv')
    shapes = O.rrdbnet_shapes(nb=nb)
    assert list(net.state_dict().keys()) == list(shapes.keys())
    assert all(tuple(v.shape) == shapes[k] for k, v in net.state_dict().items())
    sd = O.synth_state_dict(shapes, seed=1, gain=0.3)
    net.load_state_dict(sd, strict=True)
    x = O.synth_image((2, 3, 12, 10), 11).requires_grad_(True)
    out = net(x)
    pat = O.synth(tuple(out.shape), 12)
    (out * pat).sum().backward()
    keep = ['model.0.weight', 'model.0.bias', 'model.1.sub.0.RDB1.conv1.0.weight', 'model.1.sub.0.RDB2.conv3.0.bias',
            'model.1.sub.0.RDB3.conv5.0.weight', 'model.3.weight', 'model.10.weight', 'model.10.bias']
    norms, kept = grad_summary(list(net.named_parameters()), keep)
    save('rrdbnet_nb1.pt', dict(nb=nb, x_seed=11, x_shape=(2, 3, 12, 10), w_seed=1, w_gain=0.3, pat_seed=12,
                                out=out.detach(), dx=x.grad.clone(), grad_norms=norms, grads=kept))


# ---------------------------------------------------------------- G2: NLayerDiscriminator fwd + bwd
def gen_nlayer_d():
    net = arch.NLayerDiscriminator(9, n_layers=2)
    shapes = O.nlayer_d_shapes(9, 64, 2)
    assert list(net.state_dict().keys()) == list(shapes.keys())
    sd = O.synth_state_dict(shapes, seed=2, gain=1.0)
    net.load_state_dict(sd, strict=True)
    x = O.synth_image((2, 9, 32, 32), 21).requires_grad_(True)
    out = net(x)
    pat = O.synth(tuple(out.shape), 22)
    (out * pat).sum().backward()
    norms, kept = grad_summary(list(net.named_parameters()), ['model.0.weight', 'model.0.bias', 'model.8.weight', 'model.8.bias'])
    save('nlayer_d.pt', dict(x_seed=21, x_shape=(2, 9, 32, 32), w_seed=2, pat_seed=22, out=out.detach(),
                             dx=x.grad.clone(), grad_norms=norms, grads=kept))


# ---------------------------------------------------------------- G3: VGG19 features[:35]
def gen_vgg():
    net = arch.VGGFeatureExtractor(feature_layer=34, use_bn=False, use_input_norm=True, device=torch.device('cpu'))
    shapes = O.vgg19_shapes(34)
    own = [k for k in net.state_dict().keys() if k.startswith('features')]
    assert own == list(shapes.keys()), (own[:4], list(shapes.keys())[:4])
    sd = O.synth_state_dict(shapes, seed=3, gain=1.0)
    net.load_state_dict(sd, strict=False)
    x = O.synth_image((1, 3, 32, 32), 31).requires_grad_(True)
    out = net(x)
    pat = O.synth(tuple(out.shape), 32)
    (out * pat).sum().backward()
    save('vgg19.pt', dict(x_seed=31, x_shape=(1, 3, 32, 32), w_seed=3, pat_seed=32, out=out.detach(), dx=x.grad.clone()))


# ---------------------------------------------------------------- G4: filters / losses / host utils
def gen_misc():
    x = O.synth_image((2, 3, 16, 12), 41)
    d = OrderedDict(x_seed=41, x_shape=(2, 3, 16, 12))
    d['gau_low_k5'] = arch.FilterLow(kernel_size=5, gaussian=True)(x)
    d['gau_high_k5'] = arch.FilterHigh(kernel_size=5, gaussian=True)(x)
    d['avg_low_k5_incl'] = arch.FilterLow(kernel_size=5, gaussian=False, include_pad=True)(x)
    d['avg_high_k5_excl'] = arch.FilterHigh(kernel_size=5, gaussian=False, include_pad=False)(x)
    d['gau_high_k9'] = arch.FilterHigh(kernel_size=9, gaussian=True)(x)
    w = O.synth_image((2, 1, 4, 3), 42)
    d['w_seed'] = 42
    d['bilinear_x4'] = torch.nn.functional.interpolate(w, size=(16, 12), mode='bilinear', align_corners=False)
    p = O.synth((2, 1, 6, 6), 43, 3.0)
    d['p_seed'] = 43
    for t in ('vanilla', 'lsgan', 'wgan-gp'):
        g = ref_loss.GANLoss(t, 1.0, 0.0)
        d['gan_%s_real' % t] = g(p, True).clone()
        d['gan_%s_fake' % t] = g(p, False).clone()
    fa, re = ref_util.b_split(x.repeat(2, 1, 1, 1), [0, 0, 1, 1])
    d['b_split_fake'], d['b_split_real'] = fa, re
    img = ref_util.tensor2img(x[0] * 1.2 - 0.1)
    img2 = ref_util.tensor2img(x[1])
    d['tensor2img'] = torch.from_numpy(img.copy())
    d['psnr'] = ref_util.calculate_psnr(img, img2)
    big = O.synth_image((2, 3, 24, 24), 44)
    i1, i2 = ref_util.tensor2img(big[0]), ref_util.tensor2img(big[0] * 0.9 + 0.1 * big[1])
    d['ssim_seed'] = 44
    d['ssim'] = float(ref_util.calculate_ssim(i1, i2))
    save('misc.pt', d)


# ---------------------------------------------------------------- G5: DASR_Model train steps, G6: SRModel test
def make_opt(is_train, model, nb=1, fs='wavelet', ragan=False):
    opt = {
        'name': 'golden', 'model': model, 'scale': 4, 'gpu_ids': None, 'is_train': is_train, 'chop': False,
        'val_lpips': False, 'multiweights': True,
        'path': {'pretrain_model_G': None, 'pretrain_model_D_target': None, 'pretrain_model_D_source': None,
                 'models': '/tmp', 'training_state': '/tmp'},
        'network_G': {'which_model_G': 'RRDB_net', 'norm_type': None, 'mode': 'CNA', 'nf': 64, 'nb': nb, 'in_nc': 3,
                      'out_nc': 3, 'gc': 32, 'group': 1, 'scale': 4},
        'network_D': {'which_model_D': 'discriminator_patch', 'which_model_pairD': 'discriminator_patch',
                      'norm_type': 'Batch', 'act_type': 'leakyrelu', 'mode': 'CNA', 'nf': 64,
                      'in_nc': 9 if fs == 'wavelet' else 3, 'n_layers': 2},
        'train': {'lr_G': 5e-5, 'weight_decay_G': 0, 'beta1_G': 0.9, 'lr_D': 5e-5, 'weight_decay_D': 0, 'beta1_D': 0.9,
                  'lr_scheme': 'MultiStepLR', 'lr_steps': [50000, 80000], 'lr_gamma': 0.5, 'fs': fs, 'norm': True,
                  'sup_LL': True, 'fs_kernel_size': 5, 'pixel_criterion': 'l1', 'pixel_weight': 1, 'pixel_LL_weight': 1,
                  'feature_criterion': 'l1', 'feature_weight': 1e-2, 'gan_type': 'vanilla', 'ragan': ragan,
                  'gan_H_target': 1e-4, 'gan_H_source': 0, 'G_update_inter': 1, 'D_update_inter': 1,
                  'D_update_ratio': 1, 'D_init_iters': 0, 'manual_seed': 0, 'niter': 10, 'val_freq': 10},
    }
    return dict_to_nonedict(opt)


def synth_batch(B, h, w, seed):
    return {'LR_real': O.synth_image((B, 3, h, w), seed), 'LR_fake': O.synth_image((B, 3, h, w), seed + 1),
            'HR': O.synth_image((B, 3, 4 * h, 4 * w), seed + 2), 'HR_unpair': O.synth_image((B, 3, 4 * h, 4 * w), seed + 3),
            'fake_w': O.synth_image((B, 1, h, w), seed + 4)}


def gen_dasr_step(fs, name, ragan=False):
    nb = 1
    model = create_model(make_opt(True, 'DASR', nb, fs, ragan))
    in_nc_d = 9 if fs == 'wavelet' else 3
    sdG = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), seed=5, gain=0.3)
    sdD = O.synth_state_dict(O.nlayer_d_shapes(in_nc_d, 64, 2), seed=6, gain=1.0)
    sdF = O.synth_state_dict(O.vgg19_shapes(34), seed=7, gain=1.0)
    model.netG.load_state_dict(sdG, strict=True)
    model.netD_target.load_state_dict(sdD, strict=True)
    model.netF.load_state_dict(sdF, strict=False)
    B, h, w = 2, 8, 8
    keepG = ['model.0.weight', 'model.1.sub.0.RDB1.conv1.0.bias', 'model.1.sub.0.RDB2.conv5.0.weight', 'model.10.weight']
    keepD = ['model.0.weight', 'model.8.weight', 'model.8.bias']
    rec = dict(nb=nb, B=B, h=h, w=w, fs=fs, data_seeds=[51, 61], wG_seed=5, wD_seed=6, wF_seed=7, gain_G=0.3, ragan=ragan, steps=[])
    for step, seed in enumerate(rec['data_seeds'], 1):
        model.update_learning_rate() if False else None  # train.py:105 steps schedulers first; LR unchanged before 50k iters
        model.feed_data(synth_batch(B, h, w, seed), True)
        model.optimize_parameters(step)
        log = OrderedDict(model.get_current_log())
        G = model.netG.state_dict()
        D = model.netD_target.state_dict()
        rec['steps'].append(dict(
            log=log, fake_H=model.fake_H.detach().clone(),
            G_norms=OrderedDict((k, float(v.double().norm())) for k, v in G.items()),
            D_norms=OrderedDict((k, float(v.double().norm())) for k, v in D.items()),
            G_keep=OrderedDict((k, G[k].clone()) for k in keepG), D_keep=OrderedDict((k, D[k].clone()) for k in keepD),
            G_delta_norm=float(sum(((G[k] - sdG[k]).double() ** 2).sum() for k in G) ** 0.5),
            D_delta_norm=float(sum(((D[k] - sdD[k]).double() ** 2).sum() for k in D) ** 0.5)))
        print('  step', step, {k: round(v, 6) for k, v in log.items()})
    # one file per step keeps every fixture under 1 MB (tests/helpers.py load_train_steps)
    for k, s in enumerate(rec.pop('steps'), 1):
        save(name.replace('.pt', '.step%d.pt' % k), s)
    save(name, rec)


def gen_dasr_ragan():
    """`ragan: true` (DASR_model.py:242-247,273-275): relativistic average terms in the G and D losses."""
    gen_dasr_step('gau', 'dasr_step_ragan.pt', ragan=True)


def gen_sr_test():
    nb = 1
    model = create_model(make_opt(False, 'sr', nb))
    sdG = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), seed=8, gain=0.3)
    model.netG.load_state_dict(sdG, strict=True)
    lr = O.synth_image((1, 3, 10, 14), 81)
    hr = O.synth_image((1, 3, 40, 56), 82)
    model.feed_data({'LR': lr, 'HR': hr})
    model.test()
    vis = model.get_current_visuals(need_HR=True)
    SR = vis['SR'].clone()  # tensor2img clamps its argument IN PLACE (utils/util.py:186)
    # synthetic weights give a low-amplitude output: stretch it into [0,1] so the uint8 image / PSNR / SSIM are non-trivial
    sr_img = ref_util.tensor2img(SR * 8.0 + 0.5)
    hr_img = ref_util.tensor2img(vis['HR'].clone())
    save('sr_test.pt', dict(nb=nb, w_seed=8, gain=0.3, lr_seed=81, hr_seed=82, lr_shape=(1, 3, 10, 14),
                            SR=SR, sr_img=torch.from_numpy(sr_img.copy()),
                            psnr=ref_util.calculate_psnr(sr_img, hr_img), ssim=float(ref_util.calculate_ssim(sr_img, hr_img))))


if __name__ == '__main__':
    if len(sys.argv) > 1:
        for n in sys.argv[1:]:
            globals()['gen_' + n]()
        sys.exit(0)
    gen_rrdbnet()
    gen_nlayer_d()
    gen_vgg()
    gen_misc()
    gen_dasr_step('wavelet', 'dasr_step_wavelet.pt')
    gen_dasr_step('gau', 'dasr_step_gau.pt')
    gen_dasr_ragan()
    gen_sr_test()
