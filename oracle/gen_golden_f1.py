"""Generate tests/golden/f1_*.pt (SURVEY §8f.1: SRResNet + pixelshuffle, the BatchNorm VGG-style discriminators, the
ESRGAN / SRGAN train steps; one file per case, each under 1 MB) by running the UNMODIFIED reference on CPU.  Test infrastructure only.

    python oracle/gen_golden_f1.py

Harness patches (not in the reference): torchvision vgg19 is built without download; SRRaGAN_model / SRGAN_model construct
`PerceptualLoss()` unconditionally with use_gpu=True (SRRaGAN_model.py:28), which needs CUDA — replaced by a no-op
module for the CPU run (it is only used by test())."""
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

import torch  # noqa: E402
import torchvision  # noqa: E402

_orig_vgg19 = torchvision.models.vgg19
torchvision.models.vgg19 = lambda pretrained=True, **k: _orig_vgg19(weights=None)

import models.modules.architecture as arch  # noqa: E402  (reference)
import models.SRGAN_model as ref_srgan  # noqa: E402
import models.SRRaGAN_model as ref_srragan  # noqa: E402
from models import create_model  # noqa: E402
from options.options import dict_to_nonedict  # noqa: E402

from oracle import srn_oracle as O  # noqa: E402

ref_srgan.PerceptualLoss = lambda *a, **k: torch.nn.Identity()
ref_srragan.PerceptualLoss = lambda *a, **k: torch.nn.Identity()
OUT = os.path.join(ROOT, 'tests', 'golden')
torch.set_num_threads(8)


def save(name, obj):
    path = os.path.join(OUT, name)
    torch.save(obj, path)
    print('%-22s %8.1f KB' % (name, os.path.getsize(path) / 1024))


def synth_sd(net, seed, gain=1.0):
    """deterministic weights for every tensor of net.state_dict(): convs / linears kaiming-like, BatchNorm gamma ~ 1, the
    rest small; running statistics keep their defaults (fresh modules on both sides)."""
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


def module_case(net, x, seed, pat_seed, keep=6):
    sd = synth_sd(net, seed)
    net.load_state_dict(sd, strict=False)
    net.train()
    x = x.clone().requires_grad_(True)
    out = net(x)
    pat = O.synth(tuple(out.shape), pat_seed)
    (out * pat).sum().backward()
    named = list(net.named_parameters())
    norms = OrderedDict((k, float(p.grad.double().norm())) for k, p in named)
    step = max(1, len(named) // keep)
    kept = OrderedDict((k, p.grad.clone()) for k, p in named[::step] if p.grad.numel() <= 300000)
    running = OrderedDict((k, v.clone()) for k, v in net.state_dict().items() if 'running' in k or 'num_batches' in k)
    return dict(out=out.detach(), dx=x.grad.clone(), grad_norms=norms, grads=kept, running=running)


def gen_modules():
    rec = {}
    g = arch.SRResNet(3, 3, 64, 2, upscale=4, norm_type=None, act_type='relu', mode='CNA', upsample_mode='pixelshuffle')
    rec['srresnet'] = dict(cfg=dict(nb=2, norm_type=None, mode='CNA'), w_seed=301, x_seed=302, x_shape=(2, 3, 14, 10), pat_seed=303,
                           **module_case(g, O.synth_image((2, 3, 14, 10), 302), 301, 303))
    g = arch.SRResNet(3, 3, 32, 1, upscale=2, norm_type='batch', act_type='relu', mode='NAC', res_scale=0.5, upsample_mode='upconv')
    rec['srresnet_bn_nac'] = dict(cfg=dict(nb=1, nf=32, upscale=2, norm_type='batch', mode='NAC', res_scale=0.5, upsample_mode='upconv'),
                                  w_seed=311, x_seed=312, x_shape=(3, 3, 12, 8), pat_seed=313,
                                  **module_case(g, O.synth_image((3, 3, 12, 8), 312), 311, 313))
    d = arch.Discriminator_VGG_128(3, 64)
    rec['vgg128'] = dict(w_seed=321, x_seed=322, x_shape=(2, 3, 128, 128), pat_seed=323,
                         **module_case(d, O.synth_image((2, 3, 128, 128), 322), 321, 323))
    d = arch.Discriminator_VGG_192(3, 64, norm_type='batch', act_type='leakyrelu', mode='CNA')
    rec['vgg192'] = dict(w_seed=331, x_seed=332, x_shape=(2, 3, 192, 192), pat_seed=333,
                         **module_case(d, O.synth_image((2, 3, 192, 192), 332), 331, 333))
    for case, obj in rec.items():
        save('f1_%s.pt' % case, obj)


def make_opt(model):
    return dict_to_nonedict({
        'name': 'golden', 'model': model, 'scale': 4, 'gpu_ids': None, 'is_train': True, 'chop': False, 'val_lpips': False,
        'path': {'pretrain_model_G': None, 'pretrain_model_D': None, 'models': '/tmp', 'training_state': '/tmp'},
        'network_G': {'which_model_G': 'RRDB_net', 'norm_type': None, 'mode': 'CNA', 'nf': 64, 'nb': 1, 'in_nc': 3, 'out_nc': 3,
                      'gc': 32, 'group': 1, 'scale': 4},
        'network_D': {'which_model_D': 'discriminator_vgg_128', 'norm_type': 'batch', 'act_type': 'leakyrelu', 'mode': 'CNA',
                      'nf': 64, 'in_nc': 3},
        'train': {'lr_G': 1e-4, 'weight_decay_G': 0, 'beta1_G': 0.9, 'lr_D': 1e-4, 'weight_decay_D': 0, 'beta1_D': 0.9,
                  'lr_scheme': 'MultiStepLR', 'lr_steps': [50000], 'lr_gamma': 0.5, 'pixel_criterion': 'l1', 'pixel_weight': 1e-2,
                  'feature_criterion': 'l1', 'feature_weight': 1, 'gan_type': 'vanilla', 'gan_weight': 5e-3,
                  'D_update_ratio': 1, 'D_init_iters': 0, 'manual_seed': 0, 'niter': 10, 'val_freq': 10}})


def gen_steps():
    rec = {}
    for model_name in ('srragan', 'srgan'):
        model = create_model(make_opt(model_name))
        sdG = O.synth_state_dict(O.rrdbnet_shapes(nb=1), seed=341, gain=0.3)
        sdD = synth_sd(model.netD, 342)
        sdF = O.synth_state_dict(O.vgg19_shapes(34), seed=343, gain=1.0)
        model.netG.load_state_dict(sdG, strict=True)
        model.netD.load_state_dict(sdD, strict=False)
        model.netF.load_state_dict(sdF, strict=False)
        steps = []
        for step, seed in enumerate((351, 361), 1):
            data = {'LR': O.synth_image((2, 3, 32, 32), seed), 'HR': O.synth_image((2, 3, 128, 128), seed + 1)}
            model.feed_data(data, True)
            model.optimize_parameters(step)
            log = OrderedDict((k, float(v)) for k, v in model.get_current_log().items())
            G, D = model.netG.state_dict(), model.netD.state_dict()
            steps.append(dict(log=log, fake_H=model.fake_H.detach().clone(),
                              G_norms=OrderedDict((k, float(v.double().norm())) for k, v in G.items()),
                              D_norms=OrderedDict((k, float(v.double().norm())) for k, v in D.items() if 'num_batches' not in k),
                              D_running=OrderedDict((k, v.clone()) for k, v in D.items() if 'running' in k or 'num_batches' in k)))
            print(' ', model_name, 'step', step, {k: round(v, 6) for k, v in log.items()})
        rec[model_name] = dict(wG_seed=341, wD_seed=342, wF_seed=343, data_seeds=(351, 361), steps=steps)
    for model_name, obj in rec.items():
        save('f1_steps_%s.pt' % model_name, obj)


if __name__ == '__main__':
    gen_modules()
    gen_steps()
