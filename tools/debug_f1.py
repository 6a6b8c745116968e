"""Where does the 1e-3 deviation of the first-layer filter gradients of Discriminator_VGG_128 come from?
Compares (a) our kernels, (b) torch's own GPU fp32 operators (cuDNN), (c) the reference fixture (torch CPU fp32) against
the float64 evaluation of the same algorithm, per parameter; then isolates the wgrad kernel on float64-derived inputs."""
import copy
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
import torch
from oracle import srn_oracle as O
from helpers import native_forward, truth64
from test_gpu_f1 import synth_sd
from dasr_b200.srn.models.modules.architecture import Discriminator_VGG_128, Discriminator_VGG_192

torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False
for name, net in (('vgg128', Discriminator_VGG_128(3, 64)),
                  ('vgg192', Discriminator_VGG_192(3, 64, norm_type='batch', act_type='leakyrelu', mode='CNA'))):
    gg = torch.load(os.path.join(ROOT, 'tests', 'golden', 'f1_%s.pt' % name))
    net.load_state_dict(synth_sd(net, gg['w_seed']), strict=False)
    net.train()
    x = O.synth_image(gg['x_shape'], gg['x_seed'])
    pat = O.synth(tuple(gg['out'].shape), gg['pat_seed'])
    _, t_dx, t_grads = truth64(net, x, pat)
    peer = copy.deepcopy(net).cuda()
    xp = x.cuda().requires_grad_(True)
    (native_forward(peer, xp) * pat.cuda()).sum().backward()
    net.cuda()
    xo = x.cuda().requires_grad_(True)
    (net(xo) * pat.cuda()).sum().backward()
    rl = lambda a, b: float((a.double().cpu() - b.double().cpu()).abs().max() / b.double().abs().max().clamp_min(1e-30))
    print('== %s: rel-Linf vs float64 truth   ours | torch-GPU fp32 | reference fixture (torch-CPU fp32)' % name)
    print('  dx            %.2e | %.2e | %.2e' % (rl(xo.grad, t_dx), rl(xp.grad, t_dx), rl(gg['dx'], t_dx)))
    pn, pp = dict(net.named_parameters()), dict(peer.named_parameters())
    for k in gg['grads']:
        print('  %-20s %.2e | %.2e | %.2e   (|g|max %.2e)' % (k, rl(pn[k].grad, t_grads[k]), rl(pp[k].grad, t_grads[k]),
                                                             rl(gg['grads'][k], t_grads[k]), float(t_grads[k].abs().max())))
