"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle and the committed golden
fixtures generated from the reference.  Tolerances: fp32 mode 1e-3 relative L-inf (BASELINE north_star;
measured ~1e-6), bf16 tcgen05 mode 3e-2 relative L-inf on activations (operand rounding, SURVEY H2)."""
import numpy as np
import pytest
import torch

from oracle import srn_oracle as O

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-3


def rel_linf(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def cuda_sd(sd):
    return {k: v.cuda() for k, v in sd.items()}


def build_G(nb, sd):
    from dasr_b200.srn.models.modules.architecture import RRDBNet
    net = RRDBNet(3, 3, 64, nb, gc=32, upscale=4)
    net.load_state_dict(sd, strict=True)
    return net.cuda()


# ------------------------------------------------------------------------------------------------ G
def test_rrdbnet_fp32_forward_backward_vs_golden(golden):
    g = golden('rrdbnet_nb1.pt')
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['w_seed'], g['w_gain'])
    net = build_G(g['nb'], sd)
    x = O.synth_image(g['x_shape'], g['x_seed']).cuda().requires_grad_(True)
    out = net(x)
    assert out.shape == g['out'].shape
    assert rel_linf(out, g['out']) < FP32_TOL
    (out * O.synth(tuple(out.shape), g['pat_seed']).cuda()).sum().backward()
    assert rel_linf(x.grad, g['dx']) < FP32_TOL
    named = dict(net.named_parameters())
    for k, ref in g['grads'].items():
        assert rel_linf(named[k].grad, ref) < FP32_TOL, k
    for k, n in g['grad_norms'].items():
        assert abs(float(named[k].grad.double().norm()) - n) <= 1e-3 * max(n, 1e-12), k


@pytest.mark.parametrize('shape', [(1, 3, 16, 8), (2, 3, 21, 13), (1, 3, 40, 24)])
def test_rrdbnet_fp32_inference_vs_oracle(shape):
    nb = 2
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 101, 0.3)
    net = build_G(nb, sd).eval()
    net.precision = 'fp32'
    x = O.synth_image(shape, 102)
    with torch.no_grad():
        out = net(x.cuda())
        ref = O.rrdbnet_forward(x, sd, nb)
    assert rel_linf(out, ref) < FP32_TOL


@pytest.mark.parametrize('prec', ['bf16', 'bf16_layer'])
@pytest.mark.parametrize('shape', [(1, 3, 16, 8), (2, 3, 21, 13), (1, 3, 48, 40)])
def test_rrdbnet_bf16_tcgen05_vs_oracle(shape, prec):
    nb = 2
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 103, 0.3)
    net = build_G(nb, sd).eval()
    net.precision = prec
    x = O.synth_image(shape, 104)
    with torch.no_grad():
        out = net(x.cuda())
        ref = O.rrdbnet_forward(x, sd, nb)
    assert out.shape == ref.shape
    assert rel_linf(out, ref) < 1e-2          # measured 6e-4 .. 4e-3 on these shapes (bf16 operands, fp32 accumulation)
    # and the result does not depend on which A-operand path the kernel uses (shifted descriptors vs per-tap tiles)


def test_rrdbnet_bf16_batch_independence_full_width():
    """Size-independent property at the BASELINE tile width (256): a batched forward equals per-image forwards
    bit for bit (tiles never mix images; zero padding comes from TMA out-of-bounds fill)."""
    nb = 1
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 105, 0.3)
    net = build_G(nb, sd).eval()
    net.precision = 'bf16'
    x = O.synth_image((3, 3, 64, 256), 106).cuda()
    with torch.no_grad():
        full = net(x)
        parts = torch.cat([net(x[i:i + 1]) for i in range(3)], 0)
    assert torch.equal(full, parts)


def test_rrdbnet_bf16_translation_property():
    """Zero-padded conv stack is shift-equivariant away from borders: cropping the input by whole tiles moves
    the interior of the output by 4x the shift (checks tile/halo addressing at non-trivial offsets)."""
    nb = 1
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 107, 0.3)
    net = build_G(nb, sd).eval()
    net.precision = 'fp32'
    x = O.synth_image((1, 3, 96, 64), 108).cuda()
    with torch.no_grad():
        a = net(x)
        b = net(x[:, :, 16:, 8:].contiguous())
    # receptive field of nb=1: 1 + 15 + 1 (LR side) + tail < 20 LR px => compare beyond 24 LR px from the cut
    m = 24
    ia = a[:, :, 4 * (16 + m):, 4 * (8 + m):]
    ib = b[:, :, 4 * m:, 4 * m:]
    assert rel_linf(ia, ib) < 1e-5


def test_rrdbnet_bf16_training_gradients_vs_oracle():
    """Mixed-precision training mode (tcgen05 fprop + dgrad, fp32-accumulated wgrad on bf16 activations): gradients
    agree with the fp32 oracle to bf16 accuracy (relative L2 error per tensor; tolerance 0.12: bf16 activation gradients through 17 convs; the wgrad kernel itself is exact)."""
    nb = 1
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 131, 0.3)
    net = build_G(nb, sd)
    net.train_precision = 'bf16'
    x = O.synth_image((2, 3, 24, 16), 132)
    pat = O.synth((2, 3, 96, 64), 133)
    out = net(x.cuda())
    (out * pat.cuda()).sum().backward()
    p = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref = O.rrdbnet_forward(x, p, nb)
    (ref * pat).sum().backward()
    assert rel_linf(out, ref) < 3e-2
    worst = 0.0
    for k, v in net.named_parameters():
        g, r = v.grad.float().cpu(), p[k].grad
        err = float((g - r).norm() / r.norm().clamp_min(1e-20))
        worst = max(worst, err)
        assert err < 0.12, (k, err)
    assert worst > 0            # bf16 path really ran (fp32 path would give ~1e-6)


# ------------------------------------------------------------------------------------------------ D
def test_nlayer_d_vs_golden(golden):
    from dasr_b200.srn.models.modules.architecture import NLayerDiscriminator
    g = golden('nlayer_d.pt')
    sd = O.synth_state_dict(O.nlayer_d_shapes(9, 64, 2), g['w_seed'], 1.0)
    net = NLayerDiscriminator(9, n_layers=2)
    net.load_state_dict(sd, strict=True)
    net.cuda()
    x = O.synth_image(g['x_shape'], g['x_seed']).cuda().requires_grad_(True)
    out = net(x)
    assert rel_linf(out, g['out']) < FP32_TOL
    (out * O.synth(tuple(out.shape), g['pat_seed']).cuda()).sum().backward()
    assert rel_linf(x.grad, g['dx']) < FP32_TOL
    named = dict(net.named_parameters())
    for k, ref in g['grads'].items():
        assert rel_linf(named[k].grad, ref) < FP32_TOL, k
    for k, n in g['grad_norms'].items():
        assert abs(float(named[k].grad.double().norm()) - n) <= 1e-3 * max(n, 1e-12), k


@pytest.mark.parametrize('n_layers,hw,math', [(2, (64, 64), 'fma'), (3, (64, 48), 'fma'), (2, (44, 36), 'tf32')])
def test_nlayer_d_one_kernel_layers_vs_oracle_and_unfused(n_layers, hw, math, monkeypatch):
    """Conv2d(4x4) -> InstanceNorm2d -> LeakyReLU as ONE kernel (dasr_conv2d_in_lrelu_f32, taken when the batch gives >= 32
    (image, 64-channel) CTAs): batch 16 against the CPU oracle of the reference module and against the two-kernel path
    (forward, input gradient, parameter gradients).  tf32: the same with tensor-core math, tolerance of tf32 operands."""
    from dasr_b200 import ops
    from dasr_b200.srn.models.modules.architecture import NLayerDiscriminator
    sd = O.synth_state_dict(O.nlayer_d_shapes(9, 64, n_layers), 121, 1.0)
    x = O.synth_image((16, 9) + hw, 122)
    ref = O.nlayer_d_forward(x[:2], sd, n_layers)
    res = {}
    for fused in ('1', '0'):
        monkeypatch.setenv('DASR_B200_FUSED_IN', fused)
        net = NLayerDiscriminator(9, n_layers=n_layers)
        net.load_state_dict(sd, strict=True)
        net.cuda()
        xg = x.cuda().requires_grad_(True)
        launches = ops._lib.LAUNCHES
        with ops.f32_math(math):
            out = net(xg)
            (out * O.synth(tuple(out.shape), 123).cuda()).sum().backward()
        res[fused] = (out.detach(), xg.grad, [p.grad for p in net.parameters()], ops._lib.LAUNCHES - launches)
    tol = FP32_TOL if math == 'fma' else 2e-2
    assert rel_linf(res['1'][0][:2], ref) < tol
    eq = 1e-5 if math == 'fma' else 2e-2
    assert rel_linf(res['1'][0], res['0'][0]) < eq
    assert rel_linf(res['1'][1], res['0'][1]) < eq * 10
    for a, b in zip(res['1'][2], res['0'][2]):
        assert rel_linf(a, b) < eq * 10
    assert res['1'][3] == res['0'][3] - n_layers          # one launch less per normalised layer


@pytest.mark.parametrize('in_nc,hw', [(3, (36, 28)), (9, (18, 22))])
def test_nlayer_d_ragged_vs_oracle(in_nc, hw):
    from dasr_b200.srn.models.modules.architecture import NLayerDiscriminator
    sd = O.synth_state_dict(O.nlayer_d_shapes(in_nc, 64, 2), 111, 1.0)
    net = NLayerDiscriminator(in_nc, n_layers=2)
    net.load_state_dict(sd, strict=True)
    net.cuda()
    x = O.synth_image((3, in_nc) + hw, 112)
    ref = O.nlayer_d_forward(x, sd, 2)
    out = net(x.cuda())
    assert out.shape == ref.shape and rel_linf(out, ref) < FP32_TOL


# ---------------------------------------------------------------------------------------------- VGG
def test_vgg19_vs_golden(golden):
    from dasr_b200.srn.models.modules.architecture import VGGFeatureExtractor
    g = golden('vgg19.pt')
    sd = O.synth_state_dict(O.vgg19_shapes(34), g['w_seed'], 1.0)
    net = VGGFeatureExtractor(feature_layer=34, weights=sd).cuda()
    x = O.synth_image(g['x_shape'], g['x_seed']).cuda().requires_grad_(True)
    out = net(x)
    assert out.shape == g['out'].shape
    assert rel_linf(out, g['out']) < FP32_TOL
    (out * O.synth(tuple(out.shape), g['pat_seed']).cuda()).sum().backward()
    assert rel_linf(x.grad, g['dx']) < FP32_TOL


def test_vgg19_bf16_tensor_core_path_vs_golden(golden):
    """Mixed-precision perceptual-loss network (tcgen05 convs, bf16 activations): features and input gradient
    against the fp32 reference within bf16 tolerances (rel-L2; 16 stacked bf16 layers)."""
    from dasr_b200.srn.models.modules.architecture import VGGFeatureExtractor
    g = golden('vgg19.pt')
    sd = O.synth_state_dict(O.vgg19_shapes(34), g['w_seed'], 1.0)
    net = VGGFeatureExtractor(feature_layer=34, weights=sd).cuda()
    net.precision = 'bf16'
    x = O.synth_image(g['x_shape'], g['x_seed']).cuda().requires_grad_(True)
    out = net(x)
    assert out.shape == g['out'].shape

    def rel_l2(a, b):
        return float((a.detach().float().cpu() - b).norm() / b.norm())
    e_f = rel_l2(out, g['out'])
    (out * O.synth(tuple(out.shape), g['pat_seed']).cuda()).sum().backward()
    e_g = rel_l2(x.grad, g['dx'])
    cos = float(torch.nn.functional.cosine_similarity(x.grad.cpu().flatten(), g['dx'].flatten(), dim=0))
    print('vgg bf16: feature rel-L2 %.3e  dx rel-L2 %.3e  cos %.4f' % (e_f, e_g, cos))
    # The input gradient of a ReLU/max-pool stack is piecewise constant: every pre-activation within bf16 rounding of
    # zero flips its mask (~0.3 % of the elements per layer -> ~4 % rel-L2 per layer, 16 layers + 4 pools in
    # quadrature ~ 0.3).  It is the exact gradient of the bf16 network; the kernels themselves are checked
    # tightly in test_conv_tc_wide_channel_tiles.
    assert e_f < 3e-2 and e_g < 0.45 and cos > 0.9


@pytest.mark.parametrize('cin,cout,h,w', [(64, 128, 20, 12), (256, 256, 9, 17), (512, 512, 8, 8), (32, 64, 16, 8)])
def test_conv_tc_wide_channel_tiles(cin, cout, h, w):
    """tcgen05 fprop / dgrad with the filters split in Cout tiles (VGG19 widths) against torch fp32 convs on the
    same bf16-rounded operands."""
    import torch.nn.functional as F
    from dasr_b200 import engine, ops
    N = 3
    x = O.synth((N, cin, h, w), 11, 1.0).bfloat16().float()
    wt = O.synth((cout, cin, 3, 3), 12, 1.0 / (3.0 * cin ** 0.5)).bfloat16().float()
    b = O.synth((cout,), 13, 0.1)
    ref = F.relu(F.conv2d(x, wt, b, padding=1))
    xd = x.permute(0, 2, 3, 1).contiguous().bfloat16().cuda()
    od = torch.empty((N, h, w, cout), dtype=torch.bfloat16, device='cuda')
    ops.conv_tc(xd, ops.pack_filter_tc(wt.cuda(), ops.TC_FPROP), b.cuda(), od, kind=ops.TC_FPROP,
                nt=engine._pick_nt_staged(cout, cin), act=ops.ACT_RELU)
    got = od.float().permute(0, 3, 1, 2).cpu()
    assert float((got - ref).abs().max() / ref.abs().max()) < 1e-2
    gy = O.synth((N, cout, h, w), 14, 1.0).bfloat16().float()
    gref = F.conv_transpose2d(gy, wt, padding=1)
    gd = gy.permute(0, 2, 3, 1).contiguous().bfloat16().cuda()
    gi = torch.empty((N, h, w, cin), dtype=torch.bfloat16, device='cuda')
    ops.conv_tc(gd, ops.pack_filter_tc(wt.cuda(), ops.TC_DGRAD), None, gi, kind=ops.TC_DGRAD,
                nt=engine._pick_nt_staged(cin, cout))
    got = gi.float().permute(0, 3, 1, 2).cpu()
    assert float((got - gref).abs().max() / gref.abs().max()) < 1e-2


@pytest.mark.parametrize('shape', [(2, 16, 24), (3, 40, 24), (1, 64, 64)])
def test_rdb_wgrad_kernel_matches_per_conv_wgrad(shape):
    """dasr_rdb_wgrad_tc (five filter gradients of a dense block, 7 (row tile, columns, taps) jobs in one launch) against
    five dasr_conv3x3_wgrad_tc launches on the same bf16 operands: same products, different fp32 summation order."""
    from dasr_b200 import ops
    N, H, W = shape
    xb = O.synth((N, H, W, 256), 21, 1.0).bfloat16().cuda()
    ga = O.synth((N, H, W, 192), 22, 1.0).bfloat16().cuda()
    gb = O.synth((N, H, W, 64), 23, 1.0).bfloat16().cuda()
    ref, got = [], []
    for k in range(1, 6):
        cin, cout = 64 + 32 * (k - 1), (32 if k < 5 else 64)
        r = torch.empty((cout, cin, 3, 3), device='cuda')
        dy = ops.View(ga, 32, 64 + 32 * (k - 1)) if k < 5 else ops.View(gb, 64, 0)
        ops.conv3x3_wgrad_tc(ops.View(xb, cin, 0), dy, r)
        ref.append(r)
        got.append(torch.full((cout, cin, 3, 3), float('nan'), device='cuda'))
    ops.rdb_wgrad_tc(xb, ga, 64, gb, 0, got)
    torch.cuda.synchronize()
    for k in range(5):
        err = float((got[k] - ref[k]).abs().max() / ref[k].abs().max())
        assert err < 1e-5, (k + 1, err)


def test_batch_packer_matches_per_filter_packs():
    """dasr_pack_filter_tc_batch (one launch, device job table) writes bit-identical kernel-layout filters to the
    per-filter path for every key the mixed-precision forward/backward asks for."""
    from dasr_b200 import engine
    nb = 1
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 5, 0.3)
    params = [v.cuda() for v in sd.values()]
    x = O.synth_image((1, 3, 16, 24), 6).cuda()
    ref = engine._PackCache()
    out, ctx = engine.rrdb_forward_bf16_train(x, params, nb, 4, ref)
    engine.rrdb_backward_bf16(ctx, params, torch.ones_like(out), ref)
    L = engine.RRDBLayout(nb, params[0].shape[0], 4)
    bp = engine._BatchPacker(params, L, L.nf)
    bp.launch()
    torch.cuda.synchronize()
    single = {k for k in ref.d if k[0] == 'w3'}          # last layer, taps in GEMM-N: packed by the single-filter kernel (4 KB)
    assert set(ref.d.keys()) - single == set(bp.cache.d.keys())
    for k, (_, t) in ref.d.items():
        if k in single:
            continue
        got = bp.cache.d[k][1]
        assert got.shape == t.shape and got.dtype == t.dtype, k
        assert torch.equal(got, t), k
    out2, ctx2 = engine.rrdb_forward_bf16_train(x, params, nb, 4, bp.cache)
    assert torch.equal(out, out2)


# ------------------------------------------------------------------------ filters / haar / losses
def test_filters_haar_bilinear_losses(golden):
    from dasr_b200 import ops
    from dasr_b200.srn.models.modules import architecture as A
    from dasr_b200.srn.models.modules import loss as L
    g = golden('misc.pt')
    x = O.synth_image(g['x_shape'], g['x_seed']).cuda()
    assert torch.allclose(A.FilterLow(kernel_size=5, gaussian=True).cuda()(x).cpu(), g['gau_low_k5'], atol=1e-6)
    assert torch.allclose(A.FilterHigh(kernel_size=5, gaussian=True).cuda()(x).cpu(), g['gau_high_k5'], atol=1e-6)
    assert torch.allclose(A.FilterLow(kernel_size=5, gaussian=False, include_pad=True).cuda()(x).cpu(), g['avg_low_k5_incl'], atol=1e-6)
    assert torch.allclose(A.FilterHigh(kernel_size=5, gaussian=False, include_pad=False).cuda()(x).cpu(), g['avg_high_k5_excl'], atol=1e-6)
    assert torch.allclose(A.FilterHigh(kernel_size=9, gaussian=True).cuda()(x).cpu(), g['gau_high_k9'], atol=1e-6)
    w = O.synth_image((2, 1, 4, 3), g['w_seed']).cuda()
    up = torch.empty((2, 1, 16, 12), device='cuda')
    ops.bilinear(w, up)
    assert torch.allclose(up.cpu(), g['bilinear_x4'], atol=1e-6)
    p = O.synth((2, 1, 6, 6), g['p_seed'], 3.0).cuda()
    for t in ('vanilla', 'lsgan', 'wgan-gp'):
        crit = L.GANLoss(t)
        assert abs(float(crit(p, True)) - float(g['gan_%s_real' % t])) < 1e-5
        assert abs(float(crit(p, False)) - float(g['gan_%s_fake' % t])) < 1e-5
    # haar split (+norm) against the oracle restatement, forward and backward
    xr = x.clone().requires_grad_(True)
    ll, hc = L.haar_split(xr, True)
    rll, rhc = O.wavelet_s(x.cpu(), True)
    assert torch.allclose(ll.cpu(), rll, atol=1e-6) and torch.allclose(hc.cpu(), rhc, atol=1e-6)
    pa, pb = O.synth(tuple(ll.shape), 7).cuda(), O.synth(tuple(hc.shape), 8).cuda()
    ((ll * pa).sum() + (hc * pb).sum()).backward()
    xc = x.cpu().clone().requires_grad_(True)
    cl, ch = O.wavelet_s(xc, True)
    ((cl * pa.cpu()).sum() + (ch * pb.cpu()).sum()).backward()
    assert torch.allclose(xr.grad.cpu(), xc.grad, atol=1e-6)
    # filter backward (gaussian high-pass and box filter without pad counting)
    for kw in (dict(kernel_size=5, gaussian=True), dict(kernel_size=5, gaussian=False, include_pad=False)):
        xr = x.clone().requires_grad_(True)
        y = A.FilterHigh(**kw).cuda()(xr)
        pat = O.synth(tuple(y.shape), 9)
        (y * pat.cuda()).sum().backward()
        xc = x.cpu().clone().requires_grad_(True)
        (O.filter_high(xc, 5, kw['gaussian'], kw.get('include_pad', True)) * pat).sum().backward()
        assert torch.allclose(xr.grad.cpu(), xc.grad, atol=1e-6)


def test_weighted_l1_and_l1_grad():
    from dasr_b200.srn.models.modules import loss as L
    a = O.synth_image((2, 3, 12, 8), 121)
    b = O.synth_image((2, 3, 12, 8), 122)
    w = O.synth_image((2, 1, 12, 8), 123)
    ac = a.clone().requires_grad_(True)
    ref = torch.mean(w * torch.abs(ac - b))
    ref.backward()
    ag = a.cuda().requires_grad_(True)
    out = L.weighted_l1(ag, b.cuda(), w.cuda())
    (out * 3.0).backward()
    assert abs(float(out) - float(ref)) < 1e-6
    assert torch.allclose(ag.grad.cpu(), 3.0 * ac.grad, atol=1e-7)


# ------------------------------------------------------------------------------ full model, API level
from helpers import make_opt, unwrap  # noqa: E402


@pytest.mark.parametrize('name', ['dasr_step_wavelet.pt', 'dasr_step_gau.pt', 'dasr_step_ragan.pt'])
def test_dasr_model_train_steps_vs_golden(golden, name):
    """create_model -> feed_data -> optimize_parameters x2 through the public API, against the log values
    and post-step weights the reference produced for the same inputs (oracle/gen_golden.py)."""
    from dasr_b200.srn.models import create_model
    from helpers import load_train_steps
    g = load_train_steps(golden, name)
    fs = g['fs']
    opt = make_opt(True, 'DASR', g['nb'], fs)
    opt['train']['ragan'] = bool(g.get('ragan', False))        # dasr_step_ragan.pt: relativistic average GAN terms
    model = create_model(opt)
    unwrap(model.netG).load_state_dict(O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['wG_seed'], g['gain_G']))
    unwrap(model.netD_target).load_state_dict(O.synth_state_dict(O.nlayer_d_shapes(9 if fs == 'wavelet' else 3, 64, 2), g['wD_seed'], 1.0))
    unwrap(model.netF).load_state_dict(O.synth_state_dict(O.vgg19_shapes(34), g['wF_seed'], 1.0), strict=False)
    B, h, w = g['B'], g['h'], g['w']
    for step, (seed, ref) in enumerate(zip(g['data_seeds'], g['steps']), 1):
        data = {'LR_real': O.synth_image((B, 3, h, w), seed), 'LR_fake': O.synth_image((B, 3, h, w), seed + 1),
                'HR': O.synth_image((B, 3, 4 * h, 4 * w), seed + 2), 'HR_unpair': O.synth_image((B, 3, 4 * h, 4 * w), seed + 3),
                'fake_w': O.synth_image((B, 1, h, w), seed + 4)}
        model.feed_data(data, True)
        model.optimize_parameters(step)
        log = model.get_current_log()
        assert list(log.keys()) == list(ref['log'].keys())
        for k in log:
            assert abs(log[k] - ref['log'][k]) <= 1e-3 * max(1.0, abs(ref['log'][k])), (k, log[k], ref['log'][k])
        assert rel_linf(model.fake_H, ref['fake_H']) < FP32_TOL
        G, D = unwrap(model.netG).state_dict(), unwrap(model.netD_target).state_dict()
        for k, v in ref['G_keep'].items():
            assert rel_linf(G[k], v) < FP32_TOL, k
        # relativistic losses only see score DIFFERENCES: the gradient of D's last bias is mathematically zero, what
        # backward leaves there is rounding noise and Adam turns noise into a +-lr step -> not comparable
        skip = {'model.8.bias'} if g.get('ragan') else set()
        for k, v in ref['D_keep'].items():
            if k not in skip:
                assert rel_linf(D[k], v) < FP32_TOL, k
        for k, n in ref['G_norms'].items():
            assert abs(float(G[k].double().norm()) - n) <= 1e-4 * max(n, 1e-9), k
        for k, n in ref['D_norms'].items():
            if k not in skip:
                assert abs(float(D[k].double().norm()) - n) <= 1e-4 * max(n, 1e-9), k


def test_sr_model_test_path_vs_golden(golden):
    from dasr_b200.srn.models import create_model
    from dasr_b200.srn.utils import util
    g = golden('sr_test.pt')
    for prec, tol in (('fp32', FP32_TOL), ('bf16', 3e-2)):
        model = create_model(make_opt(False, 'sr', g['nb']))
        unwrap(model.netG).load_state_dict(O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['w_seed'], g['gain']))
        unwrap(model.netG).precision = prec
        model.feed_data({'LR': O.synth_image(g['lr_shape'], g['lr_seed']), 'HR': O.synth_image((1, 3, 40, 56), g['hr_seed'])})
        model.test()
        vis = model.get_current_visuals(need_HR=True)
        assert rel_linf(vis['SR'], g['SR']) < tol
        img = util.tensor2img(vis['SR'] * 8.0 + 0.5)
        hr = util.tensor2img(vis['HR'])
        if prec == 'fp32':
            assert np.abs(img.astype(int) - g['sr_img'].numpy().astype(int)).max() <= 1
            assert abs(util.calculate_psnr(img, hr) - g['psnr']) < 1e-3        # 3 decimals
            assert abs(util.calculate_ssim(img, hr) - g['ssim']) < 1e-3
        else:
            assert abs(util.calculate_psnr(img, hr) - g['psnr']) < 0.05


def test_ops_refuse_cpu_tensors():
    from dasr_b200._lib import DasrError
    from dasr_b200.srn.models.modules.architecture import RRDBNet
    net = RRDBNet(3, 3, 64, 1)
    with pytest.raises(DasrError):
        net(torch.rand(1, 3, 8, 8))


@pytest.mark.parametrize('min_size', [160000, 300])
def test_forward_chop_matches_stitched_oracle_quadrants(min_size):
    """utils/util.py:87-147 forward_chop (4 overlapping quadrants, `shave` px, recursive above min_size) with the quadrants
    batched into one device forward: equals the stitching of the oracle's per-quadrant forwards."""
    from dasr_b200.srn.utils.util import forward_chop
    nb, scale, shave = 1, 4, 6
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 141, 0.3)
    net = build_G(nb, sd).eval()
    net.precision = 'fp32'
    x = O.synth_image((1, 3, 44, 36), 142)

    def ref_chop(img):
        h, w = img.shape[-2:]
        tb = (slice(0, h // 2 + shave), slice(h - h // 2 - shave, h))
        lr = (slice(0, w // 2 + shave), slice(w - w // 2 - shave, w))
        parts = [img[..., a, b] for a in tb for b in lr]
        outs = [O.rrdbnet_forward(c, sd, nb) if h * w < 4 * min_size else ref_chop(c) for c in parts]
        H, W = scale * h, scale * w
        y = torch.empty((img.shape[0], 3, H, W))
        y[..., :H // 2, :W // 2] = outs[0][..., :H // 2, :W // 2]
        y[..., :H // 2, W - W // 2:] = outs[1][..., :H // 2, W // 2 - W:]
        y[..., H - H // 2:, :W // 2] = outs[2][..., H // 2 - H:, :W // 2]
        y[..., H - H // 2:, W - W // 2:] = outs[3][..., H // 2 - H:, W // 2 - W:]
        return y
    with torch.no_grad():
        got = forward_chop(x.cuda(), scale, net, shave=shave, min_size=min_size)
        ref = ref_chop(x)
    assert got.shape == ref.shape == (1, 3, 176, 144)
    assert rel_linf(got, ref) < FP32_TOL


def test_sr_model_test_x8_self_ensemble_vs_oracle():
    """SRModel.test_x8 (SR_model.py:102-140): mean over the 8 dihedral views, each mapped back."""
    from dasr_b200.srn.models import create_model
    nb = 1
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 151, 0.3)
    model = create_model(make_opt(False, 'sr', nb))
    unwrap(model.netG).load_state_dict(sd)
    unwrap(model.netG).precision = 'fp32'
    x = O.synth_image((1, 3, 12, 20), 152)
    model.feed_data({'LR': x})
    model.test_x8()
    outs = []
    for t in (False, True):
        for hf in (False, True):
            for vf in (False, True):
                v = x
                if vf:
                    v = v.flip(3)
                if hf:
                    v = v.flip(2)
                if t:
                    v = v.transpose(2, 3)
                o = O.rrdbnet_forward(v.contiguous(), sd, nb)
                if t:
                    o = o.transpose(2, 3)
                if hf:
                    o = o.flip(2)
                if vf:
                    o = o.flip(3)
                outs.append(o)
    ref = torch.stack(outs, 0).mean(0)
    assert rel_linf(model.fake_H, ref) < FP32_TOL


@pytest.mark.parametrize('sched', ['2', '3', '4'])
def test_dense_block_schedules_agree_with_one_launch_per_conv(sched, monkeypatch):
    """Every dense-block schedule (which launch computes which (conv, input chunk) product, partial sums in HBM) gives the
    per-layer result up to bf16 rounding of the partial sums; ragged tiles, odd tile count, three RRDBs."""
    from dasr_b200.srn.models.modules.architecture import RRDBNet
    monkeypatch.setenv('DASR_B200_SCHED', sched)
    monkeypatch.setenv('DASR_B200_GRAPH', '0')
    nb = 3
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 131, 0.3)
    net = RRDBNet(3, 3, 64, nb, gc=32, upscale=4)
    net.load_state_dict(sd, strict=True)
    net.cuda().eval()
    x = O.synth_image((3, 3, 40, 44), 132).cuda()
    with torch.no_grad():
        net.precision = 'bf16_layer'
        ref = net(x)
        net.precision = 'bf16'
        out = net(x)
        net.precision = 'fp32'
        exact = net(x)
    assert rel_linf(out, ref) < 1e-2, rel_linf(out, ref)
    assert rel_linf(out, exact) < 3e-2


def test_fused_mask_backward_matches_separate_mask_kernels(monkeypatch):
    """DASR_B200_FUSE_MASK=1: the LeakyReLU backward of x1..x4 runs inside the dgrad epilogues of the CTA-pair kernel (the
    activation gates the channels each launch completes) instead of in act_bwd kernels: same gradients up to one bf16
    rounding (measured 4e-3 rel-L2)."""
    from dasr_b200 import engine
    nb = 2
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 5, 0.3)
    params = [v.cuda() for v in sd.values()]
    x = O.synth_image((3, 3, 32, 24), 6).cuda()
    dout = O.synth((3, 3, 128, 96), 7).cuda()
    res = {}
    for mode in ('0', '1'):
        monkeypatch.setenv('DASR_B200_FUSE_MASK', mode)
        out, ctx = engine.rrdb_forward_bf16_train(x, params, nb, 4, engine._PackCache())
        _, grads, _ = engine.rrdb_backward_bf16(ctx, params, dout, engine._PackCache())
        torch.cuda.synchronize()
        res[mode] = [g.clone() for g in grads]
    for a, b in zip(res['0'], res['1']):
        assert float((a.double() - b.double()).norm() / a.double().norm().clamp_min(1e-30)) < 2e-2
