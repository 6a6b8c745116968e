"""GPU parity at the BASELINE shapes (VERDICT r1 "weak #1/#2", SURVEY §8 row g1).

  * configs[0] ("PR1 ref"): RRDBNet-23, kaiming x0.1-like gain, 1x3x256x256, fp32 kernels against the CPU oracle:
    rel-Linf <= 1e-3 (north_star), 8-bit images equal, PSNR/SSIM to 3 decimals.
  * configs[1]: 16x3x256x256 through the benchmarked bf16 tcgen05 dense-block schedule against the fp32 kernels on
    the same weights: rel-Linf reported + bounded, 8-bit image difference and PSNR/SSIM deltas reported + bounded;
    the same launches with IEEE half operands (precision 'fp16'): PSNR/SSIM to 3 decimals.
  * mixed-precision DASR_Model train steps against the reference's own two-step fixture with stated tolerances.

"rel-Linf" = max|a-b| / max|b| (SURVEY H2).  The raw output of a x0.1-initialised net spans only +-3e-4, so images
are formed with one affine map (taken from the fp32 result) that spreads the output over [0.05, 0.95]; the HR image is
the fp32 SR image plus +-12/255 deterministic noise (PSNR ~ 31 dB, the regime of real SR results).
"""
import numpy as np
import pytest
import torch

from oracle import srn_oracle as O

pytestmark = pytest.mark.gpu


def rel_linf(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))


def build_G(nb, sd):
    from dasr_b200.srn.models.modules.architecture import RRDBNet
    net = RRDBNet(3, 3, 64, nb, gc=32, upscale=4)
    net.load_state_dict(sd, strict=True)
    return net.cuda().eval()


def _affine(ref):
    lo, hi = float(ref.min()), float(ref.max())
    s = 0.9 / max(hi - lo, 1e-30)
    return s, 0.05 - lo * s


def _images(out, s, t):
    from dasr_b200.srn.utils import util
    return [util.tensor2img((out[i].float().cpu() * s + t)) for i in range(out.shape[0])]


def _hr_from(img, seed):
    noise = (O.synth(img.shape, seed, 12.0).numpy()).round()
    return np.clip(img.astype(np.float64) + noise, 0, 255).astype(np.uint8)


def _psnr_ssim(img, hr):
    from dasr_b200.srn.utils import util
    b = 4                                                # test.py crops `scale` border pixels (test.py:86-92)
    a, h = img[b:-b, b:-b], hr[b:-b, b:-b]
    return util.calculate_psnr(a, h), util.calculate_ssim(a, h)


def test_config0_fp32_nb23_256_vs_oracle():
    """BASELINE configs[0]: one 256x256 LR image, RRDBNet-23, gain 0.1, fp32 kernels vs the CPU oracle (~10 s of CPU)."""
    nb = 23
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 201, 0.1)
    net = build_G(nb, sd)
    net.precision = 'fp32'
    x = O.synth_image((1, 3, 256, 256), 202)
    with torch.no_grad():
        out = net(x.cuda()).cpu()
        ref = O.rrdbnet_forward(x, sd, nb)
    e = rel_linf(out, ref)
    s, t = _affine(ref)
    img, rimg = _images(out, s, t)[0], _images(ref, s, t)[0]
    hr = _hr_from(rimg, 203)
    p, q = _psnr_ssim(img, hr)
    rp, rq = _psnr_ssim(rimg, hr)
    ndiff = int((img != rimg).sum())
    print('config0 fp32 nb23 256x256: rel-Linf %.3e | 8-bit pixels differing %d of %d | PSNR %.6f vs %.6f | SSIM %.6f vs %.6f'
          % (e, ndiff, img.size, p, rp, q, rq))
    assert out.shape == (1, 3, 1024, 1024)
    assert e < 1e-3
    assert np.abs(img.astype(int) - rimg.astype(int)).max() <= 1
    assert abs(p - rp) < 5e-4 and abs(q - rq) < 5e-4          # 3 decimals


def test_config1_bf16_nb23_16x256_vs_fp32_kernels():
    """BASELINE configs[1] (the benchmarked path): 16x3x256x256, bf16 tcgen05 dense-block schedule, against the fp32
    kernels (themselves pinned to the oracle at this size by the test above).  bf16 operands cannot meet 1e-3 rel-Linf
    (SURVEY H2: operand rounding alone is 8.8e-3 at nb=23): the numbers are reported and bounded at ~2x what is measured."""
    nb = 23
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=nb), 201, 0.1)
    net = build_G(nb, sd)
    x = O.synth_image((16, 3, 256, 256), 204).cuda()
    with torch.no_grad():
        net.precision = 'fp32'
        ref = torch.cat([net(x[i:i + 4]).cpu() for i in range(0, 16, 4)], 0)
        res = {}
        for prec in ('bf16', 'bf16_layer', 'fp16'):
            net.precision = prec
            res[prec] = net(x).cpu()
    s, t = _affine(ref)
    rimgs = _images(ref, s, t)
    for prec, out in res.items():
        e = rel_linf(out, ref)
        rms = float((out - ref).pow(2).mean().sqrt() / ref.abs().max())
        imgs = _images(out, s, t)
        dp, dq, nd, mx = 0.0, 0.0, 0, 0
        for i in (0, 7, 15):
            hr = _hr_from(rimgs[i], 300 + i)
            p, q = _psnr_ssim(imgs[i], hr)
            rp, rq = _psnr_ssim(rimgs[i], hr)
            dp, dq = max(dp, abs(p - rp)), max(dq, abs(q - rq))
            nd += int((imgs[i] != rimgs[i]).sum())
            mx = max(mx, int(np.abs(imgs[i].astype(int) - rimgs[i].astype(int)).max()))
        print('config1 %s nb23 16x256x256 vs fp32 kernels: rel-Linf %.3e rel-rms %.3e | 8-bit: %d of %d differ, max %d LSB | '
              '|dPSNR| %.5f dB |dSSIM| %.6f (PSNR ~31 dB)' % (prec, e, rms, nd, 3 * imgs[0].size, mx, dp, dq))
        res[prec] = (e, rms, mx, dp, dq)
    # measured on B200 (round 2): rel-Linf 6.8e-4, rel-rms 1.1e-4, 2.7 % of the 8-bit pixels differ by 1 LSB,
    # |dPSNR| 0.0024 dB, |dSSIM| 0.0002 at PSNR ~31 dB — i.e. PSNR/SSIM agree to 2 decimals, not to the 3 the north star
    # asks of the tensor-core path (the fp32 kernels above do).  Bounds = ~2x the measurement.
    for prec in ('bf16', 'bf16_layer'):
        e, rms, mx, dp, dq = res[prec]
        assert e < 2e-3 and rms < 3e-4, prec
        assert mx <= 1, prec
        assert dp < 6e-3 and dq < 6e-4, prec
    # IEEE half operands on the same kernels (precision 'fp16'): 3 more significand bits.  Measured on B200: rel-Linf 9.6e-5,
    # rel-rms 2.3e-5, 0.55 % of the 8-bit values differ by 1 LSB, |dPSNR| 0.0005 dB, |dSSIM| 0.00005 at PSNR ~31 dB —
    # SSIM equal to 4 decimals, PSNR equal to 3 decimals up to a half-unit in the third (5x closer than bf16).
    e, rms, mx, dp, dq = res['fp16']
    assert e < 2e-4 and rms < 5e-5
    assert mx <= 1
    assert dp < 1e-3 and dq < 1e-4


def test_mixed_precision_dasr_steps_vs_reference_fixture(golden, monkeypatch):
    """DASR_Model in the mixed-precision training mode (tcgen05 G fprop/dgrad/wgrad, tcgen05 VGG19; fp32 D, losses, Adam)
    against the two optimisation steps the REFERENCE produced (tests/golden/dasr_step_wavelet.pt).
    Tolerances (bf16 activations, fp32 accumulation): losses 2e-3 relative (measured ~1e-4..1e-3), SR output 3e-2 rel-Linf,
    post-Adam weights: Adam moves every weight by ~lr regardless of the gradient magnitude, so the kept slices are
    compared through the UPDATE direction (cosine > 0.8: signs of near-zero gradients flip under bf16)."""
    monkeypatch.setenv('DASR_B200_TRAIN_PRECISION', 'bf16')
    from dasr_b200.srn.models import create_model
    from helpers import load_train_steps, make_opt, unwrap
    g = load_train_steps(golden, 'dasr_step_wavelet.pt')
    model = create_model(make_opt(True, 'DASR', g['nb'], g['fs']))
    sdG = O.synth_state_dict(O.rrdbnet_shapes(nb=g['nb']), g['wG_seed'], g['gain_G'])
    sdD = O.synth_state_dict(O.nlayer_d_shapes(9, 64, 2), g['wD_seed'], 1.0)
    unwrap(model.netG).load_state_dict(sdG)
    unwrap(model.netD_target).load_state_dict(sdD)
    unwrap(model.netF).load_state_dict(O.synth_state_dict(O.vgg19_shapes(34), g['wF_seed'], 1.0), strict=False)
    B, h, w = g['B'], g['h'], g['w']
    worst = {}
    for step, (seed, ref) in enumerate(zip(g['data_seeds'], g['steps']), 1):
        data = {'LR_real': O.synth_image((B, 3, h, w), seed), 'LR_fake': O.synth_image((B, 3, h, w), seed + 1),
                'HR': O.synth_image((B, 3, 4 * h, 4 * w), seed + 2), 'HR_unpair': O.synth_image((B, 3, 4 * h, 4 * w), seed + 3),
                'fake_w': O.synth_image((B, 1, h, w), seed + 4)}
        model.feed_data(data, True)
        model.optimize_parameters(step)
        log = model.get_current_log()
        assert list(log.keys()) == list(ref['log'].keys())
        for k in log:
            err = abs(log[k] - ref['log'][k]) / max(1e-3, abs(ref['log'][k]))
            worst[k] = max(worst.get(k, 0.0), err)
        e_out = rel_linf(model.fake_H, ref['fake_H'])
        worst['fake_H'] = max(worst.get('fake_H', 0.0), e_out)
        G = unwrap(model.netG).state_dict()
        if step == 1:
            cs = []
            for k, v in ref['G_keep'].items():
                w0 = sdG[k]
                du, dr = (G[k].cpu() - w0).flatten(), (v - w0).flatten()
                if float(dr.norm()) > 0:
                    cs.append(float(torch.nn.functional.cosine_similarity(du, dr, dim=0)))
            worst['update_cos_min'] = min(cs)
        for k, n in ref['G_norms'].items():
            assert abs(float(G[k].double().norm()) - n) <= 1e-3 * max(n, 1e-9), k
    print('mixed-precision DASR steps vs reference fixture: ' + ', '.join('%s %.3e' % kv for kv in worst.items()))
    for k, v in worst.items():
        if k == 'update_cos_min':
            assert v > 0.8, (k, v)
        elif k == 'fake_H':
            assert v < 3e-2, (k, v)
        elif k.startswith('disc_Score'):
            assert v < 2e-2, (k, v)
        elif k == 'loss/l_g_fea':
            assert v < 1.5e-2, (k, v)        # L1 of bf16 VGG19 features: 4.5e-3 .. 6.2e-3 measured across builds (summation order)
        else:
            assert v < 5e-3, (k, v)
