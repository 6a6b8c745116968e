"""Host-side logic (CPU): option parsing, model construction / state_dict contract, b_split, metrics,
and the data-parallel gradient bucket over gloo with world_size 2."""
import json
import os
import shlex
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import srn_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_options_parse_roundtrip(tmp_path):
    from dasr_b200.srn.options import options as option
    cfg = {
        "name": "debug_x", "model": "sr", "scale": 4, "gpu_ids": [], "chop": False,
        "datasets": {"test_1": {"name": "a", "mode": "LRHR", "dataroot_HR": "~/hr", "dataroot_LR": "~/lr.lmdb"}},
        "path": {"root": str(tmp_path), "pretrain_model_G": None},
        "network_G": {"which_model_G": "RRDB_net", "nf": 64, "nb": 23, "in_nc": 3, "out_nc": 3, "gc": 32},
    }
    p = tmp_path / 'o.json'
    p.write_text('// comment line\n' + json.dumps(cfg, indent=1).replace('"scale": 4,', '"scale": 4, // x4'))
    opt = option.parse(str(p), is_train=False)
    assert opt['is_train'] is False and opt['network_G']['scale'] == 4
    assert opt['datasets']['test_1']['phase'] == 'test' and opt['datasets']['test_1']['data_type'] == 'lmdb'
    assert opt['path']['results_root'].endswith(os.path.join('results', 'debug_x'))
    nd = option.dict_to_nonedict(opt)
    assert nd['nonexistent'] is None and nd['network_G']['norm_type'] is None
    assert 'which_model_G' in option.dict2str(nd)


def test_shipped_json_files_parse():
    """The reference's own option files parse unchanged (they are read from tests/data copies of the two
    files the north star names; paths inside are never touched at parse time)."""
    from dasr_b200.srn.options import options as option
    for name, train in (('test_sr.json', False), ('train_DASR_auto_reproduce_realsr.json', True)):
        opt = option.dict_to_nonedict(option.parse(os.path.join(ROOT, 'tests', 'data', name), is_train=train))
        assert opt['network_G']['which_model_G'] == 'RRDB_net' and opt['network_G']['nb'] == 23
        assert opt['scale'] == 4


def test_create_model_state_dict_contract_and_cpu_refusal():
    from dasr_b200._lib import DasrError
    from dasr_b200.srn.models import create_model
    from tests.test_gpu_parity import make_opt
    with pytest.warns(UserWarning):
        model = create_model(make_opt(True, 'DASR_FS_ESRGAN_patchGAN', nb=2, gpu=False))   # alias the shipped JSONs use
    assert list(model.netG.state_dict().keys()) == list(O.rrdbnet_shapes(nb=2).keys())
    assert list(model.netD_target.state_dict().keys()) == list(O.nlayer_d_shapes(9, 64, 2).keys())
    assert len(model.optimizers) == 2 and len(model.schedulers) == 2
    # G: kaiming * 0.1, zero bias (networks.py:30-44,142-143)
    w = model.netG.state_dict()['model.1.sub.0.RDB1.conv1.0.weight']
    assert abs(float(w.std()) - 0.1 * (2.0 / (64 * 9)) ** 0.5) < 0.2 * 0.1 * (2.0 / (64 * 9)) ** 0.5
    assert float(model.netG.state_dict()['model.0.bias'].abs().max()) == 0.0
    data = {k: torch.rand(1, 3, 8, 8) for k in ('LR_real', 'LR_fake')}
    data.update(HR=torch.rand(1, 3, 32, 32), HR_unpair=torch.rand(1, 3, 32, 32), fake_w=torch.rand(1, 1, 8, 8))
    with pytest.raises(DasrError):          # no CPU fallback: the product path refuses to run without CUDA
        model.feed_data(data, True)
        model.optimize_parameters(1)
    with pytest.raises(NotImplementedError):
        create_model(make_opt(True, 'De_Resnet', gpu=False))      # dead duplicate of codes/DSN in the reference (SURVEY §2)


def test_save_load_checkpoint_roundtrip(tmp_path):
    from dasr_b200.srn.models import create_model
    from tests.test_gpu_parity import make_opt
    opt = make_opt(True, 'DASR', nb=1, gpu=False)
    opt['path']['models'] = str(tmp_path)
    opt['path']['training_state'] = str(tmp_path)
    with pytest.warns(UserWarning):
        m = create_model(opt)
    m.save(7)
    m.save_training_state(1, 7)
    assert sorted(os.listdir(tmp_path)) == ['7.state', '7_D_target.pth', '7_G.pth']
    sd = torch.load(tmp_path / '7_G.pth')
    assert list(sd.keys()) == list(O.rrdbnet_shapes(nb=1).keys()) and sd['model.0.weight'].dtype == torch.float32
    opt['path']['pretrain_model_G'] = str(tmp_path / '7_G.pth')
    with pytest.warns(UserWarning):
        m2 = create_model(opt)
    assert torch.equal(m2.netG.state_dict()['model.3.weight'], sd['model.3.weight'])
    m2.resume_training(torch.load(tmp_path / '7.state'))


def test_b_split_and_metrics(golden):
    from dasr_b200.srn.utils import util
    g = golden('misc.pt')
    x = O.synth_image(g['x_shape'], g['x_seed'])
    fa, re = util.b_split(x.repeat(2, 1, 1, 1), [0, 0, 1, 1])
    assert torch.equal(fa, g['b_split_fake']) and torch.equal(re, g['b_split_real'])
    fa2, re2 = util.b_split(x.repeat(2, 1, 1, 1), [0, 1, 0, 1])
    assert torch.equal(fa2, x.repeat(2, 1, 1, 1)[[0, 2]]) and torch.equal(re2, x.repeat(2, 1, 1, 1)[[1, 3]])
    img = util.tensor2img(x[0] * 1.2 - 0.1)
    assert np.array_equal(img, g['tensor2img'].numpy())
    assert abs(util.calculate_psnr(img, util.tensor2img(x[1].clone())) - g['psnr']) < 1e-9
    big = O.synth_image((2, 3, 24, 24), g['ssim_seed'])
    i1, i2 = util.tensor2img(big[0].clone()), util.tensor2img(big[0] * 0.9 + 0.1 * big[1])
    assert abs(util.calculate_ssim(i1, i2) - g['ssim']) < 1e-9


DP_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from dasr_b200.dp import GradBucket
dist.init_process_group('gloo', init_method='tcp://127.0.0.1:%%s' %% sys.argv[2], rank=int(sys.argv[1]), world_size=2)
rank = dist.get_rank()
os.environ['DASR_B200_DP_OVERLAP'] = sys.argv[3]
torch.manual_seed(100 + rank)                       # every process draws its OWN initial weights (train.py, manual_seed null)


class ArenaNet(torch.nn.Module):
    # stands in for RRDBNet in mixed precision: its backward writes ONE flat gradient tensor in its own layout
    # ([weights | biases], not parameter order) into the bucket segment it was handed
    def __init__(self):
        super().__init__()
        self.a = torch.nn.Linear(5, 7)
        self.b = torch.nn.Linear(7, 3)
        self.arena = None

    def set_grad_arena(self, flat):
        self.arena = flat

    def forward(self, x):
        return self.b(self.a(x))

    def flat_backward(self, loss):
        ps = list(self.parameters())
        gs = torch.autograd.grad(loss, ps)
        order = [0, 2, 1, 3]                         # weights first, then biases
        o = 0
        for i in order:
            v = self.arena[o:o + ps[i].numel()].view_as(ps[i])
            v.copy_(gs[i])
            ps[i].grad = v
            o += ps[i].numel()


G, D = ArenaNet(), torch.nn.Sequential(torch.nn.Linear(4, 6), torch.nn.Linear(6, 1))
bucket = GradBucket([G, D])
assert bucket.active and bucket.numel() == sum(p.numel() for n in (G, D) for p in n.parameters())
# rank 0's weights were broadcast at construction
for p in list(G.parameters()) + list(D.parameters()):
    t = [torch.zeros_like(p), torch.zeros_like(p)]
    dist.all_gather(t, p.data)
    assert torch.equal(t[0], t[1]), 'replicas differ after construction'
assert G.arena is not None and G.arena.data_ptr() == bucket.flat.data_ptr()


def data(r):
    return torch.arange(10, dtype=torch.float32).reshape(2, 5) * (r + 1), torch.arange(8, dtype=torch.float32).reshape(2, 4) - r


def local_grads(r):
    xg, xd = data(r)
    gg = torch.autograd.grad(G(xg).sum(), list(G.parameters()))
    gd = torch.autograd.grad(D(xd).square().sum(), list(D.parameters()))
    return [g.clone() for g in gg], [g.clone() for g in gd]


ref = [local_grads(r) for r in range(2)]
for step in range(2):                               # two steps: views / arena are persistent, .grad is reset in between
    for p in list(G.parameters()) + list(D.parameters()):
        p.grad = None
    xg, xd = data(rank)
    G.flat_backward(G(xg).sum())
    bucket.reduce_segment(0)                        # starts G's exchange (no-op with overlap off)
    D(xd).square().sum().backward()
    bucket.finish()
    assert bucket.last_copies == len(list(D.parameters())), bucket.last_copies     # only D's tensors are gathered by copy
    lo, hi = bucket.flat.data_ptr(), bucket.flat.data_ptr() + 4 * bucket.numel()
    for net, k in ((G, 0), (D, 1)):
        for i, p in enumerate(net.parameters()):
            assert lo <= p.grad.data_ptr() < hi
            want = (ref[0][k][i] + ref[1][k][i]) / 2
            assert torch.allclose(p.grad, want, atol=1e-5), (step, k, i)
print('rank', rank, 'ok')
'''


def test_grad_bucket_allreduce_gloo_world2(tmp_path):
    script = tmp_path / 'w.py'
    script.write_text(DP_WORKER % ROOT)
    for k, overlap in enumerate(('1', '0')):          # overlapped per-network exchange / one all-reduce of the whole bucket
        port = str(29500 + (os.getpid() + k) % 2000)
        procs = [subprocess.Popen([sys.executable, str(script), str(r), port, overlap], stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
                 for r in range(2)]
        outs = [p.communicate(timeout=180)[0].decode() for p in procs]
        assert all(p.returncode == 0 for p in procs), outs
        assert all('ok' in o for o in outs)


def test_dsn_modules_match_reference_state_dict_layout():
    """De_resnet / Discriminator(FSD) expose the reference's state_dict keys and shapes (DSN/model.py), and a CPU
    tensor is refused loudly (no CPU fallback on the product path)."""
    import pytest
    import torch
    from oracle import dsn_oracle as D
    from dasr_b200._lib import DasrError
    from dasr_b200.dsn.model import De_resnet, Discriminator
    net = De_resnet(n_res_blocks=8, scale=4)
    shapes = D.de_resnet_shapes(8, 4)
    assert [(k, tuple(v.shape)) for k, v in net.state_dict().items()] == list(shapes.items())
    d = Discriminator(kernel_size=5, D_arch='FSD', norm_layer='Instance', filter_type='wavelet', cs='cat')
    assert [(k, tuple(v.shape)) for k, v in d.state_dict().items()] == list(D.fsd_shapes(9).items())
    with pytest.raises(DasrError):
        net(torch.zeros(1, 3, 16, 16))


def _write_tree(base, files):
    for rel, text in files.items():
        p = base / rel
        p.parent.mkdir(parents=True, exist_ok=True)
        p.write_text(text)


# A stand-in for a DASR `codes` checkout: the directory layout and the top-level module names its entry scripts import.
# Every module the dasr_b200 mirrors replace fails on import here, so a script that gets the checkout's own copy stops.
def _decoy(name):
    return 'raise ImportError("the checkout\'s own %s was imported instead of the dasr_b200 mirror")\n' % name


SRN_DECOYS = {name: _decoy(name) for name in ('models/__init__.py', 'options/__init__.py', 'options/options.py',
                                              'utils/__init__.py', 'utils/util.py')}
DSN_DECOYS = {name: _decoy(name) for name in ('model.py', 'loss.py')}

# SRN inference entry point: option file -> logger -> dataset -> create_model -> feed_data / test, like codes/SRN/test.py.
SRN_TEST_SCRIPT = r'''
import argparse
import logging

import options.options as option
import utils.util as util
from data import create_dataset
from models import create_model
from utils.receptive_cal import WINDOW      # a module only the checkout has: found through the mirror package's search path

ap = argparse.ArgumentParser()
ap.add_argument('-opt', required=True)
opt = option.dict_to_nonedict(option.parse(ap.parse_args().opt, is_train=False))
util.mkdirs([opt['path']['results_root'], opt['path']['log']])
util.setup_logger(None, opt['path']['log'], 'test.log', level=logging.INFO, screen=True)
model = create_model(opt)
for batch in create_dataset(opt['datasets']['test_1']):
    model.feed_data(batch, False)
    model.test()
'''
SRN_DATA_PACKAGE = r'''
import torch


def create_dataset(opt):
    return [{'LR': torch.rand(1, 3, 16, 16), 'LR_path': ['a.png']}]
'''


def test_reference_test_py_runs_unchanged_through_the_launcher(tmp_path):
    """Drop-in boundary: an SRN test script, executed unchanged by dasr_b200.launch from a checkout whose own `models`,
    `options` and `utils` packages sit next to it, parses its JSON, builds its dataset with the checkout's data/ package,
    creates the model through the mirror and reaches the first kernel call — which must refuse loudly on a host without
    a GPU (no CPU fallback)."""
    import json
    srn = tmp_path / 'codes' / 'SRN'
    _write_tree(srn, dict(SRN_DECOYS, **{'test.py': SRN_TEST_SCRIPT, 'data/__init__.py': SRN_DATA_PACKAGE,
                                          'utils/receptive_cal.py': 'WINDOW = 1\n'}))
    opt = {'name': 'dropin_test', 'suffix': None, 'model': 'sr', 'scale': 4, 'gpu_ids': None, 'chop': False, 'val_lpips': False,
           'save_RealorFake': False,
           'datasets': {'test_1': {'name': 'toy', 'mode': 'LRHR', 'dataroot_HR': str(tmp_path / 'HR'), 'dataroot_LR': str(tmp_path / 'LR')}},
           'path': {'root': str(tmp_path / 'out'), 'pretrain_model_G': None},
           'network_G': {'which_model_G': 'RRDB_net', 'norm_type': None, 'mode': 'CNA', 'nf': 64, 'nb': 1, 'in_nc': 3, 'out_nc': 3,
                         'gc': 32, 'group': 1}}
    cfg = tmp_path / 'test.json'
    cfg.write_text(json.dumps(opt))
    env = dict(os.environ, PYTHONPATH=ROOT, CUDA_VISIBLE_DEVICES='')
    r = subprocess.run([sys.executable, '-m', 'dasr_b200.launch', str(srn / 'test.py'), '-opt', str(cfg)], cwd=str(tmp_path), env=env,
                       capture_output=True, text=True, timeout=600)
    err = r.stderr + r.stdout
    assert r.returncode != 0
    assert 'was imported instead of the dasr_b200 mirror' not in err, err[-2000:]
    assert 'dasr_b200/srn/models/SR_model.py' in err, err[-2000:]          # the mirror, not the checkout's models package
    assert 'no CPU fallback exists' in err, err[-2000:]


def test_auto_reproduce_resolves_to_the_mirrors_after_install(tmp_path):
    """`python -m dasr_b200.install <codes>` + an unmodified driver script that shells out like codes/Auto_Reproduce.py
    (`cd ./DSN; sh <launcher>.sh` and `cd ./SRN; python train.py -opt ...`): both child scripts must import the dasr_b200
    mirrors although their own directory is first on sys.path.  The overlay log records which imports were redirected for
    which script directory."""
    codes = tmp_path / 'codes'
    py = shlex.quote(sys.executable)
    _write_tree(codes, {
        'Auto_Reproduce.py': 'import os\nos.system("cd ./DSN; sh launcher.sh")\nos.system("cd ./SRN; %s train.py -opt x.json")\n' % py,
        'DSN/launcher.sh': '%s train.py --generator DeResnet\n' % py,
        'DSN/train.py': 'import model\nimport loss\nimport utils\n',
        'DSN/utils.py': '',
        'SRN/train.py': 'import options.options\nimport utils.util\nimport models\n'})
    _write_tree(codes / 'DSN', DSN_DECOYS)
    _write_tree(codes / 'SRN', SRN_DECOYS)
    from dasr_b200 import install
    import io
    buf = io.StringIO()
    site_dir = install.install(str(codes), pth=False, out=buf)
    assert 'PYTHONPATH' in buf.getvalue() and (codes / 'SRN' / '.dasr_b200').read_text().strip() == 'SRN'
    log = tmp_path / 'overlay.log'
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([site_dir, ROOT]),
               CUDA_VISIBLE_DEVICES='', DASR_B200_OVERLAY_LOG=str(log), DASR_B200_ALLOW_RANDOM_VGG='1')
    r = subprocess.run([sys.executable, 'Auto_Reproduce.py'], cwd=str(codes), env=env, capture_output=True, text=True, timeout=900)
    assert 'was imported instead of the dasr_b200 mirror' not in r.stdout + r.stderr, r.stderr[-3000:]
    text = log.read_text() if log.exists() else ''
    dsn_dir, srn_dir = str(codes / 'DSN'), str(codes / 'SRN')
    for name in ('model', 'loss'):
        assert any(l.startswith(name + ' -> ') and 'dasr_b200/dsn/' in l and dsn_dir in l for l in text.splitlines()), (name, text, r.stderr[-3000:])
    for name in ('options', 'utils', 'models'):
        assert any(l.startswith(name + ' -> ') and 'dasr_b200/srn/' in l and srn_dir in l for l in text.splitlines()), (name, text, r.stderr[-3000:])
    # an unmarked directory is left alone
    install.uninstall(str(codes), out=buf)
    assert not (codes / 'SRN' / '.dasr_b200').exists()
    log.unlink()
    subprocess.run([sys.executable, '-c', 'import options.options'], cwd=srn_dir, env=env, capture_output=True, text=True, timeout=300)
    assert not log.exists() or 'options' not in log.read_text()


def test_bench_cpu_leg_and_generators_run():
    """bench.py: the CPU reference leg runs (tiny image) and the local deterministic generator matches the oracle's."""
    import torch
    import bench
    from oracle import srn_oracle as O
    mp_s, dt = bench.cpu_reference_forward(1, 8, 2, 1, 0)
    assert mp_s > 0 and dt > 0
    assert torch.equal(bench.synth((2, 3, 5), 9, 0.5, 0.5), O.synth((2, 3, 5), 9, 0.5, 0.5))


def test_dense_block_schedules_cover_every_product_once():
    """engine.SCHED2 / SCHED3: every (conv k, input chunk c < k) product of the dense block is computed by exactly one
    launch, launch j completes conv j (first of its contiguous column set), only reads activations that already exist and
    launch 1 initialises every partial sum."""
    from dasr_b200 import engine
    for sched in engine.SCHEDULES.values():
        assert engine.check_schedule(sched)
    bad = ((('x',), (1, 2, 3, 4, 5)), ((1,), (2,)), ((2,), (3, 4)), ((3,), (4,)), ((1, 2, 3, 4), (5,)))     # (3, x1) missing
    import pytest
    with pytest.raises(AssertionError):
        engine.check_schedule(bad)
    # channel offsets of the chunks inside the [x | x1..x4 | p5] buffer
    assert engine._sched2_chunk_offsets(64, 'x') == [0, 32] and engine._sched2_chunk_offsets(64, 3) == [128]


def test_ddm_window_ranges_reproduce_the_reference_scatter(golden):
    """dasr_b200/dsn/receptive_cal.py: the per-coordinate ranges of covering patch rows / columns (host logic feeding the
    dasr_ddm gather kernels), evaluated here with numpy, reproduce the reference's scatter-add / count
    (codes/DSN/receptive_cal.py:34-60) for the three discriminator geometries of create_dataset_modified.py:113-119 —
    including the quirk that the W axis' (jump, rf, start) are used for both axes."""
    from dasr_b200.dsn import receptive_cal as R
    for c in golden('ddm.pt'):
        H, W = c['hw']
        lh, lw = R.receptive_cal(H, c['convnet']), R.receptive_cal(W, c['convnet'])
        assert tuple(lh) == c['layer_h'] and tuple(lw) == c['layer_w']
        patch = O.synth_image(c['patch_shape'], c['patch_seed']).double().numpy()[0, 0]
        jump, rf, start = lw[1], lw[2], lw[3]
        ilo, ihi = R._windows(lh[0], H, jump, rf, start)
        jlo, jhi = R._windows(lw[0], W, jump, rf, start)
        out = np.empty((H, W))
        for y in range(H):
            for x in range(W):
                blk = patch[ilo[y]:ihi[y] + 1, jlo[x]:jhi[x] + 1]
                out[y, x] = blk.sum() / blk.size if blk.size else np.nan
        ref = c['ddm'].numpy()[0, 0]
        assert np.allclose(out, ref, rtol=1e-12, atol=1e-12, equal_nan=True), c['name']


def test_f32_math_context_and_fused_layer_eligibility(monkeypatch):
    """ops.f32_math nests (the arithmetic of the generic conv kernels inside a step); the one-kernel discriminator layer is
    taken for feature maps of at most 8 x 64 pixels (cluster of <= 8 CTAs) and can be switched off."""
    from dasr_b200 import ops
    assert ops._f32_math[-1] == 0
    with ops.f32_math('tf32'):
        assert ops._f32_math[-1] == ops.F32_MATH['tf32'] == 2
        with ops.f32_math('fma'):
            assert ops._f32_math[-1] == 1
        assert ops._f32_math[-1] == 2
    assert ops._f32_math[-1] == 0
    assert ops.conv_in_lrelu_fused_ok(32, 16, 16, 128) and ops.conv_in_lrelu_fused_ok(1, 22, 23, 64)
    assert not ops.conv_in_lrelu_fused_ok(32, 32, 32, 128)
    monkeypatch.setenv('DASR_B200_FUSED_IN', '0')
    assert not ops.conv_in_lrelu_fused_ok(32, 16, 16, 128)


def test_drop_in_entry_points_default_to_mixed_precision(monkeypatch):
    """dasr_b200.launch / the import overlay set DASR_B200_TRAIN_PRECISION=bf16 unless the user chose a mode."""
    from dasr_b200 import overlay
    monkeypatch.delenv('DASR_B200_TRAIN_PRECISION', raising=False)
    overlay._drop_in_defaults()
    assert os.environ['DASR_B200_TRAIN_PRECISION'] == 'bf16'
    monkeypatch.setenv('DASR_B200_TRAIN_PRECISION', 'fp32')
    overlay._drop_in_defaults()
    assert os.environ['DASR_B200_TRAIN_PRECISION'] == 'fp32'


def test_pair_kernel_cout_tiles_for_the_vgg_layers():
    """ops.pick_nt_pair: the Cout tile of a CTA pair is the largest multiple of 32 whose half filter set (9 taps x K x nt / 2
    x 2 B) plus an epilogue ring and four A stages fit one SM — host-side planning through dasr_conv_tc2_supported (no GPU)."""
    from dasr_b200 import ops
    assert ops.pick_nt_pair(512, 512) == 32          # conv4 / conv5: 147 KB of filters per SM
    assert ops.pick_nt_pair(256, 256) == 64
    assert ops.pick_nt_pair(128, 256) == 128
    assert ops.pick_nt_pair(64, 64) == 64
    assert ops.pick_nt_pair(64, 48) is None          # not a multiple of 32
