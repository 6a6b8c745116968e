#!/usr/bin/env python
"""bench.py — headline benchmark of the DASR SRN hot path on B200; prints one JSON result line on stdout.

Workload (BASELINE.json configs[1]): RRDBNet-23 x4 generator forward, batch 16 x 3 x 256 x 256 synthetic LR
images per GPU (weak scaling), tcgen05 bf16 kernels (fp32 accumulate), random-init weights of the
reference architecture.  metric = output megapixels / second over all GPUs.

  value : device-timed steps, inputs resident in HBM (CUDA events, max over ranks)
  e2e   : the same metric through the public API (SRModel.feed_data -> test -> get result) with PINNED HOST
          input and output buffers, H2D + D2H inside the timed region
  roofline      : the tcgen05 conv kernel (all conv_tc launches of a step bracketed by CUDA events)
  cpu_baseline  : the oracle port of the reference forward on the host cores (bounded sample)
  train         : DASR_Model train step (BASELINE configs[2]: B=32, HR crop 128) iterations / second, fp32 kernels

`--impl reference` times the reference algorithm's CPU path (oracle port of the pure-Python reference) on the host
cores with all threads.

`--steps K` is the number of timed steps of every GPU forward measurement and of `--impl reference`; the cpu_baseline
sample beside the GPU result is one forward (it only sets the scale of the comparison).  `--dump-outputs DIR` writes what
the timed GPU forward returned in its last step (see dump_outputs), so that two builds can be compared output for
output: inputs and weights are generated from fixed seeds and are identical from run to run.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# synthetic weights everywhere (no checkpoints offline): the perceptual networks run with deterministic random features
os.environ.setdefault('DASR_B200_ALLOW_RANDOM_VGG', '1')

NB, NF, BATCH, LR = 23, 64, 16, 256
FLOP_PER_LR_PIXEL = 35853696          # whole G forward, SURVEY.md §8(d): conv MACs x2, no recompute credit
METRIC = 'x4 SR output megapixels/sec (RRDBNet-23 G forward)'


def out_mp(batch, lr):
    return batch * (4 * lr) * (4 * lr) / 1e6


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1400.0)), 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)'
    return 1400.0, 'fallback (B200_PROFILING.md sustained ~1.4 PFLOP/s)'


class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                       '-lms', '100'], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(', ') for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], 0, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.strip().lower().startswith('active'):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        # median of the samples under load (upper half: the sampler also sees idle edges)
        load = sm[len(sm) // 2:] if sm else []
        return {'sm_mhz': load[len(load) // 2] if load else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


def synth(shape, seed, scale=1.0, offset=0.0):
    """Deterministic pseudo-random fp32 tensor (64-bit mix hash of the element index; no RNG state, identical on every
    rank / box).  The GPU arms generate their inputs and weights with this; oracle/ is only imported by the CPU legs."""
    import numpy as np
    import torch
    n = 1
    for d in shape:
        n *= int(d)
    x = np.arange(n, dtype=np.uint64) + np.uint64((int(seed) * 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF)
    for mul in (0xFF51AFD7ED558CCD, 0xC4CEB9FE1A85EC53):
        x ^= x >> np.uint64(33)
        x = (x * np.uint64(mul)) & np.uint64(0xFFFFFFFFFFFFFFFF)
    x ^= x >> np.uint64(33)
    u = (x >> np.uint64(40)).astype(np.float64) / float(1 << 24)
    return torch.from_numpy(((u * 2.0 - 1.0) * scale + offset).astype(np.float32)).reshape(tuple(shape))


def synth_image(shape, seed):
    return synth(shape, seed, 0.5, 0.5)


def synth_weights(net, seed=1, gain=0.1):
    """Kaiming-like magnitudes for every tensor of net.state_dict() (random-init stand-in: no checkpoints offline)."""
    import math
    sd = {}
    for i, (k, v) in enumerate(net.state_dict().items()):
        if v.dim() == 4:
            bound = gain * math.sqrt(2.0 / (v.shape[1] * v.shape[2] * v.shape[3])) * math.sqrt(3.0)
            sd[k] = synth(tuple(v.shape), seed * 1000 + i, bound)
        else:
            sd[k] = synth(tuple(v.shape), seed * 1000 + i, 0.05)
    return sd


def pick_threads():
    """Fixed policy for the CPU arms: min(32, host CPUs) intra-op threads.  (torch's oneDNN convs on this path stop
    scaling around 16-32 threads and regress when oversubscribed on a shared many-core host; round 1 probed per run and
    landed on 16 / 32 / 64 from run to run, which made the baseline jumpy.)"""
    return max(1, min(32, os.cpu_count() or 1))


def cpu_reference_forward(n_images, lr, threads, steps, warmup):
    """The reference algorithm on CPU (oracle port, fp32, torch CPU ops) — used by --impl reference and cpu_baseline."""
    import torch
    from oracle import srn_oracle as O
    torch.set_num_threads(threads)
    sd = O.synth_state_dict(O.rrdbnet_shapes(nb=NB), 1, 0.1)
    x = O.synth_image((n_images, 3, lr, lr), 7)
    with torch.no_grad():
        for _ in range(warmup):
            O.rrdbnet_forward(x, sd, NB)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.rrdbnet_forward(x, sd, NB)
        dt = (time.perf_counter() - t0) / steps
    return out_mp(n_images, lr) / dt, dt


def cpu_reference_train_step(threads, B=8):
    """configs[2] on CPU: the oracle's DASR train step (G + patch-D + VGG19 perceptual + weighted L1, both Adam steps) on a
    bounded sample of B of the 32 crops per half-batch; returns (it/s scaled to batch 32, seconds of the sample)."""
    import torch
    from oracle import srn_oracle as O
    torch.set_num_threads(threads)
    sdG = O.synth_state_dict(O.rrdbnet_shapes(nb=NB), 1, 0.1)
    sdD = O.synth_state_dict(O.nlayer_d_shapes(9, 64, 2), 2, 1.0)
    sdF = O.synth_state_dict(O.vgg19_shapes(34), 3, 1.0)
    h = 32
    data = {'LR_real': O.synth_image((B, 3, h, h), 200), 'LR_fake': O.synth_image((B, 3, h, h), 300),
            'HR': O.synth_image((B, 3, 4 * h, 4 * h), 400), 'HR_unpair': O.synth_image((B, 3, 4 * h, 4 * h), 500),
            'fake_w': O.synth_image((B, 1, h, h), 600)}
    t0 = time.perf_counter()
    O.dasr_train_step(sdG, sdD, sdF, data, NB)
    dt = time.perf_counter() - t0
    return (B / 32.0) / dt, dt


def cpu_reference_dsn_step(threads, B=4):
    """configs[4] on CPU: the oracle's DSN iteration on B of the 8 crops; returns (it/s scaled to batch 8, seconds)."""
    import torch
    from oracle import dsn_oracle as D
    from oracle import srn_oracle as O
    torch.set_num_threads(threads)
    sdG = D.synth_de_resnet(8, 4, 7, 0.7)
    sdD = O.synth_state_dict(D.fsd_shapes(9), 8, 1.0)
    sdV = O.synth_state_dict(D.vgg16_shapes(), 9, 1.0)
    inp, bic, dis = O.synth_image((B, 3, 256, 256), 700), O.synth_image((B, 3, 64, 64), 800), O.synth_image((B, 3, 64, 64), 900)
    t0 = time.perf_counter()
    D.dsn_train_step(sdG, sdD, sdV, inp, bic, dis)
    dt = time.perf_counter() - t0
    return (B / 8.0) / dt, dt


DUMP_SAMPLES = 1 << 22


def dump_outputs(dirname, sr):
    """Write the SR batch of one forward ([16, 3, 1024, 1024], 201 MB as float32) as a fixed, seeded sample of
    DUMP_SAMPLES elements: DIR/sr.npy holds their values (float32), DIR/sr_index.npy their flat positions in the batch
    (ascending, float64: exact).  48 MB in all."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    flat = sr.detach().float().reshape(-1)
    idx = np.sort(np.random.default_rng(0).choice(flat.numel(), size=DUMP_SAMPLES, replace=False))
    vals = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy()
    np.save(os.path.join(dirname, 'sr.npy'), vals)
    np.save(os.path.join(dirname, 'sr_index.npy'), idx.astype(np.float64))


def run_reference(args, rank):
    if rank != 0:
        return
    threads = pick_threads()
    steps, warm = args.steps, 1 if args.warmup > 0 else 0
    nimg = 4
    mp_s, dt = cpu_reference_forward(nimg, LR, threads, steps, warm)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': mp_s, 'unit': 'MP/s', 'n_gpus': args.gpus, 'steps': steps,
        'warmup': warm, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'RRDBNet-23 x4 inference, batch 16 x 3x256x256 per GPU (configs[1]); CPU arm: one step = a '
                               'bounded sample of 4 of the 16 images', 'inputs': 'host memory'},
        'cpu_baseline': {'value': mp_s, 'unit': 'MP/s', 'cores': threads, 'host_cpus': os.cpu_count(), 'kind': 'port',
                         'threads_policy': 'min(32, host CPUs)',
                         'sample': '4 x 3x256x256 images per step (1/4 of the batch), oracle/srn_oracle.py rrdbnet_forward, torch CPU fp32'},
        'e2e': {'value': mp_s, 'unit': 'MP/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='dasr_b200')
    ap.add_argument('--train-steps', type=int, default=20)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the output of the last timed forward step to DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the output of the GPU path; it does not apply to --impl reference')
    rank = int(os.environ.get('RANK', 0))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    if args.impl == 'reference':
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)

    from dasr_b200 import _lib
    from dasr_b200.srn.models import create_model
    from dasr_b200.srn.options.options import dict_to_nonedict
    W, K = max(args.warmup, 3), args.steps

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    opt = dict_to_nonedict({
        'name': 'bench', 'model': 'sr', 'scale': 4, 'gpu_ids': [local_rank], 'is_train': False, 'chop': False, 'val_lpips': False,
        'path': {'pretrain_model_G': None},
        'network_G': {'which_model_G': 'RRDB_net', 'norm_type': None, 'mode': 'CNA', 'nf': NF, 'nb': NB, 'in_nc': 3,
                      'out_nc': 3, 'gc': 32, 'scale': 4}})
    model = create_model(opt)
    netG = model.netG.module if hasattr(model.netG, 'module') else model.netG
    netG.load_state_dict(synth_weights(netG))
    netG.precision = os.environ.get('DASR_BENCH_PRECISION', 'bf16')   # 'bf16' (dense-block N-fused) | 'bf16_layer'
    netG.eval()

    x_host = synth_image((BATCH, 3, LR, LR), 100 + rank).pin_memory()
    x_dev = x_host.to(dev)
    y_host = torch.empty((BATCH, 3, 4 * LR, 4 * LR), dtype=torch.float32).pin_memory()

    def _rec():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    # ---------------------------------------------------------------- device-resident timing (value)
    # The forward is replayed from a CUDA graph (captured on the first call); all timing is CUDA events.
    with torch.no_grad():
        for _ in range(W):
            netG(x_dev)
        barrier()
        sampler = ClockSampler(local_rank) if rank == 0 else None
        l0 = _lib.LAUNCHES
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            out = netG(x_dev)
        e1.record()
        barrier()
        launches = _lib.LAUNCHES - l0
        ms = max_over_ranks(e0.elapsed_time(e1) / K)
        clocks = sampler.stop() if sampler else None
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, out)
        del out
        # roofline: time of the conv_tc launch sequence = step time minus the (few) non-conv kernels of a forward,
        # which are timed here on the same shapes: layout change of the input, zero fill, per-chunk feature copy,
        # and the clone of the graph's static output.
        from dasr_b200 import ops
        bf = torch.bfloat16
        xin = torch.zeros((BATCH, LR, LR, 32), dtype=bf, device=dev)
        fea = torch.empty((BATCH, LR, LR, NF), dtype=bf, device=dev)
        buf = torch.empty((BATCH, LR, LR, 256), dtype=bf, device=dev)
        big = torch.empty((BATCH, 3, 4 * LR, 4 * LR), dtype=torch.float32, device=dev)
        def _non_conv():
            xin.zero_()
            ops.nchw_to_nhwc(x_dev, ops.View(xin, 3, 0))
            ops.axpby(fea, 1.0, None, 0.0, ops.View(buf, NF, 0))
            big.clone()
            x_dev.clone()
        for _ in range(2):
            _non_conv()                          # allocator warm-up
        torch.cuda.synchronize()
        n0 = _rec()
        for _ in range(K):
            xin.zero_()
            ops.nchw_to_nhwc(x_dev, ops.View(xin, 3, 0))
            ops.axpby(fea, 1.0, None, 0.0, ops.View(buf, NF, 0))
            big.clone()
            x_dev.clone()
        n1 = _rec()
        torch.cuda.synchronize()
        non_tc_ms = n0.elapsed_time(n1) / K
        tc_ms = ms - non_tc_ms
        n_tc = launches // K - 2          # kernels of ours per forward minus the layout change of the input and the feature copy
        del xin, fea, buf, big

        # ---------------------------------------------------------------- end-to-end through the public API
        # Every step: H2D of the input from pinned host memory (feed_data), the forward (test()), D2H of the result into
        # pinned host memory.  The D2H of step k runs on a copy stream and overlaps the forward of step k+1 (two host
        # buffers); the timed region ends when the last result has landed on the host.
        y_hosts = [y_host, torch.empty_like(y_host).pin_memory()]
        copy_stream = torch.cuda.Stream()
        done = [torch.cuda.Event(), torch.cuda.Event()]

        def e2e_step(k):
            model.feed_data({'LR': x_host})          # H2D of the step's input from pinned host memory
            model.test()                             # netG forward (public API call of test.py)
            res = model.fake_H
            ready = torch.cuda.Event()
            ready.record()
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(ready)
                y_hosts[k & 1].copy_(res, non_blocking=True)   # D2H of the result
                res.record_stream(copy_stream)
                done[k & 1].record(copy_stream)

        for k in range(2):
            e2e_step(k)
        copy_stream.synchronize()
        barrier()
        e0.record()
        for k in range(K):
            if k >= 2:
                done[k & 1].synchronize()            # host buffer k&1 was consumed two steps ago
            e2e_step(k)
        torch.cuda.current_stream().wait_stream(copy_stream)
        e1.record()
        barrier()
        e2e_ms = max_over_ranks(e0.elapsed_time(e1) / K)
        # ---------------------------------------------------------------- same launches with IEEE half operands
        # (precision 'fp16': tcgen05 kind::f16 with F16 instead of BF16 operands — the mode that meets the 3-decimal
        # PSNR / SSIM gate, tests/test_gpu_parity_scale.py); reported beside the bf16 headline, not instead of it
        fp16_ms = None
        if os.environ.get('DASR_BENCH_FP16', '1') != '0' and netG.precision == 'bf16':
            netG.precision = 'fp16'
            for _ in range(max(W, 3)):
                netG(x_dev)
            barrier()
            e0.record()
            for _ in range(K):
                out = netG(x_dev)
            e1.record()
            barrier()
            fp16_ms = max_over_ranks(e0.elapsed_time(e1) / K)
            del out
            netG.precision = 'bf16'
    model.fake_H = None
    netG._graphs.clear()
    torch.cuda.empty_cache()

    # ---------------------------------------------------------------- train step (configs[2]) and DSN iteration (configs[4])
    train = dsn = None
    allreduce_ms = None
    if args.train_steps > 0:
        train = bench_train(args, dev, local_rank, world, barrier, max_over_ranks, 'bf16')
        fp32_args = argparse.Namespace(**vars(args))
        fp32_args.train_steps = min(args.train_steps, 3)            # the fp32 parity mode takes ~0.5 s per step
        train['fp32_mode'] = bench_train(fp32_args, dev, local_rank, world, barrier, max_over_ranks, 'fp32')
        dsn = bench_dsn(args, dev, rank, world, barrier, max_over_ranks, 'bf16')
        dsn['fp32_mode'] = bench_dsn(fp32_args, dev, rank, world, barrier, max_over_ranks, 'fp32')
        if world > 1:
            # the gradient exchange in isolation: NCCL all-reduce (AVG) of the 69.5 MB [G | D] bucket, CUDA events, max over ranks
            flat = torch.zeros(17366724, dtype=torch.float32, device=dev)
            for _ in range(3):
                dist.all_reduce(flat, op=dist.ReduceOp.AVG)
            barrier()
            a0, a1 = _rec(), None
            for _ in range(10):
                dist.all_reduce(flat, op=dist.ReduceOp.AVG)
            a1 = _rec()
            barrier()
            allreduce_ms = max_over_ranks(a0.elapsed_time(a1) / 10)
            del flat

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    peak, peak_src = peaks()
    flops_step = FLOP_PER_LR_PIXEL * BATCH * LR * LR
    ach = flops_step / (tc_ms * 1e-3) / 1e12
    traffic, traffic_src = None, None
    for name in ('r2_traffic.json', 'r1_traffic.json'):
        tp = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get('dram_bytes_per_launch_avg')
            traffic_src = 'static: ncu launch list of this command, profiles/%s (not re-measured in this run)' % name
            break
    line = {
        'metric': METRIC, 'value': world * out_mp(BATCH, LR) / (ms * 1e-3), 'unit': 'MP/s', 'n_gpus': world, 'steps': K,
        'warmup': W, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16',
        'data': 'synthetic',
        'config': {'workload': 'RRDBNet-23 x4 inference, batch 16 x 3x256x256 per GPU, forward_chop off (BASELINE configs[1])',
                   'weights': 'random init (deterministic synthetic), reference architecture nb=23 nf=64 gc=32',
                   'parallelism': 'dp%d (independent replicas, no collective on the inference path)' % world,
                   'l2': 'working set (3 x 537 MB dense-block buffers + 2.1 GB HR activations) >> 126 MB L2: no flush needed'},
        'e2e': {'value': world * out_mp(BATCH, LR) / (e2e_ms * 1e-3), 'unit': 'MP/s', 'ms_per_step': e2e_ms,
                'h2d_bytes_per_step': x_host.numel() * 4, 'd2h_bytes_per_step': y_host.numel() * 4,
                'api': 'SRModel.feed_data(pinned host LR) -> SRModel.test() -> pinned host copy of fake_H (copy stream, double buffered)'},
        'gpu_launches': launches,
        'clocks': clocks,
        'roofline': {'bound': 'tensor', 'kernel': 'dasr::conv_tc2_kernel / conv_tc_kernel (tcgen05 implicit-GEMM 3x3 conv)',
                     'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak, 'peak_source': peak_src,
                     'traffic': traffic, 'traffic_source': traffic_src, 'launches_per_step': n_tc, 'avg_launch_ms': tc_ms / n_tc,
                     'algorithmic_flops_per_step': flops_step, 'non_conv_ms_per_step': non_tc_ms},
    }
    if fp16_ms:
        line['fp16'] = {'value': world * out_mp(BATCH, LR) / (fp16_ms * 1e-3), 'unit': 'MP/s', 'ms_per_step': fp16_ms,
                        'note': "netG.precision='fp16': same kernels and schedule, IEEE half operands / activations"}
    detail = {'roofline_note': 'achieved = algorithmic conv FLOPs of one forward / (CUDA-event step time - CUDA-event time of the non-conv kernels of a step)'}
    if train:
        detail['train'], detail['dsn'] = train, dsn
        line['train'] = {'value': train['value'], 'unit': 'it/s', 'ms_per_step': train['ms_per_step'], 'steps': train['steps'],
                         'global_batch': 32 * world, 'dtype': 'bf16 mixed', 'fp32_mode_it_s': train['fp32_mode']['value'],
                         'allreduce_ms': allreduce_ms, 'gpu_launches_per_step': train['gpu_launches_per_step']}
        line['dsn'] = {'value': dsn['value'], 'unit': 'it/s', 'ms_per_step': dsn['ms_per_step'], 'global_batch': 8 * world,
                       'fp32_mode_it_s': dsn['fp32_mode']['value']}
    if not args.no_cpu_baseline and world == 1:
        threads = pick_threads()
        mp_s, dt = cpu_reference_forward(4, LR, threads, 1, 0)
        line['cpu_baseline'] = {'value': mp_s, 'unit': 'MP/s', 'cores': threads, 'kind': 'port', 'seconds': dt,
                                'sample': '4 x 3x256x256 images (1/4 of the batch), oracle port of RRDBNet-23 forward, torch CPU fp32, min(32, host CPUs) threads'}
        if train:
            it_s, dt = cpu_reference_train_step(threads)
            line['train']['cpu_baseline'] = {'value': it_s, 'unit': 'it/s', 'cores': threads, 'kind': 'port', 'seconds': dt,
                                             'sample': 'oracle DASR train step on 8 of the 32 crops per half batch, scaled to batch 32'}
            it_s, dt = cpu_reference_dsn_step(threads)
            line['dsn']['cpu_baseline'] = {'value': it_s, 'unit': 'it/s', 'cores': threads, 'kind': 'port', 'seconds': dt,
                                           'sample': 'oracle DSN iteration on 4 of the 8 crops, scaled to batch 8'}
    # full detail (per-mode configs, dtypes, launch counts) on stderr; stdout carries ONE compact JSON line
    sys.stderr.write('bench detail: ' + json.dumps(detail) + '\n')
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def bench_train(args, dev, local_rank, world, barrier, max_over_ranks, precision='fp32'):
    """DASR_Model.feed_data + optimize_parameters (G + D + VGG perceptual + weighted L1), B=32 per GPU, HR crop 128."""
    import warnings
    import torch
    from dasr_b200 import _lib
    from dasr_b200.srn.models import create_model
    from dasr_b200.srn.options.options import dict_to_nonedict
    B, h = 32, 32
    opt = dict_to_nonedict({
        'name': 'bench_train', 'model': 'DASR', 'scale': 4, 'gpu_ids': [local_rank], 'is_train': True, 'chop': False,
        'val_lpips': False, 'multiweights': True,
        'path': {'pretrain_model_G': None, 'pretrain_model_D_target': None, 'pretrain_model_D_source': None},
        'network_G': {'which_model_G': 'RRDB_net', 'norm_type': None, 'mode': 'CNA', 'nf': NF, 'nb': NB, 'in_nc': 3,
                      'out_nc': 3, 'gc': 32, 'scale': 4},
        'network_D': {'which_model_D': 'discriminator_patch', 'nf': 64, 'in_nc': 9, 'n_layers': 2},
        'train': {'lr_G': 5e-5, 'weight_decay_G': 0, 'beta1_G': 0.9, 'lr_D': 5e-5, 'weight_decay_D': 0, 'beta1_D': 0.9,
                  'lr_scheme': 'MultiStepLR', 'lr_steps': [50000, 80000], 'lr_gamma': 0.5, 'fs': 'wavelet', 'norm': True,
                  'sup_LL': True, 'pixel_criterion': 'l1', 'pixel_weight': 1, 'pixel_LL_weight': 1, 'feature_criterion': 'l1',
                  'feature_weight': 1e-2, 'gan_type': 'vanilla', 'ragan': False, 'gan_H_target': 1e-4, 'gan_H_source': 0,
                  'G_update_inter': 1, 'D_update_inter': 1, 'D_update_ratio': 1, 'D_init_iters': 0}})
    torch.manual_seed(0)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        model = create_model(opt)
    g = model.netG.module if hasattr(model.netG, 'module') else model.netG
    g.train_precision = precision
    f = getattr(model, 'netF', None)
    if f is not None:
        (f.module if hasattr(f, 'module') else f).precision = precision
    rank = int(os.environ.get('RANK', 0))
    data = {'LR_real': synth_image((B, 3, h, h), 200 + rank).pin_memory(), 'LR_fake': synth_image((B, 3, h, h), 300 + rank).pin_memory(),
            'HR': synth_image((B, 3, 4 * h, 4 * h), 400 + rank).pin_memory(), 'HR_unpair': synth_image((B, 3, 4 * h, 4 * h), 500 + rank).pin_memory(),
            'fake_w': synth_image((B, 1, h, h), 600 + rank).pin_memory()}
    step = 0
    for _ in range(2):
        step += 1
        model.feed_data(data, True)
        model.optimize_parameters(step)
    barrier()
    l0 = _lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.train_steps):
        step += 1
        model.feed_data(data, True)
        model.optimize_parameters(step)
    log = model.get_current_log()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / args.train_steps)
    res = {'metric': 'DASR SRN train iterations/sec (G + patch-D + VGG19 perceptual + weighted L1, Adam x2)',
           'value': 1e3 / ms, 'unit': 'it/s', 'ms_per_step': ms, 'steps': args.train_steps,
           'dtype': 'f32' if precision == 'fp32' else 'bf16 (G and VGG19: tcgen05 fprop+dgrad, G wgrad tcgen05 with fp32 accumulation; D, losses, Adam fp32)',
           'config': {'workload': 'BASELINE configs[2]: batch 32 (2B=64 LR 32x32 through G), HR crop 128, fs wavelet, per GPU',
                      'global_batch': 32 * world, 'parallelism': 'dp%d, one flat-bucket NCCL all-reduce of G+D grads per step' % world},
           'gpu_launches_per_step': (_lib.LAUNCHES - l0) // args.train_steps,
           'loss_l_g_pix': log.get('loss/l_g_pix')}
    del model
    torch.cuda.empty_cache()
    return res


def bench_dsn(args, dev, rank, world, barrier, max_over_ranks, precision='fp32'):
    """BASELINE configs[4]: DSN DeResnet + wavelet-cat FS discriminator GAN iteration, batch 8, crop 256, per GPU."""
    import warnings
    import torch
    from dasr_b200 import _lib
    from dasr_b200.dsn.loss import GeneratorLoss
    from dasr_b200.dsn.model import De_resnet, Discriminator
    from dasr_b200.dsn.train import train_iteration
    import contextlib
    import io
    torch.manual_seed(0)
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter('ignore')
        mg = De_resnet(n_res_blocks=8, scale=4).to(dev)
        md = Discriminator(kernel_size=5, D_arch='FSD', norm_layer='Instance', filter_type='wavelet', cs='cat').to(dev)
        gl = GeneratorLoss(per_type='VGG', filter='wavelet', kernel_size=5, w_col=1, w_tex=0.005, w_per=0.01, wgan=False).to(dev)
    mg.precision = precision
    gl.perceptual_loss.loss_network.precision = precision
    og = torch.optim.Adam(mg.parameters(), lr=1e-4, betas=[0.5, 0.999])
    od = torch.optim.Adam(md.parameters(), lr=1e-4, betas=[0.5, 0.999])
    B = 8
    inp = synth_image((B, 3, 256, 256), 700 + rank).to(dev)
    bic = synth_image((B, 3, 64, 64), 800 + rank).to(dev)
    dis = synth_image((B, 3, 64, 64), 900 + rank).to(dev)
    sync = None
    if world > 1:
        import torch.distributed as dist
        plist = [p for p in list(mg.parameters()) + list(md.parameters()) if p.requires_grad]

        def sync():
            flat = torch.cat([p.grad.reshape(-1) for p in plist])
            dist.all_reduce(flat)
            flat /= world
            o = 0
            for p in plist:
                p.grad = flat[o:o + p.numel()].view_as(p)
                o += p.numel()
    for _ in range(2):
        train_iteration(mg, md, gl, og, od, inp, bic, dis, grad_sync=sync, log=False)
    barrier()
    l0 = _lib.LAUNCHES
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.train_steps):
        train_iteration(mg, md, gl, og, od, inp, bic, dis, grad_sync=sync, log=False)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / args.train_steps)
    res = {'metric': 'DSN train iterations/sec (De_resnet + FS discriminator + VGG16 perceptual + LL colour loss, Adam x2)',
           'value': 1e3 / ms, 'unit': 'it/s', 'ms_per_step': ms, 'steps': args.train_steps,
           'dtype': 'f32' if precision == 'fp32' else 'bf16 (De_resnet trunk and VGG16 on tcgen05, fp32 accumulation; stride-2 tail, discriminator, losses, Adam fp32)',
           'config': {'workload': 'BASELINE configs[4]: batch 8, crop 256 -> 64, wavelet cat, per GPU', 'global_batch': B * world},
           'gpu_launches_per_step': (_lib.LAUNCHES - l0) // args.train_steps}
    del mg, md, gl
    torch.cuda.empty_cache()
    return res


if __name__ == '__main__':
    main()
