#!/usr/bin/env python
"""bench.py - headline benchmark of the Competitive-Collaboration training step on B200.

  python bench.py --gpus N --steps K --warmup W          (N>1: launched under torch.distributed.run)
  python bench.py --impl reference ...                    (the reference algorithm's CPU path: oracle port)
  python bench.py ... --dump-outputs DIR                  (also write the last timed step's outputs as DIR/<name>.npy)

One JSON line on rank 0.  metric = BASELINE.json's "train-step triplets/sec at 256x832x6lvl": frame
snippets (target + 4 references) per second through forward + losses + backward + Adam.

  value     device-resident inputs, whole step replayed as one CUDA graph, CUDA-event timed, max over ranks
  e2e       same step through the public API with HOST (pinned) inputs: H2D of the 5 frames + intrinsics and
            a D2H read of the loss inside the timed region, every step
  roofline  dominant kernel family (by measured share of the step) against the measured B200 peak;
            roofline_warploss is the fused warp+loss kernel against the HBM peak (BASELINE metric, 2nd half)
  cpu_baseline  the oracle port of the reference step on this box's host cores (bounded sample)
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

import torch  # noqa: E402

H, W, NLEVELS = 256, 832, 6
PER_GPU_BATCH = 4
CFG_WORKLOAD = {
    'cfg1': 'cfg1: DispResNet6+PoseNetB6 depth/pose step, 256x832 b4/GPU, 6 pyramid levels '
            '(photometric_reconstruction_loss + edge-aware smoothness, fwd+bwd+Adam)',
    'cfg2': 'cfg2: Back2Future flow step, 256x832 b4/GPU, 6 levels (photometric_flow_loss + SSIM + edge-aware smoothness, '
            'fwd+bwd+Adam)',
    'cfg3': 'cfg3: full CC joint step (Disp+Pose+Mask+Flow, 5 losses), 256x832 b4/GPU, 6 levels, fwd+bwd+Adam',
}


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tensor_burst=d['bf16_tflops'], tensor_sustained=d['bf16_tflops_sustained'],
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm=6650.0, tensor_burst=1590.0, tensor_sustained=1400.0, source='fallback (B200_PROFILING.md)')


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.f = tempfile.NamedTemporaryFile('w+', suffix='.csv', delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                       '--format=csv,noheader,nounits', '-lms', '100'], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return None
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.strip().split(', ') for r in open(self.f.name) if r.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
                if v.strip().lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return None
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), samples=len(sm), reasons=sorted(reasons))


# ---------------------------------------------------------------------------------------------------
def host_batches(nb, B, seed0):
    """nb synthetic batches of the reference's sample contract in PINNED host memory."""
    from cc_b200 import synth
    out = []
    for i in range(nb):
        tgt, refs = synth.frames(B, H, W, seed=seed0 + i)
        K, Kinv = synth.intrinsics(B, H, W)
        ts = [tgt] + refs + [K, Kinv]
        if torch.cuda.is_available():
            ts = [t.pin_memory() for t in ts]
        out.append(ts)
    return out


def _say(msg):
    """progress line on stderr (CCB_BENCH_VERBOSE=1): which phase a rank is in when a multi-GPU run stalls"""
    if os.environ.get('CCB_BENCH_VERBOSE'):
        sys.stderr.write('[bench rank %s %.1fs] %s\n' % (os.environ.get('RANK', '0'), time.perf_counter() - _T0, msg))
        sys.stderr.flush()


_T0 = time.perf_counter()


def measure_cfg(cfg, args, dev, rank, local, world, steps, full):
    """One configuration: device-resident graph-replay timing (`value`), host-fed timing (`e2e`), and - when
    `full` - the eager profile pass (kernel shares + roofline objects).  Returns a dict of raw numbers."""
    from cc_b200 import _lib, dist as cdist, pyramid
    from cc_b200.train_step import Trainer, HostFeeder
    B = PER_GPU_BATCH
    _say('%s: build trainer (+ parameter broadcast)' % cfg)
    trainer = Trainer(cfg, dev, seed=0)
    dump = full and bool(args.dump_outputs)
    init = initial_state(trainer) if dump else None
    hb = host_batches(4, B, seed0=1000 * rank)
    static = [torch.empty_like(t, device=dev) for t in hb[0]]
    for s, h in zip(static, hb[0]):
        s.copy_(h)
    tgt, refs, K, Kinv = static[0], static[1:5], static[5], static[6]
    in_bytes = sum(t.numel() * 4 for t in hb[0])
    torch.cuda.synchronize()
    _say('%s: eager steps' % cfg)
    pyramid.clear()
    trainer.step(tgt, refs, K, Kinv)
    if getattr(trainer, 'wcache', None) is not None and not trainer.wcache.committed:
        pyramid.clear()                       # N > 1: the first step taught the gradient buckets, this one records the weight cache
        trainer.step(tgt, refs, K, Kinv)
    c0 = _lib.lib().ccb_launch_count()
    pyramid.clear()
    trainer.step(tgt, refs, K, Kinv)
    launches_per_step = _lib.lib().ccb_launch_count() - c0
    use_graph = not args.no_graph
    graph_aux = {}
    if use_graph:
        _say('%s: capture' % cfg)
        eager_step = trainer.step

        def step_keeping_aux(*a):
            # replay() hands back only the loss; the loss terms and network outputs of the step that capture() records
            # live at fixed addresses that every replay rewrites: keep them for --dump-outputs.  Only the recorded step's,
            # and detached: a live autograd graph of capture()'s eager warm-up step would keep the parameters' gradient
            # accumulators bound to the warm-up stream, and the captured backward would then wait on uncaptured work.
            loss, aux = eager_step(*a)
            if torch.cuda.is_current_stream_capturing():
                graph_aux['aux'] = {k: [t.detach() for t in v] if isinstance(v, (list, tuple)) else
                                    (v.detach() if torch.is_tensor(v) else v) for k, v in aux.items()}
            return loss, aux
        trainer.step = step_keeping_aux
        try:
            trainer.capture(tgt, refs, K, Kinv, warmup=1)
        finally:
            del trainer.step
        assert 'aux' in graph_aux, 'Trainer.capture() did not record its step through trainer.step: the outputs of the ' \
                                   'graph are out of reach of --dump-outputs'

    def one_step():
        if use_graph:
            return trainer.replay(), graph_aux['aux']
        pyramid.clear()
        return trainer.step(tgt, refs, K, Kinv)

    def run_steps(n):
        """n steps between two CUDA events; returns the events and what the last step returned."""
        a, b, out = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True), (None, None)
        a.record()
        for _ in range(n):
            out = None                                     # the previous step's outputs do not outlive it
            out = one_step()
        b.record()
        return a, b, out

    warm = max(args.warmup, 3)
    for _ in range(warm):
        one_step()
    # ---- value: device-resident inputs --------------------------------------------------------------
    sampler = ClockSampler(local) if (rank == 0 and full) else None
    _say('%s: timed region' % cfg)
    torch.cuda.synchronize(); cdist.barrier()
    if sampler:
        sampler.start()
    e0, e1, (loss, aux) = run_steps(steps - 1 if dump else steps)
    ms_total = 0.0
    if dump:
        # The dumped (last) step starts from the seeded initial state, reset outside the timed events: after many steps the
        # state carries every earlier step's rounding (the warp backward scatters with atomics, deep BatchNorms amplify),
        # while one step from a fixed state differs between runs or builds only by that step's own rounding.
        e1.synchronize()
        ms_total = e0.elapsed_time(e1)
        reset_state(trainer, init)
        e0, e1, (loss, aux) = run_steps(1)
    torch.cuda.synchronize(); cdist.barrier()
    clocks = sampler.stop() if sampler else None
    ms_total = cdist.max_over_ranks(ms_total + e0.elapsed_time(e1), dev)
    if dump and rank == 0:
        dump_outputs(args.dump_outputs, trainer, loss, aux)
    loss = aux = None
    # ---- e2e: host inputs, H2D + D2H inside the timed region ----------------------------------------
    _say('%s: e2e region' % cfg)
    loss_host = torch.empty(1).pin_memory()
    feeder = HostFeeder(static, lambda i: hb[i % len(hb)])
    inline = (args.feed == 'inline')                       # inline: H2D straight into the graph inputs on the compute stream

    def feed(i, prefetch):
        if inline:
            for s_, h_ in zip(static, hb[i % len(hb)]):
                s_.copy_(h_, non_blocking=True)
        else:
            feeder.feed(i, prefetch=prefetch)

    for i in range(2):
        feed(i, False)
        one_step()
    torch.cuda.synchronize(); cdist.barrier()
    feeder.next = None
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for i in range(steps):
        feed(i, i + 1 < steps)                             # prefetch mode: batch i+1 crosses PCIe while step i computes
        loss = one_step()[0]
        loss_host.copy_(loss.reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()          # the reference reads loss.item() every step
    f1.record()
    torch.cuda.synchronize(); cdist.barrier()
    ms_e2e = cdist.max_over_ranks(f0.elapsed_time(f1), dev)
    res = dict(ms_total=ms_total, ms_e2e=ms_e2e, steps=steps, warm=warm, launches_per_step=int(launches_per_step),
               in_bytes=in_bytes, loss=float(loss_host[0]), clocks=clocks, use_graph=use_graph, prof={})
    # the profile pass runs whole (eager) steps, all-reduce included: EVERY rank must take part
    if full and not args.no_profile:
        _say('%s: profile pass' % cfg)
        res['prof'] = profile_pass(trainer, tgt, refs, K, Kinv)
    del trainer, feeder
    pyramid.clear()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    from cc_b200 import dist as cdist
    wd = float(os.environ.get('CCB_BENCH_WATCHDOG', '0'))
    if wd > 0:                                              # dump every thread's Python stack and exit instead of hanging
        import faulthandler
        faulthandler.dump_traceback_later(wd, exit=True, file=sys.stderr)
    _say('init process group')
    rank, local, world = cdist.init_from_env()
    assert world == args.gpus, 'WORLD_SIZE %d != --gpus %d (launch with torch.distributed.run)' % (world, args.gpus)
    dev = torch.device('cuda', local)
    torch.cuda.set_device(dev)
    numa_bound = cdist.bind_to_gpu_numa(local) if world > 1 else False
    B = PER_GPU_BATCH
    m = measure_cfg(args.cfg, args, dev, rank, local, world, args.steps, full=True)
    # the other BASELINE.json single-GPU configurations ride along as extra keys (N=1 only: scaling runs stay short)
    side = {}
    if world == 1 and not args.no_side_configs:
        for c in ('cfg1', 'cfg2', 'cfg3'):
            if c != args.cfg:
                side[c] = measure_cfg(c, args, dev, rank, local, world, args.steps, full=False)
    ref_gpu = None
    if world == 1 and not args.no_reference_gpu:
        _say('reference on the GPU')
        try:
            ref_gpu = reference_gpu(args.cfg, dev)
        except Exception as exc:                            # context number only: never lose the bench line over it
            ref_gpu = {'error': repr(exc)[:300]}
    _say('done')
    out = None
    if rank == 0:
        pk = peaks()
        tps = lambda ms, k: world * B * k / (ms * 1e-3)
        out = {
            'metric': 'train-step triplets/sec at 256x832x6lvl', 'value': tps(m['ms_total'], m['steps']), 'unit': 'triplets/s',
            'n_gpus': world, 'steps': m['steps'], 'warmup': m['warm'], 'ms_per_step': m['ms_total'] / m['steps'],
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': CFG_WORKLOAD[args.cfg], 'global_batch': world * B, 'per_gpu_batch': B,
                       'frame': '%dx%d' % (H, W), 'levels': NLEVELS, 'parallelism': 'dp%d' % world,
                       'conv_math': 'tcgen05 kind::tf32 x3 split precision (fp32-accurate, <=1e-4 parity)', 'cuda_graph': m['use_graph'],
                       'numa_bound': numa_bound,
                       'l2_policy': 'inputs and activations (>1 GB/step) exceed the 126 MB L2; no explicit flush',
                       'e2e_input_path': ('pinned host batch -> H2D on a copy stream one step ahead (HostFeeder) -> D2D into the graph inputs; '
                                          'all steps+copies inside the timed region') if args.feed == 'prefetch' else
                                         'pinned host batch -> H2D into the graph inputs on the compute stream'},
            'e2e': {'value': tps(m['ms_e2e'], m['steps']), 'unit': 'triplets/s', 'h2d_bytes_per_step': m['in_bytes'], 'd2h_bytes_per_step': 4,
                    'ms_per_step': m['ms_e2e'] / m['steps']},
            'gpu_launches': int(m['launches_per_step'] * m['steps']), 'gpu_launches_per_step': m['launches_per_step'],
            'clocks': m['clocks'], 'loss': m['loss'], 'peaks': pk,
        }
        out.update(m['prof'].get('json', {}))
        if side:
            out['configs'] = {c: {'workload': CFG_WORKLOAD[c], 'value': tps(r['ms_total'], r['steps']), 'unit': 'triplets/s',
                                  'ms_per_step': r['ms_total'] / r['steps'], 'steps': r['steps'],
                                  'e2e': {'value': tps(r['ms_e2e'], r['steps']), 'ms_per_step': r['ms_e2e'] / r['steps'],
                                          'h2d_bytes_per_step': r['in_bytes'], 'd2h_bytes_per_step': 4},
                                  'gpu_launches_per_step': r['launches_per_step'], 'loss': r['loss']} for c, r in side.items()}
        if ref_gpu is not None:
            out['reference_gpu'] = ref_gpu
        if world == 1 and not args.no_cpu_baseline:
            out['cpu_baseline'] = cpu_baseline(args.cfg, budget_s=25.0)
    return out


def _state_tensors(trainer):
    return [t for net in trainer.nets.values() for t in list(net.parameters()) + list(net.buffers())]


def initial_state(trainer):
    """Copies of the trainer's parameters and buffers as built from the seed, tensor by tensor (the optimiser's flat
    layout may be re-packed by the first data-parallel step)."""
    return [t.detach().clone() for t in _state_tensors(trainer)]


def reset_state(trainer, init):
    """Back to initial_state(): parameters and buffers restored, Adam moments and step count zero as after construction."""
    with torch.no_grad():
        for t, v in zip(_state_tensors(trainer), init):
            t.copy_(v)
        for buf in (trainer.opt.exp_avg, trainer.opt.exp_avg_sq, trainer.opt.state):
            buf.zero_()
    trainer.refresh_weights()


def dump_outputs(out_dir, trainer, loss, aux, budget=64 * 10 ** 6):
    """What the last timed step computed, as float32 out_dir/<name>.npy: the loss, the loss terms and network outputs it
    returns (aux), the parameter gradients of its backward and the BatchNorm statistics it leaves (one flat array per net).
    The step starts from the seeded initial state (measure_cfg).  At most `budget` bytes in all: every array larger than a
    common cap keeps a fixed, seeded sample of its flattened elements (the same indices whenever the sizes are the same)."""
    import numpy as np
    arrs = {'loss': loss}
    for k, v in aux.items():
        if isinstance(v, (list, tuple)):
            arrs.update({'%s_%d' % (k, i): t for i, t in enumerate(v)})
        elif torch.is_tensor(v):
            arrs[k] = v
    for n, net in trainer.nets.items():
        arrs['grads_' + n] = torch.cat([(p._ccb_grad if getattr(p, '_ccb_grad', None) is not None else torch.zeros_like(p))
                                        .reshape(-1) for p in net.parameters()])
        bufs = [b.reshape(-1) for b in net.buffers() if b.is_floating_point()]
        if bufs:
            arrs['buffers_' + n] = torch.cat(bufs)
    # the largest cap that keeps the total within budget: arrays at or under it are written whole
    left, cap = (budget - 128 * len(arrs)) // 4, None
    sizes = sorted(t.numel() for t in arrs.values())
    for i, n in enumerate(sizes):
        if n * (len(sizes) - i) > left:
            cap = left // (len(sizes) - i)
            break
        left -= n
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrs.items():
        t = t.detach()
        if cap is not None and t.numel() > cap:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), cap, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(out_dir, name + '.npy'), t.float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------
def profile_pass(trainer, tgt, refs, K, Kinv, steps=2):
    """Per-entry-point CUDA-event timing of the step (eager, on the launching stream) -> kernel shares,
    and the roofline objects for the dominant family and for the fused warp+loss kernels."""
    from cc_b200 import _lib, pyramid
    pk = peaks()
    records = []
    real = _lib.lib()

    class Proxy:
        def __getattr__(self, name):
            fn = getattr(real, name)
            if not name.startswith('ccb_') or name.endswith('_floats') or name in ('ccb_launch_count', 'ccb_last_error_string'):
                return fn

            def wrapped(*a):
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                rc = fn(*a)
                e.record()
                kern = None
                if name.startswith('ccb_conv2d_'):
                    kern = (real.ccb_debug_last_conv_kernel() or b'').decode() + ':' + name[len('ccb_conv2d_'):]
                records.append((name, a[0], s, e, kern))
                return rc
            return wrapped

    saved = _lib._lib
    for it in range(steps + 1):
        if it == 1:
            records.clear()
        _lib._lib = Proxy()
        try:
            pyramid.clear()
            trainer.step(tgt, refs, K, Kinv)
        finally:
            _lib._lib = saved
        torch.cuda.synchronize()
    fam, kern_ms = {}, {}
    for name, a0, s, e, kern in records:
        ms = s.elapsed_time(e)
        f = fam.setdefault(name, dict(ms=0.0, calls=0, flops=0.0, bytes=0.0))
        f['ms'] += ms
        f['calls'] += 1
        if name.startswith('ccb_conv2d_'):
            d = a0._obj if hasattr(a0, '_obj') else a0
            fl = 2.0 * d.B * d.Co * d.Ho * d.Wo * d.Ci * d.kh * d.kw
            f['flops'] += fl
            k = kern_ms.setdefault(kern, dict(ms=0.0, calls=0, flops=0.0))
            k['ms'] += ms; k['calls'] += 1; k['flops'] += fl
        elif name.startswith('ccb_photo_loss_'):
            d = a0._obj if hasattr(a0, '_obj') else a0
            px = sum(d.B * d.h[l] * d.w[l] for l in range(d.nlevels))
            # SURVEY 8(d): rigid 80 B/px fwd (+20 bwd) with mask; 64 (+4) without; flow 60 (+24)
            if d.mode == 0:
                per = (80 if d.has_mask else 64) if name.endswith('fwd') else (20 if d.has_mask else 4)
            else:
                per = (60 if d.has_mask else 52) if name.endswith('fwd') else (24 if d.has_mask else 16)
            f['bytes'] += float(px) * per
    total = sum(f['ms'] for f in fam.values())
    conv = {k: v for k, v in fam.items() if k.startswith('ccb_conv2d_')}
    conv_ms = sum(v['ms'] for v in conv.values())
    conv_flops = sum(v['flops'] for v in conv.values())
    photo = {k: v for k, v in fam.items() if k.startswith('ccb_photo_loss_')}
    photo_ms = sum(v['ms'] for v in photo.values())
    photo_bytes = sum(v['bytes'] for v in photo.values())
    js = {}
    if conv_ms > 0:
        ach = conv_flops / (conv_ms * 1e-3) / 1e12
        js['roofline'] = {'bound': 'tensor', 'kernel': 'conv2d fprop+dgrad+wgrad (implicit GEMM)', 'achieved': ach,
                          'peak': pk['tensor_sustained'], 'unit': 'TFLOP/s', 'frac': ach / pk['tensor_sustained'],
                          'traffic': None, 'share_of_step': conv_ms / total, 'launches': sum(v['calls'] for v in conv.values()) // steps,
                          'executed_tensor_tflops': 3.0 * ach,
                          'peak_source': pk['source'] + ' bf16 sustained; achieved counts ALGORITHMIC flops - the fp32-accurate path '
                                         'executes 3 tf32 MMAs per product (tf32 dense peak = bf16 / 2), see DESIGN.md'}
    if photo_ms > 0:
        ach = photo_bytes / (photo_ms * 1e-3) / 1e9
        js['roofline_warploss'] = {'bound': 'hbm', 'kernel': 'photo_fwd+photo_bwd (fused warp+SSIM+loss)', 'achieved': ach,
                                   'peak': pk['hbm'], 'unit': 'GB/s', 'frac': ach / pk['hbm'], 'traffic': None,
                                   'share_of_step': photo_ms / total, 'peak_source': pk['source']}
    # `roofline` = the heaviest single kernel, timed alone (spec); the aggregated convolution family moves to
    # `roofline_family` (its share of the step is what explains the headline)
    # live shares of the convolution kernels: CUDA events around every conv call of the eager step, bucketed by the kernel the
    # call dispatched to (ccb_debug_last_conv_kernel); a call's time includes its helper launches (layout copy, split-K sum)
    js['conv_kernel_shares'] = {k: {'share_of_step': round(v['ms'] / total, 4), 'calls_per_step': v['calls'] // steps,
                                    'algorithmic_tflops': round(v['flops'] / (v['ms'] * 1e-3) / 1e12, 1)}
                                for k, v in sorted(kern_ms.items(), key=lambda kv: -kv[1]['ms'])}
    try:
        single = single_kernel_roofline(pk)
        nh = [v for k, v in kern_ms.items() if k.startswith('conv_nhwc')]
        if nh:
            single['share_of_step'] = sum(v['ms'] for v in nh) / total
            single['share_source'] = 'live: CUDA events around every conv call of the profiled eager step that dispatched to conv_nhwc_kernel (fprop + dgrad)'

        if 'roofline' in js:
            js['roofline_family'] = js['roofline']
            single['family_share_of_step'] = js['roofline']['share_of_step']
        js['roofline'] = single
    except Exception as exc:                               # never lose the bench line over the side measurement
        js['roofline_kernel_error'] = repr(exc)[:200]
    js['kernel_shares'] = {k: round(v['ms'] / total, 4) for k, v in sorted(fam.items(), key=lambda kv: -kv[1]['ms'])[:8]}
    js['profiled_step_ms'] = total / steps
    return {'json': js}


def single_kernel_roofline(pk, iters=20):
    """The heaviest single convolution of the step, alone: DispResNet6's 7x7 32->32 layer (b4, 128x416, 21.4 GFLOP), which
    the dispatcher gives to conv_nhwc_kernel (channels-last slab kernel).  Duration = CUDA events around `iters` calls on
    the launching stream - a call = NCHW->NHWC copy + weight preparation + the kernel, as in the step (inputs 27 MB +
    outputs 27 MB per launch).  DRAM traffic = the committed ncu --set full capture of the same launch
    (profiles/r02_ncu_nhwc_7x7.txt), labelled as such; null if that file is absent."""
    from cc_b200 import nn as cnn, _lib
    dev = torch.device('cuda', torch.cuda.current_device())
    B, C, Hh, Ww, k = PER_GPU_BATCH, 32, H // 2, W // 2, 7
    x = torch.randn(B, C, Hh, Ww, device=dev)
    w = torch.randn(C, C, k, k, device=dev) * 0.05
    b = torch.zeros(C, device=dev)
    with torch.no_grad():
        for _ in range(3):
            cnn.conv2d(x, w, b, None, 1, 3, 'relu')
        kern = (_lib.lib().ccb_debug_last_conv_kernel() or b'').decode()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            cnn.conv2d(x, w, b, None, 1, 3, 'relu')
        e1.record()
        torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / iters
    flops = 2.0 * B * C * C * k * k * Hh * Ww
    ach = flops / (us * 1e-6) / 1e12
    traffic, traffic_src = None, None
    try:
        unit = {'byte': 1.0, 'Kbyte': 1e3, 'Mbyte': 1e6, 'Gbyte': 1e9}
        vals = {}
        for line in open(os.path.join(ROOT, 'profiles', 'r02_ncu_nhwc_7x7.txt')):
            f = line.split()
            if len(f) >= 3 and f[0] in ('dram__bytes_read.sum', 'dram__bytes_write.sum'):
                vals[f[0]] = float(f[1]) * unit[f[2]]
        if len(vals) == 2:
            traffic = sum(vals.values())
            traffic_src = 'committed capture profiles/r02_ncu_nhwc_7x7.txt (ncu --set full of this launch, kernel only), not re-measured in this run'
    except Exception:
        pass
    return {'bound': 'tensor', 'kernel': '%s_kernel<3xTF32> + layout copy + weight prep (7x7 32->32 fprop, b%d %dx%d)' % (kern, B, Hh, Ww),
            'share_of_step': None, 'share_source': None,
            'achieved': ach, 'peak': pk['tensor_burst'], 'unit': 'TFLOP/s', 'frac': ach / pk['tensor_burst'],
            'us_per_launch': us, 'algorithmic_flops_per_launch': flops, 'algorithmic_bytes_per_launch': 2.0 * B * C * Hh * Ww * 4,
            'traffic': traffic, 'traffic_source': traffic_src,
            'peak_source': pk['source'] + ' bf16 burst (kernel timed alone); 3 tf32 passes at half the bf16 rate: ceiling = peak / 6'}


# ---------------------------------------------------------------------------------------------------
def pick_cpu_threads():
    """torch CPU ops collapse when every tiny op fans out over 100+ threads (measured: 180 s/step at 128 threads
    vs ~1.3 s at 8): calibrate on a proxy (conv fwd+bwd + one loss-layer call) and use the fastest setting."""
    import torch.nn.functional as F
    from cc_b200 import synth
    from oracle import losses as OL
    n = os.cpu_count() or 1
    cands = sorted({c for c in (4, 8, 16, 32, 64, n) if c <= n})
    x = torch.randn(2, 32, 64, 208, requires_grad=True)
    w = torch.randn(32, 32, 3, 3, requires_grad=True)
    s = synth.sample(2, 64, 208, seed=3, nlevels=3)
    best, best_t = cands[0], float('inf')
    for c in cands:
        torch.set_num_threads(c)
        ts = []
        for _ in range(2):
            t0 = time.perf_counter()
            F.conv2d(x, w, None, 1, 1).sum().backward()
            d = [t.clone().requires_grad_(True) for t in s['depth']]
            OL.photometric_reconstruction_loss(s['tgt'], s['refs'], s['K'], s['Kinv'], d, [None] * 3, s['pose'], wssim=0.9).backward()
            ts.append(time.perf_counter() - t0)
        if min(ts) < best_t:
            best, best_t = c, min(ts)
    torch.set_num_threads(best)
    return best, n


def _ref_module():
    p = os.path.join(ROOT, 'baseline')
    if p not in sys.path:
        sys.path.insert(0, p)
    import ref_step
    return ref_step


def _cpu_step_timer(cfg, B, threads):
    """(run, kind, label): one reference train step on the host cores.  kind "reference" = the UNMODIFIED reference
    modules under baseline/_ref driven by baseline/ref_step.py (stub correlation op); kind "port" = the oracle
    restatement, only when baseline/_ref is absent."""
    from cc_b200 import synth
    torch.set_num_threads(threads)
    tgt, refs = synth.frames(B, H, W, seed=7)
    K, Kinv = synth.intrinsics(B, H, W)
    rs = _ref_module()
    if rs.available():
        r = rs.Ref(cfg, 'cpu')

        def run():
            t0 = time.perf_counter()
            r.step(tgt, refs, K, Kinv)
            return time.perf_counter() - t0
        return run, 'reference', 'unmodified reference modules (baseline/_ref), train.py:454-509,566-568 body, stub correlation op'
    from oracle import step as OS
    P = OS.make_params(cfg)
    opt = OS.Adam(OS.all_params(P), OS.HP['lr'], OS.HP['beta1'], OS.HP['beta2'])

    def run():
        t0 = time.perf_counter()
        OS.train_step(cfg, P, opt, tgt, refs, K, Kinv)
        return time.perf_counter() - t0
    return run, 'port', 'oracle port of the reference step (baseline/_ref absent)'


def cpu_baseline(cfg, budget_s=25.0):
    """The reference step on the host cores, bounded to ~budget_s of CPU work."""
    threads, ncores = pick_cpu_threads()
    B = 2
    run, kind, label = _cpu_step_timer(cfg, B, threads)
    t_first = run()                      # warm-up (allocator, thread pool)
    ts = [run()]
    while sum(ts) + t_first + ts[-1] < budget_s and len(ts) < 5:
        ts.append(run())
    ts.sort()
    t = ts[len(ts) // 2]
    return {'value': B / t, 'unit': 'triplets/s', 'cores': threads, 'kind': kind,
            'sample': '%s step (fwd+bwd+Adam) at b%d 256x832x6lvl: %s; torch CPU fp32, %d threads (fastest of a calibration sweep; box has %d cores), median of %d after 1 warm-up' % (cfg, B, label, threads, ncores, len(ts)),
            's_per_step': t}


def reference_gpu(cfg, dev, steps=5, warm=3):
    """BASELINE.md section 4: the reference PyTorch path itself on this B200 (cudnn.benchmark=True as train.py:299; TF32
    on = the reference's default on this hardware, TF32 off = the parity setting), same batch shape.  Context for
    the north-star's ">= 10x reference PyTorch on 1xB200"; not the denominator of the driver's ratio."""
    from cc_b200 import synth
    rs = _ref_module()
    if not rs.available():
        return {'unavailable': 'baseline/_ref missing'}
    B = PER_GPU_BATCH
    tgt, refs = synth.frames(B, H, W, seed=7)
    K, Kinv = synth.intrinsics(B, H, W)
    tgt, refs, K, Kinv = tgt.to(dev), [r.to(dev) for r in refs], K.to(dev), Kinv.to(dev)
    saved = (torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    out = {'workload': CFG_WORKLOAD[cfg], 'per_gpu_batch': B, 'steps': steps, 'warmup': warm,
           'note': 'unmodified reference modules (baseline/_ref) + pure-torch stub for the absent spatial_correlation_sampler; '
                   'loss.item() every step as train.py:563'}
    try:
        for tf32 in (True, False):
            torch.backends.cudnn.benchmark = True
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            r = rs.Ref(cfg, dev)
            for _ in range(warm):
                r.step(tgt, refs, K, Kinv).item()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                r.step(tgt, refs, K, Kinv).item()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out['tf32_on' if tf32 else 'tf32_off'] = {'ms_per_step': ms, 'value': B / (ms * 1e-3), 'unit': 'triplets/s'}
            if not tf32:
                try:                                            # kernel launches of one reference step
                    from torch.profiler import profile, ProfilerActivity
                    with profile(activities=[ProfilerActivity.CUDA]) as prof:
                        r.step(tgt, refs, K, Kinv).item()
                        torch.cuda.synchronize()
                    out['gpu_launches_per_step'] = sum(int(e.count) for e in prof.key_averages() if e.device_type is not None and 'cuda' in str(e.device_type).lower())
                except Exception as exc:
                    out['gpu_launches_per_step'] = None
                    out['launch_count_error'] = repr(exc)[:120]
            del r
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.benchmark, torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    return out


def run_reference(args):
    """--impl reference: the reference's own CPU implementation of the step (unmodified modules under baseline/_ref,
    driven by baseline/ref_step.py; oracle port only if that copy is absent), all the host threads it can use, rank 0 only."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return None
    threads, ncores = pick_cpu_threads()
    B = 2
    run, kind, label = _cpu_step_timer(args.cfg, B, threads)
    probe = run()
    if probe * (args.steps + args.warmup) > 280 and B > 1:     # keep the whole run within a few minutes
        B = 1
        run, kind, label = _cpu_step_timer(args.cfg, B, threads)
        run()
    for _ in range(max(0, args.warmup - 1)):
        run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run()
    dt = time.perf_counter() - t0
    v = B * args.steps / dt
    return {'impl': 'reference', 'metric': 'train-step triplets/sec at 256x832x6lvl', 'value': v, 'unit': 'triplets/s',
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': CFG_WORKLOAD[args.cfg], 'sample_batch_per_step': B, 'frame': '%dx%d' % (H, W),
                       'levels': NLEVELS, 'device': 'host CPU', 'reference_code': label},
            'cpu_baseline': {'value': v, 'unit': 'triplets/s', 'cores': threads, 'kind': kind,
                             'sample': '%s %s step at b%d per step, %d steps, %d threads (fastest of a sweep; %d cores)' % (label, args.cfg, B, args.steps, threads, ncores)},
            'e2e': {'value': v, 'unit': 'triplets/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cfg', default='cfg3', choices=sorted(CFG_WORKLOAD))
    ap.add_argument('--feed', default='prefetch', choices=['prefetch', 'inline'], help='e2e input path')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-profile', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-side-configs', action='store_true', help='skip the cfg1/cfg2 side measurements (N=1)')
    ap.add_argument('--no-reference-gpu', action='store_true', help='skip the reference-PyTorch-on-this-GPU context run (N=1)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the outputs of the last timed step of --cfg, run from the seeded initial state, as DIR/<name>.npy '
                         '(rank 0, at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    # Contract: rank 0 prints ONE JSON line on stdout.  Libraries chat on fd 1 (NCCL prints its version banner there):
    # park the real stdout, point fd 1 at stderr for the duration of the run, write the line to the real one at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = run_reference(args) if args.impl == 'reference' else run_ours(args)
    sys.stdout.flush()
    if out is not None:
        os.write(real_stdout, (json.dumps(out) + '\n').encode())
    if args.impl == 'ours' and int(os.environ.get('WORLD_SIZE', '1')) > 1:
        # A captured CUDA graph that contains the NCCL all-reduce keeps the communicator busy: destroy_process_group()
        # blocks forever on it (observed on 2xB200).  The result is printed; leave without the teardown.
        torch.cuda.synchronize()
        torch.distributed.barrier()
        sys.stderr.flush()
        os._exit(0)


if __name__ == '__main__':
    main()
