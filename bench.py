#!/usr/bin/env python
"""Benchmark of the ReconfigISP hot path on B200 (driver contract: one JSON line on stdout from rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload tuning|search] [--impl b200|reference|torch_eager]
                  [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...          (one rank per GPU, weak scaling)

--workload tuning (default) = BASELINE.json configs[1], the configuration `metric` is quoted on: one proxy-tuning step
  (forward + MSE + gradients of every stage parameter + Adam update) of the fixed all-classical pipeline
  Bayer_02_Demosaic_02_sRGB_11_13_01_14 (skip | bilinear demosaic | wb-manual | wb-quadratic | gamma | gtm-manual;
  SURVEY.md §8d) on 4 synthetic 12 MP RGGB raws per GPU.  Metric: ISP-stack MP/s, fwd+bwd (MP = N*H*W of the raw frame).
--workload search = configs[2]/[4]: one DARTS search iteration of the supernet (n_step=3, threshold 0.2, alpha=0: 2+4+45
  candidates; optimize_alphas + optimize_parameters = 5 supernet forward+backward passes, codes/train.py:201-215,
  darts_model.py:224-324) on 256x256 raw patches, per-GPU batch fixed.  Metric: MP/s through one supernet fwd+bwd pass.

  value        steps with the inputs already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e          the same step through the public model API from PINNED HOST buffers: feed_data() (H2D, double-buffered on a
               copy stream) -> optimize_parameters() -> loss.item() (D2H) every step.  The loaders' integer codes cross
               PCIe (u16 raw, u8 GT: 5 B/px) and are normalised on the device; `e2e_fp32` moves fp32 (16 B/px)
  roofline     the dominant kernel alone: algorithmic bytes (or FLOPs) / CUDA-event time vs the measured peak
  cpu_baseline the oracle port of the same path on the host cores, bounded sample (rank 0, N=1 only)
  --impl reference    times that CPU port as its own arm (rank 0 only under torchrun)
  --impl torch_eager  the same pipeline as stock torch ops + autograd on the B200 (BASELINE.md's "number to beat")
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ARCH = 'Bayer_02_Demosaic_02_sRGB_11_13_01_14'
ARCH_LIGHT = 'Bayer_02_Demosaic_02_sRGB_01_14'      # gamma -> tone curve (the yolo pipeline's classical tail)
H, W = 3000, 4000
FRAMES_PER_GPU = 4
ALGO_BYTES_PER_PX = 16          # read raw 4 B + GT 12 B; nothing but ~100 floats is written (DESIGN.md)
METRIC = 'ISP-stack MP/s fwd+bwd (fixed pipeline proxy-tuning step, synthetic 12MP RGGB raws)'
METRIC_SEARCH = 'DARTS supernet search MP/s (raw pixels through one supernet fwd+bwd pass; an iteration = 5 passes, 51 candidates)'
SEARCH_PATCH = 256
SEARCH_BATCH = 64               # per GPU: the size that fills a B200 (the reference's 4 x 256^2 is reported beside it)
SM_CLOCK_HZ, SMS = 1.965e9, 148


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j['hbm_gbs']), float(j['bf16_tflops']), 'measured (MEASURED_PEAKS.json)'
        except Exception:
            pass
    return 6650.0, 1590.0, 'fallback (B200_PROFILING.md)'


def static_profile():
    """Per-launch DRAM bytes / executed instructions of the step kernel from the committed ncu capture (static, labelled)."""
    p = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    try:
        return json.load(open(p))
    except Exception:
        return {}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([f.strip() for f in out.split(',')])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith('active')})
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(self.samples)}


def opt_tuning(arch=ARCH):
    return {'model': 'isp', 'is_train': True,
            'network_G': {'which_model_G': 'OriginUniversal', 'architecture': arch, 'weight_seed': 10},
            'train': {'lr_G': 1e-3, 'beta1': 0.9, 'beta2': 0.99, 'pixel_criterion': 'l2', 'lr_scheme': 'MultiStepLR',
                      'lr_steps': [20000, 40000, 60000], 'lr_gamma': 0.5},
            'path': {'pretrain_model_G': None}}


def opt_search():
    return {'model': 'darts', 'network_G': {'which_model_G': 'SuperPruneFifteenDemosFourBayerTwo', 'n_step': 3, 'n_modules': 15,
                                           'prune_threshold': 0.2, 'weight_seed': 10},
            'train': {'lr_G': 1e-3, 'momentum_G': 0.9, 'lr_meta': 1e-3, 'beta1': 0.9, 'beta2': 0.999, 'pixel_criterion': 'l2'}}


# ---- CPU arms (oracle port of the reference path; the only place bench.py executes oracle/) ---------------------------
def cpu_tuning_rate(sample_hw, reps, threads=None, warmup=1):
    """fwd + MSE + backward of the stage parameters on one frame of `sample_hw`, `warmup` untimed then `reps` timed.
    -> (MP/s, cores, seconds per rep)."""
    import torch
    from oracle import pipeline_oracle as PO
    from reconfigisp_b200.synthetic import synthetic_frames
    cores = threads or os.cpu_count()
    torch.set_num_threads(cores)
    h, w = sample_hw
    raw, gt = synthetic_frames(1, h, w, seed=10)
    pipe = PO.FixedPipeline(ARCH, 'origin', 10)

    def step():
        y, _ = pipe.forward(raw)
        loss = ((y - gt) ** 2).mean()
        nz = [l for l in pipe.logits if l.numel()]
        torch.autograd.grad(loss, nz)
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(reps):
        step()
    dt = (time.perf_counter() - t0) / reps
    return h * w / 1e6 / dt, torch.get_num_threads(), dt


def cpu_search_rate(batch, size, reps, warmup=0):
    """One DARTS iteration (5 supernet fwd+bwd passes) of the oracle supernet on `batch` patches of `size`^2, `warmup` untimed
    then `reps` timed.  -> (MP/s per pass, cores, seconds per iteration)."""
    import torch
    from oracle import pipeline_oracle as PO
    from reconfigisp_b200.synthetic import synthetic_frames
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    raw, gt = synthetic_frames(2 * batch, size, size, seed=10)
    netG, netV = PO.Supernet(3, 0.2, 10), PO.Supernet(3, 0.2, 10)

    def it():
        PO.darts_step(netG, netV, raw[:batch], gt[:batch], raw[batch:], gt[batch:], 1e-3, 0.9, 1e-3)
    for _ in range(warmup):
        it()
    t0 = time.perf_counter()
    for _ in range(reps):
        it()
    dt = (time.perf_counter() - t0) / reps
    return 5 * batch * size * size / 1e6 / dt, torch.get_num_threads(), dt


def run_reference(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return 0
    if args.workload == 'search':
        # a step = one DARTS iteration of the CPU port on a bounded sample (2 patches of 64x64 take seconds: the supernet runs
        # 51 candidates incl. median / NLM / bilateral five times)
        rate, cores, dt = cpu_search_rate(2, 64, args.steps, args.warmup)
        sample = '2+2 patches of 64x64 per iteration (train/val halves), %d iterations after %d warm-up (oracle/pipeline_oracle.py ' \
                 'darts_step, torch CPU)' % (args.steps, args.warmup)
        metric, workload = METRIC_SEARCH, 'configs[2]: DARTS search iteration, n_step=3, 51 candidates; CPU sample: %s' % sample
    else:
        # a step = one fwd+bwd of the CPU port on a bounded crop of one 12 MP frame, sized from a probe so that the whole
        # --steps/--warmup run stays within ~2 minutes
        _, _, probe_dt = cpu_tuning_rate((752, 1000), 1)
        n = args.steps + args.warmup
        scale = min(4.0, max(0.25, (120.0 / n) / max(probe_dt, 1e-3)))         # pixels relative to the probe crop
        hw = (int(752 * scale ** 0.5) // 2 * 2, int(1000 * scale ** 0.5) // 4 * 4)
        rate, cores, dt = cpu_tuning_rate(hw, args.steps, warmup=args.warmup)
        sample = '1 frame crop of %dx%d per step (oracle/pipeline_oracle.py FixedPipeline, torch CPU)' % hw
        metric, workload = METRIC, 'configs[1]: fixed pipeline %s fwd+bwd (proxy tuning), 12MP RGGB raws; CPU sample: %s' % (ARCH, sample)
    line = {'impl': 'reference', 'metric': metric, 'value': round(rate, 3), 'unit': 'MP/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': round(dt * 1e3, 2), 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {'workload': workload},
            'cpu_baseline': {'value': round(rate, 3), 'unit': 'MP/s', 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': round(rate, 3), 'unit': 'MP/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line), flush=True)
    return 0


# ---- helpers of the GPU arms ------------------------------------------------------------------------------------------
class Timer:
    def __init__(self, torch, dist, world, dev):
        self.torch, self.dist, self.world, self.dev = torch, dist, world, dev

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def __call__(self, fn, steps, warmup):
        """ms for `steps` calls of fn: barrier + synchronize on both sides, CUDA events, MAX over ranks."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms.item())


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(net, params, **scalars):
    """Host float32 copies of what a training step hands its caller: the given device scalars (the loss) and, by parameter
    name, every trainable tensor after the update (`param.<name>`) with the gradient the step computed for it (`grad.<name>`)."""
    keep = {id(p) for p in params}
    out = dict(scalars)
    for name, p in net.named_parameters():
        if id(p) in keep and p.numel():
            out['param.' + name] = p
            if p.grad is not None:
                out['grad.' + name] = p.grad
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def dump_outputs(path, arrays):
    import numpy as np
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError('--dump-outputs: %d bytes exceed the %d-byte limit' % (total, DUMP_LIMIT_BYTES))
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + '.npy'), a)


def teardown(world, dist, models):
    if world > 1:
        # teardown must never hold the job: release the captured graphs first, and leave hard if NCCL teardown stalls
        import torch
        for m in models:
            m.__dict__.pop('_graphs', None)
            m._graph = None
        torch.cuda.synchronize()
        watchdog = threading.Timer(60.0, lambda: os._exit(0))
        watchdog.daemon = True
        watchdog.start()
        dist.barrier()
        dist.destroy_process_group()
        watchdog.cancel()


# ---- workload: proxy tuning of the fixed pipeline (configs[1]) -----------------------------------------------------------
def run_tuning(args):
    import torch
    import torch.distributed as dist
    from reconfigisp_b200 import dist as D
    from reconfigisp_b200 import _lib as L
    from reconfigisp_b200 import ops
    from reconfigisp_b200.synthetic import synthetic_frames
    from reconfigisp_b200.tuning import IspModel

    local = int(os.environ.get('LOCAL_RANK', '0'))
    numa = D.bind_to_gpu_numa_node(local)          # before any pinned allocation
    rank, world, local = D.init_from_env('nccl')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    timed = Timer(torch, dist, world, dev)
    B = args.frames
    raw_h, gt_h = synthetic_frames(B, H, W, seed=10 + rank, pin=True)
    model = IspModel(opt_tuning())
    px = B * H * W
    hbm_peak, _, peak_src = peaks()

    # ---- value: inputs resident in HBM ------------------------------------------------------------------------
    model.feed_data((raw_h.to(dev), gt_h.to(dev)))
    torch.cuda.synchronize()
    sampler = ClockSampler(local)
    sampler.start()
    ms_step = timed(model.optimize_parameters, args.steps, args.warmup) / args.steps
    value = world * px / 1e6 / (ms_step / 1e3)
    # taken now: the legs below keep training the same model
    outputs = step_outputs(model.netG, model.netG.trainable_parameters, loss=model.log_dict['loss']) if args.dump_outputs else None

    # ---- e2e: host buffers through the public API; the copy of batch k+1 overlaps the step of batch k ------------
    def e2e_loop(batches):
        state = {'k': 0}
        model.feed_data(batches[0])

        def step():
            model.optimize_parameters()
            state['k'] += 1
            model.feed_data(batches[state['k'] % len(batches)])      # next batch: H2D on the copy stream, other buffer set
            return float(model.log_dict['loss'].item())              # D2H of this step's loss
        return step
    n_e2e = max(2, min(args.steps, 40))
    raw_c = torch.round(raw_h * 1023).to(torch.int16).pin_memory()
    gt_c = torch.round(gt_h * 255).to(torch.uint8).pin_memory()
    ms_codec = timed(e2e_loop([(raw_c, gt_c)]), n_e2e, 4) / n_e2e
    ms_fp32 = timed(e2e_loop([(raw_h, gt_h)]), n_e2e, 4) / n_e2e
    model.feed_data((model._bufs['img0'], model._bufs['gt0']))        # back to resident device tensors
    torch.cuda.synchronize()

    # ---- roofline of the dominant kernel (and its launches per step) -------------------------------------------------
    dm_kind, chain, keep = model.netG.fused_mse_step_plan()
    step = ops.PipelineStep(B, H, W, dm_kind, chain, dev)
    with torch.no_grad():
        table = model.netG._segment_table(keep, B).contiguous()
    l0 = L.size('risp_launch_count')
    step(model.img, model.gt, table)
    kernels_per_step = L.size('risp_launch_count') - l0              # prep + fused step kernel + finaliser
    ms_k = timed(lambda: step(model.img, model.gt, table), args.steps, args.warmup) / args.steps
    n_f = max(10, args.steps // 4)
    with torch.no_grad():
        ms_f = timed(lambda: ops.pipeline_fwd(model.img, dm_kind, chain, table), n_f, args.warmup) / n_f
        ms_d = timed(lambda: ops.demosaic(model.img, dm_kind), n_f, args.warmup) / n_f
    # ---- the same step kernel on a lighter shipped chain (gamma -> tone curve): the memory-bound regime -----------------
    light = IspModel(opt_tuning(ARCH_LIGHT))
    dm_l, chain_l, keep_l = light.netG.fused_mse_step_plan()
    step_l = ops.PipelineStep(B, H, W, dm_l, chain_l, dev)
    with torch.no_grad():
        table_l = light.netG._segment_table(keep_l, B).contiguous()
    ms_l = timed(lambda: step_l(model.img, model.gt, table_l), args.steps, args.warmup) / args.steps
    clocks = sampler.summary()          # sampled across all timed legs
    achieved = ALGO_BYTES_PER_PX * px / (ms_k / 1e3) / 1e9
    prof = static_profile()

    def frac(ms):
        return round(ALGO_BYTES_PER_PX * px / (ms / 1e3) / 1e9 / hbm_peak, 4)

    line = None
    if rank == 0:
        roof = {'bound': 'hbm', 'achieved': round(achieved, 1), 'peak': hbm_peak, 'unit': 'GB/s', 'frac': round(achieved / hbm_peak, 4),
                'traffic': None, 'kernel': 'risp::fused::fused_kernel<BILINEAR, STEP, gain|poly10|gamma|gtm>',
                'ms_per_launch': round(ms_k, 4), 'algorithmic_bytes_per_px': ALGO_BYTES_PER_PX}
        if prof.get('step_dram_bytes_per_px'):
            roof['traffic'] = prof['step_dram_bytes_per_px'] * px
            roof['traffic_source'] = 'profiles/r2_traffic.json: ncu --set full capture of this kernel at the same shape (static, not measured in this run)'
        fp32 = None
        if prof.get('step_thread_instr_per_px'):
            ips = prof['step_thread_instr_per_px'] * px / (ms_k / 1e3)
            fp32 = {'bound': 'issue', 'achieved': round(ips / 1e12, 2), 'peak': round(SMS * 128 * SM_CLOCK_HZ / 1e12, 2), 'unit': 'T thread-instr/s',
                    'frac': round(ips / (SMS * 128 * SM_CLOCK_HZ), 4), 'thread_instr_per_px': prof['step_thread_instr_per_px'],
                    'pipe_fma_pct_ncu': prof.get('step_pipe_fma_pct'), 'issue_active_pct_ncu': prof.get('step_issue_active_pct'),
                    'note': 'the step kernel is bound by the fp32 pipe and the dependent chains of its 37-parameter stage stack, not by HBM: '
                            'executed thread-instructions per pixel (ncu, static) x pixels / measured time vs 148 SMs x 128 lanes x 1.965 GHz; '
                            'a packed FFMA2/FMUL2 holds the FMA pipe for two cycles (profiles/r2_fma_rates.txt), so the pipe is busier '
                            'than the issue slots (pipe_fma_pct_ncu, static from the same capture)'}
        line = {'metric': METRIC, 'value': round(value, 1), 'unit': 'MP/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': round(ms_step, 4), 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': {'workload': 'configs[1]: fixed pipeline %s fwd+bwd (proxy tuning), %d x 12MP RGGB raws per GPU' % (ARCH, B),
                           'frame': [H, W], 'frames_per_gpu': B, 'parallelism': 'dp%d (frames sharded, one in-place all-reduce of the flat gradient buffer)' % world,
                           'l2': 'inputs %.0f MB per step > 126 MB L2 (no flush needed)' % ((4 + 12) * px / 1e6),
                           'peak_source': peak_src, 'numa_node': numa},
                'clocks': clocks,
                'e2e': {'value': round(world * px / 1e6 / (ms_codec / 1e3), 1), 'unit': 'MP/s', 'h2d_bytes_per_step': 5 * px,
                        'd2h_bytes_per_step': 4, 'ms_per_step': round(ms_codec, 3),
                        'note': 'IspModel.feed_data (pinned host u16 raw codes + u8 GT, decoded on the device, double-buffered on a copy '
                                'stream) -> optimize_parameters -> loss.item() every step'},
                'e2e_fp32': {'value': round(world * px / 1e6 / (ms_fp32 / 1e3), 1), 'unit': 'MP/s', 'h2d_bytes_per_step': 16 * px,
                             'd2h_bytes_per_step': 4, 'ms_per_step': round(ms_fp32, 3), 'note': 'same loop with fp32 host tensors (the reference loaders\' format)'},
                'fwd': {'value': round(world * px / 1e6 / (ms_f / 1e3), 1), 'unit': 'MP/s', 'ms_per_step': round(ms_f, 4), 'roofline_frac': frac(ms_f),
                        'note': 'fused inference of the same pipeline (demosaic + 4 stages in one pass, read raw 4 B + write BGR 12 B per px), data resident; '
                                'the plain 4r+12w streaming kernel of scripts/micro/stream_mix.cu reaches 0.84 of the copy peak'},
                'demosaic': {'ms_per_step': round(ms_d, 4), 'roofline_frac': frac(ms_d), 'note': 'bilinear demosaic alone through the same kernel (16 B/px)'},
                'light_pipeline': {'arch': ARCH_LIGHT, 'ms_per_step': round(ms_l, 4), 'roofline_frac': frac(ms_l),
                                   'value': round(world * px / 1e6 / (ms_l / 1e3), 1), 'unit': 'MP/s',
                                   'note': 'the same fused fwd+bwd step kernel on the gamma -> tone-curve chain (4 parameters): memory-bound regime'},
                'gpu_launches': kernels_per_step * args.steps,
                'gpu_launches_note': '%d kernels of this library per step (parameter preparation, fused step, finaliser) + torch\'s sigmoid/scale table, '
                                     'backward glue and fused Adam, all replayed from one CUDA graph' % kernels_per_step,
                'roofline': roof}
        if fp32:
            line['roofline_fp32'] = fp32
    if rank == 0 and world == 1 and not args.no_cpu:
        rate, cores, dt = cpu_tuning_rate((H, W), 8)
        line['cpu_baseline'] = {'value': round(rate, 3), 'unit': 'MP/s', 'cores': cores, 'kind': 'port',
                                'sample': '1 frame %dx%d of the workload, 1 warm-up + 8 reps of fwd+bwd = %.1f s '
                                          '(oracle/pipeline_oracle.py FixedPipeline, torch CPU)' % (H, W, 9 * dt)}
    if rank == 0:
        print(json.dumps(line), flush=True)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    teardown(world, dist, [model, light])
    return 0


# ---- workload: DARTS supernet search iteration (configs[2] / [4]) ---------------------------------------------------------
def run_search(args):
    import torch
    import torch.distributed as dist
    from reconfigisp_b200 import dist as D
    from reconfigisp_b200 import _lib as L
    from reconfigisp_b200 import ops
    from reconfigisp_b200.search import DartsModel
    from reconfigisp_b200.synthetic import synthetic_frames

    local = int(os.environ.get('LOCAL_RANK', '0'))
    numa = D.bind_to_gpu_numa_node(local)
    rank, world, local = D.init_from_env('nccl')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    timed = Timer(torch, dist, world, dev)
    hbm_peak, bf16_peak, peak_src = peaks()
    S, B = SEARCH_PATCH, args.batch
    m = DartsModel(opt_search())
    raw, gt = synthetic_frames(2 * B, S, S, seed=10 + rank, pin=True)
    host = (raw[:B], gt[:B], raw[B:], gt[B:])                     # train half / validation half (data_sampler.py:69-150)
    m.feed_data(tuple(t.to(dev) for t in host))

    def it():
        m.optimize_alphas()
        m.optimize_parameters()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = L.size('risp_launch_count')
    it()
    own_launches = L.size('risp_launch_count') - l0
    steps = args.steps
    ms_it = timed(it, steps, min(args.warmup, 3)) / steps
    px = B * S * S
    value = world * 5 * px / 1e6 / (ms_it / 1e3)
    outputs = None
    if args.dump_outputs:
        # taken now: the legs below keep searching with the same model
        outputs = step_outputs(m.netG, list(m.netG.trainable_parameters) + list(m.netG.alphas), loss=m.log_dict['loss'],
                               val_loss=m.val_loss)

    def e2e_it():
        m.feed_data(host)
        it()
        return float(m.log_dict['loss'].item())
    n_e = max(1, min(steps, 5))
    ms_e2e = timed(e2e_it, n_e, 1) / n_e

    # the reference's own batch (yolo_search.yml:16-17: 4 patches per GPU)
    m.feed_data(tuple(t[:4].to(dev) for t in host))
    ms_it4 = timed(it, max(2, min(steps, 10)), 2) / max(2, min(steps, 10))

    # ---- roofline (a): the tensor-core convolution that carries the iteration: 64->64 3x3 (Path-Restore body), in isolation
    x = torch.randn(B, 64, S, S, device=dev)
    w = torch.randn(64, 64, 3, 3, device=dev) / 24.0
    bias = torch.zeros(64, device=dev)
    xb = ops.to_blocked(x)
    with torch.no_grad():
        ms_c = timed(lambda: ops.conv2d_tc(xb, w, bias), 10, 3) / 10
    useful_tf = 2.0 * B * S * S * 64 * 64 * 9 / (ms_c / 1e3) / 1e12
    tf32_peak = bf16_peak / 2.0
    # ---- roofline (b): the fused mixed-op of one sRGB step (6 classical candidates in registers + 9 materialised CNN outputs)
    # at 12 MP: fwd 132 B/px, bwd 252 B/px (SURVEY.md §8d)
    mixed = None
    try:
        from reconfigisp_b200.modules.super_prune_fifteen_demos_four_bayer_two import mixed_op_probe
        mixed = mixed_op_probe(timed, 1, 3000, 4000, hbm_peak)
    except Exception as e:                                        # a diagnostic leg must not take the bench line down
        mixed = {'error': str(e)[:200]}
    clocks = sampler.summary()
    line = None
    if rank == 0:
        line = {'metric': METRIC_SEARCH, 'value': round(value, 2), 'unit': 'MP/s', 'n_gpus': world, 'steps': steps, 'warmup': min(args.warmup, 3),
                'ms_per_step': round(ms_it, 2), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32 (CNN candidates: 3xTF32 on tcgen05, fp32-accurate)',
                'data': 'synthetic',
                'config': {'workload': 'configs[2]/[4]: DARTS search iteration (optimize_alphas + optimize_parameters = 5 supernet fwd+bwd passes), '
                                       'n_step=3, threshold 0.2, alpha=0 (2+4+45 candidates), %d+%d patches of %dx%d per GPU' % (B, B, S, S),
                           'patch': S, 'batch_per_gpu': B, 'parallelism': 'dp%d (patches sharded; one flattened all-reduce of alpha+parameter gradients per pass)' % world,
                           'l2': 'activations of one pass: %.1f GB per GPU >> 126 MB L2' % (B * S * S * 4 * 64 * 14 * 9 / 1e9), 'peak_source': peak_src, 'numa_node': numa},
                'clocks': clocks,
                'e2e': {'value': round(world * 5 * px / 1e6 / (ms_e2e / 1e3), 2), 'unit': 'MP/s', 'h2d_bytes_per_step': 2 * 16 * px,
                        'd2h_bytes_per_step': 4, 'ms_per_step': round(ms_e2e, 2)},
                'ref_batch': {'batch_per_gpu': 4, 'ms_per_step': round(ms_it4, 2), 'value': round(world * 5 * 4 * S * S / 1e6 / (ms_it4 / 1e3), 2), 'unit': 'MP/s',
                              'note': 'the reference configuration (4 patches per GPU): launch-latency-bound'},
                'gpu_launches': own_launches * steps,
                'gpu_launches_note': '%d kernels of this library per iteration (counted by risp_launch_count)' % own_launches,
                'roofline': {'bound': 'tensor', 'achieved': round(useful_tf, 1), 'peak': round(tf32_peak, 1), 'unit': 'TFLOP/s', 'frac': round(useful_tf / tf32_peak, 4),
                             'traffic': None, 'kernel': 'risp::conv_tc_kernel 64->64 3x3, %dx%dx%d (tcgen05 kind::tf32)' % (B, S, S), 'ms_per_launch': round(ms_c, 4),
                             'note': 'useful fp32-equivalent FLOPs (2*Cin*Cout*K^2 per px) vs dense TF32 peak = measured bf16 peak / 2; the kernel issues two MMAs '
                                     'per 8 channels (kind::tf32 main term + one bf16 kind::f16 MMA for both cross terms of the hi/lo split) to stay fp32-accurate'},
                'mixed_op': mixed}
    if rank == 0 and world == 1 and not args.no_cpu:
        rate, cores, dt = cpu_search_rate(4, 96, 2)
        line['cpu_baseline'] = {'value': round(rate, 4), 'unit': 'MP/s', 'cores': cores, 'kind': 'port',
                                'sample': '2 iterations on 4+4 patches of 96x96 = %.1f s (oracle/pipeline_oracle.py darts_step, torch CPU)' % (2 * dt)}
    if rank == 0:
        print(json.dumps(line), flush=True)
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
    teardown(world, dist, [])
    return 0


# ---- eager torch on the same B200 (BASELINE.md's "number to beat") -------------------------------------------------------
def run_torch_eager(args):
    if int(os.environ.get('RANK', '0')) != 0:
        return 0
    import torch
    dev = torch.device('cuda', 0)
    from reconfigisp_b200.synthetic import synthetic_frames
    B = args.frames
    raw, gt = synthetic_frames(B, H, W, seed=10)
    raw, gt = raw.to(dev), gt.to(dev)
    # the reference's own expressions (tools_origin.py:326-357 WbQuadratic, :425-438 GtmManual) with a bilinear demosaic by
    # conv2d on the CFA masks, gamma by pow, wb by a broadcast multiply -- stock ATen kernels + autograd
    import torch.nn.functional as F
    k_g = torch.tensor([[0, 1, 0], [1, 4, 1], [0, 1, 0]], device=dev, dtype=torch.float32).view(1, 1, 3, 3) / 4
    k_rb = torch.tensor([[1, 2, 1], [2, 4, 2], [1, 2, 1]], device=dev, dtype=torch.float32).view(1, 1, 3, 3) / 4
    mask = torch.zeros(3, 1, H, W, device=dev)
    mask[2, 0, 0::2, 0::2] = 1; mask[1, 0, 0::2, 1::2] = 1; mask[1, 0, 1::2, 0::2] = 1; mask[0, 0, 1::2, 1::2] = 1    # B,G,R planes
    logits = [torch.zeros(3, device=dev, requires_grad=True), torch.zeros(30, device=dev, requires_grad=True),
              torch.zeros(1, device=dev, requires_grad=True), torch.zeros(3, device=dev, requires_grad=True)]
    with torch.no_grad():
        logits[0].fill_(-1.38); logits[1][6] = logits[1][17] = logits[1][28] = 0.406; logits[3].copy_(torch.tensor([-1.099, 0., 1.099]))
    opt = torch.optim.Adam(logits, 1e-3)

    def forward():
        rp = F.pad(raw, (1, 1, 1, 1), mode='reflect')
        planes = [F.conv2d(rp * F.pad(mask[c:c + 1], (1, 1, 1, 1)), k_g if c == 1 else k_rb) for c in range(3)]
        x = torch.cat(planes, 1)
        x = x * (torch.sigmoid(logits[0]) * 5).view(1, 3, 1, 1)
        b, g, r = x[:, 0:1], x[:, 1:2], x[:, 2:3]
        phi = torch.cat([b * b, g * g, r * r, b * g, b * r, g * r, b, g, r, torch.ones_like(b)], 1)
        P = (torch.sigmoid(logits[1]) * 10 - 5).view(3, 10)
        x = torch.einsum('ck,nkhw->nchw', P, phi).clamp(0, 1)
        x = x.clamp(1e-8, 1) ** torch.sigmoid(logits[2])
        ys = torch.cat([x.new_zeros(1), torch.sigmoid(logits[3]), x.new_ones(1)])
        out = x
        for k in range(4):
            lo, hi = k / 4, (k + 1) / 4
            out = torch.where((x >= lo) & (x < hi), ys[k] + (x - lo) * (ys[k + 1] - ys[k]) * 4, out)
        return out.clamp(0, 1)

    def step():
        opt.zero_grad()
        loss = F.mse_loss(forward(), gt)
        loss.backward()
        opt.step()
    for _ in range(max(1, min(args.warmup, 3))):
        step()
    torch.cuda.synchronize()
    n = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / n
    rate = B * H * W / 1e6 / (ms / 1e3)
    print(json.dumps({'impl': 'torch_eager', 'metric': METRIC, 'value': round(rate, 1), 'unit': 'MP/s', 'n_gpus': 1, 'steps': n, 'warmup': min(args.warmup, 3),
                      'ms_per_step': round(ms, 3), 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                      'config': {'workload': 'configs[1]: the same pipeline %s as stock torch ops + autograd + Adam on one B200, %d x 12MP' % (ARCH, B)},
                      'gpu_launches': 0, 'note': 'reference-style eager PyTorch on the same GPU; none of this repository\'s kernels'}), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None, help='timed steps (default: 200 for tuning, 20 for search)')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'torch_eager'])
    ap.add_argument('--workload', default='tuning', choices=['tuning', 'search'])
    ap.add_argument('--frames', type=int, default=FRAMES_PER_GPU, help='tuning: 12MP frames per GPU per step')
    ap.add_argument('--batch', type=int, default=SEARCH_BATCH, help='search: 256x256 patches per GPU (train half; as many again for validation)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--dump-outputs', metavar='DIR', help='b200: write the loss, the updated parameters and their gradients of the '
                    'last timed step to DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.workload == 'search' else 200        # a search iteration costs ~5000 tuning steps
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs needs --impl b200')
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        return run_reference(args)
    if args.impl == 'torch_eager':
        return run_torch_eager(args)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', str(args.gpus),
               '--master-addr', '127.0.0.1', '--master-port', str(29500 + os.getpid() % 1000), os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    return run_search(args) if args.workload == 'search' else run_tuning(args)


if __name__ == '__main__':
    sys.exit(main())
