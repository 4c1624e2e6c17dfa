"""bench.py -- frames/s of Vid2VidModelG.inference at 2048x1024 (BASELINE config 4:
`--label_nc 35 --loadSize 2048 --n_scales_spatial 3 --use_instance --fg --use_single_G`,
scripts/street/test_2048.sh) on synthetic 35-label sequences with random-init weights.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg4|cfg2|tiny] [--dump-outputs DIR]

A step = one steady-state generated frame (all three scales).  One process per GPU; N > 1 runs N
independent clips (inference has no exchange step: "replicas only", weak scaling) and reports the
whole-job frames/s = N * K / max-over-ranks time.  Prints ONE JSON line on rank 0.

The headline (`value`, `e2e`, `roofline`, `dtype`) is the PRECISE arithmetic mode (split-bf16 x3, fp32-class: the mode
whose outputs match the fp32 reference at images 5e-3 / flow 0.02 px, tests/test_gpu_precise.py); the bf16-operand mode is
measured in the same run and reported beside it under `fast`.

  value        device-resident inputs, CUDA-event timed (what the kernels can do)
  e2e          the public streaming API with HOST buffers: one pinned uint8 label frame -> H2D -> ... -> uint8 RGB frame
               (util.tensor2im on the device) -> D2H into pinned memory, every step inside the timed region
  roofline     the tcgen05 conv kernel: algorithmic conv FLOPs of a frame / summed device time of its launches
               (per-launch CUDA events, v2v_plan_profile) against MEASURED_PEAKS.json dense bf16 (burst)
  cpu_baseline the reference's own Vid2VidModelG.inference (unmodified, vendored into the git-ignored oracle/_ref by
               oracle/make_ref.py; CPU shims of oracle/ref_shim.py) timed on the host cores on a band of one steady-state
               frame of the same workload (kind "reference"; the oracle port, kind "port", only if no reference travelled)
`--impl reference` times the same CPU arm as the reference line.

`--dump-outputs DIR` (inference workloads) writes, for each precision mode, what the last timed step of each timed loop
returned: `<mode>_fake_B.npy` and `<mode>_real_A.npy` from Vid2VidModelG.inference, `<mode>_e2e_rgb.npy` from
inference_stream (the uint8 frame as float32), all on the same fixed seeded sample of DUMP_PIXELS pixel positions
(`sample_pixels.npy`), channels first.  Inputs and weights are seeded, so two builds run with the same arguments can be
compared output for output.
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

WORKLOADS = {
    # name: (W, H, n_scales, ngf, loadSize)
    'cfg4': dict(W=2048, H=1024, n_scales=3, ngf=128, desc='label2city 2048x1024 inference, n_scales_spatial=3 --fg --use_single_G'),
    'cfg2': dict(W=512, H=256, n_scales=1, ngf=128, desc='label2city 512x256 inference (use_single_G), n_scales_spatial=1 --fg'),
    'tiny': dict(W=256, H=128, n_scales=2, ngf=32, desc='plumbing: 256x128, 2 scales, ngf 32'),
    # training steps (train.py:50-93): G + multiscale D + temporal D + FlowNet2 warp losses, one clip per GPU, one flat NCCL
    # gradient all-reduce per step
    'cfg3': dict(W=1024, H=512, n_scales=2, ngf=128, train=True,
                 desc='label2city 1024x512 training step (G + multiscale D + FlowNet2 warp loss), batch-sharded, n_scales_spatial=2'),
    'cfg3_small': dict(W=256, H=128, n_scales=2, ngf=32, train=True, desc='plumbing: 256x128 training step, ngf 32'),
    # the reference-flow network of the training step on its own (models/flownet.py:25-62): FlowNetC -> S -> S || SD -> Fusion
    'flownet2': dict(W=1024, H=512, flownet=True, desc='FlowNet2 (flow, confidence) of one 1024x512 frame pair, 162.5 M parameters'),
}


def make_opt_for(wl):
    from vid2vid_b200.utils import make_opt
    w = WORKLOADS[wl]
    return make_opt(label_nc=35, use_instance=True, fg=True, fg_labels=[26], n_scales_spatial=w['n_scales'], ngf=w['ngf'],
                    use_single_G=True, loadSize=w['W'], dataroot='datasets/Cityscapes/', gpu_ids=[0])


def frame_macs(wl):
    from vid2vid_b200 import networks as NW
    opt = make_opt_for(wl)
    opt.gpu_ids = []
    w = WORKLOADS[wl]
    total = 0.0
    for s in range(w['n_scales']):
        sc = 2 ** (w['n_scales'] - 1 - s)
        total += NW.build_netG(opt, s).conv_macs(1, w['H'] // sc, w['W'] // sc)
    return total


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md): NVML every 50 ms, nvidia-smi fallback."""

    REASONS = {'hw_slowdown': 0x8, 'sw_thermal_slowdown': 0x20, 'hw_thermal_slowdown': 0x40, 'sw_power_cap': 0x4}

    def __init__(self, index, period=0.05):
        super().__init__(daemon=True)
        self.period = period
        self.index, self.sm, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        self.recording = False      # NVML init and the first (slow) queries happen during warm-up, outside the timed region
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    # the same queries whether or not we are recording, so their first-call costs are paid in warm-up
                    clk = self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM)
                    try:
                        mask = self.nvml.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        mask = self.nvml.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    if self.recording:
                        self.sm.append(clk)
                        for n, bit in self.REASONS.items():
                            if mask & bit:
                                self.reasons.add(n)
                    time.sleep(self.period)
                elif not self.recording:
                    time.sleep(0.02)
                else:
                    q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
                        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
                    o = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                       capture_output=True, text=True, timeout=5).stdout.strip().split(',')
                    self.sm.append(int(float(o[0])))
                    self.max_mhz = int(float(o[1]))
                    for n, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], o[2:]):
                        if v.strip().lower().startswith('active'):
                            self.reasons.add(n)
            except Exception:
                time.sleep(0.05)

    def summary(self):
        if not self.sm and self.nvml is not None:        # very short timed region: one sample right after it
            try:
                self.sm.append(self.nvml.nvmlDeviceGetClockInfo(self.h, self.nvml.NVML_CLOCK_SM))
            except Exception:
                pass
        sm = sorted(self.sm)
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(sm)}


def reduce_times(times_ms, world, device='cpu'):
    """Device-timed durations -> the slowest rank's (replicas finish when the last one does).  One all-reduce(MAX) on the
    job's process group (NCCL on the GPU box, gloo in the CPU tests); the data path itself has no collective."""
    import torch
    t = torch.tensor(list(times_ms), device=device, dtype=torch.float64)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return t.tolist()


def peaks():
    """(dense bf16 burst TFLOP/s, sustained TFLOP/s, HBM GB/s, source)."""
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get('bf16_tflops', 1665.0), d.get('bf16_tflops_sustained', 1381.2), d.get('hbm_gbs', 6570.9), 'measured (MEASURED_PEAKS.json)'
    return 1665.0, 1400.0, 6650.0, 'fallback (B200_PROFILING.md)'


# ----------------------------------------------------------------------------------------------- ours
MODES = ('precise', 'fast')
DUMP_PIXELS = 1 << 17       # per mode 3 + 36 + 3 float32 channels at these positions: 2 modes * 42 * 4 B * 2^17 = 44 MB
DTYPE = {'precise': 'bf16x3 (split-bf16 hi/lo operands, 3 tcgen05.mma per K block, fp32 accumulate: fp32-class)',
         'fast': 'bf16 (bf16 operands, fp32 accumulate)'}


def run_ours(args, rank, world, local_rank):
    import gc
    import numpy as np
    import torch
    import torch.distributed as dist
    from vid2vid_b200 import _lib as L
    from vid2vid_b200 import networks as NW
    from vid2vid_b200.model_g import Vid2VidModelG
    from vid2vid_b200.utils import synth_label_sequence

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    wl = WORKLOADS[args.workload]
    opt = make_opt_for(args.workload)
    opt.gpu_ids = [local_rank]
    torch.manual_seed(1234 + rank)
    model = Vid2VidModelG().initialize(opt)
    tG = opt.n_frames_G
    K, Wm = args.steps, max(args.warmup, 3)
    H, Wd = wl['H'], wl['W']
    n_frames = 2 * len(MODES) * (K + Wm + tG) + 8
    seq = synth_label_sequence(n_frames, H, Wd, label_nc=35, block=64, seed=rank)   # (1, T, 1, H, W) float ids
    seq_dev = seq.to(dev)
    seq_u8 = seq[0, :, 0].to(torch.uint8).pin_memory()                              # (T, H, W) uint8, pinned host
    out_u8 = torch.empty((H, Wd, 3), dtype=torch.uint8).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    modes = [m for m in MODES if args.modes in ('both', m)]
    dumps = {}
    if args.dump_outputs:
        pix = torch.randperm(H * Wd, generator=torch.Generator().manual_seed(0))[:DUMP_PIXELS].sort().values
        pix_dev = pix.to(dev)
        dumps['sample_pixels'] = pix.double()
    sampler = ClockSampler(local_rank)
    sampler.start()
    res = {}
    t = 0
    gc.collect()
    for mode in modes:
        NW.set_default_precision(mode)
        # ---- warm-up: first-frame generator (first call only) + W frames; instantiates this mode's CUDA graphs
        for _ in range(Wm):
            A = seq_dev[:, t:t + tG]
            model.inference(A, None, A)
            t += 1
        # ---- timed: device-resident inputs.  (A generation-2 garbage collection over the module tree costs tens of ms
        # when it lands inside a sub-second timed region: collect now, keep the collector off until the regions are done.)
        gc.collect()
        gc.disable()
        barrier()
        if mode == modes[0]:
            sampler.recording = True
        l0 = L.LAUNCHES[0]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            A = seq_dev[:, t:t + tG]
            out = model.inference(A, None, A)
            t += 1
        e1.record()
        barrier()
        if args.dump_outputs:       # (the next inference call may reuse these buffers)
            dumps[mode + '_fake_B'] = out[0][0].flatten(1)[:, pix_dev].cpu()
            dumps[mode + '_real_A'] = out[1].flatten(1)[:, pix_dev].cpu()
        ms_dev = e0.elapsed_time(e1)
        launches = L.LAUNCHES[0] - l0
        # ---- timed: end to end through the public streaming API with HOST buffers: one pinned uint8 label frame (and the
        # instance-id frame: the same synthetic map) -> H2D -> window push -> inference -> tensor2im on device -> D2H uint8
        model._win_A = None
        for _ in range(tG + 1):
            model.inference_stream(seq_u8[t], None, out_u8=out_u8)
            t += 1
        barrier()
        e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e2.record()
        for _ in range(K):
            model.inference_stream(seq_u8[t], None, out_u8=out_u8)
            t += 1
        e3.record()
        barrier()
        if args.dump_outputs:
            dumps[mode + '_e2e_rgb'] = out_u8.view(-1, 3)[pix].t().float()
        gc.enable()
        ms_e2e = e2.elapsed_time(e3)
        ms_dev, ms_e2e = reduce_times([ms_dev, ms_e2e], world, dev)
        res[mode] = dict(ms_dev=ms_dev, ms_e2e=ms_e2e, launches=launches)
    sampler.stop_flag = True
    h2d = 2 * H * Wd             # label + instance id frame, uint8
    d2h = 3 * H * Wd             # uint8 RGB frame
    if rank != 0:
        return
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumps.items():
            a = a.numpy()
            np.save(os.path.join(args.dump_outputs, name + '.npy'), a if a.dtype == np.float64 else a.astype(np.float32))

    # ---- first-frame generator (--use_single_G; runs tG - 1 times per clip, not per frame): timed separately (SURVEY 8d)
    first_ms = None
    if model.netG_i is not None:
        x = torch.zeros(1, 35, H, Wd, device=dev)
        x[:, 7] = 1.0
        model.netG_i(x)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(3):
            model.netG_i(x)
        f1.record()
        torch.cuda.synchronize()
        first_ms = f0.elapsed_time(f1) / 3

    # ---- roofline of the conv kernel per mode (per-launch CUDA events over one more frame, v2v_plan_profile)
    peak_burst, peak_sust, peak_gbs, peak_src = peaks()
    fmacs = frame_macs(args.workload)
    traffic_db = {}
    try:
        traffic_db = json.load(open(os.path.join(ROOT, 'profiles', 'conv_dram_traffic.json')))
    except Exception:
        pass

    def roofline(mode):
        conv_ms, conv_macs, other_ms, conv_launches, kind_ms = 0.0, 0.0, 0.0, 0, {}
        for s in range(wl['n_scales']):
            net = getattr(model, 'netG%d' % s)
            for key, ent in net._plans().items():
                if key[-1] != mode:
                    continue
                for kind, ms, macs in ent['plan'].profile():
                    kind_ms[kind] = kind_ms.get(kind, 0.0) + ms
                    if kind == 1:
                        conv_ms += ms
                        conv_macs += macs
                        conv_launches += 1
                    else:
                        other_ms += ms
        achieved = 2.0 * conv_macs / (conv_ms * 1e-3) / 1e12 if conv_ms > 0 else 0.0
        tj = traffic_db.get('%s_%s' % (args.workload, mode)) or (traffic_db.get(args.workload) if mode == 'fast' else None) or {}
        passes = 3 if mode == 'precise' else 1
        return {'bound': 'tensor', 'kernel': 'conv_umma_kernel (all launches of one frame)', 'achieved': achieved, 'peak': peak_burst,
                'unit': 'TFLOP/s', 'frac': achieved / peak_burst,
                'peak_source': peak_src + ': dense bf16 burst (kernels are timed one launch at a time); sustained %.1f' % peak_sust,
                'mma_passes_per_k_block': passes,
                'issued_tensor_tflops': achieved * passes, 'frac_of_issued_mma_work': achieved * passes / peak_burst,
                'traffic': tj.get('dram_bytes_per_launch_avg'),
                'traffic_unit': 'bytes per launch (dram read + write, ncu, mean over the launches of a frame)',
                'traffic_source': tj.get('source'), 'launches_per_frame': conv_launches,
                'algorithmic_flops_per_launch_avg': 2.0 * conv_macs / max(conv_launches, 1),
                'avg_launch_us': 1e3 * conv_ms / max(conv_launches, 1),
                'conv_kernel_ms_per_frame': conv_ms, 'other_kernels_ms_per_frame': other_ms,
                'ms_by_kernel_kind': {str(k): round(v, 4) for k, v in sorted(kind_ms.items())}}

    def line(mode):
        r = res[mode]
        frame_ms = r['ms_dev'] / K
        return {'value': world * K / (r['ms_dev'] * 1e-3), 'unit': 'frames/s', 'ms_per_step': frame_ms, 'dtype': DTYPE[mode],
                'e2e': {'value': world * K / (r['ms_e2e'] * 1e-3), 'unit': 'frames/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                        'api': 'Vid2VidModelG.inference_stream(pinned uint8 label frame) -> uint8 RGB frame in pinned host memory'},
                'gpu_launches': r['launches'], 'roofline': roofline(mode),
                'frame_flops_over_frame_time_tflops': 2 * fmacs / (frame_ms * 1e-3) / 1e12}

    head = line(modes[0])
    out = {
        'metric': 'frames/sec at 2048x1024 inference' if args.workload == 'cfg4' else 'frames/sec inference (%s)' % args.workload,
        'value': head['value'], 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': Wm,
        'ms_per_step': head['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': head['dtype'], 'data': 'synthetic 35-label blocky sequences, random-init weights (N(0,0.02))',
        'config': {'workload': wl['desc'], 'parallelism': 'replicas x%d (independent clips, no collective)' % world,
                   'frames_per_step': 1, 'conv_flops_per_frame': 2 * fmacs, 'precision_mode': modes[0],
                   'l2_policy': 'per-frame working set (weights 0.8 GB + activations) is far larger than the 126 MB L2'},
        'e2e': head['e2e'], 'gpu_launches': head['gpu_launches'], 'clocks': sampler.summary(), 'roofline': head['roofline'],
        'first_frame_generator_ms': first_ms,
    }
    if len(modes) > 1:
        out['fast'] = line('fast')          # the bf16-operand mode, reported beside the fp32-class headline
    if world == 1 and not args.no_cpu_baseline:
        out['cpu_baseline'] = cpu_frames_per_s(args.workload, steps=1, warm=0, budget_s=25.0)
    emit(out)


# ----------------------------------------------------------------------------------------------- CPU arm
def _cpu_model(workload, threads):
    """(step(H, n, seed) -> seconds per frame, kind).  kind 'reference': the UNMODIFIED reference Vid2VidModelG.inference
    (/root/reference here, its vendored copy oracle/_ref on the GPU box) under the CPU shims of oracle/ref_shim.py;
    kind 'port': the oracle restatement, only when no reference tree travelled."""
    import torch
    from vid2vid_b200.utils import synth_label_sequence
    wl = WORKLOADS[workload]
    torch.set_num_threads(threads)
    opt = make_opt_for(workload)
    opt.gpu_ids = []
    torch.manual_seed(0)
    from oracle import ref_shim
    if ref_shim.available():
        m = ref_shim.make_model_G(opt, single_G=None)
        kind = 'reference'

        def run(H, n, seed):
            m.fake_B_prev = [torch.zeros(2, 3, H // 2 ** s, wl['W'] // 2 ** s) for s in range(wl['n_scales'])]
            seq = synth_label_sequence(n + 2, H, wl['W'], label_nc=35, block=32, seed=seed)
            t0 = time.time()
            for t in range(n):
                m.inference(seq[:, t:t + 3], None, seq[:, t:t + 3])       # runs under torch.no_grad itself
            return (time.time() - t0) / n
    else:
        from oracle import generator_oracle as GO
        from vid2vid_b200 import networks as NW
        sds = [NW.build_netG(opt, s).state_dict() for s in range(wl['n_scales'])]
        kind = 'port'

        def run(H, n, seed):
            orc = GO.ModelGOracle(opt, sds)
            orc.fake_B_prev = [torch.zeros(2, 3, H // 2 ** s, wl['W'] // 2 ** s) for s in range(wl['n_scales'])]
            seq = synth_label_sequence(n + 2, H, wl['W'], label_nc=35, block=32, seed=seed)
            t0 = time.time()
            with torch.no_grad():
                for t in range(n):
                    orc.inference(seq[:, t:t + 3], seq[:, t:t + 3])
            return (time.time() - t0) / n
    return run, kind


def cpu_frames_per_s(workload, steps, warm, budget_s=150.0):
    """The reference on the host cores.  A step is one steady-state frame of the workload restricted to a horizontal band
    of the image (full width, height H*f, f in {1/8, 1/4, 1/2, 1}): every layer does the same work per pixel, so
    frames/s = f / seconds-per-band.  f is the largest fraction for which steps + warm bands fit in `budget_s`
    (calibrated on one 1/8 band); previous-frame state is zero-filled (the cost does not depend on the content).
    Threads: PyTorch's CPU convolutions regress beyond ~32 threads on the 128-core hosts, so a 1/16 band is timed with 32
    threads and with all cores and the faster setting is used (both numbers are reported)."""
    import torch
    wl = WORKLOADS[workload]
    band = lambda f: max(32, int(wl['H'] * f) // 32 * 32)
    all_cores = os.cpu_count()
    cand = sorted({min(all_cores, int(os.environ.get('V2V_CPU_THREADS', '32'))), all_cores})
    calib = {}
    run = kind = None
    for th in cand:
        run, kind = _cpu_model(workload, th)
        run(band(1.0 / 16), 1, 0)                     # warm the thread pool / allocator
        calib[th] = run(band(1.0 / 16), 1, 1)
    cores = min(calib, key=calib.get)
    run, kind = _cpu_model(workload, cores)
    t8 = run(band(1.0 / 8), 1, 1)                     # calibration of the band size
    frac = 1.0 / 16
    for f in (1.0, 0.5, 0.25, 0.125):
        if t8 * 8 * f * (steps + warm) <= budget_s:
            frac = f
            break
    if warm:
        run(band(frac), warm, 2)
    Hb = band(frac)
    dt = run(Hb, steps, 3)
    model = ''
    try:
        model = [l.split(':')[1].strip() for l in open('/proc/cpuinfo') if l.startswith('model name')][0]
    except Exception:
        pass
    eff = Hb / wl['H']
    return {'value': eff / dt, 'unit': 'frames/s', 'cores': cores, 'kind': kind,
            'sample': '%d step(s), each one steady-state frame of a %dx%d band (%.3f of the %s frame) through %s, torch %s CPU fp32, '
                      '%d threads (1/16-band calibration, s/band: %s), %s'
                      % (steps, wl['W'], Hb, eff, wl['desc'],
                         "the reference's own Vid2VidModelG.inference" if kind == 'reference' else 'the oracle port',
                         torch.__version__, cores, ', '.join('%d thr %.2f' % kv for kv in sorted(calib.items())), model),
            'seconds_per_step': dt}


def run_reference(args, rank, world):
    if rank != 0:
        return
    if WORKLOADS[args.workload].get('train') or WORKLOADS[args.workload].get('flownet'):
        emit({'impl': 'reference', 'unavailable': 'the CPU reference arm is defined for the headline inference workloads; '
                          'the reference training step needs its CUDA-only FlowNet2 ops (see DESIGN.md)'})
        return
    K, Wm = args.steps, args.warmup
    r = cpu_frames_per_s(args.workload, steps=K, warm=min(Wm, 1), budget_s=180.0)
    wl = WORKLOADS[args.workload]
    out = {'impl': 'reference',
           'metric': 'frames/sec at 2048x1024 inference' if args.workload == 'cfg4' else 'frames/sec inference (%s)' % args.workload,
           'value': r['value'], 'unit': 'frames/s', 'n_gpus': world, 'steps': K, 'warmup': min(Wm, 1),
           'ms_per_step': 1e3 / r['value'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
           'data': 'synthetic 35-label blocky sequences, random-init weights',
           'config': {'workload': wl['desc'], 'parallelism': 'host CPU, rank 0 only'},
           'cpu_baseline': {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
           'e2e': {'value': r['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    emit(out)


# ----------------------------------------------------------------------------------------------- training step (cfg3)
def run_train(args, rank, world, local_rank):
    """BASELINE config 3: `python bench.py --workload cfg3 [--gpus N]`.  A step = one iteration of train.py's inner loop on one
    clip per GPU (n_frames_load = 1 generated frame): generator forward (tcgen05, precise mode), FlowNet2 (no grad), image and
    temporal discriminator losses, the three backward passes (data gradients as forward convs on conv_umma_kernel, weight
    gradients on wgrad_umma_kernel, both in the split-bf16 precise arithmetic; norm / head / composite / loss backward on CUDA
    cores), ONE flat NCCL all-reduce over [G | D | D_T] and the Adam steps.  value = clips
    (= generated frames) per second over all ranks; the all-reduce is timed separately with CUDA events."""
    import gc
    import torch
    import torch.distributed as dist
    from vid2vid_b200 import _lib as L
    from vid2vid_b200 import flownet as FN
    from vid2vid_b200.model_d import Vid2VidModelD
    from vid2vid_b200.model_g import Vid2VidModelG
    from vid2vid_b200.trainer import Trainer
    from vid2vid_b200.utils import make_opt, synth_label_sequence

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    wl = WORKLOADS[args.workload]
    H, Wd = wl['H'], wl['W']
    opt = make_opt(label_nc=35, use_instance=True, fg=True, fg_labels=[26], n_scales_spatial=wl['n_scales'], ngf=wl['ngf'], num_D=3,
                   n_scales_temporal=2, n_frames_D=3, isTrain=True, no_vgg=True, gpu_ids=[local_rank], n_frames_total=30,
                   dataroot='datasets/Cityscapes/', loadSize=Wd)
    torch.manual_seed(1234)                         # identical initial weights on every rank (DataParallel replicates rank 0's)
    G = Vid2VidModelG().initialize(opt)
    D = Vid2VidModelD().initialize(opt)
    F = FN.FlowNet().initialize(opt)
    tr = Trainer(opt, G, D, F, world=world)
    # warm-up must reach the steady state of the clip: the temporal discriminators switch on as the frame history fills
    # (scale s needs tD**s * (tD - 1) + 1 frames, vid2vid_model_D.py:267-282) and build their plans at that step
    K, Wm = args.steps, max(args.warmup, opt.n_frames_D ** (opt.n_scales_temporal - 1) * (opt.n_frames_D - 1) + 3)
    tG = opt.n_frames_G
    T = K + Wm + tG + 2
    A = synth_label_sequence(T, H, Wd, label_nc=35, block=64, seed=rank).pin_memory()
    g = torch.Generator().manual_seed(77 + rank)
    coarse = torch.rand(T, 3, H // 16, Wd // 16, generator=g) * 2 - 1
    B = torch.nn.functional.interpolate(coarse, size=(H, Wd), mode='bilinear', align_corners=False).view(1, T, 3, H, Wd).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank, period=0.25)     # (NVML queries take the driver lock the ~3600 launches of a step also need)
    sampler.start()
    ar_ms = []
    orig_ar = tr.grads.all_reduce_mean

    def timed_ar(w):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        orig_ar(w)
        e1.record()
        ar_ms.append((e0, e1))
    tr.grads.all_reduce_mean = timed_ar
    t = 0
    for _ in range(Wm):
        a, b = A[:, t:t + tG].to(dev, non_blocking=True), B[:, t:t + tG].to(dev, non_blocking=True)
        tr.step(a, b, a)
        t += 1
    barrier()
    ar_ms.clear()
    sampler.recording = True
    l0 = L.LAUNCHES[0]
    gc.collect()
    gc.disable()          # (a generation-2 collection over the module / plan object graph inside a ~1 s region costs 10 % of it)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    step_wall = []
    for _ in range(K):
        t_wall = time.perf_counter()
        a, b = A[:, t:t + tG].to(dev, non_blocking=True), B[:, t:t + tG].to(dev, non_blocking=True)     # H2D of the step's inputs
        losses, _ = tr.step(a, b, a)           # ... and the D2H read of its loss values (one stacked copy to pinned host memory)
        t += 1
        step_wall.append((time.perf_counter() - t_wall) * 1e3)
    e1.record()
    barrier()
    gc.enable()
    sampler.stop_flag = True
    ms = e0.elapsed_time(e1)
    launches = L.LAUNCHES[0] - l0
    ar = sum(x.elapsed_time(y) for x, y in ar_ms) / max(len(ar_ms), 1)
    ms, ar = reduce_times([ms, ar], world, dev)
    if rank != 0:
        return
    gmacs = 0.0
    for s in range(wl['n_scales']):
        for key, ent in getattr(G, 'netG%d' % s)._plans().items():
            if 'train' in key:
                gmacs += ent['plan'].conv_macs
    peak_burst, peak_sust, peak_gbs, peak_src = peaks()
    step_ms = ms / K
    fl = 3 * 2 * gmacs                    # forward + data gradient + weight gradient of every generator convolution
    out = {'metric': 'training clips/sec (%s)' % args.workload, 'value': world * K / (ms * 1e-3), 'unit': 'clips/s', 'n_gpus': world, 'steps': K,
           'warmup': Wm, 'ms_per_step': step_ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
           'dtype': 'forward and backward convolutions ' + DTYPE['precise'] + '; norm / loss backward f32',
           'data': 'synthetic 35-label blocky clips + low-pass noise frames, random-init G / D / FlowNet2',
           'config': {'workload': wl['desc'], 'parallelism': 'dp%d: one clip per GPU, per-rank BatchNorm statistics, ONE flat NCCL all-reduce '
                      '(%.1f M fp32 gradients of [G | D | D_T0 | D_T1]) per step' % (world, tr.grads.numel / 1e6),
                      'frames_per_step': 1, 'generator_conv_flops_fwd_bwd_per_step': fl},
           'e2e': {'value': world * K / (ms * 1e-3), 'unit': 'clips/s', 'h2d_bytes_per_step': int(2 * tG * H * Wd * 4 + tG * 3 * H * Wd * 4),
                   'd2h_bytes_per_step': 9 * 4,
                   'api': 'Trainer.step(host label / frame tensors) -> host loss values, every step (the reference reads them every '
                          'print_freq steps, train.py:102-107; Trainer.step_async defers the read)'},
           'gpu_launches': launches, 'clocks': sampler.summary(),
           'all_reduce': {'ms_per_step': ar, 'share_of_step': ar / step_ms, 'bytes': tr.grads.numel * 4,
                          'algbw_gbs': tr.grads.numel * 4 / (ar * 1e-3) / 1e9 if ar > 0 else None, 'backend': 'nccl' if world > 1 else 'none (1 rank)'},
           'wall_ms_each_step': [round(x, 1) for x in step_wall],
           'hbm_used_gb': round((torch.cuda.mem_get_info(dev)[1] - torch.cuda.mem_get_info(dev)[0]) / 2 ** 30, 1),
           'roofline': {'bound': 'tensor', 'kernel': 'generator convolutions: forward + data gradient (conv_umma_kernel) + weight gradient (wgrad_umma_kernel)', 'achieved': fl / (step_ms * 1e-3) / 1e12,
                        'peak': peak_burst, 'unit': 'TFLOP/s', 'frac': fl / (step_ms * 1e-3) / 1e12 / peak_burst, 'peak_source': peak_src,
                        'traffic': None, 'note': 'whole-step time as denominator (includes the discriminators, FlowNet2, losses, optimizer); '
                        'algorithmic FLOPs: the precise mode issues 3 MMAs per algorithmic MAC'},
           'last_losses': losses}
    emit(out)


# ----------------------------------------------------------------------------------------------- FlowNet2 (a14 / a15)
def run_flownet2(args, rank, world, local_rank):
    """`python bench.py --workload flownet2`: a step = flowNet(frame_t, frame_t-1) -> (flow, confidence) for one 1024x512 pair
    (models/flownet.py:25-62; 264.3 algorithmic GMAC over the five sub-networks, SURVEY 8d).  value = pairs/s device-resident;
    e2e = two pinned fp32 host frames in, flow + confidence back to pinned host memory, every step."""
    import torch
    from vid2vid_b200 import _lib as L
    from vid2vid_b200 import flownet as FN
    from vid2vid_b200.utils import make_opt

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    wl = WORKLOADS[args.workload]
    H, Wd = wl['H'], wl['W']
    torch.manual_seed(1234)
    F = FN.FlowNet().initialize(make_opt(gpu_ids=[local_rank]))
    K, Wm = args.steps, max(args.warmup, 3)
    g = torch.Generator().manual_seed(5 + rank)
    coarse = torch.rand(K + Wm + 1, 3, H // 16, Wd // 16, generator=g)
    frames = torch.nn.functional.interpolate(coarse, size=(H, Wd), mode='bilinear', align_corners=False).pin_memory()
    frames_dev = frames.to(dev)
    out_flow = torch.empty(1, 2, H, Wd).pin_memory()
    out_conf = torch.empty(1, 1, H, Wd).pin_memory()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank)
    sampler.start()
    for t in range(Wm):
        F(frames_dev[t + 1:t + 2], frames_dev[t:t + 1])
    barrier()
    sampler.recording = True
    l0 = L.LAUNCHES[0]
    e0, e1, e2, e3 = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    e0.record()
    for t in range(Wm, Wm + K):
        F(frames_dev[t + 1:t + 2], frames_dev[t:t + 1])
    e1.record()
    barrier()
    launches = L.LAUNCHES[0] - l0
    e2.record()
    for t in range(Wm, Wm + K):
        a, b = frames[t + 1:t + 2].to(dev, non_blocking=True), frames[t:t + 1].to(dev, non_blocking=True)
        flow, conf = F(a, b)
        out_flow.copy_(flow, non_blocking=True)
        out_conf.copy_(conf, non_blocking=True)
    e3.record()
    barrier()
    sampler.stop_flag = True
    ms_dev, ms_e2e = reduce_times([e0.elapsed_time(e1), e2.elapsed_time(e3)], world, dev)
    if rank != 0:
        return
    conv_ms, conv_macs, other_ms, n_conv = 0.0, 0.0, 0.0, 0
    for key, ent in F.flowNet._plans().items():
        for kind, ms, macs in ent['plan'].profile():
            if kind == 1:
                conv_ms += ms; conv_macs += macs; n_conv += 1
            else:
                other_ms += ms
    peak_burst, peak_sust, peak_gbs, peak_src = peaks()
    ach = 2.0 * conv_macs / (conv_ms * 1e-3) / 1e12 if conv_ms else 0.0
    out = {'metric': 'frame pairs/sec (FlowNet2 1024x512)', 'value': world * K / (ms_dev * 1e-3), 'unit': 'pairs/s', 'n_gpus': world, 'steps': K,
           'warmup': Wm, 'ms_per_step': ms_dev / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': DTYPE['precise'],
           'data': 'synthetic low-pass noise frames, random-init (xavier) FlowNet2 weights',
           'config': {'workload': wl['desc'], 'parallelism': 'replicas x%d' % world, 'conv_flops_per_pair': 2.0 * conv_macs},
           'e2e': {'value': world * K / (ms_e2e * 1e-3), 'unit': 'pairs/s', 'h2d_bytes_per_step': 2 * 3 * H * Wd * 4, 'd2h_bytes_per_step': 3 * H * Wd * 4,
                   'api': 'FlowNet.forward(pinned fp32 frame pair) -> (flow, conf) in pinned host memory'},
           'gpu_launches': launches, 'clocks': sampler.summary(),
           'roofline': {'bound': 'tensor', 'kernel': 'conv_umma_kernel (all launches of the five sub-network plans)', 'achieved': ach, 'peak': peak_burst,
                        'unit': 'TFLOP/s', 'frac': ach / peak_burst, 'peak_source': peak_src, 'mma_passes_per_k_block': 3,
                        'issued_tensor_tflops': 3 * ach, 'traffic': None, 'launches_per_pair': n_conv, 'conv_kernel_ms_per_pair': conv_ms,
                        'other_plan_kernels_ms_per_pair': other_ms}}
    emit(out)


_REAL_STDOUT = None


def emit(obj):
    """The ONE JSON line of the contract, on the process's real stdout."""
    line = (json.dumps(obj) + '\n').encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def main():
    # Everything else that lands on stdout (NCCL prints its version banner there on these boxes, libraries may print notices)
    # goes to stderr instead: file descriptor 1 is pointed at stderr for the duration of the run.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg4', choices=list(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', dest='no_cpu_baseline', action='store_true')
    ap.add_argument('--modes', default='both', choices=['both', 'precise', 'fast'])
    ap.add_argument('--dump-outputs', dest='dump_outputs', metavar='DIR',
                    help='write the outputs of the last timed step as DIR/<name>.npy (inference workloads)')
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != 'ours' or WORKLOADS[args.workload].get('train') or WORKLOADS[args.workload].get('flownet')):
        ap.error('--dump-outputs is implemented for --impl ours on the inference workloads (cfg4, cfg2, tiny)')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'          # (keeps NCCL's version banner off stdout: ONE JSON line)
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    if WORKLOADS[args.workload].get('train'):
        run_train(args, rank, world, local_rank)
    elif WORKLOADS[args.workload].get('flownet'):
        run_flownet2(args, rank, world, local_rank)
    else:
        run_ours(args, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
