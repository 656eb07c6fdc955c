#!/usr/bin/env python
"""Benchmark of the flow log-density hot path (BASELINE.json metric: flow log_prob samples/sec).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun for N>1)
  python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm's CPU port (oracle/) on the host cores
  python bench.py ... --dump-outputs DIR                    # also write what the last timed step computed, to compare two builds

A step = one log_prob pass over one synthetic batch of the workload (default: configs[1], the CIFAR-10C-shaped conv-coupling
specialist, onehot+vardeq, --contextflow).  Prints ONE JSON line on rank 0.
"""
import argparse, json, os, statistics, subprocess, sys, threading, time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'flow_log_prob_samples_per_sec'
UNIT = 'samples/s'
WORKLOADS = {'cfg1': 'mnist-r 1x32x32 conv generalist', 'cfg2': 'cifar10c 3x32x32 conv specialist onehot+vardeq contextflow',
             'cfg3': 'atm 38x144x1 trans specialist eye+argmax contextflow', 'cfg4': 'smap 25x8x1 trans generalist'}
DEFAULT_BATCH = {'cfg1': 8192, 'cfg2': 8192, 'cfg3': 1024, 'cfg4': 131072}
REF_BATCH = {'cfg1': 256, 'cfg2': 256, 'cfg3': 64, 'cfg4': 256}          # reference default batch (config.py:10; BASELINE.md §3); cfg3: 64 (BASELINE.md §4)
TORCH_CUDA_BATCH = {'cfg1': 2048, 'cfg2': 2048, 'cfg3': 256, 'cfg4': 8192}
DUMP_BYTES = 64 * 10**6                                                  # --dump-outputs: all arrays of one run together


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='cfg2', choices=sorted(WORKLOADS))
    ap.add_argument('--batch', type=int, default=0, help='samples per GPU per step (0 = workload default)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--ref-device', default='cpu', choices=['cpu', 'cuda'],
                    help='--impl reference only: cpu (the contract: host cores) or cuda (the same torch op sequence run eagerly on the GPU, '
                         'the "reference torch-on-CUDA" figure of the north star; informative)')
    ap.add_argument('--path', default='log_prob', choices=['log_prob', 'train', 'reverse'],
                    help='log_prob (default): the headline forward log-density path; train / reverse: the SURVEY §8(f) rows, measured by '
                         'tools/bench_training.py / tools/bench_inverse.py (their own JSON lines)')
    ap.add_argument('--secondary', default='cfg4', choices=sorted(WORKLOADS) + [''], help='second workload measured in the same run ("" = none)')
    ap.add_argument('--tertiary', default='cfg3', choices=sorted(WORKLOADS) + [''], help='third workload measured in the same run: BASELINE configs[2], the ATM trans specialist ("" = none)')
    ap.add_argument('--no-parity', action='store_true', help='skip the oracle parity check of the timed batch (profiling runs)')
    ap.add_argument('--eager', action='store_true', help='launch every kernel from Python instead of replaying the captured CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='log_prob path of --impl ours only: after the timed steps, write the (batch, mixtures) log-probabilities the last timed '
                         'step of each workload returned as DIR/<workload>_log_prob.npy (float32, rows in batch order; a fixed, seeded sample of '
                         f'rows when all of them together exceed {DUMP_BYTES // 10**6} MB).  The image workloads (cfg1, cfg2) draw dequantisation '
                         'and encoder noise from torch\'s device generator: the same build and arguments reproduce them exactly, but two builds '
                         'that draw their noise in a different order differ by up to tens of nats per row while both are correct')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and (a.impl != 'ours' or a.path != 'log_prob'):
        ap.error('--dump-outputs covers the log_prob path of --impl ours only')
    return a


class ClockSampler(threading.Thread):
    """SM clocks + throttle reasons during the timed region (B200_PROFILING.md recipe).  NVML through pynvml when importable (a
    sample per ~20 ms), else the recipe's nvidia-smi query line (one sample per ~0.3 s).  Samples carry a timestamp; summary() keeps
    those inside the timed window [t0, t1] and, when the window was too short for any, the nearest ones taken under the same load."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
    NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n = self.nvml
        sm = float(n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM))
        try:
            power = n.nvmlDeviceGetPowerUsage(self.handle) / 1000.0
        except Exception:
            power = 0.0
        try:
            mask = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        except Exception:
            mask = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        bits = [getattr(n, 'nvmlClocksEventReasonHwSlowdown', 0x8), getattr(n, 'nvmlClocksEventReasonHwThermalSlowdown', 0x40),
                getattr(n, 'nvmlClocksEventReasonSwThermalSlowdown', 0x20), getattr(n, 'nvmlClocksEventReasonSwPowerCap', 0x4)]
        return [sm, self.max_sm, power] + [bool(mask & b) for b in bits]

    def _sample_smi(self):
        out = subprocess.run(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-i', str(self.index)],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        c = [v.strip() for v in out.split(',')]
        return [float(c[0]), float(c[1]), float(c[2])] + [v.lower().startswith('active') for v in c[3:7]]

    def run(self):
        while not self.stop_flag.is_set():
            try:
                row = self._sample_nvml() if self.nvml is not None else self._sample_smi()
                self.rows.append((time.perf_counter(), row))
            except Exception:
                pass
            self.stop_flag.wait(0.02 if self.nvml is not None else 0.05)

    def summary(self, t0=None, t1=None):
        self.stop_flag.set()
        rows = [r for t, r in self.rows if t0 is None or (t0 <= t <= t1)]
        window = 'timed region'
        if not rows and self.rows:                                      # window shorter than one sample: the samples closest to it (warm-up / e2e legs, same load)
            mid = 0.5 * (t0 + t1)
            rows = [r for _, r in sorted(self.rows, key=lambda tr: abs(tr[0] - mid))[:3]]
            window = 'nearest samples (timed region shorter than the sampling period)'
        if not rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unsampled']}
        reasons = [n for i, n in enumerate(self.NAMES) if any(r[3 + i] for r in rows)]
        return {'sm_mhz': statistics.median(r[0] for r in rows), 'sm_max_mhz': rows[0][1], 'reasons': reasons, 'samples': len(rows),
                'power_w_max': max(r[2] for r in rows), 'window': window, 'source': 'nvml' if self.nvml is not None else 'nvidia-smi'}


def _reference_forward(workload, device):
    """(log_prob(x, ctx) callable, kind, description): the UNMODIFIED reference when a complete checkout is found ($CFPP_REFERENCE, or
    baseline/_ref made by tools/install_reference.py) -- its own create_model / FlowSequential.log_prob over its own torch layers --
    else the oracle port (oracle/flow_oracle.py: the same torch op sequence, pinned to the reference by tests/golden)."""
    import torch
    from contextflow_b200 import builder, synth
    conf = synth.CONFIGS[workload]
    sys.path.insert(0, os.path.join(ROOT, 'tools'))
    import refshim
    ref = None if os.environ.get('CFPP_BENCH_FORCE_PORT') == '1' else refshim.find_reference()
    if ref is not None:
        try:
            M = refshim.import_reference(ref)
            torch.manual_seed(0)
            net = refshim.create_model(M, conf).eval()
            sd = net.state_dict(); synth.fill_state(sd, 'bench'); net.load_state_dict(sd)
            net = net.to(device)
            return (lambda x, c: net.log_prob(x, context=c)), 'reference', f'unmodified reference ({os.path.relpath(ref, ROOT) if ref.startswith(ROOT) else ref})'
        except Exception as e:                                   # an incomplete checkout: say so and use the port
            print(f'bench.py: reference checkout at {ref} not usable ({type(e).__name__}: {e}); using the oracle port', file=sys.stderr)
    from oracle import flow_oracle as O
    stack = O.build_stack(conf['cfg'], conf['data_size'], conf['mixtures'], conf['contexts'])
    model = builder.build_named(conf)
    state = model.state_dict(); synth.fill_state(state, 'bench')
    O.DEVICE = str(device)
    state = {k: v.to(device) for k, v in state.items()}

    class TorchNoise:
        def rand(self, shape): return torch.rand(shape, device=device)
        def randn(self, shape): return torch.randn(shape, device=device)
    return (lambda x, c: O.log_prob(stack, state, x, c, TorchNoise())), 'port', 'oracle port of the reference op sequence (oracle/flow_oracle.py)'


def reference_run(workload, batch, steps, warmup, device='cpu', tf32=None, seed=1234):
    """The reference's log_prob timed on the host cores (device='cpu', all threads) or eagerly on the GPU (device='cuda': the
    "reference torch-on-CUDA" figure of the north star; tf32=None keeps torch's default flags, False disables TF32 everywhere)."""
    import contextlib
    import torch
    from contextflow_b200 import synth
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    conf = synth.CONFIGS[workload]
    on_gpu = str(device).startswith('cuda')
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32)
    if tf32 is not None:
        torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = bool(tf32)
    fwd, kind, what = _reference_forward(workload, device)
    gen = torch.Generator().manual_seed(seed)
    C, H, W = conf['data_size']
    x = (torch.randint(0, 256, (batch, C, H, W), generator=gen).float() if conf['image'] else torch.rand(batch, C, H, W, generator=gen)).to(device)
    ctx = torch.stack([torch.randint(0, k, (batch,), generator=gen) for k in conf['contexts']], 1).to(device)
    dev_ctx = torch.device(device) if (on_gpu and kind == 'port') else contextlib.nullcontext()
    sync = torch.cuda.synchronize if on_gpu else (lambda: None)
    times = []
    with torch.no_grad(), dev_ctx:
        for _ in range(max(1, warmup)):                          # the first forward also triggers ActNorm's data-dependent initialisation
            fwd(x, ctx)
        sync()
        t_all = time.perf_counter()
        for _ in range(steps):
            t0 = time.perf_counter(); fwd(x, ctx); sync(); times.append(time.perf_counter() - t0)
        dt = time.perf_counter() - t_all
    torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = saved
    if on_gpu:
        flags = 'torch default flags' if tf32 is None else f'TF32 {"on" if tf32 else "off"}'
        how = f'torch CUDA eager fp32 on {torch.cuda.get_device_name(0)}, {flags}'
    else:
        how = f'torch CPU fp32, {torch.get_num_threads()} threads'
    return dict(value=batch * steps / dt, unit=UNIT, cores=cores, kind=kind, median_ms_per_step=1e3 * statistics.median(times),
                sample=f'{steps} x log_prob of a {batch}-sample {workload} batch, {what}, {how}'), dt


HBM_KERNELS_EXCLUDED = ('conv_cond_fwd', 'conv_cond_tc_fwd', 'conv_cond_tc_coupling_fwd', 'vit_cond_fwd', 'vit_tc_fwd', 'vit_tc2_fwd', 'gmm_logprob',
                        'gmm_logprob_ctxtab', 'gmm_logprob_ctxtab_cached', 'gmm_tile_logprob', 'ctx_encode_batch', 'ctx_encode', 'cn_batch', 'ctx_tables', 'linear_fwd', 'ldj_sum', 'slogdet')
TENSOR_KERNELS = ('conv_cond_tc_fwd', 'conv_cond_tc_coupling_fwd', 'vit_tc_fwd', 'vit_tc2_fwd', 'conv1x1_tc_fwd')
PAIR_KERNELS = TENSOR_KERNELS                                    # fp16 hi/lo pairs: 3 tensor products issued per algorithmic product


def config_line(workload, B, world, conf, graphed):
    C, H, W = conf['data_size']
    return {'workload': f'{workload}: {WORKLOADS[workload]}', 'batch_per_gpu': B, 'global_batch': B * world,
            'parallelism': f'dp{world} (batch-sharded, final all-gather of log-probs)',
            'l2_policy': f'{NBUF} rotating input batches; per-layer working set {12 * B * C * H * W / 1e6:.0f} MB > 126 MB L2',
            'weights': 'synthetic fill (synth.fill_state)',
            'launch': 'CUDA graph replay of the whole log_prob (contextflow_b200/graphed.py)' if graphed else 'eager (one Python call per kernel)',
            'kernel_timing': 'per-launch CUDA events in an eager pass over the same steps right after the timed region',
            'e2e_mode': 'GraphedLogProb.stream: pinned H2D of batch i+1 on a copy stream overlaps the replay of batch i; D2H of every result' if graphed
                        else 'per-step blocking copies'}


NBUF = 3


def measure(a, workload, B, rank, world, dev, with_e2e=True, parity=True):
    """One workload on this rank's GPU: device-timed value, per-kernel roofline, end-to-end leg, parity of the timed configuration."""
    import torch
    import torch.distributed as dist
    from contextflow_b200 import _cabi, builder, ops, synth
    from contextflow_b200.graphed import GraphedLogProb
    from contextflow_b200.sharded import ShardedLogProb
    conf = synth.CONFIGS[workload]
    model = builder.build_named(conf)
    sd = model.state_dict(); synth.fill_state(sd, 'bench'); model.load_state_dict(sd)
    model = model.to(dev).eval()
    M = conf['mixtures']
    # synthetic inputs: NBUF rotating device-resident batches (HBM-resident inputs; the set is larger than L2) + pinned host copies
    torch.manual_seed(1234 + rank)
    C, H, W = conf['data_size']

    def fresh():
        x = torch.randint(0, 256, (B, C, H, W)).float() if conf['image'] else torch.rand(B, C, H, W)
        ctx = torch.stack([torch.randint(0, k, (B,)) for k in conf['contexts']], 1)
        return x, ctx
    host = [tuple(t.pin_memory() for t in fresh()) for _ in range(NBUF)]
    devb = [(x.to(dev), c.to(dev)) for x, c in host]
    sharder = ShardedLogProb(lambda x, c: model.log_prob(x, c), M)
    graphed = None if a.eager else GraphedLogProb(model)

    def run(x, c):
        """One log_prob pass: a replay of the captured CUDA graph (x / c are copied into its static input buffers -- device to
        device for resident inputs, pinned host to device for the end-to-end leg), or the eager launch sequence with --eager."""
        if graphed is not None:
            return graphed(x, c, clone=False)
        return model.log_prob(x.to(dev, non_blocking=True), c.to(dev, non_blocking=True))

    def step(i):
        x, c = devb[i % NBUF]
        with torch.no_grad():
            return sharder.gather(run(x, c), B * world)   # the path's only exchange: final score gather (no-op at N=1)

    def step_e2e(i, out_host):
        hx, hc = host[i % NBUF]
        with torch.no_grad():
            lp = sharder.gather(run(hx, hc), B * world)
            out_host.copy_(lp[:out_host.shape[0]], non_blocking=True)
        torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(dev.index); sampler.start()
    for i in range(max(a.warmup, 3)):
        step(i)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    prof_range = os.environ.get('CFPP_PROFILE_RANGE') == '1'       # ncu --profile-from-start off: capture the timed steps only
    if prof_range:
        torch.cuda.profiler.start()
    l0 = _cabi.launch_count()
    t_begin = time.perf_counter()
    ev0.record()
    for i in range(a.steps):
        out = step(i)
    ev1.record()
    barrier()
    t_end = time.perf_counter()
    if prof_range:
        torch.cuda.profiler.stop()
    # a graph replay returns its static output buffer, which the passes below overwrite: copy the last timed step's result out now
    last_out = out.float().cpu() if a.dump_outputs and rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    launches = _cabi.launch_count() - l0 if graphed is None else graphed.launches_per_replay(*devb[0]) * a.steps
    # per-kernel durations: the same steps launched eagerly with a CUDA-event pair around every libcfpp launch (events cannot be
    # read back from inside a replayed graph); same kernels, same inputs, right after the timed region
    timer = ops.OpTimer(); ops.set_timer(timer)
    with torch.no_grad():
        for i in range(a.steps):
            x, c = devb[i % NBUF]
            model.log_prob_eager(x, c)
    barrier()
    ops.set_timer(None)
    # The conv couplings run fused into the conditioner's epilogue by default (h never reaches HBM), so the step has no stand-alone
    # memory-bound coupling launch to put against the HBM roof.  A few eager steps of the two-kernel route (CFPP_CONV_COND=split), outside
    # the timed region, keep that figure in the record.
    split_summ = None
    if rank == 0 and 'conv_cond_tc_coupling_fwd' in timer.summary() and os.environ.get('CFPP_CONV_COND', 'auto') in ('auto', 'fused'):
        prev = os.environ.get('CFPP_CONV_COND')
        os.environ['CFPP_CONV_COND'] = 'split'
        tsplit = ops.OpTimer(); ops.set_timer(tsplit)
        with torch.no_grad():
            for i in range(min(a.steps, 10)):
                x, c = devb[i % NBUF]
                model.log_prob_eager(x, c)
        torch.cuda.synchronize()
        ops.set_timer(None)
        if prev is None:
            os.environ.pop('CFPP_CONV_COND')
        else:
            os.environ['CFPP_CONV_COND'] = prev
        split_summ = tsplit.summary()
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    clocks = sampler.summary(t_begin, t_end)

    e2e = None
    if with_e2e:
        # end to end through the public API with host buffers (pinned H2D of x, ctx every step; D2H of every step's log-probs), timed on
        # the host clock.  Graph mode uses GraphedLogProb.stream: the copy of batch i+1 overlaps the replay of batch i.
        nout = B * world if rank == 0 else B
        outs_host = [torch.empty((nout, M), dtype=torch.float32).pin_memory() for _ in range(min(a.steps, 4))]
        gather = (lambda lp: sharder.gather(lp, B * world))

        def e2e_pass(n):
            if graphed is not None:
                with torch.no_grad():
                    graphed.stream((host[i % NBUF] for i in range(n)), [outs_host[i % len(outs_host)] for i in range(n)], post=gather if world > 1 else None)
            else:
                for i in range(n):
                    step_e2e(i, outs_host[i % len(outs_host)])
        e2e_pass(2)
        barrier()
        t0 = time.perf_counter()
        e2e_pass(a.steps)
        barrier()
        e2e_s = time.perf_counter() - t0
        te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        x0, c0 = host[0]
        e2e = {'value': world * B * a.steps / float(te.item()), 'unit': UNIT, 'h2d_bytes_per_step': x0.numel() * 4 + c0.numel() * 8, 'd2h_bytes_per_step': B * world * M * 4}

    par = None
    if parity and rank == 0:
        # parity of exactly what was timed: one of the rotating batches through the GRAPH REPLAY under a fixed seed, the same batch through
        # the eager launch sequence with its draws recorded (must be bit-identical), and a 256-row subsample of it through the CPU oracle
        # (the reference's op sequence, pinned by tests/golden) replaying those recorded noise rows.  The oracle is the checker only.
        from oracle import check
        x, c = devb[1 % NBUF]
        with torch.no_grad():
            torch.manual_seed(4242)
            rep = run(x, c).clone()
        logp, rec = check.recorded_log_prob(model, x, c, seed=4242)
        par = check.rows_parity(model, conf, x, c, seed=4242, n_rows=256, logp=logp, rec=rec)
        par['replay_equals_eager'] = bool(torch.equal(rep, logp))
        par['ok'] = bool(par['ok'] and par['replay_equals_eager'])
        del rec

    if rank != 0:
        return None
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak, hbm_src = (peaks['hbm_gbs'], 'measured (MEASURED_PEAKS.json)') if 'hbm_gbs' in peaks else (6650.0, 'fallback (B200_PROFILING.md)')
    timed_s = ms / 1e3
    if timed_s < 1.0:                                            # a sub-second timed region runs at burst clocks: the burst bf16 figure is the roof
        tf_peak, tf_src = peaks.get('bf16_tflops', 1650.0), 'bf16 burst'
    else:
        tf_peak, tf_src = peaks.get('bf16_tflops_sustained', 1400.0), 'bf16 sustained'
    tf_src += ' (MEASURED_PEAKS.json)' if peaks else ' (fallback)'
    summ = timer.summary()
    total_ms = sum(v['ms'] for v in summ.values()) or 1.0
    kernels = {}
    for name, v in sorted(summ.items(), key=lambda kv: -kv[1]['ms']):
        sec = v['ms'] / 1e3
        kernels[name] = {'share': round(v['ms'] / total_ms, 4), 'ms_per_step': round(v['ms'] / a.steps, 4), 'launches_per_step': v['n'] / a.steps,
                         'GBps': round(v['bytes'] / sec / 1e9, 1) if sec > 0 else None, 'TFLOPps': round(v['flops'] / sec / 1e12, 3) if sec > 0 else None}
        if v.get('shapes'):
            kernels[name]['by_shape'] = {k: {'ms_per_launch': round(w['ms'] / w['n'], 4), 'launches_per_step': w['n'] / a.steps,
                                             'GBps': round(w['bytes'] / (w['ms'] / 1e3) / 1e9, 1), 'TFLOPps': round(w['flops'] / (w['ms'] / 1e3) / 1e12, 3)}
                                         for k, w in v['shapes'].items() if w['ms'] > 0}

    def traffic_of(name):
        try:                                                   # DRAM bytes of one launch from the committed ncu --set full capture
            tj = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json'))).get(name)
            if tj and tj.get('batch') == B and tj.get('workload') == workload:
                return tj['dram_bytes_per_launch']
        except Exception:
            pass
        return None

    def roof_of(name):
        tv = summ[name]
        sec = tv['ms'] / 1e3
        if name in TENSOR_KERNELS:
            ach = tv['flops'] / sec / 1e12
            return {'kernel': name, 'bound': 'tensor', 'achieved': ach, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': ach / tf_peak, 'traffic': traffic_of(name),
                    'issued_tensor_TFLOPps': 3.0 * ach, 'frac_issued': 3.0 * ach / tf_peak,
                    'peak_source': tf_src + '; achieved counts ALGORITHMIC flops: the fp32-faithful fp16-pair arithmetic issues 3 tensor products per '
                                            'algorithmic one, so its own ceiling is 1/3 of this peak'}
        if name in HBM_KERNELS_EXCLUDED:                        # FP32-issue bound kernels (mixture, encoders): report flops against the tensor roof for scale
            ach = tv['flops'] / sec / 1e12
            return {'kernel': name, 'bound': 'tensor', 'achieved': ach, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': ach / tf_peak, 'traffic': traffic_of(name),
                    'peak_source': tf_src + '; this kernel is an FP32-FMA path (not a tensor-core kernel)'}
        ach = tv['bytes'] / sec / 1e9
        return {'kernel': name, 'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak, 'traffic': traffic_of(name), 'peak_source': hbm_src}

    top = next(iter(kernels))
    roof = roof_of(top)
    hbm_names = [n for n in summ if n not in HBM_KERNELS_EXCLUDED and summ[n]['bytes'] > 0]
    hb, hs = sum(summ[n]['bytes'] for n in hbm_names), sum(summ[n]['ms'] for n in hbm_names) / 1e3
    roof_hbm = {'kernels': sorted(hbm_names), 'bound': 'hbm', 'achieved': hb / hs / 1e9, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': hb / hs / 1e9 / hbm_peak,
                'ms_per_step': 1e3 * hs / a.steps, 'note': 'every HBM-bound kernel of the step together: algorithmic bytes / summed launch time'} if hs > 0 else None
    roof_c = None
    for cand in ('coupling_fwd', 'conv_cond_tc_coupling_fwd'):
        if cand in summ and cand not in TENSOR_KERNELS:
            roof_c = roof_of(cand)
    if roof_c is None and split_summ and 'coupling_fwd' in split_summ:
        tv = split_summ['coupling_fwd']
        ach = tv['bytes'] / (tv['ms'] / 1e3) / 1e9
        roof_c = {'kernel': 'coupling_fwd', 'bound': 'hbm', 'achieved': ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach / hbm_peak, 'traffic': traffic_of('coupling_fwd'),
                  'peak_source': hbm_src, 'ms_per_step': round(tv['ms'] / min(a.steps, 10), 4),
                  'note': 'the stand-alone memory-bound coupling kernel of the two-kernel route (CFPP_CONV_COND=split), timed in eager steps outside the '
                          'timed region; the timed step runs the coupling transform inside the conditioner kernel'}
    return {'value': world * B * a.steps / (ms / 1e3), 'ms_per_step': ms / a.steps, 'config': config_line(workload, B, world, conf, graphed is not None),
            'clocks': clocks, 'gpu_launches': launches, 'e2e': e2e, 'roofline': roof, 'roofline_coupling': roof_c, 'roofline_hbm_path': roof_hbm,
            'kernels': kernels, 'parity_at_bench_batch': par, 'outputs': {f'{workload}_log_prob': last_out}}


def dump_outputs(path, arrays):
    """Write each (rows, M) array as path/<name>.npy in float32.  When all of them together exceed DUMP_BYTES, each keeps the same share
    of its rows: a sorted sample drawn with a fixed seed, so that two runs with the same arguments write the same rows."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    total = sum(v.numel() * 4 for v in arrays.values())
    for name, v in arrays.items():
        v = v.numpy().astype(np.float32)
        if total > DUMP_BYTES:
            keep = max(1, v.shape[0] * DUMP_BYTES // total)
            v = v[np.sort(np.random.default_rng(0).choice(v.shape[0], keep, replace=False))]
        np.save(os.path.join(path, f'{name}.npy'), v)


def main():
    a = parse()
    if a.path != 'log_prob':                       # the "next" rows have their own measurement tools; same launch conventions (torchrun for N > 1)
        import runpy
        tool = 'bench_training.py' if a.path == 'train' else 'bench_inverse.py'
        argv = [tool, '--steps', str(a.steps)]
        if a.path == 'train':
            argv += ['--warmup', str(a.warmup), '--impl', a.impl, '--workload', a.workload]
            if a.batch:
                argv += ['--batch', str(a.batch)]
            if a.impl == 'reference':
                argv += ['--ref-device', a.ref_device]
        sys.argv = argv
        runpy.run_path(os.path.join(ROOT, 'tools', tool), run_name='__main__')
        return
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1)); local = int(os.environ.get('LOCAL_RANK', 0))
    workload = a.workload

    if a.impl == 'reference':
        # the reference arm: the reference's own implementation of the path on the host cores (all threads), same metric / unit / config as
        # this repo's arm; each step is a BOUNDED sample of the workload (one reference-default 256-sample batch, config.py:10)
        if rank != 0:
            return
        from contextflow_b200 import synth
        B = a.batch or REF_BATCH[workload]
        base, dt = reference_run(workload, B, a.steps, max(1, min(a.warmup, 2)), a.ref_device)
        cfg = config_line(workload, DEFAULT_BATCH[workload], max(a.gpus, 1), synth.CONFIGS[workload], True)
        print(json.dumps({'metric': METRIC, 'value': base['value'], 'unit': UNIT, 'impl': 'reference', 'n_gpus': a.gpus, 'steps': a.steps,
                          'warmup': a.warmup, 'ms_per_step': 1e3 * dt / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
                          'dtype': 'f32', 'data': 'synthetic', 'config': cfg,
                          'reference_arm': f'each step = log_prob of one {B}-sample batch on {a.ref_device} ({base["kind"]}); see cpu_baseline.sample',
                          'cpu_baseline': base, 'e2e': {'value': base['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))
        return

    import torch
    import torch.distributed as dist
    assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    saved_stdout = None
    if world > 1:
        # NCCL writes its version banner to stdout at communicator creation: keep this process's stdout for the ONE JSON line by
        # pointing fd 1 at stderr until the timed runs are over
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group('nccl', device_id=dev)
    B = a.batch or DEFAULT_BATCH[workload]
    res = measure(a, workload, B, rank, world, dev, parity=not a.no_parity)
    sec = None
    if a.secondary and a.secondary != workload:
        # BASELINE configs[4] names two shapes for the throughput sweep (CIFAR-shape conv AND SMAP-shape trans): the second one rides
        # along in the same line so that it is seen at every N the driver runs
        sec = measure(a, a.secondary, DEFAULT_BATCH[a.secondary], rank, world, dev, with_e2e=False, parity=not a.no_parity)
    ter = None
    if a.tertiary and a.secondary and a.tertiary not in (workload, a.secondary):
        # BASELINE configs[2] (ATM trans specialist, eye + argmax): the general ViT conditioner's shape, seen at every N as well
        ter = measure(a, a.tertiary, DEFAULT_BATCH[a.tertiary], rank, world, dev, with_e2e=False, parity=not a.no_parity)
    if saved_stdout is not None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if rank == 0:
        if a.dump_outputs:
            dump_outputs(a.dump_outputs, {k: v for r in (res, sec, ter) if r is not None for k, v in r['outputs'].items()})
        line = {'metric': METRIC, 'value': res['value'], 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': max(a.warmup, 3),
                'ms_per_step': res['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                'config': res['config'], 'clocks': res['clocks'], 'gpu_launches': res['gpu_launches'], 'e2e': res['e2e'],
                'roofline': res['roofline'], 'roofline_coupling': res['roofline_coupling'], 'roofline_hbm_path': res['roofline_hbm_path'],
                'kernels': res['kernels'], 'parity_at_bench_batch': res['parity_at_bench_batch'],
                'gradient_gate_note': 'training-direction gradients (tests/test_gpu_training.py) pass within 2e-4 of the largest entry OR 4x the reference\'s own fp32-fp64 gap (3x with the FP32 conditioner forward, CFPP_TRAIN_TC=0)'}
        if sec is not None:
            line['secondary'] = {'metric': METRIC, 'value': sec['value'], 'unit': UNIT, 'ms_per_step': sec['ms_per_step'], 'config': sec['config'],
                                 'gpu_launches': sec['gpu_launches'], 'roofline': sec['roofline'], 'roofline_coupling': sec['roofline_coupling'],
                                 'roofline_hbm_path': sec['roofline_hbm_path'], 'kernels': sec['kernels'], 'parity_at_bench_batch': sec['parity_at_bench_batch']}
        if ter is not None:
            line['tertiary'] = {'metric': METRIC, 'value': ter['value'], 'unit': UNIT, 'ms_per_step': ter['ms_per_step'], 'config': ter['config'],
                                'gpu_launches': ter['gpu_launches'], 'roofline': ter['roofline'], 'kernels': ter['kernels'],
                                'parity_at_bench_batch': ter['parity_at_bench_batch']}
        if world == 1 and not a.no_cpu_baseline:
            # bounded sample of the same workload on the host cores: ~10-20 s of CPU work (probe one step, then as many as fit)
            probe, dt1 = reference_run(workload, REF_BATCH[workload], 1, 1)
            nsteps = max(2, min(60, int(12.0 / max(dt1, 1e-3))))
            base, _ = reference_run(workload, REF_BATCH[workload], nsteps, 0)
            line['cpu_baseline'] = base
            # the north star's performance anchor: the reference's torch code run eagerly on this same GPU (B = 2048), with the flags a
            # user gets by default and with TF32 off (the parity-grade arithmetic); value / torch_cuda_baseline.value is the >= 8x target
            tcb = {}
            for key, tf in (('default_flags', None), ('tf32_off', False)):
                try:
                    r, _ = reference_run(workload, TORCH_CUDA_BATCH[workload], 10, 3, device=f'cuda:{local}', tf32=tf)
                    tcb[key] = r
                except Exception as e:
                    tcb[key] = {'unavailable': f'{type(e).__name__}: {e}'[:300]}
                torch.cuda.empty_cache()
            ok = [v['value'] for v in tcb.values() if 'value' in v]
            if ok:
                tcb['speedup_over_torch_cuda'] = {'device_timed': res['value'] / max(ok), 'e2e': res['e2e']['value'] / max(ok),
                                                  'note': 'this repo at N=1 / the faster of the two torch-on-CUDA runs; north-star target >= 8'}
            line['torch_cuda_baseline'] = tcb
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
