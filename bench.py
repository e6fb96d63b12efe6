#!/usr/bin/env python
"""Benchmark of the PIDM training step (BASELINE.json: "train samples/s Darcy 64x64 PIDM at 1/2/4/8 B200;
residual-kernel HBM GB/s").

    python bench.py --gpus N --steps K --warmup W           # this repo's engine (libpidm kernels)
    python bench.py --impl reference --steps K --warmup W   # the reference algorithm on the host CPU cores (oracle port)

One step = one iteration of the reference training loop (main.py:157-183): q_sample -> Unet3D(dim=32) -> x0_hat ->
Darcy residual -> data + residual loss -> backward -> clip(1.0) -> Adam(1e-4) -> EMA(0.99), batch 32 per GPU,
synthetic 64x64 fields, random-init weights, bf16 GEMM operands / activations with fp32 accumulation.
Prints ONE JSON line (rank 0)."""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
_IMPL = next((sys.argv[i + 1] for i, a in enumerate(sys.argv[:-1]) if a == '--impl'), 'b200')
if _IMPL in ('reference', 'cpu_extras'):
    # CPU legs: hide the GPU before torch initialises (the reference picks `cuda` whenever it is available)
    os.environ['CUDA_VISIBLE_DEVICES'] = ''
if _IMPL == 'b200':
    sys.path.insert(0, ROOT)
else:
    # reference legs import the UNMODIFIED reference `src` package (oracle/ref_arm.py): the repo root, whose `src/`
    # drop-in package would shadow it, must not be importable in this process
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or '.') != ROOT]

import torch  # noqa: E402

PER_GPU_BATCH = 32
METRIC = 'train samples/s Darcy 64x64 PIDM'
FWD_GFLOP_PER_SAMPLE = 3.98      # SURVEY.md section 3.2 (conv3x3 2.40, 1x1 0.96, attention einsums 0.36, 4x4 0.20, rest)


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm_gbs=d['hbm_gbs'], bf16_tflops=d['bf16_tflops'], bf16_sustained=d.get('bf16_tflops_sustained'),
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of the local GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception as ex:          # NVML missing: report that instead of inventing numbers
            self.nv, self.err = None, repr(ex)

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {'hw_slowdown': nv.nvmlClocksThrottleReasonHwSlowdown,
                 'hw_thermal_slowdown': nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 'sw_thermal_slowdown': nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 'sw_power_cap': nv.nvmlClocksThrottleReasonSwPowerCap}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.02)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                    'note': 'no NVML samples' + (': ' + self.err if self.nv is None else '')}
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2], 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


# --------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the oracle port of the reference training iteration on the host cores
# --------------------------------------------------------------------------------------------------
def log(msg):
    print(f'[bench {time.strftime("%H:%M:%S")}] {msg}', file=sys.stderr, flush=True)


def _ref_arm():
    """oracle/ref_arm.py, loaded by file path (the repo root is not importable in the reference legs)"""
    import importlib.util
    spec = importlib.util.spec_from_file_location('pidm_ref_arm', os.path.join(ROOT, 'oracle', 'ref_arm.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def run_reference(args, rank):
    """`--impl reference`: the reference's own training iteration on the host cores (unmodified modules from
    oracle/_ref when present, else the oracle port), `--steps` timed iterations after `--warmup` untimed ones."""
    if rank != 0:
        return
    r = _ref_arm().cpu_train_baseline(args.steps, args.warmup, PER_GPU_BATCH)
    out = {'metric': METRIC, 'value': r['value'], 'unit': 'samples/s', 'n_gpus': args.gpus, 'steps': r['steps'],
           'warmup': args.warmup, 'ms_per_step': r['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
           'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference',
           'config': {'workload': 'Darcy 64x64 PIDM train step (mean-mode x0), Unet3D dim=32, batch 32, host CPU',
                      'global_batch': PER_GPU_BATCH},
           'cpu_baseline': {k: r[k] for k in ('value', 'unit', 'cores', 'kind', 'sample')},
           'e2e': {'value': r['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
           'gpu_launches': 0}
    print(json.dumps(out), flush=True)


def run_side_leg(args):
    """internal legs spawned by the b200 arm: `--impl cpu_extras` (BASELINE.md 3.5 CPU timings) and `--impl torch_cuda`
    (the reference on the same B200 through stock PyTorch-CUDA)."""
    ra = _ref_arm()
    out = ra.cpu_extras() if args.impl == 'cpu_extras' else ra.torch_cuda_baselines(PER_GPU_BATCH)
    print(json.dumps(out), flush=True)


def spawn_leg(impl, timeout_s, *extra):
    """run `bench.py --impl <impl>` in a fresh process (own sys.path, own CUDA context) and parse its JSON line"""
    import subprocess
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', impl, *extra]
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'LOCAL_RANK', 'WORLD_SIZE', 'MASTER_ADDR', 'MASTER_PORT')}
    try:
        p = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=timeout_s, env=env,
                           cwd=ROOT)
        for line in p.stderr.splitlines():
            if line.startswith('[ref_arm'):
                print(line, file=sys.stderr, flush=True)
        lines = [l for l in p.stdout.splitlines() if l.startswith('{')]
        if p.returncode != 0 or not lines:
            return {'error': f'leg {impl} rc={p.returncode}: {p.stderr.strip().splitlines()[-1][:300] if p.stderr.strip() else ""}'}
        return json.loads(lines[-1])
    except subprocess.TimeoutExpired:
        return {'error': f'leg {impl} exceeded {timeout_s} s'}


# --------------------------------------------------------------------------------------------------
# this repo's arm
# --------------------------------------------------------------------------------------------------
def _graph_time_ms(orig_call, name, a, side):
    """Device time of one libpidm call: 20 launches captured into a CUDA graph on a private stream, replayed 5 times
    between two CUDA events (no host launch overhead, the conditions of the graph-replayed training step)."""
    a = list(a)
    a[-1] = side.cuda_stream                                  # the stream handle is the last argument of every entry point
    with torch.cuda.stream(side):
        orig_call(name, *a)
        side.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            for _ in range(20):
                orig_call(name, *a)
        g.replay()
        side.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(side)
        for _ in range(5):
            g.replay()
        e1.record(side)
        side.synchronize()
    return e0.elapsed_time(e1) / 100.0


def breakdown_one_step(engine, x0):
    """Per-entry-point device time of the libpidm calls of ONE step.  The calls (with their live operands) are recorded
    during an eager step; every distinct call is then timed by CUDA-graph replay with CUDA events on its stream
    (_graph_time_ms).  Calls that must not be repeated (the in-place optimizer update) keep the eager event time."""
    from physicsinformeddiffusionmodels_b200 import (_lib, ops, packing, denoising_utils, engine as eng_mod, residuals_darcy,
                                                     residuals_mechanics_K)
    records = []
    orig = _lib.call

    def timed(name, *a):
        if name in _lib._VALUE_RETURN:
            return orig(name, *a)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = orig(name, *a)
        e1.record()
        records.append((name, a, e0, e1))
        return r
    mods = [mo for mo in (ops, packing, denoising_utils, eng_mod, residuals_darcy, residuals_mechanics_K) if hasattr(mo, 'call')]
    for mo in mods:
        mo.call = timed
    world = engine.world
    engine.world = 1          # rank-local diagnostic step: no collective (the other ranks are not in this code path)
    try:
        engine._step_body(x0)
        torch.cuda.synchronize()
    finally:
        engine.world = world
        for mo in mods:
            mo.call = orig
    def key_of(name, a):
        return (name,) + tuple(x for x in a if isinstance(x, int) and not isinstance(x, bool) and x < (1 << 24))
    graph_ms = {}
    side = torch.cuda.Stream()
    for name, a, e0, e1 in records:
        k = key_of(name, a)
        if k in graph_ms or name in ('pidm_adam_ema_step',):
            continue
        try:
            graph_ms[k] = _graph_time_ms(orig, name, a, side)
        except Exception as ex:                                   # keep the eager number for this call
            log(f'graph timing of {name} failed ({ex}); using the eager event time')
            graph_ms[k] = None
    torch.cuda.synchronize()
    agg = {}
    detail = []
    for name, a, e0, e1 in records:
        ms = graph_ms.get(key_of(name, a))
        if ms is None:
            ms = e0.elapsed_time(e1)
        nbytes = 0.0
        detail.append((round(ms * 1e3, 1), name, [x for x in a if isinstance(x, int) and not isinstance(x, bool) and x < (1 << 24)][:14]))
        flop = 0.0
        if name == 'pidm_conv2d_tc_general':
            B, Hin, Win, Cin, Ho, Wo, Cout, KH, KW, stride, tr = (a[5], a[6], a[7], a[8], a[9], a[10], a[11], a[12], a[13],
                                                                 a[14], a[16])
            taps = KH * KW / (stride * stride) if tr else KH * KW
            flop = 2.0 * B * Ho * Wo * Cout * taps * Cin
            # algorithmic bytes: input + output (+ residual) activations in bf16, packed weights once
            nbytes = 2.0 * (B * Hin * Win * Cin + B * Ho * Wo * Cout * (2 if a[3] is not None else 1) + KH * KW * Cin * Cout)
        elif name == 'pidm_conv2d_simt':
            B, Cin, Ho, Wo, Cout, KH, KW, stride, tr = a[5], a[8], a[9], a[10], a[11], a[12], a[13], a[14], a[16]
            taps = KH * KW / (stride * stride) if tr else KH * KW       # useful taps of the transposed gather
            flop = 2.0 * B * Ho * Wo * Cout * taps * Cin
        elif name == 'pidm_conv2d_wgrad_tc':
            B, CAr, GH, GW, CB, KH, KW = a[3], a[7], a[8], a[9], a[10], a[11], a[12]
            flop = 2.0 * B * GH * GW * CB * KH * KW * CAr
        elif name == 'pidm_conv2d_wgrad_simt':
            B, Cin, Ho, Wo, Cout, KH, KW, stride, tr = a[4], a[7], a[9], a[10], a[11], a[12], a[13], a[14], a[16]
            taps = KH * KW / (stride * stride) if tr else KH * KW
            flop = 2.0 * B * Ho * Wo * Cout * taps * Cin
        d = agg.setdefault(name, {'ms': 0.0, 'calls': 0, 'flop': 0.0, 'bytes': 0.0})
        d['ms'] += ms
        d['calls'] += 1
        d['flop'] += flop
        d['bytes'] += nbytes
    if os.environ.get('PIDM_BENCH_DETAIL'):
        with open(os.environ['PIDM_BENCH_DETAIL'], 'w') as f:
            for us, name, ints in sorted(detail, key=lambda r: -r[0]):
                f.write(f'{us:9.1f} us  {name:28s} {ints}\n')
    return agg


def sampling_bench(model, dev, n_steps=250, batches=(16, 64, 256)):
    """BASELINE.json configs[3]: ancestral sampling loop with per-step Darcy residual evaluation (engine.SampleEngine: 10
    steps per captured CUDA graph, weights packed once per loop, initial noise drawn on the device), device-timed, at
    three batch sizes in mean mode (x0 = network output) and at batch 16 with `x0_estimation: sample` (two network calls
    per step + the DDIM jump, reference ddim_steps = 0)."""
    from physicsinformeddiffusionmodels_b200.denoising_utils import DenoisingDiffusion
    from physicsinformeddiffusionmodels_b200.engine import SampleEngine
    from physicsinformeddiffusionmodels_b200.residuals_darcy import ResidualsDarcy
    was_training = model.training
    model.eval()
    diff = DenoisingDiffusion(n_steps, dev)

    def run(batch, use_ddim_x0):
        res = ResidualsDarcy(model=model, fd_acc=2, pixels_per_dim=64, pixels_at_boundary=True, reverse_d1=True, device=dev,
                             bcs='none', domain_length=1., use_ddim_x0=use_ddim_x0, ddim_steps=0)
        eng = SampleEngine(model, diff, res, batch=batch)
        eng.sample()                                      # captures the graph + one full warm-up loop
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        x, r, _ = eng.sample()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        return {'batch': batch, 'ms_per_loop': ms, 'ms_per_step': ms / n_steps, 'samples_per_s': batch / (ms * 1e-3),
                'final_abs_residual_mean': float(r.abs().mean().item()), 'finite': bool(torch.isfinite(x).all().item())}
    out = {'workload': f'Darcy 64x64 ancestral sampling (p_sample_loop), {n_steps} steps, Darcy residual evaluated every step, '
                       'bf16 activations, 10 steps per CUDA graph', 'mean_mode': [run(b, False) for b in batches],
           'sample_mode_ddim0': run(batches[0], True)}
    best = max(out['mean_mode'], key=lambda d: d['samples_per_s'])
    out.update({k: best[k] for k in ('batch', 'ms_per_loop', 'ms_per_step', 'samples_per_s')})      # headline: best batch
    model.train(was_training)
    return out


def mechanics_bench(dev, pk, batch=32, steps=10, warmup=4):
    """BASELINE.json configs[2]: topology-optimisation (mechanics) 64x64, PIDM loss, batch 32, one B200 -- the model the
    reference trains for this study, Unet3D(dim=128, channels=10, out_dim=3, sigmoid_last_channel=True) (main.py:102-109,
    126), through TrainEngine (CUDA graph), device-timed; plus the matrix-free residual kernel against the HBM roofline
    on a working set larger than L2."""
    from physicsinformeddiffusionmodels_b200 import ops
    from physicsinformeddiffusionmodels_b200._lib import call, stream
    from physicsinformeddiffusionmodels_b200.denoising_utils import DenoisingDiffusion
    from physicsinformeddiffusionmodels_b200.engine import TrainEngine
    from physicsinformeddiffusionmodels_b200.residuals_mechanics_K import ResidualsMechanics
    from physicsinformeddiffusionmodels_b200.unet_model import Unet3D
    torch.manual_seed(0)
    model = Unet3D(dim=128, channels=10, out_dim=3, sigmoid_last_channel=True).to(dev)
    n_params = sum(p.numel() for p in model.parameters() if p.requires_grad)
    diff = DenoisingDiffusion(100, dev)
    res = ResidualsMechanics(model=model, pixels_per_dim=64, pixels_at_boundary=True, no_BC_folder='', device=dev)
    eng = TrainEngine(model, diff, res, lr=1e-4, max_norm=1.0, ema_mu=0.99, c_data=1.0, c_residual=1e-2, c_ineq=0.,
                      lambda_opt=1e-3, use_graph=True)
    g = torch.Generator(device='cpu').manual_seed(5)
    cond = torch.rand(batch, 3, 65, 65, generator=g)
    cond[:, 0] = (0.3 + 0.4 * torch.rand(batch, generator=g))[:, None, None]
    x0 = torch.cat((0.2 * torch.randn(batch, 2, 65, 65, generator=g), torch.rand(batch, 1, 65, 65, generator=g).clamp(1e-3, 1.)), 1)
    bcs = torch.zeros(batch, 4, 65, 65)
    bcs[:, 0, :, 0] = 1.; bcs[:, 1, :, 0] = 1.; bcs[:, 3, 32, 64] = -1.
    inp = torch.cat((cond, x0, bcs), dim=1).to(dev)
    for _ in range(warmup):
        out = eng.step(inp)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = eng.step(inp)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    gf_sample = 47.3 * 3                       # SURVEY 8d: 47.3 GFLOP/sample forward, x3 for fwd + bwd
    r = {'workload': f'mechanics (topology optimisation) 64x64 PIDM train step, Unet3D(dim=128, ch=10, out=3), batch {batch}, '
                     'bf16 activations, CUDA graph, c_residual=1e-2, lambda_opt=1e-3 (configs[2])',
         'trainable_parameters': n_params, 'ms_per_step': ms, 'samples_per_s': batch / (ms * 1e-3),
         'model_tflops_at_value': gf_sample * batch / (ms * 1e-3) / 1e3, 'last_loss': float(out[0].item()),
         'finite': bool(torch.isfinite(out[0]).item())}
    try:      # the same convolution kernels at 128 .. 1024 channels: per-entry-point device time of one step
        agg = breakdown_one_step(eng, inp)
        peak = pk['bf16_sustained'] or pk['bf16_tflops']
        conv = agg.get('pidm_conv2d_tc_general')
        if conv and conv['flop']:
            tf = conv['flop'] / (conv['ms'] * 1e-3) / 1e12
            r['roofline_conv'] = {'bound': 'tensor', 'kernel': 'pidm_conv2d_tc_general (the convolution kernels of the headline '
                                  'workload, here at 128-1024 channels)', 'achieved': tf, 'peak': peak, 'unit': 'TFLOP/s',
                                  'frac': tf / peak, 'ms': conv['ms'], 'launches_per_step': conv['calls'], 'traffic': None,
                                  'how': 'as roofline.how: algorithmic FLOPs / CUDA-graph-replayed device time of every launch'}
        tot = sum(v['ms'] for v in agg.values())
        r['kernel_time_breakdown_ms'] = {k: {'ms': round(v['ms'], 4), 'calls': v['calls'],
                                             'tflops': (v['flop'] / (v['ms'] * 1e-3) / 1e12) if v['flop'] else None}
                                         for k, v in sorted(agg.items(), key=lambda kv: -kv[1]['ms'])[:8]}
        r['kernel_time_total_ms'] = tot
    except Exception as ex:
        r['roofline_conv'] = {'error': repr(ex)[:300]}
    eng.close()
    del eng, model
    torch.cuda.empty_cache()
    # ---- residual kernel alone, B = 8192 (1.24 GB working set >> 126 MB L2)
    Bs = 8192
    u = torch.randn(Bs, 2, 65, 65, device=dev) * 0.1
    rho = torch.rand(Bs, 64, 64, device=dev)
    bc = torch.zeros(Bs, 4, 65, 65, device=dev)
    bc[:, 0, :, 0] = 1.; bc[:, 1, :, 0] = 1.; bc[:, 3, 32, 64] = -1.
    rr = torch.empty(Bs, 8450, device=dev)
    cc = torch.empty(Bs, device=dev)
    fn = lambda: call('pidm_mechanics_residual_fwd', u, rho, bc, res.KE, rr, cc, Bs, 64, stream())
    for _ in range(3):
        fn()
    e0.record()
    for _ in range(10):
        fn()
    e1.record()
    torch.cuda.synchronize()
    ms_k = e0.elapsed_time(e1) / 10
    alg = Bs * (2 * 4225 + 4096 + 4 * 4225 + 8450) * 4          # read u, rho, bcs; write residual (SURVEY 8d: ~152 KB/sample)
    gbs = alg / ms_k / 1e6
    r['roofline_mechanics'] = {'bound': 'hbm', 'kernel': 'mech_node_kernel<0> (pidm_mechanics_residual_fwd), B=8192 standalone sweep',
                               'achieved': gbs, 'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': gbs / pk['hbm_gbs'],
                               'traffic': None, 'ms_per_launch': ms_k, 'algorithmic_bytes': alg,
                               'reference_path_bytes_per_sample': 285.6e6 * 4,
                               'note': 'matrix-free K(rho)u - f; the reference assembles a dense 8450 x 8450 stiffness matrix '
                                       '(285.6 MB per sample, written >= 4 times)'}
    return r


def residual_kernel_sweep(pk):
    """Standalone HBM sweep of the Darcy residual kernel at B = 32768 (2.7 GB working set >> 126 MB L2)."""
    from physicsinformeddiffusionmodels_b200 import ops
    from physicsinformeddiffusionmodels_b200._lib import call, stream
    Bs = 32768
    x = torch.randn(Bs, 2, 64, 64, device='cuda')
    fs = torch.zeros(4096, device='cuda')
    fs[:8 * 64].view(8, 64)[:, :8] = 10.0
    r = torch.empty(Bs, 4096, 3, device='cuda')
    res = {}
    for mode in ('fwd', 'loss'):
        if mode == 'loss':
            tgt = torch.randn_like(x)
            t = torch.randint(0, 100, (Bs,), device='cuda')
            tab = torch.rand(100, device='cuda') + 0.1
            sums = torch.zeros(3, device='cuda')
            gx = torch.empty_like(x)
            fn = lambda: call('pidm_darcy_pidm_loss', x, x, tgt, fs, t, tab, tab, 1.0, 1e-3, sums, gx, None, Bs, 64, 1.0,
                              1, 1, stream())
            alg_bytes = Bs * (2 * 4096 * 4 * 3)        # read x0_hat + target, write gradient
        else:
            fn = lambda: call('pidm_darcy_residual_fwd', x, fs, r, Bs, 64, 1.0, 1, 1, stream())
            alg_bytes = Bs * 81920                     # SURVEY.md 8d: read 2*P^2*4, write 3*P^2*4 per sample
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 10
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        res[mode] = dict(ms=ms, gbs=alg_bytes / ms / 1e6, bytes=alg_bytes)
    g = res['fwd']['gbs']
    return {'bound': 'hbm', 'kernel': 'darcy_kernel<0> (pidm_darcy_residual_fwd), B=32768 standalone sweep',
            'achieved': g, 'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': g / pk['hbm_gbs'], 'traffic': None,
            'peak_source': pk['source'], 'ms_per_launch': res['fwd']['ms'], 'algorithmic_bytes': res['fwd']['bytes'],
            'fused_loss_grad_variant': {'achieved': res['loss']['gbs'], 'frac': res['loss']['gbs'] / pk['hbm_gbs'],
                                        'ms_per_launch': res['loss']['ms'], 'algorithmic_bytes': res['loss']['bytes']}}


DUMP_SAMPLE = 1 << 22      # sampled parameter positions: params + EMA = 2 x 16.8 MB of float32


def dump_step_outputs(path, eng, out):
    """`--dump-outputs DIR`: what the last timed step handed its caller, as DIR/<name>.npy in float32 -- the values
    TrainEngine.step returns (loss, data_loss, residual_abs_mean) and the weights it left in the model (params_sample,
    and their EMA shadow ema_sample).  The weights are the trainable parameters flattened in named_parameters() order
    and sampled at DUMP_SAMPLE fixed positions (seeded, ascending), so that two builds can be compared position by
    position.  The inputs are the same in every run, but weight gradients are summed with fp32 atomics and the
    optimizer steps before the dump amplify that rounding: two runs of `--steps 20 --warmup 5` on one B200 (1000 W
    power limit) agreed to 0.3 % in the loss and 1e-3 in the weights.  Call before any further step: the returned
    tensors are the graph's static outputs."""
    import numpy as np
    named = [(n, p) for n, p in eng.model.named_parameters() if p.requires_grad]
    ema = eng.ema_state_dict()
    n_total = sum(p.numel() for _, p in named)
    idx = torch.randperm(n_total, generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    idx = idx.to(out[0].device)
    arrays = dict(zip(('loss', 'data_loss', 'residual_abs_mean'), out))
    arrays['params_sample'] = torch.cat([p.detach().reshape(-1) for _, p in named])[idx]
    arrays['ema_sample'] = torch.cat([ema[n].reshape(-1) for n, _ in named])[idx]
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(path, name + '.npy'), t.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step computed to DIR/<name>.npy (b200 arm)')
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference', 'cpu_extras', 'torch_cuda'])
    ap.add_argument('--no-torch-cuda-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-sampling', action='store_true')
    ap.add_argument('--no-mechanics', action='store_true')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to the b200 arm')
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'reference':
        return run_reference(args, rank)
    if args.impl in ('cpu_extras', 'torch_cuda'):
        return run_side_leg(args)
    assert args.warmup >= 3, 'timing rules: at least 3 warm-up steps'
    import torch.distributed as dist
    from physicsinformeddiffusionmodels_b200 import _lib, ops
    from physicsinformeddiffusionmodels_b200.denoising_utils import DenoisingDiffusion
    from physicsinformeddiffusionmodels_b200.engine import TrainEngine
    from physicsinformeddiffusionmodels_b200.residuals_darcy import ResidualsDarcy
    from physicsinformeddiffusionmodels_b200.unet_model import Unet3D
    assert torch.cuda.is_available(), 'bench.py (b200 arm) needs a CUDA device; there is no CPU fallback'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    assert world == args.gpus, f'--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)'
    if world > 1:
        # the secondary workloads and the CPU / stock-PyTorch baselines are single-GPU legs (reported at N = 1 only): at
        # N > 1 the other ranks would sit in a barrier for minutes while rank 0 runs them
        args.no_cpu_baseline = args.no_sampling = args.no_mechanics = args.no_torch_cuda_baseline = True
    ops.set_precision('bf16')
    torch.manual_seed(0)                              # identical initial weights on every rank
    model = Unet3D(dim=32, channels=2).to(dev)
    diff = DenoisingDiffusion(100, dev)
    res = ResidualsDarcy(model=model, fd_acc=2, pixels_per_dim=64, pixels_at_boundary=True, reverse_d1=True, device=dev,
                         bcs='none', domain_length=1.)
    # data parallel: t / eps are drawn for the GLOBAL batch from a generator that is identical on every rank and sliced
    # to the rank's rows (SURVEY 8e: the N-rank job consumes the random numbers of the one-process run on N*32 samples)
    eng = TrainEngine(model, diff, res, lr=1e-4, max_norm=1.0, ema_mu=0.99, c_data=1.0, c_residual=1e-3,
                      use_graph=not args.no_graph, world=world, rank=rank, global_draws=True)
    B = PER_GPU_BATCH
    gdata = torch.Generator().manual_seed(1234 + rank)                     # different data per rank
    x0_dev = torch.randn(B, 2, 64, 64, generator=gdata).to(dev)
    x0_host = torch.randn(B, 2, 64, 64, generator=gdata).pin_memory()
    torch.cuda.manual_seed(1234)                                          # identical noise stream on every rank
    loss_host = torch.zeros(1).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ------------------------------------------------------------------------------
    import faulthandler
    faulthandler.dump_traceback_later(240, repeat=True, file=sys.stderr)
    log('warm-up (first call captures the CUDA graph)')
    for _ in range(args.warmup):
        eng.step(x0_dev)
    barrier()
    log('timed region')
    launches0 = _lib.launch_count
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = eng.step(x0_dev)
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1)
    last_loss = float(out[0].item())
    log(f'device-resident: {ms / args.steps:.3f} ms/step')
    if args.dump_outputs and rank == 0:
        dump_step_outputs(args.dump_outputs, eng, out)
    # ---- end to end: pinned host batch -> H2D -> step -> D2H loss, every step ------------------------------------
    for _ in range(3):
        x0_dev.copy_(x0_host, non_blocking=True)
        loss_host.copy_(eng.step(x0_dev)[0].reshape(1), non_blocking=True)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        x0_dev.copy_(x0_host, non_blocking=True)
        loss_host.copy_(eng.step(x0_dev)[0].reshape(1), non_blocking=True)
        torch.cuda.current_stream().synchronize()    # the caller reads the loss every step
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    # kernels per step: count libpidm entry calls of one eager step (each call launches >= 1 kernel)
    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()

    extra = {}
    if rank == 0:
        log(f'e2e: {ms_e2e / args.steps:.3f} ms/step; per-kernel breakdown of one eager step')
        pk = peaks()
        c0 = _lib.launch_count
        agg = breakdown_one_step(eng, x0_dev)
        calls_per_step = _lib.launch_count - c0
        total_ms = sum(d['ms'] for d in agg.values())
        top = sorted(agg.items(), key=lambda kv: -kv[1]['ms'])
        name, d = top[0]
        tensor_names = ('pidm_conv2d_tc_general', 'pidm_conv2d_simt', 'pidm_conv2d_wgrad_simt',
                        'pidm_conv2d_wgrad_tc')
        if name in tensor_names and d['flop'] > 0:
            ach = d['flop'] / (d['ms'] * 1e-3) / 1e12
            peak = pk['bf16_sustained'] or pk['bf16_tflops']
            roof = {'bound': 'tensor', 'kernel': name, 'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s',
                    'frac': ach / peak, 'traffic': None, 'launches_per_step': d['calls'],
                    'share_of_step_kernel_time': d['ms'] / total_ms, 'peak_source': pk['source'] + ', sustained figure',
                    'how': 'algorithmic 2*M*N*K FLOPs of every launch of this entry point in one step / device time of '
                           'those launches (each distinct call replayed from a CUDA graph, CUDA events on its stream)'}
            if d.get('bytes'):
                # the U-Net is narrow (32..256 channels): its convolutions are bound by operand / activation movement
                # long before the tensor pipe, so the same launches are also reported against the HBM roofline
                roof['algorithmic_bytes'] = d['bytes']
                roof['hbm_view'] = {'achieved': d['bytes'] / (d['ms'] * 1e-3) / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
                                    'frac': d['bytes'] / (d['ms'] * 1e-3) / 1e9 / pk['hbm_gbs']}
            prof = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles')
            tpath = next((os.path.join(prof, f) for f in ('r02_step_traffic.json', 'r01_step_traffic.json')
                          if os.path.exists(os.path.join(prof, f))), None)
            if tpath:
                prefix = {'pidm_conv2d_tc_general': 'conv_tc_kernel',
                          'pidm_conv2d_wgrad_tc': 'wgrad'}.get(name)
                if prefix:
                    tr = json.load(open(tpath))
                    roof['traffic'] = sum(v['dram_bytes'] for k, v in tr.items() if k.startswith(prefix))
                    roof['traffic_note'] = ('STATIC, not measured in this run: dram__bytes_read.sum + dram__bytes_write.sum summed '
                                            'over the launches of this kernel in ONE step, from the committed ncu launch '
                                            f'list profiles/{os.path.basename(tpath)} (same command, scripts/gpu_final.sh); '
                                            'compare with algorithmic_bytes')
        else:
            roof = {'bound': 'hbm', 'kernel': name, 'achieved': None, 'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': None,
                    'traffic': None, 'share_of_step_kernel_time': d['ms'] / total_ms}
        extra['roofline'] = roof
        log('residual kernel sweep')
        extra['roofline_residual'] = residual_kernel_sweep(pk)
        extra['kernel_time_breakdown_ms'] = {k: {'ms': round(v['ms'], 4), 'calls': v['calls'],
                                                 'tflops': (v['flop'] / (v['ms'] * 1e-3) / 1e12) if v['flop'] else None}
                                             for k, v in top[:12]}
        extra['gpu_launches'] = calls_per_step * args.steps * world
        extra['launches_note'] = (f'{calls_per_step} libpidm entry-point calls per step per GPU (each issues 1-3 kernels); '
                                  'replayed from a CUDA graph' if not args.no_graph else 'eager')
        if not args.no_sampling:
            log('sampling loop (configs[3]): 250 ancestral steps, batch 16 / 64 / 256, mean and sample mode')
            extra['sampling'] = sampling_bench(model, dev)
        if not args.no_mechanics:
            log('mechanics workload (configs[2]): Unet3D(dim=128), batch 32')
            try:
                extra['mechanics'] = mechanics_bench(dev, pk)
            except Exception as ex:                      # a secondary workload must not take the headline line down
                extra['mechanics'] = {'error': repr(ex)[:400]}
        if not args.no_torch_cuda_baseline:
            log('torch_cuda_baseline: the reference on this GPU through stock PyTorch-CUDA (subprocess)')
            extra['torch_cuda_baseline'] = spawn_leg('torch_cuda', 240)
        if not args.no_cpu_baseline:
            log('cpu_baseline: the reference training iteration on the host cores (subprocess)')
            cb = spawn_leg('reference', 300, '--steps', '3', '--warmup', '1')
            extra['cpu_baseline'] = cb.get('cpu_baseline', cb)
            log('cpu extras: residual operator and p_sample_loop of the reference on the host cores (subprocess)')
            extra['cpu_baseline_extras'] = spawn_leg('cpu_extras', 300)
    if world > 1:
        dist.barrier()
    if rank == 0:
        faulthandler.cancel_dump_traceback_later()
        sps = world * B * args.steps / (ms * 1e-3)
        sps_e2e = world * B * args.steps / (ms_e2e * 1e-3)
        tflops = 3 * FWD_GFLOP_PER_SAMPLE * 1e9 * sps / 1e12
        out = {'metric': METRIC, 'value': sps, 'unit': 'samples/s', 'n_gpus': world, 'steps': args.steps,
               'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
               'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
               'config': {'workload': 'Darcy 64x64 PIDM train step: q_sample + Unet3D(dim=32,ch=2) fwd/bwd + Darcy '
                                      'residual loss + clip + Adam + EMA (configs[1])',
                          'global_batch': world * B, 'per_gpu_batch': B, 'parallelism': f'dp{world}',
                          'cuda_graph': not args.no_graph,
                          'l2': 'no explicit flush: one step streams >1 GB of activations and gradients (dqkv alone 201 MB) '
                                'through the 126 MB L2, so weights/activations are cold at every layer',
                          'model_tflops_at_value': tflops, 'last_loss': last_loss},
               'clocks': clocks,
               'e2e': {'value': sps_e2e, 'unit': 'samples/s', 'ms_per_step': ms_e2e / args.steps,
                       'h2d_bytes_per_step': world * x0_host.numel() * 4, 'd2h_bytes_per_step': world * 4,
                       'api': 'pinned host batch -> TrainEngine.step -> loss read back, every step'}}
        out.update(extra)
        print(json.dumps(out), flush=True)
    if world > 1:
        # orderly teardown: the captured graphs hold NCCL kernels, so they go first, then the communicator
        faulthandler.cancel_dump_traceback_later()
        sys.stdout.flush()
        sys.stderr.flush()
        watchdog = threading.Timer(60.0, lambda: os._exit(0))   # the result is printed: a stuck teardown must not stall the driver
        watchdog.daemon = True
        watchdog.start()
        eng.close()
        dist.barrier()
        dist.destroy_process_group()
        watchdog.cancel()


if __name__ == '__main__':
    main()
