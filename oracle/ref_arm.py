"""Reference arm of bench.py.  TEST / MEASUREMENT INFRASTRUCTURE ONLY -- never imported by the product package.

Runs the UNMODIFIED reference modules (jhbastek/PhysicsInformedDiffusionModels `src/*.py`) through the import shims in
oracle/ref_shims/ (SURVEY.md section 8c: einops_exts, rotary_embedding_torch, findiff, solidspy, matplotlib, imageio):

* on the host CPU cores  -> `bench.py --impl reference` / the `cpu_baseline` block       (kind = "reference")
* on the B200 through stock PyTorch-CUDA (cuDNN / cuBLAS) -> the `torch_cuda_baseline` block, the comparison point
  SURVEY 2b / BASELINE.md 3.7 ask for (the reference ships no GPU kernels of its own)

The reference sources are NOT part of this repository: `__graft_entry__.build()` copies them into the git-ignored
oracle/_ref/ when the original project is at hand (oracle/fetch_reference.py).  When oracle/_ref/ is absent every
function here falls back to the oracle port (oracle/pidm_oracle.py, kind = "port") and says so.

This module must be loaded BY FILE PATH in a process whose sys.path does not contain the repo root: the repo's `src/`
drop-in package (a regular package) would shadow the reference's `src/` (a namespace package) regardless of order.
"""
import importlib.util
import os
import sys
import time
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF_DIR = os.path.join(HERE, '_ref')


def reference_available():
    return os.path.isfile(os.path.join(REF_DIR, 'src', 'unet_model.py'))


def _load_oracle():
    spec = importlib.util.spec_from_file_location('pidm_oracle', os.path.join(HERE, 'pidm_oracle.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_reference():
    """-> namespace with the reference's classes.  Call once, before anything imported `src`."""
    sys.path[:] = [p for p in sys.path if os.path.abspath(p or '.') != ROOT]
    sys.path.insert(0, os.path.join(HERE, 'ref_shims'))
    sys.path.insert(0, REF_DIR)
    warnings.filterwarnings('ignore')
    import src.unet_model as um
    assert os.path.abspath(um.__file__).startswith(REF_DIR), f'wrong src package on the path: {um.__file__}'
    import src.denoising_utils as du
    import src.residuals_darcy as rd
    return dict(Unet3D=um.Unet3D, DenoisingDiffusion=du.DenoisingDiffusion, EMA=du.EMA, ResidualsDarcy=rd.ResidualsDarcy,
                du=du)


def usable_cores():
    """Cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open('/sys/fs/cgroup/cpu/cpu.cfs_quota_us').read())
            per = int(open('/sys/fs/cgroup/cpu/cpu.cfs_period_us').read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


def log(msg):
    print(f'[ref_arm {time.strftime("%H:%M:%S")}] {msg}', file=sys.stderr, flush=True)


class _Timer:
    """wall clock on the CPU, CUDA events on the GPU"""

    def __init__(self, device):
        import torch
        self.cuda = str(device).startswith('cuda')
        self.torch = torch

    def __enter__(self):
        if self.cuda:
            self.e0, self.e1 = self.torch.cuda.Event(enable_timing=True), self.torch.cuda.Event(enable_timing=True)
            self.torch.cuda.synchronize()
            self.e0.record()
        else:
            self.t0 = time.perf_counter()
        return self

    def __exit__(self, *a):
        if self.cuda:
            self.e1.record()
            self.torch.cuda.synchronize()
            self.seconds = self.e0.elapsed_time(self.e1) * 1e-3
        else:
            self.seconds = time.perf_counter() - self.t0


# ------------------------------------------------------------------------------------------------------------------
# the training iteration of the reference, main.py:157-183, on `device`
# ------------------------------------------------------------------------------------------------------------------
def build_reference_step(ref, device, batch):
    """model / diffusion / residuals / optimizer / EMA exactly as main.py:116-143 builds them for gov_eqs='darcy'."""
    import torch
    ref['du'].device = torch.device(device)          # the module-level `device` the reference reads at :322
    torch.manual_seed(0)
    model = ref['Unet3D'](dim=32, channels=2).to(device)
    diff = ref['DenoisingDiffusion'](100, device)
    res = ref['ResidualsDarcy'](model=model, fd_acc=2, pixels_per_dim=64, pixels_at_boundary=True, reverse_d1=True,
                                device=device, bcs='none', domain_length=1.)
    opt = torch.optim.Adam(model.parameters(), lr=1.e-4)
    ema = ref['EMA'](0.99)
    ema.register(model)
    x0 = torch.randn(batch, 2, 64, 64, device=device)

    def step():
        model.train()
        loss, data_loss, residual_loss, _, _ = diff.model_estimation_loss(
            x0, residual_func=res, c_data=1., c_residual=1e-3, c_ineq=0., lambda_opt=0.)
        opt.zero_grad()
        loss.backward()
        torch.nn.utils.clip_grad_norm_(model.parameters(), 1.)
        opt.step()
        ema.update(model)                              # steady state of the loop (iteration > ema_start)
        return loss
    return step, model, diff, res


def build_port_step(device, batch, channels_last=False):
    """the oracle restatement of the same iteration (functional F.conv2d / group_norm / einsum, autograd, Adam, EMA)"""
    import torch
    O = _load_oracle()
    cfg = O.unet_config(dim=32, channels=2)
    sd = O.make_test_state_dict(cfg, 0)
    sdr = {k: v.to(device).clone().requires_grad_('freqs' not in k) for k, v in sd.items()}
    train = [v for v in sdr.values() if v.requires_grad]
    m = [torch.zeros_like(p) for p in train]
    v = [torch.zeros_like(p) for p in train]
    ema = [p.detach().clone() for p in train]
    tables = {k: t.to(device) for k, t in O.diffusion_tables(100).items()}
    if str(device).startswith('cuda'):
        # the restatement builds the source field on the host at every call: keep one device copy (CUDA-graph capture
        # cannot contain a pageable host-to-device copy)
        fs = {}
        orig_source = O.darcy_source

        def cached_source(pixels=64, w=0.125, r=10.0, dtype=torch.float32):
            key = (pixels, dtype)
            if key not in fs:
                fs[key] = orig_source(pixels, w, r, dtype).to(device)
            return fs[key]
        O.darcy_source = cached_source
    torch.manual_seed(0)
    x0 = torch.randn(batch, 2, 64, 64, device=device)
    state = {'it': 0}

    def step():
        t = torch.randint(0, 100, (batch,), device=device)
        e = torch.randn_like(x0)
        for p in train:
            p.grad = None
        loss, _ = O.darcy_training_loss(sdr, cfg, x0, t, e, tables, 1.0, 1e-3)
        loss.backward()
        with torch.no_grad():
            grads = [p.grad if p.grad is not None else torch.zeros_like(p) for p in train]
            state['it'] += 1
            O.adam_ema_step(train, grads, m, v, ema, state['it'])
        return loss
    return step


def time_steps(step, device, steps, warmup, sync_each=True):
    import torch
    for _ in range(warmup):
        step()
    times = []
    for it in range(steps):
        with _Timer(device) as tm:
            out = step()
            if sync_each and str(device).startswith('cuda'):
                float(out)                              # the loop reads the loss (pbar / logging)
        times.append(tm.seconds)
    return times


def cpu_train_baseline(steps, warmup, batch=32):
    import torch
    ncores = usable_cores()
    torch.set_num_threads(ncores)
    if reference_available():
        ref = load_reference()
        step, *_ = build_reference_step(ref, 'cpu', batch)
        kind, what = 'reference', 'unmodified reference modules (oracle/_ref/src) + import shims'
    else:
        step = build_port_step('cpu', batch)
        kind, what = 'port', 'oracle/pidm_oracle.py restatement (oracle/_ref is absent)'
    log(f'cpu train baseline: kind={kind}, {ncores} usable cores (os.cpu_count()={os.cpu_count()}), batch {batch}')
    times = time_steps(step, 'cpu', steps, warmup, sync_each=False)
    sec = sum(times) / len(times)
    return dict(value=batch / sec, unit='samples/s', cores=ncores, kind=kind, ms_per_step=sec * 1e3, steps=len(times),
                sample=f'{len(times)} training iterations (main.py:157-183 body: loss, backward, clip, Adam, EMA) at batch '
                       f'{batch} after {warmup} warm-up, torch {torch.__version__} CPU fp32, {ncores} threads; {what}')


def cpu_extras(budget_s=120.0):
    """BASELINE.md 3.5: the reference's residual operator alone (fwd, fwd+bwd) at B=32 and B=4096, and its
    p_sample_loop (100-step schedule, B=8, per-step residual) -- a bounded number of steps, extrapolated."""
    import torch
    ncores = usable_cores()
    torch.set_num_threads(ncores)
    out = {'cores': ncores}
    if not reference_available():
        out['unavailable'] = 'oracle/_ref is absent'
        return out
    ref = load_reference()
    _, model, diff, res = build_reference_step(ref, 'cpu', 2)
    out['kind'] = 'reference'
    for B in (32, 4096):
        x = torch.randn(B, 2, 64, 64)
        res.compute_residual(x[:2], pass_through=True)
        t0 = time.perf_counter()
        res.compute_residual(x, pass_through=True)
        fwd = time.perf_counter() - t0
        xg = x.clone().requires_grad_(True)
        t0 = time.perf_counter()
        r = res.compute_residual(xg, pass_through=True)['residual']
        (r * r).sum().backward()
        fb = time.perf_counter() - t0
        out[f'residual_operator_B{B}'] = {
            'fwd_ms': fwd * 1e3, 'fwd_bwd_ms': fb * 1e3, 'fwd_gbs_algorithmic': B * 81920 / fwd / 1e9,
            'fwd_bwd_gbs_algorithmic': B * (81920 + 114688) / fb / 1e9,
            'note': 'ResidualsDarcy.compute_residual(pass_through=True), residuals_darcy.py:106-207; algorithmic bytes '
                    '81,920 B/sample fwd + 114,688 B/sample bwd (SURVEY 8d)'}
        log(f'residual operator B={B}: fwd {fwd * 1e3:.1f} ms, fwd+bwd {fb * 1e3:.1f} ms')
    # sampling: every step of the loop costs the same (one network call + residual), so time `n_run` steps
    model.eval()
    B, n_run = 8, 10
    d = ref['DenoisingDiffusion'](n_run, 'cpu')
    t0 = time.perf_counter()
    d.p_sample_loop(None, (B, 2, 64, 64), save_output=True, surpress_noise=True, residual_func=res, eval_residuals=True)
    sec = time.perf_counter() - t0
    per_step = sec / n_run
    out['p_sample_loop'] = {'batch': B, 'steps_timed': n_run, 's_per_step': per_step,
                            's_per_100_step_loop_extrapolated': per_step * 100,
                            'samples_per_s_250_steps_extrapolated': B / (per_step * 250),
                            'note': 'DenoisingDiffusion.p_sample_loop (denoising_utils.py:494-545) with per-step residual '
                                    f'evaluation, {n_run} steps timed (every step = one network call + residual), '
                                    'extrapolated linearly to 100 / 250 steps'}
    log(f'p_sample_loop B={B}: {per_step:.3f} s per step')
    return out


def torch_cuda_baselines(batch=32, steps=10, warmup=3):
    """The same reference code on the B200 via stock PyTorch-CUDA kernels: eager fp32 (TF32 off), TF32, bf16 autocast
    (+ channels_last for the port), and the port under a CUDA graph.  Device-timed per step."""
    import torch
    assert torch.cuda.is_available()
    dev = 'cuda'
    out = {'batch': batch, 'torch': torch.__version__, 'cudnn': torch.backends.cudnn.version(),
           'note': 'one iteration of main.py:157-183 (loss, backward, clip, Adam, EMA) per step, CUDA events around each '
                   'step incl. the loss read-back the loop does; reference = unmodified modules, port = oracle restatement'}

    def run(name, step, **ctx):
        try:
            times = time_steps(step, dev, steps, warmup)
            ms = 1e3 * sorted(times)[len(times) // 2]
            out[name] = {'ms_per_step': ms, 'samples_per_s': batch / (ms * 1e-3), **ctx}
            log(f'torch-cuda {name}: {ms:.2f} ms/step')
        except Exception as ex:                                     # report, never hide
            out[name] = {'error': repr(ex)[:300]}
            log(f'torch-cuda {name}: FAILED {ex!r}')

    def set_tf32(on):
        torch.backends.cuda.matmul.allow_tf32 = on
        torch.backends.cudnn.allow_tf32 = on
    torch.backends.cudnn.benchmark = True
    if reference_available():
        ref = load_reference()
        step, model, diff, res = build_reference_step(ref, dev, batch)
        set_tf32(False)
        run('reference_eager_fp32', step, kind='reference')
        set_tf32(True)
        run('reference_eager_tf32', step, kind='reference')

        def step_amp():
            with torch.autocast('cuda', dtype=torch.bfloat16):
                return step()
        run('reference_autocast_bf16', step_amp, kind='reference',
            note='torch.autocast(bfloat16) around the whole iteration; the residual operator then also runs in bf16 for '
                 'its conv2d stencils, which the reference never does -- speed only, not a valid training setup')
    else:
        out['reference'] = {'unavailable': 'oracle/_ref is absent'}
    set_tf32(False)
    pstep = build_port_step(dev, batch)
    run('port_eager_fp32', pstep, kind='port')
    set_tf32(True)
    run('port_eager_tf32', pstep, kind='port')
    # CUDA graph of the port iteration (TF32): functional code, no host syncs inside
    try:
        gstep = build_port_step(dev, batch)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            for _ in range(3):
                gstep()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            static_loss = gstep()

        def replay():
            g.replay()
            return static_loss
        run('port_cuda_graph_tf32', replay, kind='port', note='whole iteration captured once, replayed')
    except Exception as ex:
        out['port_cuda_graph_tf32'] = {'error': repr(ex)[:300]}
        log(f'torch-cuda graph capture failed: {ex!r}')
    best = min((v['ms_per_step'] for v in out.values() if isinstance(v, dict) and 'ms_per_step' in v), default=None)
    out['best_ms_per_step'] = best
    return out
