"""bench.py contract.  On the CPU: the reference arm (`--impl reference`) runs the reference training iteration on the
host cores and prints ONE JSON line with the result keys (no GPU, none of this repository's kernels).  On the GPU:
`--dump-outputs` of this repository's arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '1'],
                         capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith('{')]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    assert d['impl'] == 'reference'
    if 'unavailable' in d:
        return
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['metric'] == 'train samples/s Darcy 64x64 PIDM' and d['unit'] == 'samples/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['ms_per_step'] > 0
    assert d['steps'] == 2 and d['warmup'] == 1
    cb = d['cpu_baseline']
    assert cb['kind'] in ('reference', 'port') and cb['cores'] >= 1 and cb['sample'] and cb['value'] == d['value']
    assert d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    assert d.get('gpu_launches', 0) == 0


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step(tmp_path):
    """`--dump-outputs DIR`: float32 .npy files of the last timed step, 64 MB at most, the loss equal to the one the JSON
    line reports, and the weights sampled at the documented positions (first 2^22 of a seed-0 permutation of the
    trainable elements in named_parameters() order, ascending): rebuilt here from the seed-0 initial model, they must
    have moved by the 5 optimizer updates and by no more than Adam's per-step bound allows."""
    import torch
    from physicsinformeddiffusionmodels_b200.unet_model import Unet3D
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '2', '--warmup', '3', '--dump-outputs', str(tmp_path),
           '--no-sampling', '--no-mechanics', '--no-torch-cuda-baseline', '--no-cpu-baseline']
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith('{')][-1])
    assert d['steps'] == 2
    names = sorted(os.listdir(tmp_path))
    assert names == ['data_loss.npy', 'ema_sample.npy', 'loss.npy', 'params_sample.npy', 'residual_abs_mean.npy'], names
    assert sum(os.path.getsize(tmp_path / n) for n in names) <= 64 << 20
    arrays = {n[:-4]: np.load(tmp_path / n) for n in names}
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
    assert arrays['params_sample'].shape == arrays['ema_sample'].shape == (1 << 22,)
    assert float(arrays['loss']) == d['config']['last_loss']
    torch.manual_seed(0)                                     # the initial weights of bench.py
    trainable = [p for p in Unet3D(dim=32, channels=2).parameters() if p.requires_grad]
    flat = torch.cat([p.detach().reshape(-1) for p in trainable])
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:1 << 22].sort().values
    init = flat[idx].numpy()
    params, ema = arrays['params_sample'], arrays['ema_sample']
    bound = 5 * 4 * 1e-4                                     # 3 warm-up + 2 timed Adam updates at lr 1e-4
    assert (params != init).mean() > 0.5                     # not the initial (stale) weights
    assert np.abs(params - init).max() <= bound              # the same positions as the initial weights
    assert np.abs(ema - init).max() <= bound and (ema != params).any()
