"""The reference's OWN driver scripts, executed against this repository's drop-in `src/` package.

`oracle/_ref/{main.py,main_toy.py}` are the unmodified files of the reference (copied by `__graft_entry__.build()`
when the original project is at hand, not part of this repository; the tests skip without them).  The scripts hard-code their run length (300,000 training
iterations, a 10^4-point data set, W&B tracking), so the test rewrites exactly those LITERALS -- listed in `EDITS` below,
each asserted to occur -- and nothing else: imports, model construction, loss call, optimizer / clip / EMA sequence,
sampling call, checkpoint call all execute as written by the reference's authors.  matplotlib (not installed here) is
replaced by the accept-everything shim in oracle/ref_shims."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, 'oracle', '_ref')
SHIMS = os.path.join(ROOT, 'oracle', 'ref_shims')


def _run(script_text, cwd, timeout=900):
    path = os.path.join(cwd, 'driver.py')
    with open(path, 'w') as f:
        f.write(script_text)
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([ROOT, SHIMS]), WANDB_MODE='disabled')
    r = subprocess.run([sys.executable, path], cwd=cwd, env=env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r


def _edit(text, edits):
    for old, new in edits:
        assert text.count(old) >= 1, f'literal not found in the reference script: {old!r}'
        text = text.replace(old, new)
    return text


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, 'main.py')), reason='reference scripts not fetched (oracle/_ref)')
def test_reference_main_py_runs_on_the_drop_in_package(tmp_path):
    """main.py (Darcy, model.yaml as shipped except diff_steps): 2 training iterations incl. validation loss, EMA,
    sampling with residual evaluation, CSV dumps and the checkpoint."""
    EDITS = [('train_iterations = 300000', 'train_iterations = 2'),
             ('train_batch_size = 64', 'train_batch_size = 2'),
             ('no_samples = 8', 'no_samples = 2')]
    text = _edit(open(os.path.join(REF, 'main.py')).read(), EDITS)
    yaml_text = _edit(open(os.path.join(REF, 'model.yaml')).read(), [('diff_steps: 100', 'diff_steps: 4')])
    with open(tmp_path / 'model.yaml', 'w') as f:
        f.write(yaml_text)
    rng = np.random.default_rng(0)
    for split in ('train', 'valid'):
        os.makedirs(tmp_path / 'data' / 'darcy' / split)
        for name in ('p_data.csv', 'K_data.csv'):
            np.savetxt(tmp_path / 'data' / 'darcy' / split / name, rng.standard_normal((4, 64 * 64)).astype(np.float32),
                       delimiter=',')
    r = _run(text, str(tmp_path))
    run_dir = tmp_path / 'trained_models' / 'run_1'
    assert (run_dir / 'model' / 'checkpoint_2.pt').exists(), r.stdout[-2000:]
    stats = run_dir / 'training' / 'step_2' / 'sample_statistics.csv'
    assert stats.exists()
    vals = np.genfromtxt(stats, delimiter=',', skip_header=1)[:, 1]
    assert np.isfinite(vals).all()
    assert 'test loss at iteration 0' in r.stdout


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, 'main_toy.py')), reason='reference scripts not fetched (oracle/_ref)')
def test_reference_main_toy_py_runs_on_the_drop_in_package(tmp_path):
    """main_toy.py (configs[0]): 2 epochs over a 512-point data set, sampling + CSV dump at epoch 0, checkpoint."""
    EDITS = [("'train_num_steps': 400", "'train_num_steps': 1"),
             ("'no_samples': 1000", "'no_samples': 64"),
             ("'wandb_track': True", "'wandb_track': False"),
             ('sample_hypersphere(10**4', 'sample_hypersphere(512')]
    text = _edit(open(os.path.join(REF, 'main_toy.py')).read(), EDITS)
    r = _run(text, str(tmp_path))
    out = tmp_path / 'trained_models' / 'toy' / 'run_1'
    assert (out / 'model' / 'checkpoint_1.pt').exists(), r.stdout[-2000:]
    pts = np.loadtxt(out / 'csv' / 'step_0_sample.csv', delimiter=',')
    assert pts.shape == (64, 2) and np.isfinite(pts).all()
