"""The drop-in CLIs end to end on a GPU: train.py (reference flags) on gzip TFRecords -> checkpoint -> resume -> sample.py;
bench.py's output dump."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(args, cwd, timeout=600):
    env = dict(os.environ, PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable] + args, cwd=cwd, env=env, capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout


def test_train_checkpoint_resume_sample(tmp_path):
    from progen_b200.data import write_tfrecords
    import numpy as np
    rng = np.random.default_rng(0)
    aa = 'ACDEFGHIKLMNPQRSTVWY'
    seqs = ['[tax=Mammalia] # ' + ''.join(rng.choice(list(aa), size=int(rng.integers(20, 100)))) for _ in range(48)]
    data = tmp_path / 'train_data'
    data.mkdir()
    write_tfrecords(str(data / f'0.{len(seqs) - 8}.train.tfrecord.gz'), seqs[:-8])
    write_tfrecords(str(data / '0.8.valid.tfrecord.gz'), seqs[-8:])
    cfgdir = tmp_path / 'configs' / 'model'
    cfgdir.mkdir(parents=True)
    (cfgdir / 'tiny.toml').write_text('num_tokens = 256\ndim = 128\ndepth = 2\ndim_head = 64\nheads = 2\nwindow_size = 64\n'
                                      'seq_len = 128\nglobal_mlp_depth = 1\n')
    common = ['--config_path', str(cfgdir), '--model_name', 'tiny', '--data_path', str(data), '--checkpoint_path',
              str(tmp_path / 'ckpts'), '--wandb_off', '--batch_size', '4', '--grad_accum_every', '2', '--checkpoint_every', '1',
              '--validate_every', '2', '--sample_every', '3', '--prime_length', '8']
    out = run([os.path.join(ROOT, 'train.py')] + common + ['--num_steps', '3', '--cuda_graph'], cwd=str(tmp_path))   # captured after 2 eager micro-steps
    assert 'loss:' in out and 'valid_loss:' in out and 'checkpoint to start at sequence index of 8' in out
    losses = [float(l.split()[-1]) for l in out.splitlines() if l.startswith('loss:')]
    assert len(losses) == 3 and all(l == l and l < 7.0 for l in losses)
    # resume: model config and position come from the checkpoint (train.py:99-100,126-128)
    out2 = run([os.path.join(ROOT, 'train.py')] + common + ['--num_steps', '1', '--mixed_precision'], cwd=str(tmp_path))
    assert 'starting from sequence 24' in out2
    out3 = run([os.path.join(ROOT, 'sample.py'), '--checkpoint_path', str(tmp_path / 'ckpts'), '--prime', '[tax=Mammalia] #',
                '--greedy'], cwd=str(tmp_path))
    assert 'sequence length: 128' in out3 and '*' * 40 in out3


def test_bench_dump_outputs_repeat(tmp_path):
    """bench.py --dump-outputs: the last timed step's loss, logits, gradient and parameters as float .npy files of at most
    64 MB, the same in two runs with the same arguments (seeded inputs; only the order of atomic reductions may differ)"""
    import numpy as np
    dumps = []
    for r in range(2):
        d = tmp_path / f'run{r}'
        out = run([os.path.join(ROOT, 'bench.py'), '--config', 'tiny', '--steps', '2', '--warmup', '1', '--no-cpu-baseline',
                   '--dump-outputs', str(d)], cwd=str(tmp_path))
        lines = [l for l in out.splitlines() if l.strip()]
        assert len(lines) == 1
        j = json.loads(lines[0])
        assert j['steps'] == 2
        files = sorted(d.iterdir())
        assert [f.name for f in files] == ['grads.npy', 'logits.npy', 'loss.npy', 'params.npy']
        assert sum(f.stat().st_size for f in files) <= 64 << 20
        arrays = {f.stem: np.load(f) for f in files}
        assert all(a.dtype in (np.float32, np.float64) and a.size > 0 and np.isfinite(a).all() for a in arrays.values())
        assert abs(float(arrays['loss'][0]) - j['final_loss']) <= 1e-6 * abs(j['final_loss'])
        dumps.append(arrays)
    a, b = dumps
    for k in a:
        assert a[k].shape == b[k].shape, k
        assert np.abs(a[k] - b[k]).max() <= 1e-2 * max(1e-6, float(np.abs(a[k]).max())), k
