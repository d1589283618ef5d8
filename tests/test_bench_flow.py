"""bench.py's control flow on CPU (tests/bench_dryrun.py replaces the CUDA-facing pieces): ONE JSON line with the extra
C5 / C3 legs, single process and world-size-2 gloo; a leg or a teardown that hangs must not lose the line."""
import json
import os
import socket
import subprocess
import sys
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRY = os.path.join(ROOT, 'tests', 'bench_dryrun.py')
FLAGS = ['--no-cpu-baseline', '--no-gpu-reference', '--no-fp32-parity', '--steps', '2']


def _port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _run(world, extra=(), hang='', limit=240):
    env = dict(os.environ, DRYRUN_HANG=hang)
    if world == 1:
        cmd = [sys.executable, DRY] + FLAGS + list(extra)
    else:
        cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', f'--nproc-per-node={world}', '--master-addr', '127.0.0.1',
               '--master-port', str(_port()), DRY, '--gpus', str(world)] + FLAGS + list(extra)
    t0 = time.time()
    p = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=limit, cwd=ROOT)
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith('{')]
    return p.returncode, lines, time.time() - t0, p.stderr


def test_one_line_with_both_extra_legs_single_process():
    rc, lines, _, err = _run(1)
    assert rc == 0 and len(lines) == 1, err[-2000:]
    line = json.loads(lines[0])
    for key in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype',
                'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline'):
        assert key in line
    c5, c3 = line['c5_sharded_search'], line['c3_strong_split']
    assert 'error' not in c5 and 'error' not in c3, (c5, c3)
    assert c5['indices_bit_exact_vs_pairwise'] is True and c5['merged_equals_gathered_lists'] is None and c5['gpu_launches'] == 3 * c5['steps']
    assert c3['scaling'] == 'strong' and c3['output_finite'] is True
    assert line['four_terms_author_weights']['output_finite'] is True and 'w_lpips=10' in line['four_terms_author_weights']['config']['workload']
    rc, lines, _, err = _run(1, ['--no-extras'])
    assert rc == 0 and len(lines) == 1 and 'c5_sharded_search' not in json.loads(lines[0]), err[-2000:]


def test_dump_outputs_of_the_last_timed_step(tmp_path):
    import numpy as np
    out = tmp_path / 'out'
    rc, lines, _, err = _run(1, ['--no-extras', '--warmup', '3', '--steps', '4', '--dump-outputs', str(out)])
    assert rc == 0 and len(lines) == 1, err[-2000:]
    assert json.loads(lines[0])['steps'] == 4
    assert sorted(os.listdir(out)) == ['img.npy', 'w_aug.npy']
    img, w = np.load(out / 'img.npy'), np.load(out / 'w_aug.npy')
    assert img.dtype == w.dtype == np.float32 and img.shape == (2, 3, 4, 4) and w.shape == (2, 1, 8)
    assert (img == 3 + 4).all()                  # the stand-in's pixels count its calls: 3 warm-up + 4 timed steps


def test_dump_outputs_sample_fixed_rows_beyond_the_limit(tmp_path):
    import numpy as np
    import torch

    import bench
    a, b = torch.arange(64.0).reshape(16, 4), -torch.arange(32.0).reshape(16, 2)
    for d in ('x', 'y'):
        bench.dump_outputs(str(tmp_path / d), {'a': a, 'b': b.double()}, limit=200)
    ra, rb = np.load(tmp_path / 'x' / 'a.npy'), np.load(tmp_path / 'x' / 'b.npy')
    assert ra.dtype == rb.dtype == np.float32 and ra.nbytes + rb.nbytes <= 200 and ra.shape == (8, 4) and rb.shape == (8, 2)
    rows = ra[:, 0].astype(np.int64) // 4
    assert (np.diff(rows) > 0).all() and (rb[:, 0] == -2 * rows).all()          # the same ascending rows of both arrays
    assert (np.load(tmp_path / 'y' / 'a.npy') == ra).all()                       # and the same rows in every run
    bench.dump_outputs(str(tmp_path / 'z'), {'a': a}, limit=a.numel() * 4)
    assert (np.load(tmp_path / 'z' / 'a.npy') == a.numpy()).all()


def test_two_ranks_gloo_merge_check_and_teardown():
    rc, lines, _, err = _run(2)
    assert rc == 0 and len(lines) == 1, err[-2000:]
    line = json.loads(lines[0])
    c5, c3 = line['c5_sharded_search'], line['c3_strong_split']
    assert line['n_gpus'] == 2 and c5['n_gpus'] == 2 and c5['merged_equals_gathered_lists'] is True and c5['indices_bit_exact_vs_pairwise'] is True
    assert c5['gpu_launches'] == 4 * c5['steps'] and 'NCCL all-gather' in c5['config']['workload']
    assert c3['n_gpus'] == 2 and 'split over 2 rank(s)' in c3['config']['parallelism'] and 'four_terms_author_weights' not in line


def test_hung_extra_leg_keeps_the_headline_line():
    rc, lines, dt, err = _run(2, ['--extras-timeout', '4'], hang='c5', limit=120)
    assert rc == 0 and len(lines) == 1, err[-2000:]
    line = json.loads(lines[0])
    assert 'watchdog' in line and 'c5_sharded_search' not in line and line['value'] > 0 and dt < 90


def test_hung_teardown_ends_with_exit_code_zero():
    rc, lines, dt, err = _run(2, ['--teardown-timeout', '3'], hang='teardown', limit=120)
    assert rc == 0 and len(lines) == 1 and dt < 90, err[-2000:]
    assert 'watchdog' not in json.loads(lines[0])


def test_c5_config_line_two_ranks():
    rc, lines, _, err = _run(2, ['--config', 'c5', '--steps', '1'])
    assert rc == 0 and len(lines) == 1, err[-2000:]
    line = json.loads(lines[0])
    assert line['metric'] == 'nearest-code queries/sec' and line['merged_equals_gathered_lists'] is True
