"""The tap-GEMM kernel has two mainloops: single-CTA MMAs (M = 128) and CTA pairs (cta_group::2, M = 256 over
two SMs, four-tile work items at BN = 128).  The planner mixes them per launch (csrc/plan.cuh::make_b_map);
LA_CTA2 forces one everywhere.  The switch is read once per process, so each forced mode runs the parity tests
of tests/test_gpu_parity.py / tests/test_gpu_disc.py and the clamp tests of tests/test_gpu_act_clamp.py in a child process.
"""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
@pytest.mark.parametrize('mode', ['0', '2'])
def test_parity_suite_in_forced_pair_mode(mode):
    env = dict(os.environ, LA_CTA2=mode)
    sel = ('synthesis_matches_oracle or simt_twin or augment_loop_matches_oracle or reference_golden or ragged_batches '
           'or single_channel_wide or logits_loss_and_gradient or realism_term or (test_clamp_ and not without_staged)')
    r = subprocess.run([sys.executable, '-m', 'pytest', '-x', '-q', '-m', 'gpu', '-k', sel,
                        os.path.join(ROOT, 'tests', 'test_gpu_parity.py'), os.path.join(ROOT, 'tests', 'test_gpu_disc.py'),
                        os.path.join(ROOT, 'tests', 'test_gpu_act_clamp.py')],
                       cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    tail = (r.stdout or '')[-2000:] + (r.stderr or '')[-1000:]
    assert r.returncode == 0, tail
    assert ' passed' in r.stdout and 'failed' not in r.stdout, tail
