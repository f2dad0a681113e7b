"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the agreed keys, and
the cuda arm refuses to run (no CPU fallback) when there is no device."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize('workload', ['fifo60k', 'dlas60k', 'sjf10k', 'env512x10k'])
def test_reference_arm_prints_one_json_line(workload):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--workload', workload,
                        '--no-python-reference'], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'simulated_events_per_sec' and d['unit'] == 'events/s'
    assert d['higher_is_better'] is True and d['value'] > 0 and d['scaling'] == 'weak' and d['vs_baseline'] is None
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': 'events/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config'] and d['config']['name'] == workload


def test_reference_arm_reports_the_staged_python_reference():
    """When __graft_entry__.build() staged the unmodified reference under oracle/_ref/reference, the CPU arm times it for real
    on a 2 000-job trace and reports it beside the port."""
    if not os.path.exists(os.path.join(ROOT, 'oracle', '_ref', 'reference', 'run_sim.py')):
        pytest.skip('build() staged no reference under oracle/_ref/reference')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0', '--workload', 'sjf10k'],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.strip()][0])
    rp = d['cpu_baseline']['reference_python']
    assert rp['cores'] == 1 and rp['events_per_s'] > 0 and 'dead-code loop' in rp['sample']


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_cuda_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1'], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and 'no CPU fallback' in (r.stderr + r.stdout)
