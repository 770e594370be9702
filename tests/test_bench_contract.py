"""CPU: bench.py's reference arm prints ONE JSON line with the keys of every bench line (the B200 arm needs a GPU and refuses
without one).  GPU: the B200 arm's --dump-outputs."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1', '--ref_envs', '8'],
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'paac_env_steps_per_sec' and d['unit'] == 'env-steps/s'
    assert d['higher_is_better'] is True and d['scaling'] == 'weak' and d['vs_baseline'] is None and d['gpu_launches'] == 0
    assert d['value'] > 0 and d['ms_per_step'] > 0 and d['steps'] >= 1 and d['warmup'] >= 3
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['value'] == d['value'] and d['cpu_baseline']['cores'] >= 1
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    # the arm says what it really ran: the bounded sample, not the 4096-env workload
    assert d['config']['envs_timed'] == 8 and d['config']['env_steps_per_step'] == 8 * 5 and 'workload' in d['config']


def test_reference_arm_other_ranks_do_nothing():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1'], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_b200_arm_refuses_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '1'], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                       text=True, timeout=300)
    assert r.returncode != 0 and 'no CPU fallback' in (r.stderr + r.stdout)


@pytest.mark.parametrize('argv,message', [(['--steps', '0'], '--steps must be at least 1'),
                                          (['--dump-outputs', 'out'], '--dump-outputs writes the outputs of the B200 arm')])
def test_reference_arm_refuses_bad_arguments(argv, message):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference'] + argv,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=120)
    assert r.returncode == 2 and message in r.stderr and r.stdout == ''


@pytest.mark.gpu
def test_b200_arm_dumps_the_last_timed_step(tmp_path):
    """--dump-outputs: float32 arrays of the last timed step, under 64 MB; the same arguments give the same inputs."""
    got = []
    for run in ('a', 'b'):
        out = str(tmp_path / run)
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--envs', '64', '--steps', '2', '--warmup', '1',
                            '--no_cpu_baseline', '--no_e2e', '--no_variants', '--dump-outputs', out],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        d = json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])
        assert d['steps'] == 2 and d['dumped_outputs']['dir'] == out
        arrays = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
        assert len(arrays) == d['dumped_outputs']['arrays'] and all(a.dtype == np.float32 for a in arrays.values())
        assert sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out)) <= 64 << 20
        assert arrays['actions'].shape == (5, 64) and arrays['pi'].shape == (5, 64, 6)
        assert arrays['observed_states'].shape == (5, 16, 84, 84, 4) and arrays['params'].shape == arrays['grads'].shape
        assert np.isfinite(arrays['loss']).all() and np.all((arrays['actions'] >= 0) & (arrays['actions'] < 6))
        assert np.allclose(arrays['pi'].sum(-1), 1.0, atol=1e-5)
        got.append(arrays)
    # the preprocessed observations depend on the seeded frames alone: bit-identical from run to run
    assert np.array_equal(got[0]['env_index'], got[1]['env_index'])
    assert np.array_equal(got[0]['observed_states'], got[1]['observed_states'])
