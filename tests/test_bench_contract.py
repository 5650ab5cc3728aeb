"""bench.py's contract on the CPU: the five BASELINE configurations are selectable, and the reference arm
(`--impl reference`: the CPU oracle port timed on the host cores) prints ONE JSON line with the benchmark's result keys and
times exactly --steps steps; on a GPU, --dump-outputs writes the last timed step's results."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_configs_are_the_baseline_configs():
    import bench
    base = json.load(open(os.path.join(ROOT, 'BASELINE.json')))
    assert set(bench.CONFIGS) == {'cfg1', 'cfg2', 'cfg3', 'cfg4', 'cfg5'} and len(base['configs']) == 5
    bench.select_config('cfg4')
    assert bench.IMAGE[:2] == (128, 128) and bench.SAVP_HPARAMS['sequence_length'] == 16
    bench.select_config('cfg2')
    assert bench.IMAGE == (64, 64, 3) and bench.PER_GPU_BATCH == 16 and bench.SAVP_HPARAMS['sequence_length'] == 12
    assert bench.SAVP_HPARAMS['context_frames'] == 2


def test_reference_arm_prints_the_contract_line():
    env = dict(os.environ, CUDA_VISIBLE_DEVICES='')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '1'],
                       capture_output=True, text=True, timeout=600, env=env)
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert r.returncode == 0 and len(lines) == 1, r.stderr[-500:]
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'frames/s' and d['higher_is_better'] is True and d['value'] > 0
    assert d['metric'].startswith('frames/sec SAVP 64x64') and d['n_gpus'] == 1 and d['data'] == 'synthetic'
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and abs(cb['value'] - d['value']) < 1e-9 and 'training steps' in cb['sample']
    assert d['steps'] == 2 and cb['sample'].startswith('2 full training steps')
    assert d['e2e'] == dict(value=d['value'], unit='frames/s', h2d_bytes_per_step=0, d2h_bytes_per_step=0)
    assert d['config']['workload'] and d['ms_per_step'] > 0


def test_bench_rejects_a_step_count_below_one_and_dumps_of_the_reference_arm():
    for extra in (['--steps', '0'], ['--impl', 'reference', '--dump-outputs', 'out']):
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and 'error' in r.stderr, (extra, r.stderr[-500:])


def _bench_dump(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', str(steps), '--warmup', '1', '--no-cpu',
                        '--no-roofline', '--dump-outputs', str(out)], capture_output=True, text=True, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert r.returncode == 0 and len(lines) == 1, r.stderr[-2000:]
    files = sorted(out.iterdir())
    assert sum(p.stat().st_size for p in files) <= 64 << 20
    return json.loads(lines[0]), {p.name[:-4]: np.load(p) for p in files}


@pytest.mark.gpu
def test_dump_outputs_holds_the_last_timed_step_and_is_reproducible(tmp_path):
    """--dump-outputs: float32 / float64 arrays under 64 MB in all; the loss terms are the ones the JSON line reports.  The
    last timed step starts from the seeded initial state whatever --steps is, so a run of 3 steps dumps what a run of 1 step
    dumps, up to the fp32 summation order of the atomics inside that one step."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip('no CUDA device')
    d, arrays = _bench_dump(tmp_path / 'a', 3)
    assert d['steps'] == 3 and d['losses_finite']
    assert all(a.dtype in (np.float32, np.float64) for a in arrays.values())
    assert arrays['gen_images'].shape == (16, 11, 64, 64, 3) and arrays['gen_images_enc'].shape == (16, 11, 64, 64, 3)
    assert arrays['zs_mu_enc'].shape == (16, 11, 8) and arrays['zs_log_sigma_sq_enc'].shape == (16, 11, 8)
    assert all(np.isfinite(a).all() for a in arrays.values())
    for k, v in d['losses'].items():                     # the JSON line rounds to 6 decimals
        assert abs(float(arrays[k]) - v) <= 1e-6, (k, float(arrays[k]), v)
    _, again = _bench_dump(tmp_path / 'b', 1)
    assert sorted(again) == sorted(arrays)
    diffs = {k: float(np.linalg.norm(again[k].astype(np.float64) - arrays[k]) / (np.linalg.norm(arrays[k]) + 1e-12)) for k in arrays}
    print('run-to-run relative L2 of the dumped arrays:', diffs)
    assert np.abs(again['gen_images'] - arrays['gen_images']).max() <= 1e-3
    assert all(v <= 1e-2 for v in diffs.values()), diffs
