"""bench.py contract pieces: the reference arm (the oracle timed on the host cores) prints one JSON line with the keys
a reader of the result expects; --dump-outputs writes the top-k of the last timed step (CPU: sampling and files; GPU:
the values against the oracle)."""
import json
import os
import subprocess
import sys

import pytest

import oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--users', '300',
                          '--items', '500', '--d', '16', '--steps', '1', '--warmup', '1', '--cpu-budget', '0.5'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line['impl'] == 'reference' and line['metric'] == 'predict_rank_pairs_per_s' and line['unit'] == 'pairs/s'
    assert line['higher_is_better'] is True and line['value'] > 0 and line['steps'] == 1 and line['n_gpus'] == 1
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    assert line['cpu_baseline']['value'] == line['value'] and line['cpu_baseline']['sample']
    assert line['e2e'] == {'value': line['value'], 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in line['config'] and line['gpu_launches'] == 0


def test_reference_arm_under_torchrun_env_only_rank0_prints():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2',
                          '--users', '64', '--items', '64', '--d', '8', '--steps', '1', '--warmup', '0'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith('{')]


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location('bench', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_writes_a_seeded_sample_within_budget(tmp_path, monkeypatch):
    import numpy as np
    import torch
    bench = _bench_module()
    monkeypatch.setattr(bench, 'DUMP_BYTES', 100 * (8 + 3 * 12))        # room for 100 rows of a top-3
    from tensorrec_b200.kernels import PackedTopK
    n_users, k = 1000, 3
    top = PackedTopK(n_users, k, 'cpu')
    top.items.copy_(torch.arange(n_users * k, dtype=torch.int32).reshape(n_users, k))
    top.scores.copy_(-torch.arange(n_users * k, dtype=torch.float32).reshape(n_users, k) / 7)
    dumps = []
    for run in range(2):
        out = tmp_path / str(run)
        bench.dump_topk(str(out), top, first_user=5000)
        dumps.append({p.stem: np.load(str(p)) for p in out.iterdir()})
    got = dumps[0]
    assert sorted(got) == ['topk_items', 'topk_scores', 'user_ids']
    assert got['user_ids'].dtype == np.float64 and got['topk_items'].dtype == np.float64
    assert got['topk_scores'].dtype == np.float32
    rows = got['user_ids'].astype(np.int64) - 5000
    assert len(rows) == 100 and np.all(np.diff(rows) > 0) and rows[-1] < n_users
    assert np.array_equal(got['topk_items'], top.items.numpy()[rows].astype(np.float64))
    assert np.array_equal(got['topk_scores'], top.scores.numpy()[rows])
    for name in got:
        assert np.array_equal(got[name], dumps[1][name])                  # the same rows on every run


@pytest.mark.gpu
def test_dump_outputs_holds_the_oracle_top_k(tmp_path):
    """Integer-valued weights: the timed path's top-k equals the oracle's bit for bit, ties included."""
    import numpy as np
    bench = _bench_module()
    argv = ['--users', '3000', '--items', '5000', '--d', '64', '--scores', 'ties', '--steps', '2', '--warmup', '1',
            '--no-extra', '--no-clocks', '--cpu-budget', '0.2', '--parity-users', '64']
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + argv + ['--dump-outputs', str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.splitlines()[-1])['steps'] == 2
    got = {p.stem: np.load(str(p)) for p in tmp_path.iterdir()}
    assert np.array_equal(got['user_ids'], np.arange(3000))
    args = type('Args', (), dict(users=3000, items=5000, d=64, scores='ties'))()
    uf, itf, wu, wi, bu, bi = bench.make_problem(args)
    scores = oracle.OracleModel([wu], wi, bu, bi).predict(uf, itf)
    exp_items, exp_scores = oracle.top_k_from_scores(scores, 10)
    assert np.array_equal(got['topk_items'], exp_items) and np.array_equal(got['topk_scores'], exp_scores)


def test_dump_outputs_and_steps_are_checked():
    for extra in (['--impl', 'reference', '--dump-outputs', 'x'], ['--workload', 'dense', '--dump-outputs', 'x'],
                  ['--steps', '0']):
        out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + extra, capture_output=True, text=True,
                             timeout=300, cwd=ROOT)
        assert out.returncode == 2 and 'error' in out.stderr, extra
