"""CPU: the committed bench lines carry every key of the bench contract, and bench.py parses without a GPU."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

REQUIRED = ['metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
            'vs_baseline', 'dtype', 'data', 'config', 'e2e', 'gpu_launches', 'clocks', 'roofline']


def _load(name):
    return json.load(open(os.path.join(ROOT, 'profiles', name)))


def test_own_arm_line_has_the_contract_keys():
    d = _load('bench_r02_v14.json')
    for k in REQUIRED + ['cpu_baseline']:
        assert k in d, k
    base = json.load(open(os.path.join(ROOT, 'BASELINE.json')))
    assert d['metric'] in base['metric'] and d['unit'] == 'tuples/s' and d['higher_is_better'] is True
    assert d['scaling'] == 'weak' and d['vs_baseline'] is None and d['data'] == 'synthetic'
    assert 'workload' in d['config'] and 'model' not in d['config']
    assert d['warmup'] >= 3 and d['gpu_launches'] > 0
    e = d['e2e']
    assert e['h2d_bytes_per_step'] > 0 and e['d2h_bytes_per_step'] > 0 and e['value'] != d['value']
    r = d['roofline']
    for k in ('bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'):
        assert k in r, k
    assert r['bound'] in ('hbm', 'tensor') and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
    assert r['traffic'] and r['frac'] > 0.3                      # round 2: attention at > 0.3 of the measured bf16 peak
    assert d['value'] > 350 and d['run']['attention_split'] == 'fp16 hi/lo'
    p = d['pose_auc_parity']
    assert p['max_abs_diff_pt'] <= 0.5 and p['n_errors'] == 320
    c = d['cpu_baseline']
    assert c['kind'] in ('reference', 'port') and c['cores'] >= 1 and c['sample']
    assert not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}


def test_reference_arm_line():
    d = _load('bench_r02_v14_reference_arm.json')
    assert d['steps'] == 20 and d['warmup'] == 5            # the arm honours --steps / --warmup
    assert d['impl'] == 'reference' and d['unit'] == 'tuples/s' and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_two_gpu_line_scales():
    one, two = _load('bench_r02_g16_quick.json'), _load('bench_r02_v8_2gpu.json')      # same commit
    assert two['n_gpus'] == 2 and two['run']['parallelism'] == 'dp2'
    assert two['value'] > 1.9 * one['value']             # whole-job aggregate, weak scaling


def test_eight_gpu_line_scales():
    one, eight = _load('bench_r02_v14.json'), _load('bench_r02_v15_8gpu.json')
    assert eight['n_gpus'] == 8 and eight['run']['parallelism'] == 'dp8' and eight['scaling'] == 'weak'
    assert eight['value'] > 0.95 * 8 * one['value']


def test_training_line_cfg5():
    """bench.py --config cfg5: training iterations per second (stage 1 of BASELINE configs[4])."""
    d = _load('bench_r02_cfg5_h.json')
    for k in REQUIRED:
        assert k in d, k
    assert d['unit'] == 'steps/s' and d['scaling'] == 'weak' and d['config']['workload'].startswith('train_stage1')
    assert d['warmup'] >= 3 and d['gpu_launches'] > 1000 and d['value'] > 7.0
    assert abs(d['value'] * d['ms_per_step'] - 1000.0) < 1.0 and d['tuples_per_s'] == d['value'] * d['units_per_step']
    assert d['loss_first_last'][1] < 0.2 * d['loss_first_last'][0]              # the optimiser steps really train
    assert d['e2e']['h2d_bytes_per_step'] > 1e7 and 'not built' in d['run']['stage']
    first = _load('bench_r02_cfg5_a.json')
    assert d['value'] > 3.0 * first['value']                                    # 2.1 -> 7.4 steps/s over the round
    two = _load('bench_r02_cfg5_2gpu.json')                                     # data parallel, gradient all-reduce over NCCL
    assert two['n_gpus'] == 2 and two['tuples_per_s'] > 1.9 * d['tuples_per_s'] and 'all-reduce' in two['run']['collective']


def test_pair_config_lines():
    for name, unit_min in (('bench_r02_v14_cfg2.json', 2000), ('bench_r02_v14_cfg4.json', 400)):
        d = _load(name)
        for k in REQUIRED + ['cpu_baseline']:
            assert k in d, (name, k)
        assert d['unit'] == 'pairs/s' and d['value'] > unit_min
        assert d['pose_auc_parity']['max_abs_diff_pt'] <= 0.1


def test_bench_cli_parses_without_gpu():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--help'], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and '--impl' in r.stdout and '--gpus' in r.stdout and '--dump-outputs' in r.stdout


def test_dump_outputs_exact_small_sampled_large(tmp_path):
    """bench.py --dump-outputs: small outputs stored exactly as float32 / float64, a large one as a seeded sample that
    keeps the total within the budget, the same positions on every run."""
    import numpy as np
    import torch
    import bench
    big = np.arange(1 << 16, dtype=np.float32).reshape(64, 1024)
    arrays = {'scores': torch.from_numpy(big), 'matches': torch.arange(-1, 99), 'success': torch.tensor([True, False]),
              'cost': np.linspace(0.0, 1.0, 7), 'view_ids': [0, 1]}
    budget = 1 << 16
    stored = bench.dump_outputs(str(tmp_path / 'a'), arrays, budget=budget)
    bench.dump_outputs(str(tmp_path / 'b'), arrays, budget=budget)
    assert sorted(stored) == ['cost', 'matches', 'scores', 'success']
    assert sorted(os.listdir(tmp_path / 'a')) == sorted(n + '.npy' for n in stored)
    a = {n: np.load(tmp_path / 'a' / (n + '.npy')) for n in stored}
    assert sum(v.nbytes for v in a.values()) <= budget
    assert a['matches'].dtype == np.float64 and np.array_equal(a['matches'], np.arange(-1, 99))
    assert a['success'].dtype == np.float32 and a['success'].tolist() == [1.0, 0.0]
    assert a['cost'].dtype == np.float64 and np.array_equal(a['cost'], arrays['cost'])
    s = a['scores']                      # element k of `big` is k: the sample holds its own (increasing) positions
    assert s.dtype == np.float32 and 0 < s.size < big.size and np.all(np.diff(s) > 0)
    for n in stored:
        assert np.array_equal(a[n], np.load(tmp_path / 'b' / (n + '.npy')))
