"""bench.py on CPU: the reference arm prints one JSON line with the contract's keys (the GPU arm needs a B200)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _last_json(text):
    lines = [ln for ln in text.splitlines() if ln.startswith('{')]
    assert lines, text
    return json.loads(lines[-1])


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
                          '--cpu-frames', '1'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = _last_json(out.stdout)
    assert d['impl'] == 'reference' and d['unit'] == 'frames/s' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['steps'] == 1 and d['warmup'] == 0
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config'] and d['gpu_launches'] == 0


def test_reference_arm_is_silent_on_other_ranks():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2'],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ''


def test_workload_names_and_defaults():
    sys.path.insert(0, ROOT)
    import bench
    old = sys.argv
    try:
        sys.argv = ['bench.py']
        a = bench.parse()
    finally:
        sys.argv = old
    assert (a.gpus, a.impl, a.workload) == (1, 'ours', 'pald576') and a.steps >= 1 and a.warmup >= 3
    assert bench.BYTES_PER_FRAME == 3317760 and bench.DECODE_BYTES_PER_FRAME == 1658880


def test_dump_outputs_is_a_fixed_sample_within_64_mb(tmp_path):
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    n, h, w = 64, 576, 720
    g = torch.Generator().manual_seed(1)
    comp = torch.randint(0, 256, (n, h, w), dtype=torch.uint8, generator=g)
    out = torch.randint(0, 256, (n, h, w, 3), dtype=torch.uint8, generator=g)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), 100, composite=comp, rgb=out)
    bench.dump_outputs(str(tmp_path / 'c'), 100, bench.DUMP_BYTES // 16, 'one_preset.', composite=comp, rgb=out)
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == ['composite.npy', 'frame_index.npy', 'rgb.npy', 'row_index.npy']
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in names) <= 64 * 10 ** 6
    assert sum(os.path.getsize(tmp_path / 'c' / f) for f in os.listdir(tmp_path / 'c')) <= 64 * 10 ** 6 // 16
    assert sorted(os.listdir(tmp_path / 'c')) == ['one_preset.' + f for f in names]
    frames, rows = (np.load(tmp_path / 'a' / f) for f in ('frame_index.npy', 'row_index.npy'))
    assert frames.dtype == rows.dtype == np.float64 and len(frames) == (64 * 10 ** 6 - 4096) // (16 + 4 * 4 * w)
    assert len(np.unique(frames)) == n and ((frames - 100) * h + rows == np.unique((frames - 100) * h + rows)).all()
    f, r = frames.astype(np.int64) - 100, rows.astype(np.int64)
    for name, x in (('composite', comp), ('rgb', out)):
        got = np.load(tmp_path / 'a' / (name + '.npy'))
        assert got.dtype == np.float32 and np.array_equal(got, x.numpy()[f, r])
        assert np.array_equal(got, np.load(tmp_path / 'b' / (name + '.npy')))


def test_committed_bench_lines_carry_the_contract():
    """The lines bench.py printed on the B200 boxes (profiles/r2_bench*.json) have every key of the measurement contract: the base
    keys, `clocks`, `parity` within 1 LSB, `e2e` with its byte counts and the two beside-forms, `gpu_launches` > 0,
    `roofline` (HBM, live achieved / measured peak), `roofline_fma` and `cpu_baseline`."""
    for name, n in (('r2_bench.json', 1), ('r2_bench_n2.json', 2), ('r2_bench_n8.json', 8)):
        with open(os.path.join(ROOT, 'profiles', name)) as f:
            d = _last_json(f.read())
        for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                  'vs_baseline', 'dtype', 'data', 'config', 'clocks', 'e2e', 'gpu_launches', 'roofline', 'cpu_baseline'):
            assert k in d, (name, k)
        assert d['n_gpus'] == n and d['unit'] == 'frames/s' and d['scaling'] == 'weak' and d['vs_baseline'] is None
        assert d['warmup'] >= 3 and d['config']['timed_region_s'] >= 1.5 and 'workload' in d['config']
        assert not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
        assert max(d['parity'][k] for k in ('max_lsb_comp', 'max_lsb_rgb', 'e2e_max_lsb_comp', 'e2e_max_lsb_rgb')) <= 1
        e = d['e2e']
        assert e['value'] > 0 and e['h2d_bytes_per_step'] > 0 and e['d2h_bytes_per_step'] > 0
        assert e['with_composite_out']['value'] > 0 and e['two_calls']['value'] > 0 and 0 < e['frac_of_copy_peak'] < 1.2
        assert d['gpu_launches'] > 0
        r = d['roofline']
        assert r['bound'] == 'hbm' and r['unit'] == 'GB/s' and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
        assert 0 < d['roofline_fma']['frac'] < 1
        c = d['cpu_baseline']
        assert c['kind'] == 'port' and c['cores'] >= 1 and c['value'] > 0 and c['sample']
        assert d['value'] / c['value'] > 100          # the GPU arm against the CPU port on the same box
