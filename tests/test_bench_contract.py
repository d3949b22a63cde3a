"""bench.py contract checks that need no GPU: the reference arm prints exactly ONE JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'lines/s' and d['higher_is_better'] is True
    for k in ('metric', 'value', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'scaling', 'vs_baseline', 'dtype', 'data', 'config',
              'cpu_baseline', 'e2e'):
        assert k in d, k
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0
    assert d['value'] > 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK='1', LOCAL_RANK='1', WORLD_SIZE='2', MASTER_ADDR='127.0.0.1', MASTER_PORT='29999')
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    assert p.stdout.strip() == ''


def test_per_stage_roofline_arithmetic():
    sys.path.insert(0, ROOT)
    import bench
    work = bench.stage_work()
    pk = {'tf_sustained': 1000.0, 'hbm_gbs': 5000.0}
    r = bench.per_stage_roofline({'L_5.xproj': 0.1, 'decode': 0.05, 'unknown': 1.0, 'O_6': 0.0}, work, pk, 64)
    assert set(r) == {'L_5.xproj', 'decode'}
    fl = 2 * 200 * 768 * 2048 * 64
    assert abs(r['L_5.xproj']['tflops'] - fl / 1e-4 / 1e12) < 0.01 and abs(r['L_5.xproj']['tensor_frac'] - r['L_5.xproj']['tflops'] / 1000.0) < 1e-3
    assert r['decode']['tflops'] == 0 and r['decode']['gbs'] > 0


def test_dump_outputs_writes_float_arrays_with_unwritten_slots_zeroed(tmp_path):
    sys.path.insert(0, ROOT)
    import numpy as np
    import bench
    from kraken_b200.dist import ResultBlocks
    rb = ResultBlocks(2, 3, 5, pin=False)
    rb.t.fill_(7)                                            # stands for whatever an earlier run left in the buffer
    v = rb.views(1)
    v['counts'][:] = [0, 2, 5]
    v['labels'][1, :2] = [4, 9]; v['starts'][1, :2] = [0, 3]; v['ends'][1, :2] = [1, 4]; v['confs'][1, :2] = [0.5, 0.25]
    bench.dump_outputs(str(tmp_path / 'out'), {k: a.copy() for k, a in v.items()})
    got = {f[:-4]: np.load(tmp_path / 'out' / f) for f in os.listdir(tmp_path / 'out')}
    assert sorted(got) == ['confs', 'counts', 'ends', 'labels', 'starts']
    assert got['confs'].dtype == np.float32 and all(got[k].dtype == np.float64 for k in ('counts', 'labels', 'starts', 'ends'))
    assert got['counts'].tolist() == [0, 2, 5]
    assert got['labels'][0].tolist() == [0] * 5 and got['labels'][1].tolist() == [4, 9, 0, 0, 0] and got['labels'][2].tolist() == [7] * 5
    assert got['confs'][1].tolist() == [0.5, 0.25, 0, 0, 0]


def test_dump_outputs_only_for_the_gpu_cfg2_arm():
    p = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--dump-outputs', 'unused'],
                       capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert p.returncode == 2 and '--dump-outputs' in p.stderr and not os.path.exists(os.path.join(ROOT, 'unused'))
