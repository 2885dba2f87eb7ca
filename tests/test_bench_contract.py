"""bench.py contract checks that run without a GPU: the reference arm (CPU oracle port) prints one JSON line with the
keys the driver reads."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.timeout(600)
def test_reference_arm_json_line():
    env = dict(os.environ, OMP_NUM_THREADS='1')     # torchrun exports this; the arm must still use every core
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '1', '--steps', '1',
                        '--warmup', '0', '--skip-cloud-opt'], capture_output=True, text=True, env=env, cwd=ROOT, timeout=550)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line['impl'] == 'reference' and line['higher_is_better'] is True and line['n_gpus'] == 1
    for key in ('metric', 'value', 'unit', 'steps', 'warmup', 'ms_per_step', 'scaling', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in line, key
    assert line['unit'] == 'image-pairs/s' and line['value'] > 0
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    assert line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    if (os.cpu_count() or 1) > 1:
        assert line['cpu_baseline']['cores'] > 1, 'reference arm must not stay on the single thread torchrun grants'


def test_host_threads_respects_cgroup_quota_and_cap():
    sys.path.insert(0, ROOT)
    import bench
    n = bench.host_threads()
    assert 1 <= n <= 64 and n <= len(os.sched_getaffinity(0))
    assert bench.host_threads(cap=2) <= 2


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1',
                        '--warmup', '0'], capture_output=True, text=True, env=env, cwd=ROOT, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_build_roofline_on_a_recorded_breakdown():
    """The `roofline` object is assembled by a pure function: feed it the per-kernel breakdown of a recorded run."""
    sys.path.insert(0, ROOT)
    import bench
    rec = json.loads(open(os.path.join(ROOT, 'profiles', 'r01_bench_v13.json')).read().strip().splitlines()[-1])
    prof = {k: dict(count=v['launches'], ms=v['ms'], flops=(v['tflops'] or 0.0) * v['ms'] * 1e9, bytes=(v['gbs'] or 0.0) * v['ms'] * 1e6)
            for k, v in rec['kernels'].items()}
    pk = dict(hbm=6556.2, tf_burst=1683.2, tf_sustained=1439.4, source='test')
    for world in (1, 8):
        r = bench.build_roofline(prof, pk, rec['value'] * world, world)
        json.dumps(r)                                     # serialisable
        assert r['bound'] == 'tensor' and r['unit'] == 'TFLOP/s' and r['kernel'] == 'gemm_tcgen05_2cta_bn256'
        assert abs(r['frac'] - r['achieved'] / r['peak']) < 1e-12 and 0.5 < r['frac'] < 1.0
        assert r['peak'] == pk['tf_sustained'] and 0 < r['frac_of_burst_peak'] < r['frac']
        assert r['traffic'] and r['traffic'] < 1.2 * bench.ncu_traffic()[r['kernel']]['algorithmic_bytes']
        ws = r['whole_step']
        assert abs(ws['achieved'] - rec['value'] * world * bench.GFLOP_PER_PAIR / 1e3) < 1e-6
        assert abs(ws['frac'] - ws['achieved'] / (pk['tf_sustained'] * world)) < 1e-12
    # a class the table has no capture for: traffic stays null
    odd = bench.build_roofline({'some_kernel': dict(count=1, ms=1.0, flops=1e12, bytes=0.0)}, pk, 1.0, 1)
    assert odd['traffic'] is None and odd['traffic_note'] is None and odd['achieved'] == 1000.0


def test_dump_outputs_whole_or_fixed_sample_within_the_limit(tmp_path, monkeypatch):
    """--dump-outputs: the arrays as returned when they fit; otherwise the same seeded pixel positions in every array and every
    run, float32, within DUMP_MAX_BYTES."""
    sys.path.insert(0, ROOT)
    import numpy as np
    import torch
    import bench
    assert bench.DUMP_SAMPLE_PX * 32 + 4 * 4096 <= bench.DUMP_MAX_BYTES
    g = torch.Generator().manual_seed(0)
    B, H, W = 2, 8, 12
    r1 = dict(pts3d=torch.randn((B, H, W, 3), generator=g), conf=torch.rand((B, H, W), generator=g))
    r2 = dict(pts3d=torch.randn((B, H, W, 3), generator=g), conf=torch.rand((B, H, W), generator=g))
    names = dict(pred1_pts3d=r1['pts3d'], pred1_conf=r1['conf'], pred2_pts3d_in_other_view=r2['pts3d'], pred2_conf=r2['conf'])
    info = bench.dump_outputs(str(tmp_path / 'full'), r1, r2)
    assert info['sample'] is None and sorted(os.listdir(tmp_path / 'full')) == sorted(n + '.npy' for n in names)
    for n, t in names.items():
        a = np.load(tmp_path / 'full' / (n + '.npy'))
        assert a.dtype == np.float32 and np.array_equal(a, t.numpy())
    monkeypatch.setattr(bench, 'DUMP_MAX_BYTES', 4096 + 100 * 32)
    monkeypatch.setattr(bench, 'DUMP_SAMPLE_PX', 50)
    for run in ('a', 'b'):
        info = bench.dump_outputs(str(tmp_path / run), r1, r2)
        assert info['sample'] and sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= bench.DUMP_MAX_BYTES
    idx = np.sort(np.random.default_rng(bench.DUMP_SEED).choice(B * H * W, 50, replace=False))
    for n, t in names.items():
        a, b = np.load(tmp_path / 'a' / (n + '.npy')), np.load(tmp_path / 'b' / (n + '.npy'))
        assert a.dtype == np.float32 and np.array_equal(a, b)
        assert np.array_equal(a, t.reshape(B * H * W, *t.shape[3:]).numpy()[idx]), n


def test_steps_must_be_positive():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '0', '--warmup', '0'],
                       capture_output=True, text=True, cwd=ROOT, timeout=120)
    assert r.returncode == 2 and '--steps must be at least 1' in r.stderr
