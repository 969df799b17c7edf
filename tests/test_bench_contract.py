"""bench.py's reference arm on the CPU (no GPU needed): the JSON line keeps the driver's contract, other ranks stay quiet,
--dump-outputs writes what the timed path returned. On the GPU: the product arm dumps the same arrays as the oracle."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle_lib as ol

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DUMP_FILES = ('pcm.npy', 'pcm_packets.npy', 'out_bytes.npy', 'status.npy')


@pytest.fixture(scope='module')
def cache(tmp_path_factory):
    return str(tmp_path_factory.mktemp('alac_b200_cache'))


def _run(cache, env_extra, *extra_args, impl='reference'):
    env = dict(os.environ, ALAC_B200_CACHE=cache, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', impl, '--workload', 'smoke', '--steps', '1',
                           '--warmup', '1', *extra_args], capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)


def _load_dump(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in DUMP_FILES}


def test_reference_arm_line(cache):
    r = _run(cache, {})
    assert r.returncode == 0, r.stderr[-500:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, lines  # ONE JSON line on stdout, everything else on stderr
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'decoded PCM samples/s' and d['unit'] == 'samples/s'
    assert d['higher_is_better'] is True and d['vs_baseline'] is None and d['dtype'] == 'int32' and d['data'] == 'synthetic'
    assert d['steps'] == 1 and d['warmup'] == 1 and d['n_gpus'] == 1 and d['gpu_launches'] == 0
    assert d['value'] > 0 and d['ms_per_step'] > 0 and d['config']['workload'].startswith('smoke')
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == d['value'] and cb['sample']
    assert d['e2e'] == {'value': d['value'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_reference_arm_other_ranks_do_nothing(cache):
    r = _run(cache, {'RANK': '1', 'WORLD_SIZE': '2', 'LOCAL_RANK': '1'})
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_reference_arm_dump_outputs(cache, tmp_path, monkeypatch):
    """--dump-outputs: float arrays under 64 MB, the same from run to run, and the PCM of the sampled packets is what
    decoding those packets one by one gives."""
    dumps = []
    for k in range(2):
        d = str(tmp_path / f'dump{k}')
        r = _run(cache, {}, '--dump-outputs', d)
        assert r.returncode == 0, r.stderr[-500:]
        assert sorted(os.listdir(d)) == sorted(DUMP_FILES)
        assert sum(os.path.getsize(os.path.join(d, f)) for f in DUMP_FILES) <= 64 << 20
        dumps.append(_load_dump(d))
    for f in dumps[0]:
        assert dumps[0][f].dtype in (np.float32, np.float64), f
        assert np.array_equal(dumps[0][f], dumps[1][f]), f
    monkeypatch.setenv('ALAC_B200_CACHE', cache)
    import bench
    wl = bench.build_workload('smoke', seed=2, threads=2)
    n = len(wl['sizes'])
    got = dumps[0]
    idx = got['pcm_packets'].astype(np.int64)
    assert idx[0] == 0 and idx[-1] == n - 1 and len(idx) == len(np.unique(idx))
    assert got['pcm'].shape == (len(idx), 4096, 2) and got['status'].shape == got['out_bytes'].shape == (n,)
    assert (got['status'] == 0).all() and got['out_bytes'].sum() == wl['frames'] * 2 * 3
    for row, i in zip(got['pcm'], idx):
        p = bytes(wl['packed'][int(wl['offsets'][i]):int(wl['offsets'][i]) + int(wl['sizes'][i])])
        st, pcm = ol.decode_packet(wl['cfg'], p)
        want = ol.pcm_bytes_to_int(pcm, 24, 2)
        assert st == 0 and np.array_equal(row[:len(want)], want) and not row[len(want):].any(), i


@pytest.mark.gpu
def test_product_arm_dump_equals_reference_arm(cache, tmp_path):
    """The CUDA path's last timed step, as --dump-outputs writes it, equals the CPU oracle's arrays exactly."""
    ours, ref = str(tmp_path / 'ours'), str(tmp_path / 'ref')
    r = _run(cache, {}, '--only-main', '--no-cpu-baseline', '--dump-outputs', ours, impl='ours')
    assert r.returncode == 0, r.stderr[-1000:]
    assert json.loads(r.stdout)['steps'] == 1
    r = _run(cache, {}, '--dump-outputs', ref)
    assert r.returncode == 0, r.stderr[-500:]
    a, b = _load_dump(ours), _load_dump(ref)
    for f in a:
        assert a[f].dtype == b[f].dtype and np.array_equal(a[f], b[f]), f
