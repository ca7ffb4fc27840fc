"""bench.py contract pieces that can be checked without a GPU: the reference arm's JSON line (the unmodified reference when a
tree is present, else the oracle port, on a tiny workload) and that the product arm refuses to run without CUDA instead of
falling back to anything."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args, timeout=600, **extra_env):
    env = dict(os.environ, COUNCIL_CPU_THREADS='4', **extra_env)
    return subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), *args], capture_output=True, text=True, timeout=timeout,
                          cwd=ROOT, env=env)


import pytest


@pytest.mark.parametrize('disable_ref', ['0', '1'])
def test_reference_arm_prints_one_contract_line(disable_ref):
    r = run_bench('--impl', 'reference', '--workload', 'tiny_64_n2_b2', '--steps', '1', '--warmup', '0', COUNCIL_REF_DISABLE=disable_ref)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'images/s' and d['higher_is_better'] is True
    assert d['metric'] == 'training images/sec (gen+dis step)' and d['steps'] == 1 and d['warmup'] == 0
    assert d['value'] > 0 and abs(d['value'] - 1e3 / d['ms_per_step']) < 1e-6 * d['value']
    assert d['config']['workload'] == 'tiny_64_n2_b2' and 'model' not in d['config']
    cb = d['cpu_baseline']
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    import ref_runner
    have_ref = disable_ref == '0' and ref_runner.find_reference() is not None
    assert cb['kind'] == ('reference' if have_ref else 'port') and cb['unmodified'] is have_ref
    assert cb['cores'] == 4 and cb['host_cores'] >= 1 and cb['value'] == d['value']
    assert cb['batch_ran'] == 1 and d['config']['batch_ran'] == 1 and d['config']['batch_per_gpu'] == 2  # the sample's batch is stated
    assert d['e2e'] == {'value': d['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_reference_arm_other_ranks_exit_without_work():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--workload', 'tiny_64_n2_b2',
                        '--steps', '1', '--warmup', '0'], capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_dump_outputs_after_one_step(tmp_path):
    """--dump-outputs: float32 arrays of the published losses and a fixed sample of the updated parameters, at most 64 MB."""
    import numpy as np
    import torch
    import bench
    from council_gan_b200.trainer_council import Council_Trainer
    from ops_torch import TorchOps
    hp, n, b, size, it = bench.load_hp('tiny_64_n2_b2')
    torch.manual_seed(1)
    tr = Council_Trainer(hp, 'cpu', _ops=TorchOps('cpu'))
    xa, xb = bench.synth(b, size, 123)
    bench.dump_outputs(tr, str(tmp_path / 'pre'))
    tr.dis_update(xa, xb, hp)
    tr.dis_council_update(xa, xb, hp)
    tr.gen_update(xa, xb, hp, it)
    for out in ('a', 'b'):
        bench.dump_outputs(tr, str(tmp_path / out))
    names = sorted(os.listdir(tmp_path / 'a'))
    assert names == ['loss_dis_council_total.npy', 'loss_dis_total.npy', 'loss_gen_total.npy', 'params_dis_a2b.npy',
                     'params_dis_council_a2b.npy', 'params_gen_a2b.npy']
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in names) <= 64 << 20
    for f in names:
        a = np.load(tmp_path / 'a' / f)
        assert a.dtype == np.float32 and np.isfinite(a).all() and np.array_equal(a, np.load(tmp_path / 'b' / f)), f
    assert np.array_equal(np.load(tmp_path / 'a' / 'loss_gen_total.npy'), np.array([float(v) for v in tr.loss_gen_total_s], np.float32))
    for fam in ('gen', 'dis', 'dis_council'):  # the dump holds the parameters after the step, not before it
        f = 'params_%s_a2b.npy' % fam
        assert not np.array_equal(np.load(tmp_path / 'a' / f), np.load(tmp_path / 'pre' / f)), f
    # the documented sample: the generators' state_dicts in key order, concatenated over the members, at seeded sorted positions
    full = torch.cat([v.detach().float().reshape(-1) for m in tr.gen_a2b_s for v in m.state_dict().values()]).numpy()
    idx = np.sort(np.random.default_rng(0).choice(full.size, bench.DUMP_SAMPLE, replace=False))
    assert np.array_equal(np.load(tmp_path / 'a' / 'params_gen_a2b.npy'), full[idx])


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip('CUDA present: the product arm runs')
    r = run_bench('--workload', 'tiny_64_n2_b2', '--steps', '1', '--warmup', '0', '--no-cpu-baseline', timeout=300)
    assert r.returncode != 0, 'the product arm must fail loudly without a GPU, not fall back'
    assert r.stdout.strip() == ''
