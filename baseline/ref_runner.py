"""Runs the UNMODIFIED reference (Onr/Council-GAN) training step for the comparison legs of bench.py.

MEASUREMENT INFRASTRUCTURE ONLY -- never imported by the product package (council_gan_b200).

Where the reference comes from, in this order (SURVEY.md section 8c/8d):
  1. ``$COUNCIL_REF_DIR``                (a checkout of Onr/Council-GAN)
  2. ``<repo>/oracle/_ref``              (git-ignored install made by ``oracle/install_reference.py`` during the build; it
                                          travels with a copy of the built tree, like a pip --target install would)
If neither exists, callers fall back to the oracle port (oracle/council_oracle.py: a plain-PyTorch restatement that
is pinned against the reference's own outputs) and say so (``kind: "port"``).

Two ways of running it:
  * device ``'cpu'``   -- the reference hard-codes ``.cuda(dev)``; ``Tensor.cuda`` / ``Module.cuda`` are rebound to ``.to(dev)``
                          in THIS process (out-of-tree shim, the reference files are untouched).  Use a subprocess.
  * device ``'cuda:N'`` -- native: stock PyTorch + cuDNN, the library-kernel baseline SURVEY.md 2.1 names ("*that* is the
                          GPU-side number to beat").  cudnn.deterministic = True exactly as train.py:61 sets it; a second
                          number with cudnn.benchmark (autotuned algorithms) is reported beside it.
"""
from __future__ import annotations

import os
import sys
import time
import types

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
NEEDED = ('trainer_council.py', 'networks.py', 'utils.py', 'data.py')


def find_reference():
    if os.environ.get('COUNCIL_REF_DISABLE') == '1':  # tests: exercise the oracle-port fallback
        return None
    for p in (os.environ.get('COUNCIL_REF_DIR'), os.path.join(ROOT, 'oracle', '_ref')):
        if p and all(os.path.exists(os.path.join(p, f)) for f in NEEDED):
            return p
    return None


def import_reference(ref_dir, cpu_shim):
    """-> the reference's Council_Trainer class (unmodified source, imported from ref_dir)."""
    sys.modules.setdefault('torchfile', types.ModuleType('torchfile'))  # utils.py:6; used only by load_vgg16 (dead at vgg_w = 0)
    if ref_dir not in sys.path:
        sys.path.insert(0, ref_dir)
    if cpu_shim:
        import torch.nn as nn
        torch.Tensor.cuda = lambda self, device=None, *a, **k: self.to(device if device is not None else 'cpu')
        nn.Module.cuda = lambda self, device=None: self.to(device if device is not None else 'cpu')
    import trainer_council as ref_tc
    assert os.path.dirname(os.path.abspath(ref_tc.__file__)) == os.path.abspath(ref_dir), \
        'imported %s, not the reference in %s' % (ref_tc.__file__, ref_dir)
    return ref_tc.Council_Trainer


def seed_like_train_py(seed):
    """train.py:55-61 (seed_torch)."""
    import random
    import numpy as np
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    if torch.cuda.is_available():
        torch.cuda.manual_seed(seed)


def make_step(trainer, hp, x_a, x_b, iteration):
    """train.py:241-250: dis_update -> dis_council_update -> gen_update on one minibatch."""
    def step():
        hp['iteration'] = iteration
        trainer.dis_update(x_a, x_b, hp)
        if hp['council']['numberOfCouncil_dis_relative_iteration'] > 0:
            trainer.dis_council_update(x_a, x_b, hp)
        trainer.gen_update(x_a, x_b, hp, iteration)
    return step


def build_reference_trainer(hp, device, ref_dir=None):
    ref_dir = ref_dir or find_reference()
    if ref_dir is None:
        raise FileNotFoundError('no reference tree (COUNCIL_REF_DIR, oracle/_ref)')
    cls = import_reference(ref_dir, cpu_shim=(str(device) == 'cpu'))
    seed_like_train_py(hp.get('random_seed', 1))
    tr = cls(hp, str(device))
    tr.cuda(str(device))  # train.py:87
    return tr, ref_dir


def time_cpu(step, steps, warmup):
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    return (time.perf_counter() - t0) / steps


def time_gpu(step, steps, warmup, device):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize(device)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize(device)
    return e0.elapsed_time(e1) * 1e-3 / steps


def gpu_library_baseline(hp, x_a, x_b, iteration, device, steps=10, warmup=3, tuned=True):
    """The unmodified reference on the GPU under stock PyTorch + cuDNN (train.py:241-251 path).

    -> dict(value images/s, ms_per_step, kind, torch, cudnn, settings ..., value_cudnn_benchmark ...)
    Falls back to the oracle port moved to the device when no reference tree is present (kind "port")."""
    import copy
    hp = copy.deepcopy(hp)
    B = x_a.size(0)
    info = {'torch': torch.__version__, 'cudnn': torch.backends.cudnn.version(), 'batch': B, 'steps': steps, 'warmup': warmup,
            'allow_tf32_cudnn': bool(torch.backends.cudnn.allow_tf32), 'allow_tf32_matmul': bool(torch.backends.cuda.matmul.allow_tf32),
            'unit': 'images/s'}
    xa, xb = x_a.to(device).detach(), x_b.to(device).detach()  # train.py:228
    ref_dir = find_reference()
    prev = (torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark)
    try:
        if ref_dir is not None:
            torch.backends.cudnn.deterministic = True  # train.py:61
            torch.backends.cudnn.benchmark = False
            tr, _ = build_reference_trainer(hp, device, ref_dir)
            step = make_step(tr, hp, xa, xb, iteration)
            info['kind'] = 'unmodified'
            info['source'] = ref_dir
        else:
            sys.path.insert(0, os.path.join(ROOT, 'oracle'))
            import council_oracle as co
            states = co.synth_all_states(hp, seed=7)
            states = {k: [{kk: vv.to(device) for kk, vv in sd.items()} for sd in lst] for k, lst in states.items()}
            tr = co.OracleTrainer(hp, states)
            step = make_step(tr, hp, xa, xb, iteration)
            info['kind'] = 'port'
            info['source'] = 'oracle/council_oracle.py on the device (no reference tree on this box)'
        dt = time_gpu(step, steps, warmup, device)
        info.update(value=B / dt, ms_per_step=dt * 1e3, settings='cudnn.deterministic=True, cudnn.benchmark=False (train.py:61)')
        info['losses'] = {'gen': [float(v) for v in tr.loss_gen_total_s], 'dis': [float(v) for v in tr.loss_dis_total_s]}
        if tuned:
            torch.backends.cudnn.deterministic = False
            torch.backends.cudnn.benchmark = True
            dt2 = time_gpu(step, steps, max(warmup, 3), device)
            info.update(value_cudnn_benchmark=B / dt2, ms_per_step_cudnn_benchmark=dt2 * 1e3)
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = prev
    del tr
    torch.cuda.empty_cache()
    return info
