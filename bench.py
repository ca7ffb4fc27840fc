#!/usr/bin/env python
"""bench.py -- training images/sec of the Council-GAN step (dis_update + dis_council_update + gen_update).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one full training iteration (train.py:241-250 order) over one synthetic minibatch.
Default workload = BASELINE.json configs[1]: male2female 256x256, council_size=4, batch 8 per GPU
(weak scaling: configs[3] is the same at 8 GPUs, global batch 64).  All gates open (iteration 60001).

Prints ONE JSON line (rank 0).  `value` = images/sec with inputs resident in HBM; `e2e` = the same through
the public Council_Trainer API with HOST (pinned) image tensors: H2D copies and the D2H loss read are inside
the timed region.  `roofline` is for the dominant convolution kernel, timed live with CUDA events on the
launching stream in a second timed region of the same K steps (the headline region carries no per-kernel events).

`--dump-outputs DIR` writes what the last step of the headline region handed its caller (see dump_outputs) as DIR/<name>.npy;
inputs, initial weights and noise are seeded, so two builds run with the same arguments can be compared output for output.

Comparison legs (measurement infrastructure, baseline/ref_runner.py):
  * `cpu_baseline` / `--impl reference`: the UNMODIFIED reference (`$COUNCIL_REF_DIR` -> oracle/_ref; else the
    oracle port, `kind: "port"`) on the host cores, on a bounded sample of the workload (batch 1 -- the batch really run is
    printed), with the thread count chosen by a sweep at THIS workload (host core count printed);
  * `gpu_library_baseline` (and `--impl reference-gpu`): the same unmodified reference on the same B200 under stock
    PyTorch + cuDNN at the workload's full batch (train.py:241-251 path, cudnn.deterministic as train.py:61, plus a
    cudnn.benchmark number) -- the comparator SURVEY.md 2.1 names.
Before timing, the first step of our arm is checked against the reference's golden losses for the workload (1e-3).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import yaml  # noqa: E402

WORKLOADS = {
    # name: (config yaml, council_size, per-GPU batch, image size, iteration with every gate open)
    'male2female_256_n4_b8': ('male2female', 4, 8, 256, 60001),
    'selfie2anime_256_n4_b4': ('selfie2anime', 4, 4, 256, 2001),
    'glasses_128_n2_b1': ('glasses', 2, 1, 128, 20001),
    'male2female_512_n6_b2': ('male2female', 6, 2, 512, 60001),
    'tiny_64_n2_b2': ('glasses', 2, 2, 64, 20001),
}
ALG_GMAC_PER_IMAGE_MEMBER_256 = 486.7  # SURVEY.md section 8(d): algorithmic work, K=4


def load_hp(workload):
    cfg, n, b, size, it = WORKLOADS[workload]
    hp = yaml.safe_load(open(os.path.join(ROOT, 'configs', cfg + '.yaml')))
    hp['council']['council_size'] = n
    hp['batch_size'] = b
    hp['iteration'] = it
    for k in ('new_size', 'crop_image_height', 'crop_image_width'):
        hp[k] = size
    return hp, n, b, size, it


def synth(batch, size, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(batch, 3, size, size, generator=g) * 2 - 1, torch.rand(batch, 3, size, size, generator=g) * 2 - 1


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(',')])
            except Exception:
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons),
                'samples': len(sm)}


GOLDEN_FOR = {'male2female_256_n4_b8': 'm2f256_n4_b8', 'selfie2anime_256_n4_b4': 'anime256_n4_b4',
              'male2female_512_n6_b2': 'm2f512_n6_b2', 'glasses_128_n2_b1': 'glasses128_n2_b1'}


def reference_cpu_rate(workload, steps, warmup):
    """images/sec of the reference's own CPU implementation on a bounded sample (batch 1) of the workload.
    -> (rate, seconds per step, info dict for cpu_baseline)."""
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    import ref_runner as rr
    hp, n, b, size, it = load_hp(workload)
    sample_batch = 1
    hp['batch_size'] = sample_batch
    host = os.cpu_count() or 1
    x_a, x_b = synth(sample_batch, size, 123)
    ref_dir = rr.find_reference()
    if ref_dir is not None:
        tr, _ = rr.build_reference_trainer(hp, 'cpu', ref_dir)
        kind, what = 'reference', 'the unmodified reference (%s) on CPU, .cuda(dev) rebound to .to(dev)' % ref_dir
    else:
        sys.path.insert(0, os.path.join(ROOT, 'oracle'))
        import council_oracle as co
        tr = co.OracleTrainer(hp, co.synth_all_states(hp, seed=7))
        co.seed_all(1)
        kind, what = 'port', 'oracle/council_oracle.py (plain-PyTorch restatement pinned against the reference; no reference tree on this box)'
    step = rr.make_step(tr, hp, x_a, x_b, it)
    # thread count: measured at THIS workload (one dis_update per candidate), not assumed
    forced = os.environ.get('COUNCIL_CPU_THREADS')
    sweep = {}
    if forced:
        cores = max(1, min(host, int(forced)))
    else:
        cands = sorted(set(c for c in (4, 8, 16, 32, 64, host) if c <= host))
        torch.set_num_threads(cands[0])
        hp['iteration'] = it
        tr.dis_update(x_a, x_b, hp)  # page-in / allocator warm-up
        for c in cands:
            torch.set_num_threads(c)
            t0 = time.perf_counter()
            tr.dis_update(x_a, x_b, hp)
            sweep[str(c)] = round(time.perf_counter() - t0, 3)
            if sweep[str(c)] > 3.0 * min(sweep.values()):
                break  # oversubscribed: larger counts only get worse
        cores = int(min(sweep, key=sweep.get))
    torch.set_num_threads(cores)
    dt = rr.time_cpu(step, steps, warmup)
    info = {'value': sample_batch / dt, 'unit': 'images/s', 'cores': cores, 'host_cores': host, 'kind': kind,
            'unmodified': kind == 'reference', 'batch_ran': sample_batch, 'thread_sweep_s_per_dis_update': sweep,
            'sample': 'one full iteration (dis + dis_council + gen update) of the same config at batch %d (config batch %d): %s; '
                      '%d torch threads chosen by the sweep on a %d-core host' % (sample_batch, b, what, cores, host)}
    return sample_batch / dt, dt, info


def reference_cpu_subprocess(workload):
    """cpu_baseline leg of our arm: the reference arm in a clean process (its .cuda shim and thread settings stay there)."""
    r = subprocess.run([sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--workload', workload, '--steps', '1',
                        '--warmup', '1'], capture_output=True, text=True, timeout=1500, cwd=ROOT,
                       env={k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')})
    for line in reversed(r.stdout.splitlines()):
        if line.startswith('{'):
            return json.loads(line)['cpu_baseline']
    return {'error': (r.stderr or r.stdout)[-400:]}


def parity_check(trainer_cls, workload, dev, tc):
    """First step of our arm vs the reference's golden losses for this workload (tests/golden, generated from the unmodified
    reference by oracle/make_golden.py).  Checker use of oracle/ only: the synthetic parameter/input generators."""
    case = GOLDEN_FOR.get(workload)
    path = os.path.join(ROOT, 'tests', 'golden', '%s.json' % case)
    if case is None or not os.path.exists(path):
        return {'checked': False, 'why': 'no golden fixture for this workload'}
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    import council_oracle as co
    from common import load_golden, setup_case
    gold = load_golden(case)
    hp, states, x_a, x_b = setup_case(gold)
    co.seed_all(hp['random_seed'])
    tr = trainer_cls(hp, dev)
    tr.ops.set_tensor_core_mode(tc)
    for name, lst in states.items():
        fam, d = name.rsplit('_', 1)
        for i, sd in enumerate(lst):
            getattr(tr, '%s_%s_s' % (fam, d))[i].load_state_dict(sd)
    co.seed_all(gold['rng_seed'])
    tr.dis_update(x_a, x_b, hp)
    tr.dis_council_update(x_a, x_b, hp)
    tr.gen_update(x_a, x_b, hp, gold['iteration'])
    worst = 0.0
    for got, want in ((tr.loss_dis_total_s, gold['loss_dis_total']), (tr.loss_dis_council_total_s, gold['loss_dis_council_total']),
                      (tr.loss_gen_total_s, gold['loss_gen_total'])):
        for g, w in zip(got, want):
            worst = max(worst, abs(float(g) - w) / abs(w))
    del tr
    torch.cuda.empty_cache()
    return {'checked': True, 'case': case, 'worst_rel_loss_err_vs_reference': worst, 'tol': 1e-3, 'ok': bool(worst < 1e-3)}


DUMP_SAMPLE = 1 << 20  # parameter values kept per network family (4 MB of float32): a few families stay far below 64 MB


def dump_outputs(trainer, out_dir):
    """Write what a caller of the step receives after it, as float32 DIR/<name>.npy: the per-member total losses the three
    updates publish, and per network family (gen/dis/dis_council x direction) every member's updated state_dict, flattened
    in key order and concatenated over the members.  A family larger than DUMP_SAMPLE values keeps a fixed, seeded sample
    of them (same positions, in increasing order, on every run of the same workload)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    for name in ('loss_dis_total', 'loss_dis_council_total', 'loss_gen_total'):
        vals = getattr(trainer, name + '_s', None)
        if vals is not None:
            arrays[name] = np.array([float(v) for v in vals], dtype=np.float32)
    for d in ('a2b', 'b2a'):
        for fam in ('gen', 'dis', 'dis_council'):
            members = getattr(trainer, '%s_%s_s' % (fam, d), None)
            if not members:
                continue
            # a generator's state_dict mixes device parameters with host-side norm running statistics
            flat = torch.cat([v.detach().to('cpu', torch.float32).reshape(-1) for m in members for v in m.state_dict().values()]).numpy()
            if flat.size > DUMP_SAMPLE:
                flat = flat[np.sort(np.random.default_rng(0).choice(flat.size, DUMP_SAMPLE, replace=False))]
            arrays['params_%s_%s' % (fam, d)] = flat
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'reference-gpu'])
    ap.add_argument('--workload', default='male2female_256_n4_b8', choices=list(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-baseline', action='store_true')
    ap.add_argument('--no-parity-check', action='store_true')
    ap.add_argument('--tc', type=int, default=1, help='0: SIMT fp32 kernels only, 1: tcgen05 TF32 where supported')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    assert args.warmup >= 0 and args.steps >= 1
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    hp, n_members, batch, size, it = load_hp(args.workload)
    scale = (size / 256.0) ** 2
    metric, unit = 'training images/sec (gen+dis step)', 'images/s'
    config = {'workload': args.workload, 'council_size': n_members, 'batch_per_gpu': batch, 'global_batch': batch * world,
              'image': '%dx%d' % (size, size), 'parallelism': 'dp%d' % world, 'iteration': it,
              'l2': 'per-step working set (saved activations, several GB) >> 126 MB L2; no explicit flush'}

    # ------------------------------------------------------------------ reference arm: the reference's own CPU path
    if args.impl == 'reference':
        if rank != 0:
            return 0
        rate, dt, info = reference_cpu_rate(args.workload, args.steps, args.warmup)
        config['batch_ran'] = info['batch_ran']
        line = {'impl': 'reference', 'metric': metric, 'value': rate, 'unit': unit, 'n_gpus': args.gpus, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config, 'cpu_baseline': info,
                'e2e': {'value': rate, 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ library-kernel arm: the reference on the GPU (stock PyTorch + cuDNN)
    if args.impl == 'reference-gpu':
        if rank != 0:
            return 0
        sys.path.insert(0, os.path.join(ROOT, 'baseline'))
        import ref_runner as rr
        torch.cuda.set_device(local_rank)
        dev = 'cuda:%d' % local_rank
        x_a, x_b = synth(batch, size, 123)
        sampler = ClockSampler(local_rank)
        sampler.start()
        info = rr.gpu_library_baseline(hp, x_a, x_b, it, dev, steps=args.steps, warmup=args.warmup)
        clocks = sampler.stop()
        line = {'impl': 'reference-gpu', 'metric': metric, 'value': info['value'], 'unit': unit, 'n_gpus': 1, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': info['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
                'vs_baseline': None, 'dtype': 'tf32 (cudnn.allow_tf32 as shipped)', 'data': 'synthetic', 'config': config,
                'clocks': clocks, 'gpu_library_baseline': info}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dev = 'cuda:%d' % local_rank
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device(dev))
    from council_gan_b200 import Council_Trainer
    import random
    import numpy as np
    random.seed(1)
    np.random.seed(1)
    torch.manual_seed(1)
    parity = None
    if world == 1 and not args.no_parity_check:
        parity = parity_check(Council_Trainer, args.workload, dev, args.tc)
        if parity.get('checked') and not parity['ok']:
            print('PARITY CHECK FAILED: %r' % (parity,), file=sys.stderr)
    random.seed(1)
    np.random.seed(1)
    torch.manual_seed(1)
    trainer = Council_Trainer(hp, dev)
    ops = trainer.ops
    ops.set_tensor_core_mode(args.tc)
    xa_h, xb_h = synth(batch * world, size, 123)
    xa_h = xa_h[rank * batch:(rank + 1) * batch].contiguous().pin_memory()
    xb_h = xb_h[rank * batch:(rank + 1) * batch].contiguous().pin_memory()
    xa_d, xb_d = xa_h.to(dev), xb_h.to(dev)

    def step(xa, xb):
        trainer.dis_update(xa, xb, hp)
        trainer.dis_council_update(xa, xb, hp)
        trainer.gen_update(xa, xb, hp, it)
        trainer.update_learning_rate()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    for _ in range(max(args.warmup, 0)):
        step(xa_d, xb_d)
    sampler = ClockSampler(local_rank)  # every rank samples its own GPU: the step is power-limited and max-over-ranks timed
    sampler.start()
    l0 = ops.launch_count()
    ms = timed(lambda: step(xa_d, xb_d), args.steps)   # the headline timed region: nothing but the step's own launches in the stream
    launches = ops.launch_count() - l0
    if args.dump_outputs and rank == 0:  # the regions below keep training the same trainer
        dump_outputs(trainer, args.dump_outputs)
    # second timed region of the same K steps with a CUDA-event pair around every convolution / HBM-pass launch (per-kernel averages for
    # the roofline): ~800 event records per step cost host time (the 128x128 configuration is launch-bound) and sit between kernels that
    # would otherwise overlap their launch, so they are kept out of the headline region; shares are taken against THIS region's time
    ops.start_timing()
    ms_prof = timed(lambda: step(xa_d, xb_d), args.steps)
    ktimes = ops.stop_timing()
    clocks = sampler.stop()
    if world > 1:  # median SM clock of every rank's GPU during the timed region (the slowest GPU sets the step time)
        mhz = torch.tensor([float(clocks['sm_mhz'] or 0.0)], device=dev)
        allm = [torch.zeros_like(mhz) for _ in range(world)]
        dist.all_gather(allm, mhz)
        clocks['sm_mhz_per_rank'] = [float(t.item()) for t in allm]
    ms_per_step = ms / args.steps
    value = batch * world / (ms_per_step * 1e-3)

    # end to end through the public API with HOST tensors: every step gets its own pinned minibatch (as train.py:225-228's data
    # loader does), so the H2D copy and the NCHW -> channels-last conversion happen inside every timed step; the losses are
    # read back to the host at the end of every step
    d2h = [0]
    host_batches = [(xa_h.clone().pin_memory(), xb_h.clone().pin_memory()) for _ in range(args.steps + 1)]
    it_host = iter(host_batches)
    misses0 = trainer.img_cache_misses

    def e2e_step():
        xa, xb = next(it_host)
        step(xa, xb)
        vals = [float(v) for v in trainer.loss_gen_total_s] + [float(v) for v in trainer.loss_dis_total_s]
        d2h[0] = 4 * len(vals) + 4 * 6 * n_members
        return vals

    e2e_step()
    m1 = trainer.img_cache_misses
    ms_e2e = timed(e2e_step, args.steps) / args.steps
    assert trainer.img_cache_misses - m1 == 2 * args.steps, 'every e2e step must upload its own two image batches'
    e2e = {'value': batch * world / (ms_e2e * 1e-3), 'unit': unit, 'ms_per_step': ms_e2e,
           'h2d_bytes_per_step': int(2 * xa_h.numel() * 4), 'd2h_bytes_per_step': int(d2h[0]),
           'fresh_host_tensors_per_step': True, 'image_uploads_in_timed_region': int(trainer.img_cache_misses - m1)}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # roofline of the dominant kernel (largest share of the timed region among the timed conv launches)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    roofline = None
    roofline_hbm = None
    hbm_times = {k: v for k, v in (ktimes or {}).items() if k.startswith('hbm:')}
    ktimes = {k: v for k, v in (ktimes or {}).items() if not k.startswith('hbm:')}
    if hbm_times:
        # the largest HBM-bound kernel group of the step: algorithmic bytes / measured launch time vs the measured copy bandwidth
        hkey, (h_ms, h_cnt, h_bytes) = max(hbm_times.items(), key=lambda kv: kv[1][0])
        hbm_peak = peaks.get('hbm_gbs', 6500.0)
        h_ach = h_bytes / (h_ms / h_cnt * 1e-3) / 1e9
        roofline_hbm = {'bound': 'hbm', 'kernel': hkey[4:], 'achieved': h_ach, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': h_ach / hbm_peak,
                        'bytes_per_launch': h_bytes, 'launches': h_cnt, 'avg_ms': h_ms / h_cnt, 'share_of_step': h_ms / ms_prof,
                        'all_hbm_kernels_ms_per_step': round(sum(v[0] for v in hbm_times.values()) / args.steps, 3),
                        'peak_source': 'MEASURED_PEAKS.json hbm_gbs (copy bandwidth)' if peaks else 'fallback 6500'}
    # MEASURED_PEAKS.json has no TF32 figure: measure the library TF32 GEMM on this box (cuBLAS through torch.matmul, 8192^3, best of
    # 10 after warm-up) as a second, like-for-like denominator for the TF32 convolution kernels
    tf32_lib = None
    try:
        prev = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        ma = torch.randn(8192, 8192, device=dev)
        mb = torch.randn(8192, 8192, device=dev)
        for _ in range(3):
            torch.matmul(ma, mb)
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(ma, mb)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        tf32_lib = 2.0 * 8192 ** 3 / (best * 1e-3) / 1e12
        torch.backends.cuda.matmul.allow_tf32 = prev
        del ma, mb
    except Exception:
        pass
    if ktimes:
        key, (tot_ms, cnt, flops) = max(ktimes.items(), key=lambda kv: kv[1][0])
        tf32_peak = peaks.get('bf16_tflops_sustained', 1400.0) / 2.0  # TF32 runs at half the bf16 tensor rate
        ach = flops / (tot_ms / cnt * 1e-3) / 1e12
        traffic = tensor_pipe = None
        try:
            ent = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json'))).get(key, {})
            traffic, tensor_pipe = ent.get('traffic_bytes'), ent.get('tensor_pipe_pct')
        except Exception:
            pass
        roofline = {'bound': 'tensor', 'kernel': key, 'achieved': ach, 'peak': tf32_peak, 'unit': 'TFLOP/s', 'frac': ach / tf32_peak,
                    'frac_of_nominal_tf32_1100': ach / 1100.0, 'flops_per_launch': flops,
                    'tf32_cublas_tflops_measured_here': tf32_lib, 'frac_of_tf32_cublas': (ach / tf32_lib) if tf32_lib else None,
                    'traffic': traffic, 'tensor_pipe_pct_ncu': tensor_pipe, 'launches': cnt, 'avg_ms': tot_ms / cnt, 'share_of_step': tot_ms / ms_prof,
                    'timed_region_ms_per_step': ms_prof / args.steps,
                    'peak_source': ('MEASURED_PEAKS.json bf16_tflops_sustained / 2 (TF32 operands)' if peaks else 'fallback 1400/2')}
    alg_tflop = 2 * ALG_GMAC_PER_IMAGE_MEMBER_256 * 1e9 * scale * n_members * batch * world / 1e12
    line = {'metric': metric, 'value': value, 'unit': unit, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'tf32' if args.tc else 'f32', 'data': 'synthetic', 'config': config, 'clocks': clocks, 'e2e': e2e,
            'gpu_launches': int(launches), 'tensor_map_cache': ops.tensor_map_cache_stats(), 'roofline': roofline, 'roofline_hbm': roofline_hbm,
            'step_algorithmic_tflops': alg_tflop / (ms_per_step * 1e-3) / world,
            'kernel_times_ms_per_step': ({k: round(v[0] / args.steps, 3) for k, v in sorted(ktimes.items(), key=lambda kv: -kv[1][0])[:60]}
                                         if ktimes else None),
            'hbm_kernel_times_ms_per_step': ({k[4:]: round(v[0] / args.steps, 3) for k, v in sorted(hbm_times.items(), key=lambda kv: -kv[1][0])[:20]}
                                             if hbm_times else None),
            'losses': {'gen': [float(v) for v in trainer.loss_gen_total_s], 'dis': [float(v) for v in trainer.loss_dis_total_s]}}
    line['parity_check'] = parity
    if world == 1 and not args.no_gpu_baseline:
        # the comparator SURVEY.md 2.1 / 8d names: the unmodified reference on this same GPU under stock PyTorch + cuDNN
        torch.cuda.empty_cache()
        sys.path.insert(0, os.path.join(ROOT, 'baseline'))
        import ref_runner as rr
        try:
            gb = rr.gpu_library_baseline(hp, xa_h, xb_h, it, dev, steps=args.steps, warmup=args.warmup)
            gb['ours_over_baseline'] = value / gb['value']
            gb['ours_over_baseline_cudnn_benchmark'] = value / gb['value_cudnn_benchmark'] if gb.get('value_cudnn_benchmark') else None
        except Exception as e:  # the comparison leg must never take the product line down
            gb = {'error': '%s: %s' % (type(e).__name__, str(e)[:300])}
        line['gpu_library_baseline'] = gb
    if not args.no_cpu_baseline:
        line['cpu_baseline'] = reference_cpu_subprocess(args.workload)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == '__main__':
    sys.exit(main())
