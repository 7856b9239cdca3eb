#!/usr/bin/env python
"""bench.py -- the legs of BASELINE.json's metric, one JSON line per run.

  python bench.py --gpus N --steps K --warmup W                       headline: CDAE training samples/s, configs[2]
  python bench.py --workload {c1,c2,c4_sampled,c4_full,small} ...     the other configs of the metric
  python bench.py --impl reference [--workload ...]                   the reference-semantics CPU path (oracle port)
  python bench.py ... --dump-outputs DIR                              also the outputs of the last timed step, as .npy
  N > 1: launched by torch.distributed.run, one rank per GPU (c3: data-parallel / item-sharded step; c4_*: users
  partitioned over ranks, no collective)

A "step" = one pass of the hot path over one batch: an optimizer step on B sampled users (CDAE) / pairs (DMF), or the
ranking of one block of users (c4).  Every line carries `value` (inputs resident in HBM, CUDA events on the launching
stream), `e2e` (the public call with host buffers: H2D of the inputs and D2H of the result inside the timed region),
`roofline` (dominant kernel, timed live with CUDA events inside libdrb in a separate pass) and `cpu_baseline` (the
oracle port on the host cores, bounded sample, rank 0 at N=1).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

C3 = dict(name='c3', title='cdae_ml20m_shape', origin='BASELINE.json configs[2]', model='cdae', n_users=138493,
          n_items=26744, nnz=20_000_000, hidden=200, batch=4096, q=0.2, lr=1e-3, reg=1e-3, neg_ratio=5, seed=10,
          zipf_a=1.0, mask='philox')
C1 = dict(name='c1', title='cdae_ml100k_shape', origin='BASELINE.json configs[0]', model='cdae', n_users=943,
          n_items=1682, nnz=100_000, hidden=50, batch=64, q=0.2, lr=1e-3, reg=1e-3, neg_ratio=5, seed=10, zipf_a=0.0,
          mask='mt19937')
SMALL = dict(name='small', title='cdae_small_debug', origin='debug shape, not a BASELINE.json config', model='cdae',
             n_users=6040, n_items=3706, nnz=1_000_000, hidden=200, batch=1024, q=0.2, lr=1e-3, reg=1e-3, neg_ratio=5,
             seed=10, zipf_a=1.0, mask='philox')
C2 = dict(name='c2', title='dmf_ml1m_shape', origin='BASELINE.json configs[1]', model='dmf', n_users=6040, n_items=3706,
          nnz=1_000_000, towers=[64, 32], batch=256, lr=1e-3, reg=1e-4, neg_ratio=5, seed=10, zipf_a=0.0)
C4S = dict(C3, name='c4_sampled', title='ranking_evaluation_leave1out_100neg', origin='BASELINE.json configs[3]',
           model='rank_sampled', n_neg=100, k=10)
C4F = dict(C3, name='c4_full', title='full_catalog_top100', origin='BASELINE.json configs[3]', model='topk', k=100,
           score_batch=int(os.environ.get('DRB_BENCH_SCORE_BATCH', -1)))   # users per scoring block (fit(score_batch=));
                                                                           # -1: one 256-user tile per pair of SMs
C5 = dict(name='c5', title='cdae_10m_x_1m_item_sharded', origin='BASELINE.json configs[4]', model='cdae_sharded',
          n_users=10_000_000, n_items=1_000_000, nnz=1_000_000_000, hidden=256, batch=4096, q=0.2, lr=1e-3, reg=1e-3,
          seed=10, zipf_a=1.0, neg_total=1024)
WORKLOADS = {c['name']: c for c in (C3, C1, SMALL, C2, C4S, C4F, C5)}


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], tf=d['bf16_tflops_sustained'], tf_burst=d['bf16_tflops'], src='measured')
    return dict(hbm=6650.0, tf=1400.0, tf_burst=1590.0, src='fallback')


def load_traffic():
    """ncu --set full DRAM bytes per launch, from the newest profiles/*traffic.json."""
    best = None
    pdir = os.path.join(ROOT, 'profiles')
    for f in sorted(os.listdir(pdir)) if os.path.isdir(pdir) else []:
        if f.endswith('traffic.json'):
            best = os.path.join(pdir, f)
    return json.load(open(best)).get('dram_bytes_per_launch', {}) if best else {}


def make_data(cfg):
    import drecpy_b200 as drb
    t = time.time()
    u, i, v = drb.synthetic_interactions(cfg['n_users'], cfg['n_items'], cfg['nnz'], seed=cfg['seed'],
                                         zipf_a=cfg['zipf_a'])
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    ds.csr(1e-3)
    return ds, time.time() - t


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader,nounits',
                                          '-lms', '50', '-i', str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            time.sleep(0.25)                   # let the first samples arrive before the timed region starts
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if r and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for j, n in enumerate(names) if any(len(r) > 3 + j and r[3 + j].startswith('Active') for r in self.rows)]
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


class Dist:
    """torch.distributed plumbing: one process per GPU, NCCL."""

    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get('RANK', '0'))
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(self.local)
        self.dev = torch.device(f'cuda:{self.local}')
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group('nccl', device_id=self.dev)
            self.dist = dist

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], device=self.dev, dtype=self.torch.float64)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        t = self.torch.tensor([float(x)], device=self.dev, dtype=self.torch.float64)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def finish(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()


def timed_steps(D, run_step, warmup, steps, flush_l2=False):
    """W untimed + K timed steps, CUDA events on the current stream, barrier + synchronize on both sides, max over
    ranks.  flush_l2: a 256 MiB memset between steps and every step timed on its own (L2-resident working sets)."""
    torch = D.torch
    for s in range(warmup):
        run_step(s)
    D.barrier()
    clocks = ClockSampler(D.local).start()
    if not flush_l2:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for s in range(warmup, warmup + steps):
            run_step(s)
        e1.record()
        D.barrier()
        ms = e0.elapsed_time(e1)
    else:
        junk = torch.empty(256 << 20, dtype=torch.uint8, device=D.dev)
        evs = []
        for s in range(warmup, warmup + steps):
            junk.fill_(s & 0xff)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            run_step(s)
            b.record()
            evs.append((a, b))
        D.barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
    info = clocks.stop()
    return D.max_over_ranks(ms), info


def profile_kernels(ctx, run_step, passes):
    from drecpy_b200 import _lib
    lib = _lib.load()
    _lib.check(lib.drb_ctx_profile_enable(ctx, 1))
    for s in range(passes):
        run_step(s)
    prof = _lib.profile_read(ctx)
    _lib.check(lib.drb_ctx_profile_enable(ctx, 0))
    return {k: round(v[0] / passes, 5) for k, v in prof.items()}


DUMP_BUDGET = 60_000_000           # bytes over all files of --dump-outputs: under 64 MB with room for the .npy headers


def dump_outputs(out_dir, arrays):
    """Writes the device tensors a caller of the timed path receives after its last step as out_dir/<name>.npy, so that
    two builds run with the same arguments can be compared output for output.  float64 stays float64, integers become
    float64 (exact), other floats float32.  Smallest first, a tensor is written whole when it fits an equal share of the
    budget still left, otherwise as a fixed sample of its rows, in row order: the first rows of numpy
    default_rng(0).permutation(n_rows).  So the sample depends only on the shapes, and two tensors with the same number
    of rows share the sampled rows of the smaller sample."""
    import torch
    os.makedirs(out_dir, exist_ok=True)

    def np_dtype(t):
        return np.float32 if t.dtype.is_floating_point and t.dtype != torch.float64 else np.float64
    items = sorted(arrays.items(), key=lambda kv: kv[1].numel() * np.dtype(np_dtype(kv[1])).itemsize)
    left = DUMP_BUDGET
    for j, (name, t) in enumerate(items):
        dt = np_dtype(t)
        row = int(np.prod(t.shape[1:])) * np.dtype(dt).itemsize
        share = left // (len(items) - j)
        if t.dim() and t.shape[0] * row > share:
            idx = np.sort(np.random.default_rng(0).permutation(t.shape[0])[:max(1, share // row)])
            t = t[torch.as_tensor(idx, device=t.device)]
        h = np.ascontiguousarray(t.detach().cpu().numpy(), dtype=dt)
        np.save(os.path.join(out_dir, name + '.npy'), h)
        left -= h.nbytes


def base_line(cfg, metric, unit, value, world, K, W, ms_total, config, clocks, launches, scaling='weak'):
    return {'metric': metric, 'value': value, 'unit': unit, 'n_gpus': world, 'steps': K, 'warmup': W,
            'ms_per_step': ms_total / K, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': config, 'clocks': clocks, 'gpu_launches': int(launches)}


def hbm_roofline(kernel, alg_bytes, ms, peaks, traffic=None, note=None):
    gbs = alg_bytes / (ms * 1e-3) / 1e9 if ms and ms > 0 else None
    return {'kernel': kernel, 'bound': 'hbm', 'achieved': gbs, 'peak': peaks['hbm'], 'unit': 'GB/s',
            'frac': gbs / peaks['hbm'] if gbs else None, 'traffic': traffic, 'peak_source': f"{peaks['src']} copy",
            'algorithmic_bytes_per_launch': alg_bytes, 'ms_per_launch': ms, 'note': note}


# ========================================================================================== CDAE training (c3, c1, small)
def cdae_config(cfg, n_gpus, parallelism=None, flush=False):
    big = cfg['name'] == 'c3'
    return {'workload': f"{cfg['title']}: CDAE hidden_factors={cfg['hidden']} bce q={cfg['q']} on synthetic "
                        f"{cfg['n_users']}x{cfg['n_items']} / {cfg['nnz']} interactions ({cfg['origin']})",
            'batch_per_gpu': cfg['batch'], 'global_batch': cfg['batch'] * n_gpus, 'neg_ratio': cfg['neg_ratio'],
            'label_mode': 'batch_mean', 'adam': 'dense, per-variable step counter',
            'mask_rng': {'philox': 'philox (device; documented deviation from the MT19937 stream)',
                         'mt19937': 'mt19937 (bit-exact replay of cdae.py:63-64 on the host, keep bytes uploaded)',
                         'mt19937_device': 'mt19937 (bit-exact replay of cdae.py:63-64 on the device by jump-ahead, '
                                           'one k_mt_keep launch per step)'}[cfg['mask']],
            'item_popularity': f"zipf a={cfg['zipf_a']}" if cfg['zipf_a'] else 'uniform',
            'parallelism': parallelism or f'dp{n_gpus}',
            'l2': ('per-step working set (params + Adam state + dz ~ 2.7 GB) exceeds the 126 MB L2; no flush needed'
                   if big else ('L2 flushed between steps (256 MiB memset), every step timed on its own' if flush else
                                'working set is L2 resident; back-to-back steps'))}


def cdae_roofline(kernels, cfg, n_params, peaks, traffic_table, world=1):
    """Dominant family = the three output-layer GEMMs (forward + fused loss epilogue, dW'^T, dh): tensor bound.
    achieved = ALGORITHMIC flops (SURVEY 8d: 6*K*I per sampled user) / their time; peak = measured sustained bf16."""
    hidden, n_items, batch = cfg['hidden'], cfg['n_items'], cfg['batch']
    gemm = {k: v for k, v in kernels.items() if k.startswith('k_sgemm') or k.startswith('k_umma')}
    gemm_ms = sum(gemm.values())
    flops = 6.0 * hidden * n_items * batch
    achieved = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else None
    tc_path = any(k.startswith('k_umma') for k in kernels)
    traffic = None
    if tc_path and traffic_table and cfg['name'] == 'c3':
        traffic = sum(traffic_table.get(k, 0) for k in gemm) or None
    adam_ms = kernels.get('k_adam', float('nan'))
    # 28 B per parameter (w, m, v read + written, g read); the gradient of user-table rows without a sampled user is
    # known to be zero and is not read: at most `batch * world` of the n_users rows carry one
    ld = -(-hidden // 4) * 4
    v_rows_untouched = max(0, cfg['n_users'] - batch * max(1, world))
    adam_bytes = 28.0 * n_params - 4.0 * v_rows_untouched * ld
    adam_gbs = adam_bytes / (adam_ms * 1e-3) / 1e9
    return {'kernel': ' + '.join(sorted(gemm)) + (' (tcgen05 split-precision GEMMs: output layer fwd + fused loss '
                                                   "epilogue, dW'^T, dh)" if tc_path else ' (fp32 FFMA path)'),
            'bound': 'tensor', 'achieved': achieved, 'peak': peaks['tf'], 'unit': 'TFLOP/s',
            'frac': (achieved / peaks['tf']) if achieved else None, 'traffic': traffic,
            'algorithmic_flops_per_step': flops, 'ms_per_step_family': gemm_ms,
            'note': 'achieved counts the algorithmic fp32 flops (6*K*I per sampled user); every fp32-accurate product is '
                    'issued as 3 reduced-precision MMAs, so the issued-MMA rate is 3x achieved',
            'peak_source': f"{peaks['src']} bf16 sustained",
            'share_of_step': gemm_ms / sum(kernels.values()) if kernels else None,
            'secondary': {'k_adam': {'bound': 'hbm', 'achieved': adam_gbs, 'peak': peaks['hbm'], 'unit': 'GB/s',
                                     'frac': adam_gbs / peaks['hbm'], 'algorithmic_bytes_per_step': adam_bytes}}}


def dp_parity(D):
    """N-rank step vs the single-rank step on the same GLOBAL batch (mini problem), both parallel modes; printed in
    the bench line so multi-GPU correctness is visible in the driver's own run.  Every rank takes part; rank 0 also
    runs the single-rank model."""
    import torch
    import drecpy_b200 as drb
    from drecpy_b200.parallel import DataParallel
    U, I, K, B, steps = 1003, 2501, 72, 128, 5
    u, i, v = drb.synthetic_interactions(U, I, 60000, seed=4)
    ds = drb.InteractionData(u, i, v)
    rng = np.random.default_rng(5)

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo))
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    w = {'W': glorot((I, K), I, K), 'W_': glorot((K, I), K, I), 'V': glorot((U, K), U, K), 'b': glorot((K,), K, K),
         'b_': glorot((I,), I, I)}
    ref_losses, ref_w = None, None
    if D.rank == 0:
        ref = drb.CDAE(hidden_factors=K, seed=10, verbose=False, rng_mode='philox', device=str(D.dev))
        ref.fit(ds, epochs=0, batch_size=B * D.world, init_weights=w)
        ref_losses = []
        for s in range(1, steps + 1):
            ref._step = s
            ref_losses.append(ref._train_step(B * D.world, 1e-3, want_loss=True))
        ref_w = {k: getattr(ref, k).detach().clone() for k in ('W', 'W_', 'V', 'b', 'b_')}
        del ref
    out = {}
    for mode in ('data', 'items'):
        m = drb.CDAE(hidden_factors=K, seed=10, verbose=False, rng_mode='philox', device=str(D.dev))
        m.fit(ds, epochs=0, batch_size=B, init_weights=w, data_parallel=DataParallel(D.dist), parallel_mode=mode)
        losses = []
        for s in range(1, steps + 1):
            m._step = s
            losses.append(m._train_step(B, 1e-3, want_loss=True))
        full = m.gather_full_weights()
        if D.rank == 0:
            loss_rel = max(abs(a - b) / abs(b) for a, b in zip(losses, ref_losses))
            w_rel = max(float((full[k] - ref_w[k]).abs().max() / ref_w[k].abs().max()) for k in ref_w)
            out[mode] = {'loss_rel': loss_rel, 'w_rel': w_rel, 'steps': steps, 'ok': bool(loss_rel < 1e-4 and w_rel < 5e-4)}
        del m
        D.barrier()
    torch.cuda.empty_cache()
    if D.rank == 0:
        out['shape'] = f'{U}x{I}, K={K}, global batch {B * D.world}, {D.world} ranks vs 1 rank'
    return out


def cdae_cpu_arm(cfg, ds, steps, warmup, budget_s):
    """Reference-semantics CPU path: oracle port of the step (batch-mean labels, per-variable Adam counter, dense Adam
    + L2; numpy / BLAS on all host cores) fed by the oracle's own sampler -- nothing from libdrb.  The corruption draw
    is the reference's MT19937 stream at c1 and a numpy Bernoulli draw at the large shapes (cheaper than the reference's
    n_items Python draws per user).  Sampler time is also reported on its own."""
    import random
    from oracle.cdae import CDAEOracle, corruption_keep_mt
    from oracle.sampler import PointSamplerOracleCSR
    rng = np.random.default_rng(1)
    U, I, K, B = cfg['n_users'], cfg['n_items'], cfg['hidden'], cfg['batch']

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo))
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    o = CDAEOracle(glorot((I, K), I, K), glorot((K, I), K, I), glorot((U, K), U, K), glorot((K,), K, K),
                   glorot((I,), I, I), ds.csr(), interaction_threshold=1e-3, corruption_level=cfg['q'],
                   learning_rate=cfg['lr'])
    sampler = PointSamplerOracleCSR(ds.uid, ds.iid, ds.interaction, cfg['neg_ratio'], 1e-3, cfg['seed'])
    mask_rng, brng = random.Random(cfg['seed']), np.random.default_rng(0)
    t_sampler = [0.0]

    def one(b):
        t0 = time.time()
        uids = np.array([t[0] for t in sampler.sample(b)])
        t_sampler[0] += time.time() - t0
        if cfg['mask'] == 'mt19937':
            keep = np.stack([corruption_keep_mt(mask_rng, I, cfg['q']) for _ in uids])
        else:
            keep = brng.random((b, I)) >= cfg['q']
        return float(o.step(uids, keep, cfg['reg']))
    t0 = time.time()
    one(min(B, 512))
    t_cal = time.time() - t0
    b_ref = B
    while b_ref > 256 and t_cal * max(1.0, b_ref / 512 * 0.6) * (steps + warmup) > budget_s:
        b_ref //= 2
    n_steps = steps
    if t_cal * (steps + warmup) < 0.2 * budget_s:                     # tiny shapes: enough steps for ~10 s of CPU work
        n_steps = int(min(2000, max(steps, 10.0 / max(t_cal, 1e-4))))
    for _ in range(warmup):
        one(b_ref)
    t_sampler[0] = 0.0
    t0 = time.time()
    for _ in range(n_steps):
        loss = one(b_ref)
    dt = time.time() - t0
    return dict(samples_per_s=b_ref * n_steps / dt, batch=b_ref, seconds=dt, loss=loss, steps=n_steps,
                sampler_seconds=t_sampler[0])


def run_cdae_reference(args, cfg):
    ds, _ = make_data(cfg)
    r = cdae_cpu_arm(cfg, ds, max(1, args.steps), args.warmup, 150.0)
    sample = (f"{r['steps']} timed oracle steps of {r['batch']} sampled users on the full {cfg['title']} shape, oracle "
              f"sampler included ({r['sampler_seconds']:.2f} s of {r['seconds']:.1f} s); rank 0 only")
    config = cdae_config(cfg, 1, 'cpu, one process')
    config.update({'batch_per_gpu': None, 'global_batch': r['batch'],
                   'reference_arm': f"oracle port (numpy/BLAS) + oracle sampler, batch {r['batch']} per step on rank 0 "
                                    f"only, whatever --gpus says ({args.gpus}); no libdrb on this arm"})
    return {'impl': 'reference', 'metric': 'cdae_training_samples_per_sec', 'value': r['samples_per_s'],
            'unit': 'samples/s', 'n_gpus': args.gpus, 'steps': r['steps'], 'warmup': args.warmup,
            'ms_per_step': 1e3 * r['seconds'] / r['steps'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config,
            'cpu_baseline': {'value': r['samples_per_s'], 'unit': 'samples/s', 'cores': os.cpu_count(), 'kind': 'port',
                             'sample': sample},
            'e2e': {'value': r['samples_per_s'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'loss_last': r['loss']}


def run_cdae_native(args, cfg, D, arrays=None):
    import torch
    import drecpy_b200 as drb
    from drecpy_b200 import _lib
    from drecpy_b200.parallel import DataParallel
    rank, world, dev = D.rank, D.world, D.dev
    parity = dp_parity(D) if world > 1 and not args.no_dp_parity else None
    ds, t_data = make_data(cfg)
    B, K, W = cfg['batch'], args.steps, args.warmup
    m = drb.CDAE(hidden_factors=cfg['hidden'], corruption_level=cfg['q'], loss='bce', seed=cfg['seed'], verbose=False,
                 rng_mode=cfg['mask'], device=str(dev))
    m.fit(ds, epochs=0, batch_size=B, learning_rate=cfg['lr'], neg_ratio=cfg['neg_ratio'], reg_rate=cfg['reg'],
          sampler=drb.PointSampler(ds, cfg['neg_ratio'], 1e-3, cfg['seed'] + rank),
          data_parallel=DataParallel(D.dist), dp_sampler='independent', parallel_mode=args.parallel)
    items_mode = args.parallel == 'items' and world > 1
    Bs = B * world if items_mode else B          # item-sharded: every rank steps the whole global batch

    # ---- device-resident inputs for the `value` leg
    lib = _lib.load()
    batches = []
    pos_indptr = m._h_indptr                      # the (possibly item-sharded) CSR the model gathers from
    if items_mode:                                # all ranks must step the same users
        m._sampler = drb.PointSampler(ds, cfg['neg_ratio'], 1e-3, cfg['seed'])
    mt = cfg['mask'] == 'mt19937'
    n_batches = min(K + W, 64)
    for _ in range(n_batches):
        u = m._sampler.sample_arrays(Bs)[0]
        off = np.zeros(Bs + 1, np.int32)
        _lib.check(lib.drb_batch_offsets(_lib.np_ptr(u), Bs, _lib.np_ptr(pos_indptr), _lib.np_ptr(off)))
        keep_dev = None
        if mt:
            keep = np.zeros(max(int(off[-1]), 16), np.uint8)
            _lib.check(lib.drb_cdae_corruption_keep_mt(m._mask_rng.handle, _lib.np_ptr(u), Bs, cfg['n_items'],
                                                       float(cfg['q']), _lib.np_ptr(m._h_indptr),
                                                       _lib.np_ptr(m._h_indices), _lib.np_ptr(off), _lib.np_ptr(keep),
                                                       len(keep)))
            keep_dev = torch.from_numpy(keep).to(dev)
        batches.append((torch.from_numpy(u.copy()).to(dev), torch.from_numpy(off).to(dev), keep_dev))
    loss_dev = torch.zeros(2, device=dev)

    def step(s):
        bt = batches[s % n_batches]
        m.step_device(bt[0], bt[1], bt[2], cfg['reg'], loss_dev)
    flush = cfg['name'] != 'c3' and not args.no_flush
    launches0 = [0]

    def step_counted(s):
        if s == W:
            launches0[0] = m.launch_count()
        step(s)
    ms_total, clock_info = timed_steps(D, step_counted, W, K, flush_l2=flush)
    launches = m.launch_count() - launches0[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'loss': loss_dev, 'W': m.W, 'W_': m.W_, 'V': m.V, 'b': m.b, 'b_': m.b_})
    loss_value = m.global_loss(loss_dev)                        # collective when parallel: every rank calls it
    ms_warm = None
    if flush:                                                   # also the steady-state, L2-warm number
        ms_warm, _ = timed_steps(D, step, 3, K, flush_l2=False)

    # ---- e2e leg: the per-step body of fit(): host sampler -> pinned staging -> H2D -> step -> D2H loss
    for _ in range(3):
        m._step += 1
        m._train_step(B, cfg['reg'], want_loss=True, prefetch=True)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        m._step += 1
        loss_e2e = m._train_step(B, cfg['reg'], want_loss=True, prefetch=True)   # exactly what fit() runs per epoch
    torch.cuda.synchronize()
    t_e2e = D.max_over_ranks(time.perf_counter() - t0)
    h2d = 4 * B + 4 * (B + 1) + (int(batches[0][1][-1].item()) if mt else 0)

    # ---- roofline leg: per-kernel CUDA-event timing inside libdrb (separate pass; all ranks: the step has collectives)
    kernels = profile_kernels(m._ctx, step, 5)
    if rank != 0:
        return None
    peaks = load_peaks()
    n_params = int(m._L.total)                                   # parameters this rank updates (its shard when item-sharded)
    roofline = cdae_roofline(kernels, cfg, n_params, peaks, load_traffic(), D.world)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        r = cdae_cpu_arm(cfg, ds, 2, 1, 60.0)
        cpu = {'value': r['samples_per_s'], 'unit': 'samples/s', 'cores': os.cpu_count(), 'kind': 'port',
               'sample': f"{r['steps']} timed oracle steps of {r['batch']} sampled users on the full shape (numpy/BLAS "
                         f"on all cores + oracle sampler, {r['sampler_seconds']:.2f} s of {r['seconds']:.1f} s)"}
    value = B * world * K / (ms_total * 1e-3)
    line = base_line(cfg, 'cdae_training_samples_per_sec', 'samples/s', value, world, K, W, ms_total,
                     cdae_config(cfg, world, f'item-sharded x{world}' if items_mode else f'dp{world}', flush),
                     clock_info, launches, scaling='strong' if cfg.get('strong') else 'weak')
    line.update({'e2e': {'value': B * world * K / t_e2e, 'unit': 'samples/s', 'h2d_bytes_per_step': h2d,
                         'd2h_bytes_per_step': 4, 'ms_per_step': 1e3 * t_e2e / K},
                 'roofline': roofline, 'cpu_baseline': cpu, 'kernels_ms_per_step': kernels,
                 'loss_last': loss_value, 'loss_last_e2e': loss_e2e, 'data_gen_s': round(t_data, 1)})
    if ms_warm is not None:
        line['value_l2_warm'] = B * world * K / (ms_warm * 1e-3)
    if parity is not None:
        line['dp_parity'] = parity
    del m, batches
    torch.cuda.empty_cache()
    if world == 1 and not args.no_extras and cfg['name'] == 'c3':
        # the other legs of BASELINE.json's metric, measured after the headline with their own roofline / cpu_baseline
        # (each is a full bench line of its own workload; `python bench.py --workload X` prints the same line alone)
        extras = {}
        sub = argparse.Namespace(**vars(args))
        sub.warmup, sub.dump_outputs = max(args.warmup, 3), None
        for name in ('c2', 'c4_sampled', 'c4_full', 'c1'):
            try:
                extras[name] = RUNNERS[WORKLOADS[name]['model']][0](sub, dict(WORKLOADS[name]), D,
                                                                     arrays=(ds.user, ds.item, ds.interaction))
            except Exception as exc:          # never lose the headline line because of a secondary measurement
                extras[name] = {'error': repr(exc)}
        line['extras'] = extras
    return line


# ========================================================================================== DMF training (c2)
def dmf_config(cfg, n_gpus, flush):
    return {'workload': f"{cfg['title']}: DMF towers {cfg['towers']}/{cfg['towers']} cosine + normalised BCE on synthetic "
                        f"{cfg['n_users']}x{cfg['n_items']} / {cfg['nnz']} interactions ({cfg['origin']})",
            'batch_per_gpu': cfg['batch'], 'global_batch': cfg['batch'] * n_gpus, 'neg_ratio': cfg['neg_ratio'],
            'adam': 'dense, per-tower step counter', 'parallelism': f'dp{n_gpus}',
            'l2': 'L2 flushed between steps (256 MiB memset), every step timed on its own' if flush else
                  'working set (2.5 MB of weights) is L2 resident; back-to-back steps'}


def dmf_weights(cfg, seed=2):
    rng = np.random.default_rng(seed)

    def tower(in_dim):
        out = []
        for f in cfg['towers']:
            lim = np.sqrt(6.0 / (in_dim + f))
            out.append((rng.uniform(-lim, lim, (in_dim, f)).astype(np.float32), np.zeros(f, np.float32)))
            in_dim = f
        return out
    return {'user_nn': tower(cfg['n_items']), 'item_nn': tower(cfg['n_users'])}


def dmf_cpu_arm(cfg, ds, budget_s=12.0):
    from oracle.dmf import DMFOracle
    from oracle.sampler import PointSamplerOracleCSR
    w = dmf_weights(cfg)
    vals = ds.interaction
    mn = 0 if vals.min() == 1 else vals.min()
    o = DMFOracle(w['user_nn'], w['item_nn'], ds.csr(), ds.csc(), mn, vals.max(), learning_rate=cfg['lr'])
    so = PointSamplerOracleCSR(ds.uid, ds.iid, ds.interaction, cfg['neg_ratio'], 1e-3, cfg['seed'])
    B = cfg['batch']

    def one():
        t = so.sample(B)
        return float(o.step([x[0] for x in t], [x[1] for x in t], [o.standardize(x[2]) for x in t], cfg['reg']))
    one()
    t0, n = time.time(), 0
    while time.time() - t0 < budget_s:
        loss = one()
        n += 1
    dt = time.time() - t0
    return dict(samples_per_s=B * n / dt, steps=n, seconds=dt, loss=loss)


def run_dmf_reference(args, cfg):
    ds, _ = make_data(cfg)
    r = dmf_cpu_arm(cfg, ds, 20.0)
    return {'impl': 'reference', 'metric': 'dmf_training_samples_per_sec', 'value': r['samples_per_s'],
            'unit': 'samples/s', 'n_gpus': args.gpus, 'steps': r['steps'], 'warmup': 1,
            'ms_per_step': 1e3 * r['seconds'] / r['steps'], 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': dmf_config(cfg, 1, False),
            'cpu_baseline': {'value': r['samples_per_s'], 'unit': 'samples/s', 'cores': os.cpu_count(), 'kind': 'port',
                             'sample': f"{r['steps']} oracle steps of {cfg['batch']} pairs (numpy/BLAS + oracle sampler), "
                                       f"{r['seconds']:.1f} s, rank 0 only"},
            'e2e': {'value': r['samples_per_s'], 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}


def run_dmf_native(args, cfg, D, arrays=None):
    import torch
    import drecpy_b200 as drb
    from drecpy_b200.parallel import DataParallel
    ds, _ = make_data(cfg)
    B, K, W = cfg['batch'], args.steps, args.warmup
    kw = {}
    if D.world > 1:
        kw = dict(data_parallel=DataParallel(D.dist))
    m = drb.DMF(user_factors=list(cfg['towers']), item_factors=list(cfg['towers']), seed=cfg['seed'], verbose=False,
                device=str(D.dev))
    m.fit(ds, epochs=0, batch_size=B, learning_rate=cfg['lr'], neg_ratio=cfg['neg_ratio'], reg_rate=cfg['reg'],
          init_weights=dmf_weights(cfg), sampler=drb.PointSampler(ds, cfg['neg_ratio'], 1e-3, cfg['seed'] + D.rank),
          **kw)
    dev = D.dev
    nb = min(K + W, 128)
    batches = []
    for _ in range(nb):
        uu, ii, vv = m._sampler.sample_arrays(B)
        batches.append((torch.from_numpy(uu.copy()).to(dev), torch.from_numpy(ii.copy()).to(dev),
                        torch.from_numpy(m.labels_from_values(vv)).to(dev)))
    loss = torch.zeros(2, device=dev)

    def step(s):
        m.step_device(*batches[s % nb], cfg['reg'], loss)
    flush = not args.no_flush
    l0 = [0]

    def step_counted(s):
        if s == W:
            l0[0] = m.launch_count()
        step(s)
    ms_total, clock_info = timed_steps(D, step_counted, W, K, flush_l2=flush)
    launches = m.launch_count() - l0[0]
    if args.dump_outputs and D.rank == 0:
        out = {'loss': loss}
        for tower in ('user_nn', 'item_nn'):
            for j, (kernel, bias) in enumerate(m.tower_weights(tower)):
                out[f'{tower}_kernel_{j}'], out[f'{tower}_bias_{j}'] = kernel, bias
        dump_outputs(args.dump_outputs, out)
    ms_warm, _ = timed_steps(D, step, 3, K, flush_l2=False)
    # end to end through fit()'s step (host sampler -> H2D -> step -> D2H loss): median over chunks of 50 steps
    chunks = []
    for _ in range(3):
        m._step += 1
        m._train_step(B, cfg['reg'], want_loss=True, prefetch=True)
    for _ in range(5):
        t0 = time.perf_counter()
        for _ in range(50):
            m._step += 1
            m._train_step(B, cfg['reg'], want_loss=True, prefetch=True)
        chunks.append((time.perf_counter() - t0) / 50)
    t_e2e = D.max_over_ranks(float(np.median(chunks)))
    kernels = profile_kernels(m._ctx, step, 10)
    if D.rank != 0:
        return None
    peaks = load_peaks()
    # algorithmic bytes of the sparse first layers (SURVEY 8d): gather (4*64+4+4) B per stored entry of the sampled
    # users' rows and items' columns, scatter 8*64 B per entry
    csr, csc = ds.csr(), ds.csc()
    du, di = np.diff(csr[0]), np.diff(csc[0])
    nnz_batch = float(np.mean([du[b[0].cpu().numpy()].sum() + di[b[1].cpu().numpy()].sum() for b in batches[:16]]))
    w0 = cfg['towers'][0]
    g_ms = kernels.get('k_gather', 0.0)
    s_ms = kernels.get('k_scatter', 0.0)
    dom = 'k_scatter' if s_ms >= g_ms else 'k_gather'
    alg = (8.0 * w0 if dom == 'k_scatter' else (4.0 * w0 + 8)) * nnz_batch
    roofline = hbm_roofline(f'{dom} (both towers: 2 launches per step)', alg, kernels.get(dom, 0.0), peaks,
                            note=f'{nnz_batch:.0f} stored entries per batch; the tables (1.5 + 0.95 MB) are L2 resident '
                                 'and the step is launch / latency bound, so this fraction is reported, not aimed at')
    roofline['step_algorithmic_bytes'] = (12.0 * w0 + 8) * nnz_batch
    roofline['share_of_step'] = kernels.get(dom, 0.0) / max(sum(kernels.values()), 1e-9)
    cpu = None
    if not args.no_cpu_baseline:
        r = dmf_cpu_arm(cfg, ds)
        cpu = {'value': r['samples_per_s'], 'unit': 'samples/s', 'cores': os.cpu_count(), 'kind': 'port',
               'sample': f"{r['steps']} oracle steps of {B} pairs (numpy/BLAS + oracle sampler), {r['seconds']:.1f} s"}
    line = base_line(cfg, 'dmf_training_samples_per_sec', 'samples/s', B * D.world * K / (ms_total * 1e-3), D.world, K, W,
                     ms_total, dmf_config(cfg, D.world, flush), clock_info, launches)
    line.update({'value_l2_warm': B * D.world * K / (ms_warm * 1e-3),
                 'e2e': {'value': B * D.world / t_e2e, 'unit': 'samples/s', 'h2d_bytes_per_step': 12 * B,
                         'd2h_bytes_per_step': 4, 'ms_per_step': 1e3 * t_e2e},
                 'roofline': roofline, 'cpu_baseline': cpu, 'kernels_ms_per_step': kernels,
                 'launches_per_step': launches / K, 'loss_last': float(loss[0])})
    return line


# ========================================================================================== ranking (c4_sampled, c4_full)
def rank_setup(cfg, D, arrays):
    """configs[3]: the reference's leave-1-out split of the C3 data, a K=200 model fitted for a few steps."""
    import drecpy_b200 as drb
    if arrays is None:
        arrays = drb.synthetic_interactions(cfg['n_users'], cfg['n_items'], cfg['nnz'], seed=cfg['seed'],
                                            zipf_a=cfg['zipf_a'])
    t0 = time.perf_counter()
    train, test = drb.leave_k_out(drb.InteractionData(*arrays), k=1, min_user_interactions=0, seed=10,
                                  max_concurrent_threads=16, verbose=False)
    t_split = time.perf_counter() - t0
    train.assign_internal_ids()
    m = drb.CDAE(hidden_factors=cfg['hidden'], seed=cfg['seed'], verbose=False, rng_mode='philox', device=str(D.dev))
    sb = cfg.get('score_batch', 0)
    if sb < 0:      # the score filter runs CTA pairs over 256-user tiles: a block of (SMs / 2) tiles is one tile per pair
        import torch
        sb = (torch.cuda.get_device_properties(D.dev).multi_processor_count // 2) * 256
    m.fit(train, epochs=3, batch_size=4096, score_batch=sb)
    return train, test, m, t_split


def rank_config(cfg, n_gpus, what):
    return {'workload': f"{cfg['title']}: {what} for all users of the CDAE K={cfg['hidden']} model on synthetic "
                        f"{cfg['n_users']}x{cfg['n_items']} / {cfg['nnz']} interactions ({cfg['origin']})",
            'parallelism': f'users partitioned over {n_gpus} GPU(s), no collective',
            'l2': 'inputs per step (CSR rows, candidate / output lists, both weight tables: > 200 MB) exceed the 126 MB L2'}


def oracle_for(m, train):
    from oracle.cdae import CDAEOracle
    return CDAEOracle(m.W.cpu().numpy(), m.W_.cpu().numpy(), m.V.cpu().numpy(), m.b.cpu().numpy(), m.b_.cpu().numpy(),
                      train.csr(), interaction_threshold=1e-3)


def run_rank_sampled_native(args, cfg, D, arrays=None):
    import torch
    import drecpy_b200 as drb
    from drecpy_b200 import evaluation as ev
    train, test, m, t_split = rank_setup(cfg, D, arrays)
    kw = dict(k=cfg['k'], n_pos_interactions=1, n_neg_interactions=cfg['n_neg'], generate_negative_pairs=True,
              novelty=True, seed=10)
    # ---- device-resident leg: the candidate lists of this rank's users live in HBM; one step ranks all of them
    data = drb.InteractionData.from_dataset(test)
    users, t_indptr, t_order = ev._group_by_user(data)
    cand_off, cand, pos_off, pos, skipped, _, _ = ev.generate_candidates(
        m, data, users, np.ascontiguousarray(t_indptr), t_order, 1e-3, 1, cfg['n_neg'], True, False, 10)
    active = np.flatnonzero(skipped == 0)
    lo, hi = (len(active) * D.rank) // D.world, (len(active) * (D.rank + 1)) // D.world
    mine = active[lo:hi]
    C = cfg['n_neg'] + 1
    iids = train.items_to_iids(cand).astype(np.int32)
    padded = np.stack([iids[cand_off[u]:cand_off[u] + C] for u in mine]) if len(mine) else np.zeros((0, C), np.int32)
    uids = train.users_to_uids(users[mine]).astype(np.int32)
    d_u = torch.as_tensor(uids, device=D.dev)
    d_c = torch.as_tensor(np.ascontiguousarray(padded), device=D.dev)
    d_n = torch.full((len(mine),), C, dtype=torch.int32, device=D.dev)
    out = m.rank_candidates_device(d_u, d_c, d_n, True)
    K, W = args.steps, max(3, args.warmup)
    l0 = [0]

    def step(s):
        if s == W:
            l0[0] = m.launch_count()
        m.rank_candidates_device(d_u, d_c, d_n, True, out=out)
    ms_total, clock_info = timed_steps(D, step, W, K)
    launches = m.launch_count() - l0[0]
    if args.dump_outputs and D.rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(('iids', 'scores', 'n_out'), out)))
    n_users_total = int(D.sum_over_ranks(len(mine)))
    kernels = profile_kernels(m._ctx, step, 2)
    # ---- e2e leg: the public call (host candidate generation, H2D, rank, D2H of the ranked lists, metrics); N=1 only
    e2e_t, res = [], None
    if D.world == 1:
        for _ in range(3):
            t0 = time.perf_counter()
            res = drb.ranking_evaluation(m, test, metrics=[drb.HitRatio(), drb.NDCG()], verbose=False, **kw)
            e2e_t.append(time.perf_counter() - t0)
    if D.rank != 0:
        return None
    peaks = load_peaks()
    Kh = cfg['hidden']
    deg = np.diff(train.csr(1e-3)[0])[uids].astype(np.float64)
    alg_gather = float((4.0 * Kh + 4) * deg.sum() + 4.0 * Kh * len(uids))
    alg_rank = float(len(uids)) * C * (4.0 * Kh + 12)
    g_ms, r_ms = kernels.get('k_gather', 0.0), kernels.get('k_rank_candidates', 0.0)
    dom = ('k_rank_candidates', alg_rank, r_ms) if r_ms >= g_ms else ('k_gather', alg_gather, g_ms)
    n_launch = max(1, -(-len(uids) // m._max_batch))
    roofline = hbm_roofline(f'{dom[0]} ({n_launch} launches per step, summed)', dom[1], dom[2], peaks,
                            note='sampled-candidate scoring: h gather (4K per stored positive) + 101 candidate rows of '
                                 "W'^T per user (SURVEY 8d: ~196 KB/user); W and W' (21 MB each) are L2 resident")
    roofline['step_algorithmic_bytes'] = alg_gather + alg_rank
    roofline['step_achieved_gbs'] = (alg_gather + alg_rank) * D.world / (ms_total / K * 1e-3) / 1e9
    cpu = None
    if D.world == 1 and not args.no_cpu_baseline:
        cpu = rank_sampled_cpu_arm(cfg, m, train, test, kw)
    line = base_line(cfg, 'sampled_ranking_users_per_sec', 'users/s', n_users_total * K / (ms_total * 1e-3), D.world, K,
                     W, ms_total, rank_config(cfg, D.world, f'leave-1-out ranking_evaluation, 1 positive + {cfg["n_neg"]} '
                                                               f'generated negatives, HitRatio/NDCG@{cfg["k"]}'),
                     clock_info, launches)
    line.update({'roofline': roofline, 'cpu_baseline': cpu, 'kernels_ms_per_step': kernels, 'users': n_users_total,
                 'leave_k_out_s': t_split})
    if e2e_t:
        t = float(np.median(e2e_t))
        line['e2e'] = {'value': len(active) / t, 'unit': 'users/s', 'seconds': t, 'repeats': len(e2e_t),
                       'h2d_bytes_per_step': int(len(active) * (C * 4 + 8)), 'd2h_bytes_per_step': int(len(active) * (C * 8 + 4)),
                       'what': 'drecpy_b200.ranking_evaluation(model, test, ...) wall time, median of 3: native '
                               'candidate generation on the host, H2D, rank, D2H of the ranked lists, metrics'}
        line['metrics'] = res
    return line


def rank_sampled_cpu_arm(cfg, m, train, test, kw, n_users=1500):
    """Oracle protocol (per-user Random(seed+idx) candidates, oracle scoring, heapq order, metrics) on the first
    n_users test users."""
    import heapq
    from oracle.cdae import sigmoid
    from oracle.ranking import ranking_evaluation_oracle
    o = oracle_for(m, train)
    seen, pos = train.csr(), train.csr(1e-3)
    raw = train.raw_items
    tu = test.user.tolist()
    order, s = [], set()
    for x in tu:
        if x not in s:
            s.add(x)
            order.append(x)
        if len(order) == n_users:
            break
    train_pos = {}
    for usr in order:
        uid = train.user_to_uid(usr)
        if uid is not None:
            train_pos[usr] = set(raw[pos[1][pos[0][uid]:pos[0][uid + 1]]].tolist())

    def rank_fn(user, items, novelty):
        uid = train.user_to_uid(user)
        p = o.predict(uid)                                           # cdae.py:84-88: all I outputs, as the reference does
        cand = set(x for x in (train.item_to_iid(it) for it in items) if x is not None)
        if novelty:
            cand -= set(seen[1][seen[0][uid]:seen[0][uid + 1]].tolist())
        return [train.iid_to_item(i) for _, i in heapq.nlargest(len(cand), [(p[i], i) for i in cand])]
    t0 = time.time()
    res = ranking_evaluation_oracle(rank_fn, tu, test.item.tolist(), test.interaction.tolist(), train_pos, m.n_items,
                                    1e-3, n_test_users=n_users, metrics=('HitRatio', 'NDCG'), **kw)
    dt = time.time() - t0
    return {'value': n_users / dt, 'unit': 'users/s', 'cores': os.cpu_count(), 'kind': 'port',
            'sample': f'oracle protocol + oracle scoring for the first {n_users} test users, {dt:.1f} s', 'metrics': res}


def run_topk_native(args, cfg, D, arrays=None):
    import torch
    train, test, m, _ = rank_setup(cfg, D, arrays)
    k = cfg['k']
    lo, hi = (m.n_users * D.rank) // D.world, (m.n_users * (D.rank + 1)) // D.world
    uids = torch.arange(lo, hi, dtype=torch.int32, device=D.dev)
    K, W = args.steps, max(3, args.warmup)
    l0 = [0]
    last = [None]

    def step(s):
        if s == W:
            l0[0] = m.launch_count()
        last[0] = m.topk_batch(uids, k, novelty=True, return_device=True)
    ms_total, clock_info = timed_steps(D, step, W, K)
    launches = m.launch_count() - l0[0]
    if args.dump_outputs and D.rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(('iids', 'scores', 'n_out'), last[0])))
    kernels = profile_kernels(m._ctx, step, 2)
    # ---- e2e: host uids -> H2D -> top-k -> D2H of the ranked lists (iids, scores, counts)
    h_u = np.arange(lo, hi, dtype=np.int32)
    m.topk_batch(h_u, k, novelty=True)
    D.barrier()
    ts = []
    for _ in range(3):
        t0 = time.perf_counter()
        oi, os_, on = m.topk_batch(h_u, k, novelty=True)
        ts.append(time.perf_counter() - t0)
    t_e2e = D.max_over_ranks(float(np.median(ts)))
    if D.rank != 0:
        return None
    peaks = load_peaks()
    n = hi - lo
    flops = 2.0 * cfg['hidden'] * cfg['n_items'] * n
    gemm = {kk: v for kk, v in kernels.items() if kk.startswith('k_umma') or kk.startswith('k_sgemm')}
    dom_ms = sum(gemm.values()) if gemm else sum(kernels.values())
    ach = flops / (dom_ms * 1e-3) / 1e12 if dom_ms else None
    traffic = load_traffic()
    roofline = {'kernel': ' + '.join(sorted(gemm)) or 'all', 'bound': 'tensor', 'achieved': ach, 'peak': peaks['tf'],
                'unit': 'TFLOP/s', 'frac': ach / peaks['tf'] if ach else None,
                'traffic': sum(traffic.get(kk, 0) for kk in gemm) or None,
                'algorithmic_flops_per_step': flops, 'ms_per_step_family': dom_ms,
                'peak_source': f"{peaks['src']} bf16 sustained",
                'share_of_step': dom_ms / max(sum(kernels.values()), 1e-9),
                'note': "2*K*I flops per user (h W'^T over the whole catalog), fp32-accurate split products; the fused "
                        'epilogue keeps the top-k on chip'}
    cpu = None
    if D.world == 1 and not args.no_cpu_baseline:
        o = oracle_for(m, train)
        t0, nu = time.time(), 0
        while time.time() - t0 < 10.0:
            o.rank(nu * 97 % m.n_users, range(m.n_items), k, True)     # full forward + heapq.nlargest, as cdae.py:90-103
            nu += 1
        dt = time.time() - t0
        cpu = {'value': nu / dt, 'unit': 'users/s', 'cores': os.cpu_count(), 'kind': 'port',
               'sample': f'oracle _rank over range(n_items) + heapq.nlargest({k}) for {nu} users, {dt:.1f} s'}
    total = m.n_users
    line = base_line(cfg, 'full_catalog_ranked_users_per_sec', 'users/s', total * K / (ms_total * 1e-3), D.world, K, W,
                     ms_total, rank_config(cfg, D.world, f'full-catalog top-{k} with novelty filter'), clock_info, launches)
    line.update({'e2e': {'value': total / t_e2e, 'unit': 'users/s', 'seconds': t_e2e, 'h2d_bytes_per_step': 4 * n,
                         'd2h_bytes_per_step': n * (8 * k + 4)},
                 'roofline': roofline, 'cpu_baseline': cpu, 'kernels_ms_per_step': kernels, 'users': total,
                 'n_out_min': int(on.min())})
    return line


def run_rank_reference(args, cfg):
    """CPU arm of the c4 workloads: needs a fitted model; the oracle is trained for 3 oracle steps of 512 users (the
    throughput of scoring does not depend on the weights)."""
    import drecpy_b200 as drb
    from oracle.cdae import CDAEOracle
    arrays = drb.synthetic_interactions(cfg['n_users'], cfg['n_items'], cfg['nnz'], seed=cfg['seed'], zipf_a=cfg['zipf_a'])
    ds = drb.InteractionData(*arrays)
    ds.assign_internal_ids()
    rng = np.random.default_rng(1)
    U, I, K = cfg['n_users'], cfg['n_items'], cfg['hidden']

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo))
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    o = CDAEOracle(glorot((I, K), I, K), glorot((K, I), K, I), glorot((U, K), U, K), glorot((K,), K, K),
                   glorot((I,), I, I), ds.csr(), interaction_threshold=1e-3)
    k = cfg['k']
    C = cfg.get('n_neg', 0) + 1
    t0, nu = time.time(), 0
    brng = np.random.default_rng(0)
    while time.time() - t0 < 20.0:
        uid = nu * 97 % U
        cand = range(I) if cfg['model'] == 'topk' else brng.integers(0, I, C).tolist()
        o.rank(uid, cand, k if cfg['model'] == 'topk' else C, True)
        nu += 1
    dt = time.time() - t0
    metric = 'full_catalog_ranked_users_per_sec' if cfg['model'] == 'topk' else 'sampled_ranking_users_per_sec'
    what = f'full-catalog top-{k}' if cfg['model'] == 'topk' else f'{C} sampled candidates'
    return {'impl': 'reference', 'metric': metric, 'value': nu / dt, 'unit': 'users/s', 'n_gpus': args.gpus, 'steps': nu,
            'warmup': 0, 'ms_per_step': 1e3 * dt / nu, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': rank_config(cfg, 1, what),
            'cpu_baseline': {'value': nu / dt, 'unit': 'users/s', 'cores': os.cpu_count(), 'kind': 'port',
                             'sample': f'oracle _rank ({what}) for {nu} users, {dt:.1f} s, rank 0 only'},
            'e2e': {'value': nu / dt, 'unit': 'users/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}


# ========================================================================================== configs[4]: item-sharded CDAE
def run_c5_native(args, cfg, D, arrays=None):
    """CDAE K=256 on 10 M users x 1 M items / 1 B interactions, W / W' / b' sharded by item range and V by user range over
    the ranks, sampled outputs (positives + neg_total drawn items per sampled user; the dense output layer of cdae.py:76
    would cost 6.3 PFLOP per 4096-user step here).  Every rank generates only its own columns, on its GPU.  Per step the
    ranks exchange two all-reduces of batch x hidden activations (partial pre-activation, partial dh): rows of the tables
    never travel.  --c5-scale shrinks users / items / interactions by that factor for a quick run."""
    import torch
    import drecpy_b200 as drb
    from drecpy_b200 import _lib
    from drecpy_b200.parallel import DataParallel
    sc = args.c5_scale
    U, I, nnz = int(cfg['n_users'] * sc), int(cfg['n_items'] * sc), int(cfg['nnz'] * sc)
    world, rank, dev = D.world, D.rank, D.dev
    B, K, W = cfg['batch'], args.steps, args.warmup
    Bg = B * world
    neg_per_group = max(1, cfg['neg_total'] // world)      # one negative-sampling group per rank (= per item shard)
    torch.cuda.reset_peak_memory_stats(dev)
    t0 = time.time()
    indptr, indices = drb.synthetic_item_shard(U, I, nnz, rank, world, seed=cfg['seed'], zipf_a=cfg['zipf_a'], device=str(dev))
    t_data = time.time() - t0
    nnz_local = int(indices.shape[0])
    m = drb.CDAE(hidden_factors=cfg['hidden'], corruption_level=cfg['q'], loss='bce', seed=cfg['seed'], verbose=False,
                 rng_mode='philox', device=str(dev), output='sampled', neg_per_group=neg_per_group)
    m.fit_item_shard((indptr, indices), U, I, B, DataParallel(D.dist), learning_rate=cfg['lr'], reg_rate=cfg['reg'])
    lib = _lib.load()
    if world == 1:
        Bg = B
    batches = []
    nb = min(K + W, 16)
    for _ in range(nb):
        u = m._sampler.sample_arrays(Bg)[0].copy()
        off = np.zeros(Bg + 1, np.int32)
        _lib.check(lib.drb_batch_offsets(_lib.np_ptr(u), Bg, _lib.np_ptr(m._h_indptr), _lib.np_ptr(off)))
        batches.append((torch.from_numpy(u).to(dev), torch.from_numpy(off).to(dev)))
    loss_dev = torch.zeros(2, device=dev)

    def step(s):
        bt = batches[s % nb]
        m.step_device(bt[0], bt[1], None, cfg['reg'], loss_dev)
    l0 = [0]

    def step_counted(s):
        if s == W:
            l0[0] = m.launch_count()
        step(s)
    ms_total, clock_info = timed_steps(D, step_counted, W, K)
    launches = m.launch_count() - l0[0]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {'loss': loss_dev, 'W': m.W, 'W_': m.W_, 'V': m.V, 'b': m.b, 'b_': m.b_})
    loss_value = m.global_loss(loss_dev)
    # e2e: host sampler -> pinned staging -> H2D -> step -> D2H loss, exactly fit()'s per-step body
    for _ in range(2):
        m._step += 1
        m._train_step(B, cfg['reg'], want_loss=True, prefetch=True)
    D.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        m._step += 1
        loss_e2e = m._train_step(B, cfg['reg'], want_loss=True, prefetch=True)
    torch.cuda.synchronize()
    t_e2e = D.max_over_ranks(time.perf_counter() - t0)
    kernels = profile_kernels(m._ctx, step, 3)
    mem_gb = D.max_over_ranks(torch.cuda.max_memory_allocated(dev) / 2 ** 30)
    nnz_total = int(D.sum_over_ranks(nnz_local))
    if rank != 0:
        return None
    peaks = load_peaks()
    ld = int(m._L.ld)
    deg_loc = float(np.mean([float(b[1][-1].item()) for b in batches[:4]])) / Bg       # local positives per sampled user
    n_params = int(m._L.total)
    adam_ms, so_ms = kernels.get('k_adam', 0.0), kernels.get('k_sampled_out', 0.0)
    alg_so = 8.0 * ld * (deg_loc + neg_per_group) * Bg
    if adam_ms >= so_ms:
        roofline = hbm_roofline('k_adam (dense Adam + L2 over this rank\'s shard: V rows dominate)', 28.0 * n_params, adam_ms, peaks,
                                note='reference semantics: every row of V, W, W\' is updated every step (recommender_abc.py:328-334)')
    else:
        roofline = hbm_roofline('k_sampled_out', alg_so, so_ms, peaks)
    roofline['secondary'] = {'k_sampled_out': {'bound': 'hbm', 'achieved': alg_so / (so_ms * 1e-3) / 1e9 if so_ms else None,
                                               'peak': peaks['hbm'], 'unit': 'GB/s', 'algorithmic_bytes': alg_so,
                                               'note': '8*K bytes per scored (user, item): W\' row in, gradient row out (atomics)'},
                             'k_adam': {'bound': 'hbm', 'achieved': 28.0 * n_params / (adam_ms * 1e-3) / 1e9 if adam_ms else None,
                                        'peak': peaks['hbm'], 'unit': 'GB/s'}}
    roofline['share_of_step'] = max(adam_ms, so_ms) / max(sum(kernels.values()), 1e-9)
    config = {'workload': f"{cfg['title']}: CDAE hidden_factors={cfg['hidden']} bce q={cfg['q']}, sampled outputs (positives + "
                          f"{neg_per_group * world} drawn items per sampled user; extension, see DESIGN.md), synthetic {U}x{I} / "
                          f"{nnz_total} interactions ({cfg['origin']}{'' if sc == 1.0 else f', scaled by {sc}'})",
              'batch_per_gpu': B, 'global_batch': Bg, 'parallelism': f'item-sharded x{world} (W, W\', b\' by item range, V by user range)',
              'mask_rng': 'philox (device)', 'adam': 'dense, per-variable step counter',
              'bytes_exchanged_per_step_per_rank': 2 * Bg * ld * 4,
              'exchange': 'two all-reduces of global_batch x hidden fp32 activations (partial pre-activation, partial dh); rows of W / W\' / V never travel',
              'memory_per_rank_gb': round(mem_gb, 2), 'interactions_per_rank': nnz_local,
              'l2': 'per-step working set (this rank\'s tables + Adam state: tens of GB) far exceeds the 126 MB L2'}
    line = base_line(cfg, 'cdae_training_samples_per_sec', 'samples/s', Bg * K / (ms_total * 1e-3), world, K, W, ms_total,
                     config, clock_info, launches)
    line.update({'e2e': {'value': Bg * K / t_e2e, 'unit': 'samples/s', 'h2d_bytes_per_step': 8 * Bg + 4, 'd2h_bytes_per_step': 4,
                         'ms_per_step': 1e3 * t_e2e / K},
                 'roofline': roofline, 'cpu_baseline': None, 'kernels_ms_per_step': kernels, 'loss_last': loss_value,
                 'loss_last_e2e': loss_e2e, 'data_gen_s': round(t_data, 1)})
    return line


def run_c5_reference(args, cfg):
    """CPU arm of configs[4]: the sampled-output oracle on a shape scaled down until its dense intermediates fit (the
    oracle, like the reference, densifies the sampled users' rows: 4096 x 1 M floats at full size)."""
    import random
    import drecpy_b200 as drb
    from oracle.cdae import CDAESampledOracle
    sc = 0.02
    U, I, nnz, K, B = int(cfg['n_users'] * sc), int(cfg['n_items'] * sc), int(cfg['nnz'] * sc), cfg['hidden'], 512
    u, i, v = drb.synthetic_interactions(U, I, nnz, seed=cfg['seed'], zipf_a=cfg['zipf_a'])
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    rng = np.random.default_rng(1)
    U, I = ds.count_unique('uid'), ds.count_unique('iid')

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo))
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    o = CDAESampledOracle(glorot((I, K), I, K), glorot((K, I), K, I), glorot((U, K), U, K), glorot((K,), K, K),
                          glorot((I,), I, I), ds.csr(), interaction_threshold=1e-3, corruption_level=cfg['q'],
                          learning_rate=cfg['lr'], n_groups=8, neg_per_group=cfg['neg_total'] // 8, seed=cfg['seed'])
    brng = np.random.default_rng(0)
    t0, n = time.time(), 0
    while time.time() - t0 < 25.0 and n < max(1, args.steps):
        uids = brng.integers(0, U, B)
        keep = brng.random((B, I)) >= cfg['q']
        loss = float(o.step_sampled(uids, keep, cfg['reg'], n + 1))
        n += 1
    dt = time.time() - t0
    config = {'workload': f"{cfg['title']} scaled by {sc} ({U}x{I} / {len(u)} interactions), batch {B}: CPU arm of {cfg['origin']}",
              'parallelism': 'cpu, one process', 'global_batch': B}
    return {'impl': 'reference', 'metric': 'cdae_training_samples_per_sec', 'value': B * n / dt, 'unit': 'samples/s',
            'n_gpus': args.gpus, 'steps': n, 'warmup': 0, 'ms_per_step': 1e3 * dt / n, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': config,
            'cpu_baseline': {'value': B * n / dt, 'unit': 'samples/s', 'cores': os.cpu_count(), 'kind': 'port',
                             'sample': f'{n} sampled-output oracle steps of {B} users on the scaled-down shape, {dt:.1f} s, rank 0 only'},
            'e2e': {'value': B * n / dt, 'unit': 'samples/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'loss_last': loss}


RUNNERS = {'cdae_sharded': (run_c5_native, run_c5_reference), 'cdae': (run_cdae_native, run_cdae_reference), 'dmf': (run_dmf_native, run_dmf_reference),
           'rank_sampled': (run_rank_sampled_native, run_rank_reference), 'topk': (run_topk_native, run_rank_reference)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='native', choices=['native', 'reference'])
    ap.add_argument('--workload', default='c3', choices=sorted(WORKLOADS))
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-extras', action='store_true')
    ap.add_argument('--no-flush', action='store_true', help='c1 / c2: back-to-back steps instead of an L2 flush per step')
    ap.add_argument('--no-dp-parity', action='store_true')
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'],
                    help='c3, N>1: weak = 4096 users per GPU (default, the driver\'s curve); strong = 4096 users globally')
    ap.add_argument('--mask', default=None, choices=['philox', 'mt19937', 'mt19937_device'],
                    help='CDAE workloads: corruption-mask generator (default: philox at c3, the host MT19937 replay at c1)')
    ap.add_argument('--c5-scale', type=float, default=1.0, help='c5: shrink users / items / interactions by this factor')
    ap.add_argument('--parallel', default='data', choices=['data', 'items'],
                    help='N>1: data = replicated weights + gradient all-reduce; items = item-sharded weights')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last one computed (rank 0) as DIR/<name>.npy, '
                         'float32 / float64, at most 64 MB in all (larger outputs as a fixed sample of their rows)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the native path; the reference arm has none')
    cfg = dict(WORKLOADS[args.workload])
    if args.mask and 'mask' in cfg:
        cfg['mask'] = args.mask
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.scaling == 'strong' and cfg['model'] == 'cdae' and world > 1:
        assert cfg['batch'] % world == 0
        cfg['batch'] //= world                        # the global batch stays what BASELINE.json names
        cfg['strong'] = True
    native, reference = RUNNERS[cfg['model']]
    if args.impl == 'reference':
        if int(os.environ.get('RANK', '0')) == 0:
            print(json.dumps(reference(args, cfg)), flush=True)
        return
    D = Dist()
    line = native(args, cfg, D)
    if D.rank == 0 and line is not None:
        print(json.dumps(line), flush=True)
    D.finish()


if __name__ == '__main__':
    main()
