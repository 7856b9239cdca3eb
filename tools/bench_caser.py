#!/usr/bin/env python
"""Caser on one GPU at the ml-1m shape (6040 x 3706, 1 M rows, 512 windows per step) and the ml-20m shape
(138,493 x 26,744, 20 M rows, 4096 windows per step), default sizes (L=5, T=3, d=50, n_v=4, n_h=16, neg_ratio=5),
synthetic interactions and timestamps from a seed.  Prints one JSON line: per shape the step time (CUDA events over
--steps graph-replayed steps after --warmup), windows/s, the update kernel's share of the step with its algorithmic
bytes (params, m, v, grads read, params, m, v written: 28 bytes per parameter) from a profiled pass of its own, and
full-catalog top-100 users/s; and the card name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = {'ml-1m': (6040, 3706, 1_000_209, 512), 'ml-20m': (138_493, 26_744, 20_000_263, 4096)}


def card():
    import torch
    out = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        out['power_limit'], out['max_sm_clock'] = [x.strip() for x in q.split(',')]
    except Exception as e:        # the card name is still reported
        out['power_limit'] = f'unavailable ({e.__class__.__name__})'
    return out


def run_shape(name, steps, warmup, topk_users):
    import torch
    import drecpy_b200 as drb
    from drecpy_b200 import _lib
    U, I, nnz, B = SHAPES[name]
    u, i, v = drb.synthetic_interactions(U, I, nnz, seed=10)
    ts = np.random.default_rng(11).integers(0, 10 ** 9, len(u))
    m = drb.Caser(seed=10, verbose=False)
    t0 = time.time()
    m.fit(drb.InteractionData(u, i, v, timestamp=ts), epochs=0, batch_size=B, neg_ratio=5)
    setup_s = time.time() - t0
    for s in range(1, warmup + 1):
        m._step = s
        m._train_step(B, 1e-3)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for s in range(warmup + 1, warmup + steps + 1):
        m._step = s
        m._train_step(B, 1e-3)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / steps
    loss = m._train_step(B, 1e-3, want_loss=True)
    # profiled pass (direct launches, events around every kernel): the update kernel's share of the step
    lib = _lib.load()
    _lib.check(lib.drb_ctx_profile_enable(m._ctx, 1))
    for s in range(20):
        m._step += 1
        m._train_step(B, 1e-3)
    prof = _lib.profile_read(m._ctx)
    _lib.check(lib.drb_ctx_profile_enable(m._ctx, 0))
    total = sum(ms for ms, _ in prof.values())
    upd = sum(ms for k, (ms, _) in prof.items() if k.startswith('k_adam') or k.startswith('k_optim'))
    n_params = int(m._params.numel())
    upd_ms = upd / 20
    users = np.arange(min(U, topk_users), dtype=np.int32)
    m.topk_batch(users[:min(len(users), 1024)], 100)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.topk_batch(users, 100)
    torch.cuda.synchronize()
    topk_s = time.perf_counter() - t0
    return {'shape': name, 'users': U, 'items': I, 'rows': len(u), 'batch': B, 'setup_s': round(setup_s, 2),
            'step_ms': round(step_ms, 4), 'windows_per_s': round(B / step_ms * 1e3), 'loss': loss,
            'params': n_params, 'update_ms': round(upd_ms, 4), 'update_share_of_profiled_step': round(upd / total, 3),
            'update_bytes': 28 * n_params, 'update_GBps': round(28 * n_params / (upd_ms * 1e-3) / 1e9, 1),
            'profiled_kernels_ms': {k: round(ms / c, 4) for k, (ms, c) in prof.items()},
            'top100_users_per_s': round(len(users) / topk_s), 'top100_users': len(users)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=200)
    ap.add_argument('--warmup', type=int, default=20)
    ap.add_argument('--shapes', default='ml-1m,ml-20m')
    ap.add_argument('--topk-users', type=int, default=32768)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_caser: no CUDA device (the measurement needs a B200)')
    res = {'card': card(), 'results': [run_shape(s, a.steps, a.warmup, a.topk_users) for s in a.shapes.split(',')]}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
