#!/usr/bin/env python
"""DMF full-catalog top-k (drb_dmf_topk): ranked users/s, one JSON line per shape.

  python tools/bench_dmf_topk.py [--steps K] [--warmup W] [--shapes c2,ml20m]

value            users/s of drb_dmf_topk over every user, k = 100, novelty on, uids and outputs resident on the device,
                 CUDA events around K back-to-back calls after W warm-up calls
e2e              users/s of recommend_batch(all raw user ids, n=100): host ids in, host arrays out
previous_route   users/s of m._rank(uid, range(n_items), 100, True) -- what recommend() ran before drb_dmf_topk --
                 on a fixed sample of 200 users
kernels_ms_per_step, roofline, cpu_baseline (DMFOracle forward over the catalog + heapq.nlargest, bounded), gpu,
bitwise_equal_rank_path (drb_dmf_topk rows == drb_dmf_rank_candidates over the catalog, ids and score bits, on a sample
of users at the timed shape, checked in the same run).
The c2 shape (6040 x 3706) is launch-size work: one block of users, a few microseconds per kernel.
"""
import argparse
import heapq
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

K_TOP = 100
SHAPES = {
    'c2': dict(bench.C2, title='dmf_ml1m_shape_full_catalog_top100', score_batch=8192,
               note='launch-size work: one block of 6040 users, the whole catalog per call is 22 M scores'),
    'ml20m': dict(bench.C2, name='ml20m', title='dmf_ml20m_shape_full_catalog_top100', origin='ml-20m shape',
                  n_users=138493, n_items=26744, nnz=20_000_000, zipf_a=1.0, score_batch=32768, note=None),
}


def gpu_info():
    """name, power limit (W), max SM clock (MHz) of device 0, read only."""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader,nounits',
                              '-i', '0'], capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        return {'name': out[0].strip(), 'power_limit_w': float(out[1]), 'max_sm_mhz': float(out[2])}
    except Exception as e:
        return {'name': None, 'power_limit_w': None, 'max_sm_mhz': None, 'error': str(e)}


def cpu_arm(cfg, ds, m, budget_s):
    """DMFOracle forward over the catalog in item chunks + heapq.nlargest, for as long as the budget allows; users/s
    from the item-scores/s rate (a user = n_items scores)."""
    from oracle.dmf import DMFOracle
    w = bench.dmf_weights(cfg)
    o = DMFOracle(w['user_nn'], w['item_nn'], ds.csr(), ds.csc(), m.min_interaction, m.max_interaction)
    I, chunk = m.n_items, 256
    rng = np.random.default_rng(1)
    t0, scored, done = time.time(), 0, 0
    while time.time() - t0 < budget_s:
        uid = int(rng.integers(0, m.n_users))
        p = np.empty(I, np.float32)
        for c in range(0, I, chunk):
            ids = np.arange(c, min(I, c + chunk))
            p[ids] = o.forward(np.full(len(ids), uid), ids)[0]
            scored += len(ids)
            if time.time() - t0 > budget_s:
                break
        else:
            seen = set(ds.user_items(uid).tolist())
            heapq.nlargest(K_TOP, ((float(p[i]), i) for i in range(I) if i not in seen))
            done += 1
    dt = time.time() - t0
    return {'value': scored / I / dt, 'unit': 'users/s', 'cores': os.cpu_count(), 'kind': 'port',
            'sample': f'{scored} item scores ({done} users completed) in {dt:.1f} s, numpy/BLAS oracle, chunks of {chunk} items'}


def run(cfg, args, D):
    import torch
    import drecpy_b200 as drb
    from drecpy_b200 import _lib
    lib = _lib.load()
    ds, _ = bench.make_data(cfg)
    m = drb.DMF(user_factors=cfg['towers'], item_factors=cfg['towers'], seed=10, verbose=False)
    m.fit(ds, epochs=0, batch_size=cfg['batch'], init_weights=bench.dmf_weights(cfg), score_batch=cfg['score_batch'])
    U, I, w = m.n_users, m.n_items, cfg['towers'][-1]
    d_u = torch.arange(U, dtype=torch.int32, device=D.dev)
    nb = lib.drb_dmf_topk_scratch_bytes(m._native, K_TOP)
    scratch = torch.empty(nb, dtype=torch.uint8, device=D.dev)
    o_i = torch.empty((U, K_TOP), dtype=torch.int32, device=D.dev)
    o_s = torch.empty((U, K_TOP), dtype=torch.float32, device=D.dev)
    o_n = torch.empty(U, dtype=torch.int32, device=D.dev)

    def step(s):
        _lib.check(lib.drb_dmf_topk(m._native, _lib.t_ptr(d_u), U, K_TOP, 1, _lib.t_ptr(scratch), nb, _lib.t_ptr(o_i),
                                    _lib.t_ptr(o_s), _lib.t_ptr(o_n)))

    l0 = m.launch_count()
    step(0)
    launches = m.launch_count() - l0
    ms, clocks = bench.timed_steps(D, step, args.warmup, args.steps)
    ms_step = ms / args.steps
    flagged = int((o_n < 0).sum())

    # the same answer as the rank path, ids and score bits, on a sample of users
    rng = np.random.default_rng(0)
    sample = np.sort(rng.choice(U, 256, replace=False)).astype(np.int32)
    d_s = torch.as_tensor(sample, device=D.dev)
    cat = torch.arange(I, dtype=torch.int32, device=D.dev)
    ri, rs, rn = m._rank_device(d_s, cat.expand(len(sample), -1).contiguous(),
                                torch.full((len(sample),), I, dtype=torch.int32, device=D.dev), True)
    gi, gs, gn = o_i[d_s.long()], o_s[d_s.long()], o_n[d_s.long()]
    valid = torch.arange(K_TOP, device=D.dev)[None, :] < gn[:, None].long()
    bitwise = bool(torch.equal(gn, torch.clamp(rn, max=K_TOP)) and
                   torch.equal(torch.where(valid, gi, -1), torch.where(valid, ri[:, :K_TOP], -1)) and
                   torch.equal(torch.where(valid, gs.view(torch.int32), 0), torch.where(valid, rs[:, :K_TOP].contiguous().view(torch.int32), 0)))

    kernels = bench.profile_kernels(m._ctx, step, 2)
    # previous route: recommend() before drb_dmf_topk = _rank over the catalog, one user per call
    prev_users = sample[:200]
    m._rank(int(prev_users[0]), range(I), K_TOP, True)
    torch.cuda.synchronize()
    t0 = time.time()
    for uid in prev_users:
        m._rank(int(uid), range(I), K_TOP, True)
    prev = len(prev_users) / (time.time() - t0)
    # end to end: raw ids in, host arrays out
    users = ds.raw_users
    m.recommend_batch(users[:1024], n=K_TOP)
    t0 = time.time()
    items, scores, counts = m.recommend_batch(users, n=K_TOP)
    e2e_s = time.time() - t0

    gpu = gpu_info()
    sms = torch.cuda.get_device_properties(D.dev).multi_processor_count
    flops = 2.0 * w * U * I
    ffma_peak = sms * 128 * 2 * gpu['max_sm_mhz'] * 1e6 if gpu['max_sm_mhz'] else None
    gather_bytes = ds.csr()[1].size * (8 + 4 * cfg['towers'][0])      # index + value + one first-layer row per entry
    k_ms = sum(kernels.values())
    filt_ms = kernels.get('k_dmf_topk_filter')
    line = bench.base_line(cfg, 'dmf_full_catalog_ranked_users_per_sec', 'users/s', U / (ms_step * 1e-3), 1,
                           args.steps, args.warmup, ms, {
                               'workload': f"{cfg['title']}: DMF towers {cfg['towers']}/{cfg['towers']}, top-{K_TOP} over "
                                           f"the whole catalog for all {U} users, novelty on, synthetic {U}x{I} / "
                                           f"{cfg['nnz']} interactions (zipf_a={cfg['zipf_a']}), blocks of "
                                           f"{m._max_batch} users", 'note': cfg['note']}, clocks, launches)
    line.update({
        'overflow_users_rerun': flagged,
        'e2e': {'value': U / e2e_s, 'unit': 'users/s', 'seconds': e2e_s, 'call': 'recommend_batch(all users, n=100)'},
        'previous_route': {'value': prev, 'unit': 'users/s', 'users': len(prev_users),
                           'call': 'm._rank(uid, range(n_items), 100, True) per user (recommend() before this change)'},
        'speedup_vs_previous_route': U / (ms_step * 1e-3) / prev,
        'kernels_ms_per_step': kernels,
        'roofline': {
            'ffma': {'flops': flops, 'peak_flops_per_s': ffma_peak,
                     'peak': f'{sms} SMs x 128 FP32 lanes x 2 x max SM clock {gpu["max_sm_mhz"]} MHz (derived)',
                     'bound_ms': flops / ffma_peak * 1e3 if ffma_peak else None,
                     'filter_kernel_ms': filt_ms,
                     'frac_of_filter_kernel': (flops / ffma_peak * 1e3) / filt_ms if ffma_peak and filt_ms else None,
                     'note': 'the exact score is 32 products + 31 adds in tree order plus the normalisation: about '
                             '63 FP32 instructions per score, 2 w flops counted'},
            'gather': {'bytes': gather_bytes, 'hbm_bytes_per_s': 7.7e12,
                       'bound_ms': gather_bytes / 7.7e12 * 1e3, 'peak_source': 'HGX B200 data sheet, one GPU',
                       'note': 'user-tower first layer: one index, one value and one 64-float row per stored entry'},
            'kernels_ms_total': k_ms},
        'cpu_baseline': cpu_arm(cfg, ds, m, args.cpu_budget),
        'gpu': gpu,
        'bitwise_equal_rank_path': bitwise, 'bitwise_sample_users': len(sample),
    })
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--shapes', default='c2,ml20m')
    ap.add_argument('--cpu-budget', type=float, default=8.0)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be >= 1')
    D = bench.Dist()
    for name in args.shapes.split(','):
        print(json.dumps(run(SHAPES[name], args, D)), flush=True)


if __name__ == '__main__':
    main()
