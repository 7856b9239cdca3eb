#!/usr/bin/env python
"""predictive_evaluation at the ml-20m shape: test rows/s of the whole call, one JSON line per model.

  python tools/bench_predictive_evaluation.py [--models cdae,dmf] [--repeats R]

Data: synthetic 138,493 x 26,744, 20 M interactions (zipf 1.0), leave_k_out(k=0.2) (about 4 M test rows); CDAE K=200
and DMF [64, 32] (fitted for 2 epochs).  The call: predictive_evaluation(model, test) (RMSE, MSE) over every test row.

value            test rows/s of the whole call (best of R repeats after one warm-up call)
parts            of a separate call with timings= (the library brackets every launch with CUDA events there): host
                 selection, predict_batch wall time, pair-kernel and user-side (K1 gather / tower GEMMs, argument
                 check) kernel time, per-kernel breakdown
grouping         grouping 4 M (uid, iid) pairs by user: torch on the device (upload, stable sort, unique_consecutive,
                 cumsum; what predict_batch does) and NumPy on the host (stable argsort, unique, cumsum), best of 3
general          the per-row model.predict loop on the first 1,000 rows, rows/s
equal_to_general the batched dict equals the per-row dict at n_test_predictions=2000, with y_pred bitwise equal
gpu              name, power limit and SM clock of device 0, read in the same run
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.bench_recommendation_evaluation import SHAPE, build_model, gpu_info   # noqa: E402


def grouping(m, test):
    """Seconds to group the test pairs by internal uid: on the device with torch, and on the host with NumPy."""
    import torch
    uids, iids = m._pair_ids(test.user, test.item)
    dev, host = [], []
    for _ in range(3):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        d_u = torch.from_numpy(uids).to(m._dev)
        d_i = torch.from_numpy(iids).to(m._dev)
        s_u, order = torch.sort(d_u, stable=True)
        users, counts = torch.unique_consecutive(s_u, return_counts=True)
        off = torch.cumsum(counts, 0)
        p_iid = d_i[order]
        torch.cuda.synchronize()
        dev.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        order_h = np.argsort(uids, kind='stable')
        users_h, counts_h = np.unique(uids[order_h], return_counts=True)
        off_h = np.cumsum(counts_h)
        p_iid_h = iids[order_h]
        host.append(time.perf_counter() - t0)
    assert np.array_equal(users.cpu().numpy(), users_h) and np.array_equal(off.cpu().numpy(), off_h)
    assert np.array_equal(p_iid.cpu().numpy(), p_iid_h)
    return {'pairs': len(uids), 'torch_device_s': min(dev), 'numpy_host_s': min(host)}


def run(name, args, train, test):
    import torch
    import drecpy_b200 as drb
    m, desc = build_model(name, train)
    drb.predictive_evaluation(m, test)                           # warm-up: every shape of the call
    best, res = None, None
    for _ in range(args.repeats):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = drb.predictive_evaluation(m, test)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, res = dt, r
    tm = {}
    drb.predictive_evaluation(m, test, timings=tm)
    n_rows = tm['n_rows']
    small_f, small_s = {}, {}
    eq = (drb.predictive_evaluation(m, test, n_test_predictions=2000, timings=small_f) ==
          drb.predictive_evaluation(m, test, n_test_predictions=2000, timings=small_s, force_python=True))
    eq = bool(eq and np.array_equal(small_f['y_pred'].view(np.uint64), small_s['y_pred'].view(np.uint64)))
    t0 = time.perf_counter()
    gen = {}
    drb.predictive_evaluation(m, test, n_test_predictions=1000, force_python=True, timings=gen)
    gen_rate = len(gen['y_pred']) / (time.perf_counter() - t0)
    return {
        'metric': f'predictive_evaluation_{name}_rows_per_sec', 'value': n_rows / best, 'unit': 'rows/s',
        'workload': f"predictive_evaluation (RMSE, MSE) of all {len(test)} test rows, {desc}, synthetic "
                    f"{SHAPE['n_users']}x{SHAPE['n_items']} / {SHAPE['nnz']} interactions (zipf {SHAPE['zipf_a']}), "
                    f"leave_k_out(k=0.2)",
        'seconds': best, 'repeats': args.repeats, 'rows': n_rows, 'result': res,
        'parts': {'host_select_s': tm['host_select_s'], 'predict_batch_s': tm['predict_batch_s'],
                  'pair_kernel_ms': tm['pair_kernel_ms'], 'user_side_kernel_ms': tm['user_side_kernel_ms'],
                  'kernels_ms': tm['kernels_ms']},
        'grouping': grouping(m, test),
        'general': {'value': gen_rate, 'unit': 'rows/s', 'rows': len(gen['y_pred']),
                    'call': 'model.predict per row (first 1000 counted rows)'},
        'equal_to_general': eq,
        'gpu': gpu_info(),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--models', default='cdae,dmf')
    ap.add_argument('--repeats', type=int, default=3)
    args = ap.parse_args()
    if args.repeats < 1:
        ap.error('--repeats must be >= 1')
    import drecpy_b200 as drb
    u, i, v = drb.synthetic_interactions(SHAPE['n_users'], SHAPE['n_items'], SHAPE['nnz'], seed=SHAPE['seed'],
                                         zipf_a=SHAPE['zipf_a'])
    train, test = drb.leave_k_out(drb.InteractionData(u, i, v), k=0.2, seed=10, max_concurrent_threads=16)
    train.assign_internal_ids()
    for name in args.models.split(','):
        print(json.dumps(run(name, args, train, test)), flush=True)


if __name__ == '__main__':
    main()
