#!/usr/bin/env python
"""recommendation_evaluation at the ml-20m shape: users/s of the whole call, one JSON line per model.

  python tools/bench_recommendation_evaluation.py [--models cdae,dmf] [--repeats R]

Data: synthetic 138,493 x 26,744, 20 M interactions (zipf 1.0), leave_k_out(k=1); CDAE K=200 and DMF [64, 32]
(fitted for 2 epochs).  The call: recommendation_evaluation(model, test, k=[10, 100], novelty=True) for all users.

value            users/s of the whole call (best of R repeats after one warm-up call)
parts            of the timed call: host protocol (candidate generation, tables, metric tail), top-k and the metric
                 kernel (CUDA events), upload + launch, copy of the per-user arrays
route_a          recommend_batch(users, n=100) to host arrays, then drb_eval_metrics on the host, in the same run;
                 equal_to_route_a: the result dicts are equal and the per-user dcg / idcg / hits / n_rec bitwise equal
route_b          the reference-shaped per-user loop (model.recommend + the metric classes) on a fixed sample of 200
                 users, users/s
gpu              name, power limit and SM clock of device 0, read in the same run
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K_LIST = [10, 100]
SHAPE = dict(n_users=138493, n_items=26744, nnz=20_000_000, zipf_a=1.0, seed=10)


def gpu_info():
    """name, power limit (W), current and max SM clock (MHz) of device 0, read only."""
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm',
                              '--format=csv,noheader,nounits', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(',')
        return {'name': out[0].strip(), 'power_limit_w': float(out[1]), 'sm_mhz': float(out[2]),
                'max_sm_mhz': float(out[3])}
    except Exception as e:
        return {'name': None, 'power_limit_w': None, 'sm_mhz': None, 'max_sm_mhz': None, 'error': str(e)}


def route_a(m, ds_test, users, ks, n_pos=None, novelty=False, low=None, seed=0, threshold=None, chunk=8192):
    """Per-user metric sums of `users` (raw ids, in the order the evaluation visited them) from recommend_batch's host
    arrays and the host C++ drb_eval_metrics, with the distinct items of each user's evaluated set (and their first
    test values) as both its test table and its candidate list.  Returns (result dict, per-user arrays)."""
    import pandas as pd
    from drecpy_b200 import _lib, evaluation as E
    from drecpy_b200.dataset import InteractionData
    thr = m.interaction_threshold if threshold is None else threshold
    train_eval = ds_test is None
    data = InteractionData.from_dataset(m.interaction_dataset if train_eval else ds_test)
    all_users, t_indptr, t_order = E._group_by_user(data)
    cand_off, cand, pos_off, pos, _, t_item, t_val = E.generate_candidates(
        m, data, all_users, t_indptr, t_order, thr, n_pos, None, False, train_eval, seed)
    idx = pd.Index(all_users).get_indexer(users)
    K = max(ks)
    items, _, counts = m.recommend_batch(users, n=K, novelty=novelty, interaction_threshold=low, chunk=chunk)
    keys, vals, lens, p_keys, p_lens, p_distinct = [], [], [], [], [], []
    for i in idx.tolist():
        first = {}
        for it, v in zip(t_item[t_indptr[i]:t_indptr[i + 1]].tolist(), t_val[t_indptr[i]:t_indptr[i + 1]].tolist()):
            first.setdefault(it, v)
        c = list(dict.fromkeys(cand[cand_off[i]:cand_off[i + 1]].tolist()))
        keys += c
        vals += [first[it] for it in c]
        lens.append(len(c))
        p = pos[pos_off[i]:pos_off[i + 1]].tolist()
        p_keys += p
        p_lens.append(len(p))
        p_distinct.append(len(set(p)))
    n = len(idx)
    off = np.zeros(n + 1, np.int64)
    np.cumsum(lens, out=off[1:])
    p_off = np.zeros(n + 1, np.int64)
    np.cumsum(p_lens, out=p_off[1:])
    keys, vals = np.asarray(keys, np.int64), np.asarray(vals, np.float64)
    p_keys = np.asarray(p_keys if p_keys else [0], np.int64)
    ranked = np.ascontiguousarray(items, np.int64)
    n_out = np.ascontiguousarray(counts, np.int32)
    ks_c = np.asarray(ks, np.int64)
    dcg, idcg = np.zeros((n, len(ks))), np.zeros((n, len(ks)))
    hits = np.zeros((n, len(ks)), np.int64)
    b, e = np.ascontiguousarray(off[:-1]), np.ascontiguousarray(off[1:])
    pb, pe = np.ascontiguousarray(p_off[:-1]), np.ascontiguousarray(p_off[1:])
    P = _lib.np_ptr
    _lib.check(_lib.load().drb_eval_metrics(n, P(b), P(e), P(keys), P(vals), P(ranked), K, P(n_out), P(b), P(e),
                                            P(keys), P(pb), P(pe), P(p_keys), P(ks_c), len(ks),
                                            min(16, os.cpu_count() or 1), P(dcg), P(idcg), P(hits)))
    n_rec = np.minimum(n_out[:, None].astype(np.int64), ks_c[None, :])
    metrics = [E.Precision(), E.Recall(), E.HitRatio(), E.NDCG()]
    sums = {(mm.name, k_): [0, 0] for mm in metrics for k_ in ks}
    E._metric_sums_from_user_values(sums, metrics, ks, dcg, idcg, hits, n_rec, np.asarray(p_lens, np.int64),
                                    np.asarray(p_distinct, np.int64))
    return E._metric_results(sums), {'dcg': dcg, 'idcg': idcg, 'hits': hits, 'n_rec': n_rec}


def bitwise_equal(per_user, ref):
    return (np.array_equal(per_user['dcg'].view(np.int64), ref['dcg'].view(np.int64))
            and np.array_equal(per_user['idcg'].view(np.int64), ref['idcg'].view(np.int64))
            and np.array_equal(per_user['hits'].astype(np.int64), ref['hits'])
            and np.array_equal(per_user['n_rec'].astype(np.int64), ref['n_rec']))


def route_b(m, test, users, ks, novelty):
    """The reference-shaped loop: model.recommend per user, then the metric classes (ranking_evaluation's dispatch)."""
    from drecpy_b200 import evaluation as E
    rows = {}
    for u, it, v in zip(test.user.tolist(), test.item.tolist(), test.interaction.tolist()):
        rows.setdefault(u, []).append((it, v))
    metrics = [E.Precision(), E.Recall(), E.HitRatio(), E.NDCG()]
    sums = {(mm.name, k_): [0, 0] for mm in metrics for k_ in ks}
    t0 = time.perf_counter()
    for u in users:
        r = rows[u]
        recs = [it for _, it in m.recommend(u, n=max(ks), novelty=novelty)]
        positives = [it for it, v in r if v >= m.interaction_threshold]
        rel = {it: 0 for it in recs}
        for it, v in reversed(r):
            rel[it] = v
        best = min(positives, key=lambda it: rel[it]) if positives else None
        E._call_metrics(sums, metrics, ks, recs, positives, best, rel)
    return len(users) / (time.perf_counter() - t0)


def build_model(name, train):
    import drecpy_b200 as drb
    if name == 'cdae':
        m = drb.CDAE(hidden_factors=200, seed=10, verbose=False, rng_mode='philox')
        m.fit(train, epochs=2, batch_size=4096)
        return m, 'CDAE K=200'
    m = drb.DMF(user_factors=[64, 32], item_factors=[64, 32], seed=10, verbose=False)
    m.fit(train, epochs=2, batch_size=4096, score_batch=32768)
    return m, 'DMF [64, 32]'


def run(name, args, train, test):
    import torch
    import drecpy_b200 as drb
    m, desc = build_model(name, train)
    n_test_users = len(np.unique(test.user))
    drb.recommendation_evaluation(m, test, k=K_LIST, novelty=True)                 # warm-up: every shape of the call
    best, tm, res = None, None, None
    for _ in range(args.repeats):
        t = {}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = drb.recommendation_evaluation(m, test, k=K_LIST, novelty=True, timings=t)
        dt = time.perf_counter() - t0
        if best is None or dt < best:
            best, tm, res = dt, t, r
    per_user = tm.pop('per_user')
    t0 = time.perf_counter()
    ref, ref_pu = route_a(m, test, per_user['users'], K_LIST, novelty=True)
    a_s = time.perf_counter() - t0
    sample = np.random.default_rng(0).choice(per_user['users'], 200, replace=False).tolist()
    b_rate = route_b(m, test, sample, K_LIST, True)
    return {
        'metric': f'recommendation_evaluation_{name}_users_per_sec', 'value': tm['n_users'] / best, 'unit': 'users/s',
        'workload': f"recommendation_evaluation(k={K_LIST}, novelty=True) of all {n_test_users} test users, {desc}, "
                    f"synthetic {SHAPE['n_users']}x{SHAPE['n_items']} / {SHAPE['nnz']} interactions "
                    f"(zipf {SHAPE['zipf_a']}), leave_k_out(k=1)",
        'seconds': best, 'repeats': args.repeats, 'evaluated_users': tm['n_users'], 'result': res,
        'parts': {'host_protocol_s': tm['host_protocol_s'], 'upload_and_launch_s': tm['launch_and_upload_s'],
                  'copy_back_s': tm['copy_back_s'], 'topk_ms': tm['topk_ms'],
                  'metrics_kernel_ms': tm['metrics_kernel_ms']},
        'route_a': {'seconds': a_s, 'value': tm['n_users'] / a_s, 'unit': 'users/s',
                    'call': 'recommend_batch(users, n=100) + drb_eval_metrics (host)'},
        'equal_to_route_a': bool(ref == res and bitwise_equal(per_user, ref_pu)),
        'route_b': {'value': b_rate, 'unit': 'users/s', 'users': len(sample),
                    'call': 'model.recommend + metric classes per user (reference-shaped loop)'},
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
    train, test = drb.leave_k_out(drb.InteractionData(u, i, v), k=1, seed=10, max_concurrent_threads=16)
    train.assign_internal_ids()
    for name in args.models.split(','):
        print(json.dumps(run(name, args, train, test)), flush=True)


if __name__ == '__main__':
    main()
