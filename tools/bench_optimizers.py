#!/usr/bin/env python
"""The CDAE training step at the ml-20m shape (bench.py's c3) with every optimizer fit(optimizer=...) runs natively.

  python tools/bench_optimizers.py [--steps K] [--warmup W] [--only sgd,adam,...]

Data and model: bench.py's C3 (synthetic 138,493 x 26,744, 20 M interactions, zipf 1.0; K=200, B=4096, philox mask),
device-resident batches fed through step_device.  One JSON line per optimizer:

step_ms              CUDA-event time of K steps / K (after W warm-up steps), profiling off
update_ms            the update kernel's (K4) CUDA-event time per step, from a separate profiled run of K steps
update_kernel        its profiler name (k_adam, k_optim_sgd, ...)
bytes_per_param      state bytes K4 moves per parameter: w read + written, g read, each slot read + written
alg_bytes_per_step   bytes_per_param x parameters, less the 4 B gradient read of every element of an untouched V row
                     (users not in the batch; counted per batch)
update_gbs / of_peak alg_bytes_per_step / update_ms, and that over the HBM peak bench.py divides by (bench.load_peaks():
                     the measured copy peak of MEASURED_PEAKS.json, else bench.py's fallback figure); peak_gbs and
                     peak_src say which
gpu                  name, power limit and SM clock of device 0, read in the same run
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

OPTIMIZERS = {
    'adam': (None, 28),
    'sgd': ({'name': 'SGD', 'learning_rate': 0.1}, 12),
    'sgd_momentum': ({'name': 'SGD', 'learning_rate': 0.1, 'momentum': 0.9}, 20),
    'rmsprop': ({'name': 'RMSprop'}, 20),
    'rmsprop_centered': ({'name': 'RMSprop', 'centered': True}, 28),
    'rmsprop_momentum': ({'name': 'RMSprop', 'momentum': 0.9}, 28),
    'rmsprop_centered_momentum': ({'name': 'RMSprop', 'momentum': 0.9, 'centered': True}, 36),
    'adagrad': ({'name': 'Adagrad'}, 20),
    'adamax': ({'name': 'Adamax'}, 28),
    'amsgrad': ({'name': 'Adam', 'amsgrad': True}, 36),
}


def run(name, args, ds, cfg, gpu, peaks):
    import torch
    import drecpy_b200 as drb
    from drecpy_b200 import _lib
    opt, bpp = OPTIMIZERS[name]
    B = cfg['batch']
    m = drb.CDAE(hidden_factors=cfg['hidden'], corruption_level=cfg['q'], seed=cfg['seed'], verbose=False,
                 rng_mode='philox')
    m.fit(ds, epochs=0, batch_size=B, learning_rate=cfg['lr'], reg_rate=cfg['reg'], optimizer=opt)
    lib = _lib.load()
    batches, untouched = [], []
    for _ in range(16):
        u = m._sampler.sample_arrays(B)[0]
        off = np.zeros(B + 1, np.int32)
        _lib.check(lib.drb_batch_offsets(_lib.np_ptr(u), B, _lib.np_ptr(m._h_indptr), _lib.np_ptr(off)))
        batches.append((torch.from_numpy(u.copy()).to(m._dev), torch.from_numpy(off).to(m._dev)))
        untouched.append(m.n_users - len(np.unique(u)))
    loss = torch.zeros(2, device=m._dev)

    def steps(n, first):
        for s in range(first, first + n):
            bt = batches[s % len(batches)]
            m.step_device(bt[0], bt[1], None, cfg['reg'], loss)
    steps(args.warmup, 0)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    steps(args.steps, args.warmup)
    e1.record()
    torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / args.steps
    _lib.check(lib.drb_ctx_profile_enable(m._ctx, 1))
    steps(args.steps, args.warmup + args.steps)
    prof = _lib.profile_read(m._ctx)
    _lib.check(lib.drb_ctx_profile_enable(m._ctx, 0))
    kname = [k for k in prof if k == 'k_adam' or k.startswith('k_optim_')]
    assert len(kname) == 1, prof
    update_ms = prof[kname[0]][0] / args.steps
    n_params = int(m._L.total)
    alg = bpp * n_params - 4 * m._L.ld * float(np.mean(untouched))
    loss_v = float(loss[0].item())
    return {'optimizer': name, 'config': m.optimizer, 'step_ms': step_ms, 'update_ms': update_ms,
            'update_kernel': kname[0], 'bytes_per_param': bpp, 'params': n_params, 'alg_bytes_per_step': alg,
            'update_gbs': alg / (update_ms * 1e-3) / 1e9, 'of_peak': alg / (update_ms * 1e-3) / 1e9 / peaks['hbm'],
            'peak_gbs': peaks['hbm'], 'peak_src': peaks['src'],
            'loss_last': loss_v, 'finite': bool(np.isfinite(loss_v)), 'steps': args.steps, 'warmup': args.warmup,
            'shape': f"{cfg['n_users']} x {cfg['n_items']}, {cfg['nnz']} interactions, K={cfg['hidden']}, B={B}",
            'gpu': gpu}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--only', default=','.join(OPTIMIZERS))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('bench_optimizers: needs a CUDA device (there is no CPU measurement)')
    import bench
    from tools.bench_recommendation_evaluation import gpu_info
    cfg = bench.C3
    ds, _ = bench.make_data(cfg)
    gpu, peaks = gpu_info(), bench.load_peaks()
    for name in args.only.split(','):
        print(json.dumps(run(name, args, ds, cfg, gpu, peaks)), flush=True)


if __name__ == '__main__':
    main()
