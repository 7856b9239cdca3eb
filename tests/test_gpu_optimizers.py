"""fit(optimizer=...) on the GPU: every supported Keras optimizer against the oracle (oracle/optim.py) on identical
seeded inputs, injected initial weights and sampler / mask streams; graph replay, the Adam default spelled three ways,
and save / load of the optimizer slots.  Tolerances are those of tests/test_gpu_parity.py."""
import random

import numpy as np
import pytest
import torch

import drecpy_b200 as drb
from drecpy_b200 import _lib, optimizers
from oracle import philox as ophilox
from oracle.cdae import corruption_keep_mt
from oracle.optim import CDAEOptimOracle, CDAESampledOptimOracle, DMFOptimOracle
from oracle.sampler import PointSamplerOracle

pytestmark = pytest.mark.gpu

OPTIMIZERS = {
    'sgd': {'name': 'SGD', 'learning_rate': 0.1},
    'sgd_momentum': {'name': 'SGD', 'learning_rate': 0.1, 'momentum': 0.9},
    'sgd_nesterov': {'name': 'SGD', 'learning_rate': 0.1, 'momentum': 0.9, 'nesterov': True},
    'rmsprop': {'name': 'RMSprop'},
    'rmsprop_centered': {'name': 'RMSprop', 'centered': True},
    # with momentum 0.9 RMSprop's step is up to ~30 x lr (g / sqrt(0.1 g^2) summed over ~10 steps): elements whose
    # gradient is fp32 rounding noise drift apart by that much, so these two run at lr 1e-4
    'rmsprop_momentum': {'name': 'RMSprop', 'learning_rate': 1e-4, 'momentum': 0.9},
    'rmsprop_centered_momentum': {'name': 'RMSprop', 'learning_rate': 1e-4, 'momentum': 0.9, 'centered': True},
    'adagrad': {'name': 'Adagrad', 'learning_rate': 0.01},
    'adamax': {'name': 'Adamax'},
    'amsgrad': {'name': 'Adam', 'amsgrad': True},
    'sgd_momentum_decay': {'name': 'SGD', 'learning_rate': 0.1, 'momentum': 0.9, 'decay': 0.002},
}


def _dataset(U, I, nnz, seed=10):
    u, i, v = drb.synthetic_interactions(U, I, nnz, seed=seed)
    ds = drb.InteractionData(u, i, v)
    ds.assign_internal_ids()
    return ds


def _cdae_weights(U, I, K, seed=1):
    rng = np.random.default_rng(seed)

    def glorot(shape, fi, fo):
        lim = np.sqrt(6.0 / (fi + fo))
        return rng.uniform(-lim, lim, shape).astype(np.float32)
    return {'W': glorot((I, K), I, K), 'W_': glorot((K, I), K, I), 'V': glorot((U, K), U, K),
            'b': glorot((K,), K, K), 'b_': glorot((I,), I, I)}


def rel_err(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def _cdae(ds, K, B, w, opt, **kw):
    m = drb.CDAE(hidden_factors=K, corruption_level=0.2, seed=10, verbose=False, **kw)
    m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, neg_ratio=5, reg_rate=1e-3, init_weights=w, optimizer=opt)
    return m


def _oracle_opt(opt):
    return dict(opt)          # the raw config: oracle.optim fills in the Keras defaults itself


@pytest.mark.parametrize('case', list(OPTIMIZERS))
def test_cdae_c1_100_steps_vs_oracle(case):
    """C1: 943 x 1682, 100k interactions, K=50, q=0.2, bce, B=64, the bit-exact sampler and MT19937 mask stream."""
    opt = OPTIMIZERS[case]
    ds = _dataset(943, 1682, 100000)
    U, I, K, B = 943, 1682, 50, 64
    w = _cdae_weights(U, I, K)
    m = _cdae(ds, K, B, w, opt)
    o = CDAEOptimOracle(w['W'], w['W_'], w['V'], w['b'], w['b_'], ds.csr(), interaction_threshold=1e-3,
                        optimizer=_oracle_opt(opt))
    so, pr = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, 5, 1e-3, 10), random.Random(10)
    l, lo = [], []
    for s in range(1, 101):
        m._step = s
        l.append(m._train_step(B, 1e-3, want_loss=True))
        uids = np.array([t[0] for t in so.sample(B)])
        keep = np.stack([corruption_keep_mt(pr, I, o.q) for _ in uids])
        lo.append(float(o.step(uids, keep, 1e-3)))
    l, lo = np.array(l), np.array(lo)
    assert np.all(np.isfinite(l))
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-3, (case, l[-5:], lo[-5:])
    for name in ('W', 'W_', 'V', 'b', 'b_'):
        assert rel_err(getattr(m, name).cpu().numpy(), getattr(o, name)) < 2e-3, (case, name)
    assert rel_err(m.W_.cpu().numpy(), w['W_']) > 1e-5, case          # the update moved the weights
    if case == 'amsgrad':
        # v-hat is a running maximum of v, and it differs from v where v has shrunk (user rows sampled once and then
        # decayed under the L2 gradient alone): plain Adam run in its place would leave the third arena at zero
        vhat, v = m._optim_x, m._adam_v
        assert bool(torch.all(vhat >= v)) and bool(torch.any(vhat > v))


def _dmf_weights(U, I, uf, itf, seed=2):
    rng = np.random.default_rng(seed)

    def tower(in_dim, factors):
        out = []
        for f in factors:
            lim = np.sqrt(6.0 / (in_dim + f))
            out.append((rng.uniform(-lim, lim, (in_dim, f)).astype(np.float32),
                        rng.uniform(0.0, 0.05, f).astype(np.float32)))
            in_dim = f
        return out
    return {'user_nn': tower(I, uf), 'item_nn': tower(U, itf)}


@pytest.mark.parametrize('case', list(OPTIMIZERS))
def test_dmf_steps_vs_oracle(case):
    opt = OPTIMIZERS[case]
    U, I, B = 400, 600, 64
    ds = _dataset(U, I, 20000, seed=5)
    w = _dmf_weights(U, I, [64, 32], [64, 32])
    m = drb.DMF(user_factors=[64, 32], item_factors=[64, 32], seed=10, verbose=False)
    m.fit(ds, epochs=0, batch_size=B, learning_rate=1e-3, neg_ratio=5, reg_rate=1e-4, init_weights=w, optimizer=opt)
    o = DMFOptimOracle(w['user_nn'], w['item_nn'], ds.csr(), ds.csc(), m.min_interaction, m.max_interaction,
                       optimizer=_oracle_opt(opt))
    so = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, 5, 1e-3, 10)
    l, lo = [], []
    for s in range(1, 41):
        m._step = s
        l.append(m._train_step(B, 1e-4, want_loss=True))
        t = so.sample(B)
        lo.append(float(o.step([x[0] for x in t], [x[1] for x in t], [o.standardize(x[2]) for x in t], 1e-4)))
    l, lo = np.array(l), np.array(lo)
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-3, (case, l[-3:], lo[-3:])
    for (k, b), (ko, bo) in zip(m.tower_weights('user_nn') + m.tower_weights('item_nn'), o.user_layers + o.item_layers):
        assert rel_err(k.cpu().numpy(), ko) < 2e-3, case
        assert rel_err(b.cpu().numpy(), bo) < 2e-3, case


def test_cdae_sampled_output_step_vs_oracle():
    """The sampled-output step with centered RMSprop and momentum (the third arena) against CDAESampledOptimOracle."""
    opt = OPTIMIZERS['rmsprop_centered_momentum']
    ds = _dataset(211, 389, 9000, seed=4)
    U, I, B, K = 211, 389, 48, 36
    w = _cdae_weights(U, I, K)
    m = _cdae(ds, K, B, w, opt, rng_mode='philox', output='sampled', neg_per_group=20, neg_groups=2)
    assert m._optim_x is not None
    o = CDAESampledOptimOracle(w['W'], w['W_'], w['V'], w['b'], w['b_'], ds.csr(), interaction_threshold=1e-3,
                               n_groups=2, neg_per_group=20, seed=10, optimizer=_oracle_opt(opt))
    so = PointSamplerOracle(ds.uid, ds.iid, ds.interaction, 5, 1e-3, 10)
    pos = ds.csr(1e-3)
    l, lo = [], []
    for s in range(1, 16):
        m._step = s
        l.append(m._train_step(B, 1e-3, want_loss=True))
        uids = np.array([t[0] for t in so.sample(B)])
        keep = np.ones((B, I), bool)
        for b, u in enumerate(uids):
            items = pos[1][pos[0][u]:pos[0][u + 1]]
            keep[b, items] = ophilox.keep_mask(items, b, s, 10, o.q)
        lo.append(float(o.step_sampled(uids, keep, 1e-3, s)))
    l, lo = np.array(l), np.array(lo)
    assert np.max(np.abs(l - lo) / np.abs(lo)) < 1e-4, (l, lo)
    for name in ('W', 'W_', 'V', 'b', 'b_'):
        assert rel_err(getattr(m, name).cpu().numpy(), getattr(o, name)) < 5e-4, name


def _steps(m, n, B, first=1):
    losses = []
    for s in range(first, first + n):
        m._step = s
        losses.append(m._train_step(B, 1e-3, want_loss=True))
    return losses


def test_cdae_graph_replay_equals_direct_launches(monkeypatch):
    """AMSGrad through the replayed CUDA graph and through direct launches.  At B = 2 no gradient element receives more
    than two atomic additions, which commute: the two runs are bitwise equal.  At B = 48 the losses agree to the last
    bits.  Switching the optimizer of a model whose step was captured re-captures it (no stale replay)."""
    ds = _dataset(300, 500, 15000, seed=8)
    w = _cdae_weights(300, 500, 24)
    opt = OPTIMIZERS['amsgrad']
    for B, exact in ((2, True), (48, False)):
        runs = []
        for graph in ('1', '0'):
            monkeypatch.setenv('DRB_GRAPH', graph)
            m = _cdae(ds, 24, B, w, opt)
            n0 = m.launch_count()
            losses = _steps(m, 12, B)
            runs.append((np.array(losses), m.launch_count() - n0, [t.cpu().numpy() for t in
                                                                   (m._params, m._adam_m, m._adam_v, m._optim_x)]))
        assert runs[0][1] > runs[1][1]                       # the graph run replayed (one k_set_scalars per step)
        if exact:
            assert np.array_equal(runs[0][0], runs[1][0])
            for a, b in zip(runs[0][2], runs[1][2]):
                assert np.array_equal(a, b)
        else:
            assert np.allclose(runs[0][0], runs[1][0], rtol=2e-6, atol=0)
            assert rel_err(runs[0][2][0], runs[1][2][0]) < 1e-5
    # switch the optimizer of a live model (graph captured for SGD) and compare with direct launches
    final = []
    for graph in ('1', '0'):
        monkeypatch.setenv('DRB_GRAPH', graph)
        m = _cdae(ds, 24, 2, w, OPTIMIZERS['sgd_momentum'])
        _steps(m, 6, 2)
        m.optimizer = optimizers.parse({'name': 'Adagrad', 'learning_rate': 0.05})
        m._adam_m.fill_(0.1)
        m._apply_optimizer()
        losses = _steps(m, 6, 2, first=7)
        final.append((np.array(losses), m._params.cpu().numpy()))
    assert np.array_equal(final[0][0], final[1][0]) and np.array_equal(final[0][1], final[1][1])


def test_dmf_graph_replay_after_an_optimizer_switch(monkeypatch):
    """Adamax, then SGD with momentum on the same live model: graph replay against direct launches.  A replay of the
    graph captured for Adamax would keep taking Adamax steps; the run that never switches shows how far apart that
    ends up.  The tower scatter adds with atomics, and Adamax's first steps are about lr in size whatever the gradient's
    magnitude, so the two runs agree to 1e-4 of the weights' scale rather than bit for bit."""
    U, I, B = 300, 500, 64
    ds = _dataset(U, I, 15000, seed=8)
    w = _dmf_weights(U, I, [64, 32], [64, 32])
    runs = []
    for graph, switch in (('1', True), ('0', True), ('1', False)):
        monkeypatch.setenv('DRB_GRAPH', graph)
        m = drb.DMF(user_factors=[64, 32], item_factors=[64, 32], seed=10, verbose=False)
        m.fit(ds, epochs=0, batch_size=B, reg_rate=1e-4, init_weights=w, optimizer={'name': 'Adamax'})
        losses = [m._train_step(B, 1e-4, want_loss=True) for m._step in range(1, 6)]
        if switch:
            m.optimizer = optimizers.parse({'name': 'SGD', 'learning_rate': 0.5, 'momentum': 0.5})
            m._adam_m.zero_()
            m._apply_optimizer()
        losses += [m._train_step(B, 1e-4, want_loss=True) for m._step in range(6, 11)]
        runs.append((np.array(losses), m._params.cpu().numpy()))
    assert np.allclose(runs[0][0], runs[1][0], rtol=2e-6, atol=0)
    assert rel_err(runs[0][1], runs[1][1]) < 1e-4
    assert rel_err(runs[2][1], runs[1][1]) > 100 * rel_err(runs[0][1], runs[1][1])


class _KerasStub:
    def __init__(self, **config):
        self.config = config

    def get_config(self):
        return dict(self.config)


@pytest.mark.parametrize('cls', ['CDAE', 'DMF'])
def test_adam_spelled_three_ways_is_bitwise_the_default(cls):
    ds = _dataset(120, 200, 4000, seed=9)
    spellings = [None, {'name': 'Adam'},
                 _KerasStub(name='Adam', learning_rate=0.001, decay=0.0, beta_1=0.9, beta_2=0.999, epsilon=1e-07,
                            amsgrad=False)]
    out = []
    for opt in spellings:
        m = drb.CDAE(hidden_factors=12, seed=10, verbose=False) if cls == 'CDAE' else \
            drb.DMF(user_factors=[16, 8], item_factors=[16, 8], seed=10, verbose=False)
        m.fit(ds, epochs=8, batch_size=2, optimizer=opt)
        assert m.optimizer['name'] == 'Adam' and m._optim_x is None
        out.append([t.cpu().numpy() for t in (m._params, m._adam_m, m._adam_v)])
    for other in out[1:]:
        for a, b in zip(out[0], other):
            assert np.array_equal(a, b)


@pytest.mark.parametrize('opt', ['amsgrad', 'rmsprop_centered_momentum', 'adagrad'])
def test_save_load_round_trips_every_slot_arena(tmp_path, opt):
    ds = _dataset(120, 200, 4000, seed=9)
    m = drb.CDAE(hidden_factors=12, seed=10, verbose=False)
    m.fit(ds, epochs=6, batch_size=16, optimizer=OPTIMIZERS[opt])
    assert (m._optim_x is not None) == (opt != 'adagrad')
    path = str(tmp_path / 'model.joblib')
    m.save(path)
    m2 = drb.CDAE.load(path)
    assert m2.optimizer == m.optimizer
    for k in ('_params', '_adam_m', '_adam_v', '_optim_x'):
        a, b = getattr(m, k), getattr(m2, k)
        assert (a is None) == (b is None), k
        if a is not None:
            assert b.device.type == 'cuda' and torch.equal(a, b), k
    p = m.predict(ds.uid_to_user(0), ds.iid_to_item(0))
    assert m2.predict(ds.uid_to_user(0), ds.iid_to_item(0)) == p


def test_native_setter_refuses_bad_descriptors():
    ds = _dataset(60, 80, 1200, seed=3)
    m = drb.CDAE(hidden_factors=8, seed=10, verbose=False)
    m.fit(ds, epochs=1, batch_size=8)
    lib = _lib.load()
    import ctypes as C
    for fields, msg in (({'kind': 9}, b'unknown optimizer kind'), ({'kind': 1, 'momentum': -1.0}, b'momentum'),
                        ({'kind': 0, 'amsgrad': 1, 'beta1': 0.9, 'beta2': 0.999, 'epsilon': 1e-7}, b'third_state'),
                        ({'kind': 3, 'epsilon': 0.0}, b'epsilon'), ({'kind': 2, 'rho': 2.0, 'epsilon': 1e-7}, b'rho')):
        d = _lib.OptimDesc(**fields)
        assert lib.drb_cdae_set_optimizer(m._native, C.byref(d)) == -1
        assert msg in lib.drb_last_error()
    m._train_step(8, 1e-3)            # the model still runs its (unchanged) Adam
