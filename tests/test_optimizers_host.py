"""fit(optimizer=...) without a GPU: the oracle's Keras updates (oracle/optim.py) against torch.optim in float64 where the
formulas coincide and against hand-written float64 loops where they do not, and the parsing / refusals of
drecpy_b200.optimizers (the dict fit() keeps as self.optimizer and the native descriptor built from it)."""
import numpy as np
import pytest
import torch

import drecpy_b200 as drb
from drecpy_b200 import _lib, optimizers
from oracle.optim import KerasOptimizer

D = np.float64


def _grads(n_steps, shape=(7, 5), seed=0):
    rng = np.random.default_rng(seed)
    return [rng.normal(0, 1, shape) * rng.uniform(0.1, 2.0) for _ in range(n_steps)]


def _run_oracle(config, w0, grads, ts=None):
    opt = KerasOptimizer(config)
    w = np.array(w0, D)
    s = opt.slots(w)
    for j, g in enumerate(grads):
        opt.update(w, s, np.array(g, D), ts[j] if ts is not None else j + 1)
    return w


def _run_torch(make, w0, grads):
    p = torch.nn.Parameter(torch.tensor(w0, dtype=torch.float64))
    opt = make([p])
    for g in grads:
        p.grad = torch.tensor(g, dtype=torch.float64)
        opt.step()
    return p.detach().numpy()


W0 = np.random.default_rng(1).normal(0, 0.3, (7, 5))


@pytest.mark.parametrize('config,make', [
    ({'name': 'SGD', 'learning_rate': 0.05}, lambda p: torch.optim.SGD(p, lr=0.05)),
    ({'name': 'SGD', 'learning_rate': 0.05, 'momentum': 0.9}, lambda p: torch.optim.SGD(p, lr=0.05, momentum=0.9)),
    ({'name': 'SGD', 'learning_rate': 0.05, 'momentum': 0.8, 'nesterov': True},
     lambda p: torch.optim.SGD(p, lr=0.05, momentum=0.8, nesterov=True)),
    ({'name': 'RMSprop', 'learning_rate': 0.01, 'rho': 0.85, 'epsilon': 1e-6},
     lambda p: torch.optim.RMSprop(p, lr=0.01, alpha=0.85, eps=1e-6)),
    ({'name': 'RMSprop', 'learning_rate': 0.01, 'rho': 0.9, 'epsilon': 1e-6, 'centered': True},
     lambda p: torch.optim.RMSprop(p, lr=0.01, alpha=0.9, eps=1e-6, centered=True)),
    ({'name': 'Adagrad', 'learning_rate': 0.1, 'initial_accumulator_value': 0.3, 'epsilon': 1e-7},
     lambda p: torch.optim.Adagrad(p, lr=0.1, initial_accumulator_value=0.3, eps=1e-7)),
    ({'name': 'Adagrad', 'learning_rate': 0.1, 'initial_accumulator_value': 0.1, 'epsilon': 1e-7, 'decay': 0.05},
     lambda p: torch.optim.Adagrad(p, lr=0.1, lr_decay=0.05, initial_accumulator_value=0.1, eps=1e-7)),
], ids=['sgd', 'sgd_momentum', 'sgd_nesterov', 'rmsprop', 'rmsprop_centered', 'adagrad', 'adagrad_decay'])
def test_oracle_matches_torch_optim_float64(config, make):
    grads = _grads(12)
    got = _run_oracle(config, W0, grads)
    want = _run_torch(make, W0, grads)
    assert np.max(np.abs(got - want)) <= 1e-12 * max(1.0, np.abs(want).max()), config
    assert np.max(np.abs(got - W0)) > 1e-3          # the weights moved


def _loop_rmsprop_momentum(w, grads, lr, rho, mom, eps, centered):
    w = w.copy()
    ms, mg, mv = np.zeros_like(w), np.zeros_like(w), np.zeros_like(w)
    for g in grads:
        ms = ms + (g * g - ms) * (1 - rho)
        if centered:
            mg = mg + (g - mg) * (1 - rho)
            d = ms - mg * mg + eps                    # epsilon inside the square root in this branch
        else:
            d = ms + eps
        mv = mv * mom + lr * g / np.sqrt(d)
        w = w - mv
    return w


@pytest.mark.parametrize('centered', [False, True])
def test_rmsprop_with_momentum_puts_epsilon_inside_the_square_root(centered):
    grads = _grads(10, seed=2)
    cfg = {'name': 'RMSprop', 'learning_rate': 0.01, 'rho': 0.8, 'momentum': 0.7, 'epsilon': 0.05,
           'centered': centered}
    got = _run_oracle(cfg, W0, grads)
    want = _loop_rmsprop_momentum(W0, grads, 0.01, 0.8, 0.7, 0.05, centered)
    assert np.allclose(got, want, rtol=1e-13, atol=1e-15)
    # eps = 0.05 is large on purpose: the momentum == 0 branch (eps outside the root) gives different weights
    cfg0 = dict(cfg, momentum=0.0)
    assert np.max(np.abs(_run_oracle(cfg0, W0, grads) - want)) > 1e-3


def test_adamax_against_a_float64_loop():
    grads = _grads(15, seed=3)
    lr, b1, b2, eps = 0.02, 0.85, 0.99, 1e-6
    w, m, u = W0.copy(), np.zeros_like(W0), np.zeros_like(W0)
    for t, g in enumerate(grads, 1):
        m = m + (g - m) * (1 - b1)
        u = np.maximum(b2 * u, np.abs(g))
        w = w - lr / (1 - b1 ** t) * (m / (u + eps))
    got = _run_oracle({'name': 'Adamax', 'learning_rate': lr, 'beta_1': b1, 'beta_2': b2, 'epsilon': eps}, W0, grads)
    assert np.allclose(got, w, rtol=1e-13, atol=1e-15)


def test_amsgrad_against_a_float64_loop():
    rng = np.random.default_rng(4)
    grads = [rng.normal(0, 1, W0.shape) * (3.0 if t < 3 else 0.2) for t in range(14)]    # v shrinks: vhat matters
    lr, b1, b2, eps = 0.01, 0.9, 0.95, 1e-7
    w, m, v, vh = W0.copy(), np.zeros_like(W0), np.zeros_like(W0), np.zeros_like(W0)
    for t, g in enumerate(grads, 1):
        alpha = lr * np.sqrt(1 - b2 ** t) / (1 - b1 ** t)
        m = m + (g - m) * (1 - b1)
        v = v + (g * g - v) * (1 - b2)
        vh = np.maximum(vh, v)
        w = w - m * alpha / (np.sqrt(vh) + eps)
    cfg = {'name': 'Adam', 'learning_rate': lr, 'beta_1': b1, 'beta_2': b2, 'epsilon': eps, 'amsgrad': True}
    got = _run_oracle(cfg, W0, grads)
    assert np.allclose(got, w, rtol=1e-13, atol=1e-15)
    assert np.max(np.abs(_run_oracle(dict(cfg, amsgrad=False), W0, grads) - w)) > 1e-4


@pytest.mark.parametrize('name', ['SGD', 'RMSprop', 'Adamax', 'Adam'])
def test_decay_follows_the_per_variable_counters(name):
    """Keras-2 decay: lr_t = lr / (1 + decay * iterations), iterations = t - 1 of the variable being updated.  With the
    per-variable counters of Q2 (CDAE: t = 5(s-1)+j+1) variable j of step s sees lr / (1 + decay (5(s-1)+j))."""
    grads = _grads(6, seed=5)
    lr, decay, j = 0.01, 0.03, 3
    ts = [5 * (s - 1) + j + 1 for s in range(1, 7)]
    cfg = {'name': name, 'learning_rate': lr, 'decay': decay}
    got = _run_oracle(cfg, W0, grads, ts)
    w, a = W0.copy(), [np.zeros_like(W0) for _ in range(2)]
    for t, g in zip(ts, grads):
        lr_t = lr / (1 + decay * (t - 1))
        if name == 'SGD':
            w = w - lr_t * g
        elif name == 'RMSprop':
            a[0] = 0.9 * a[0] + 0.1 * g * g
            w = w - lr_t * g / (np.sqrt(a[0]) + 1e-7)
        elif name == 'Adamax':
            a[0] = a[0] + (g - a[0]) * 0.1
            a[1] = np.maximum(0.999 * a[1], np.abs(g))
            w = w - lr_t / (1 - 0.9 ** t) * (a[0] / (a[1] + 1e-7))
        else:
            a[0] = a[0] + (g - a[0]) * 0.1
            a[1] = a[1] + (g * g - a[1]) * 0.001
            w = w - lr_t * np.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t) * a[0] / (np.sqrt(a[1]) + 1e-7)
    assert np.allclose(got, w, rtol=1e-12, atol=1e-15)
    assert np.max(np.abs(_run_oracle(dict(cfg, decay=0.0), W0, grads, ts) - w)) > 1e-6


def test_oracle_adam_equals_adam_update_in_float32():
    from oracle.cdae import adam_update
    grads = [g.astype(np.float32) for g in _grads(9, seed=6)]
    w, m, v = W0.astype(np.float32), np.zeros(W0.shape, np.float32), np.zeros(W0.shape, np.float32)
    for t, g in enumerate(grads, 1):
        adam_update(w, m, v, g, 1e-3, t)
    opt = KerasOptimizer({'name': 'Adam'})
    w2 = W0.astype(np.float32)
    s = opt.slots(w2)
    for t, g in enumerate(grads, 1):
        opt.update(w2, s, g, t)
    assert np.array_equal(w, w2)


# ------------------------------------------------------------------ parsing (drecpy_b200.optimizers)
class _KerasStub:
    """What a tf.keras optimizer offers: get_config() with Keras-shaped keys (TensorFlow itself is not needed)."""

    def __init__(self, **config):
        self.config = config

    def get_config(self):
        return dict(self.config)


def test_default_and_unnamed_dicts_are_todays_adam():
    assert optimizers.parse(None, 0.005) == {'name': 'Adam', 'learning_rate': 0.005, 'beta_1': 0.9, 'beta_2': 0.999,
                                             'epsilon': 1e-7, 'amsgrad': False, 'decay': 0.0}
    o = optimizers.parse({'beta_2': 0.99, 'epsilon': 1e-8}, 0.01)
    assert (o['name'], o['learning_rate'], o['beta_1'], o['beta_2'], o['epsilon']) == ('Adam', 0.01, 0.9, 0.99, 1e-8)
    assert optimizers.parse({'learning_rate': 0.2}, 0.01)['learning_rate'] == 0.2
    # every Adam argument of an unnamed dict is honoured, decay and amsgrad included; other keys are refused
    o = optimizers.parse({'learning_rate': 0.01, 'decay': 1e-4, 'amsgrad': True}, 0.5)
    assert (o['name'], o['learning_rate'], o['decay'], o['amsgrad']) == ('Adam', 0.01, 1e-4, True)
    assert optimizers.parse({'lr': 0.03}, 0.5)['learning_rate'] == 0.03
    with pytest.raises(ValueError, match='momentum'):
        optimizers.parse({'momentum': 0.9})
    with pytest.raises(NotImplementedError, match='clipping'):
        optimizers.parse({'clipnorm': 1.0})


def test_named_dicts_take_the_keras_defaults():
    assert optimizers.parse({'name': 'SGD'}, 0.5) == {'name': 'SGD', 'learning_rate': 0.01, 'momentum': 0.0,
                                                      'nesterov': False, 'decay': 0.0}
    o = optimizers.parse({'name': 'rmsprop', 'momentum': 0.9, 'centered': True})
    assert o == {'name': 'RMSprop', 'learning_rate': 0.001, 'rho': 0.9, 'momentum': 0.9, 'epsilon': 1e-7,
                 'centered': True, 'decay': 0.0}
    assert optimizers.parse({'name': 'Adagrad'})['initial_accumulator_value'] == 0.1
    assert optimizers.parse({'name': 'Adamax', 'lr': 0.02})['learning_rate'] == 0.02
    assert optimizers.parse({'name': 'Adam', 'amsgrad': True, 'decay': 1e-4})['amsgrad'] is True


def test_keras_shaped_get_config_is_read():
    stub = _KerasStub(name='SGD', learning_rate=np.float32(0.1), decay=0.0, momentum=0.9, nesterov=True)
    assert optimizers.parse(stub) == {'name': 'SGD', 'learning_rate': float(np.float32(0.1)), 'momentum': 0.9,
                                      'nesterov': True, 'decay': 0.0}
    stub = _KerasStub(name='Adam', learning_rate=0.001, decay=0.0, beta_1=0.9, beta_2=0.999, epsilon=None,
                      amsgrad=False, clipnorm=None, global_clipnorm=None, clipvalue=None, weight_decay=None,
                      use_ema=False, ema_momentum=0.99, jit_compile=True, is_legacy_optimizer=False)
    assert optimizers.parse(stub) == optimizers.parse(None, 0.001)


@pytest.mark.parametrize('opt,match', [
    ({'name': 'SGD', 'learning_rate': {'class_name': 'ExponentialDecay', 'config': {}}}, 'schedules'),
    (_KerasStub(name='Adam', learning_rate=lambda: 0.1), 'schedules'),
    ({'name': 'Adam', 'clipnorm': 1.0}, 'clipping'),
    (_KerasStub(name='SGD', clipvalue=0.5), 'clipping'),
    ({'name': 'RMSprop', 'global_clipnorm': 2.0}, 'clipping'),
    ({'name': 'Nadam'}, 'Nadam'),
    (_KerasStub(name='Ftrl', learning_rate=0.001), 'Ftrl'),
    ({'name': 'Adadelta'}, 'Adadelta'),
    ({'name': 'AdamW', 'weight_decay': 0.004}, 'AdamW'),
    ({'name': 'Adam', 'weight_decay': 0.004}, 'weight_decay'),
    ('adam', 'neither a dict nor a Keras optimizer'),
])
def test_refusals_name_what_is_supported(opt, match):
    with pytest.raises(NotImplementedError, match=match) as e:
        optimizers.parse(opt)
    assert 'SGD' in str(e.value) and 'Adamax' in str(e.value) and 'Adagrad' in str(e.value)


def test_out_of_range_values_are_value_errors():
    for bad in ({'name': 'SGD', 'momentum': 1.5}, {'name': 'RMSprop', 'rho': -0.1}, {'name': 'Adamax', 'beta_1': 1.0},
                {'name': 'Adagrad', 'epsilon': 0.0}, {'name': 'Adam', 'decay': -1.0},
                {'name': 'Adagrad', 'initial_accumulator_value': -0.1}):
        with pytest.raises(ValueError):
            optimizers.parse(bad)


@pytest.mark.parametrize('cls', [drb.CDAE, drb.DMF])
def test_fit_refuses_before_touching_a_device(cls):
    u, i, v = drb.synthetic_interactions(30, 40, 300, seed=1)
    ds = drb.InteractionData(u, i, v)
    with pytest.raises(NotImplementedError, match='Nadam'):
        cls(verbose=False, seed=1).fit(ds, epochs=1, optimizer={'name': 'Nadam'})
    with pytest.raises(NotImplementedError, match='clipping'):
        cls(verbose=False, seed=1).fit(ds, epochs=1, optimizer=_KerasStub(name='Adam', clipnorm=1.0))


def test_native_descriptor_and_slots():
    d = optimizers.native_desc(optimizers.parse({'name': 'RMSprop', 'momentum': 0.5, 'centered': True}), 4096)
    assert (d.kind, d.centered, d.third_state) == (2, 1, 4096)
    assert abs(d.momentum - 0.5) < 1e-7 and abs(d.rho - 0.9) < 1e-7 and abs(d.epsilon - 1e-7) < 1e-13
    assert isinstance(d, _lib.OptimDesc)
    d = optimizers.native_desc({'learning_rate': 0.001, 'beta_1': 0.8, 'beta_2': 0.99, 'epsilon': 1e-8})   # an old dict
    assert (d.kind, d.amsgrad, d.decay) == (0, 0, 0.0) and abs(d.beta1 - 0.8) < 1e-7
    third = {'SGD': False, 'Adagrad': False, 'Adamax': False}
    for name, want in third.items():
        assert optimizers.needs_third_state({'name': name, **optimizers.parse({'name': name})}) is want
    assert optimizers.needs_third_state(optimizers.parse({'name': 'Adam', 'amsgrad': True}))
    assert optimizers.needs_third_state(optimizers.parse({'name': 'RMSprop', 'momentum': 0.1, 'centered': True}))
    assert not optimizers.needs_third_state(optimizers.parse({'name': 'RMSprop', 'centered': True}))
    assert optimizers.initial_m(optimizers.parse({'name': 'Adagrad', 'initial_accumulator_value': 0.25})) == 0.25
    assert optimizers.initial_m(optimizers.parse(None)) == 0.0
