"""Oracle restatement of the Keras optimizers fit(optimizer=...) accepts (numpy; test infrastructure).

PARITY UNPINNED (TensorFlow absent, see oracle/__init__.py).  Restates the Keras-2 / TF 2.0-2.3 OptimizerV2 dense
updates, one apply_gradients per variable (recommender_abc.py:328-334), g = gradient with the L2 term folded in:
  SGD      momentum == 0: ResourceApplyGradientDescent  w -= lr_t g
           momentum > 0:  ResourceApplyKerasMomentum    a = a momentum - lr_t g; w += a  (nesterov: w += a momentum - lr_t g)
  RMSprop  momentum == 0: the Python branch of _resource_apply_dense
                          ms = rho ms + (1-rho) g^2; centered: mg = rho mg + (1-rho) g, d = ms - mg^2, else d = ms;
                          w -= lr_t g / (sqrt(d) + eps)
           momentum > 0:  ApplyRMSProp / ApplyCenteredRMSProp (eps inside the square root)
                          ms += (g^2 - ms)(1-rho); centered: mg += (g - mg)(1-rho), d = ms - mg^2 + eps, else
                          d = ms + eps; mom = mom momentum + lr_t g / sqrt(d); w -= mom
  Adagrad  ResourceApplyAdagradV2: acc (starts at initial_accumulator_value) += g^2; w -= lr_t g / (sqrt(acc) + eps)
  Adamax   ResourceApplyAdaMax: m += (g - m)(1-b1); u = max(b2 u, |g|); w -= lr_t / (1 - b1^t) (m / (u + eps))
  Adam     ResourceApplyAdam (oracle.cdae.adam_update); amsgrad: ResourceApplyAdamWithAmsgrad, vhat = max(vhat, v),
           w -= (m alpha_t) / (sqrt(vhat) + eps)
lr_t = lr / (1 + decay (t - 1)) (Keras-2 decay; t - 1 = the optimizer's iterations before this update).  Every
scalar and element operation runs in the dtype of the arrays passed (float32 for the parity tests; float64 lets tests
compare the formulas with torch.optim).  CDAEOptimOracle / CDAESampledOptimOracle / DMFOptimOracle (below) are the
training-step oracles with one of these optimizers in place of their default Adam.
"""
import numpy as np

KERAS_DEFAULTS = {
    'SGD': {'learning_rate': 0.01, 'momentum': 0.0, 'nesterov': False},
    'RMSprop': {'learning_rate': 0.001, 'rho': 0.9, 'momentum': 0.0, 'epsilon': 1e-7, 'centered': False},
    'Adagrad': {'learning_rate': 0.001, 'initial_accumulator_value': 0.1, 'epsilon': 1e-7},
    'Adamax': {'learning_rate': 0.001, 'beta_1': 0.9, 'beta_2': 0.999, 'epsilon': 1e-7},
    'Adam': {'learning_rate': 0.001, 'beta_1': 0.9, 'beta_2': 0.999, 'epsilon': 1e-7, 'amsgrad': False},
}


class KerasOptimizer:
    """config: {'name': one of KERAS_DEFAULTS, hyper-parameters (Keras defaults where missing), 'decay'}."""

    def __init__(self, config):
        self.name = config['name']
        self.c = dict(KERAS_DEFAULTS[self.name], decay=0.0)
        self.c.update({k: v for k, v in config.items() if k != 'name'})

    def slots(self, w):
        """The slot arrays of variable w, in the order update() reads them."""
        c, z = self.c, (lambda: np.zeros_like(w))
        if self.name == 'SGD':
            return [z()] if c['momentum'] > 0 else []
        if self.name == 'RMSprop':
            return [z()] + ([z()] if c['centered'] else []) + ([z()] if c['momentum'] > 0 else [])
        if self.name == 'Adagrad':
            return [np.full_like(w, c['initial_accumulator_value'])]
        if self.name == 'Adamax':
            return [z(), z()]
        return [z(), z()] + ([z()] if c['amsgrad'] else [])

    def lr_t(self, t, dt):
        lr = dt(self.c['learning_rate'])
        if self.c['decay']:
            lr = lr / (dt(1) + dt(self.c['decay']) * dt(t - 1))
        return lr

    def update(self, w, s, g, t):
        """One dense update of w (in place) with gradient g at per-variable step t (= iterations + 1)."""
        dt, c = w.dtype.type, self.c
        lr = self.lr_t(t, dt)
        one = dt(1)
        if self.name == 'SGD':
            mom = dt(c['momentum'])
            if c['momentum'] == 0:
                w -= lr * g
                return
            a = s[0]
            a[...] = a * mom - lr * g
            w += a * mom - lr * g if c['nesterov'] else a
        elif self.name == 'RMSprop':
            rho, eps, mom = dt(c['rho']), dt(c['epsilon']), dt(c['momentum'])
            ms = s[0]
            if c['momentum'] == 0:
                ms[...] = rho * ms + (one - rho) * (g * g)
                d = ms
                if c['centered']:
                    mg = s[1]
                    mg[...] = rho * mg + (one - rho) * g
                    d = ms - mg * mg
                w -= lr * g / (np.sqrt(d) + eps)
                return
            ms += (g * g - ms) * (one - rho)
            d = ms + eps
            if c['centered']:
                mg = s[1]
                mg += (g - mg) * (one - rho)
                d = ms - mg * mg + eps
            mv = s[-1]
            mv[...] = mv * mom + lr * g / np.sqrt(d)
            w -= mv
        elif self.name == 'Adagrad':
            acc = s[0]
            acc += g * g
            w -= lr * g / (np.sqrt(acc) + dt(c['epsilon']))
        elif self.name == 'Adamax':
            b1, b2, eps = dt(c['beta_1']), dt(c['beta_2']), dt(c['epsilon'])
            m, u = s
            m += (g - m) * (one - b1)
            u[...] = np.maximum(b2 * u, np.abs(g))
            w -= lr / (one - np.power(b1, dt(t), dtype=w.dtype)) * (m / (u + eps))
        else:
            b1, b2, eps = dt(c['beta_1']), dt(c['beta_2']), dt(c['epsilon'])
            alpha = lr * np.sqrt(one - np.power(b2, dt(t), dtype=w.dtype), dtype=w.dtype) / \
                (one - np.power(b1, dt(t), dtype=w.dtype))
            m, v = s[0], s[1]
            m += (g - m) * (one - b1)
            v += (g * g - v) * (one - b2)
            if c['amsgrad']:
                vh = s[2]
                np.maximum(vh, v, out=vh)
                w -= (m * alpha) / (np.sqrt(vh) + eps)
            else:
                w -= alpha * m / (np.sqrt(v) + eps)


# ---------------------------------------------------------------------------------------------------------------------
# The CDAE / DMF oracles with an optimizer other than their default Adam: same forward / backward (grads), same
# per-variable step counters (Q2), the update of `optimizer` (a config dict as above) instead of adam_update.
from .cdae import CDAEOracle, CDAESampledOracle, F     # noqa: E402
from .dmf import DMFOracle                             # noqa: E402


class _WithOptimizer:
    def _init_optimizer(self, optimizer, variables):
        self.opt = KerasOptimizer(optimizer)
        self.slots = [self.opt.slots(x) for x in variables]

    def _apply_cdae(self, grads):
        self.step_count += 1
        s = self.step_count
        for j, (w, g) in enumerate(zip(self.vars, grads)):
            t = 5 * (s - 1) + j + 1 if self.adam_t == 'per_variable' else s     # Q2
            self.opt.update(w, self.slots[j], g.astype(F), t)


class CDAEOptimOracle(_WithOptimizer, CDAEOracle):
    def __init__(self, *args, optimizer, **kw):
        super().__init__(*args, **kw)
        self._init_optimizer(optimizer, self.vars)

    def step(self, uids, keep, reg_rate):
        total, grads = self.grads(uids, keep, reg_rate)
        self._apply_cdae(grads)
        return total


class CDAESampledOptimOracle(_WithOptimizer, CDAESampledOracle):
    def __init__(self, *args, optimizer, **kw):
        super().__init__(*args, **kw)
        self._init_optimizer(optimizer, self.vars)

    def step_sampled(self, uids, keep, reg_rate, step):
        total, grads = self.grads_sampled(uids, keep, reg_rate, step)
        self._apply_cdae(grads)
        return total


class DMFOptimOracle(_WithOptimizer, DMFOracle):
    """Variables in the order [user tower (kernel, bias) per layer, item tower (kernel, bias) per layer]."""

    def __init__(self, *args, optimizer, **kw):
        super().__init__(*args, **kw)
        self._init_optimizer(optimizer, [x for g in self.groups for kb in g for x in kb])

    def step(self, uids, iids, labels, reg_rate):
        total, all_grads = self.grads(uids, iids, labels, reg_rate)
        self.step_count += 1
        s = self.step_count
        j = 0
        for gidx, (layers, grads) in enumerate(zip(self.groups, all_grads)):
            t = 2 * (s - 1) + gidx + 1 if self.adam_t == 'per_variable' else s      # Q2: one counter per tower
            for (k, b), (gk, gb) in zip(layers, grads):
                self.opt.update(k, self.slots[j], gk.astype(F), t)
                self.opt.update(b, self.slots[j + 1], gb.astype(F), t)
                j += 2
        return total
