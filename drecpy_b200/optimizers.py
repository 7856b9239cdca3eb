"""The `optimizer=` keyword of fit(): which Keras optimizers run natively, and how they reach the update kernel.

The reference's fit() takes any tf.keras optimizer (recommender_abc.py:153, applied per variable at :328-334).  This
package runs five of them in its dense update kernel (K4, csrc/optim.cu), with the Keras-2 / TF 2.0-2.3 OptimizerV2
semantics restated in include/drb.h (drb_optim_desc) and oracle/optim.py:

  SGD(learning_rate=0.01, momentum=0.0, nesterov=False)
  RMSprop(learning_rate=0.001, rho=0.9, momentum=0.0, epsilon=1e-7, centered=False)
  Adagrad(learning_rate=0.001, initial_accumulator_value=0.1, epsilon=1e-7)
  Adamax(learning_rate=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-7)
  Adam(learning_rate=0.001, beta_1=0.9, beta_2=0.999, epsilon=1e-7, amsgrad=False)

each with the Keras-2 `decay` (lr_t = lr / (1 + decay * iterations)).  fit(optimizer=...) accepts None (Adam with fit's
learning_rate), a dict without 'name' (overrides of that Adam: learning_rate, beta_1, beta_2, epsilon, amsgrad, decay;
other keys are refused), a dict with 'name', or any object with get_config() -- a tf.keras optimizer is read through its config, so TensorFlow
is never imported.  Learning-rate schedules, gradient clipping and every other optimizer raise NotImplementedError.
"""
import math

from . import _lib

DRB_OPT = {'Adam': 0, 'SGD': 1, 'RMSprop': 2, 'Adagrad': 3, 'Adamax': 4}

# Keras defaults per optimizer (every hyper-parameter the native update reads), before 'decay'
KERAS_DEFAULTS = {
    'SGD': {'learning_rate': 0.01, 'momentum': 0.0, 'nesterov': False},
    'RMSprop': {'learning_rate': 0.001, 'rho': 0.9, 'momentum': 0.0, 'epsilon': 1e-7, 'centered': False},
    'Adagrad': {'learning_rate': 0.001, 'initial_accumulator_value': 0.1, 'epsilon': 1e-7},
    'Adamax': {'learning_rate': 0.001, 'beta_1': 0.9, 'beta_2': 0.999, 'epsilon': 1e-7},
    'Adam': {'learning_rate': 0.001, 'beta_1': 0.9, 'beta_2': 0.999, 'epsilon': 1e-7, 'amsgrad': False},
}
_BOOL = ('nesterov', 'centered', 'amsgrad')
_CLIP = ('clipnorm', 'clipvalue', 'global_clipnorm')

SUPPORTED = ('drecpy_b200 runs these Keras optimizers natively: SGD (momentum, nesterov), RMSprop (rho, momentum, '
             'centered), Adagrad (initial_accumulator_value), Adamax and Adam (amsgrad), each with epsilon and the '
             'Keras-2 decay, with a constant learning rate and without gradient clipping.  Pass one of them (a tf.keras '
             'optimizer or a dict with its name and arguments), a dict of Adam overrides, or None')


def parse(opt, learning_rate=0.001):
    """The optimizer dict fit() keeps as self.optimizer: {'name', 'learning_rate', <hyper-parameters>, 'decay'}."""
    if opt is None or (isinstance(opt, dict) and 'name' not in opt):
        # overrides of the default Adam: learning_rate (default: fit's) and every Adam argument, decay and amsgrad
        # included; a key Adam does not have is refused rather than dropped
        opt = dict(opt or {})
        unknown = sorted(set(opt) - set(KERAS_DEFAULTS['Adam']) - {'lr', 'decay', *_CLIP})
        if unknown:
            raise ValueError(f'optimizer dict without a name holds Adam overrides; Adam has no {", ".join(unknown)} '
                             f'(give the dict a "name" for another optimizer).  {SUPPORTED}.')
        opt.setdefault('learning_rate', opt.pop('lr', learning_rate))
        opt['name'] = 'Adam'
    if isinstance(opt, dict):
        config = dict(opt)
    elif callable(getattr(opt, 'get_config', None)):
        config = dict(opt.get_config())
    else:
        raise NotImplementedError(f'optimizer {opt!r} is neither a dict nor a Keras optimizer.  {SUPPORTED}.')
    name = {k.lower(): k for k in KERAS_DEFAULTS}.get(str(config.get('name')).lower())
    if name is None:
        raise NotImplementedError(f"optimizer {config.get('name')!r} is not supported.  {SUPPORTED}.")
    for k in _CLIP:
        if config.get(k) is not None:
            raise NotImplementedError(f'{name}: gradient clipping ({k}={config[k]!r}) is not supported.  {SUPPORTED}.')
    if config.get('weight_decay') not in (None, 0, 0.0) or config.get('use_ema'):
        raise NotImplementedError(f'{name}: weight_decay and use_ema are not supported.  {SUPPORTED}.')
    lr = config.get('learning_rate', config.get('lr', KERAS_DEFAULTS[name]['learning_rate']))
    if isinstance(lr, dict) or callable(lr):
        raise NotImplementedError(f'{name}: learning-rate schedules ({lr!r}) are not supported.  {SUPPORTED}.')
    out = {'name': name, 'learning_rate': _number(name, 'learning_rate', lr)}
    for k, default in KERAS_DEFAULTS[name].items():
        if k == 'learning_rate':
            continue
        v = config.get(k, default)
        if v is None and k == 'epsilon':
            v = 1e-7                                              # Keras: epsilon=None means backend.epsilon()
        out[k] = bool(v) if k in _BOOL else _number(name, k, v)
    out['decay'] = _number(name, 'decay', config.get('decay', 0.0) or 0.0)
    _check_ranges(out)
    return out


def _number(name, key, v):
    try:
        x = float(v)
    except (TypeError, ValueError):
        raise NotImplementedError(f'{name}: {key}={v!r} is not a number.  {SUPPORTED}.') from None
    if not math.isfinite(x):
        raise ValueError(f'{name}: {key} must be finite (got {x})')
    return x


def _check_ranges(o):
    bad = []
    if o['learning_rate'] < 0 or o['decay'] < 0:
        bad.append('learning_rate and decay must be >= 0')
    if 'momentum' in o and not 0.0 <= o['momentum'] <= 1.0:
        bad.append('momentum must be in [0, 1]')
    if 'rho' in o and not 0.0 <= o['rho'] <= 1.0:
        bad.append('rho must be in [0, 1]')
    if 'beta_1' in o and not (0.0 <= o['beta_1'] < 1.0 and 0.0 <= o['beta_2'] < 1.0):
        bad.append('beta_1 and beta_2 must be in [0, 1)')
    if o['name'] not in ('SGD', 'Adam') and not o['epsilon'] > 0.0:
        bad.append('epsilon must be > 0')
    if o.get('initial_accumulator_value', 0.0) < 0.0:
        bad.append('initial_accumulator_value must be >= 0')
    if bad:
        raise ValueError(f"{o['name']}: " + '; '.join(bad))


def _named(o):
    """self.optimizer of any age (a dict without 'name' is the Adam of earlier versions) as a parsed dict."""
    return o if 'name' in o else parse(o, o.get('learning_rate', 0.001))


def needs_third_state(o):
    """AMSGrad's vhat and centered RMSprop's momentum live in a third arena; every other slot in adam_m / adam_v."""
    o = _named(o)
    return (o['name'] == 'Adam' and o['amsgrad']) or (o['name'] == 'RMSprop' and o['centered'] and o['momentum'] > 0)


def initial_m(o):
    """Initial value of the adam_m arena: Adagrad's accumulator starts at initial_accumulator_value, all else at 0."""
    o = _named(o)
    return o['initial_accumulator_value'] if o['name'] == 'Adagrad' else 0.0


def native_desc(o, third_state_ptr=None):
    """drb_optim_desc of an optimizer dict; third_state_ptr: device pointer of the third arena (or None)."""
    o = _named(o)
    d = _lib.OptimDesc()
    d.kind = DRB_OPT[o['name']]
    d.momentum = o.get('momentum', 0.0)
    d.nesterov = int(o.get('nesterov', False))
    d.rho = o.get('rho', 0.0)
    d.centered = int(o.get('centered', False))
    d.beta1, d.beta2 = o.get('beta_1', 0.0), o.get('beta_2', 0.0)
    d.epsilon = o.get('epsilon', 0.0)
    d.amsgrad = int(o.get('amsgrad', False))
    d.decay = o.get('decay', 0.0)
    d.third_state = third_state_ptr
    return d
