"""Float64 restatement of Caser (Tang & Wang, WSDM 2018) as drecpy_b200.Caser trains and scores it (test infrastructure).

PARITY WITH DRecPy's TensorFlow Caser UNPINNED: DRecPy's caser.py / list_sampler.py are not in this tree, and its
ListSampler cannot run on Python >= 3.11 (rng.sample on a set).  This module is the definition the kernels are held to
(drecpy_b200/csrc/caser.cu), as CDAESampledOracle is for the sampled-output extension of CDAE:
  sequences   a user's training rows with interaction >= threshold, sorted by (sort column, row order)
  batch       example b: window idx = (philox(0, b) << 32 | philox(1, b)) mod n_windows over all (user, start) windows of
              L + T consecutive items (binary search in the per-user prefix sums); L inputs, T targets (label 1);
              T * neg_ratio negatives, item = philox(q * 32 + a, b) mod n_items, redrawn while stored for the user,
              a < 32, the last attempt kept.  Counter (c0, b, step_lo, step_hi), key (seed_lo ^ salt, seed_hi).
  dropout     element e of c = [vertical (c d + k); pooled horizontal ((h - 1) n_h + f)]: kept when
              u = (philox(e, b) >> 8) 2^-24 >= rate, then scaled by 1 / (1 - rate); training only
  forward     E^ = E[S]; o~ = Fv^T E^ + bv; o[h, f] = max_i relu(<E^[i:i+h], Fh_h[:, :, f]> + bh_h[f]);
              z = relu(c W_fc + b_fc); x = [z; P[u]]; y_j = x . W2[j] + b2[j]
  loss        Keras-2 BCE over sigmoid(y), mean over B T (1 + neg_ratio) terms, plus reg sum w^2 over E, P, Fv, Fh, fc, W2
  update      the Keras rule of oracle/optim.py per tensor, g = gradient + 2 reg w, t = step for every tensor
"""
import numpy as np

from .philox import philox_first
from .optim import KerasOptimizer

KERAS_EPS = 1e-7
SALT_WINDOW, SALT_NEG, SALT_DROP = 0x9E3779B9, 0x3C6EF372, 0xDAA66D2B
L2_TENSORS = ('E', 'P', 'Fv', 'Fh', 'fc', 'W2')


def sequences(uid, iid, interaction, n_users, threshold=None, sort_values=None):
    """(indptr [n_users + 1], items): each user's rows with interaction >= threshold, sorted by (sort value, row)."""
    seqs = [[] for _ in range(n_users)]
    rows = [r for r in range(len(uid)) if threshold is None or interaction[r] >= threshold]
    key = (lambda r: (sort_values[r], r)) if sort_values is not None else (lambda r: r)
    for r in sorted(rows, key=key):
        seqs[uid[r]].append(int(iid[r]))
    indptr = np.zeros(n_users + 1, np.int64)
    indptr[1:] = np.cumsum([len(s) for s in seqs])
    return indptr, np.array([x for s in seqs for x in s], np.int32)


def window_offsets(indptr, L, T):
    n = np.maximum(np.diff(indptr) - (L + T) + 1, 0)
    off = np.zeros(len(n) + 1, np.int64)
    off[1:] = np.cumsum(n)
    return off


def _philox(c0, b, step, seed, salt):
    c0 = np.asarray(c0, np.uint32)
    return philox_first(c0, np.full_like(c0, b), np.full_like(c0, step & 0xFFFFFFFF), np.full_like(c0, step >> 32),
                        (seed & 0xFFFFFFFF) ^ salt, seed >> 32)


def sample_batch(indptr, seq, win_off, seen, n_items, L, T, neg_ratio, batch, seed, step):
    """(users [B], items [B, L + T + T neg_ratio]) of one step; seen = (indptr, sorted indices) of all stored rows."""
    n_win = int(win_off[-1])
    users = np.zeros(batch, np.int32)
    items = np.zeros((batch, L + T + T * neg_ratio), np.int32)
    s_ptr, s_idx = seen
    for b in range(batch):
        hi = int(_philox([0], b, step, seed, SALT_WINDOW)[0])
        lo = int(_philox([1], b, step, seed, SALT_WINDOW)[0])
        idx = ((hi << 32) | lo) % n_win
        u = int(np.searchsorted(win_off, idx, side='right') - 1)
        start = idx - int(win_off[u])
        users[b] = u
        items[b, :L + T] = seq[indptr[u] + start: indptr[u] + start + L + T]
        stored = set(s_idx[s_ptr[u]:s_ptr[u + 1]].tolist())
        for q in range(T * neg_ratio):
            draws = _philox(np.arange(32) + q * 32, b, step, seed, SALT_NEG) % np.uint32(n_items)
            item = int(draws[-1])
            for x in draws.tolist():
                if x not in stored:
                    item = x
                    break
            items[b, L + T + q] = item
    return users, items


def dropout_scale(n_elems, batch, seed, step, rate):
    """[B, n_elems] factors: 1 / (1 - rate) where kept, 0 where dropped (all ones when rate == 0)."""
    out = np.ones((batch, n_elems))
    if rate <= 0:
        return out
    for b in range(batch):
        x = _philox(np.arange(n_elems), b, step, seed, SALT_DROP)
        u = (x >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
        out[b] = np.where(u >= np.float32(rate), 1.0 / (1.0 - rate), 0.0)
    return out


class CaserOracle:
    """w: {'E' [I, d], 'P' [U, d], 'Fv' [L, n_v], 'bv' [n_v], 'Fh': [h x d x n_h for h = 1..L], 'bh': [n_h] * L,
    'fc' [n_v d + n_h L, d], 'bfc' [d], 'W2' [I, 2d], 'b2' [I]} (copied to float64)."""

    def __init__(self, w, optimizer=None):
        self.w = {k: ([np.array(x, np.float64) for x in v] if isinstance(v, (list, tuple)) else np.array(v, np.float64))
                  for k, v in w.items()}
        self.L, self.n_v = self.w['Fv'].shape
        self.d = self.w['E'].shape[1]
        self.n_h = self.w['bh'][0].shape[0]
        self.opt = KerasOptimizer(optimizer or {'name': 'Adam'})
        self.slots = {k: ([self.opt.slots(x) for x in v] if isinstance(v, list) else self.opt.slots(v))
                      for k, v in self.w.items()}
        self.step_count = 0

    def forward(self, users, inputs, scale=None):
        """inputs [B, L] item ids (-1: zero row); scale [B, F] dropout factors or None.  x [B, 2d] and the cache."""
        w, L, d = self.w, self.L, self.d
        eh = np.where((inputs >= 0)[:, :, None], w['E'][np.maximum(inputs, 0)], 0.0)              # [B, L, d]
        ov = np.einsum('lc,bld->bcd', w['Fv'], eh) + w['bv'][None, :, None]                       # [B, n_v, d]
        oh, amax = [], []
        for h in range(1, L + 1):
            conv = np.stack([np.einsum('bqd,qdf->bf', eh[:, i:i + h], w['Fh'][h - 1]) for i in range(L - h + 1)], 1)
            conv = conv + w['bh'][h - 1][None, None, :]                                          # [B, L-h+1, n_h]
            am = conv.argmax(axis=1)
            best = np.take_along_axis(conv, am[:, None, :], 1)[:, 0]
            oh.append(np.maximum(best, 0.0))
            amax.append(np.where(best > 0, am, -1))
        c0 = np.concatenate([ov.reshape(len(users), -1)] + oh, axis=1)                           # [B, F]
        c = c0 * scale if scale is not None else c0
        z = np.maximum(c @ w['fc'] + w['bfc'], 0.0)
        x = np.concatenate([z, w['P'][users]], axis=1)
        return x, dict(eh=eh, c=c, z=z, amax=amax, scale=scale)

    def scores(self, x, items):
        return np.einsum('bk,bjk->bj', x, self.w['W2'][items]) + self.w['b2'][items]

    def loss_and_grads(self, users, items, L, T, scale, reg_rate):
        """Reported loss and the raw gradients (without the L2 term) of one batch."""
        w, d, n_v, n_h = self.w, self.d, self.n_v, self.n_h
        B = len(users)
        inputs, tgt = items[:, :L], items[:, L:]
        x, cache = self.forward(users, inputs, scale)
        y = self.scores(x, tgt)
        t = np.zeros_like(y)
        t[:, :T] = 1.0
        p = 1.0 / (1.0 + np.exp(-y))
        pc = np.clip(p, KERAS_EPS, 1 - KERAS_EPS)
        n = y.size
        data = -(t * np.log(pc + KERAS_EPS) + (1 - t) * np.log(1 - pc + KERAS_EPS)).sum() / n
        inside = (p >= KERAS_EPS) & (p <= 1 - KERAS_EPS)
        gy = np.where(inside, -(t / (pc + KERAS_EPS) - (1 - t) / (1 - pc + KERAS_EPS)) / n * p * (1 - p), 0.0)
        g = {k: ([np.zeros_like(x_) for x_ in v] if isinstance(v, list) else np.zeros_like(v)) for k, v in w.items()}
        W2t = w['W2'][tgt]                                                # [B, J, 2d]
        np.add.at(g['W2'], tgt, gy[:, :, None] * x[:, None, :])
        np.add.at(g['b2'], tgt, gy)
        dx = np.einsum('bj,bjk->bk', gy, W2t)
        np.add.at(g['P'], users, dx[:, d:])
        dz = dx[:, :d] * (cache['z'] > 0)
        g['bfc'] = dz.sum(0)
        g['fc'] = cache['c'].T @ dz
        dc = dz @ w['fc'].T
        if cache['scale'] is not None:
            dc = dc * cache['scale']
        eh = cache['eh']
        dov = dc[:, :n_v * d].reshape(B, n_v, d)
        g['Fv'] = np.einsum('bcd,bld->lc', dov, eh)
        g['bv'] = dov.sum(axis=(0, 2))
        deh = np.einsum('lc,bcd->bld', w['Fv'], dov)
        for h in range(1, self.L + 1):
            do = dc[:, n_v * d + (h - 1) * n_h: n_v * d + h * n_h]        # [B, n_h]
            am = cache['amax'][h - 1]
            act = am >= 0
            g['bh'][h - 1] = (do * act).sum(0)
            for b in range(B):
                for f in np.flatnonzero(act[b]):
                    i0 = am[b, f]
                    g['Fh'][h - 1][:, :, f] += do[b, f] * eh[b, i0:i0 + h]
                    deh[b, i0:i0 + h] += do[b, f] * w['Fh'][h - 1][:, :, f]
        np.add.at(g['E'], inputs, deh)
        reg = reg_rate * sum((x_ ** 2).sum() for k in L2_TENSORS for x_ in (w[k] if isinstance(w[k], list) else [w[k]]))
        return data + reg, g, data

    def step(self, users, items, L, T, scale, reg_rate):
        """One training step on a given batch: the loss before the update."""
        loss, g, _ = self.loss_and_grads(users, items, L, T, scale, reg_rate)
        self.step_count += 1
        t = self.step_count
        for k, v in self.w.items():
            reg = 2 * reg_rate if k in L2_TENSORS else 0.0
            if isinstance(v, list):
                for j, x_ in enumerate(v):
                    self.opt.update(x_, self.slots[k][j], g[k][j] + reg * x_, t)
            else:
                self.opt.update(v, self.slots[k], g[k] + reg * v, t)
        return loss

    def user_inputs(self, indptr, seq, uids):
        """[n, L] the last L items of each sequence, left-padded with -1."""
        out = np.full((len(uids), self.L), -1, np.int64)
        for r, u in enumerate(uids):
            s = seq[indptr[u]:indptr[u + 1]][-self.L:]
            if len(s):
                out[r, self.L - len(s):] = s
        return out

    def predict_all(self, indptr, seq, uids):
        """sigmoid scores [n, n_items] without dropout."""
        x, _ = self.forward(np.asarray(uids), self.user_inputs(indptr, seq, uids))
        return 1.0 / (1.0 + np.exp(-(x @ self.w['W2'].T + self.w['b2'])))
