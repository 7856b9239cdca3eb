"""Caser (Tang & Wang, "Personalized Top-N Sequential Recommendation via Convolutional Sequence Embedding", WSDM 2018)
on the native B200 step -- the third of DRecPy's deep recommenders.

The model, its window sampler and its dropout stream are those of oracle/caser.py (float64); parity with DRecPy's
TensorFlow Caser and its MT19937 ListSampler is unpinned (DESIGN.md section 8).  A training step is one native call:
the batch of `batch_size` windows is drawn on the GPU (nothing crosses from the host), then the fused forward +
backward kernel, the dense update of the whole parameter arena and the loss.  Scoring uses the user representation
x = [z; P[u]] from the last L items of each user's training sequence and CDAE's exact scoring launches, so predict,
predict_batch, rank, recommend, recommend_batch and topk_batch give a user bit-identical scores.
Keyword init_weights={'E', 'P', 'Fv', 'bv', 'Fh' (list of L arrays [h, d, n_h]), 'bh' (list of L arrays [n_h]), 'fc',
'bfc', 'W2', 'b2'} injects every initial value (shapes of oracle.caser.CaserOracle).
"""
import ctypes as C
import random

import numpy as np

from . import _lib
from .dataset import _argsort_stable
from .recommender import DeepRecommenderABC


class Caser(DeepRecommenderABC):
    _SET_OPTIMIZER = 'drb_caser_set_optimizer'

    def __init__(self, L=5, T=3, d=50, n_v=4, n_h=16, dropout_rate=0.5, sort_column='timestamp', **kwds):
        super(Caser, self).__init__(**kwds)
        self.L, self.T, self.d, self.n_v, self.n_h = int(L), int(T), int(d), int(n_v), int(n_h)
        self.dropout_rate = float(dropout_rate)
        self.sort_column = sort_column
        if not 0.0 <= self.dropout_rate < 1.0:
            raise ValueError(f'Caser: dropout_rate must be in [0, 1) (got {dropout_rate})')
        lay = _lib.CaserLayout()
        lib = _lib.load()
        if lib.drb_caser_layout(1, 1, self.L, self.T, self.d, self.n_v, self.n_h, C.byref(lay)) != 0:
            raise ValueError(lib.drb_last_error().decode())
        self._init_weights = kwds.get('init_weights')
        self._native = None
        self._ctx = None

    # ------------------------------------------------------------------ sequences
    def _sequences(self):
        """(indptr [n_users + 1] int64, items int32): each user's rows with interaction >= interaction_threshold in
        (sort_column, row) order."""
        data = self._data
        sel = np.flatnonzero(data.interaction >= self.interaction_threshold) if self.interaction_threshold is not None \
            else np.arange(len(data))
        if self.sort_column is not None:
            ts = getattr(data, self.sort_column, None)
            if ts is None:
                raise ValueError(f'Caser: the dataset has no "{self.sort_column}" column to order the sequences by '
                                 f'(pass sort_column=None to use row order)')
            sel = sel[np.argsort(np.asarray(ts)[sel], kind='stable')]
        sel = sel[_argsort_stable(data.uid[sel])]
        indptr = np.zeros(self.n_users + 1, np.int64)
        np.cumsum(np.bincount(data.uid[sel], minlength=self.n_users), out=indptr[1:])
        return indptr, np.ascontiguousarray(data.iid[sel].astype(np.int32))

    # ------------------------------------------------------------------ setup
    def _pre_fit(self, learning_rate, neg_ratio, reg_rate, batch_size=32, **kwds):
        import torch
        self._torch = torch
        if not torch.cuda.is_available():
            raise RuntimeError('drecpy_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        if int(neg_ratio) != neg_ratio or neg_ratio < 0:
            raise ValueError(f'Caser: neg_ratio must be a non-negative integer (got {neg_ratio})')
        self.neg_ratio = int(neg_ratio)
        self._dev = torch.device(self.device or f'cuda:{torch.cuda.current_device()}')
        self._max_batch = int(max(batch_size, 32, min(1024, self.n_users)))
        indptr, seq = self._sequences()
        win = np.maximum(np.diff(indptr) - (self.L + self.T) + 1, 0)
        win_off = np.zeros(self.n_users + 1, np.int64)
        np.cumsum(win, out=win_off[1:])
        if win_off[-1] == 0:
            raise ValueError(f'Caser: no user has L + T = {self.L + self.T} training items to draw a window from')
        self._seq_host = (indptr, seq, win_off)
        lay = _lib.CaserLayout()
        _lib.check(_lib.load().drb_caser_layout(self.n_users, self.n_items, self.L, self.T, self.d, self.n_v, self.n_h,
                                                C.byref(lay)))
        self._L = lay
        self._params = torch.zeros(lay.total, dtype=torch.float32, device=self._dev)
        self._alloc_optimizer_slots()
        self._grads = torch.zeros_like(self._params)
        self._init(kwds.get('init_weights', self._init_weights))
        self._build_native()

    def weights(self, arena=None):
        """{name: view} into the parameter arena (or another arena of its layout, e.g. self._grads), shaped as the
        init_weights keyword takes them."""
        lay, d, L, n_h = self._L, self.d, self.L, self.n_h
        p = self._params if arena is None else arena
        F = self.n_v * d + n_h * L

        def v(off, rows, cols, ld=None):
            ld = ld or cols
            return p[off:off + rows * ld].view(rows, ld)[:, :cols]
        fh, bh, o = [], [], lay.off_fh
        for h in range(1, L + 1):
            fh.append(p[o:o + h * d * n_h].view(h, d, n_h))
            o += h * d * n_h
            bh.append(p[lay.off_bh + (h - 1) * n_h: lay.off_bh + h * n_h])
        return {'E': v(lay.off_e, self.n_items, d, lay.ld_e), 'P': v(lay.off_p, self.n_users, d, lay.ld_e),
                'Fv': v(lay.off_fv, L, self.n_v), 'bv': p[lay.off_bv:lay.off_bv + self.n_v], 'Fh': fh, 'bh': bh,
                'fc': v(lay.off_fc, F, d), 'bfc': p[lay.off_bfc:lay.off_bfc + d],
                'W2': v(lay.off_w2, self.n_items, 2 * d, lay.ld_x), 'b2': p[lay.off_b2:lay.off_b2 + self.n_items]}

    def _init(self, given):
        torch = self._torch
        gen = torch.Generator().manual_seed(abs(int(self.seed)) if self.seed is not None else random.getrandbits(62))
        d, L = self.d, self.L

        def normal(shape):                                  # N(0, (1/d)^2)
            return torch.randn(shape, generator=gen, dtype=torch.float32) / d

        def glorot(shape, fan_in, fan_out):                 # Keras Conv2D / Dense glorot_uniform
            lim = float(np.sqrt(6.0 / (fan_in + fan_out)))
            return (torch.rand(shape, generator=gen, dtype=torch.float32) * 2 - 1) * lim
        w = self.weights()
        F = self.n_v * d + self.n_h * L
        init = {'E': normal((self.n_items, d)), 'P': normal((self.n_users, d)),
                'Fv': glorot((L, self.n_v), L, L * self.n_v), 'bv': torch.zeros(self.n_v),
                'Fh': [glorot((h, d, self.n_h), h * d, h * d * self.n_h) for h in range(1, L + 1)],
                'bh': [torch.zeros(self.n_h) for _ in range(L)],
                'fc': glorot((F, d), F, d), 'bfc': torch.zeros(d),
                'W2': normal((self.n_items, 2 * d)), 'b2': torch.zeros(self.n_items)}
        for k, dst in w.items():
            src = (given or {}).get(k, init[k]) if given is not None else init[k]
            if given is not None and k not in given:
                raise KeyError(f'init_weights: "{k}" is missing')
            pairs = zip(dst, src) if isinstance(dst, list) else [(dst, src)]
            for dv, sv in pairs:
                sv = torch.as_tensor(np.asarray(sv), dtype=torch.float32)
                assert tuple(sv.shape) == tuple(dv.shape), f'init_weights["{k}"]: expected {tuple(dv.shape)}, got {tuple(sv.shape)}'
                dv.copy_(sv)

    def _build_native(self):
        torch = self._torch
        lib = _lib.load()
        dev = self._dev
        self._ctx = _lib.vp()
        _lib.check(lib.drb_ctx_create(dev.index or 0, C.byref(self._ctx)))
        self._stream = torch.cuda.current_stream(dev)
        _lib.check(lib.drb_ctx_set_stream(self._ctx, _lib.vp(self._stream.cuda_stream)))
        indptr, seq, win_off = self._seq_host
        s_ptr, s_idx, _ = self._data.csr()
        self._dev_seq = {k: torch.from_numpy(np.ascontiguousarray(a)).to(dev) for k, a in
                         (('indptr', indptr), ('seq', seq if len(seq) else np.zeros(1, np.int32)), ('win', win_off),
                          ('s_ptr', s_ptr), ('s_idx', s_idx if len(s_idx) else np.zeros(1, np.int32)))}
        ws = lib.drb_caser_workspace_bytes(self.n_users, self.n_items, self.L, self.T, self.d, self.n_v, self.n_h,
                                           self.neg_ratio, self._max_batch)
        if ws < 0:
            raise RuntimeError(f'libdrb error: {lib.drb_last_error().decode()}')
        self._workspace = torch.empty(ws, dtype=torch.uint8, device=dev)
        D = _lib.CaserDesc()
        D.n_users, D.n_items, D.L, D.T, D.d = self.n_users, self.n_items, self.L, self.T, self.d
        D.n_v, D.n_h, D.neg_ratio, D.dropout_rate = self.n_v, self.n_h, self.neg_ratio, self.dropout_rate
        D.params, D.adam_m, D.adam_v, D.grads = (self._params.data_ptr(), self._adam_m.data_ptr(),
                                                 self._adam_v.data_ptr(), self._grads.data_ptr())
        t = self._dev_seq
        D.seq, D.seq_indptr, D.win_off, D.n_windows = (t['seq'].data_ptr(), t['indptr'].data_ptr(), t['win'].data_ptr(),
                                                       int(win_off[-1]))
        D.seen_indptr, D.seen_indices = t['s_ptr'].data_ptr(), t['s_idx'].data_ptr()
        D.workspace, D.workspace_bytes, D.max_batch = self._workspace.data_ptr(), ws, self._max_batch
        self._native = _lib.vp()
        _lib.check(lib.drb_caser_create(self._ctx, C.byref(D), C.byref(self._native)))
        ptr = _lib.vp()
        _lib.check(lib.drb_caser_loss_buffer(self._native, C.byref(ptr)))
        off = ptr.value - self._workspace.data_ptr()
        self._loss_dev = self._workspace[off:off + 8].view(torch.float32)
        self._loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        self._apply_optimizer()

    def _params_tensor(self):
        return self._params

    def __getstate__(self):
        st = super(Caser, self).__getstate__()
        st.pop('_dev_seq', None)            # device copies of the sequences: rebuilt by _build_native on load
        return st

    # ------------------------------------------------------------------ training step
    def philox_seed(self):
        return abs(int(self.seed)) & 0xFFFFFFFFFFFFFFFF if self.seed is not None else 0

    def step_args(self, reg_rate):
        o = self.optimizer
        a = _lib.CaserStepArgs()
        a.learning_rate = o['learning_rate']
        a.beta1, a.beta2, a.epsilon = o.get('beta_1', 0.9), o.get('beta_2', 0.999), o.get('epsilon', 1e-7)
        a.reg_rate = reg_rate
        a.t = self._step
        a.philox_seed, a.philox_step = self.philox_seed(), self._step
        return a

    def _train_step(self, batch_size, reg_rate, want_loss=False, **kwds):
        with self._lock:
            args = self.step_args(reg_rate)
            _lib.check(_lib.load().drb_caser_step(self._native, int(batch_size), C.byref(args),
                                                  _lib.t_ptr(self._loss_dev)))
            if not want_loss:
                return None
            self._loss_host.copy_(self._loss_dev, non_blocking=True)
            self._stream.synchronize()
            return float(self._loss_host[0])

    def last_batch(self):
        """(users [B], items [B, L + T + T neg_ratio]) of the last step, as numpy arrays (tests)."""
        u, it, row = _lib.vp(), _lib.vp(), _lib.i32()
        _lib.check(_lib.load().drb_caser_batch_buffer(self._native, C.byref(u), C.byref(it), C.byref(row)))
        self.synchronize()
        n = self._max_batch
        torch = self._torch
        base = self._workspace.data_ptr()
        users = self._workspace[u.value - base:u.value - base + 4 * n].view(torch.int32).cpu().numpy()
        items = self._workspace[it.value - base:it.value - base + 4 * n * row.value].view(torch.int32)
        return users, items.view(n, row.value).cpu().numpy()

    def launch_count(self):
        return _lib.load().drb_ctx_launch_count(self._ctx)

    def synchronize(self):
        _lib.check(_lib.load().drb_ctx_synchronize(self._ctx))

    # ------------------------------------------------------------------ scoring
    def user_rep(self, uids):
        """x = [z; P[u]] for internal user ids, float32 [n, 2d]."""
        torch = self._torch
        with self._lock:
            u = torch.as_tensor(np.asarray(uids, np.int32), device=self._dev)
            out = torch.empty((len(u), self._L.ld_x), dtype=torch.float32, device=self._dev)
            for o in range(0, len(u), self._max_batch):
                n = min(self._max_batch, len(u) - o)
                _lib.check(_lib.load().drb_caser_user_rep(self._native, _lib.t_ptr(u[o:]), n, _lib.t_ptr(out[o:])))
            return out[:, :2 * self.d].cpu().numpy()

    def _predict(self, uid, iid=None, **kwds):
        if uid is None: return None
        torch = self._torch
        with self._lock:
            u = torch.tensor([uid], dtype=torch.int32, device=self._dev)
            out = torch.empty(self._L.items_pad, dtype=torch.float32, device=self._dev)
            _lib.check(_lib.load().drb_caser_predict_all(self._native, _lib.t_ptr(u), 1, _lib.t_ptr(out)))
            predictions = out[:self.n_items].cpu().numpy()
        return predictions if iid is None else predictions[iid]

    def _launch_predict_pairs(self, users, pair_off, pair_iid, pair_dst, out):
        _lib.check(_lib.load().drb_caser_predict_pairs(self._native, _lib.t_ptr(users), users.numel(),
                                                       _lib.t_ptr(pair_off), _lib.t_ptr(pair_iid), _lib.t_ptr(pair_dst),
                                                       out.numel(), _lib.t_ptr(out)))

    def _rank_batch(self, uids, cand, cand_count, novelty):
        torch = self._torch
        with self._lock:
            d_u = torch.as_tensor(np.ascontiguousarray(uids, np.int32), device=self._dev)
            d_c = torch.as_tensor(np.ascontiguousarray(cand, np.int32), device=self._dev)
            d_n = torch.as_tensor(np.ascontiguousarray(cand_count, np.int32), device=self._dev)
            n, max_c = d_c.shape
            o_i = torch.empty((n, max_c), dtype=torch.int32, device=self._dev)
            o_s = torch.empty((n, max_c), dtype=torch.float32, device=self._dev)
            o_n = torch.empty(n, dtype=torch.int32, device=self._dev)
            _lib.check(_lib.load().drb_caser_rank_candidates(self._native, _lib.t_ptr(d_u), n, _lib.t_ptr(d_c),
                                                             _lib.t_ptr(d_n), max_c, int(bool(novelty)),
                                                             _lib.t_ptr(o_i), _lib.t_ptr(o_s), _lib.t_ptr(o_n)))
            return o_i.cpu().numpy(), o_s.cpu().numpy(), o_n.cpu().numpy()

    def topk_batch(self, uids, k, novelty=True, return_device=False):
        """Full-catalog top-k for many users: (iids [n, k], scores [n, k], n_out [n]), 1 <= k <= 2048; row r is what
        _rank_batch returns for uids[r] over range(n_items), truncated to k, with the same score bits."""
        torch = self._torch
        k = int(k)
        with self._lock:
            d_u = uids if torch.is_tensor(uids) else torch.as_tensor(np.ascontiguousarray(uids, np.int32), device=self._dev)
            n = d_u.numel()
            o_i = torch.empty((n, k), dtype=torch.int32, device=self._dev)
            o_s = torch.empty((n, k), dtype=torch.float32, device=self._dev)
            o_n = torch.empty(n, dtype=torch.int32, device=self._dev)
            _lib.check(_lib.load().drb_caser_topk(self._native, _lib.t_ptr(d_u), n, k, int(bool(novelty)),
                                                  _lib.t_ptr(o_i), _lib.t_ptr(o_s), _lib.t_ptr(o_n)))
            if return_device:
                return o_i, o_s, o_n
            return o_i.cpu().numpy(), o_s.cpu().numpy(), o_n.cpu().numpy()

    def _topk_device_scores(self, uids, k, novelty):
        return self.topk_batch(uids, k, novelty, return_device=True)

    def _recommend(self, uid, n, novelty, threshold):
        if n <= 2048:
            o_i, o_s, o_n = self.topk_batch(np.array([uid], np.int32), int(n), novelty)
            ranked = [(o_s[0, j], int(o_i[0, j])) for j in range(int(o_n[0]))]
        else:
            ranked = self._rank(uid, range(self.n_items), n, novelty)
        if threshold is None:
            return ranked
        return [x for x in ranked if x[0] >= threshold]
