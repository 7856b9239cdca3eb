"""DMF (Deep Matrix Factorization) on the native B200 step -- drop-in for DRecPy's DMF.

Mirrors DRecPy/Recommender/dmf.py: constructor :22-44 (same asserts), _pre_fit :46-62 (two Dense(relu) towers,
Glorot kernels, zero biases, l2(reg) on kernels), _sample_batch :64-73 (labels (r-min)/(max-min) when use_nce),
_preprocess_input :75-86 (raw-valued rows / columns, l2-normalised when l2_norm_vectors) and
_predict_batch / _compute_batch_loss :88-99 (now drb_dmf_step), _predict :101-106.
Keyword init_weights={'user_nn': [(kernel, bias), ...], 'item_nn': [...]} injects initial weights (Keras shapes:
kernel [in, out], bias [out]); adam_t='per_variable' keeps the reference's per-tower Adam step counter (Q2).
"""
import ctypes as C
import random

import numpy as np

from . import _lib
from .parallel import DataParallel
from .recommender import DeepRecommenderABC
from .sampler import PointSampler

_RING = 4


class DMF(DeepRecommenderABC):
    def __init__(self, user_factors=None, item_factors=None, use_nce=True, l2_norm_vectors=True, **kwds):
        super(DMF, self).__init__(**kwds)
        self.user_factors = user_factors
        if self.user_factors is None:
            self.user_factors = [64, 32]
        assert type(self.user_factors) is list, 'The "user_factors" argument must be of type list (ex: [64, 32]).'
        assert len(self.user_factors) > 0, 'The "user_factors" argument must have at least 1 element.'
        self.item_factors = item_factors
        if self.item_factors is None:
            self.item_factors = [64, 32]
        assert type(self.item_factors) is list, 'The "item_factors" argument must be of type list (ex: [64, 32]).'
        assert len(self.item_factors) > 0, 'The "item_factors" argument must have at least 1 element.'
        assert self.user_factors[-1] == self.item_factors[-1], \
            f'The last user and item factors dimension must be equal ({self.user_factors[-1]} != {self.item_factors[-1]})'
        self.use_nce = use_nce
        self.l2_norm_vectors = l2_norm_vectors
        self.adam_t = kwds.get('adam_t', 'per_variable')
        self._native = None
        self._ctx = None

    # ------------------------------------------------------------------ setup
    def _pre_fit(self, learning_rate, neg_ratio, reg_rate, batch_size=32, **kwds):
        import torch
        self._torch = torch
        if not torch.cuda.is_available():
            raise RuntimeError('drecpy_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        self._dev = torch.device(self.device or f'cuda:{torch.cuda.current_device()}')
        self._max_batch = int(max(batch_size, min(1024, max(self.n_users, self.n_items)), kwds.get('score_batch', 0)))
        # data parallel over pair mini-batches: batch_size is PER RANK; replicated weights, one gradient all-reduce
        self._dp = kwds.get('data_parallel') or DataParallel()
        self._alloc_and_init(kwds.get('init_weights', None))
        self._build_native()
        self._sampler = kwds.get('sampler') or PointSampler(self._data, neg_ratio, self.interaction_threshold, self.seed)
        self._slots = []
        for _ in range(_RING):
            s = {'uid': torch.empty(batch_size, dtype=torch.int32).pin_memory(),
                 'iid': torch.empty(batch_size, dtype=torch.int32).pin_memory(),
                 'lab': torch.empty(batch_size, dtype=torch.float32).pin_memory(),
                 'val': np.empty(batch_size, np.float64), 'event': None}
            s['uid_np'], s['iid_np'], s['lab_np'] = s['uid'].numpy(), s['iid'].numpy(), s['lab'].numpy()
            self._slots.append(s)
        self._slot_idx = 0
        self._loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        self._next = None

    def _factor_arrays(self):
        uf = (C.c_int32 * len(self.user_factors))(*self.user_factors)
        itf = (C.c_int32 * len(self.item_factors))(*self.item_factors)
        return uf, itf

    def _alloc_and_init(self, init_weights):
        torch = self._torch
        lib = _lib.load()
        uf, itf = self._factor_arrays()
        L = _lib.DmfLayout()
        _lib.check(lib.drb_dmf_layout(self.n_users, self.n_items, uf, len(self.user_factors), itf,
                                      len(self.item_factors), C.byref(L)))
        self._L = L
        self._params = torch.zeros(L.total, dtype=torch.float32, device=self._dev)
        self._adam_m = torch.zeros_like(self._params)
        self._adam_v = torch.zeros_like(self._params)
        self._grads = torch.zeros_like(self._params)
        gen = torch.Generator().manual_seed(abs(int(self.seed)) if self.seed is not None else random.getrandbits(62))
        for name, factors in (('user_nn', self.user_factors), ('item_nn', self.item_factors)):
            given = (init_weights or {}).get(name)
            for l, (k_view, b_view) in enumerate(self.tower_weights(name)):
                if given is not None:
                    k = torch.as_tensor(np.asarray(given[l][0]), dtype=torch.float32)
                    b = torch.as_tensor(np.asarray(given[l][1]), dtype=torch.float32)
                    assert tuple(k.shape) == tuple(k_view.shape), f'{name}[{l}] kernel: expected {tuple(k_view.shape)}'
                else:                                   # Keras Dense defaults: glorot_uniform kernel, zero bias
                    fan_in, fan_out = k_view.shape
                    lim = float(np.sqrt(6.0 / (fan_in + fan_out)))
                    k = (torch.rand((fan_in, fan_out), generator=gen, dtype=torch.float32) * 2 - 1) * lim
                    b = torch.zeros(fan_out)
                k_view.copy_(k)
                b_view.copy_(b)

    def tower_weights(self, name):
        """[(kernel [in, out], bias [out])] views into the parameter arena, Keras-shaped."""
        L = self._L
        user = name == 'user_nn'
        factors = self.user_factors if user else self.item_factors
        offs_k = L.off_kernel_user if user else L.off_kernel_item
        offs_b = L.off_bias_user if user else L.off_bias_item
        lds = L.ld_user if user else L.ld_item
        in_dim = self.n_items if user else self.n_users
        out = []
        for l, f in enumerate(factors):
            k = self._params[offs_k[l]:offs_k[l] + in_dim * lds[l]].view(in_dim, lds[l])[:, :f]
            b = self._params[offs_b[l]:offs_b[l] + f]
            out.append((k, b))
            in_dim = f
        return out

    def _build_native(self):
        torch = self._torch
        lib = _lib.load()
        dev = self._dev
        self._ctx = _lib.vp()
        _lib.check(lib.drb_ctx_create(dev.index or 0, C.byref(self._ctx)))
        self._stream = torch.cuda.current_stream(dev)
        _lib.check(lib.drb_ctx_set_stream(self._ctx, _lib.vp(self._stream.cuda_stream)))
        self._dev_sparse = {}
        for name, (indptr, indices, data) in (('csr', self._data.csr()), ('csc', self._data.csc())):
            vals = data.astype(np.float32)                    # tf.convert_to_tensor(..., dtype=tf.float32), dmf.py:79
            t = {'indptr': torch.from_numpy(np.ascontiguousarray(indptr)).to(dev),
                 'indices': torch.from_numpy(np.ascontiguousarray(indices)).to(dev),
                 'values': torch.from_numpy(vals).to(dev), 'scale': None}
            if self.l2_norm_vectors:                          # x * rsqrt(max(sum x^2, 1e-12)), dmf.py:82-84
                ss = np.zeros(len(indptr) - 1, np.float32)
                rows = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))
                np.add.at(ss, rows, vals * vals)
                scale = (np.float32(1) / np.sqrt(np.maximum(ss, np.float32(1e-12)))).astype(np.float32)
                t['scale'] = torch.from_numpy(scale).to(dev)
            self._dev_sparse[name] = t
        uf, itf = self._factor_arrays()
        ws_bytes = lib.drb_dmf_workspace_bytes(self.n_users, self.n_items, uf, len(self.user_factors), itf,
                                               len(self.item_factors), self._max_batch)
        assert ws_bytes > 0
        self._workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        d = _lib.DmfDesc()
        d.n_users, d.n_items = self.n_users, self.n_items
        d.n_layers_user, d.n_layers_item = len(self.user_factors), len(self.item_factors)
        for l, f in enumerate(self.user_factors): d.user_factors[l] = f
        for l, f in enumerate(self.item_factors): d.item_factors[l] = f
        d.params, d.adam_m, d.adam_v, d.grads = (self._params.data_ptr(), self._adam_m.data_ptr(),
                                                 self._adam_v.data_ptr(), self._grads.data_ptr())
        for name in ('csr', 'csc'):
            t = self._dev_sparse[name]
            setattr(d, f'{name}_indptr', t['indptr'].data_ptr())
            setattr(d, f'{name}_indices', t['indices'].data_ptr())
            setattr(d, f'{name}_values', t['values'].data_ptr())
            setattr(d, f'{name}_row_scale', t['scale'].data_ptr() if t['scale'] is not None else None)
        d.workspace, d.workspace_bytes, d.max_batch = self._workspace.data_ptr(), ws_bytes, self._max_batch
        self._native = _lib.vp()
        _lib.check(lib.drb_dmf_create(self._ctx, C.byref(d), C.byref(self._native)))
        ptr = _lib.vp()
        _lib.check(lib.drb_dmf_loss_buffer(self._native, C.byref(ptr)))
        off = ptr.value - self._workspace.data_ptr()
        self._loss_dev = self._workspace[off:off + 8].view(torch.float32)

    def _params_tensor(self):
        return self._params

    # ------------------------------------------------------------------ training step
    def step_args(self, reg_rate):
        o = self.optimizer
        a = _lib.DmfStepArgs()
        a.learning_rate, a.beta1, a.beta2, a.epsilon = o['learning_rate'], o['beta_1'], o['beta_2'], o['epsilon']
        a.reg_rate = reg_rate
        s = self._step
        for g in range(2):
            a.t[g] = 2 * (s - 1) + g + 1 if self.adam_t == 'per_variable' else s      # Q2
        return a

    def labels_from_values(self, values, out=None):
        """dmf.py:69: _standardize_value(interaction) when use_nce, else the raw interaction."""
        v = np.asarray(values, np.float64)
        lab = (v - self.min_interaction) / (self.max_interaction - self.min_interaction) if self.use_nce else v
        if out is None:
            return lab.astype(np.float32)
        out[:] = lab
        return out

    def _acquire_slot(self):
        slot = self._slots[self._slot_idx]
        self._slot_idx = (self._slot_idx + 1) % _RING
        if slot['event'] is not None:
            slot['event'].synchronize()
        return slot

    def _prepare_batch(self, slot, batch_size):
        self._sampler.sample_arrays(batch_size, out=(slot['uid_np'], slot['iid_np'], slot['val']))
        self.labels_from_values(slot['val'], out=slot['lab_np'])

    def _train_step(self, batch_size, reg_rate, want_loss=False, prefetch=False, **kwds):
        lib = _lib.load()
        with self._lock:
            nxt = getattr(self, '_next', None)
            if nxt is not None and nxt[1] == batch_size:
                slot = nxt[0]
            else:
                slot = self._acquire_slot()
                self._prepare_batch(slot, batch_size)
            self._next = None
            if self._dp.active:
                d = self._dp_buffers(batch_size)
                d['uid'].copy_(slot['uid'][:batch_size], non_blocking=True)
                d['iid'].copy_(slot['iid'][:batch_size], non_blocking=True)
                d['lab'].copy_(slot['lab'][:batch_size], non_blocking=True)
                self._step -= 1                  # step_device advances it again
                self.step_device(d['uid'], d['iid'], d['lab'], reg_rate, d['loss'])
            else:
                args = self.step_args(reg_rate)
                _lib.check(lib.drb_dmf_step_host(self._native, _lib.np_ptr(slot['uid_np']), _lib.np_ptr(slot['iid_np']),
                                                 _lib.np_ptr(slot['lab_np']), batch_size, C.byref(args), None))
                if want_loss:
                    self._loss_host.copy_(self._loss_dev, non_blocking=True)
            ev = self._torch.cuda.Event()
            ev.record(self._stream)
            slot['event'] = ev
            if prefetch:
                nslot = self._acquire_slot()
                self._prepare_batch(nslot, batch_size)
                self._next = (nslot, batch_size)
            if not want_loss:
                return None
            if self._dp.active:
                return self.global_loss(self._dp_dev['loss'])
            ev.synchronize()
            return float(self._loss_host[0])

    def _dp_buffers(self, batch_size):
        torch = self._torch
        if not hasattr(self, '_dp_dev') or self._dp_dev['uid'].numel() != batch_size:
            self._dp_dev = {'uid': torch.empty(batch_size, dtype=torch.int32, device=self._dev),
                            'iid': torch.empty(batch_size, dtype=torch.int32, device=self._dev),
                            'lab': torch.empty(batch_size, dtype=torch.float32, device=self._dev),
                            'loss': torch.zeros(2, dtype=torch.float32, device=self._dev)}
        return self._dp_dev

    def global_loss(self, loss2):
        """Reported loss of the global batch from this rank's [loss, batch term] pair (a collective when parallel)."""
        return float(self._dp.global_loss(loss2).item()) if self._dp.active else float(loss2[0].item())

    def step_device(self, uids_dev, iids_dev, labels_dev, reg_rate, loss_dev):
        """One step on device-resident pairs.  Data parallel: forward + backward on this rank's pairs with the loss mean
        over the global batch, ONE all-reduce of the gradient arena (2.5 MB at the ml-1m shape), then the identical
        Adam update on every rank."""
        self._step += 1
        args = self.step_args(reg_rate)
        lib = _lib.load()
        ptrs = (self._native, _lib.t_ptr(uids_dev), _lib.t_ptr(iids_dev), _lib.t_ptr(labels_dev), uids_dev.numel(),
                C.byref(args), _lib.t_ptr(loss_dev))
        dp = getattr(self, '_dp', None)
        if dp is None or not dp.active:
            _lib.check(lib.drb_dmf_step(*ptrs))
            return
        gb = uids_dev.numel() * dp.world
        _lib.check(lib.drb_dmf_step_phases(*ptrs, 1, gb))
        dp.all_reduce_sum(self._grads)
        _lib.check(lib.drb_dmf_step_phases(*ptrs, 2, gb))

    def launch_count(self):
        return _lib.load().drb_ctx_launch_count(self._ctx)

    def synchronize(self):
        _lib.check(_lib.load().drb_ctx_synchronize(self._ctx))

    # ------------------------------------------------------------------ scoring
    def forward_pairs(self, uids, iids):
        """Un-rescaled p = max(1e-6, cosine) for (uid, iid) pairs (dmf.py:88-96)."""
        torch = self._torch
        with self._lock:
            d_u = torch.as_tensor(np.ascontiguousarray(uids, np.int32), device=self._dev)
            d_i = torch.as_tensor(np.ascontiguousarray(iids, np.int32), device=self._dev)
            out = torch.empty(d_u.numel(), dtype=torch.float32, device=self._dev)
            _lib.check(_lib.load().drb_dmf_forward_pairs(self._native, _lib.t_ptr(d_u), _lib.t_ptr(d_i),
                                                         d_u.numel(), _lib.t_ptr(out)))
            return out.cpu().numpy()

    def _predict(self, uid, iid, **kwds):
        if uid is None or iid is None: return None
        return self._rescale_value(self.forward_pairs([uid], [iid])[0])

    def _sync_item_cache(self):
        # the library caches the item tower of the whole catalog between steps; in-place writes to the arena from
        # Python (weight injection, _revert_weights) bump the tensor version -> tell it
        if getattr(self, '_params_version', None) != self._params._version:
            _lib.check(_lib.load().drb_dmf_invalidate_cache(self._native))
            self._params_version = self._params._version

    def _rank_device(self, d_u, d_c, d_n, novelty):
        """drb_dmf_rank_candidates on device arrays: (iids, un-rescaled scores, n_out) as device tensors."""
        torch = self._torch
        n, max_c = d_c.shape
        self._sync_item_cache()
        o_i = torch.empty((n, max_c), dtype=torch.int32, device=self._dev)
        o_s = torch.empty((n, max_c), dtype=torch.float32, device=self._dev)
        o_n = torch.empty(n, dtype=torch.int32, device=self._dev)
        _lib.check(_lib.load().drb_dmf_rank_candidates(self._native, _lib.t_ptr(d_u), n, _lib.t_ptr(d_c),
                                                       _lib.t_ptr(d_n), max_c, int(bool(novelty)),
                                                       _lib.t_ptr(o_i), _lib.t_ptr(o_s), _lib.t_ptr(o_n)))
        return o_i, o_s, o_n

    def _rank_batch(self, uids, cand, cand_count, novelty):
        torch = self._torch
        with self._lock:
            d_u = torch.as_tensor(np.ascontiguousarray(uids, np.int32), device=self._dev)
            d_c = torch.as_tensor(np.ascontiguousarray(cand, np.int32), device=self._dev)
            d_n = torch.as_tensor(np.ascontiguousarray(cand_count, np.int32), device=self._dev)
            o_i, o_s, o_n = self._rank_device(d_u, d_c, d_n, novelty)
            # rank() reports rescaled predictions (recommender_abc.py:460 calls _predict -> _rescale_value)
            scores = self._rescale_value(o_s.cpu().numpy())
            return o_i.cpu().numpy(), scores, o_n.cpu().numpy()

    def topk_batch(self, uids, k, novelty=True, return_device=False):
        """Full-catalog top-k for many users: (iids [n, k], scores [n, k], n_out [n]).  Row r is what _rank_batch
        returns for uids[r] over range(n_items), truncated to k: the same item ids, and scores computed bit for bit
        as the rank path computes them (drb_dmf_topk), rescaled as rank() reports them.  1 <= k <= 2048.
        return_device=True: device tensors (scores rescaled on the device)."""
        torch = self._torch
        lib = _lib.load()
        k = int(k)
        with self._lock:
            self._sync_item_cache()
            nb = lib.drb_dmf_topk_scratch_bytes(self._native, k)
            if nb < 0:
                msg = lib.drb_last_error()
                raise RuntimeError(f'libdrb error: {msg.decode() if msg else ""}')
            scratch = getattr(self, '_topk_scratch', None)
            if scratch is None or scratch.numel() < nb:    # allocated once, grown when a larger k needs more
                scratch = self._topk_scratch = torch.empty(nb, dtype=torch.uint8, device=self._dev)
            d_u = uids if torch.is_tensor(uids) else torch.as_tensor(np.ascontiguousarray(uids, np.int32), device=self._dev)
            n = d_u.numel()
            o_i = torch.empty((n, k), dtype=torch.int32, device=self._dev)
            o_s = torch.empty((n, k), dtype=torch.float32, device=self._dev)
            o_n = torch.empty(n, dtype=torch.int32, device=self._dev)
            _lib.check(lib.drb_dmf_topk(self._native, _lib.t_ptr(d_u), n, k, int(bool(novelty)), _lib.t_ptr(scratch),
                                        scratch.numel(), _lib.t_ptr(o_i), _lib.t_ptr(o_s), _lib.t_ptr(o_n)))
            if n and int(o_n.min()) < 0:
                # more candidate lists of one block overflowed than the device-side fallback has rows for: those
                # users go through the rank path over the whole catalog, a few at a time (n x n_items candidates)
                bad = torch.nonzero(o_n < 0).flatten()
                cat = torch.arange(self.n_items, dtype=torch.int32, device=self._dev)
                for o in range(0, bad.numel(), 256):
                    rows = bad[o:o + 256]
                    c = rows.numel()
                    r_i, r_s, r_n = self._rank_device(d_u[rows].contiguous(), cat.expand(c, -1).contiguous(),
                                                      torch.full((c,), self.n_items, dtype=torch.int32,
                                                                 device=self._dev), novelty)
                    o_i[rows], o_s[rows], o_n[rows] = r_i[:, :k], r_s[:, :k], torch.clamp(r_n, max=k)
            if return_device:
                return o_i, self._rescale_value(o_s), o_n
            return o_i.cpu().numpy(), self._rescale_value(o_s.cpu().numpy()), o_n.cpu().numpy()

    def _recommend(self, uid, n, novelty, threshold):
        if n <= 2048:
            o_i, o_s, o_n = self.topk_batch(np.array([uid], np.int32), int(n), novelty)
            ranked = [(o_s[0, j], int(o_i[0, j])) for j in range(int(o_n[0]))]
        else:
            ranked = self._rank(uid, range(self.n_items), n, novelty)
        if threshold is None:
            return ranked
        return [x for x in ranked if x[0] >= threshold]
