"""CDAE (Collaborative Denoising Auto-Encoder) on the native B200 step -- drop-in for DRecPy's CDAE.

Mirrors DRecPy/Recommender/cdae.py: constructor :25-32, _pre_fit :34-45 (Glorot-uniform W[I,K], W_[K,I], V[U,K]
and -- as in the reference -- Glorot-initialised biases b[K], b_[I]; variable order [W, W_, V, b, b_]),
_sample_batch :47-48, the per-user reconstruct / loss / reg math :50-82 (now drb_cdae_step), _predict :84-88 and
_rank :90-103 (now drb_cdae_rank_candidates / drb_cdae_topk).

New keywords, all with reference-faithful defaults:
  label_mode='batch_mean'   the Keras-2 (B,B,I) loss broadcast of the reference (SURVEY.md Q1); 'per_user' = the
                            per-user targets of the CDAE paper
  rng_mode='mt19937'        bit-exact replay of the reference's corruption stream (n_items draws per sampled user,
                            cdae.py:63-64) on the host; 'mt19937_device' = the same stream, bit for bit, replayed on
                            the GPU by jump-ahead (mask_stream.py: 1.4 ms instead of ~0.3 s per 4096-user step);
                            'philox' = counter-based mask generated on the GPU (documented deviation)
  adam_t='per_variable'     Adam step counter advances once per variable (Q2); 'per_step' = textbook Adam
  init_weights=None         dict with any of W, W_, V, b, b_ (reference shapes) to inject initial weights
  gemm='auto'               'tcgen05' = 3xTF32 tensor-core GEMMs (fp32-accurate), 'ffma' = exact-fp32 CUDA-core GEMMs
"""
import ctypes as C
import os
import random

import numpy as np

from . import _lib, optimizers
from .parallel import DataParallel, data_parallel_step
from .recommender import DeepRecommenderABC
from .sampler import PointSampler

_RING = 4


class UniformUserSampler:
    """Seeded uniform user ids with PointSampler's array interface (sample_arrays).  For the sharded 10 M-user shape,
    where the reference sampler's membership structures do not exist on any single rank; CDAE uses only the uid of a
    sampled pair (cdae.py:52), and the reference's stream draws its users uniformly too."""

    def __init__(self, n_users, seed):
        self.n_users, self.rng = n_users, np.random.default_rng(abs(int(seed)))

    def sample_arrays(self, n, out=None):
        u = self.rng.integers(0, self.n_users, n, dtype=np.int32)
        if out is None:
            return u, np.zeros(n, np.int32), np.zeros(n, np.float64)
        out[0][:n] = u
        return out


class CDAE(DeepRecommenderABC):
    _SET_OPTIMIZER = 'drb_cdae_set_optimizer'

    def __init__(self, hidden_factors=50, corruption_level=0.2, loss='bce', **kwds):
        super(CDAE, self).__init__(**kwds)
        self.hidden_factors = hidden_factors
        self.corruption_level = corruption_level
        if loss not in ('mse', 'bce'):
            raise Exception(f'Loss function "{loss}" is not supported. Supported losses: "mse", "bce".')
        self.loss = loss
        self.label_mode = kwds.get('label_mode', 'batch_mean')
        self.rng_mode = kwds.get('rng_mode', 'mt19937')
        self.adam_t = kwds.get('adam_t', 'per_variable')
        self.gemm = kwds.get('gemm', 'auto')
        assert self.gemm in _lib.DRB_GEMM
        # output='sampled' (extension, not a reference behaviour): the training step scores each sampled user's
        # positives plus neg_groups x neg_per_group drawn items instead of the whole catalog (oracle: CDAESampledOracle)
        self.output = kwds.get('output', 'dense')
        self.neg_per_group = int(kwds.get('neg_per_group', 64))
        self.neg_groups = int(kwds.get('neg_groups', 1))
        assert self.output in ('dense', 'sampled')
        assert self.label_mode in _lib.DRB_LABEL and self.rng_mode in ('mt19937', 'mt19937_device', 'philox')
        assert self.adam_t in ('per_variable', 'per_step')
        self._native = None
        self._ctx = None

    # ------------------------------------------------------------------ setup
    def _pre_fit(self, learning_rate, neg_ratio, reg_rate, batch_size=32, **kwds):
        import torch
        self._torch = torch
        if not torch.cuda.is_available():
            raise RuntimeError('drecpy_b200 needs a CUDA device (sm_100a); there is no CPU fallback')
        self._dev = torch.device(self.device or f'cuda:{torch.cuda.current_device()}')
        self._max_batch = int(max(batch_size, min(1024, self.n_users), kwds.get('score_batch', 0)))
        # data parallel over user mini-batches: batch_size is PER RANK, the step uses the global batch
        self._dp = kwds.get('data_parallel') or DataParallel()
        self._dp_sampler = kwds.get('dp_sampler', 'replay')
        # parallel_mode='data'  : replicated weights, the mini-batch is split over ranks (gradients all-reduced)
        # parallel_mode='items' : W, W', b' sharded by item range and V by user range; every rank runs the whole
        #                         global batch against its items and only batch x hidden activations are exchanged
        self._parallel_mode = kwds.get('parallel_mode', 'data')
        assert self._parallel_mode in ('data', 'items')
        self._sharded = self._parallel_mode == 'items' and self._dp.active
        if self._sharded:
            w, r = self._dp.world, self._dp.rank
            per_i, per_u = -(-self.n_items // w), -(-self.n_users // w)
            self._ilo, self._ihi = min(self.n_items, r * per_i), min(self.n_items, (r + 1) * per_i)
            self._ulo, self._uhi = min(self.n_users, r * per_u), min(self.n_users, (r + 1) * per_u)
            assert self._ihi > self._ilo and self._uhi > self._ulo, 'more ranks than items / users'
            self._max_batch = int(max(batch_size * w, kwds.get('score_batch', 0)))
        else:
            self._ilo, self._ihi, self._ulo, self._uhi = 0, self.n_items, 0, self.n_users
        self._nI, self._nU = self._ihi - self._ilo, self._uhi - self._ulo
        self._alloc_and_init(kwds.get('init_weights', None))
        self._build_native()
        self._sampler = kwds.get('sampler') or PointSampler(self._data, neg_ratio, self.interaction_threshold, self.seed)
        mask_seed = self.seed if self.seed is not None else random.SystemRandom().getrandbits(63)
        self._mask_seed = abs(int(mask_seed))
        self._mask_rng = _lib.HostRng(self._mask_seed)      # replays self._rng of recommender_abc.py:74
        self._mask_stream = None
        if self.rng_mode == 'mt19937_device':
            if self._dp.active:
                raise NotImplementedError("rng_mode='mt19937_device' is single-process (the stream is sequential over "
                                          "the global batch); use 'philox' when data parallel")
            from .mask_stream import DeviceMaskStream
            self._mask_stream = DeviceMaskStream(self._mask_rng, self.n_items, self.corruption_level, self._torch,
                                                 self._dev, self._ctx, self._d_indptr, self._d_indices)
        self._setup_staging(batch_size)

    def fit_item_shard(self, shard_csr, n_users, n_items, batch_size, data_parallel, learning_rate=0.001,
                       reg_rate=0.001, sampler=None, **kwds):
        """Item-sharded training set-up for catalogs that never exist in one piece (BASELINE.json configs[4]: 10 M users
        x 1 M items, 1 B interactions): every rank passes only ITS columns of the interaction matrix,
        shard_csr = (indptr int64 [n_users + 1], indices int32 re-based to the shard, column-sorted), for the contiguous
        item range rank * ceil(n_items / world) ...  Weights are drawn per shard on the device; `sampler` must yield the
        same user ids on every rank (default: a seeded uniform user sampler).  No epochs are run: drive _train_step /
        step_device.  The reference has no counterpart (it is single-process and dense)."""
        import torch
        self._torch = torch
        self.n_users, self.n_items, self.n_rows = int(n_users), int(n_items), int(shard_csr[1].shape[0])
        self.min_interaction, self.max_interaction = 0, 5
        self.optimizer = optimizers.parse(kwds.pop('optimizer', None), learning_rate)
        self._step = 0
        self.epoch_weights = {}
        idx = shard_csr[1]                                   # numpy, or a torch tensor already on this rank's GPU
        self._shard_csr = (np.ascontiguousarray(shard_csr[0], np.int64),
                           idx if torch.is_tensor(idx) else np.ascontiguousarray(idx, np.int32))
        self._pre_fit(learning_rate, 5, reg_rate, batch_size=batch_size, data_parallel=data_parallel,
                      parallel_mode='items', sampler=sampler or UniformUserSampler(self.n_users, self.seed or 0), **kwds)
        self.fitted = True

    def _alloc_and_init(self, init_weights):
        torch = self._torch
        lib = _lib.load()
        L = _lib.CdaeLayout()
        _lib.check(lib.drb_cdae_layout(self._nU, self._nI, self.hidden_factors, C.byref(L)))
        self._L = L
        dev = self._dev
        self._params = torch.zeros(L.total, dtype=torch.float32, device=dev)
        self._alloc_optimizer_slots()
        self._grads = torch.zeros_like(self._params)
        K, I, U = self.hidden_factors, self.n_items, self.n_users
        gen = torch.Generator().manual_seed(abs(int(self.seed)) if self.seed is not None else random.getrandbits(62))

        def glorot(shape, fan_in, fan_out):       # tf.initializers.GlorotUniform (cdae.py:35-41)
            lim = float(np.sqrt(6.0 / (fan_in + fan_out)))
            return (torch.rand(shape, generator=gen, dtype=torch.float32) * 2 - 1) * lim
        if getattr(self, '_shard_csr', None) is not None:
            # catalogs that only exist sharded (10 M x 1 M): draw this rank's rows only, on the device (same Glorot limits)
            dgen = torch.Generator(device=dev).manual_seed(abs(int(self.seed or 0)) * 1000 + self._dp.rank)

            def dglorot(view, fan_in, fan_out):
                lim = float(np.sqrt(6.0 / (fan_in + fan_out)))
                view.copy_((torch.rand(view.shape, generator=dgen, dtype=torch.float32, device=dev) * 2 - 1) * lim)
            dglorot(self.W, I, K); dglorot(self.W_, K, I); dglorot(self.V, U, K); dglorot(self.b_, I, I)
            self.b.copy_(glorot((K,), K, K))               # replicated: the same on every rank
            return
        init = {'W': glorot((I, K), I, K), 'W_': glorot((K, I), K, I), 'V': glorot((U, K), U, K),
                'b': glorot((K,), K, K), 'b_': glorot((I,), I, I)}
        for k, v in (init_weights or {}).items():
            assert k in init, f'unknown weight {k}'
            v = torch.as_tensor(np.asarray(v), dtype=torch.float32)
            assert tuple(v.shape) == tuple(init[k].shape), f'{k}: expected shape {tuple(init[k].shape)}'
            init[k] = v
        il, ih, ul, uh = self._ilo, self._ihi, self._ulo, self._uhi      # the whole range unless item-sharded
        self.W.copy_(init['W'][il:ih])
        self.W_.copy_(init['W_'][:, il:ih])
        self.V.copy_(init['V'][ul:uh])
        self.b.copy_(init['b'])
        self.b_.copy_(init['b_'][il:ih])

    def _build_native(self):
        torch = self._torch
        lib = _lib.load()
        dev, L = self._dev, self._L
        self._ctx = _lib.vp()
        _lib.check(lib.drb_ctx_create(dev.index or 0, C.byref(self._ctx)))
        self._stream = torch.cuda.current_stream(dev)
        _lib.check(lib.drb_ctx_set_stream(self._ctx, _lib.vp(self._stream.cuda_stream)))
        shard = getattr(self, '_shard_csr', None)
        if shard is not None:                                # fit_item_shard: this rank's columns only, already re-based
            pos = seen = (shard[0], shard[1], None)
        else:
            pos = self._data.csr(self.interaction_threshold)     # positives: cdae.py:61
            seen = self._data.csr()                              # every stored row: cdae.py:93-98
            if self._sharded:                                    # keep the columns of this rank's item range, re-based
                pos, seen = [self._restrict_columns(c, self._ilo, self._ihi) for c in (pos, seen)]
        self._h_indptr = np.ascontiguousarray(pos[0])
        self._d_indptr = torch.from_numpy(self._h_indptr).to(dev)
        if torch.is_tensor(pos[1]):                          # shard generated on the device: indices never visit the host
            self._h_indices, self._d_indices = None, pos[1].to(dev).contiguous()
        else:
            self._h_indices = np.ascontiguousarray(pos[1])
            self._d_indices = torch.from_numpy(self._h_indices).to(dev)
        if seen[0] is pos[0] and seen[1] is pos[1]:          # one CSR serves both roles: no second copy in HBM
            self._d_seen_indptr, self._d_seen_indices = self._d_indptr, self._d_indices
        else:
            self._d_seen_indptr = torch.from_numpy(np.ascontiguousarray(seen[0])).to(dev)
            self._d_seen_indices = torch.from_numpy(np.ascontiguousarray(seen[1])).to(dev)
        sampled = getattr(self, 'output', 'dense') == 'sampled'
        ws_fn = lib.drb_cdae_workspace_bytes_sampled if sampled else lib.drb_cdae_workspace_bytes
        ws_bytes = ws_fn(self._nU, self._nI, self.hidden_factors, self._max_batch)
        assert ws_bytes > 0
        self._workspace = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        d = _lib.CdaeDesc()
        d.n_users, d.n_items, d.hidden = self._nU, self._nI, self.hidden_factors
        d.params, d.adam_m, d.adam_v, d.grads = (self._params.data_ptr(), self._adam_m.data_ptr(),
                                                 self._adam_v.data_ptr(), self._grads.data_ptr())
        d.csr_indptr, d.csr_indices = self._d_indptr.data_ptr(), self._d_indices.data_ptr()
        d.seen_indptr, d.seen_indices = self._d_seen_indptr.data_ptr(), self._d_seen_indices.data_ptr()
        d.corruption_level = float(self.corruption_level)
        d.loss_kind = _lib.DRB_LOSS[self.loss]
        d.label_mode = _lib.DRB_LABEL[self.label_mode]
        d.workspace, d.workspace_bytes, d.max_batch = self._workspace.data_ptr(), ws_bytes, self._max_batch
        d.gemm_path = _lib.DRB_GEMM[self.gemm]
        if sampled:
            d.output_mode, d.neg_per_group = 1, self.neg_per_group
            d.neg_groups = self._dp.world if getattr(self, '_sharded', False) else self.neg_groups
        self._native = _lib.vp()
        _lib.check(lib.drb_cdae_create(self._ctx, C.byref(d), C.byref(self._native)))
        ptr, cnt = _lib.vp(), _lib.i64()
        _lib.check(lib.drb_cdae_label_count_buffer(self._native, C.byref(ptr), C.byref(cnt)))
        off = ptr.value - self._workspace.data_ptr()
        self._label_count = self._workspace[off:off + 4 * cnt.value].view(torch.float32)   # all-reduced when DP
        _lib.check(lib.drb_cdae_loss_buffer(self._native, C.byref(ptr)))
        off = ptr.value - self._workspace.data_ptr()
        self._loss_dev = self._workspace[off:off + 8].view(torch.float32)
        _lib.check(lib.drb_cdae_h_buffer(self._native, C.byref(ptr), C.byref(cnt)))
        off = ptr.value - self._workspace.data_ptr()
        self._h_buf = self._workspace[off:off + 4 * cnt.value].view(torch.float32).view(-1, L.ld)
        _lib.check(lib.drb_cdae_dz1_buffer(self._native, C.byref(ptr), C.byref(cnt)))
        off = ptr.value - self._workspace.data_ptr()
        self._dz1 = self._workspace[off:off + 4 * cnt.value].view(torch.float32).view(-1, L.ld)
        self._apply_optimizer()

    @staticmethod
    def _restrict_columns(csr, lo, hi):
        indptr, indices, data = csr
        keep = (indices >= lo) & (indices < hi)
        rows = np.repeat(np.arange(len(indptr) - 1), np.diff(indptr))[keep]
        out = np.zeros(len(indptr), np.int64)
        np.cumsum(np.bincount(rows, minlength=len(indptr) - 1), out=out[1:])
        return out, (indices[keep] - lo).astype(np.int32), data[keep]

    def _setup_staging(self, batch_size):
        if self._sharded:
            batch_size = batch_size * self._dp.world
        torch = self._torch
        deg = np.diff(self._h_indptr)
        # users are drawn WITH replacement, so no sum over distinct users bounds a batch's positives; start from a
        # typical batch and let prepare_batch grow the slot when drb_batch_offsets reports more (_ensure_keep)
        cap = int(min(batch_size * int(deg.max(initial=0)), 4 * batch_size * float(deg.mean()) + 4096)) if len(deg) else 0
        self._slots = []
        for _ in range(_RING):
            s = {'uid': torch.empty(batch_size, dtype=torch.int32).pin_memory(),
                 'iid': np.empty(batch_size, np.int32), 'val': np.empty(batch_size, np.float64),
                 'off': torch.empty(batch_size + 1, dtype=torch.int32).pin_memory(),
                 'keep': torch.empty(max(cap, 16), dtype=torch.uint8).pin_memory(),
                 'event': None}
            s['uid_np'], s['off_np'], s['keep_np'] = s['uid'].numpy(), s['off'].numpy(), s['keep'].numpy()
            self._slots.append(s)
        self._slot_idx = 0
        self._loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
        self._next = None

    # ------------------------------------------------------------------ weights as reference-shaped views
    def _seg(self, off, rows, ld):
        return self._params[off:off + rows * ld].view(rows, ld)

    @property
    def W(self):
        return self._seg(self._L.off_w, self._nI, self._L.ld)[:, :self.hidden_factors]

    @property
    def W_(self):     # reference layout [K, I]; stored item-major
        return self._seg(self._L.off_w2t, self._nI, self._L.ld)[:, :self.hidden_factors].t()

    @property
    def V(self):
        return self._seg(self._L.off_v, self._nU, self._L.ld)[:, :self.hidden_factors]

    @property
    def b(self):
        return self._params[self._L.off_b:self._L.off_b + self.hidden_factors]

    @property
    def b_(self):
        return self._params[self._L.off_b2:self._L.off_b2 + self._nI]

    def _params_tensor(self):
        return self._params

    # ------------------------------------------------------------------ training step
    def step_args(self, reg_rate):
        o = self.optimizer
        a = _lib.CdaeStepArgs()
        a.learning_rate = o['learning_rate']       # the rest of the optimizer is the model's drb_optim_desc
        a.beta1, a.beta2, a.epsilon = o.get('beta_1', 0.9), o.get('beta_2', 0.999), o.get('epsilon', 1e-7)
        a.reg_rate = reg_rate
        s = self._step
        for j in range(5):
            a.t[j] = 5 * (s - 1) + j + 1 if self.adam_t == 'per_variable' else s     # Q2
        a.philox_seed = self._mask_seed
        a.philox_step = s
        dp = getattr(self, '_dp', None)
        if dp is not None and dp.active and getattr(self, '_sharded', False):
            a.shard_items, a.item_offset, a.n_items_global = 1, self._ilo, self.n_items
        elif dp is not None and dp.active:
            a.global_batch = self._cur_batch * dp.world
            a.slot_offset = self._cur_batch * dp.rank
            a.skip_user_grad = 1
        return a

    def prepare_batch(self, slot, batch_size):
        """Host side of one step: sample B triples (only uid is used, cdae.py:52) and build the mask inputs."""
        lib = _lib.load()
        dp = self._dp
        if self._sharded:
            # every rank replays the same stream and processes the WHOLE global batch against its own items
            n = batch_size * dp.world
            self._sampler.sample_arrays(n, out=(slot['uid_np'], slot['iid'], slot['val']))
            if self.rng_mode == 'mt19937':
                raise NotImplementedError("item-sharded training needs rng_mode='philox'")
            batch_size = n
        elif dp.active and self._dp_sampler == 'replay':
            # every rank replays the global stream and keeps its slice (== a single-process run with batch N*B)
            gu, _, _ = self._sampler.sample_arrays(batch_size * dp.world)
            lo, hi = dp.shard(batch_size * dp.world)
            slot['uid_np'][:] = gu[lo:hi]
            if self.rng_mode == 'mt19937':
                raise NotImplementedError("data parallel training needs rng_mode='philox' (the MT19937 corruption "
                                          "stream is sequential over the global batch)")
        else:
            self._sampler.sample_arrays(batch_size, out=(slot['uid_np'], slot['iid'], slot['val']))
        _lib.check(lib.drb_batch_offsets(_lib.np_ptr(slot['uid_np']), batch_size, _lib.np_ptr(self._h_indptr),
                                         _lib.np_ptr(slot['off_np'])))
        if self.rng_mode == 'mt19937':
            self._ensure_keep(slot, int(slot['off_np'][batch_size]))
            _lib.check(lib.drb_cdae_corruption_keep_mt(
                self._mask_rng.handle, _lib.np_ptr(slot['uid_np']), batch_size, self.n_items,
                float(self.corruption_level), _lib.np_ptr(self._h_indptr), _lib.np_ptr(self._h_indices),
                _lib.np_ptr(slot['off_np']), _lib.np_ptr(slot['keep_np']), len(slot['keep_np'])))
            return _lib.np_ptr(slot['keep_np'])
        return None

    def _ensure_keep(self, slot, nnz):
        """The pinned keep buffer of a staging slot holds one byte per positive of the batch; grow it when a batch
        (users repeat: sampling is with replacement) holds more than any batch so far."""
        if nnz <= len(slot['keep_np']):
            return
        if slot['event'] is not None:
            slot['event'].synchronize()               # an H2D copy out of the old buffer may still be in flight
        slot['keep'] = self._torch.empty(int(nnz * 1.25) + 4096, dtype=self._torch.uint8).pin_memory()
        slot['keep_np'] = slot['keep'].numpy()

    def _acquire_slot(self):
        slot = self._slots[self._slot_idx]
        self._slot_idx = (self._slot_idx + 1) % _RING
        if slot['event'] is not None:
            slot['event'].synchronize()          # the async H2D of the step that last used this slot is done
        return slot

    def _train_step(self, batch_size, reg_rate, want_loss=False, prefetch=False, **kwds):
        """One optimizer step through the host-buffer C-ABI entry.  With prefetch=True the NEXT batch is sampled
        and its mask built on the host while the GPU runs this step (the fit loop does this on every epoch but the
        last, so the sampler streams end exactly where the reference's would)."""
        lib = _lib.load()
        with self._lock:
            nxt = getattr(self, '_next', None)
            if nxt is not None:
                ready = nxt[2].result() if hasattr(nxt[2], 'result') else nxt[2]   # the prefetch thread is done with the
            if nxt is not None and nxt[1] == batch_size:                            # sampler from here on
                slot, keep_ptr = nxt[0], ready
            else:
                slot = self._acquire_slot()
                keep_ptr = self.prepare_batch(slot, batch_size)
            self._next = None
            self._cur_batch = batch_size
            if prefetch:
                # the NEXT batch is sampled (and, in 'mt19937' mode, its mask replayed) by a worker thread while this
                # thread enqueues the step and the GPU runs it: ctypes releases the GIL inside the native sampler
                nslot = self._acquire_slot()
                pool = self._prefetch_pool()
                self._next = (nslot, batch_size, pool.submit(self._prepare_in_thread, nslot, batch_size) if pool
                              else None)
            if self._dp.active or self._mask_stream is not None:
                self._enqueue_step_dp(slot, batch_size * (self._dp.world if self._sharded else 1), reg_rate)
            else:
                args = self.step_args(reg_rate)
                _lib.check(lib.drb_cdae_step_host(self._native, _lib.np_ptr(slot['uid_np']),
                                                  _lib.np_ptr(slot['off_np']), keep_ptr, batch_size, C.byref(args),
                                                  None))
                if want_loss:
                    self._loss_host.copy_(self._loss_dev, non_blocking=True)
            ev = self._torch.cuda.Event()
            ev.record(self._stream)
            slot['event'] = ev
            if prefetch and self._next[2] is None:       # no worker thread (DRB_PREFETCH_THREAD=0): prepare it here
                self._next = (self._next[0], batch_size, self.prepare_batch(self._next[0], batch_size))
            if not want_loss:
                return None
            if self._dp.active or self._mask_stream is not None:
                return self.global_loss(self._dp_dev['loss'])
            ev.synchronize()
            return float(self._loss_host[0])

    def _prefetch_pool(self):
        """One worker thread for the host side of the next batch (None when DRB_PREFETCH_THREAD=0)."""
        pool = getattr(self, '_pool', None)
        if pool is None and os.environ.get('DRB_PREFETCH_THREAD', '1') != '0':
            from concurrent.futures import ThreadPoolExecutor
            pool = self._pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix='drb-prefetch')
        return pool

    def _prepare_in_thread(self, slot, batch_size):
        with self._torch.cuda.device(self._dev):          # a growing pinned keep buffer is allocated for this device
            return self.prepare_batch(slot, batch_size)

    def _finish_fit(self):
        nxt = getattr(self, '_next', None)                # a batch prefetched before an early stop: let the worker finish
        if nxt is not None and hasattr(nxt[2], 'result'):
            nxt[2].result()

    def _enqueue_step_dp(self, slot, batch_size, reg_rate):
        torch = self._torch
        if not hasattr(self, '_dp_dev'):
            self._dp_dev = {'uid': torch.empty(batch_size, dtype=torch.int32, device=self._dev),
                            'off': torch.empty(batch_size + 1, dtype=torch.int32, device=self._dev),
                            'loss': torch.zeros(2, dtype=torch.float32, device=self._dev)}
        d = self._dp_dev
        d['uid'].copy_(slot['uid'][:batch_size], non_blocking=True)
        d['off'].copy_(slot['off'][:batch_size + 1], non_blocking=True)
        self._step -= 1                      # step_device advances it again
        self.step_device(d['uid'], d['off'], None, reg_rate, d['loss'])

    def global_loss(self, loss2):
        """Reported loss of the global batch from this rank's [loss, batch term] pair (a collective when parallel)."""
        dp = self._dp
        if not dp.active:
            return float(loss2[0].item())
        if self._sharded:                     # every rank holds the terms of its items and its share of the L2 sum
            t = loss2[0:1].clone()
            dp.all_reduce_sum(t)
            return float(t.item())
        return float(dp.global_loss(loss2).item())

    def step_device(self, uids_dev, keep_off_dev, keep_dev, reg_rate, loss_dev):
        """One step on device-resident inputs (torch tensors); keep_dev=None selects the philox mask.
        loss_dev: float32[2] device tensor ([0] reported loss, [1] its batch term of this rank)."""
        self._step += 1
        self._cur_batch = uids_dev.numel()
        if keep_dev is None and getattr(self, '_mask_stream', None) is not None:
            # the reference's MT19937 corruption stream, replayed on the device for this batch
            cap = int(uids_dev.numel()) * int(max(1, np.diff(self._h_indptr).max(initial=1)))
            if getattr(self, '_keep_dev', None) is None or self._keep_dev.numel() < cap:
                self._keep_dev = self._torch.empty(cap, dtype=self._torch.uint8, device=self._dev)
            keep_dev = self._keep_dev
            self._mask_stream.fill(uids_dev, keep_off_dev, keep_dev)
        args = self.step_args(reg_rate)
        if keep_dev is not None:
            args.keep_bytes = keep_dev.numel()        # lets the small shapes replay the step as a CUDA graph
        lib = _lib.load()
        ptrs = (self._native, _lib.t_ptr(uids_dev), _lib.t_ptr(keep_off_dev), _lib.t_ptr(keep_dev), uids_dev.numel(),
                C.byref(args), _lib.t_ptr(loss_dev))
        dp = getattr(self, '_dp', None)
        if dp is None or not dp.active:
            _lib.check(lib.drb_cdae_step(*ptrs))
            return
        if self._sharded:
            return self._step_device_sharded(uids_dev, args, ptrs)
        # data parallel: drecpy_b200.parallel.data_parallel_step runs the phases with the collectives between them
        torch = self._torch
        L = self._L
        B = uids_dev.numel()
        if not hasattr(self, '_dp_gather') or self._dp_gather[0].shape[0] != B * dp.world:
            self._dp_gather = (torch.empty((B * dp.world, L.ld), dtype=torch.float32, device=self._dev),
                               torch.empty(B * dp.world, dtype=torch.int32, device=self._dev))
        rows_all, uids_all = self._dp_gather

        def run_phase(mask):
            _lib.check(lib.drb_cdae_step_phases(*ptrs, mask))

        def add_user_rows(u_all, r_all):       # user-row gradients: B x K rows travel, never the U x K table
            _lib.check(lib.drb_cdae_scatter_user_rows(self._native, _lib.t_ptr(u_all), _lib.t_ptr(r_all), u_all.numel()))
        data_parallel_step(dp, run_phase, self._label_count if self.label_mode == 'batch_mean' else None, self._grads,
                           L.off_w, L.off_v, self._dz1[:B], uids_dev, rows_all, uids_all, add_user_rows)

    def _step_device_sharded(self, uids_dev, args, ptrs):
        """Item-sharded step: rows of W / W' / V never travel; the two exchanges are all-reduces of batch x hidden
        activations (the partial pre-activation of the hidden layer and the partial dh)."""
        torch, lib, dp = self._torch, _lib.load(), self._dp
        n = uids_dev.numel()
        owned = (uids_dev >= self._ulo) & (uids_dev < self._uhi)
        v_rows = torch.where(owned, uids_dev - self._ulo, torch.full_like(uids_dev, -1)).contiguous()
        args.v_rows = v_rows.data_ptr()
        PREP, GA, UPD, GB, GC, GA2, GC2 = 1, 2, 4, 8, 16, 32, 64
        _lib.check(lib.drb_cdae_step_phases(*ptrs, PREP | GA))
        dp.all_reduce_sum(self._h_buf[:n])
        _lib.check(lib.drb_cdae_step_phases(*ptrs, GA2 | GB | GC))
        dp.all_reduce_sum(self._dz1[:n])
        _lib.check(lib.drb_cdae_step_phases(*ptrs, GC2 | UPD))
        self._keepalive = v_rows             # the kernels read it asynchronously

    def gather_full_weights(self):
        """Reference-shaped full weights {W, W_, V, b, b_} on every rank (all-gather of the shards)."""
        torch, dp = self._torch, self._dp
        out = {'b': self.b.clone()}
        if not getattr(self, '_sharded', False):
            out.update(W=self.W.clone(), W_=self.W_.clone(), V=self.V.clone(), b_=self.b_.clone())
            return out
        K = self.hidden_factors

        def gather_rows(local, total, per):
            pad = torch.zeros((per, local.shape[1]), dtype=torch.float32, device=self._dev)
            pad[:local.shape[0]] = local
            full = torch.empty((per * dp.world, local.shape[1]), dtype=torch.float32, device=self._dev)
            dp.dist.all_gather_into_tensor(full, pad, group=dp.group)
            return full[:total]
        per_i, per_u = -(-self.n_items // dp.world), -(-self.n_users // dp.world)
        out['W'] = gather_rows(self.W.contiguous(), self.n_items, per_i)
        out['W_'] = gather_rows(self.W_.t().contiguous(), self.n_items, per_i).t()
        out['V'] = gather_rows(self.V.contiguous(), self.n_users, per_u)
        out['b_'] = gather_rows(self.b_.reshape(-1, 1).contiguous(), self.n_items, per_i).reshape(-1)
        return out

    def launch_count(self):
        return _lib.load().drb_ctx_launch_count(self._ctx)

    def synchronize(self):
        _lib.check(_lib.load().drb_ctx_synchronize(self._ctx))

    # ------------------------------------------------------------------ scoring
    def _predict(self, uid, iid=None, **kwds):
        if uid is None: return None
        torch = self._torch
        with self._lock:
            u = torch.tensor([uid], dtype=torch.int32, device=self._dev)
            out = torch.empty(self._L.items_pad, dtype=torch.float32, device=self._dev)
            _lib.check(_lib.load().drb_cdae_predict_all(self._native, _lib.t_ptr(u), 1, _lib.t_ptr(out)))
            predictions = out[:self.n_items].cpu().numpy()
        return predictions if iid is None else predictions[iid]

    def predict_batch(self, user_ids, item_ids, skip_errors=False, chunk=1 << 22):
        if getattr(self, '_sharded', False) or getattr(self, '_shard_csr', None) is not None:
            raise NotImplementedError('predict_batch: an item-sharded CDAE holds only its shard of the output layer, '
                                      'so its scores are not predict() values')
        return super().predict_batch(user_ids, item_ids, skip_errors, chunk)

    def _launch_predict_pairs(self, users, pair_off, pair_iid, pair_dst, out):
        _lib.check(_lib.load().drb_cdae_predict_pairs(self._native, _lib.t_ptr(users), users.numel(),
                                                      _lib.t_ptr(pair_off), _lib.t_ptr(pair_iid), _lib.t_ptr(pair_dst),
                                                      out.numel(), _lib.t_ptr(out)))

    def hidden(self, uids):
        torch = self._torch
        with self._lock:
            u = torch.as_tensor(np.asarray(uids, np.int32), device=self._dev)
            out = torch.empty((len(u), self._L.ld), dtype=torch.float32, device=self._dev)
            for o in range(0, len(u), self._max_batch):
                n = min(self._max_batch, len(u) - o)
                _lib.check(_lib.load().drb_cdae_hidden(self._native, _lib.t_ptr(u[o:]), n, _lib.t_ptr(out[o:])))
            return out[:, :self.hidden_factors].cpu().numpy()

    def rank_candidates_device(self, d_u, d_c, d_n, novelty, out=None):
        """drb_cdae_rank_candidates on device tensors: uids [n] int32, cand [n, max_c] int32 internal ids, counts [n].
        Returns device tensors (iids [n, max_c], scores [n, max_c], n_out [n]); `out` reuses a previous result."""
        torch = self._torch
        n, max_c = d_c.shape
        with self._lock:
            o_i, o_s, o_n = out if out is not None else (
                torch.empty((n, max_c), dtype=torch.int32, device=self._dev),
                torch.empty((n, max_c), dtype=torch.float32, device=self._dev),
                torch.empty(n, dtype=torch.int32, device=self._dev))
            _lib.check(_lib.load().drb_cdae_rank_candidates(self._native, _lib.t_ptr(d_u), n, _lib.t_ptr(d_c),
                                                            _lib.t_ptr(d_n), max_c, int(bool(novelty)),
                                                            _lib.t_ptr(o_i), _lib.t_ptr(o_s), _lib.t_ptr(o_n)))
        return o_i, o_s, o_n

    def _rank_batch(self, uids, cand, cand_count, novelty):
        torch = self._torch
        with self._lock:
            d_u = torch.as_tensor(np.ascontiguousarray(uids, np.int32), device=self._dev)
            d_c = torch.as_tensor(np.ascontiguousarray(cand, np.int32), device=self._dev)
            d_n = torch.as_tensor(np.ascontiguousarray(cand_count, np.int32), device=self._dev)
            o_i, o_s, o_n = self.rank_candidates_device(d_u, d_c, d_n, novelty)
            return self._to_host(o_i, o_s, o_n)

    def _to_host(self, *tensors):
        """Device results -> numpy arrays through pinned host memory (torch's caching host allocator keeps the blocks,
        so only the first call pays for pinning; a pageable .cpu() of the 111 MB of ranked lists of the ml-20m shape
        took three times as long as computing them).  The arrays own their pinned block until they are dropped."""
        torch = self._torch
        host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in tensors]
        for h, t in zip(host, tensors):
            h.copy_(t, non_blocking=True)
        torch.cuda.current_stream(self._dev).synchronize()
        return tuple(h.numpy() for h in host)

    def topk_batch(self, uids, k, novelty=True, return_device=False, exact=False):
        """Full-catalog top-k for many users: (iids [n,k], scores [n,k], n_out [n]).  exact=True forces the exact-fp32
        score rows + radix select instead of the tensor-core path."""
        torch = self._torch
        lib = _lib.load()
        with self._lock:
            d_u = uids if torch.is_tensor(uids) else torch.as_tensor(np.ascontiguousarray(uids, np.int32), device=self._dev)
            n = d_u.numel()
            o_i = torch.empty((n, k), dtype=torch.int32, device=self._dev)
            o_s = torch.empty((n, k), dtype=torch.float32, device=self._dev)
            o_n = torch.empty(n, dtype=torch.int32, device=self._dev)
            fn = lib.drb_cdae_topk_exact if exact else lib.drb_cdae_topk
            _lib.check(fn(self._native, _lib.t_ptr(d_u), n, k, int(bool(novelty)), _lib.t_ptr(o_i), _lib.t_ptr(o_s),
                          _lib.t_ptr(o_n)))
            if not exact and n and int(o_n.min()) < 0:
                # more candidate lists of one block overflowed than the device-side fallback has rows for (only
                # possible with adversarial score distributions): those users go through the exact path
                bad = torch.nonzero(o_n < 0).flatten()
                b_i = torch.empty((bad.numel(), k), dtype=torch.int32, device=self._dev)
                b_s = torch.empty((bad.numel(), k), dtype=torch.float32, device=self._dev)
                b_n = torch.empty(bad.numel(), dtype=torch.int32, device=self._dev)
                b_u = d_u[bad].contiguous()
                _lib.check(lib.drb_cdae_topk_exact(self._native, _lib.t_ptr(b_u), bad.numel(), k, int(bool(novelty)),
                                                   _lib.t_ptr(b_i), _lib.t_ptr(b_s), _lib.t_ptr(b_n)))
                o_i[bad], o_s[bad], o_n[bad] = b_i, b_s, b_n
            if return_device:
                return o_i, o_s, o_n
            return self._to_host(o_i, o_s, o_n)

    def _recommend(self, uid, n, novelty, threshold):
        if n <= 2048:
            o_i, o_s, o_n = self.topk_batch(np.array([uid], np.int32), int(n), novelty)
            ranked = [(o_s[0, j], int(o_i[0, j])) for j in range(int(o_n[0]))]
        else:
            ranked = self._rank(uid, range(self.n_items), n, novelty)
        if threshold is None:
            return ranked
        return [x for x in ranked if x[0] >= threshold]
