"""DeepRecommenderABC: RecommenderABC's public surface with the batch loop moved onto the native B200 step.

Mirrors DRecPy/Recommender/recommender_abc.py:
  __init__   :54-95     verbose / interaction_threshold / seed keywords, self._rng = random.Random(seed)
  fit        :97-264    same signature and keywords (epoch_callback_fn, epoch_callback_freq,
                        early_stopping_rule, early_stopping_freq, optimizer), same callback / early-stopping /
                        revert cadence; the tf.GradientTape body (:190-205) is replaced by one native step
  predict    :354-383   rank :421-452   recommend :391-411   save / load :503-524
Deliberate, observationally-equivalent change (SURVEY.md Q3): weights are snapshotted only on callback epochs
(the only epochs _revert_weights can ever be asked for) instead of deep-copied every step.
Subclasses implement _pre_fit / _train_step / _predict / _rank_batch on top of libdrb; overriding the math hooks
with arbitrary framework code is not supported (there is no TensorFlow and no CPU fallback).
"""
import logging
import random
import threading
from abc import ABC, abstractmethod

import numpy as np

from .dataset import InteractionData
from .loss_tracker import LossTracker


class InvalidEpochValidationResultsException(Exception):
    pass


def _is_invalid_validation_exc(e):
    return e.__class__.__name__ == 'InvalidEpochValidationResultsException'


class DeepRecommenderABC(ABC):
    def __init__(self, **kwds):
        self.verbose = kwds.get('verbose', True)
        self.min_interaction = None
        self.max_interaction = None
        self.seed = kwds.get('seed', None)
        self.device = kwds.get('device', None)          # torch device string; default: current CUDA device

        self.fitted = False
        self.n_users = 0
        self.n_items = 0
        self.n_rows = 0
        self.interaction_threshold = kwds.get('interaction_threshold', 1e-3)
        self.interaction_dataset = None
        self.epoch_weights = {}
        self.optimizer = None

        self._data = None
        self._loss_tracker = None
        self._rng = random.Random(self.seed)             # recommender_abc.py:74 (kept for API parity)
        self._lock = threading.RLock()                   # ranking_evaluation calls rank() from 4 threads
        self._step = 0

        self._logger = logging.getLogger(f'{self.__class__.__name__}_CLOGGER')
        if not self._logger.handlers:
            ch = logging.StreamHandler()
            ch.setFormatter(logging.Formatter('[%(asctime)s] (%(levelname)s) %(name)s: %(message)s'))
            self._logger.addHandler(ch)
        self._logger.propagate = False
        self._logger.setLevel(logging.INFO)

    # ------------------------------------------------------------------ fit (recommender_abc.py:97-264)
    def fit(self, interaction_dataset, epochs=50, batch_size=32, learning_rate=0.001, neg_ratio=5, reg_rate=0.001,
            copy_dataset=False, **kwds):
        self.interaction_dataset = interaction_dataset
        if copy_dataset and hasattr(interaction_dataset, '__copy__'):
            self._info('Cloning new dataset instance...')
            self.interaction_dataset = interaction_dataset.__copy__()
        self.interaction_dataset.assign_internal_ids()
        self._data = InteractionData.from_dataset(self.interaction_dataset)
        self._data.assign_internal_ids()

        self.min_interaction = self._data.min('interaction')
        if self.min_interaction == 1: self.min_interaction = 0          # recommender_abc.py:141
        self.max_interaction = self._data.max('interaction')
        self.n_users = self._data.count_unique('uid')
        self.n_items = self._data.count_unique('iid')
        self.n_rows = len(self._data)

        self._loss_tracker = kwds.get('loss_tracker') or LossTracker()
        self._log_initial_info()
        self._info('Creating auxiliary structures...')

        opt = kwds.get('optimizer', None)
        if opt is not None and not isinstance(opt, dict):
            raise NotImplementedError('drecpy_b200 runs Keras-Adam natively; pass optimizer=None or a dict with '
                                      'beta_1 / beta_2 / epsilon / learning_rate overrides')
        self.optimizer = {'learning_rate': learning_rate, 'beta_1': 0.9, 'beta_2': 0.999, 'epsilon': 1e-7}
        if opt:
            self.optimizer.update(opt)
        self._step = 0
        self.epoch_weights = {}
        self._pre_fit(learning_rate, neg_ratio, reg_rate, batch_size=batch_size, **kwds)
        self.fitted = True

        progress_desc = ''
        epoch_callback_fn = kwds.get('epoch_callback_fn', None)
        epoch_callback_ret, epoch_callback_res_registered = None, True
        epoch_callback_freq = kwds.get('epoch_callback_freq', 5)
        early_stopping_rule = kwds.get('early_stopping_rule', None)
        early_stopping_freq = kwds.get('early_stopping_freq', 5)
        early_stopping_best_epoch = None
        track = self.verbose or early_stopping_rule is not None

        if self.verbose and epoch_callback_fn is not None:
            epoch_callback_ret = epoch_callback_fn(self)
            assert type(epoch_callback_ret) is dict, \
                f'The return type of the epoch_callback_fn should be dict, but found {type(epoch_callback_ret)}'
            for metric in epoch_callback_ret:
                self._loss_tracker.add_epoch_callback_result(metric, epoch_callback_ret[metric], 0)

        _iter = range(1, epochs + 1)
        if self.verbose:
            from tqdm import tqdm
            _iter = tqdm(range(1, epochs + 1), total=epochs, desc='Fitting model...', position=0, leave=True)
        e = 0
        for e in _iter:
            self._step = e
            loss = self._train_step(batch_size, reg_rate, want_loss=track, prefetch=(e < epochs), **kwds)

            if track:
                self._loss_tracker.add_epoch_loss(loss)
                if epoch_callback_fn is not None and e % epoch_callback_freq == 0:
                    epoch_callback_res_registered = False
                    self._store_epoch_weights(e)           # Q3: snapshot only where a revert can land
                    epoch_callback_ret = epoch_callback_fn(self)
                    assert isinstance(epoch_callback_ret, dict), \
                        f'The return type of the epoch_callback_fn should be dict, but found {type(epoch_callback_ret)}'
                progress_desc = f'Fitting model... Epoch {e} Loss: {loss:.4f}'
                if epoch_callback_ret is not None:
                    for metric in epoch_callback_ret:
                        progress_desc += f' | {metric}: {epoch_callback_ret[metric]}'
                        if not epoch_callback_res_registered:
                            self._loss_tracker.add_epoch_callback_result(metric, epoch_callback_ret[metric], e)
                    epoch_callback_res_registered = True

            if early_stopping_rule is not None and e % early_stopping_freq == 0:
                if e not in self.epoch_weights:
                    self._store_epoch_weights(e)           # a rule may name any epoch it was evaluated on
                try:
                    early_stopping_best_epoch = early_stopping_rule.compute(
                        self._loss_tracker.epoch_losses, self._loss_tracker.epoch_callback_results,
                        self._loss_tracker.called_epochs)
                    if early_stopping_rule.stop_training(e, early_stopping_best_epoch, epochs):
                        break
                except Exception as exc:
                    if not _is_invalid_validation_exc(exc): raise
                    self._warn(f'Failed to compute early stopping rule {early_stopping_rule.__class__.__name__}: {exc}')

            if early_stopping_best_epoch is not None:
                progress_desc += f' | {early_stopping_rule.__class__.__name__} best epoch: {early_stopping_best_epoch}'
            if self.verbose:
                _iter.set_description(progress_desc)

        if early_stopping_rule is not None and e % early_stopping_freq != 0:
            try:
                early_stopping_best_epoch = early_stopping_rule.compute(
                    self._loss_tracker.epoch_losses, self._loss_tracker.epoch_callback_results,
                    self._loss_tracker.called_epochs)
            except Exception as exc:
                if not _is_invalid_validation_exc(exc): raise
                self._warn(f'Failed to compute early stopping rule {early_stopping_rule.__class__.__name__}: {exc}')

        if early_stopping_best_epoch is not None and early_stopping_best_epoch != epochs:
            self._info(f'Reverting network weights to epoch {early_stopping_best_epoch} due to the evaluation of the '
                       f'early stopping rule {early_stopping_rule.__class__.__name__}.')
            self._revert_weights(early_stopping_best_epoch)

        self._finish_fit()
        self._info('Model fitted.')

    # ------------------------------------------------------------------ hooks
    @abstractmethod
    def _pre_fit(self, learning_rate, neg_ratio, reg_rate, **kwds):
        """Allocate device arenas / CSR, create the native model and the sampler."""

    @abstractmethod
    def _train_step(self, batch_size, reg_rate, want_loss, **kwds):
        """Sample one batch and run one native optimizer step; returns the float loss if want_loss else None."""

    @abstractmethod
    def _predict(self, uid, iid, **kwds):
        pass

    @abstractmethod
    def _rank_batch(self, uids, cand, cand_count, novelty):
        """uids [n], cand [n, max_cand] internal ids, cand_count [n] -> (iids [n, max_cand], scores, n_out)."""

    def _finish_fit(self):
        pass

    def _params_tensor(self):
        raise NotImplementedError

    # ------------------------------------------------------------------ snapshots (recommender_abc.py:336-352, Q3)
    def _store_epoch_weights(self, epoch):
        p = self._params_tensor()
        self.epoch_weights[epoch] = p.detach().clone() if p.numel() < (1 << 27) else p.detach().cpu()

    def _revert_weights(self, epoch):
        if epoch == 0 or epoch == self._step:
            # reference: epoch_weights[0 - 1] == the last step's weights, i.e. a no-op revert
            self._info(f'Network weights reverted from epoch {self._step} to epoch {epoch}.')
            return
        if epoch not in self.epoch_weights:
            # snapshots exist on callback / early-stopping epochs only (Q3); a rule that names any other epoch cannot
            # be honoured -- say so instead of claiming a revert
            self._logger.warning(f'No weight snapshot for epoch {epoch} (snapshots: {sorted(self.epoch_weights)}); '
                                 f'network weights stay at epoch {self._step}.')
            return
        p = self._params_tensor()
        p.copy_(self.epoch_weights[epoch].to(p.device))
        self._info(f'Network weights reverted from epoch {self._step} to epoch {epoch}.')

    # ------------------------------------------------------------------ public scoring API
    def predict(self, user_id, item_id, skip_errors=False, **kwds):
        assert self.fitted is True, 'The model requires to be fitted before being able to make predictions.'
        ds = self._data
        assert skip_errors or ds.user_to_uid(user_id) is not None, f'User {user_id} was not found.'
        assert skip_errors or ds.item_to_iid(item_id) is not None, f'Item {item_id} was not found.'
        prediction = None
        try:
            uid, iid = ds.user_to_uid(user_id), ds.item_to_iid(item_id)
            prediction = self._predict(uid, iid, **kwds)
            if prediction is None:
                raise Exception(f'Failed to predict(user_id={user_id}, item_id={item_id}): None was returned.')
        except Exception as e:
            if not skip_errors: raise e
        return prediction

    def recommend(self, user_id, n=None, novelty=True, interaction_threshold=None, **kwds):
        assert self.fitted is True, 'The model requires to be fitted before being able to make predictions.'
        assert self._data.user_to_uid(user_id) is not None, f'User {user_id} was not found.'
        if n is None: n = self.n_items
        uid = self._data.user_to_uid(user_id)
        recs = self._recommend(uid, n, novelty, interaction_threshold)
        return [(r, self._data.iid_to_item(iid)) for r, iid in recs]

    def _recommend(self, uid, n, novelty, threshold):
        ranked_items = self._rank(uid, range(0, self.n_items), n, novelty)
        if threshold is None:
            return ranked_items
        return list(filter(lambda x: x[0] >= threshold, ranked_items))

    def recommend_batch(self, user_ids, n=10, novelty=True, interaction_threshold=None, chunk=8192):
        """Batched recommend() over raw user ids: (items [U, n] raw ids, scores [U, n], counts [U]); row r holds what
        recommend(user_ids[r], n, novelty, interaction_threshold) returns, counts[r] entries of it.  Padding: -1 for
        integer raw item ids (None otherwise) and NaN scores.  1 <= n <= 2048; users go to the model's full-catalog
        top-k (topk_batch) `chunk` at a time."""
        assert self.fitted is True, 'The model requires to be fitted before being able to make predictions.'
        n = int(n)
        if not 1 <= n <= 2048:
            raise ValueError(f'recommend_batch: n must be in [1, 2048] (got {n}); use recommend() for longer lists')
        data = self._data
        user_ids = np.asarray(user_ids)
        uids = np.asarray(data.users_to_uids(user_ids)).astype(np.int32) if len(user_ids) else np.zeros(0, np.int32)
        unknown = np.flatnonzero(uids < 0)
        if len(unknown):
            raise AssertionError(f'User {user_ids[unknown[0]]} was not found.')
        raw = data.raw_items
        U = len(uids)
        int_ids = np.issubdtype(raw.dtype, np.integer)
        items = np.full((U, n), -1, np.int64) if int_ids else np.full((U, n), None, object)
        scores, counts = None, np.zeros(U, np.int64)
        for o in range(0, U, chunk):
            oi, os_, on = self.topk_batch(uids[o:o + chunk], n, novelty)
            on = np.asarray(on, np.int64)
            if scores is None:
                scores = np.full((U, n), np.nan, os_.dtype)
            valid = np.arange(n)[None, :] < on[:, None]
            if interaction_threshold is not None:      # scores are descending: the threshold keeps a prefix
                valid &= os_ >= interaction_threshold
                on = valid.sum(axis=1)
            items[o:o + chunk] = np.where(valid, raw[np.where(valid, oi, 0)], items[o:o + chunk])
            scores[o:o + chunk] = np.where(valid, os_, scores[o:o + chunk])
            counts[o:o + chunk] = on
        if scores is None:
            scores = np.full((U, n), np.nan, np.float32)
        return items, scores, counts

    def rank(self, user_id, item_ids, novelty=True, skip_invalid_items=True, **kwds):
        assert self.fitted is True, 'The model requires to be fitted before being able to make predictions.'
        assert self._data.user_to_uid(user_id) is not None, f'User {user_id} was not found.'
        uid = self._data.user_to_uid(user_id)
        iids = []
        for item_id in item_ids:
            iid = self._data.item_to_iid(item_id)
            if iid is not None:
                iids.append(iid)
            elif not skip_invalid_items:
                raise Exception(f'Item {item_id} was not found.')
        n = kwds.get('n', len(iids))
        assert n <= len(iids), \
            f'The number of best items to return must be <= len(item_ids) (current value is {n} > {len(iids)})'
        ranked_list = self._rank(uid, iids, n, novelty)
        return [(r, self._data.iid_to_item(iid)) for r, iid in ranked_list]

    def _rank(self, uid, iids, n, novelty):
        """[(score, iid)] ordered like heapq.nlargest over (score, iid) tuples (recommender_abc.py:454-461)."""
        iids = np.asarray(list(iids), dtype=np.int32)
        if len(iids) == 0 or n <= 0:
            return []
        out_i, out_s, n_out = self._rank_batch(np.array([uid], np.int32), iids[None, :],
                                               np.array([len(iids)], np.int32), novelty)
        k = min(int(n_out[0]), n)
        return [(out_s[0, j], int(out_i[0, j])) for j in range(k)]

    def rank_batch(self, user_ids, item_id_lists, novelty=True):
        """Batched rank() over raw ids: returns one ranked raw-item list per user (invalid items skipped).  A user
        the model was not trained on gets an empty list (rank() would assert; per-user callers skip such users)."""
        uids = self._data.users_to_uids(np.asarray(user_ids)).astype(np.int32)
        known = uids >= 0
        lens = [len(x) for x in item_id_lists]
        flat = np.concatenate([np.asarray(x) for x in item_id_lists]) if sum(lens) else np.zeros(0, np.int64)
        iids = self._data.items_to_iids(flat)
        max_c = max(1, max(lens) if lens else 1)
        cand = np.zeros((len(uids), max_c), np.int32)
        cnt = np.zeros(len(uids), np.int32)
        o = 0
        for r, ln in enumerate(lens):
            v = iids[o:o + ln]
            v = v[v >= 0]
            cand[r, :len(v)] = v
            cnt[r] = len(v) if known[r] else 0
            o += ln
        out_i, out_s, n_out = self._rank_batch(np.where(known, uids, 0).astype(np.int32), cand, cnt, novelty)
        items = self._data.raw_items
        return [items[out_i[r, :n_out[r]]].tolist() for r in range(len(uids))], out_s, n_out

    def rank_arrays(self, user_ids, cand, cand_off, novelty=True, chunk=32768):
        """Batched rank() over flat arrays: user_ids [n] raw, cand raw item ids with offsets cand_off [n+1].
        Returns (ranked raw items [n, Cmax] padded with -1, n_out [n]).  Unknown items are skipped
        (skip_invalid_items=True); users must be known."""
        data = self._data
        uids = data.users_to_uids(user_ids).astype(np.int32)
        assert (uids >= 0).all(), 'unknown user in rank_arrays'
        n = len(uids)
        lens = np.diff(cand_off).astype(np.int64)
        c_max = int(max(1, lens.max() if n else 1))
        iids = data.items_to_iids(cand).astype(np.int32)
        if n and (lens == c_max).all() and cand_off[0] == 0:          # uniform lists (the sampled protocol): a reshape
            padded = np.ascontiguousarray(iids.reshape(n, c_max))
        else:
            padded = np.full((n, c_max), -1, np.int32)
            rows = np.repeat(np.arange(n), lens)
            cols = np.arange(len(cand)) - np.repeat(cand_off[:-1], lens)
            padded[rows, cols] = iids
        out_items = np.full((n, c_max), -1, np.int64)
        n_out = np.zeros(n, np.int32)
        raw = data.raw_items
        for o in range(0, n, chunk):
            oi, _, on = self._rank_batch(uids[o:o + chunk], padded[o:o + chunk], lens[o:o + chunk].astype(np.int32),
                                         novelty)
            if (on == oi.shape[1]).all():                                # nothing filtered: every slot is valid
                out_items[o:o + chunk, :oi.shape[1]] = raw[oi]
            else:
                valid = np.arange(oi.shape[1])[None, :] < on[:, None]
                out_items[o:o + chunk, :oi.shape[1]] = np.where(valid, raw[np.where(valid, oi, 0)], -1)
            n_out[o:o + chunk] = on
        return out_items, n_out

    def _standardize_value(self, value):
        return (value - self.min_interaction) / (self.max_interaction - self.min_interaction)

    def _rescale_value(self, value):
        return self.min_interaction + (self.max_interaction - self.min_interaction) * value

    # ------------------------------------------------------------------ logging (recommender_abc.py:471-501)
    def _log_initial_info(self):
        self._info(f'Max. interaction value: {self.max_interaction}')
        self._info(f'Min. interaction value: {self.min_interaction}')
        self._info(f'Interaction threshold value: {self.interaction_threshold}')
        self._info(f'Number of unique users: {self.n_users}')
        self._info(f'Number of unique items: {self.n_items}')
        self._info(f'Number of training points: {self.n_rows}')
        sparsity = round(100 * (1 - (self.n_rows / (self.n_users * self.n_items))), 4)
        self._info(f'Sparsity level: approx. {sparsity}%')

    def _info(self, msg, **kw):
        if self.verbose: self._logger.info(msg)

    def _warn(self, msg, **kw):
        if self.verbose: self._logger.warning(msg)

    # ------------------------------------------------------------------ persistence (recommender_abc.py:503-524)
    _TRANSIENT = ('_native', '_ctx', '_torch', '_workspace', '_slots', '_loss_host', '_loss_dev', '_stream', '_lock',
                  '_mask_rng', '_mask_stream', '_keep_dev', '_sampler', '_dp', '_dp_dev', '_dp_gather', '_label_count', '_dz1', '_h_buf', '_keepalive', '_next', '_pool',
                  '_d_indptr', '_d_indices', '_d_seen_indptr', '_d_seen_indices', '_dev_sparse', '_logger', '_dev',
                  '_topk_scratch')

    def __getstate__(self):
        """joblib/pickle: device arenas go to host tensors, native handles are dropped and rebuilt on load."""
        st = {k: v for k, v in self.__dict__.items() if k not in self._TRANSIENT}
        for k in ('_params', '_adam_m', '_adam_v', '_grads'):
            if k in st: st[k] = st[k].cpu()
        L = getattr(self, '_L', None)
        st['_L'] = (type(L), {f: (list(getattr(L, f)) if hasattr(getattr(L, f), '__len__') else getattr(L, f))
                              for f, _ in L._fields_}) if L is not None else None
        st['epoch_weights'] = {}
        return st

    def __setstate__(self, st):
        L = st.pop('_L', None)
        self.__dict__.update(st)
        self._lock = threading.RLock()
        self._logger = logging.getLogger(f'{self.__class__.__name__}_CLOGGER')
        self._native = self._ctx = None
        if L is not None and self.fitted:
            import torch
            from .parallel import DataParallel
            self._torch = torch
            cls, fields = L
            self._L = cls()
            for f, v in fields.items():
                if isinstance(v, list):
                    arr = getattr(self._L, f)
                    for j, x in enumerate(v): arr[j] = x
                else:
                    setattr(self._L, f, v)
            self._dp = DataParallel()
            self._dev = torch.device(self.device or f'cuda:{torch.cuda.current_device()}')
            for k in ('_params', '_adam_m', '_adam_v', '_grads'):
                setattr(self, k, getattr(self, k).to(self._dev))
            self._build_native()

    def save(self, save_path):
        from joblib import dump
        dump(self, save_path)

    @staticmethod
    def load(load_path):
        from joblib import load
        return load(load_path)
