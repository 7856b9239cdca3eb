"""ctypes binding of libdrb.so (include/drb.h).  Host code is Python; PyTorch only owns device buffers.

There is no CPU fallback: if the library is missing the import of any compute path fails loudly; device entry
points fail with a RuntimeError when no sm_100 GPU is present.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libdrb.so')

DRB_LOSS = {'bce': 0, 'mse': 1}
DRB_LABEL = {'batch_mean': 0, 'per_user': 1}
DRB_GEMM = {'auto': 0, 'ffma': 1, 'tcgen05': 2, 'tcgen05_tf32': 3}
DMF_MAX_LAYERS = 8

vp = C.c_void_p
i32, i64, u64, f32, f64 = C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_double


class CdaeLayout(C.Structure):
    _fields_ = [('off_w2t', i64), ('off_w', i64), ('off_v', i64), ('off_b', i64), ('off_b2', i64), ('total', i64),
                ('ld', i32), ('items_pad', i32)]


class CdaeDesc(C.Structure):
    _fields_ = [('n_users', i32), ('n_items', i32), ('hidden', i32),
                ('params', vp), ('adam_m', vp), ('adam_v', vp), ('grads', vp),
                ('csr_indptr', vp), ('csr_indices', vp), ('seen_indptr', vp), ('seen_indices', vp),
                ('corruption_level', f32), ('loss_kind', i32), ('label_mode', i32),
                ('workspace', vp), ('workspace_bytes', i64), ('max_batch', i32), ('gemm_path', i32),
                ('output_mode', i32), ('neg_per_group', i32), ('neg_groups', i32)]


class OptimDesc(C.Structure):
    _fields_ = [('kind', i32), ('momentum', f32), ('nesterov', i32), ('rho', f32), ('centered', i32), ('beta1', f32),
                ('beta2', f32), ('epsilon', f32), ('amsgrad', i32), ('decay', f32), ('third_state', vp)]


class CdaeStepArgs(C.Structure):
    _fields_ = [('learning_rate', f32), ('beta1', f32), ('beta2', f32), ('epsilon', f32), ('reg_rate', f32),
                ('t', i32 * 5), ('philox_seed', u64), ('philox_step', u64), ('global_batch', i32),
                ('slot_offset', i32), ('skip_user_grad', i32), ('shard_items', i32), ('item_offset', i32),
                ('n_items_global', i64), ('v_rows', vp), ('keep_bytes', i64)]


class DmfLayout(C.Structure):
    _fields_ = [('n_layers_user', i32), ('n_layers_item', i32),
                ('off_kernel_user', i64 * DMF_MAX_LAYERS), ('off_bias_user', i64 * DMF_MAX_LAYERS),
                ('off_kernel_item', i64 * DMF_MAX_LAYERS), ('off_bias_item', i64 * DMF_MAX_LAYERS),
                ('ld_user', i32 * DMF_MAX_LAYERS), ('ld_item', i32 * DMF_MAX_LAYERS), ('total', i64)]


class DmfDesc(C.Structure):
    _fields_ = [('n_users', i32), ('n_items', i32), ('n_layers_user', i32), ('n_layers_item', i32),
                ('user_factors', i32 * DMF_MAX_LAYERS), ('item_factors', i32 * DMF_MAX_LAYERS),
                ('params', vp), ('adam_m', vp), ('adam_v', vp), ('grads', vp),
                ('csr_indptr', vp), ('csr_indices', vp), ('csr_values', vp), ('csr_row_scale', vp),
                ('csc_indptr', vp), ('csc_indices', vp), ('csc_values', vp), ('csc_row_scale', vp),
                ('workspace', vp), ('workspace_bytes', i64), ('max_batch', i32)]


class DmfStepArgs(C.Structure):
    _fields_ = [('learning_rate', f32), ('beta1', f32), ('beta2', f32), ('epsilon', f32), ('reg_rate', f32),
                ('t', i32 * 2)]


class CaserLayout(C.Structure):
    _fields_ = [('off_e', i64), ('off_p', i64), ('off_w2', i64), ('off_fv', i64), ('off_fh', i64), ('off_fc', i64),
                ('off_bv', i64), ('off_bh', i64), ('off_bfc', i64), ('off_b2', i64), ('total', i64),
                ('ld_e', i32), ('ld_x', i32), ('items_pad', i32)]


class CaserDesc(C.Structure):
    _fields_ = [('n_users', i32), ('n_items', i32), ('L', i32), ('T', i32), ('d', i32), ('n_v', i32), ('n_h', i32),
                ('neg_ratio', i32), ('dropout_rate', f32), ('params', vp), ('adam_m', vp), ('adam_v', vp),
                ('grads', vp), ('seq', vp), ('seq_indptr', vp), ('win_off', vp), ('n_windows', i64),
                ('seen_indptr', vp), ('seen_indices', vp), ('workspace', vp), ('workspace_bytes', i64),
                ('max_batch', i32)]


class CaserStepArgs(C.Structure):
    _fields_ = [('learning_rate', f32), ('beta1', f32), ('beta2', f32), ('epsilon', f32), ('reg_rate', f32),
                ('t', i32), ('philox_seed', u64), ('philox_step', u64)]


P = C.POINTER

# name -> (restype, argtypes); every symbol include/drb.h declares
SIGNATURES = {
    'drb_version': (C.c_int, []),
    'drb_last_error': (C.c_char_p, []),
    'drb_ctx_create': (C.c_int, [C.c_int, P(vp)]),
    'drb_ctx_destroy': (C.c_int, [vp]),
    'drb_ctx_set_stream': (C.c_int, [vp, vp]),
    'drb_ctx_synchronize': (C.c_int, [vp]),
    'drb_ctx_launch_count': (i64, [vp]),
    'drb_ctx_profile_enable': (C.c_int, [vp, C.c_int]),
    'drb_ctx_profile_read': (C.c_int, [vp, C.c_char_p, i64, vp, vp, i32, P(i32)]),
    'drb_rng_create': (C.c_int, [u64, P(vp)]),
    'drb_rng_destroy': (C.c_int, [vp]),
    'drb_rng_seed': (C.c_int, [vp, u64]),
    'drb_rng_random': (f64, [vp]),
    'drb_rng_getrandbits': (u64, [vp, C.c_int]),
    'drb_rng_randbelow': (i64, [vp, i64]),
    'drb_rng_random_fill': (C.c_int, [vp, i64, vp]),
    'drb_rng_sample_indices': (C.c_int, [vp, i64, i64, vp]),
    'drb_rng_shuffle_i64': (C.c_int, [vp, i64, vp]),
    'drb_rng_window': (C.c_int, [vp, vp]),
    'drb_rng_set_window': (C.c_int, [vp, vp]),
    'drb_rng_skip': (C.c_int, [vp, i64]),
    'drb_mtjump_create': (C.c_int, [i64, i32, P(vp)]),
    'drb_mtjump_destroy': (C.c_int, [vp]),
    'drb_mtjump_polys': (C.c_int, [vp, vp]),
    'drb_mtjump_apply_host': (C.c_int, [vp, i32, vp, vp]),
    'drb_rng_getstate': (C.c_int, [vp, vp]),
    'drb_rng_setstate': (C.c_int, [vp, vp]),
    'drb_sampler_create': (C.c_int, [i32, i32, vp, vp, vp, vp, vp, f64, u64, P(vp)]),
    'drb_sampler_destroy': (C.c_int, [vp]),
    'drb_sampler_sample': (C.c_int, [vp, i64, vp, vp, vp]),
    'drb_sampler_getstate': (C.c_int, [vp, vp]),
    'drb_sampler_setstate': (C.c_int, [vp, vp]),
    'drb_cdae_corruption_keep_mt': (C.c_int, [vp, vp, i32, i32, f64, vp, vp, vp, vp, i64]),
    'drb_mt_keep_device': (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, u64]),
    'drb_batch_offsets': (C.c_int, [vp, i32, vp, vp]),
    'drb_cdae_layout': (C.c_int, [i32, i32, i32, P(CdaeLayout)]),
    'drb_cdae_workspace_bytes': (i64, [i32, i32, i32, i32]),
    'drb_cdae_workspace_bytes_sampled': (i64, [i32, i32, i32, i32]),
    'drb_cdae_create': (C.c_int, [vp, P(CdaeDesc), P(vp)]),
    'drb_cdae_destroy': (C.c_int, [vp]),
    'drb_cdae_set_optimizer': (C.c_int, [vp, P(OptimDesc)]),
    'drb_cdae_step': (C.c_int, [vp, vp, vp, vp, i32, P(CdaeStepArgs), vp]),
    'drb_cdae_step_phases': (C.c_int, [vp, vp, vp, vp, i32, P(CdaeStepArgs), vp, i32]),
    'drb_cdae_label_count_buffer': (C.c_int, [vp, P(vp), P(i64)]),
    'drb_cdae_loss_buffer': (C.c_int, [vp, P(vp)]),
    'drb_dmf_loss_buffer': (C.c_int, [vp, P(vp)]),
    'drb_cdae_dz1_buffer': (C.c_int, [vp, P(vp), P(i64)]),
    'drb_cdae_h_buffer': (C.c_int, [vp, P(vp), P(i64)]),
    'drb_cdae_scatter_user_rows': (C.c_int, [vp, vp, vp, i32]),
    'drb_cdae_step_host': (C.c_int, [vp, vp, vp, vp, i32, P(CdaeStepArgs), vp]),
    'drb_cdae_hidden': (C.c_int, [vp, vp, i32, vp]),
    'drb_cdae_rank_candidates': (C.c_int, [vp, vp, i32, vp, vp, i32, i32, vp, vp, vp]),
    'drb_cdae_topk': (C.c_int, [vp, vp, i32, i32, i32, vp, vp, vp]),
    'drb_cdae_topk_exact': (C.c_int, [vp, vp, i32, i32, i32, vp, vp, vp]),
    'drb_cdae_predict_all': (C.c_int, [vp, vp, i32, vp]),
    'drb_cdae_predict_pairs': (C.c_int, [vp, vp, i32, vp, vp, vp, i32, vp]),
    'drb_dmf_layout': (C.c_int, [i32, i32, vp, i32, vp, i32, P(DmfLayout)]),
    'drb_dmf_workspace_bytes': (i64, [i32, i32, vp, i32, vp, i32, i32]),
    'drb_dmf_create': (C.c_int, [vp, P(DmfDesc), P(vp)]),
    'drb_dmf_destroy': (C.c_int, [vp]),
    'drb_dmf_set_optimizer': (C.c_int, [vp, P(OptimDesc)]),
    'drb_dmf_step': (C.c_int, [vp, vp, vp, vp, i32, P(DmfStepArgs), vp]),
    'drb_dmf_step_phases': (C.c_int, [vp, vp, vp, vp, i32, P(DmfStepArgs), vp, i32, i32]),
    'drb_dmf_grads_buffer': (C.c_int, [vp, P(vp), P(i64)]),
    'drb_dmf_step_host': (C.c_int, [vp, vp, vp, vp, i32, P(DmfStepArgs), vp]),
    'drb_dmf_forward_pairs': (C.c_int, [vp, vp, vp, i32, vp]),
    'drb_dmf_predict_pairs': (C.c_int, [vp, vp, i32, vp, vp, vp, i32, vp]),
    'drb_dmf_rank_candidates': (C.c_int, [vp, vp, i32, vp, vp, i32, i32, vp, vp, vp]),
    'drb_dmf_invalidate_cache': (C.c_int, [vp]),
    'drb_dmf_topk_scratch_bytes': (i64, [vp, i32]),
    'drb_dmf_topk': (C.c_int, [vp, vp, i32, i32, i32, vp, i64, vp, vp, vp]),
    'drb_caser_layout': (C.c_int, [i32, i32, i32, i32, i32, i32, i32, P(CaserLayout)]),
    'drb_caser_workspace_bytes': (i64, [i32, i32, i32, i32, i32, i32, i32, i32, i32]),
    'drb_caser_create': (C.c_int, [vp, P(CaserDesc), P(vp)]),
    'drb_caser_destroy': (C.c_int, [vp]),
    'drb_caser_set_optimizer': (C.c_int, [vp, P(OptimDesc)]),
    'drb_caser_step': (C.c_int, [vp, i32, P(CaserStepArgs), vp]),
    'drb_caser_loss_buffer': (C.c_int, [vp, P(vp)]),
    'drb_caser_batch_buffer': (C.c_int, [vp, P(vp), P(vp), P(i32)]),
    'drb_caser_user_rep': (C.c_int, [vp, vp, i32, vp]),
    'drb_caser_predict_all': (C.c_int, [vp, vp, i32, vp]),
    'drb_caser_predict_pairs': (C.c_int, [vp, vp, i32, vp, vp, vp, i32, vp]),
    'drb_caser_rank_candidates': (C.c_int, [vp, vp, i32, vp, vp, i32, i32, vp, vp, vp]),
    'drb_caser_topk': (C.c_int, [vp, vp, i32, i32, i32, vp, vp, vp]),
    'drb_debug_cdae_capture_logits': (C.c_int, [vp, vp]),
    'drb_debug_split_tf32': (C.c_int, [vp, vp, i32, i32, i32, vp, vp, vp, vp, i32, i32]),
    'drb_debug_umma_gemm': (C.c_int, [vp, vp, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp, i32, i32, vp, i32]),
    'drb_debug_split_f16': (C.c_int, [vp, vp, i32, i32, i32, f32, vp, vp, i32, vp, vp, i32, i32]),
    'drb_debug_umma_gemm_f16': (C.c_int, [vp, vp, vp, i32, vp, vp, i32, i32, i32, i32, i32, i32, i32, f32, vp, i32, i32, vp, i32]),
    'drb_eval_candidates': (C.c_int, [i64, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, i64, f64, i64, f64, i32, i32, i64,
                                      i32, i64, vp, vp, vp, vp, vp]),
    'drb_leave_k_out': (C.c_int, [i64, vp, i64, f64, i32, i64, i64, i32, vp]),
    'drb_eval_lookup': (C.c_int, [i64, vp, vp, vp, vp, vp, vp, vp, f64, i32, vp]),
    'drb_eval_metrics': (C.c_int, [i64, vp, vp, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, vp]),
    'drb_eval_topk_metrics': (C.c_int, [vp, i32, vp, vp, i32, vp, i32, f64, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32,
                                        vp, vp, vp, vp]),
}

_lib = None


def load():
    """Loads libdrb.so; raises if it has not been built (python -m drecpy_b200.build / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f'{LIB_PATH} not found: build it with `python drecpy_b200/build.py` '
                           '(drecpy_b200 has no CPU fallback)')
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code):
    if code != 0:
        msg = load().drb_last_error()
        raise RuntimeError(f'libdrb error {code}: {msg.decode() if msg else ""}')


def np_ptr(a):
    """Raw pointer of a C-contiguous numpy array (caller keeps it alive)."""
    assert a.flags['C_CONTIGUOUS']
    return a.ctypes.data_as(vp)


def t_ptr(t):
    """Raw device/host pointer of a torch tensor."""
    return vp(t.data_ptr()) if t is not None else vp(0)


class HostRng:
    """CPython random.Random replay living in libdrb (used for the CDAE corruption stream)."""

    def __init__(self, seed):
        self._h = vp()
        check(load().drb_rng_create(abs(int(seed)), C.byref(self._h)))

    def __del__(self):
        if getattr(self, '_h', None) and _lib is not None:
            _lib.drb_rng_destroy(self._h)
            self._h = None

    def random(self):
        return load().drb_rng_random(self._h)

    def randbelow(self, n):
        return load().drb_rng_randbelow(self._h, n)

    def getstate(self):
        st = np.zeros(625, np.uint32)
        check(load().drb_rng_getstate(self._h, np_ptr(st)))
        return st

    def setstate(self, st):
        st = np.ascontiguousarray(st, np.uint32)
        check(load().drb_rng_setstate(self._h, np_ptr(st)))

    @property
    def handle(self):
        return self._h


def profile_read(ctx):
    """{kernel name: (total ms, launches)} accumulated since profiling was enabled / last read."""
    names = C.create_string_buffer(4096)
    ms = np.zeros(64, np.float64)
    cnt = np.zeros(64, np.int64)
    n = i32(0)
    check(load().drb_ctx_profile_read(ctx, names, 4096, np_ptr(ms), np_ptr(cnt), 64, C.byref(n)))
    keys = names.value.decode().split('\n')[:n.value]
    return {k: (float(ms[j]), int(cnt[j])) for j, k in enumerate(keys)}
