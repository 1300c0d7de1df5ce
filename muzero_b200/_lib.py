"""ctypes binding of ``libmuzero_b200.so`` (the C ABI in include/muzero_b200.h).

There is no fallback: if the shared library is missing this module raises at
import of the first symbol, and every entry point that touches the device
requires CUDA.  Build with ``python -c "import __graft_entry__ as g; g.build()"``.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libmuzero_b200.so')

MZ_OK, MZ_EINVAL, MZ_ECUDA, MZ_ENOMEM, MZ_ESTATE = 0, -1, -2, -3, -4
MZ_DEVERR_POOL_FULL, MZ_DEVERR_NAN_POLICY = 1, 2
MZ_NET_MLP, MZ_NET_BOARD, MZ_NET_ATARI = 0, 1, 2

VIEWS = ['EDGES', 'PRIOR', 'ROOT_W', 'ROOT_N', 'MINMAX', 'COUNT', 'LEAF_PARENT', 'LEAF_ACTION', 'LEAF_DEPTH',
         'SRC_SLOT', 'DST_SLOT', 'PATH', 'NODE_PARENT', 'NODE_MOVE', 'NODE_VALUE', 'RNG_KEY', 'RNG_POS', 'HIDDEN', 'REWARD',
         'VALUE', 'ERROR', 'STATS', 'EDGE_W', 'EDGE_REWARD']
VIEW = {name: i for i, name in enumerate(VIEWS)}


class PoolConfig(C.Structure):
    _fields_ = [('num_trees', C.c_int32), ('num_actions', C.c_int32), ('num_simulations', C.c_int32),
                ('hidden_bytes', C.c_int32), ('is_board_game', C.c_int32), ('has_known_bounds', C.c_int32),
                ('bound_min', C.c_double), ('bound_max', C.c_double), ('discount', C.c_double)]


class TrainConfig(C.Structure):
    _fields_ = [('in_channels', C.c_int32), ('board_h', C.c_int32), ('board_w', C.c_int32), ('num_actions', C.c_int32),
                ('num_planes', C.c_int32), ('num_res_blocks', C.c_int32), ('batch', C.c_int32),
                ('unroll_steps', C.c_int32)]


class NetConfig(C.Structure):
    _fields_ = [('kind', C.c_int32), ('in_channels', C.c_int32), ('in_h', C.c_int32), ('in_w', C.c_int32),
                ('num_actions', C.c_int32), ('num_planes', C.c_int32), ('num_res_blocks', C.c_int32),
                ('hidden_dim', C.c_int32), ('value_support', C.c_int32), ('reward_support', C.c_int32)]


class DebugTensor(C.Structure):
    _fields_ = [('ptr', C.c_void_p), ('kind', C.c_int32), ('stage', C.c_int32), ('index', C.c_int32),
                ('plane_rows', C.c_int32), ('groups', C.c_int32), ('h', C.c_int32), ('w', C.c_int32),
                ('batch', C.c_int32), ('src', C.c_int32), ('residual', C.c_int32)]


MZ_DEBUG_MAX_LAYERS = 34
MZ_DEBUG_OBS, MZ_DEBUG_CONV, MZ_DEBUG_POOL, MZ_DEBUG_NORM, MZ_DEBUG_MLP = 0, 1, 2, 3, 4


class DebugLaunch(C.Structure):
    _fields_ = ([(k, C.c_int32) for k in ('num_layers', 'tile_rows', 'resident', 'khalf', 'pair', 'sub', 'multi_pass',
                                          'grid', 'num_tiles', 'cg', 'n', 'h', 'w', 'batch')] +
                [(k, C.c_int32 * MZ_DEBUG_MAX_LAYERS) for k in ('out', 'pass_', 'flags', 'dep0', 'res_layer', 'fwd')])


_P = C.c_void_p
# name -> (restype, argtypes); every symbol include/muzero_b200.h declares
PROTOTYPES = {
    'mz_last_error': (C.c_char_p, []),
    'mz_version': (C.c_int, []),
    'mz_set_pdl': (C.c_int, [C.c_int]),
    'mz_device_check': (C.c_int, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'mz_pool_arena_bytes': (C.c_int, [C.POINTER(PoolConfig), C.POINTER(C.c_size_t)]),
    'mz_pool_create': (C.c_int, [C.POINTER(PoolConfig), C.POINTER(C.c_double), _P, C.c_size_t, C.POINTER(_P)]),
    'mz_pool_destroy': (C.c_int, [_P]),
    'mz_pool_set_tree_ctas': (C.c_int, [_P, C.c_int]),
    'mz_pool_view': (C.c_int, [_P, C.c_int, C.POINTER(_P), C.POINTER(C.c_size_t)]),
    'mz_rng_seed': (C.c_int, [_P, _P, _P]),
    'mz_dirichlet': (C.c_int, [_P, C.c_double, _P, _P]),
    'mz_search_reset': (C.c_int, [_P, _P, _P, C.c_double, _P, _P, _P, _P]),
    'mz_select': (C.c_int, [_P, _P]),
    'mz_replay_sample_uniform': (C.c_int, [C.c_int64, C.c_int32, _P, _P, _P, _P, _P]),
    'mz_replay_sample_prioritized': (C.c_int, [C.c_int64, C.c_int32, _P, C.c_float, C.c_float, _P, _P, _P, _P, _P, _P, _P]),
    'mz_replay_scatter': (C.c_int, [_P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int64, _P]),
    'mz_replay_gather': (C.c_int, [_P, _P, _P, C.c_int64, C.c_int64, _P]),
    'mz_replay_update_priorities': (C.c_int, [_P, _P, _P, C.c_int32, _P]),
    'mz_expand_backup': (C.c_int, [_P, _P, _P, _P]),
    'mz_expand_backup_select': (C.c_int, [_P, _P, _P, _P]),
    'mz_root_policy': (C.c_int, [_P, _P, _P, C.c_int, _P, _P, _P, _P, _P]),
    'mz_net_hidden_bytes': (C.c_int, [C.POINTER(NetConfig), C.POINTER(C.c_int32)]),
    'mz_net_arena_bytes': (C.c_int, [C.POINTER(NetConfig), C.c_int32, C.POINTER(C.c_size_t)]),
    'mz_net_create': (C.c_int, [C.POINTER(NetConfig), C.POINTER(_P), C.c_int32, C.c_int32, _P, C.c_size_t,
                                C.POINTER(_P)]),
    'mz_net_destroy': (C.c_int, [_P]),
    'mz_net_initial': (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    'mz_net_initial_frames': (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    'mz_net_initial_search': (C.c_int, [_P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, C.c_int32, _P, C.c_double,
                                        C.c_double, _P, _P, _P]),
    'mz_net_recurrent': (C.c_int, [_P, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'mz_search_run': (C.c_int, [_P, _P, _P]),
    'mz_net_set_fused_search': (C.c_int, [_P, C.c_int32]),
    'mz_net_set_cta_limit': (C.c_int, [_P, C.c_int32]),
    'mz_net_profile_begin': (C.c_int, [_P]),
    'mz_net_debug_capture_bytes': (C.c_int, [_P, C.c_int32, C.POINTER(C.c_size_t)]),
    'mz_net_debug_capture': (C.c_int, [_P, _P, C.c_size_t]),
    'mz_net_debug_tensor': (C.c_int, [_P, C.c_int32, C.POINTER(DebugTensor), C.POINTER(C.c_int32)]),
    'mz_net_debug_launch': (C.c_int, [_P, C.c_int32, C.POINTER(DebugLaunch), C.POINTER(C.c_int32)]),
    'mz_net_profile_end': (C.c_int, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    'mz_env_arena_bytes': (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_size_t)]),
    'mz_env_create': (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.c_size_t, C.POINTER(_P)]),
    'mz_env_destroy': (C.c_int, [_P]),
    'mz_env_view': (C.c_int, [_P, C.c_int32, C.POINTER(_P), C.POINTER(C.c_size_t)]),
    'mz_env_reset': (C.c_int, [_P, _P, _P, _P]),
    'mz_env_step': (C.c_int, [_P, _P, _P, _P, _P, _P, _P]),
    'mz_targets_nstep': (C.c_int, [C.c_int32, C.c_int32, _P, _P, _P, C.c_int32, _P, _P, _P, _P]),
    'mz_targets_mc': (C.c_int, [C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    'mz_unroll_sequences': (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                      _P, _P]),
    'mz_train_arena_bytes': (C.c_int, [C.POINTER(TrainConfig), C.POINTER(C.c_size_t)]),
    'mz_train_create': (C.c_int, [C.POINTER(TrainConfig), _P, C.c_size_t, C.POINTER(_P)]),
    'mz_train_destroy': (C.c_int, [_P]),
    'mz_train_bind': (C.c_int, [_P, C.POINTER(_P), C.c_int32, _P]),
    'mz_train_begin_step': (C.c_int, [_P, _P]),
    'mz_train_tower_forward': (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    'mz_train_tower_backward': (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P]),
    'mz_head_conv_forward': (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P]),
    'mz_head_conv_scratch_bytes': (C.c_size_t, [C.c_int64, C.c_int32, C.c_int32]),
    'mz_head_conv_backward': (C.c_int, [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _P]),
    'mz_head_tail_forward': (C.c_int, [_P] * 10 + [C.c_int32] * 5 + [C.c_float, C.c_float, _P]),
    'mz_head_tail_backward': (C.c_int, [_P] * 11 + [C.c_int32] * 5 + [_P]),
    'mz_adam_chunk_elements': (C.c_int, []),
    'mz_adam_step': (C.c_int, [_P, _P, _P, C.c_int32, _P, _P, C.c_double, C.c_double, C.c_double, C.c_double, _P]),
    'mz_train_stacked_calls': (C.c_int, [_P, C.POINTER(C.c_int32)]),
    'mz_train_tower_forward_calls': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    'mz_train_tower_backward_calls': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    'mz_train_join': (C.c_int, [_P, _P]),
    'mz_train_end_step': (C.c_int, [_P, _P]),
    'mz_train_debug_view': (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(_P), C.POINTER(C.c_size_t),
                                      C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    'mz_launch_count': (C.c_uint64, []),
}

_lib = None


def lib() -> C.CDLL:
    """The loaded library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f'{LIB_PATH} is missing: the CUDA extension has not been built '
                              '(run __graft_entry__.build()); muzero_b200 has no CPU fallback')
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)          # AttributeError here = header/library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


class MuZeroB200Error(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc == MZ_OK:
        return
    msg = lib().mz_last_error().decode()
    if rc == MZ_EINVAL:
        raise ValueError(msg)
    if rc == MZ_ENOMEM:
        raise MemoryError(msg)
    raise MuZeroB200Error(f'[{rc}] {msg}')


def ptr(t) -> int:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), 'the C ABI takes contiguous CUDA tensors'
    return t.data_ptr()


def current_stream() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
