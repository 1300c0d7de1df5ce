"""CPU tests of the drop-in boundary: the C-ABI library loads, exports every
symbol include/muzero_b200.h declares, its host-only entry points behave, and
the Python mirror keeps the reference's interface.  No compute calls (no GPU)."""
import ctypes as C
import inspect
import os
import re

import numpy as np
import pytest
import torch

from conftest import ROOT
from muzero_b200 import _lib


def header_symbols():
    src = open(os.path.join(ROOT, 'include', 'muzero_b200.h')).read()
    src = re.sub(r'/\*.*?\*/', '', src, flags=re.S)
    return sorted(set(re.findall(r'\b(mz_[a-z_0-9]+)\s*\(', src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.lib()
    names = header_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f'{n} declared in the header but not exported'
    assert sorted(_lib.PROTOTYPES) == names, 'ctypes prototypes and header disagree'


def test_view_enum_matches_header():
    src = open(os.path.join(ROOT, 'include', 'muzero_b200.h')).read()
    body = src[src.index('enum mz_view {'):src.index('MZ_VIEW__COUNT')]
    names = re.findall(r'MZ_VIEW_([A-Z_]+)\b', re.sub(r'/\*.*?\*/', '', body, flags=re.S))
    assert names == _lib.VIEWS


def test_host_only_entry_points():
    lib = _lib.lib()
    assert lib.mz_version() == 100
    cfg = _lib.PoolConfig(num_trees=4096, num_actions=10, num_simulations=25, hidden_bytes=256, is_board_game=1,
                          has_known_bounds=1, bound_min=-1.0, bound_max=1.0, discount=1.0)
    n = C.c_size_t()
    assert lib.mz_pool_arena_bytes(C.byref(cfg), C.byref(n)) == 0
    edges = 4096 * 26 * 10 * 16
    hidden = 4096 * 26 * 256
    assert edges + hidden < n.value < 1.2 * (edges + hidden) + (1 << 20) + 4096 * 624 * 4 * 1.1
    # the reference asserts discount == 1 for board games (mcts.py:349-350)
    cfg.discount = 0.997
    assert lib.mz_pool_arena_bytes(C.byref(cfg), C.byref(n)) == _lib.MZ_EINVAL
    assert b'mcts.py:349' in lib.mz_last_error()
    with pytest.raises(ValueError):
        _lib.check(_lib.MZ_EINVAL)
    cfg.discount, cfg.num_simulations = 1.0, 70000
    assert lib.mz_pool_arena_bytes(C.byref(cfg), C.byref(n)) == _lib.MZ_EINVAL
    ncfg = _lib.NetConfig(kind=_lib.MZ_NET_MLP, in_channels=81, in_h=1, in_w=1, num_actions=10, num_planes=256,
                          num_res_blocks=0, hidden_dim=64, value_support=1, reward_support=1)
    hb = C.c_int32()
    assert lib.mz_net_hidden_bytes(C.byref(ncfg), C.byref(hb)) == 0 and hb.value == 256
    assert lib.mz_net_arena_bytes(C.byref(ncfg), 4096, C.byref(n)) == 0 and n.value >= 2 * 126092 * 4


def test_uct_search_signature_is_the_reference_one():
    from muzero_b200.mcts import uct_search
    sig = inspect.signature(uct_search)
    assert list(sig.parameters) == ['state', 'network', 'device', 'config', 'temperature', 'actions_mask',
                                    'current_player', 'opponent_player', 'deterministic']
    assert sig.parameters['deterministic'].default is False


def test_config_mirrors_reference_values():
    import muzero_b200 as mz
    c = mz.make_gomoku_config(use_tensorboard=False)
    assert (c.num_simulations, c.discount, c.root_dirichlet_alpha, c.root_exploration_eps) == (200, 1.0, 0.03, 0.25)
    assert (c.pb_c_base, c.pb_c_init, c.known_bounds, c.is_board_game) == (19652, 1.25, mz.KnownBounds(-1, 1), True)
    assert (c.num_planes, c.num_res_blocks, c.unroll_steps, c.weight_decay) == (128, 8, 5, 1e-4)
    t = mz.make_tictactoe_config(use_tensorboard=False)
    assert (t.num_simulations, t.root_dirichlet_alpha, t.num_planes, t.hidden_dim) == (25, 0.25, 256, 64)
    assert t.visit_softmax_temperature_fn(5, 0) == 1.0 and t.visit_softmax_temperature_fn(6, 0) == 0.1
    k = mz.make_classic_config(use_tensorboard=False)
    assert (k.num_simulations, k.discount, k.known_bounds, k.value_support_size) == (50, 0.997, None, 31)
    assert [k.visit_softmax_temperature_fn(0, s) for s in (0, 30000, 60000)] == [1.0, 0.5, 0.25]
    a = mz.make_atari_config(use_tensorboard=False)
    assert (a.num_simulations, a.value_support_size, a.reward_support_size, a.td_steps) == (30, 61, 61, 10)


def test_reference_checkpoints_load_unchanged():
    import muzero_b200 as mz
    from conftest import GOLDEN
    for name, kw in (('tictactoe', dict(input_shape=(9, 3, 3), num_actions=10, num_planes=256, value_support_size=1,
                                        reward_support_size=1, hidden_dim=64)),
                     ('cartpole', dict(input_shape=(4, 5), num_actions=2, num_planes=512, value_support_size=31,
                                       reward_support_size=31, hidden_dim=64))):
        sd = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, f'ckpt_{name}.npz')).items()}
        net = mz.MuZeroMLPNet(**kw)
        net.load_state_dict(sd)                      # strict: every key present, nothing extra
        assert list(net.state_dict().keys()) == list(sd.keys())


def test_conv_state_dict_keys_follow_the_reference_names():
    import muzero_b200 as mz
    net = mz.MuZeroBoardGameNet((9, 9, 9), 82, 2, 32)
    keys = list(net.state_dict().keys())
    for k in ('represent_net.conv_block.0.weight', 'represent_net.res_blocks.1.conv_block2.1.running_var',
              'dynamics_net.conv_block.0.weight', 'dynamics_net.reward_head.4.bias',
              'prediction_net.policy_net.4.weight', 'prediction_net.value_net.0.weight'):
        assert k in keys
    assert net.state_dict()['dynamics_net.conv_block.0.weight'].shape == (32, 32 + 82, 3, 3)
    at = mz.MuZeroAtariNet((16, 96, 96), 18, 2, 128, 61, 61)
    assert at.state_dict()['represent_net.conv_1.weight'].shape == (128, 16, 3, 3)
    assert at.state_dict()['prediction_net.value_net.4.weight'].shape == (61, 36)


def test_no_cpu_fallback():
    import muzero_b200 as mz
    net = mz.MuZeroMLPNet((4, 5), 2, 512, 31, 31, 64)
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match='CUDA only'):
            net.initial_inference(torch.zeros(1, 4, 5))
        with pytest.raises(RuntimeError):
            mz.SearchPool(4, 2, mz.make_classic_config(use_tensorboard=False), 256, device='cpu')


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, 'muzero_b200')
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle\b', src, flags=re.M), f'{f} imports the oracle'


def test_fma_division_sequence_is_correctly_rounded(tmp_path):
    """div_by_count of csrc/mcts.cu (reciprocal + one FMA correction) == IEEE division for every visit count:
    compiled and searched on the CPU (tools/fastdiv_check.c, 5 % of the full search)."""
    import shutil
    import subprocess
    if shutil.which('gcc') is None or 'fma' not in open('/proc/cpuinfo').read():
        pytest.skip('needs gcc and a CPU with FMA')
    exe = str(tmp_path / 'fastdiv_check')
    subprocess.run(['gcc', '-O2', '-mfma', '-ffp-contract=off', '-o', exe, os.path.join(ROOT, 'tools', 'fastdiv_check.c'),
                    '-lm'], check=True)
    r = subprocess.run([exe, '5'], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    assert ' 0 mismatches' in r.stdout


def test_conv_hidden_slot_layout_round_trip_on_cpu():
    """The engine's hidden-state slot of a conv net is [C/8][H*W][8] fp16, no padding around the board:
    reference layout -> slot -> reference layout."""
    import muzero_b200 as mz
    net = mz.MuZeroBoardGameNet((9, 9, 9), 82, 1, 32)
    assert net.grid_pad == 0
    assert net.hidden_bytes == 9 * 9 * 32 * 2
    h = (torch.arange(2 * 32 * 81, dtype=torch.float32).reshape(2, 32, 9, 9) % 251) / 256.0    # fp16-exact values
    slots = net.hidden_from_reference(h)
    assert slots.dtype == torch.uint8 and tuple(slots.shape) == (2, net.hidden_bytes)
    assert torch.equal(net.hidden_to_reference(slots), h)
    # element (q = y*W + x, c) of a slot lives at ((c/8) * PB + q) * 8 + c % 8, PB = 81
    v = slots.view(torch.float16).reshape(2, 4, 81, 8)
    assert float(v[1, 2, 3 * 9 + 5, 7]) == float(h[1, 2 * 8 + 7, 3, 5])
