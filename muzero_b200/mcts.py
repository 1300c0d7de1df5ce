"""Batched GPU tree search: drop-in ``uct_search`` plus ``uct_search_batch``.

Reference interface mirrored here (michaelnny/muzero, muzero/mcts.py):
  mcts.py:302-407  uct_search(state, network, device, config, temperature, actions_mask,
                              current_player, opponent_player, deterministic=False)
                   -> (action: int, pi: float64[A], root value: float)

All tree arithmetic happens in the CUDA kernels of csrc/mcts.cu behind the C
ABI (include/muzero_b200.h).  This module only validates arguments the way the
reference does, draws the Dirichlet noise from numpy when bit-exact stream
continuity with ``np.random`` is requested, and sequences the launches.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import _lib
from .network import MuZeroNet, StackedFrames


def _capture(enqueue) -> 'torch.cuda.CUDAGraph':
    """Capture one search into a CUDA graph.  The tree / MLP kernels are launched with the programmatic-dependent-launch
    attribute (a kernel's prologue overlaps its predecessor's tail); should a driver refuse such launches under stream
    capture, the library falls back to ordinary launches and the capture is repeated."""
    try:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            enqueue()
        return g
    except Exception:                                           # noqa: BLE001
        _lib.check(_lib.lib().mz_set_pdl(0))
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            enqueue()
        return g


def pb_c_table(num_simulations: int, pb_c_base: float, pb_c_init: float) -> np.ndarray:
    """The exploration factor of mcts.py:193-195 for every parent visit count,
    evaluated with CPython ``math`` exactly as the reference evaluates it."""
    return np.array([(math.log((n + pb_c_base + 1) / pb_c_base) + pb_c_init) * math.sqrt(n)
                     for n in range(num_simulations + 2)], dtype=np.float64)


class SearchPool:
    """GPU-resident node pool + search state for ``num_trees`` independent trees.

    Replaces the ``Node`` / ``MinMaxStats`` object graph of mcts.py:33-217 with
    the struct-of-arrays arena described in DESIGN.md.
    """

    def __init__(self, num_trees: int, num_actions: int, config, hidden_bytes: int,
                 device: Union[str, torch.device] = 'cuda') -> None:
        if config.is_board_game:
            assert config.discount == 1.0            # mcts.py:349-350
        self.device = torch.device(device)
        if self.device.type != 'cuda':
            raise RuntimeError('SearchPool lives on a CUDA device (no CPU fallback)')
        if self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.B, self.A, self.S = int(num_trees), int(num_actions), int(config.num_simulations)
        self.hidden_bytes = int(hidden_bytes)
        kb = config.known_bounds
        self.cfg = _lib.PoolConfig(
            num_trees=self.B, num_actions=self.A, num_simulations=self.S, hidden_bytes=self.hidden_bytes,
            is_board_game=int(bool(config.is_board_game)), has_known_bounds=int(kb is not None),
            bound_min=float(kb.min) if kb is not None else 0.0, bound_max=float(kb.max) if kb is not None else 0.0,
            discount=float(config.discount))
        lib = _lib.lib()
        nbytes = C.c_size_t()
        _lib.check(lib.mz_pool_arena_bytes(C.byref(self.cfg), C.byref(nbytes)))
        with torch.cuda.device(self.device):
            self.arena = torch.empty(nbytes.value + 256, dtype=torch.uint8, device=self.device)
            self._base = (self.arena.data_ptr() + 255) // 256 * 256
            table = pb_c_table(self.S, config.pb_c_base, config.pb_c_init)
            self.handle = C.c_void_p()
            _lib.check(lib.mz_pool_create(C.byref(self.cfg), table.ctypes.data_as(C.POINTER(C.c_double)),
                                          self._base, nbytes.value, C.byref(self.handle)))
        self.arena_bytes = nbytes.value
        self._views = {}
        # mz_pool_create zeroes the MT19937 states, and an all-zero state emits 0 forever (NaN Dirichlet noise, a
        # degenerate tie-break).  Every new pool therefore starts from OS entropy -- NOT from np.random, whose global
        # stream the drop-in uct_search must leave exactly where the reference would.  seed() / set_rng_states()
        # replace these streams when a reproducible search is wanted.
        self.seed(np.random.SeedSequence().generate_state(self.B, dtype=np.uint32))

    def __del__(self):
        try:
            if getattr(self, 'handle', None):
                _lib.lib().mz_pool_destroy(self.handle)
                self.handle = None
        except Exception:
            pass

    # -- typed views into the arena ------------------------------------------
    _VIEW_TYPES = {
        'EDGES': (torch.uint8, 8), 'EDGE_W': (torch.float64, None), 'EDGE_REWARD': (torch.float32, None), 'PRIOR': (torch.float64, None), 'ROOT_W': (torch.float64, None),
        'ROOT_N': (torch.int32, None), 'MINMAX': (torch.float64, 2), 'COUNT': (torch.int32, None),
        'LEAF_PARENT': (torch.int32, None), 'LEAF_ACTION': (torch.int32, None), 'LEAF_DEPTH': (torch.int32, None),
        'SRC_SLOT': (torch.int32, None), 'DST_SLOT': (torch.int32, None), 'PATH': (torch.int32, None),
        'NODE_PARENT': (torch.int32, None), 'NODE_MOVE': (torch.int32, None), 'NODE_VALUE': (torch.float32, None),
        'RNG_KEY': (torch.int32, 624),
        'RNG_POS': (torch.int32, None), 'HIDDEN': (torch.uint8, None), 'REWARD': (torch.float32, None),
        'VALUE': (torch.float32, None), 'ERROR': (torch.int32, None), 'STATS': (torch.int64, None),
    }

    def view(self, name: str) -> torch.Tensor:
        """Zero-copy tensor over one of the pool's buffers (see enum mz_view)."""
        if name not in self._views:
            p, n = C.c_void_p(), C.c_size_t()
            _lib.check(_lib.lib().mz_pool_view(self.handle, _lib.VIEW[name], C.byref(p), C.byref(n)))
            off = p.value - self.arena.data_ptr()
            dt, _ = self._VIEW_TYPES[name]
            self._views[name] = self.arena[off:off + n.value].view(dt)
        return self._views[name]

    @property
    def hidden(self) -> torch.Tensor:
        """[B*(S+1), hidden_bytes] uint8 slot array."""
        return self.view('HIDDEN').view(self.B * (self.S + 1), max(self.hidden_bytes, 1)) \
            if self.hidden_bytes else self.view('HIDDEN')

    def _call(self, fn, *args):
        with torch.cuda.device(self.device):
            _lib.check(fn(self.handle, *args, _lib.current_stream()))

    # -- RNG -------------------------------------------------------------------
    def seed(self, seeds) -> None:
        """``np.random.seed(seeds[t])`` for each tree, done on the device."""
        s = torch.as_tensor(np.asarray(seeds, dtype=np.uint32).astype(np.int64), device=self.device).to(torch.int32)
        assert s.shape == (self.B,)
        self._call(_lib.lib().mz_rng_seed, _lib.ptr(s.contiguous()))

    def set_rng_states(self, states: Sequence) -> None:
        """Load numpy legacy states (``RandomState.get_state()`` tuples), one per tree."""
        keys = np.stack([np.asarray(st[1], dtype=np.uint32) for st in states]).view(np.int32)
        pos = np.array([st[2] for st in states], dtype=np.int32)
        self.view('RNG_KEY').view(self.B, 624).copy_(torch.from_numpy(keys))
        self.view('RNG_POS').copy_(torch.from_numpy(pos))

    def get_rng_states(self):
        keys = self.view('RNG_KEY').view(self.B, 624).cpu().numpy().view(np.uint32)
        pos = self.view('RNG_POS').cpu().numpy()
        return [('MT19937', keys[t].copy(), int(pos[t]), 0, 0.0) for t in range(self.B)]

    def dirichlet(self, alpha: float) -> torch.Tensor:
        out = torch.empty((self.B, self.A), dtype=torch.float64, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().mz_dirichlet(self.handle, float(alpha), _lib.ptr(out), _lib.current_stream()))
        return out

    # -- search steps ------------------------------------------------------------
    def reset(self, pi_probs: torch.Tensor, noise: Optional[torch.Tensor], eps: float,
              mask: Optional[torch.Tensor], players: Optional[torch.Tensor],
              root_reward: Optional[torch.Tensor] = None) -> None:
        assert pi_probs.dtype == torch.float32 and pi_probs.shape == (self.B, self.A)
        if mask is not None:
            assert mask.shape == pi_probs.shape          # mcts.py:293
        self._call(_lib.lib().mz_search_reset, _lib.ptr(pi_probs), _lib.ptr(noise), float(eps), _lib.ptr(mask),
                   _lib.ptr(players), _lib.ptr(root_reward))

    def select(self) -> None:
        self._call(_lib.lib().mz_select)

    def expand_backup(self, reward: Optional[torch.Tensor] = None, value: Optional[torch.Tensor] = None) -> None:
        self._call(_lib.lib().mz_expand_backup, _lib.ptr(reward), _lib.ptr(value))

    def root_policy(self, mask: Optional[torch.Tensor], temperature: torch.Tensor, deterministic: bool):
        dev = self.device
        action = torch.empty(self.B, dtype=torch.int32, device=dev)
        pi = torch.empty((self.B, self.A), dtype=torch.float64, device=dev)
        rootv = torch.empty(self.B, dtype=torch.float64, device=dev)
        visits = torch.empty((self.B, self.A), dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().mz_root_policy(self.handle, _lib.ptr(mask), _lib.ptr(temperature),
                                                 int(bool(deterministic)), _lib.ptr(action), _lib.ptr(pi),
                                                 _lib.ptr(rootv), _lib.ptr(visits), _lib.current_stream()))
        return action, pi, rootv, visits

    def check_errors(self) -> None:
        """Synchronising read of the sticky device error word."""
        e = int(self.view('ERROR').cpu()[0])
        if e:
            self.view('ERROR').zero_()
        if e & _lib.MZ_DEVERR_POOL_FULL:
            raise RuntimeError('Node already expanded.')          # mcts.py:90-91: more expansions than slots
        if e & _lib.MZ_DEVERR_NAN_POLICY:
            raise ValueError('probabilities contain NaN')           # what np.random.choice raises (mcts.py:404)

    # -- debug / parity ------------------------------------------------------------
    def dump_tree(self, t: int) -> dict:
        """Host copy of tree ``t`` as node-indexed arrays (expansion order), the
        same shape as ``oracle.mcts_oracle.SearchTrace``."""
        A, n = self.A, self.S + 1
        count = int(self.view('COUNT')[t].cpu())
        hot = self.view('EDGES').view(self.B, n * A * 8)[t].cpu().numpy().view(
            np.dtype([('N', '<u2'), ('child', '<u2'), ('Q', '<f4')])).reshape(n, A)
        rec = np.zeros((n, A), dtype=np.dtype([('W', '<f8'), ('R', '<f4'), ('N', '<u2'), ('child', '<u2')]))
        rec['N'], rec['child'] = hot['N'], hot['child']
        visited = hot['N'] > 0                            # the cold words of an edge are defined once it was visited
        rec['W'] = np.where(visited, self.view('EDGE_W').view(self.B, n * A)[t].cpu().numpy().reshape(n, A), 0.0)
        rec['R'] = np.where(visited, self.view('EDGE_REWARD').view(self.B, n * A)[t].cpu().numpy().reshape(n, A), 0.0)
        parent = self.view('NODE_PARENT').view(self.B, n)[t].cpu().numpy()[:count].copy()
        move = self.view('NODE_MOVE').view(self.B, n)[t].cpu().numpy()[:count].copy()
        N = np.zeros(count, np.int32); W = np.zeros(count, np.float64); R = np.zeros(count, np.float64)
        N[0] = int(self.view('ROOT_N')[t].cpu()); W[0] = float(self.view('ROOT_W')[t].cpu())
        for i in range(1, count):
            e = rec[parent[i], move[i]]
            assert e['child'] == i, (i, e)
            N[i], W[i], R[i] = e['N'], e['W'], e['R']
        children = np.where(rec['child'][:count] == 0xFFFF, -1, rec['child'][:count].astype(np.int32))
        mm = self.view('MINMAX').view(self.B, 2)[t].cpu().numpy()
        value = self.view('NODE_VALUE').view(self.B, n)[t].cpu().numpy()[:count].copy()
        return dict(num_nodes=count, N=N, W=W, R=R, parent=parent, move=move, children=children, value=value,
                    prior=self.view('PRIOR').view(self.B, A)[t].cpu().numpy().copy(), minmax=(mm[0], mm[1]))


# ---------------------------------------------------------------------------
# argument checks shared by both entry points (same messages as the reference)
# ---------------------------------------------------------------------------
def _check_temperature(temperature) -> None:
    # generate_play_policy, mcts.py:268-269
    if not isinstance(temperature, float) or not 0.0 <= temperature <= 1.0:
        raise ValueError(f'Expect `temperature` to be float type in the range [0.0, 1.0], got {temperature}')


def _noise_enabled(config, deterministic: bool) -> bool:
    use = (not deterministic) and config.root_dirichlet_alpha > 0.0 and config.root_exploration_eps > 0.0  # mcts.py:361
    if use:
        eps, alpha = config.root_exploration_eps, config.root_dirichlet_alpha
        if not isinstance(eps, float) or not 0.0 <= eps <= 1.0:           # mcts.py:239-240
            raise ValueError(f'Expect `eps` to be a float in the range [0.0, 1.0], got {eps}')
        if not isinstance(alpha, float) or not 0.0 <= alpha <= 1.0:       # mcts.py:241-242
            raise ValueError(f'Expect `alpha` to be a float in the range [0.0, 1.0], got {alpha}')
    return use


_POOLS = {}
# MZ_NO_FUSED_ROOT=1: initial inference, Dirichlet draw and root reset as three separate launches (the round-1 chain;
# kept for the test that pins the fused epilogue to it bit for bit)
_FUSED_ROOT = os.environ.get('MZ_NO_FUSED_ROOT', '0') != '1'


def _pool_for(B, A, config, hidden_bytes, device) -> SearchPool:
    kb = config.known_bounds
    key = (B, A, config.num_simulations, hidden_bytes, str(device), bool(config.is_board_game),
           None if kb is None else (float(kb.min), float(kb.max)), float(config.discount),
           float(config.pb_c_base), float(config.pb_c_init))
    if key not in _POOLS:
        if len(_POOLS) >= 4:
            _POOLS.pop(next(iter(_POOLS)))
        _POOLS[key] = SearchPool(B, A, config, hidden_bytes, device)
    return _POOLS[key]


def clear_pools() -> None:
    _POOLS.clear()


# ---------------------------------------------------------------------------
# batched entry point (additive API)
# ---------------------------------------------------------------------------
class SearchPlan:
    """One batched search = ONE CUDA-graph replay.

    Holds the node pool, static input/output buffers and, per variant
    (noise source, mask present, deterministic), a captured graph of
        initial_inference -> [device Dirichlet] -> reset -> S x (select, recurrent_inference,
        expand+backup) -> root policy
    so a search costs one graph launch instead of 3*S+3 kernel launches from Python.
    """

    def __init__(self, network: MuZeroNet, config, num_trees: int, pool: Optional[SearchPool] = None,
                 instance: int = 0, buffers: Optional[dict] = None) -> None:
        self.network, self.config = network, config
        self.instance = int(instance)            # which engine instance of the network this plan drives
        self.cta_limit = 0                       # SMs the tower kernels of this plan may use (0: all)
        self.dev = next(network.parameters()).device
        self.B, self.A, self.S = int(num_trees), network.num_actions, int(config.num_simulations)
        self.pool = pool if pool is not None else SearchPool(self.B, self.A, config, network.hidden_bytes, self.dev)
        assert self.pool.B == self.B and self.pool.A == self.A and self.pool.S == self.S
        B, A, dev = self.B, self.A, self.dev
        obs_elems = int(np.prod(network.input_shape))
        spec = dict(obs=((B, obs_elems), torch.float32, 0), mask=((B, A), torch.uint8, 1),
                    players=((B, 2), torch.int32, 1), temps=((B,), torch.float64, 1), noise=((B, A), torch.float64, 0),
                    pi0=((B, A), torch.float32, None), v0=((B,), torch.float32, None),
                    action=((B,), torch.int32, None), pi=((B, A), torch.float64, None),
                    root_value=((B,), torch.float64, None), visits=((B, A), torch.int32, None))
        for name, (shape, dt, fill) in spec.items():
            if buffers is not None:              # views into a larger plan's static buffers (PipelinedSearchPlan)
                t = buffers[name]
                assert tuple(t.shape) == shape and t.dtype == dt and t.is_contiguous()
            elif fill is None:
                t = torch.empty(shape, dtype=dt, device=dev)
            else:
                t = torch.full(shape, fill, dtype=dt, device=dev)
            setattr(self, name, t)
        self.root_slots = (torch.arange(B, dtype=torch.int32, device=dev) * (self.S + 1)).contiguous()
        # compact Atari observations (StackedFrames): uint8 frames + plane values, allocated on first use
        self.frames = None if buffers is None else buffers.get('frames')
        self.planes = None if buffers is None else buffers.get('planes')
        self.obs_mode = 'f32'                    # which observation buffers the next run() reads
        self._graphs = {}
        self._eng = None
        self.launches_per_search = 0
        self.use_graph = True

    def use_frames(self) -> None:
        """Switch this plan to compact observations (network.StackedFrames): allocates the static frame buffers."""
        if self.frames is None:
            c, h, w = self.network.input_shape
            self.frames = torch.zeros((self.B, c // 2, h, w), dtype=torch.uint8, device=self.dev)
            self.planes = torch.zeros((self.B, c - c // 2), dtype=torch.float32, device=self.dev)
        self.obs_mode = 'u8'

    def _enqueue(self, noise_mode: str, has_mask: bool, deterministic: bool) -> None:
        """Enqueue one whole search on the current stream (pure C-ABI calls, static pointers)."""
        lib, pool, cfg = _lib.lib(), self.pool, self.config
        eng = self.network.engine(self.B, self.instance)
        _lib.check(lib.mz_net_set_cta_limit(eng['handle'], self.cta_limit))     # engines are shared between plans
        stream = _lib.current_stream()
        hidden = pool.hidden.data_ptr() if pool.hidden_bytes else None
        mask_p = self.mask.data_ptr() if has_mask else None
        frames_p = self.frames.data_ptr() if self.obs_mode == 'u8' else None
        planes_p = self.planes.data_ptr() if self.obs_mode == 'u8' else None
        obs_p = None if self.obs_mode == 'u8' else self.obs.data_ptr()
        eps = cfg.root_exploration_eps if noise_mode != 'none' else 0.0
        # alphas are float32 in the reference (np.ones_like(prob) * alpha)
        alpha = float(np.float32(cfg.root_dirichlet_alpha)) if noise_mode == 'device' else 0.0
        noise_p = self.noise.data_ptr() if noise_mode != 'none' else None
        if _FUSED_ROOT:
            # initial inference whose policy epilogue draws the noise and prepares the roots (one launch chain, no
            # separate dirichlet / reset kernels)
            _lib.check(lib.mz_net_initial_search(eng['handle'], pool.handle, self.B, obs_p, frames_p, planes_p, hidden,
                                                 self.root_slots.data_ptr(), self.pi0.data_ptr(), self.v0.data_ptr(),
                                                 {'none': 0, 'given': 1, 'device': 2}[noise_mode], noise_p, alpha,
                                                 float(eps), mask_p, self.players.data_ptr(), stream))
        else:
            if self.obs_mode == 'u8':
                _lib.check(lib.mz_net_initial_frames(eng['handle'], self.B, frames_p, planes_p, hidden,
                                                     self.root_slots.data_ptr(), self.pi0.data_ptr(),
                                                     self.v0.data_ptr(), stream))
            else:
                _lib.check(lib.mz_net_initial(eng['handle'], self.B, obs_p, hidden, self.root_slots.data_ptr(),
                                              self.pi0.data_ptr(), self.v0.data_ptr(), stream))
            if noise_mode == 'device':
                _lib.check(lib.mz_dirichlet(pool.handle, alpha, noise_p, stream))
            _lib.check(lib.mz_search_reset(pool.handle, self.pi0.data_ptr(), noise_p, float(eps), mask_p,
                                           self.players.data_ptr(), None, stream))
        # the simulation loop (mcts.py:372-390): one persistent launch for the MLP nets, the per-simulation launch
        # chain otherwise -- the library decides (mz_search_run)
        _lib.check(lib.mz_search_run(eng['handle'], pool.handle, stream))
        _lib.check(lib.mz_root_policy(pool.handle, mask_p, self.temps.data_ptr(), int(deterministic),
                                      self.action.data_ptr(), self.pi.data_ptr(), self.root_value.data_ptr(),
                                      self.visits.data_ptr(), stream))

    def run(self, noise_mode: str = 'device', has_mask: bool = True, deterministic: bool = False) -> None:
        """Execute one search over the current contents of the static input buffers."""
        eng = self.network.engine(self.B, self.instance)
        if eng is not self._eng:                 # weights changed -> engine rebuilt -> old graphs are stale
            self._graphs.clear()
            self._eng = eng
        with torch.cuda.device(self.dev):
            if not self.use_graph:
                self._enqueue(noise_mode, has_mask, deterministic)
                return
            key = (noise_mode, has_mask, deterministic, self.obs_mode)
            g = self._graphs.get(key)
            if g is None:
                lib = _lib.lib()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):     # eager warm-up: lazy module/attribute setup must not be captured
                    n0 = lib.mz_launch_count()
                    self._enqueue(noise_mode, has_mask, deterministic)
                    self.launches_per_search = int(lib.mz_launch_count() - n0)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                # that eager pass WAS this call's search (capture below records, it does not execute)
                self._graphs[key] = _capture(lambda: self._enqueue(noise_mode, has_mask, deterministic))
                return
            g.replay()


class _PoolGroup:
    """The pools of a PipelinedSearchPlan seen as one pool of B trees (tree t lives in part t // (B / parts))."""

    def __init__(self, pools) -> None:
        self.pools = list(pools)
        self.B = sum(p.B for p in self.pools)
        self.A, self.S, self.hidden_bytes = self.pools[0].A, self.pools[0].S, self.pools[0].hidden_bytes

    def _split(self, seq):
        out, o = [], 0
        for p in self.pools:
            out.append(seq[o:o + p.B])
            o += p.B
        return out

    def seed(self, seeds) -> None:
        for p, s in zip(self.pools, self._split(np.asarray(seeds))):
            p.seed(s)

    def set_rng_states(self, states) -> None:
        for p, s in zip(self.pools, self._split(list(states))):
            p.set_rng_states(s)

    def get_rng_states(self):
        return [st for p in self.pools for st in p.get_rng_states()]

    def check_errors(self) -> None:
        for p in self.pools:
            p.check_errors()

    def stats(self) -> np.ndarray:
        return sum(p.view('STATS').cpu().numpy().astype(np.int64) for p in self.pools)

    def dump_tree(self, t: int) -> dict:
        per = self.pools[0].B
        return self.pools[t // per].dump_tree(t % per)


class PipelinedSearchPlan:
    """B trees searched as ``parts`` independent sub-batches whose launch chains are interleaved on separate
    streams inside ONE CUDA graph.

    Trees never interact, so the result is bit-identical to one SearchPlan over all B trees.  What changes is
    the schedule: a simulation is select -> recurrent inference (a persistent kernel that fills every SM) ->
    heads -> expand+backup, and the tree kernels are latency-bound on the deepest tree (a warp per tree, ~2000
    cycles per level) while all other SMs idle.  With two sub-batches in flight the tree kernels of one overlap
    the tensor-core tower of the other (the conv kernel leaves room for one small CTA per SM).  Each part has
    its own node pool and its own engine instance (activation buffers); weights are shared read-only.
    """

    def __init__(self, network: MuZeroNet, config, num_trees: int, parts: int = 2, cta_limit: int = 0,
                 tree_ctas: Optional[int] = None) -> None:
        assert parts >= 1 and num_trees % parts == 0, 'num_trees must be a multiple of parts'
        self.network, self.config = network, config
        # cta_limit > 0: every part's persistent tower kernel uses at most that many SMs, so the towers of the
        # parts run SIDE BY SIDE (small batches: a tower is bound by tile dependencies between layers, not by SMs)
        self.cta_limit = int(cta_limit)
        self.dev = next(network.parameters()).device
        self.B, self.A, self.S = int(num_trees), network.num_actions, int(config.num_simulations)
        B, A, dev, per = self.B, self.A, self.dev, int(num_trees) // parts
        obs_elems = int(np.prod(network.input_shape))
        self.obs = torch.zeros((B, obs_elems), dtype=torch.float32, device=dev)
        self.mask = torch.ones((B, A), dtype=torch.uint8, device=dev)
        self.players = torch.ones((B, 2), dtype=torch.int32, device=dev)
        self.temps = torch.ones(B, dtype=torch.float64, device=dev)
        self.noise = torch.zeros((B, A), dtype=torch.float64, device=dev)
        self.pi0 = torch.empty((B, A), dtype=torch.float32, device=dev)
        self.v0 = torch.empty(B, dtype=torch.float32, device=dev)
        self.action = torch.empty(B, dtype=torch.int32, device=dev)
        self.pi = torch.empty((B, A), dtype=torch.float64, device=dev)
        self.root_value = torch.empty(B, dtype=torch.float64, device=dev)
        self.visits = torch.empty((B, A), dtype=torch.int32, device=dev)
        names = ('obs', 'mask', 'players', 'temps', 'noise', 'pi0', 'v0', 'action', 'pi', 'root_value', 'visits')
        self.parts = [SearchPlan(network, config, per, instance=i,
                                 buffers={n: getattr(self, n)[i * per:(i + 1) * per] for n in names})
                      for i in range(parts)]
        # Large conv-net sub-batches that each fill the GPU (cta_limit == 0): the fused tree kernel of a part runs as
        # `tree_ctas` persistent CTAs on SMs of its own and the towers get the rest (see mz_pool_set_tree_ctas) --
        # a tree warp beside the tower's warps is several times slower AND slows the tower.
        env = os.environ.get('MZ_TREE_CTAS')
        self.tree_ctas = int(env) if env is not None else (4 if tree_ctas is None else int(tree_ctas))
        if parts < 2 or self.cta_limit or network.kind == _lib.MZ_NET_MLP or A > 128:
            self.tree_ctas = 0
        if self.tree_ctas:
            sms = torch.cuda.get_device_properties(dev).multi_processor_count
            self.cta_limit = sms - self.tree_ctas
            for part in self.parts:
                _lib.check(_lib.lib().mz_pool_set_tree_ctas(part.pool.handle, self.tree_ctas))
        for part in self.parts:
            part.cta_limit = self.cta_limit
        self.pool = _PoolGroup([p.pool for p in self.parts])
        self.frames = self.planes = None
        self.obs_mode = 'f32'
        self._streams = [torch.cuda.Stream(device=dev) for _ in range(parts - 1)]
        self._graphs = {}
        self._engs = None
        self.use_graph = True

    @property
    def launches_per_search(self) -> int:
        return sum(p.launches_per_search for p in self.parts)

    def use_frames(self) -> None:
        if self.frames is None:
            c, h, w = self.network.input_shape
            self.frames = torch.zeros((self.B, c // 2, h, w), dtype=torch.uint8, device=self.dev)
            self.planes = torch.zeros((self.B, c - c // 2), dtype=torch.float32, device=self.dev)
            per = self.B // len(self.parts)
            for i, part in enumerate(self.parts):
                part.frames, part.planes = self.frames[i * per:(i + 1) * per], self.planes[i * per:(i + 1) * per]
        self.obs_mode = 'u8'
        for part in self.parts:
            part.obs_mode = 'u8'

    def _enqueue_all(self, noise_mode, has_mask, deterministic) -> None:
        """Fork one stream per extra part off the current stream, enqueue every part, join."""
        main = torch.cuda.current_stream()
        for s in self._streams:
            s.wait_stream(main)
        self.parts[0]._enqueue(noise_mode, has_mask, deterministic)
        for part, s in zip(self.parts[1:], self._streams):
            with torch.cuda.stream(s):
                part._enqueue(noise_mode, has_mask, deterministic)
        for s in self._streams:
            main.wait_stream(s)

    def run(self, noise_mode: str = 'device', has_mask: bool = True, deterministic: bool = False) -> None:
        engs = [p.network.engine(p.B, p.instance) for p in self.parts]
        if self._engs is None or any(a is not b for a, b in zip(engs, self._engs)):
            self._graphs.clear()                 # weights changed -> engines rebuilt -> old graphs are stale
            self._engs = engs
        with torch.cuda.device(self.dev):
            if not self.use_graph:
                self._enqueue_all(noise_mode, has_mask, deterministic)
                return
            key = (noise_mode, has_mask, deterministic, self.obs_mode)
            g = self._graphs.get(key)
            if g is None:
                lib = _lib.lib()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):     # eager warm-up (this call's search), one part after the other
                    for part in self.parts:
                        n0 = lib.mz_launch_count()
                        part._enqueue(noise_mode, has_mask, deterministic)
                        part.launches_per_search = int(lib.mz_launch_count() - n0)
                torch.cuda.current_stream().wait_stream(side)
                torch.cuda.synchronize()
                self._graphs[key] = _capture(lambda: self._enqueue_all(noise_mode, has_mask, deterministic))
                return
            g.replay()


_PLANS = {}


def pipeline_shape(network, B: int):
    """(parts, cta_limit) of the plan uct_search_batch builds for B trees of this network.

    Conv nets with large batches (>= two 256-row tiles per SM and part): two sub-batches that each use the whole GPU,
    so the tree kernels of one overlap the tower of the other.  Smaller batches run as one plan: giving two
    sub-batches half of the SMs each (cta_limit = 74, towers side by side) was measured on the Atari-shaped config
    (1024 trees, 196 tiles per layer) and changes nothing -- a tower launch there is bound by the tile dependencies
    between layers (~1.3 tiles per CTA and layer), whatever the number of SMs."""
    if network.kind == _lib.MZ_NET_MLP or B % 2:
        return 1, 0
    h, w = network.latent_hw
    if (B // 2) * h * w >= 2 * 148 * 256:
        return 2, 0
    return 1, 0


def _plan_for(network, config, B) -> SearchPlan:
    kb = config.known_bounds
    key = (id(network), B, config.num_simulations, bool(config.is_board_game),
           None if kb is None else (float(kb.min), float(kb.max)), float(config.discount),
           float(config.pb_c_base), float(config.pb_c_init), float(config.root_dirichlet_alpha),
           float(config.root_exploration_eps))
    if key in _PLANS and _PLANS[key].network is not network:      # id() reused after garbage collection
        del _PLANS[key]
    if key not in _PLANS:
        if len(_PLANS) >= 4:
            _PLANS.pop(next(iter(_PLANS)))
        # large conv-net batches: two sub-batches in flight (each still fills the GPU's tile grid)
        parts, limit = pipeline_shape(network, B)
        _PLANS[key] = PipelinedSearchPlan(network, config, B, parts, limit) if parts > 1 else \
            SearchPlan(network, config, B)
    plan = _PLANS[key]
    plan.config = config
    return plan


@torch.no_grad()
def uct_search_batch(states, network: MuZeroNet, config, temperature, actions_mask, current_player, opponent_player,
                     deterministic: bool = False, rng=None, noise=None, plan: Optional[SearchPlan] = None):
    """``uct_search`` for B independent trees at once, everything on the GPU.

    states          [B, *obs] array/tensor (host or device), or network.StackedFrames (uint8 frames + action-plane
                    values: the compact form of a MuZeroAtariNet observation, a quarter of the upload)
    temperature     float or float64[B]
    actions_mask    bool[B, A] or None
    current_player / opponent_player   int or int[B]
    rng             None: each tree continues its device-resident MT19937 stream
                    (seed it with ``plan.pool.seed``) and, when noise is on, the
                    Dirichlet sample is drawn on the device from that stream;
                    list of B ``np.random.RandomState``: numpy-exact mode — the
                    Dirichlet sample is drawn by numpy from each stream, the
                    stream is continued on the device for tie-breaks and the final
                    draw, and written back, i.e. tree t consumes its stream exactly
                    as the reference ``uct_search`` would.
    noise           optional float64[B, A] pre-drawn Dirichlet samples (overrides both).

    Returns (actions int32[B], pi float64[B, A], root_values float64[B]) as CUDA tensors.
    """
    compact = isinstance(states, StackedFrames)
    if not compact:
        states = torch.as_tensor(states) if not torch.is_tensor(states) else states
    B = (states.frames if compact else states).shape[0]
    if config.is_board_game:
        assert config.discount == 1.0                                     # mcts.py:349-350
    if np.isscalar(temperature):
        _check_temperature(temperature)
        temps = np.full(B, temperature, dtype=np.float64)
    else:
        temps = np.asarray(temperature, dtype=np.float64)
        if temps.shape != (B,) or not ((temps >= 0.0) & (temps <= 1.0)).all():
            raise ValueError(f'Expect `temperature` to be float type in the range [0.0, 1.0], got {temperature}')
    use_noise = _noise_enabled(config, deterministic)
    if plan is None:
        plan = _plan_for(network, config, B)
    A, dev, pool = plan.A, plan.dev, plan.pool

    if compact:
        plan.use_frames()
        plan.frames.copy_(torch.as_tensor(states.frames), non_blocking=True)
        plan.planes.copy_(torch.as_tensor(states.planes), non_blocking=True)
    else:
        if plan.obs_mode != 'f32':
            plan.obs_mode = 'f32'
            for part in getattr(plan, 'parts', []):
                part.obs_mode = 'f32'
        plan.obs.copy_(states.reshape(B, -1), non_blocking=True)
    has_mask = actions_mask is not None
    if has_mask:
        m = actions_mask if torch.is_tensor(actions_mask) else torch.from_numpy(np.asarray(actions_mask, dtype=np.bool_))
        assert tuple(m.shape) == (B, A)                                   # mcts.py:293
        plan.mask.copy_(m, non_blocking=True)
    cur = np.broadcast_to(np.asarray(current_player, dtype=np.int32), (B,))
    opp = np.broadcast_to(np.asarray(opponent_player, dtype=np.int32), (B,))
    # players and temperatures rarely change between calls: upload them only when they do (each of these pageable
    # copies costs a synchronising ~30 us, a tenth of a whole Tic-Tac-Toe search)
    players = np.stack([cur, opp], axis=1)
    cache = plan.__dict__.setdefault('_host_inputs', {})
    if cache.get('players') is None or not np.array_equal(cache['players'], players):
        plan.players.copy_(torch.from_numpy(players))
        cache['players'] = players.copy()
    if cache.get('temps') is None or not np.array_equal(cache['temps'], temps):
        plan.temps.copy_(torch.from_numpy(temps))
        cache['temps'] = temps.copy()

    noise_mode = 'none'
    if use_noise:
        noise_mode = 'device'
        if noise is not None:
            plan.noise.copy_(torch.as_tensor(np.asarray(noise, dtype=np.float64)))
            noise_mode = 'given'
        elif rng is not None:
            alphas = np.ones(A, dtype=np.float32) * config.root_dirichlet_alpha   # np.ones_like(prob) * alpha
            plan.noise.copy_(torch.from_numpy(np.stack([r.dirichlet(alphas) for r in rng])))
            noise_mode = 'given'
    states_in = [r.get_state() for r in rng] if rng is not None else None
    if states_in is not None:
        pool.set_rng_states(states_in)
    plan.run(noise_mode, has_mask, deterministic)
    if rng is not None:
        for r, st in zip(rng, pool.get_rng_states()):
            old = r.get_state()
            r.set_state(('MT19937', st[1], st[2], old[3], old[4]))
    return plan.action.clone(), plan.pi.clone(), plan.root_value.clone()


# ---------------------------------------------------------------------------
# the reference's entry point
# ---------------------------------------------------------------------------
class _GlobalNumpyStream:
    """Adapter giving ``np.random``'s global stream the RandomState methods used above."""
    dirichlet = staticmethod(lambda a: np.random.dirichlet(a))
    get_state = staticmethod(lambda: np.random.get_state())
    set_state = staticmethod(lambda s: np.random.set_state(s))


@torch.no_grad()
def uct_search(state: np.ndarray, network, device, config, temperature: float, actions_mask: np.ndarray,
               current_player: int, opponent_player: int, deterministic: bool = False) -> Tuple[int, np.ndarray, float]:
    """Drop-in for ``muzero.mcts.uct_search`` (mcts.py:302-407), one tree on the GPU.

    Consumes ``np.random``'s global MT19937 stream exactly like the reference
    (Dirichlet sample, tie-breaks, final action draw) and leaves it where the
    reference would.  ``network`` is either a ``muzero_b200`` network (inference in
    the CUDA engine) or any object with the reference's ``initial_inference`` /
    ``recurrent_inference`` methods (then only the tree runs on the GPU and the
    network is called once per simulation, like the reference does).
    """
    _check_temperature(temperature)
    dev = torch.device(device)
    mask = None if actions_mask is None else np.asarray(actions_mask)[None, :]
    if isinstance(network, MuZeroNet):
        a, pi, q = uct_search_batch(np.asarray(state)[None, ...], network, config, temperature, mask,
                                    current_player, opponent_player, deterministic, rng=[_GlobalNumpyStream])
        _plan_for(network, config, 1).pool.check_errors()
        return int(a[0].cpu()), pi[0].cpu().numpy(), float(q[0].cpu())
    return _uct_search_external(state, network, dev, config, temperature, actions_mask, current_player,
                                opponent_player, deterministic)


def _uct_search_external(state, network, dev, config, temperature, actions_mask, current_player, opponent_player,
                         deterministic):
    """Tree on the GPU, network = caller's object (batch-1 calls on ``dev``'s side)."""
    if config.is_board_game:
        assert config.discount == 1.0
    gpu = dev if dev.type == 'cuda' else torch.device('cuda', torch.cuda.current_device())
    st = torch.from_numpy(np.asarray(state)).to(device=dev, dtype=torch.float32)
    out0 = network.initial_inference(st[None, ...])
    prior = np.asarray(out0.pi_probs)
    if not isinstance(prior, np.ndarray) or prior.ndim != 1 or prior.dtype not in (np.float32, np.float64):
        raise ValueError(f'Expect `prior` to be a 1D float numpy.array, got {prior}')      # mcts.py:92-93
    A = prior.shape[0]
    use_noise = _noise_enabled(config, deterministic)
    noise_d = None
    if use_noise:
        noise_d = torch.from_numpy(np.random.dirichlet(np.ones_like(prior) * config.root_dirichlet_alpha)[None]).to(gpu)
    mask_d = None
    if actions_mask is not None:
        assert np.asarray(actions_mask).shape == prior.shape                            # mcts.py:293
        mask_d = torch.from_numpy(np.asarray(actions_mask, dtype=np.uint8)[None].copy()).to(gpu)
    pool = _pool_for(1, A, config, 0, gpu)
    pool.set_rng_states([np.random.get_state()])
    players = torch.tensor([[current_player, opponent_player]], dtype=torch.int32, device=gpu)
    rr = torch.tensor([float(out0.reward)], dtype=torch.float32, device=gpu)
    pool.reset(torch.from_numpy(prior.astype(np.float32))[None].to(gpu).contiguous(), noise_d,
               config.root_exploration_eps if use_noise else 0.0, mask_d, players, rr)
    hidden = {0: out0.hidden_state}
    rv = torch.empty(2, dtype=torch.float32, device=gpu)
    for i in range(config.num_simulations):
        pool.select()
        par = int(pool.view('LEAF_PARENT')[0].cpu())
        a = int(pool.view('LEAF_ACTION')[0].cpu())
        h = torch.from_numpy(np.asarray(hidden[par])).to(device=dev, dtype=torch.float32)
        o = network.recurrent_inference(h[None, ...], torch.tensor([[a]], dtype=torch.long, device=dev))
        hidden[i + 1] = o.hidden_state
        rv.copy_(torch.tensor([float(o.reward), float(o.value)], dtype=torch.float32))
        pool.expand_backup(rv[0:1], rv[1:2])
    temps = torch.tensor([temperature], dtype=torch.float64, device=gpu)
    action, pi, rootv, _ = pool.root_policy(mask_d, temps, deterministic)
    pool.check_errors()
    stt = pool.get_rng_states()[0]
    old = np.random.get_state()
    np.random.set_state(('MT19937', stt[1], stt[2], old[3], old[4]))
    return int(action[0].cpu()), pi[0].cpu().numpy(), float(rootv[0].cpu())
