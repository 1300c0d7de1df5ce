"""Shapes and runs shared by tests/test_conv_pair_gpu.py and tests/golden/make_golden_pair.py.

Gomoku net (9x9 board, 128 planes, 8 residual blocks: the recurrent inference is one 33-conv dataflow launch).  A
256-row tile holds 256 / 81 = 3.2 boards, so B boards make ceil(81 B / 256) tiles and ceil(tiles / 2) pair items.
"""
from __future__ import annotations

import hashlib
import os

import numpy as np
import torch

# (name, boards, cta_limit (0: every SM), MZ_CONV_TILE_ROWS (None: the launch's own choice))
CASES = [
    ('bench_1024', 1024, 144, None),   # the bench's sub-batch: 324 tiles, 162 pair items on 72 pairs
    ('odd_tiles', 1000, 0, None),      # 317 tiles: the last pair item's odd tile is a null tile
    ('odd_limit', 100, 7, '256'),      # 32 tiles on 3 pairs of a 7-CTA limit, 16 items rotating by 1 per layer
    ('few_items', 315, 103, '256'),    # 100 tiles = 50 items, fewer than the 51 pairs the limit leaves room for
    ('one_each', 40, 12, '256'),       # 13 tiles (odd) = 7 items on 6 pairs: one pair takes two items per layer
]


def digest(t: torch.Tensor) -> np.ndarray:
    b = t.detach().contiguous().cpu().view(torch.uint8).numpy().tobytes()
    return np.frombuffer(hashlib.sha256(b).digest(), dtype=np.uint8).copy()


def build_net():
    import muzero_b200 as mz
    from oracle.network_oracle import randomize_batchnorm
    torch.manual_seed(0)
    net = mz.MuZeroBoardGameNet((9, 9, 9), 82, 8, 128).eval()
    randomize_batchnorm(net, 1000)
    return net.cuda()


def run_case(net, batch: int, cta_limit: int, rows) -> dict:
    from muzero_b200 import _lib
    old = os.environ.pop('MZ_CONV_TILE_ROWS', None)
    if rows is not None:
        os.environ['MZ_CONV_TILE_ROWS'] = rows
    try:
        gen = np.random.RandomState(batch)
        obs = torch.from_numpy(gen.randint(0, 2, size=(batch, 9, 9, 9)).astype(np.float32)).cuda()
        act = torch.from_numpy(gen.randint(0, 82, size=batch)).cuda()
        _lib.check(_lib.lib().mz_net_set_cta_limit(net.engine(batch)['handle'], cta_limit))
        hid, pi0, v0 = net.initial_inference_batch(obs)
        hid1, r, pi1, v1 = net.recurrent_inference_batch(hid, act)
        torch.cuda.synchronize()
    finally:
        _lib.check(_lib.lib().mz_net_set_cta_limit(net.engine(batch)['handle'], 0))
        os.environ.pop('MZ_CONV_TILE_ROWS', None)
        if old is not None:
            os.environ['MZ_CONV_TILE_ROWS'] = old
    return dict(h0=digest(hid), pi0=digest(pi0), v0=digest(v0), h1=digest(hid1), r=digest(r), pi1=digest(pi1),
                v1=digest(v1))


def run_search(net, parts: int, trees: int = 2048, sims: int = 6) -> dict:
    """One Gomoku search of `trees` trees: parts = 2 is the bench's two-stream PipelinedSearchPlan (the tree kernel
    of one sub-batch beside the tower of the other), parts = 1 one SearchPlan over the whole batch."""
    import muzero_b200 as mz
    cfg = mz.make_gomoku_config(use_tensorboard=False)
    cfg.num_simulations = sims
    gen = np.random.RandomState(23)
    obs = gen.randint(0, 2, size=(trees, 9, 9, 9)).astype(np.int8)
    # every action legal: with illegal ones a random-init net can put every visit of a tree below an illegal first
    # pick, and the visit policy is then 0 / 0 (the reference's own pathology, see test_conv_gpu.py)
    mask = np.ones((trees, 82), dtype=bool)
    plan = mz.mcts.PipelinedSearchPlan(net, cfg, trees, parts=2) if parts == 2 else mz.mcts.SearchPlan(net, cfg, trees)
    for _ in range(2):                         # eager pass, then the captured graph
        streams = [np.random.RandomState(700 + t) for t in range(trees)]
        a, pi, q = mz.uct_search_batch(obs, net, cfg, 1.0, mask, 1, 2, rng=streams, plan=plan)
        plan.pool.check_errors()
    torch.cuda.synchronize()
    return dict(action=digest(a), pi=digest(pi), root_value=digest(q))
