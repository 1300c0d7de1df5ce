"""GPU tests of the tcgen05 ResNet towers (bf16 x bf16 -> fp32) against the fp32 torch
restatement of the reference and the reference's own recorded outputs.

Stated tolerance (fp16 activations and weights, fp32 accumulation in TMEM, fp32 heads):
  hidden state (min-max normalised to [0,1]):  |err| <= 0.005   (measured <= 0.002)
  policy probabilities:                        |err| <= 0.02    (measured <= 0.0096 on random-init nets with |logit| ~ 40)
  value / reward:                              |err| <= 0.02 * max(1, |ref|_max)   (measured <= 0.014)
"""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, bits
from oracle import mcts_oracle as orc
from oracle.network_oracle import OracleNet, randomize_batchnorm
from oracle.stubnet import ReplayStub

pytestmark = pytest.mark.gpu
TOL_H = 0.005      # hidden state, normalised to [0, 1]
TOL_PV = 0.02      # policy probabilities (absolute); value / reward (relative to max(1, |ref|max))


def build_board(input_shape, num_actions, blocks, planes, seed):
    import muzero_b200 as mz
    torch.manual_seed(seed)
    net = mz.MuZeroBoardGameNet(input_shape, num_actions, blocks, planes).eval()
    randomize_batchnorm(net, 1000 + seed)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    onet = OracleNet('board', sd, num_actions, 1, 1, blocks)
    return net.cuda(), onet


def report(name, got, ref, tol, scale=None):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    err = np.abs(got - ref)
    scale = max(1.0, float(np.abs(ref).max())) if scale is None else scale
    print(f'{name}: max|err|={err.max():.4g} mean|err|={err.mean():.4g} ref|max|={np.abs(ref).max():.4g} '
          f'(tol {tol * scale:.4g})')
    assert np.isfinite(got).all(), f'{name}: non-finite output'
    assert err.max() <= tol * scale, f'{name}: max err {err.max():.4g} > {tol * scale:.4g} at {np.unravel_index(err.argmax(), err.shape)}'


@pytest.mark.parametrize('shape,A,planes', [((3, 3, 3), 10, 32), ((9, 5, 5), 26, 64), ((9, 9, 9), 82, 128),
                                            ((17, 15, 15), 226, 128)])
@pytest.mark.parametrize('batch', [1, 7, 300])
def test_single_conv_layers_blocks0(shape, A, planes, batch):
    """num_res_blocks = 0 isolates ONE tensor-core conv per function: the representation
    conv (few input planes), the dynamics conv (C planes + per-action bias table, QUIRK C)
    and the 1x1-conv heads."""
    net, onet = build_board(shape, A, 0, planes, seed=batch)
    gen = np.random.RandomState(batch)
    obs = gen.randint(0, 2, size=(batch,) + shape).astype(np.float32)
    hid, pi, v = net.initial_inference_batch(torch.from_numpy(obs).cuda())
    h_ref, pi_ref, v_ref = onet.initial_batch(obs)
    report('rep hidden', net.hidden_to_reference(hid).cpu().numpy(), h_ref.numpy(), TOL_H)
    report('pi0', pi.cpu().numpy(), pi_ref.numpy(), TOL_PV)
    report('v0', v.cpu().numpy(), v_ref.numpy(), TOL_PV)
    act = gen.randint(0, A, size=batch)
    src = torch.arange(batch - 1, -1, -1, dtype=torch.int32).cuda()
    dst = (torch.arange(batch, dtype=torch.int32) * 2 + 1).cuda()
    out = net.new_hidden(2 * batch + 1)
    slots_in = net.hidden_from_reference(h_ref.cuda())
    _, r, pi2, v2 = net.recurrent_inference_batch(slots_in, torch.from_numpy(act).cuda(), src_index=src, hidden_out=out,
                                                  dst_index=dst)
    h2_ref, r_ref, pi2_ref, v2_ref = onet.recurrent_batch(h_ref.flip(0), act)
    report('dyn hidden', net.hidden_to_reference(out)[1::2].cpu().numpy(), h2_ref.numpy(), TOL_H)
    report('reward', r.cpu().numpy(), r_ref.numpy(), TOL_PV)
    report('v1', v2.cpu().numpy(), v2_ref.numpy(), TOL_PV)
    report('pi1', pi2.cpu().numpy(), pi2_ref.numpy(), TOL_PV)
    assert (out.view(torch.float16)[0::2] == 0).all()        # untouched slots stay untouched


@pytest.fixture(params=['auto', '128', '256'])
def tile_rows(request, monkeypatch):
    """The conv kernel has a 256-row-tile (throughput) and a 128-row split-K (latency) variant, chosen from the
    number of tiles per SM; MZ_CONV_TILE_ROWS forces one so that both are exercised at test sizes."""
    if request.param == 'auto':
        monkeypatch.delenv('MZ_CONV_TILE_ROWS', raising=False)
    else:
        monkeypatch.setenv('MZ_CONV_TILE_ROWS', request.param)
    return request.param


@pytest.mark.parametrize('name,kind,kw,seed', [
    ('board_small', 'board', dict(input_shape=(5, 5, 5), num_actions=26, num_res_blocks=2, num_planes=32), 3),
    ('gomoku', 'board', dict(input_shape=(9, 9, 9), num_actions=82, num_res_blocks=8, num_planes=128), 0),
])
def test_towers_vs_reference_recording(name, kind, kw, seed, tile_rows):
    """Single-item reference API against the reference's own recorded outputs
    (tests/golden/net_golden.npz; the recording stores hidden states as float16)."""
    net, onet = build_board(kw['input_shape'], kw['num_actions'], kw['num_res_blocks'], kw['num_planes'], seed)
    z = np.load(os.path.join(GOLDEN, 'net_golden.npz'))
    tol_h = TOL_H
    for j in range(2):
        g = {k: z[f'{name}_{j}_{k}'] for k in ('obs', 'actions', 'h0', 'pi0', 'v0', 'h', 'r', 'v', 'pi')}
        o = net.initial_inference(torch.from_numpy(g['obs'])[None].cuda())
        assert o.hidden_state.shape == g['h0'].shape and o.hidden_state.dtype == np.float32
        assert isinstance(o.value, float) and o.reward == 0.0
        report(f'{name}/{j} h0', o.hidden_state, g['h0'].astype(np.float32), TOL_H)
        report(f'{name}/{j} pi0', o.pi_probs, g['pi0'], TOL_PV)
        report(f'{name}/{j} v0', o.value, g['v0'], TOL_PV)
        h = g['h0'].astype(np.float32)
        for i, a in enumerate(g['actions']):
            o = net.recurrent_inference(torch.from_numpy(h)[None].cuda(), torch.tensor([[int(a)]]).cuda())
            report(f'{name}/{j} h[{i}]', o.hidden_state, g['h'][i].astype(np.float32), TOL_H)
            report(f'{name}/{j} r[{i}]', o.reward, g['r'][i], TOL_PV)
            report(f'{name}/{j} v[{i}]', o.value, g['v'][i], TOL_PV)
            report(f'{name}/{j} pi[{i}]', o.pi_probs, g['pi'][i], TOL_PV)
            h = g['h'][i].astype(np.float32)


@pytest.mark.parametrize('batch', [5, 129, 2048])
def test_gomoku_batched_vs_torch_fp32(batch):
    net, onet = build_board((9, 9, 9), 82, 8, 128, seed=0)
    gen = np.random.RandomState(batch)
    nref = min(batch, 24)                                  # torch-CPU fp32 reference on a subset of rows
    obs = gen.randint(0, 2, size=(batch, 9, 9, 9)).astype(np.float32)
    hid, pi, v = net.initial_inference_batch(torch.from_numpy(obs).cuda())
    rows = np.sort(gen.choice(batch, size=nref, replace=False))
    h_ref, pi_ref, v_ref = onet.initial_batch(obs[rows])
    report('h0', net.hidden_to_reference(hid)[rows].cpu().numpy(), h_ref.numpy(), TOL_H)
    report('pi0', pi[rows].cpu().numpy(), pi_ref.numpy(), TOL_PV)
    report('v0', v[rows].cpu().numpy(), v_ref.numpy(), TOL_PV)
    act = gen.randint(0, 82, size=batch)
    _, r, pi2, v2 = net.recurrent_inference_batch(hid, torch.from_numpy(act).cuda())
    h2_ref, r_ref, pi2_ref, v2_ref = onet.recurrent_batch(h_ref, act[rows])
    report('r', r[rows].cpu().numpy(), r_ref.numpy(), TOL_PV)
    report('v1', v2[rows].cpu().numpy(), v2_ref.numpy(), TOL_PV)
    report('pi1', pi2[rows].cpu().numpy(), pi2_ref.numpy(), TOL_PV)


def test_gomoku_search_replays_bit_exact_in_oracle(tile_rows):
    """Whole batched Gomoku search on the GPU with the tensor-core network; every tree, fed the
    per-node (reward, value) the engine produced, is rebuilt bit-for-bit by the CPU oracle."""
    import muzero_b200 as mz
    net, onet = build_board((9, 9, 9), 82, 2, 32, seed=1)
    cfg = mz.make_gomoku_config(use_tensorboard=False)
    cfg.num_simulations = 60
    B, A, S = 48, 82, 60
    gen = np.random.RandomState(5)
    obs = gen.randint(0, 2, size=(B, 9, 9, 9)).astype(np.int8)
    mask = gen.rand(B, A) < 0.8
    mask[:, -1] = True
    streams = [np.random.RandomState(300 + t) for t in range(B)]
    plan = mz.mcts.SearchPlan(net, cfg, B)
    action, pi, rootv = mz.uct_search_batch(obs, net, cfg, 1.0, mask, 1, 2, rng=streams, plan=plan)
    plan.pool.check_errors()
    pi0 = plan.pi0.cpu().numpy()
    for t in range(0, B, 4):
        d = plan.pool.dump_tree(t)
        rs = np.random.RandomState(300 + t)
        stub = ReplayStub(pi0[t], d['R'][1:].astype(np.float32), d['value'][1:], d['parent'], d['move'])
        a_o, pi_o, q_o, tr = orc.uct_search(obs[t].astype(np.float32), stub, 'cpu', cfg, 1.0, mask[t], 1, 2, False,
                                            rng=rs, return_trace=True)
        assert np.array_equal(tr.N, d['N']) and np.array_equal(bits(tr.W), bits(d['W']))
        assert a_o == int(action[t]) and np.array_equal(bits(pi_o), bits(pi[t].cpu().numpy()))
        assert bits(q_o)[0] == bits(rootv[t].item())[0]
        assert rs.get_state()[2] == streams[t].get_state()[2]
    # second search through the captured CUDA graph gives the same answer as the eager first one
    streams2 = [np.random.RandomState(300 + t) for t in range(B)]
    a2, pi2, q2 = mz.uct_search_batch(obs, net, cfg, 1.0, mask, 1, 2, rng=streams2, plan=plan)
    assert torch.equal(a2, action) and torch.equal(pi2, pi) and torch.equal(q2, rootv)


def test_gomoku_15x15_wide_board_and_226_actions():
    """The reference's class-default Gomoku (15x15, 8 history planes -> 17 observation planes, 226 actions,
    games/gomoku.py:31-36): wider halo / tile geometry in the conv kernel, the A > 128 path of the select kernel,
    a 226-row action table.  Network vs fp32 torch, and a batched search replayed bit-exactly in the oracle."""
    import muzero_b200 as mz
    net, onet = build_board((17, 15, 15), 226, 2, 64, seed=3)
    gen = np.random.RandomState(15)
    B, A = 40, 226
    obs = gen.randint(0, 2, size=(B, 17, 15, 15)).astype(np.float32)
    hid, pi, v = net.initial_inference_batch(torch.from_numpy(obs).cuda())
    h_ref, pi_ref, v_ref = onet.initial_batch(obs)
    report('15x15 h0', net.hidden_to_reference(hid).cpu().numpy(), h_ref.numpy(), TOL_H)
    report('15x15 pi0', pi.cpu().numpy(), pi_ref.numpy(), TOL_PV)
    report('15x15 v0', v.cpu().numpy(), v_ref.numpy(), TOL_PV)
    act = gen.randint(0, A, size=B)
    hid2, r, pi2, v2 = net.recurrent_inference_batch(hid, torch.from_numpy(act).cuda())
    h2_ref, r_ref, pi2_ref, v2_ref = onet.recurrent_batch(h_ref, act)
    report('15x15 h1', net.hidden_to_reference(hid2).cpu().numpy(), h2_ref.numpy(), TOL_H)
    report('15x15 r', r.cpu().numpy(), r_ref.numpy(), TOL_PV)
    report('15x15 v1', v2.cpu().numpy(), v2_ref.numpy(), TOL_PV)
    report('15x15 pi1', pi2.cpu().numpy(), pi2_ref.numpy(), TOL_PV)

    cfg = mz.make_gomoku_config(use_tensorboard=False)
    cfg.num_simulations = 40
    # every action legal: with illegal actions a random-init net at A = 226 reproduces the reference's own
    # pathology (the first simulation ties over ALL actions, mcts.py:104-127 with N_root = 0; a tree whose first
    # pick is illegal can spend every visit below it, and generate_play_policy then divides 0 by 0 ->
    # ValueError('probabilities contain NaN'), covered by test_error_paths_match_reference_exceptions)
    mask = np.ones((B, A), dtype=bool)
    streams = [np.random.RandomState(500 + t) for t in range(B)]
    plan = mz.mcts.SearchPlan(net, cfg, B)
    action, pi, rootv = mz.uct_search_batch(obs, net, cfg, 1.0, mask, 1, 2, rng=streams, plan=plan)
    plan.pool.check_errors()
    pi0 = plan.pi0.cpu().numpy()
    for t in range(0, B, 5):
        d = plan.pool.dump_tree(t)
        rs = np.random.RandomState(500 + t)
        stub = ReplayStub(pi0[t], d['R'][1:].astype(np.float32), d['value'][1:], d['parent'], d['move'])
        a_o, pi_o, q_o, tr = orc.uct_search(obs[t], stub, 'cpu', cfg, 1.0, mask[t], 1, 2, False, rng=rs,
                                            return_trace=True)
        assert np.array_equal(tr.N, d['N']) and np.array_equal(bits(tr.W), bits(d['W']))
        assert a_o == int(action[t]) and np.array_equal(bits(pi_o), bits(pi[t].cpu().numpy()))
        assert bits(q_o)[0] == bits(rootv[t].item())[0] and rs.get_state()[2] == streams[t].get_state()[2]


def test_pipelined_plan_is_bit_identical_to_single_plan():
    """Two half-batches interleaved on two streams in one CUDA graph (PipelinedSearchPlan) give exactly the
    trees, actions, policies, root values and RNG positions of one SearchPlan over the whole batch: trees
    are independent and a network row does not depend on which other rows share its launch."""
    import muzero_b200 as mz
    net, _ = build_board((9, 9, 9), 82, 2, 32, seed=1)
    cfg = mz.make_gomoku_config(use_tensorboard=False)
    cfg.num_simulations = 40
    B, A = 64, 82
    gen = np.random.RandomState(11)
    obs = gen.randint(0, 2, size=(B, 9, 9, 9)).astype(np.int8)
    mask = gen.rand(B, A) < 0.8
    mask[:, -1] = True
    out = []
    for plan in (mz.mcts.SearchPlan(net, cfg, B), mz.mcts.PipelinedSearchPlan(net, cfg, B, parts=2)):
        res = []
        for rep in range(3):                       # eager warm-up pass, graph capture, graph replay
            streams = [np.random.RandomState(900 + t) for t in range(B)]
            a, pi, q = mz.uct_search_batch(obs, net, cfg, 1.0, mask, 1, 2, rng=streams, plan=plan)
            plan.pool.check_errors()
            res.append((a.cpu().numpy(), pi.cpu().numpy(), q.cpu().numpy(), [s.get_state()[2] for s in streams],
                        [plan.pool.dump_tree(t) for t in (0, 31, 32, 63)]))
        for r in res[1:]:
            assert np.array_equal(r[0], res[0][0]) and np.array_equal(bits(r[1]), bits(res[0][1]))
        out.append(res[-1])
    single, piped = out
    assert np.array_equal(single[0], piped[0])
    assert np.array_equal(bits(single[1]), bits(piped[1])) and np.array_equal(bits(single[2]), bits(piped[2]))
    assert single[3] == piped[3]
    for d0, d1 in zip(single[4], piped[4]):
        assert np.array_equal(d0['N'], d1['N']) and np.array_equal(bits(d0['W']), bits(d1['W']))
        assert np.array_equal(d0['parent'], d1['parent']) and np.array_equal(d0['move'], d1['move'])
        assert np.array_equal(d0['value'][1:], d1['value'][1:])          # slot 0 (the root) is never written


def build_atari(kw, seed):
    import muzero_b200 as mz
    torch.manual_seed(seed)
    net = mz.MuZeroAtariNet(**kw).eval()
    randomize_batchnorm(net, 1000 + seed)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    onet = OracleNet('atari', sd, kw['num_actions'], kw['value_support_size'], kw['reward_support_size'],
                     kw['num_res_blocks'])
    return net.cuda(), onet


ATARI_SMALL = dict(input_shape=(4, 96, 96), num_actions=6, num_res_blocks=2, num_planes=128, value_support_size=21,
                   reward_support_size=21)


def test_atari_net_vs_reference_recording(tile_rows):
    """MuZeroAtariNet: strided representation (SIMT stride-2 convs + avg pools around tcgen05 residual
    blocks at 48x48 / 24x24 / 12x12), 6x6 latent towers, support heads; against the reference's recording."""
    net, onet = build_atari(ATARI_SMALL, 5)
    z = np.load(os.path.join(GOLDEN, 'net_golden.npz'))
    for j in range(2):
        g = {k: z[f'atari_small_{j}_{k}'] for k in ('obs', 'actions', 'h0', 'pi0', 'v0', 'h', 'r', 'v', 'pi')}
        o = net.initial_inference(torch.from_numpy(g['obs'])[None].cuda())
        assert o.hidden_state.shape == (128, 6, 6)
        report(f'atari/{j} h0', o.hidden_state, g['h0'].astype(np.float32), TOL_H)
        report(f'atari/{j} pi0', o.pi_probs, g['pi0'], TOL_PV)
        report(f'atari/{j} v0', o.value, g['v0'], TOL_PV)
        h = g['h0'].astype(np.float32)
        for i, a in enumerate(g['actions']):
            o = net.recurrent_inference(torch.from_numpy(h)[None].cuda(), torch.tensor([[int(a)]]).cuda())
            report(f'atari/{j} h[{i}]', o.hidden_state, g['h'][i].astype(np.float32), TOL_H)
            report(f'atari/{j} r[{i}]', o.reward, g['r'][i], TOL_PV)
            report(f'atari/{j} v[{i}]', o.value, g['v'][i], TOL_PV)
            report(f'atari/{j} pi[{i}]', o.pi_probs, g['pi'][i], TOL_PV)
            h = g['h'][i].astype(np.float32)


def test_atari_batched_vs_torch_fp32():
    net, onet = build_atari(ATARI_SMALL, 5)
    gen = np.random.RandomState(3)
    B = 5
    obs = gen.randint(0, 256, size=(B, 4, 96, 96)).astype(np.float32)
    obs[:, 2:] = ((gen.randint(0, 6, size=(B, 2, 1, 1)) + 1) / 6).astype(np.float32)
    hid, pi, v = net.initial_inference_batch(torch.from_numpy(obs).cuda())
    h_ref, pi_ref, v_ref = onet.initial_batch(obs)
    report('atari h0', net.hidden_to_reference(hid).cpu().numpy(), h_ref.numpy(), TOL_H)
    report('atari pi0', pi.cpu().numpy(), pi_ref.numpy(), TOL_PV)
    report('atari v0', v.cpu().numpy(), v_ref.numpy(), TOL_PV)
    act = gen.randint(0, 6, size=B)
    _, r, pi2, v2 = net.recurrent_inference_batch(net.hidden_from_reference(h_ref.cuda()), torch.from_numpy(act).cuda())
    _, r_ref, pi2_ref, v2_ref = onet.recurrent_batch(h_ref, act)
    report('atari r', r.cpu().numpy(), r_ref.numpy(), TOL_PV)
    report('atari v1', v2.cpu().numpy(), v2_ref.numpy(), TOL_PV)
    report('atari pi1', pi2.cpu().numpy(), pi2_ref.numpy(), TOL_PV)


# ---------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[3] at its FULL shape (VERDICT r1 item 1a): 16 stacked planes, 18 actions, 8 blocks, support 61
# ---------------------------------------------------------------------------------------------------------------
ATARI_C4 = dict(input_shape=(16, 96, 96), num_actions=18, num_res_blocks=8, num_planes=128, value_support_size=61,
                reward_support_size=61)


def _chain_vs_recording(net, z, name, label, TOL_PV=TOL_PV):
    from test_net_golden_cpu import golden_obs
    # value / reward tolerance is relative to the scale of the head's outputs over the whole recording (a single
    # scalar's own magnitude says nothing about the head: a random-init value head ranges over +-30 and one of its
    # outputs may happen to be 2)
    vs = max(1.0, max(float(np.abs(z[f'{name}_{j}_{k}']).max()) for j in range(2) for k in ('v0', 'v')))
    rs = max(1.0, max(float(np.abs(z[f'{name}_{j}_r']).max()) for j in range(2)))
    for j in range(2):
        obs = golden_obs(z, name, j)
        g = {k: z[f'{name}_{j}_{k}'] for k in ('actions', 'h0', 'pi0', 'v0', 'h', 'r', 'v', 'pi')}
        o = net.initial_inference(torch.from_numpy(obs)[None].cuda())
        assert o.hidden_state.shape == g['h0'].shape and o.hidden_state.dtype == np.float32
        report(f'{label}/{j} h0', o.hidden_state, g['h0'].astype(np.float32), TOL_H)
        report(f'{label}/{j} pi0', o.pi_probs, g['pi0'], TOL_PV)
        report(f'{label}/{j} v0', o.value, g['v0'], TOL_PV, vs)
        h = g['h0'].astype(np.float32)
        for i, a in enumerate(g['actions']):
            o = net.recurrent_inference(torch.from_numpy(h)[None].cuda(), torch.tensor([[int(a)]]).cuda())
            report(f'{label}/{j} h[{i}]', o.hidden_state, g['h'][i].astype(np.float32), TOL_H)
            report(f'{label}/{j} r[{i}]', o.reward, g['r'][i], TOL_PV, rs)
            report(f'{label}/{j} v[{i}]', o.value, g['v'][i], TOL_PV, vs)
            report(f'{label}/{j} pi[{i}]', o.pi_probs, g['pi'][i], TOL_PV)
            h = g['h'][i].astype(np.float32)


def test_atari_c4_full_shape_vs_reference_recording(tile_rows):
    """MuZeroAtariNet((16, 96, 96), 18, 8, 128, 61, 61) -- the benchmarked shape -- against the reference's own
    recorded outputs (tests/golden/net_golden_r2.npz): 16-plane observation packing, both stride-2 tcgen05 convs, the
    full-depth towers, the support-61 heads."""
    net, _ = build_atari(ATARI_C4, 0)
    _chain_vs_recording(net, np.load(os.path.join(GOLDEN, 'net_golden_r2.npz')), 'atari_c4', 'atari_c4')


def test_atari_c4_search_replays_in_the_oracle_and_rows_match_fp32():
    """One 64-tree x 50-simulation search with the C4 network: every tree rebuilt bit-for-bit by the CPU oracle from
    the network outputs the engine produced, and sampled rows of the initial / recurrent inference compared with the
    fp32 torch restatement of the reference network."""
    import muzero_b200 as mz
    from parity_util import check_rows_against_oracle_net, replay_tree_in_oracle
    net, onet = build_atari(ATARI_C4, 0)
    cfg = mz.make_atari_config(use_tensorboard=False)
    cfg.num_simulations = 50
    B, A, S = 64, 18, 50
    gen = np.random.RandomState(44)
    obs = gen.randint(0, 256, size=(B, 16, 96, 96)).astype(np.float32)
    obs[:, 8:] = ((gen.randint(0, A, size=(B, 8, 1, 1)) + 1) / A).astype(np.float32)
    mask = np.ones((B, A), dtype=bool)
    streams = [np.random.RandomState(700 + t) for t in range(B)]
    plan = mz.mcts.SearchPlan(net, cfg, B)
    action, pi, rootv = mz.uct_search_batch(obs, net, cfg, 1.0, mask, 1, 1, rng=streams, plan=plan)
    plan.pool.check_errors()
    action_h, rootv_h = action.cpu(), rootv.cpu().numpy()
    noise = plan.noise.cpu().numpy()
    for t in range(B):
        rs = np.random.RandomState(700 + t)
        nz = rs.dirichlet(np.ones(A, dtype=np.float32) * cfg.root_dirichlet_alpha)
        assert np.array_equal(nz, noise[t])                    # numpy-exact mode: the host drew the noise
        replay_tree_in_oracle(plan, t, cfg, 1.0, mask[t], (1, 1), action_h, pi, rootv_h, rs, noise=nz)
        assert rs.get_state()[2] == streams[t].get_state()[2]
    # initial inference of 4 observations and 64 recurrent rows vs fp32 torch
    rows4 = [0, 21, 42, 63]
    h_ref, pi_ref, v_ref = onet.initial_batch(obs[rows4])
    S1 = S + 1
    roots = net.hidden_to_reference(plan.pool.hidden.view(B, S1, -1)[rows4, 0]).cpu().numpy()
    report('c4 root hidden', roots, h_ref.numpy(), TOL_H)
    report('c4 pi0', plan.pi0[rows4].cpu().numpy(), pi_ref.numpy(), TOL_PV)
    report('c4 v0', plan.v0[rows4].cpu().numpy(), v_ref.numpy(), TOL_PV)
    rows = [(int(t), int(k)) for t, k in zip(gen.choice(B, size=64), gen.randint(1, S1, size=64))]
    check_rows_against_oracle_net(net, onet, plan, rows, TOL_H, TOL_PV)


# ---------------------------------------------------------------------------------------------------------------
# Every network shape the reference builds (VERDICT r1 item 7): the ResNet Tic-Tac-Toe variant (16 planes,
# config.py:126-127), the class defaults 256 planes x 16 blocks (network.py:543-549) and the Atari class defaults
# 256 planes x 16 blocks with support 601 (network.py:504-512)
# ---------------------------------------------------------------------------------------------------------------
R2_SHAPES = {
    'ttt_resnet': ('board', dict(input_shape=(9, 3, 3), num_actions=10, num_res_blocks=2, num_planes=16), 7),
    'board_256x16': ('board', dict(input_shape=(9, 9, 9), num_actions=82, num_res_blocks=16, num_planes=256), 8),
    'atari_default': ('atari', dict(input_shape=(4, 96, 96), num_actions=6, num_res_blocks=16, num_planes=256,
                                    value_support_size=601, reward_support_size=601), 9),
}


def _build_r2(name):
    kind, kw, seed = R2_SHAPES[name]
    if kind == 'board':
        return build_board(kw['input_shape'], kw['num_actions'], kw['num_res_blocks'], kw['num_planes'], seed)
    return build_atari(kw, seed)


@pytest.mark.parametrize('name', list(R2_SHAPES))
def test_every_reference_network_shape_vs_reference_recording(name):
    net, _ = _build_r2(name)
    _chain_vs_recording(net, np.load(os.path.join(GOLDEN, 'net_golden_r2.npz')), name, name)


@pytest.mark.parametrize('name,batch,nref', [('ttt_resnet', 1000, 24), ('board_256x16', 300, 6)])
def test_new_board_shapes_batched_vs_torch_fp32(name, batch, nref, TOL_PV=TOL_PV):
    """Multi-tile dataflow launches of the padded (16 -> 32 planes) and the two-pass (256 planes) towers, with slot
    indirection on both sides, against fp32 torch on a subset of rows."""
    net, onet = _build_r2(name)
    kw = R2_SHAPES[name][1]
    A = kw['num_actions']
    gen = np.random.RandomState(batch)
    obs = gen.randint(0, 2, size=(batch,) + kw['input_shape']).astype(np.float32)
    hid, pi, v = net.initial_inference_batch(torch.from_numpy(obs).cuda())
    rows = np.sort(gen.choice(batch, size=nref, replace=False))
    h_ref, pi_ref, v_ref = onet.initial_batch(obs[rows])
    report(f'{name} h0', net.hidden_to_reference(hid)[rows].cpu().numpy(), h_ref.numpy(), TOL_H)
    report(f'{name} pi0', pi[rows].cpu().numpy(), pi_ref.numpy(), TOL_PV)
    report(f'{name} v0', v[rows].cpu().numpy(), v_ref.numpy(), TOL_PV)
    act = gen.randint(0, A, size=batch)
    src = torch.arange(batch - 1, -1, -1, dtype=torch.int32).cuda()
    dst = (torch.arange(batch, dtype=torch.int32) * 2 + 1).cuda()
    out = net.new_hidden(2 * batch + 1)
    _, r, pi2, v2 = net.recurrent_inference_batch(hid, torch.from_numpy(act).cuda(), src_index=src, hidden_out=out,
                                                  dst_index=dst)
    # row i read slot batch-1-i: reference rows for the sampled OUTPUT rows
    src_rows = batch - 1 - rows
    h_in = net.hidden_to_reference(hid)[src_rows].cpu()
    h2_ref, r_ref, pi2_ref, v2_ref = onet.recurrent_batch(h_in, act[rows])
    report(f'{name} h1', net.hidden_to_reference(out)[1::2][rows].cpu().numpy(), h2_ref.numpy(), TOL_H)
    report(f'{name} r', r[rows].cpu().numpy(), r_ref.numpy(), TOL_PV)
    # one scale for the value head over both calls (see _chain_vs_recording)
    vs = max(1.0, float(np.abs(v_ref.numpy()).max()), float(np.abs(v2_ref.numpy()).max()))
    report(f'{name} v1', v2[rows].cpu().numpy(), v2_ref.numpy(), TOL_PV, vs)
    # 16-block random-init towers put |logit| ~ 100 on the policy head: a relative logit error of 4e-4 (fp16 operands
    # through 49 convs) moves a probability by up to 0.04 where two logits nearly tie; stated tolerance 0.05 there
    report(f'{name} pi1', pi2[rows].cpu().numpy(), pi2_ref.numpy(), 0.05 if kw['num_res_blocks'] >= 16 else TOL_PV)
    assert (out.view(torch.float16)[0::2] == 0).all()        # untouched slots stay untouched
    if name == 'ttt_resnet':                                 # channels 16..31 of a slot are the zero padding
        pb = 9
        raw = out.view(torch.float16).reshape(2 * batch + 1, 4, pb, 8)
        assert (raw[1::2, 2:] == 0).all()


def test_resnet_tictactoe_variant_through_the_drop_in_uct_search():
    """The reference's own smoke configuration (tests/tictactoe/run_training_test.py:30-35: use_mlp_net=False ->
    MuZeroBoardGameNet(input_shape, num_actions, 2, 16)) through the unchanged uct_search signature."""
    import muzero_b200 as mz
    net, _ = _build_r2('ttt_resnet')
    cfg = mz.make_tictactoe_config(use_mlp_net=False, use_tensorboard=False)
    assert (cfg.num_planes, cfg.num_res_blocks) == (16, 2)
    gen = np.random.RandomState(3)
    obs = gen.randint(0, 2, size=(9, 3, 3)).astype(np.float32)
    mask = np.ones(10, dtype=bool)
    np.random.seed(11)
    a, pi, q = mz.uct_search(obs, net, 'cuda', cfg, 1.0, mask, 1, 2)
    plan = mz.mcts._plan_for(net, cfg, 1)
    d = plan.pool.dump_tree(0)
    np.random.seed(11)
    stub = ReplayStub(plan.pi0[0].cpu().numpy(), d['R'][1:].astype(np.float32), d['value'][1:], d['parent'], d['move'])
    a_o, pi_o, q_o = orc.uct_search(obs, stub, 'cpu', cfg, 1.0, mask, 1, 2)
    assert a == a_o and np.array_equal(bits(pi), bits(pi_o)) and bits(q)[0] == bits(q_o)[0]


def test_stacked_frames_equal_their_float32_expansion():
    """mz_net_initial_frames / StackedFrames: an Atari observation handed over as uint8 frames + action-plane values
    (gym_env.py:306-313) must give exactly what its float32 expansion gives -- hidden slots, policy, value, and a whole
    batched search."""
    import muzero_b200 as mz
    net, _ = build_atari(ATARI_SMALL, 5)
    gen = np.random.RandomState(8)
    B, A = 9, 6
    frames = torch.from_numpy(gen.randint(0, 256, size=(B, 2, 96, 96)).astype(np.uint8))
    planes = torch.from_numpy(((gen.randint(0, A, size=(B, 2)) + 1) / A).astype(np.float32))
    sf = mz.StackedFrames(frames, planes)
    full = sf.expand()
    assert full.shape == (B, 4, 96, 96) and full.dtype == torch.float32
    h1, pi1, v1 = net.initial_inference_batch(sf)
    h2, pi2, v2 = net.initial_inference_batch(full.cuda())
    assert torch.equal(h1, h2) and torch.equal(pi1, pi2) and torch.equal(v1, v2)
    cfg = mz.make_atari_config(use_tensorboard=False)
    cfg.num_simulations = 8
    out = []
    for obs in (sf, full):
        plan = mz.mcts.SearchPlan(net, cfg, B)
        streams = [np.random.RandomState(40 + t) for t in range(B)]
        a, pi, q = mz.uct_search_batch(obs, net, cfg, 1.0, np.ones((B, A), bool), 1, 1, rng=streams, plan=plan)
        a2, pi_2, q2 = mz.uct_search_batch(obs, net, cfg, 1.0, np.ones((B, A), bool), 1, 1,
                                           rng=[np.random.RandomState(40 + t) for t in range(B)], plan=plan)   # graph replay
        assert torch.equal(a, a2) and torch.equal(pi, pi_2)
        out.append((a.cpu(), pi.cpu(), q.cpu()))
    assert all(torch.equal(x, y) for x, y in zip(*out))
