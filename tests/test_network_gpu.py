"""GPU tests of the network kernels against the fp32 torch restatement of the reference
(oracle/network_oracle.py) and against the reference's own recorded outputs
(tests/golden/net_golden.npz).  Floating point: tolerances stated per test."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN, bits
from oracle import mcts_oracle as orc
from oracle.network_oracle import OracleNet
from oracle.stubnet import ReplayStub

pytestmark = pytest.mark.gpu

MLPS = {
    'tictactoe': dict(input_shape=(9, 3, 3), num_actions=10, num_planes=256, value_support_size=1,
                      reward_support_size=1, hidden_dim=64),
    'cartpole': dict(input_shape=(4, 5), num_actions=2, num_planes=512, value_support_size=31,
                     reward_support_size=31, hidden_dim=64),
    'lunarlander': dict(input_shape=(4, 9), num_actions=4, num_planes=512, value_support_size=31,
                        reward_support_size=31, hidden_dim=64),
}
# initial_inference: fp32 SIMT kernels vs fp32 torch, only the summation order differs
MLP_TOL = dict(rtol=2e-4, atol=2e-4)
# recurrent_inference: tcgen05 path, fp16 operands (hidden state in [0,1], trained weights) with fp32 accumulation.
# Stated tolerance: |err| <= 5e-3 * max(1, |ref|max) on hidden state, reward and value (measured on the three
# checkpoints at batch 4096: hidden <= 1.4e-3, reward / value <= 2.4e-3 of scale), <= 1e-2 on policy probabilities
# (measured <= 2.3e-3).
TC_TOL, TC_TOL_PI = 5e-3, 1e-2


def close_tc(got, ref, tol=TC_TOL, scale=None):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    scale = max(1.0, float(np.abs(ref).max())) if scale is None else scale
    err = float(np.abs(got - ref).max())
    assert np.isfinite(got).all() and err <= tol * scale, f'max err {err:.4g} > {tol * scale:.4g}'


# random-init nets that reach the one-launch search kernel's two-chunk and global-action-table paths
RANDOM_MLPS = {
    'p512_a8': dict(input_shape=(4, 5), num_actions=8, num_planes=512, value_support_size=31, reward_support_size=31,
                    hidden_dim=64),
    'p256_a20': dict(input_shape=(4, 5), num_actions=20, num_planes=256, value_support_size=31,
                     reward_support_size=31, hidden_dim=64),
}


def load_mlp(name):
    import muzero_b200 as mz
    if name in RANDOM_MLPS:
        kw = RANDOM_MLPS[name]
        torch.manual_seed(kw['num_planes'] + kw['num_actions'])
        net = mz.MuZeroMLPNet(**kw)
        sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    else:
        sd = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, f'ckpt_{name}.npz')).items()}
        kw = MLPS[name]
        net = mz.MuZeroMLPNet(**kw)
        net.load_state_dict(sd)
    net = net.cuda().eval()
    orc_net = OracleNet('mlp', sd, kw['num_actions'], kw['value_support_size'], kw['reward_support_size'])
    return net, orc_net, kw


@pytest.mark.parametrize('name', list(MLPS))
def test_mlp_single_item_api_vs_reference_recording(name):
    """initial_inference + chained recurrent_inference, the reference's own API and types."""
    net, _, kw = load_mlp(name)
    z = np.load(os.path.join(GOLDEN, 'net_golden.npz'))
    for j in range(4):
        g = {k: z[f'{name}_{j}_{k}'] for k in ('obs', 'actions', 'h0', 'pi0', 'v0', 'h', 'r', 'v', 'pi')}
        o = net.initial_inference(torch.from_numpy(g['obs'])[None].cuda())
        assert isinstance(o.value, float) and isinstance(o.reward, float) and o.reward == 0.0
        assert o.hidden_state.dtype == np.float32 and o.hidden_state.shape == (64,)
        assert o.pi_probs.dtype == np.float32 and o.pi_probs.shape == (kw['num_actions'],)
        np.testing.assert_allclose(o.hidden_state, g['h0'], **MLP_TOL)
        np.testing.assert_allclose(o.pi_probs, g['pi0'], **MLP_TOL)
        np.testing.assert_allclose(o.value, g['v0'], **MLP_TOL)
        h = g['h0']
        for i, a in enumerate(g['actions']):
            # feed the REFERENCE's hidden state so errors do not compound along the chain
            o = net.recurrent_inference(torch.from_numpy(h)[None].cuda(), torch.tensor([[int(a)]]).cuda())
            close_tc(o.hidden_state, g['h'][i])
            close_tc(o.reward, g['r'][i])
            close_tc(o.value, g['v'][i])
            close_tc(o.pi_probs, g['pi'][i], TC_TOL_PI)
            h = g['h'][i]


@pytest.mark.parametrize('name', list(MLPS))
@pytest.mark.parametrize('batch', [1, 31, 100, 4096])
def test_mlp_batched_vs_torch_fp32(name, batch):
    net, onet, kw = load_mlp(name)
    gen = np.random.RandomState(batch)
    obs = gen.standard_normal((batch,) + kw['input_shape']).astype(np.float32)
    hidden, pi, value = net.initial_inference_batch(torch.from_numpy(obs).cuda())
    h_ref, pi_ref, v_ref = onet.initial_batch(obs)
    np.testing.assert_allclose(net.hidden_to_reference(hidden).cpu().numpy(), h_ref.numpy(), **MLP_TOL)
    np.testing.assert_allclose(pi.cpu().numpy(), pi_ref.numpy(), **MLP_TOL)
    np.testing.assert_allclose(value.cpu().numpy(), v_ref.numpy(), **MLP_TOL)
    act = gen.randint(0, kw['num_actions'], size=batch)
    # gather through slot indices like the search does: reversed order in, strided order out
    src = torch.arange(batch - 1, -1, -1, dtype=torch.int32).cuda()
    dst = (torch.arange(batch, dtype=torch.int32) * 2).cuda()
    out = net.new_hidden(2 * batch)
    slots_in = net.hidden_from_reference(h_ref.cuda())
    _, reward, pi2, value2 = net.recurrent_inference_batch(slots_in, torch.from_numpy(act).cuda(), src_index=src,
                                                           hidden_out=out, dst_index=dst)
    h2_ref, r_ref, pi2_ref, v2_ref = onet.recurrent_batch(h_ref.flip(0), act)
    close_tc(net.hidden_to_reference(out)[::2].cpu().numpy(), h2_ref.numpy())
    close_tc(reward.cpu().numpy(), r_ref.numpy())
    close_tc(value2.cpu().numpy(), v2_ref.numpy())
    close_tc(pi2.cpu().numpy(), pi2_ref.numpy(), TC_TOL_PI)
    assert (net.hidden_to_reference(out)[1::2] == 0).all()          # untouched slots stay untouched
    # policy head skipped (what the search asks for): same reward/value
    _, reward3, pi3, value3 = net.recurrent_inference_batch(slots_in, torch.from_numpy(act).cuda(), src_index=src,
                                                            want_policy=False)
    assert pi3 is None and torch.equal(reward3, reward) and torch.equal(value3, value2)
    # the fp32 SIMT kernel (MZ_MLP_SIMT=1 selects it for every call) stays within the fp32 tolerance: covered by
    # initial_inference above, which always runs on it


def test_engine_tracks_weight_updates():
    net, onet, kw = load_mlp('tictactoe')
    obs = torch.zeros((3,) + kw['input_shape']).cuda()
    _, pi_a, _ = net.initial_inference_batch(obs)
    with torch.no_grad():
        net.prediction_net.policy_net[2].bias.add_(torch.arange(10.0).cuda())
    _, pi_b, _ = net.initial_inference_batch(obs)
    assert not torch.allclose(pi_a, pi_b)
    sd = {k: v.cpu() for k, v in net.state_dict().items()}
    ref = OracleNet('mlp', sd, 10, 1, 1).initial_batch(obs.cpu())[1]
    np.testing.assert_allclose(pi_b.cpu().numpy(), ref.numpy(), **MLP_TOL)


@pytest.mark.parametrize('name,B,deterministic', [('tictactoe', 256, False), ('cartpole', 128, True),
                                                  ('lunarlander', 64, False)])
def test_search_with_engine_network_replays_bit_exact_in_oracle(name, B, deterministic):
    """T2 of SURVEY.md §8c: run the whole batched search on the GPU with its own network,
    record what the network said for every node, feed exactly that to the oracle: trees,
    policies, actions, root values and RNG streams must be bit-identical."""
    import muzero_b200 as mz
    net, onet, kw = load_mlp(name)
    cfg = mz.make_tictactoe_config(use_tensorboard=False) if name == 'tictactoe' else \
        mz.make_classic_config(use_tensorboard=False)
    A, S = kw['num_actions'], cfg.num_simulations
    gen = np.random.RandomState(B)
    if name == 'tictactoe':
        obs = gen.randint(0, 2, size=(B,) + kw['input_shape']).astype(np.float32)
        mask = gen.rand(B, A) < 0.7
        mask[:, -1] = True
        cur, opp = gen.randint(1, 3, size=B), None
        opp = 3 - cur
    else:
        obs = gen.standard_normal((B,) + kw['input_shape']).astype(np.float32)
        mask = np.ones((B, A), bool)
        cur = opp = np.ones(B, int)
    dev = torch.device('cuda', 0)
    pool = mz.SearchPool(B, A, cfg, net.hidden_bytes, dev)
    streams = [np.random.RandomState(1000 + t) for t in range(B)]
    # instrumented copy of uct_search_batch's loop (same calls, plus recording)
    root_slots = torch.arange(B, dtype=torch.int32, device=dev) * (S + 1)
    _, pi0, _ = net.initial_inference_batch(torch.from_numpy(obs).to(dev), hidden_out=pool.hidden, dst_index=root_slots)
    noise = None
    if not deterministic:
        noise = np.stack([r.dirichlet(np.ones(A, np.float32) * cfg.root_dirichlet_alpha) for r in streams])
    pool.set_rng_states([r.get_state() for r in streams])
    mask_d = torch.from_numpy(mask.astype(np.uint8)).to(dev)
    players = torch.from_numpy(np.stack([cur, opp], 1).astype(np.int32)).to(dev)
    pool.reset(pi0, None if noise is None else torch.from_numpy(noise).to(dev),
               cfg.root_exploration_eps if noise is not None else 0.0, mask_d, players)
    rec_r = torch.empty((S, B), device=dev); rec_v = torch.empty((S, B), device=dev)
    rec_p = torch.empty((S, B), dtype=torch.int32, device=dev); rec_a = torch.empty((S, B), dtype=torch.int32, device=dev)
    for i in range(S):
        pool.select()
        _, r, _, v = net.recurrent_inference_batch(pool.hidden, pool.view('LEAF_ACTION'),
                                                   src_index=pool.view('SRC_SLOT'), hidden_out=pool.hidden,
                                                   dst_index=pool.view('DST_SLOT'), want_policy=False)
        rec_r[i], rec_v[i] = r, v
        rec_p[i].copy_(pool.view('LEAF_PARENT')); rec_a[i].copy_(pool.view('LEAF_ACTION'))
        pool.expand_backup(r, v)
    temps = torch.full((B,), 1.0, dtype=torch.float64, device=dev)
    action, pi, rootv, _ = pool.root_policy(mask_d, temps, deterministic)
    pool.check_errors()
    states = pool.get_rng_states()
    rec_r, rec_v, rec_p, rec_a = (x.cpu().numpy() for x in (rec_r, rec_v, rec_p, rec_a))
    pi0 = pi0.cpu().numpy()
    for t in range(0, B, max(1, B // 24)):
        rs = np.random.RandomState(1000 + t)
        stub = ReplayStub(pi0[t], rec_r[:, t], rec_v[:, t], np.concatenate([[-1], rec_p[:, t]]),
                          np.concatenate([[-1], rec_a[:, t]]))
        a_o, pi_o, q_o, tr = orc.uct_search(obs[t], stub, 'cpu', cfg, 1.0, mask[t], int(cur[t]), int(opp[t]),
                                            deterministic, rng=rs, return_trace=True)
        d = pool.dump_tree(t)
        assert np.array_equal(d['N'], tr.N) and np.array_equal(bits(d['W']), bits(tr.W))
        assert np.array_equal(d['parent'], tr.parent) and np.array_equal(d['move'], tr.move)
        assert a_o == int(action[t]) and np.array_equal(bits(pi_o), bits(pi[t].cpu().numpy()))
        assert bits(q_o)[0] == bits(rootv[t].item())[0]
        assert states[t][2] == rs.get_state()[2] and np.array_equal(states[t][1], rs.get_state()[1])
    # and the network values it was fed are the reference network's, to tolerance, at the recorded nodes
    t = 0
    hid = net.hidden_to_reference(pool.hidden.view(B, S + 1, -1)[t]).cpu()
    for i in range(0, S, 5):
        h_ref, r_ref, _, v_ref = onet.recurrent_batch(hid[rec_p[i, t]][None], np.array([rec_a[i, t]]))
        scale = max(1.0, float(np.abs(rec_v[:, t]).max()), float(np.abs(rec_r[:, t]).max()))
        close_tc(rec_r[i, t], r_ref.numpy()[0], scale=scale)
        close_tc(rec_v[i, t], v_ref.numpy()[0], scale=scale)
        close_tc(hid[i + 1].numpy(), h_ref.numpy()[0])


def test_public_batch_entry_point_matches_manual_loop():
    """uct_search_batch (numpy-exact rng mode) == the single-tree drop-in uct_search, tree by tree."""
    import muzero_b200 as mz
    net, _, kw = load_mlp('tictactoe')
    cfg = mz.make_tictactoe_config(use_tensorboard=False)
    B, A = 12, 10
    gen = np.random.RandomState(0)
    obs = gen.randint(0, 2, size=(B,) + kw['input_shape']).astype(np.int8)
    mask = gen.rand(B, A) < 0.7
    mask[:, -1] = True
    streams = [np.random.RandomState(50 + t) for t in range(B)]
    a_b, pi_b, q_b = mz.uct_search_batch(obs, net, cfg, 1.0, mask, 1, 2, rng=streams)
    for t in range(B):
        np.random.seed(50 + t)
        a, pi, q = mz.uct_search(obs[t], net, 'cuda', cfg, 1.0, mask[t], 1, 2)
        assert a == int(a_b[t]) and np.array_equal(bits(pi), bits(pi_b[t].cpu().numpy()))
        assert bits(q)[0] == bits(q_b[t].item())[0]
        assert np.random.get_state()[2] == streams[t].get_state()[2]
        assert np.array_equal(np.random.get_state()[1], streams[t].get_state()[1])


@pytest.mark.parametrize('family', ['mlp', 'conv'])
@pytest.mark.parametrize('noise_mode', ['none', 'given', 'device'])
def test_fused_root_epilogue_equals_the_separate_launches(family, noise_mode, monkeypatch):
    """mz_net_initial_search (Dirichlet draw + noise mix + mask + renormalise + root reset fused behind the policy
    softmax of the initial inference) against mz_net_initial + mz_dirichlet + mz_search_reset: every byte of the
    pool after the root preparation, the noise, the RNG streams, and the finished search."""
    import muzero_b200 as mz
    torch.manual_seed(2)
    if family == 'mlp':
        net = mz.MuZeroMLPNet((9, 3, 3), 10, 256, 1, 1, 64).cuda().eval()
        cfg = mz.make_tictactoe_config(use_tensorboard=False)
        B, A, shape = 70, 10, (9, 3, 3)
    else:
        net = mz.MuZeroBoardGameNet((5, 5, 5), 26, 2, 32).cuda().eval()
        cfg = mz.make_gomoku_config(use_tensorboard=False)
        cfg.num_simulations = 12
        B, A, shape = 37, 26, (5, 5, 5)
    gen = np.random.RandomState(9)
    obs = gen.randint(0, 2, size=(B,) + shape).astype(np.float32)
    mask = gen.rand(B, A) < 0.7
    mask[:, -1] = True
    given = gen.dirichlet(np.ones(A) * 0.3, size=B)
    out = []
    for fused in (False, True):
        monkeypatch.setattr(mz.mcts, '_FUSED_ROOT', fused)
        plan = mz.mcts.SearchPlan(net, cfg, B)
        plan.use_graph = False
        plan.pool.seed(np.arange(B) + 31)
        plan.obs.copy_(torch.from_numpy(obs).reshape(B, -1)); plan.mask.copy_(torch.from_numpy(mask))
        plan.players.copy_(torch.tensor([[1, 2]] * B, dtype=torch.int32))
        plan.noise.copy_(torch.from_numpy(given))
        net.engine(B, plan.instance)                     # engine creation launches its repacking kernels: not counted
        n0 = mz._lib.lib().mz_launch_count()
        plan.run(noise_mode, True, False)
        launches = mz._lib.lib().mz_launch_count() - n0
        torch.cuda.synchronize()
        plan.pool.check_errors()
        names = ('EDGES', 'EDGE_W', 'EDGE_REWARD', 'PRIOR', 'MINMAX', 'ROOT_W', 'ROOT_N', 'COUNT', 'NODE_PARENT', 'NODE_MOVE',
                 'RNG_KEY', 'RNG_POS')
        state = {k: plan.pool.view(k).cpu().numpy().view(np.uint8).copy() for k in names}
        state['noise'] = plan.noise.cpu().numpy().view(np.uint8).copy()
        state['pi'] = plan.pi.cpu().numpy().view(np.uint8).copy()
        state['action'] = plan.action.cpu().numpy().copy()
        out.append((state, launches))
    (sep, n_sep), (fus, n_fus) = out
    for k in sep:
        assert np.array_equal(sep[k], fus[k]), f'{family}/{noise_mode}: {k} differs'
    assert n_fus == n_sep - (2 if noise_mode == 'device' else 1)


def test_fp16_networks_rarely_change_a_search():
    """Search-level effect of fp16 tensor-core inference (VERDICT r1 item 9): 256 Tic-Tac-Toe searches with the
    checkpoint network, engine vs the oracle search driven by the fp32 torch network on the same inputs, noise and
    RNG streams.  Bound (measured: see profiles/r2_fp16_search_stats.json): the sampled action differs in <= 5 % of
    the trees, the mean L1 distance between the visit policies is <= 0.05."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(GOLDEN), '..', 'tools'))
    from fp16_search_stats import search_stats
    s = search_stats('tictactoe', 256)
    print(s)
    assert s['sampled_action_differs'] <= 0.05 and s['mean_l1_visit_policy'] <= 0.05


@pytest.mark.parametrize('name,B', [('tictactoe', 300), ('cartpole', 200), ('lunarlander', 130), ('tictactoe', 4096),
                                    ('tictactoe', 4800), ('p512_a8', 200), ('p256_a20', 200)])
@pytest.mark.parametrize('noise_mode', ['device', 'none'])
def test_one_launch_search_kernel_equals_the_launch_chain(name, B, noise_mode):
    """mz_search_run's persistent kernels for the MLP nets -- one launch per search: 32 trees per CTA with a warp per
    tree (Tic-Tac-Toe up to 32 trees per SM), or 128 trees per CTA with a thread per tree (the other cases here, on
    request; the random-init nets take the warp-per-tree kernel's two-chunk and global-action-table paths) -- against
    the per-simulation launch chain (warp-per-tree / thread-per-tree tree kernels + one tcgen05
    launch per simulation), which the lock-step and replay tests pin to the oracle: trees, statistics, hidden states,
    RNG streams, policies and actions, byte for byte."""
    import muzero_b200 as mz
    from muzero_b200 import _lib
    net, _, kw = load_mlp(name)
    cfg = {'tictactoe': mz.make_tictactoe_config, 'cartpole': mz.make_classic_config, 'lunarlander': mz.make_classic_config,
           'p512_a8': mz.make_classic_config, 'p256_a20': mz.make_classic_config}[name](use_tensorboard=False)
    A = kw['num_actions']
    gen = np.random.RandomState(B + A)
    obs = gen.standard_normal((B,) + kw['input_shape']).astype(np.float32)
    mask = gen.rand(B, A) < 0.8
    mask[:, 0] = True
    board = bool(cfg.is_board_game)
    out = []
    for fused in (0, 1):
        plan = mz.mcts.SearchPlan(net, cfg, B)
        plan.use_graph = False
        eng = net.engine(B, plan.instance)
        _lib.check(_lib.lib().mz_net_set_fused_search(eng['handle'], fused))
        plan.pool.seed(np.arange(B) + 77)
        plan.obs.copy_(torch.from_numpy(obs).reshape(B, -1)); plan.mask.copy_(torch.from_numpy(mask))
        plan.players.copy_(torch.tensor([[1, 2 if board else 1]] * B, dtype=torch.int32))
        n0 = _lib.lib().mz_launch_count()
        plan.run(noise_mode, True, False)
        launches = _lib.lib().mz_launch_count() - n0
        torch.cuda.synchronize()
        plan.pool.check_errors()
        names = ('EDGES', 'EDGE_W', 'EDGE_REWARD', 'PRIOR', 'MINMAX', 'ROOT_W', 'ROOT_N', 'COUNT', 'NODE_PARENT',
                 'NODE_MOVE', 'RNG_KEY', 'RNG_POS', 'HIDDEN')
        state = {k: plan.pool.view(k).cpu().numpy().view(np.uint8).copy() for k in names}
        # the root's entry of NODE_VALUE is never written (the search does not use the root value)
        state['NODE_VALUE'] = plan.pool.view('NODE_VALUE').view(B, -1)[:, 1:].cpu().numpy().view(np.uint8).copy()
        state['pi'] = plan.pi.cpu().numpy().view(np.uint8).copy()
        state['action'] = plan.action.cpu().numpy().copy()
        state['root_value'] = plan.root_value.cpu().numpy().view(np.uint8).copy()
        state['stats'] = plan.pool.view('STATS').cpu().numpy()[:4].copy()
        out.append((state, launches))
        _lib.check(_lib.lib().mz_net_set_fused_search(eng['handle'], 0))
    (chain, n_chain), (fus, n_fus) = out
    for k in chain:
        assert np.array_equal(chain[k], fus[k]), f'{name}: {k} differs between the launch chain and the one-launch kernel'
    S = cfg.num_simulations
    if 'MZ_FUSED_SEARCH' not in os.environ and 'MZ_NO_FUSED_ROOT' not in os.environ:      # process-wide overrides
        assert n_chain == n_fus + 2 * S and n_fus <= 4      # initial inference (+ root setup fused), search, root policy
