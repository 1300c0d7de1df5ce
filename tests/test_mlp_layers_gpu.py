"""Layer-by-layer tests of the MLP inference kernels (csrc/mlp.cu) -- the fp32 SIMT kernels mlp_initial_kernel and
mlp_recurrent_kernel, and the tcgen05 kernel mlp_tc_kernel in each of its launch forms -- against a float64
computation fed the engine's OWN stored tensors (``mz_net_debug_capture``: with capture on, every intermediate of a
call keeps a region of its own, and every launch is recorded with the form the host chose for it).

u = 2^-24 (fp32), ulp16(r) the fp16 spacing at |r| (2^-24 below 2^-14).  Weights are the fp32 state_dict tensors;
the tcgen05 kernel reads them as W16 = fp16(clamp(w, +-65504)) (pack_linear_kernel).  Every bound carries a floor of
(steps) 2^-149 for fp32 subnormals.

* tcgen05 hidden layer (per net, every 256-column chunk, stored fp16 by epilogue 1): inputs X16 = fp16(clamp(x)) of the
  gathered slot (transition), of the captured raw transition output (reward) or of its fp32 normalisation (value,
  policy).  R = X16 W16^T + b1 [+ T_a], where T_a is the fp32 first-layer weight column of the action
  (action_column_kernel, not rounded to fp16), ref = clamp(R, 0, 65504), and
      |H - ref| <= ulp16(ref) + (64/16 + 2) u (|X16| |W16|^T + |b1| + |T_a|).
  The products fp16 x fp16 are exact in fp32; the K = 64 input runs as 4 MMAs of K = 16 into an fp32 accumulator,
  one round-to-nearest per step, each step erring by at most u times the magnitude sum; the bias and the action column
  add one rounding each; ReLU does not grow an error and the conversion to fp16 adds half an ulp16 (inside ulp16(ref)).
* tcgen05 second Linear (fp32 output + b2 before the transform): input the captured fp16 hidden layer M, so
  |Y - (M W2_16^T + b2)| <= (P/16 + 2) u (|M| |W2_16|^T + |b2|): P/16 MMA steps and the bias.  No fp16 term: tight.
* SIMT Linear (fp32 weights, captured fp32 input): dense_cols seeds an fp32 FMA chain with the bias and adds the
  action's weight row after it, so |Y - ref| <= (K + 2) u mag; dense_tiny (outputs < 16 of a head's second layer)
  sums 32 lane chains of ceil(K/32) FMAs, a 5-level butterfly and the bias: (ceil(K/32) + 7) u mag.
* Normalisation (util.py:31-36) is all explicit round-to-nearest intrinsics in both kernels, so it is restated in fp32
  torch and must match BIT FOR BIT: tcgen05 (h - mn) * RN(1 / RN(RN(mx - mn) + 1e-8)), SIMT (h - mn) / RN(RN(mx - mn)
  + 1e-8).  hidden_out holds those bits in the slots dst_index names, and every other slot keeps its bytes.  In the
  split form both CTAs of a tile run the transition: their raw outputs must be the same bits (part 1's feeds the value
  and policy nets, part 0's the reward net and hidden_out).
* Output transforms on the captured fp32 logits (so the logit error is 0): test_conv_layers_gpu.transform_ratio, whose
  constants are for 32 lane sums (SIMT: support_to_scalar, softmax_rows) or, seq=True, for one thread summing the n
  terms in order (tcgen05: support_scalar_regs and the policy epilogue): the sums of n terms err by (n - 1) u each,
  expectation and normaliser together by 2n u, against n/32 + 5 for lane sums.  A support of one is the logit itself.
* Capture off vs on: every case runs both ways and the slots, pi, value and reward are the same bytes.
* Forms: each case asserts, from the launch records, the forms it is named for, and ``test_cases_cover_every_form``
  that together they reach every form.  Large batches are checked on a sample of rows: the first and last, both
  rows at every 128-row boundary, and 8 random ones.

``test_reference_flags_planted_errors`` checks the reference itself on the CPU.
Measured worst error / bound over all cases (NVIDIA B200, 1000 W power limit): tcgen05 hidden layer 0.50, tcgen05
second Linear 0.47, SIMT Linear 0.14, policy 0.30, value 0.65, reward 0.63; normalisation, hidden_out and the two
split-form transition copies bit-identical."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

from test_conv_layers_gpu import U32, safe_ratio, transform_ratio, ulp16

NETS = ('representation', 'transition', 'reward', 'value', 'policy')
PREFIX = ('represent_net.net', 'dynamics_net.transition_net', 'dynamics_net.reward_net', 'prediction_net.value_net',
          'prediction_net.policy_net')
FORMS = ('simt_initial', 'simt_recurrent', 'tc_split_policy', 'tc_split_no_policy', 'tc_one_cta', 'tc_multi_tile',
         'one_chunk', 'two_chunks', 'tab_global', 'tab_smem', 'policy_wide')
SUB = 2.0 ** -149


# ---- the float64 reference (device-agnostic; runs on the sampled rows, on the CPU) ---------------------------------
def f16(x):
    return x.float().clamp(-65504.0, 65504.0).half().double()


def normalise_fp32(raw, tc):
    """The kernels' min-max normalisation restated in fp32 (every operation rounds once, as their _rn intrinsics)."""
    h = raw.float()
    mn, mx = h.amin(1, keepdim=True), h.amax(1, keepdim=True)
    den = (mx - mn) + torch.tensor(1e-8, dtype=torch.float32)
    return (h - mn) * (1.0 / den) if tc else (h - mn) / den


def linear_ratio(Y, X, W, b, steps, tab=None, relu=False, half_out=False):
    R = X @ W.T + b
    mag = X.abs() @ W.abs().T + b.abs()
    if tab is not None:
        R, mag = R + tab, mag + tab.abs()
    if relu:
        R = R.clamp_min(0.0)
    bound = steps * (U32 * mag + SUB)
    if half_out:
        R = R.clamp(max=65504.0)
        bound = bound + ulp16(R)
    return safe_ratio((Y - R).abs(), bound)


def structure(recs, tc, nsplit, recurrent, policy):
    """{(net, layer, part): the (net, layer, part) it reads (None: observation / slots)} from the network's structure."""
    want = {}
    parts = range(nsplit) if tc else [0]
    n0 = 1 if recurrent else 0
    for part in parts:
        runs = lambda n: nsplit == 1 or n == 1 or (n == 2) == (part == 0)
        want[(n0, 0, part)] = None
        want[(n0, 1, part)] = (n0, 0, part)
        if not tc:
            want[(n0, 2, part)] = (n0, 1, part)
        heads = ([2] if recurrent else []) + [3] + ([4] if policy else [])
        for n in heads:
            if tc and not runs(n):
                continue
            want[(n, 0, part)] = (n0, 1, part) if (n == 2 or tc) else (n0, 2, part)
            want[(n, 1, part)] = (n, 0, part)
    return want


def check_call(sd, cfg, recs, tc, nsplit, x_in, action=None, outputs=None, hidden=None, per=None):
    """Every check of one recorded call.  recs: {(net, layer, part): float64 [rows, cols]} on the sampled rows;
    x_in: the observation (initial) or the gathered slots (recurrent), float64; outputs: {'pi', 'value', 'reward'};
    hidden: the sampled rows of the slots the call wrote (float32).  Returns {check: (worst ratio, where)}."""
    worst = {}
    recurrent = action is not None

    def note(check, v, where):
        if per is not None:
            per[(check, where)] = max(v, per.get((check, where), 0.0))
        if check not in worst or not v <= worst[check][0]:
            worst[check] = (v, where)
    HD, P = cfg['HD'], cfg['P']
    n0 = 1 if recurrent else 0
    norm = {}
    for (net, layer, part), Y in sorted(recs.items()):
        where = f'{NETS[net]} {layer} part {part}'
        pre = PREFIX[net]
        if layer == 2:
            continue
        if layer == 0:
            w = sd[pre + '.0.weight'].double()
            b = sd[pre + '.0.bias'].double()
            tab = None
            if net == n0:
                X = x_in
                if recurrent:
                    tab = w[:, HD + action.long()].T
                    w = w[:, :HD]
            elif net == 2:
                X = recs[(n0, 1, part)]
            else:
                raw = recs[(n0, 1, part)]
                X = normalise_fp32(raw, True).double() if tc else recs[(n0, 2, part)]
            if tc:
                note('tc_hidden', linear_ratio(Y, f16(X), f16(w), b, HD // 16 + 2, tab, relu=True, half_out=True), where)
            else:
                note('simt_linear', linear_ratio(Y, X, w, b, X.shape[1] + 2, tab, relu=True), where)
        else:
            M = recs[(net, 0, part)]
            w = sd[pre + '.2.weight'].double()
            b = sd[pre + '.2.bias'].double()
            if tc:
                note('tc_out', linear_ratio(Y, M, f16(w), b, P // 16 + 2), where)
            else:
                tiny = net >= 2 and w.shape[0] < 16
                note('simt_linear', linear_ratio(Y, M, w, b, math.ceil(P / 32) + 7 if tiny else P + 2), where)
            if net == n0:
                nm = normalise_fp32(Y, tc)
                norm[part] = nm
                if not tc:
                    got = recs[(n0, 2, part)].float()
                    note('norm_bits', 0.0 if torch.equal(got, nm) else math.inf, f'{NETS[net]} 2 part 0')
    if tc and len(norm) == 2:
        note('split_parts_equal', 0.0 if torch.equal(recs[(n0, 1, 0)], recs[(n0, 1, 1)]) else math.inf, 'transition')
    if hidden is not None:
        note('hidden_out_bits', 0.0 if torch.equal(hidden, norm[0]) else math.inf, 'hidden_out')
    if outputs:
        for key, net, kind in (('reward', 2, cfg['rkind']), ('value', 3, cfg['vkind']), ('pi', 4, 2)):
            if key not in outputs:
                continue
            lg = [v for (n, l, _), v in recs.items() if n == net and l == 1][0]
            note('head_' + key, transform_ratio(outputs[key], lg, torch.zeros_like(lg), kind, seq=tc), key)
    return worst


# ---- the reference checked on the CPU against an eager float64 run ----------------------------------------------------
def _eager_record(sd, cfg, tc, slots, action):
    """The records a recurrent call would make, from an eager float64 run of the MLP nets (the normalisation in fp32,
    which the check requires bit for bit).  tc: the split form's two parts, fp16 operands as the tcgen05 kernel
    rounds them."""
    HD = cfg['HD']
    recs = {}
    lin = lambda pre, x, j: x @ sd[f'{pre}.{j}.weight'].double().T + sd[f'{pre}.{j}.bias'].double()
    q = f16 if tc else (lambda x: x)
    w = sd[PREFIX[1] + '.0.weight'].double()
    for part in ((0, 1) if tc else (0,)):
        h = (q(slots) @ q(w[:, :HD]).T + sd[PREFIX[1] + '.0.bias'].double() + w[:, HD + action.long()].T).clamp_min(0)
        recs[(1, 0, part)] = h
        raw = h @ q(sd[PREFIX[1] + '.2.weight'].double()).T + sd[PREFIX[1] + '.2.bias'].double()
        recs[(1, 1, part)] = raw
        nm = normalise_fp32(raw, tc).double()
        if not tc:
            recs[(1, 2, part)] = nm
        for n, x in ((2, raw), (3, nm), (4, nm)):
            if tc and (n == 2) != (part == 0):
                continue
            pre = PREFIX[n]
            hn = (q(x) @ q(sd[pre + '.0.weight'].double()).T + sd[pre + '.0.bias'].double()).clamp_min(0)
            recs[(n, 0, part)] = hn
            recs[(n, 1, part)] = hn @ q(sd[pre + '.2.weight'].double()).T + sd[pre + '.2.bias'].double()
    return recs


def _support(lg):
    n = lg.shape[1]
    if n == 1:
        return lg.view(-1)
    hi = (n - 1) // 2
    x = (torch.softmax(lg, 1) * torch.linspace(-hi, hi, n, dtype=torch.float64)).sum(1)
    return torch.sign(x) * ((torch.sqrt(1 + 4e-3 * (1e-3 + 1 + x.abs())) / 2e-3 - 500) ** 2 - 1)


def _cpu_net(P, A, S, seed):
    import muzero_b200 as mz
    torch.manual_seed(seed)
    net = mz.MuZeroMLPNet((4, 5), A, P, S, S, 64)
    # weights exactly representable in fp16, so that the float64 run and the tcgen05 reference use the same operands
    sd = {k: v.detach().half().double() for k, v in net.state_dict().items()}
    return sd, dict(HD=64, P=P, A=A, vkind=int(S > 1), rkind=int(S > 1))


@pytest.mark.parametrize('tc', [True, False], ids=['tcgen05', 'simt'])
def test_reference_flags_planted_errors(tc):
    """Records of an eager float64 run pass every check with wide margin, and each planted error is flagged at its
    layer: 3 fp16 ulps on one hidden-chunk element; chunk 1 computed with chunk 0's bias columns; the action column of
    a + 1 on one row; the min-max taken over 63 of 64 columns; the reward net fed the normalised state instead of the
    raw one; a padded policy column included in the softmax; one term of a SIMT K-tail dropped."""
    P, A = (512, 10) if tc else (50, 10)
    sd, cfg = _cpu_net(P, A, 31, 3)
    sd[PREFIX[1] + '.2.bias'][63] = 8.0             # column 63 holds every row's maximum
    g = torch.Generator().manual_seed(4)
    B = 6
    slots = torch.rand(B, 64, generator=g, dtype=torch.float64).float().double()
    action = torch.randint(0, A, (B,), generator=g)
    recs = _eager_record(sd, cfg, tc, slots, action)
    outs = dict(reward=_support(recs[(2, 1, 0)]), value=_support(recs[(3, 1, 1 if tc else 0)]),
                pi=torch.softmax(recs[(4, 1, 1 if tc else 0)], 1))
    hidden = normalise_fp32(recs[(1, 1, 0)], tc)
    nsplit = 2 if tc else 1
    worst = check_call(sd, cfg, recs, tc, nsplit, slots, action, outs, hidden)
    assert max(v for v, _ in worst.values()) <= 1e-2, worst
    want = {'tc_hidden', 'tc_out', 'split_parts_equal'} if tc else {'simt_linear', 'norm_bits'}
    assert want | {'hidden_out_bits', 'head_reward', 'head_value', 'head_pi'} <= set(worst), worst

    def flagged(mutate, check, where):
        r = {k: v.clone() for k, v in recs.items()}
        o = {k: v.clone() for k, v in outs.items()}
        hid = mutate(r, o)
        per = {}
        check_call(sd, cfg, r, tc, nsplit, slots, action, o, hidden if hid is None else hid, per=per)
        assert per.get((check, where), 0.0) > 1.0, (check, where, per)
    lin0 = 'tc_hidden' if tc else 'simt_linear'

    def bump(r, o):                   # 3 fp16 ulps on the largest element of the transition's hidden layer
        d = r[(1, 0, 0)].view(-1)
        k = int(d.abs().argmax())
        d[k] += 3 * ulp16(d[k])
    flagged(bump, lin0, 'transition 0 part 0')

    if tc:
        def chunk_bias(r, o):         # chunk 1 (columns 256..511) with chunk 0's bias columns
            pre = PREFIX[3]
            b = sd[pre + '.0.bias'].double().clone()
            b[256:] = b[:256]
            x = f16(normalise_fp32(r[(1, 1, 1)], True).double())
            r[(3, 0, 1)] = (x @ f16(sd[pre + '.0.weight'].double()).T + b).clamp_min(0)
        flagged(chunk_bias, 'tc_hidden', 'value 0 part 1')

    def next_action(r, o):            # row 2 takes the action column of a + 1
        w = sd[PREFIX[1] + '.0.weight'].double()
        q = f16 if tc else (lambda x: x)
        a = (int(action[2]) + 1) % A
        r[(1, 0, 0)][2] = (q(slots[2]) @ q(w[:, :64]).T + sd[PREFIX[1] + '.0.bias'].double() + w[:, 64 + a]).clamp_min(0)
    flagged(next_action, lin0, 'transition 0 part 0')

    def min_max_63(r, o):             # normalised over 63 of the 64 columns
        raw = r[(1, 1, 0)].float()
        mn, mx = raw[:, :63].amin(1, keepdim=True), raw[:, :63].amax(1, keepdim=True)
        den = (mx - mn) + torch.tensor(1e-8, dtype=torch.float32)
        nm = (raw - mn) * (1.0 / den) if tc else (raw - mn) / den
        if not tc:
            r[(1, 2, 0)] = nm.double()
        return nm
    flagged(min_max_63, 'hidden_out_bits', 'hidden_out')

    def reward_normalised(r, o):      # the reward net reads the normalised state
        pre = PREFIX[2]
        q = f16 if tc else (lambda x: x)
        x = normalise_fp32(r[(1, 1, 0)], tc).double()
        r[(2, 0, 0)] = (q(x) @ q(sd[pre + '.0.weight'].double()).T + sd[pre + '.0.bias'].double()).clamp_min(0)
    flagged(reward_normalised, lin0, 'reward 0 part 0')

    def padded_policy(r, o):          # a padded (zero) policy column in the softmax
        lg = r[(4, 1, 1 if tc else 0)]
        o['pi'] = torch.softmax(torch.cat([lg, torch.zeros_like(lg[:, :1])], 1), 1)[:, :A]
    flagged(padded_policy, 'head_pi', 'pi')

    if not tc:
        def k_tail(r, o):             # transition second layer: K = 50, the tail term k = 49 of one element dropped
            M = r[(1, 0, 0)]
            w = sd[PREFIX[1] + '.2.weight'].double()
            t = M[:, 49:50] * w[:, 49].view(1, -1)
            i, j = divmod(int(t.abs().argmax()), t.shape[1])
            r[(1, 1, 0)][i, j] -= t[i, j]
        flagged(k_tail, 'simt_linear', 'transition 1 part 0')


# ---- the engine (GPU) -----------------------------------------------------------------------------------------------
def launch_forms(L):
    f = set()
    if L['tile_rows'] == 32:
        f.add('simt_recurrent' if L['sub'] else 'simt_initial')
        return f
    if L['pair'] == 2:
        f.add('tc_split_policy' if L['n'] else 'tc_split_no_policy')
    elif L['num_tiles'] > L['grid']:
        f.add('tc_multi_tile')
    else:
        f.add('tc_one_cta')
    f.add({1: 'one_chunk', 2: 'two_chunks'}[L['multi_pass']])
    f.add('tab_smem' if L['resident'] else 'tab_global')
    if L['n'] and L['w'] > 32:
        f.add('policy_wide')
    return f


# name: (checkpoint or None, input shape, actions, planes, support, hidden, batch, environment, forms it must show,
#        forms it must not show)
TC_ALL = {'tc_split_policy', 'tc_split_no_policy', 'tc_one_cta', 'tc_multi_tile'}
CASES = {
    'tictactoe_4096_split': ('tictactoe', (9, 3, 3), 10, 256, 1, 64, 4096, {},
                             {'tc_split_policy', 'tc_split_no_policy', 'one_chunk', 'tab_smem'}, set()),
    'tictactoe_1_split': ('tictactoe', (9, 3, 3), 10, 256, 1, 64, 1, {}, {'tc_split_policy', 'tc_split_no_policy'},
                          set()),
    'cartpole_129_split': ('cartpole', (4, 5), 2, 512, 31, 64, 129, {},
                           {'tc_split_policy', 'tc_split_no_policy', 'two_chunks'}, set()),
    'cartpole_16384_one_cta': ('cartpole', (4, 5), 2, 512, 31, 64, 16384, {}, {'tc_one_cta', 'two_chunks'},
                               {'tc_split_policy', 'tc_multi_tile'}),
    'tictactoe_10000_one_cta': ('tictactoe', (9, 3, 3), 10, 256, 1, 64, 10000, {}, {'tc_one_cta', 'one_chunk'},
                                {'tc_split_policy', 'tc_multi_tile'}),
    'cartpole_40000_multi_tile': ('cartpole', (4, 5), 2, 512, 31, 64, 40000, {}, {'tc_multi_tile'}, set()),
    'p512_a10_global_table': (None, (4, 5), 10, 512, 31, 64, 300, {}, {'tab_global', 'two_chunks'}, {'tab_smem'}),
    'p256_a20_global_table': (None, (4, 5), 20, 256, 31, 64, 300, {}, {'tab_global', 'one_chunk'}, {'tab_smem'}),
    'p256_a40_policy_wide': (None, (4, 5), 40, 256, 31, 64, 300, {}, {'policy_wide'}, set()),
    'p256_a64_policy_wide': (None, (4, 5), 64, 256, 31, 64, 300, {}, {'policy_wide'}, set()),
    'p256_a65_policy_simt': (None, (4, 5), 65, 256, 31, 64, 300, {}, {'simt_recurrent', 'tc_split_no_policy'},
                             {'tc_split_policy'}),
    'p256_a1': (None, (4, 5), 1, 256, 31, 64, 300, {}, {'tc_split_policy'}, set()),
    'support32_tc': (None, (4, 5), 4, 256, 32, 64, 300, {}, {'tc_split_policy'}, set()),
    'support33_simt': (None, (4, 5), 4, 256, 33, 64, 300, {}, {'simt_recurrent'}, TC_ALL),
    'support601_simt': (None, (4, 5), 4, 256, 601, 64, 100, {}, {'simt_recurrent'}, TC_ALL),
    'hidden32_simt': (None, (4, 5), 4, 256, 31, 32, 100, {}, {'simt_recurrent'}, TC_ALL),
    'hidden128_simt': (None, (4, 5), 4, 256, 31, 128, 100, {}, {'simt_recurrent'}, TC_ALL),
    'p100_simt': (None, (4, 5), 4, 100, 31, 64, 100, {}, {'simt_recurrent'}, TC_ALL),
    'p50_simt': (None, (4, 5), 4, 50, 31, 64, 100, {}, {'simt_recurrent'}, TC_ALL),
    'odd_input_3x7': (None, (3, 7), 4, 256, 31, 64, 100, {}, {'simt_initial', 'tc_split_policy'}, set()),
    'tictactoe_forced_simt': ('tictactoe', (9, 3, 3), 10, 256, 1, 64, 300, {'MZ_MLP_SIMT': '1'}, {'simt_recurrent'},
                              TC_ALL),
    'p768_simt': (None, (4, 5), 4, 768, 1, 64, 100, {}, {'simt_recurrent'}, TC_ALL),
    'p1024_simt': (None, (4, 5), 4, 1024, 1, 64, 100, {}, {'simt_recurrent'}, TC_ALL),
    'p1536_simt': (None, (4, 5), 4, 1536, 1, 64, 100, {}, {'simt_recurrent'}, TC_ALL),
    'gather_edge': (None, (4, 5), 10, 256, 31, 64, 300, {}, {'tc_split_policy'}, set()),
}


def _sample(batch, seed):
    s = {0, batch - 1}
    for k in range(128, batch, 128):
        s.update((k - 1, k))
    s.update(np.random.RandomState(seed).choice(batch, min(batch, 8), replace=False).tolist())
    return torch.tensor(sorted(s))


def _make_net(ckpt, shape, A, P, S, HD):
    import muzero_b200 as mz
    from conftest import GOLDEN
    torch.manual_seed(P * 1000 + A * 10 + S + HD)
    net = mz.MuZeroMLPNet(shape, A, P, S, S, HD)
    if ckpt:
        net.load_state_dict({k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, f'ckpt_{ckpt}.npz')).items()})
    return net.cuda().eval()


def run_case(name, monkeypatch):
    from muzero_b200 import _lib
    ckpt, shape, A, P, S, HD, batch, env, forms, not_forms = CASES[name]
    for k in ('MZ_MLP_SIMT',):
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    net = _make_net(ckpt, shape, A, P, S, HD)
    sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
    cfg = dict(HD=HD, P=P, A=A, vkind=int(S > 1), rkind=int(S > 1))
    e = net.engine(batch)
    lib, h = _lib.lib(), e['handle']
    gen = torch.Generator(device='cuda').manual_seed(13)
    obs = torch.randn((batch,) + shape, device='cuda', generator=gen)
    nslots = 2 * batch + 3
    dst0 = torch.randperm(nslots, device='cuda', generator=gen)[:batch].int()
    src1 = dst0[torch.randperm(batch, device='cuda', generator=gen)]
    dst1 = torch.randperm(nslots, device='cuda', generator=gen)[:batch].int()
    act = torch.randint(0, A, (batch,), device='cuda', generator=gen).int()
    fill = (torch.rand((nslots, HD), device='cuda', generator=gen) * 2 - 1).contiguous().view(torch.uint8)
    edge = None
    if name == 'gather_edge':          # parent states outside [0, 1] and beyond the fp16 range (clamped to +-65504)
        ev = torch.randn((nslots, HD), device='cuda', generator=gen) * 3.0
        ev[::3] *= 4e4
        ev[1::7, ::5] = 1e6
        ev[2::7, 1::5] = -1e6
        edge = ev.contiguous().view(torch.uint8)

    def calls():
        h0 = fill.clone()
        _, pi0, v0 = net.initial_inference_batch(obs, hidden_out=h0, dst_index=dst0)
        r0 = record()
        hin = h0 if edge is None else edge
        h1 = fill.clone()
        _, r1, pi1, v1 = net.recurrent_inference_batch(hin, act, src_index=src1, hidden_out=h1, dst_index=dst1)
        rec1 = record()
        h2 = fill.clone()
        _, r2, _, v2 = net.recurrent_inference_batch(hin, act, src_index=src1, hidden_out=h2, dst_index=dst1,
                                                     want_policy=False)
        rec2 = record()
        torch.cuda.synchronize()
        return (h0, pi0, v0, h1, r1, pi1, v1, h2, r2, v2), (r0, rec1, rec2)

    buf = None
    rows = _sample(batch, 14)
    rows_d = rows.cuda()

    def record():
        if buf is None:
            return None
        n = C.c_int32()
        _lib.check(lib.mz_net_debug_tensor(h, -1, None, C.byref(n)))
        tens = []
        for i in range(n.value):
            t = _lib.DebugTensor()
            _lib.check(lib.mz_net_debug_tensor(h, i, C.byref(t), C.byref(n)))
            assert t.kind == _lib.MZ_DEBUG_MLP
            off = t.ptr - buf.data_ptr()
            raw = buf[off:off + t.plane_rows * t.h * t.w].view(torch.float16 if t.w == 2 else torch.float32)
            data = raw.view(t.plane_rows, t.h)[:, :t.groups][rows_d].double().cpu()
            tens.append(dict(net=t.stage, layer=t.index, part=t.batch, src=t.src, data=data))
        _lib.check(lib.mz_net_debug_launch(h, -1, None, C.byref(n)))
        launches = []
        for i in range(n.value):
            L = _lib.DebugLaunch()
            _lib.check(lib.mz_net_debug_launch(h, i, C.byref(L), C.byref(n)))
            launches.append({k: getattr(L, k) for k in ('tile_rows', 'pair', 'grid', 'num_tiles', 'multi_pass', 'n',
                                                          'resident', 'sub', 'num_layers', 'h', 'w', 'batch')})
        return tens, launches

    off, _ = calls()
    nb = C.c_size_t()
    _lib.check(lib.mz_net_debug_capture_bytes(h, batch, C.byref(nb)))
    buf = torch.empty(nb.value + 256, dtype=torch.uint8, device='cuda')
    base = (buf.data_ptr() + 255) // 256 * 256
    _lib.check(lib.mz_net_debug_capture(h, base, nb.value))
    try:
        on, recs = calls()
    finally:
        _lib.check(lib.mz_net_debug_capture(h, None, 0))
    bad, worst, seen = [], {}, set()
    for k, (a, b) in enumerate(zip(off, on)):
        if not torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8)):
            bad.append(f'output {k} differs between capture off and on')
    h0, pi0, v0, h1, r1, pi1, v1, h2, r2, v2 = on
    hin = h0 if edge is None else edge
    calls_out = ((0, dict(pi=pi0, value=v0), h0, dst0), (1, dict(pi=pi1, value=v1, reward=r1), h1, dst1),
                 (2, dict(value=v2, reward=r2), h2, dst1))
    for (call, out, hs, di), (tens, launches) in zip(calls_out, recs):
        assert len(launches) == 1, launches
        L = launches[0]
        seen |= launch_forms(L)
        tc = L['tile_rows'] == 128
        nsplit = L['pair']
        if L['batch'] != batch or L['h'] != P or L['w'] != A or L['sub'] != (call > 0) or L['n'] != ('pi' in out):
            bad.append(f'call {call}: launch record {L}')
        recd = {(t['net'], t['layer'], t['part']): t['data'] for t in tens}
        key = [(t['net'], t['layer'], t['part']) for t in tens]
        want = structure(recd, tc, nsplit, call > 0, 'pi' in out)
        if set(key) != set(want) or len(key) != len(set(key)):
            bad.append(f'call {call}: recorded tensors {sorted(key)}, structure says {sorted(want)}')
            continue
        for t in tens:
            k = (t['net'], t['layer'], t['part'])
            got = None if t['src'] < 0 else key[t['src']]
            if got != want[k]:
                bad.append(f'call {call}: {k} reads {got}, structure says {want[k]}')
        if call == 0:
            x_in, a = obs.reshape(batch, -1)[rows_d].double().cpu(), None
        else:
            x_in = hin.view(torch.float32).view(-1, HD)[src1[rows_d].long()].double().cpu()
            a = act[rows_d].long().cpu()
        hidden = hs.view(torch.float32).view(-1, HD)[di[rows_d].long()].cpu()
        outs = {k: v[rows_d].double().cpu() for k, v in out.items()}
        w = check_call(sd, cfg, recd, tc, nsplit, x_in, a, outs, hidden)
        for k, (v, where) in w.items():
            if k not in worst or not v <= worst[k][0]:
                worst[k] = (v, f'call {call} {where}')
            if not v <= 1.0:
                bad.append(f'call {call} {where}: {k} {v:.4g} > 1')
        keep = torch.ones(nslots, dtype=torch.bool, device='cuda')
        keep[di.long()] = False
        if not torch.equal(hs.view(nslots, -1)[keep], fill.view(nslots, -1)[keep]):
            bad.append(f'call {call}: a slot not named by dst_index changed')
    missing = forms - seen
    extra = not_forms & seen
    if extra:
        bad.append(f'forms {sorted(extra)} ran, which this case must not run')
    if missing:
        bad.append(f'forms {sorted(missing)} not run (ran {sorted(seen)})')
    net.release_engine()
    del net, buf
    torch.cuda.empty_cache()
    return worst, bad, seen


_SEEN = {}


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(CASES))
def test_every_layer_against_float64_on_the_engines_own_tensors(case, monkeypatch):
    worst, bad, seen = run_case(case, monkeypatch)
    _SEEN[case] = seen
    print(f'\n{case}: forms {sorted(seen)}; ' + ', '.join(f'{k} {v:.3g} ({w})' for k, (v, w) in worst.items()))
    assert not bad, '\n'.join(bad[:40])


@pytest.mark.gpu
def test_cases_cover_every_form(monkeypatch):
    """Together the cases run every form of the engine (the host's heuristics may move a case to another form, but no
    form drops out of the suite unnoticed)."""
    seen = set()
    for case in CASES:
        s = _SEEN.get(case)
        if s is None:
            s = run_case(case, monkeypatch)[2]
        seen |= s
    assert seen >= set(FORMS), sorted(set(FORMS) - seen)


@pytest.mark.gpu
def test_too_wide_net_is_refused_cleanly():
    """num_planes = 2048 fits neither kernel (the tcgen05 kernel's weight-block table, the SIMT kernel's shared memory):
    mz_net_create fails with MZ_EINVAL and says why."""
    import muzero_b200 as mz
    net = mz.MuZeroMLPNet((4, 5), 4, 2048, 1, 1, 64).cuda().eval()
    with pytest.raises(ValueError, match='too wide'):
        net.engine(8)
