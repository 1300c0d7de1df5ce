"""Layer-by-layer tests of the inference conv engine (csrc/conv.cu): every conv, pool, normalisation and head of an
initial and a recurrent inference against a float64 computation fed the engine's OWN stored tensors
(``mz_net_debug_capture``: with capture on, every conv / pool output of a call keeps a region of its own, and every
conv3x3_kernel launch is recorded with the form the host chose for it).

Comparing whole towers with the fp32 oracle (tests/test_conv_gpu.py) has to be loose, since errors compound through
up to 49 layers; here each layer gets the engine's own input, so the ReLU decisions are the engine's and what is left
is rounding.  u = 2^-24 (fp32), ulp16(r) the fp16 spacing at |r| (2^-24 below 2^-14).

* Weights: bn_fold_kernel is restated in fp32 torch (correctly rounded sqrt and division, as the build has no
  --use_fast_math): s = g / sqrt(var + 1e-5), W16 = fp16(clamp(fp32(w * s))) -- the exact packed operand.  The bias
  beta - mean * s may be contracted to an FMA, so it enters the bound as |beta| + |mean * s| rather than by its bits.
  The Atari stride-2 convs use s = 1 and no bias.
* Conv layer (every 128-column pass, every form): R = conv3x3_f64(X, W16) + b [+ T[action]] [+ residual],
  ref = clamp(R, 0, 65504), and every stored element A satisfies
      |A - ref| <= ulp16(ref) + 2^-16 (conv3x3_f64(|X|, |W16|) + |beta| + |mean s| + |T| + |residual|) + e_T.
  The products fp16 x fp16 are exact in fp32.  A layer with Cin (padded) input channels runs 9 Cin / 16 MMAs of K = 16
  into an fp32 TMEM accumulator, at most 144 (Cin = 256); taking one round-to-nearest per MMA step, each step errs by
  at most u times its partial sum, and every partial sum is bounded by the magnitude sum M = conv3x3_f64(|X|, |W16|).
  The epilogue adds at most four more fp32 terms (the split-K half, bias, table, residual), each rounding once, so the
  fp32 value is within (144 + 4) u (M + |bias| + |T| + |residual|) < 2^-16 (...) = 256 u (...), and the conversion
  to fp16 adds half an ulp16(ref), inside the ulp16(ref) term.  (A truncating accumulator would double the per-step
  term, to 296 u at Cin = 256; the 256-plane cases measure the same 0.49 of the bound as the others.)  T is the dynamics' action table: in float64 from the
  QUIRK C planes (a comb, not constant planes), and action_table_kernel sums its m non-zero terms in fp32 and then
  scales, so e_T = u (m + 1) s conv3x3_f64(E_a, |w_action|).  Stride-2 convs store the even positions of the stride-1
  result.  Taps across a board edge are zero padding, so a board's outputs depend on that board alone and large
  batches are checked on a sample: the first and last boards, every board that straddles a 128-row boundary (hence
  every 256-row one too) and 8 random ones.
* Padding: channels >= num_planes (16-plane nets) are +0 in every stored tensor and slot; slots not named by
  dst_index keep their bytes.
* Normalised outputs (min-max over the num_planes real channels of a position, util.py:31-36), D = max - min + 1e-8
  over the captured raw row: the fused epilogue normalises the fp32 value v before rounding it, and the stored raw
  row is fp16(v), so v, min and max each differ from the captured values by at most ulp16(max|A|) / 2; the
  numerator (v - min) moves by at most ulp16(max|A|) and the denominator by as much, which moves the quotient (<= 1)
  by at most another ulp16(max|A|) / D.  Bound: ulp16(ref) + 2 ulp16(max|A|) / D + 2^-20 (the fp32 subtraction,
  reciprocal and product).  normalise_rows_kernel (256-plane towers) reads the stored row itself: same bound.  The
  normalised copy the prediction tower reads and every slot the call writes hold the same bits.
* Pools, AvgPool2d(3, 2, 1) with count_include_pad: an fp32 sum of <= 9 fp16 values times fp32(1/9):
  ref = avg_pool2d_f64(X), bound ulp16(ref) + 2^-20 avg_pool2d_f64(|X|).  The second pool also normalises, from its
  fp32 (unrounded) averages: bound ulp16(ref) + 2^-18 max|P| / D + 2^-20, P the float64 averages of the position.
* Heads (1x1 conv with the folded fp32 weights, ReLU, Linear, output transform) on the captured tower output F:
  the 1x1 conv is a sequential fp32 FMA chain over C channels, so |dh| <= (C + 2) u (sum|F w1| + |beta1| + |mean1 s1|);
  ReLU does not grow it; the Linear runs K = mid h w terms as 32 lane chains of ceil(K/32) FMAs and a 5-level
  butterfly, so |dlogit| <= (ceil(K/32) + 7) u (sum|f w2| + |b2|) + sum|w2| |dh|.  That logit bound e is carried
  through the float64 Jacobian J of the output transform (autograd): |dy| <= |J| e, plus for softmax
  p u (16 + out/32 + 2 max|l - m|) (expf within 2 ulp, the shift l - m, the lane sums, the division) + 2^-148
  (probabilities below 2^-126 are fp32 subnormals, whose spacing is 2^-149 whatever their size) and for
  support -> scalar the same relative error on the expectation x times |sp'(x)|, plus the fp32 evaluation of
  signed_parabolic: with a = 1 + 0.004 (1.001 + |x|) and z = sqrt(a) / 2 / 0.001 - 500, dz = 500 sqrt(a) 4u + ulp32(z)
  and |dy| gains 2 |z| dz + 2 ulp32(z^2) (z^2 - 1 cancels near x = 0, where this term dominates).
* Capture off vs on: every case runs both ways and the hidden slots, pi, value and reward are the same bytes -- with
  capture off a residual block writes its output over its input, so a race between that store and a late reader of
  the old contents would show here.
* Forms: each case asserts, from the launch record, the form it is named for, and
  ``test_cases_cover_every_form`` asserts that together they reach every form of the engine.

``test_reference_flags_planted_errors`` checks the reference itself on the CPU.
Measured worst error / bound over all cases (NVIDIA B200, 1000 W power limit): conv 0.49, normalisation 0.49,
pool 0.50, normalising pool 0.50, policy head 0.30, value head 0.020, reward head 0.015; padding channels all +0."""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

U32 = 2.0 ** -24
FORMS = ('single', 'sub', 'dataflow256', 'pair', 'pair_null_tile', 'splitk128', 'resident128', 'resident256',
         'khalf', 'multi_pass', 'split_in_block', 'n32')


# ---- the float64 reference (device-agnostic) --------------------------------------------------------------------
def ulp16(r):
    return torch.exp2(torch.floor(torch.log2(r.abs().clamp_min(2.0 ** -14))) - 10)


def ulp32(r):
    return torch.exp2(torch.floor(torch.log2(r.abs().clamp_min(2.0 ** -126))) - 23)


def conv3x3(x, w, stride=1):
    y = F.conv2d(x, w, padding=1)
    return y[:, :, ::2, ::2] if stride == 2 else y


def fold(sd, conv, bn, cin=None, dev='cpu'):
    """(W16 float64, bias float64, |beta| + |mean s| float64, s float64) of conv + eval BatchNorm as bn_fold_kernel and
    pack_conv_kernel make them; bn None: scale 1, no bias."""
    w = sd[conv + '.weight'].float().to(dev)
    if cin is not None:
        w = w[:, :cin]
    if bn is None:
        s = torch.ones(w.shape[0], device=dev)
        b = babs = torch.zeros(w.shape[0], dtype=torch.float64, device=dev)
    else:
        g, beta, mean, var = (sd[f'{bn}.{k}'].float().to(dev) for k in ('weight', 'bias', 'running_mean', 'running_var'))
        s = g / torch.sqrt(var + 1e-5)
        b = (beta - mean * s).double()
        babs = beta.double().abs() + (mean.double() * s.double()).abs()
    w16 = (w * s.view(-1, *([1] * (w.dim() - 1)))).clamp(-65504.0, 65504.0).half().double()
    return w16, b, babs, s.double()


def comb_planes(action, A, h, w):
    """QUIRK C (network.py:440-444): flat element f of the [A*h*w] block is 1 iff f % A == action."""
    b = action.shape[0]
    planes = F.one_hot(action.reshape(b, 1).long(), A).double()
    return torch.repeat_interleave(planes, repeats=h * w, dim=1).reshape(b, A, h, w)


def conv_ratio(A, X, w16, b, babs, stride=1, res=None, tab=None, tab_err=None):
    """max error / bound of one conv layer (module docstring).  A, X, res, tab: float64 [B, C, H, W]."""
    R = conv3x3(X, w16, stride) + b.view(1, -1, 1, 1)
    mag = conv3x3(X.abs(), w16.abs(), stride) + babs.view(1, -1, 1, 1)
    extra = 0.0
    if tab is not None:
        R, mag, extra = R + tab, mag + tab.abs(), tab_err
    if res is not None:
        R, mag = R + res, mag + res.abs()
    ref = R.clamp(0.0, 65504.0)
    return float(((A - ref).abs() / (ulp16(ref) + 2.0 ** -16 * mag + extra)).max())


def normalise_ratio(Nm, raw, n_real, pool_scale=False):
    """Normalised tensor Nm against min-max over the first n_real channels of raw (float64 [B, C, H, W])."""
    r = raw[:, :n_real]
    lo, hi = r.amin(1, keepdim=True), r.amax(1, keepdim=True)
    D = hi - lo + 1e-8
    ref = (r - lo) / D
    top = r.abs().amax(1, keepdim=True)
    slack = (2.0 ** -18 * top if pool_scale else 2.0 * ulp16(top)) / D + 2.0 ** -20
    return float(((Nm[:, :n_real] - ref).abs() / (ulp16(ref) + slack)).max())


def pool_ratio(P, X):
    ref = F.avg_pool2d(X, 3, 2, 1)
    return float(((P - ref).abs() / (ulp16(ref) + 2.0 ** -20 * F.avg_pool2d(X.abs(), 3, 2, 1))).max())


def _nonzero(pad):
    """Padding channels must be +0: 0 if they are, else infinity (as a ratio)."""
    return 0.0 if pad.numel() == 0 or bool((pad == 0).all() and not torch.signbit(pad).any()) else math.inf


def signed_parabolic(x, eps=1e-3):
    z = torch.sqrt(1 + 4 * eps * (eps + 1 + torch.abs(x))) / 2 / eps - 1 / 2 / eps
    return torch.sign(x) * (torch.square(z) - 1)


def head_ratio(Y, Fm, sd, prefix, kind, n_real):
    """Y: the engine's head output (float64 [B] or [B, out]); Fm: the captured tower output (float64 [B, C, H, W])."""
    dev = Fm.device
    w1, b1, b1abs, _ = fold(sd, prefix + '.0', prefix + '.1', dev=dev)
    w1 = (sd[prefix + '.0.weight'].float().to(dev)[:, :, 0, 0] *
          (sd[prefix + '.1.weight'].float().to(dev) / torch.sqrt(sd[prefix + '.1.running_var'].float().to(dev) + 1e-5))
          .view(-1, 1)).double()                                   # scale_rows_kernel: fp32 w * s, kept in fp32
    x = Fm[:, :n_real]
    B, Cn, H, W = x.shape
    h = torch.einsum('bchw,mc->bmhw', x, w1) + b1.view(1, -1, 1, 1)
    dh = (Cn + 2) * U32 * (torch.einsum('bchw,mc->bmhw', x.abs(), w1.abs()) + b1abs.view(1, -1, 1, 1))
    f, df = h.clamp_min(0.0).flatten(1), dh.flatten(1)
    w2 = sd[prefix + '.4.weight'].double().to(dev)
    b2 = sd[prefix + '.4.bias'].double().to(dev)
    K = f.shape[1]
    logit = f @ w2.T + b2
    e = (math.ceil(K / 32) + 7) * U32 * (f.abs() @ w2.abs().T + b2.abs()) + df @ w2.abs().T
    return transform_ratio(Y, logit, e, kind)


def safe_ratio(err, bound):
    """max err / bound, where a zero bound admits only a zero error."""
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, math.inf, 0.0))
    return float(r.max()) if r.numel() else 0.0


def transform_ratio(Y, logit, e, kind, seq=False):
    """Y: the engine's output (float64 [B] or [B, out]) of the output transform `kind` (0 identity, 1 support ->
    scalar, 2 softmax) of fp32 logits known to within e (float64 [B, n], like logit).  seq: one thread sums the n
    terms in order; else 32 lanes sum n / 32 each and a butterfly combines them (module docstring)."""
    if kind == 0:
        return safe_ratio((Y.view(-1) - logit.view(-1)).abs(), e.view(-1))
    dev = logit.device
    n = logit.shape[1]
    lg = logit.detach().requires_grad_(True)
    if kind == 2:
        out = torch.softmax(lg, 1)
    else:
        hi = (n - 1) // 2
        p = torch.softmax(lg, 1)
        xs = (p * torch.linspace(-hi, hi, n, dtype=torch.float64, device=dev)).sum(1)
        out = signed_parabolic(xs)
    Jabs = torch.stack([torch.autograd.grad(out[:, j].sum() if kind == 2 else out.sum(), lg, retain_graph=True)[0].abs()
                        for j in range(n if kind == 2 else 1)], 1)          # [B, outputs, logits]
    bound = (Jabs * e.unsqueeze(1)).sum(2)
    spread = (logit - logit.amax(1, keepdim=True)).abs().amax(1, keepdim=True)
    rel = U32 * (16 + (2 * n if seq else n / 32) + 2 * spread)
    out = out.detach()
    if kind == 2:
        bound = bound + out * rel + 2.0 ** -148        # expf and the division round into fp32 subnormals (2^-149)
    else:
        p = torch.softmax(logit, 1)
        sup = torch.linspace(-hi, hi, n, dtype=torch.float64, device=dev)
        xs = (p * sup).sum(1)
        dx = rel.view(-1) * (p * sup.abs()).sum(1) + ulp32(xs)
        if n % 2 == 0:            # support points -maxv + i * fp32(2 maxv / (n - 1)) are not integers
            dx = dx + 4 * U32 * (hi + 1)
        a = 1 + 0.004 * (1.001 + xs.abs())
        z = a.sqrt() / 2 / 1e-3 - 500
        dsp = 2 * z.abs() * 0.004 / 2 / 1e-3 / 2 / a.sqrt()          # |d signed_parabolic / dx|
        dz = 500 * a.sqrt() * 4 * U32 + ulp32(z)
        bound = bound.view(-1) + dsp * dx + 2 * z.abs() * dz + 2 * ulp32(z * z)
        out = out.view(-1)
    return float(((Y.reshape(out.shape) - out).abs() / bound.reshape(out.shape)).max())


# ---- the structure of a net: which weights each stored tensor is made with ------------------------------------------
def conv_names(kind, stage, index, blocks):
    """(conv prefix, BatchNorm prefix or None, stride, residual: whether the block input is added) of conv `index` of
    `stage`."""
    def blk(p, j):
        i, second = divmod(j, 2)
        return f'{p}.{i}.conv_block{2 if second else 1}.0', f'{p}.{i}.conv_block{2 if second else 1}.1', 1, bool(second)
    if stage == 2:
        return blk('prediction_net.res_blocks', index)
    if stage == 1:
        return ('dynamics_net.conv_block.0', 'dynamics_net.conv_block.1', 1, False) if index == 0 else \
            blk('dynamics_net.res_blocks', index - 1)
    if kind == 'board':
        return ('represent_net.conv_block.0', 'represent_net.conv_block.1', 1, False) if index == 0 else \
            blk('represent_net.res_blocks', index - 1)
    if index == 0:
        return 'represent_net.conv_1', None, 2, False
    if index == 5:
        return 'represent_net.conv_2', None, 2, False
    j = index - 1 if index < 5 else index - 6
    return blk(f'represent_net.res_blocks_{1 + j // 4 if index < 5 else 2 + j // 4}', j % 4)


def wiring(kind, tensors):
    """{tensor index: (input tensor index or 'slots', residual tensor index or None)} derived from the network's
    structure (not from the record), for every conv / pool / normalised tensor of a call.  tensors: list of dicts."""
    at = {(t['kind'], t['stage'], t['index']): i for i, t in enumerate(tensors)}
    conv = lambda s, j: at[('conv', s, j)]
    out = {}
    for i, t in enumerate(tensors):
        s, j = t['stage'], t['index']
        if t['kind'] == 'conv':
            if j == 0:
                src = at[('obs', 0, 0)] if s == 0 else ('slots' if s == 1 else
                                                         at.get(('norm', 0, 0), at.get(('norm', 1, 0), at.get(('pool', 0, 1)))))
            elif kind == 'atari' and s == 0 and j == 10:
                src = at[('pool', 0, 0)]
            else:
                src = conv(s, j - 1)
            _, _, _, has_res = conv_names(kind, s, j, 0)
            res = None
            if has_res:
                res = out[conv(s, j - 1)][0]
            out[i] = (src, res)
        elif t['kind'] == 'pool':
            out[i] = (conv(0, 9 if j == 0 else 13), None)
        elif t['kind'] == 'norm':
            last = max(jj for (k, ss, jj) in at if k == 'conv' and ss == s)
            out[i] = (conv(s, last), None)
    return out


def check_call(kind, sd, cfg, tensors, slots_in=None, action=None, outputs=None, heads_from=None, per=None):
    """Every check of one recorded call.  tensors: list of dicts (kind, stage, index, data float64 [B, C, H, W]);
    slots_in: float64 [B, C, H, W] dynamics input; outputs: {'pi', 'value', 'reward'} float64.  Returns
    {check: (worst ratio, where)}; per, if given, receives {(check, where): ratio}."""
    n_real, blocks = cfg['planes'], cfg['blocks']
    worst = {}

    def note(check, v, where):
        if per is not None:
            per[(check, where)] = max(v, per.get((check, where), 0.0))
        if check not in worst or not v <= worst[check][0]:
            worst[check] = (v, where)
    wire = wiring(kind, tensors)
    get = lambda k: slots_in if k == 'slots' else tensors[k]['data']
    for i, t in enumerate(tensors):
        where = f"{t['kind']} {t['stage']}.{t['index']}"
        if t['kind'] == 'conv':
            src, res = wire[i]
            X = get(src)
            cp, bp, stride, _ = conv_names(kind, t['stage'], t['index'], blocks)
            w16, b, babs, s = fold(sd, cp, bp, dev=X.device)
            c_real = w16.shape[1] if t['stage'] != 1 or t['index'] != 0 else n_real
            tab = tab_err = None
            if t['stage'] == 1 and t['index'] == 0:
                wa = sd[cp + '.weight'].double().to(X.device)[:, n_real:]
                E = comb_planes(action, cfg['actions'], X.shape[2], X.shape[3]).to(X.device)
                sc = s.view(1, -1, 1, 1)
                tab = conv3x3(E, wa) * sc
                m = conv3x3(E, torch.ones_like(wa[:1]))
                tab_err = U32 * (m + 1) * conv3x3(E, wa.abs()) * sc.abs()
                w16 = w16[:, :n_real]
            Xr = X[:, :c_real]
            n_out = w16.shape[0]
            A = t['data']
            note('conv', conv_ratio(A[:, :n_out], Xr, w16, b, babs, stride, None if res is None else get(res)[:, :n_out],
                                    tab, tab_err), where)
            note('padding', _nonzero(A[:, n_out:]), where)
        elif t['kind'] == 'pool':
            X = get(wire[i][0])
            if t['index'] == 0:
                note('pool', pool_ratio(t['data'], X), where)
            else:
                note('pool_norm', normalise_ratio(t['data'], F.avg_pool2d(X, 3, 2, 1), n_real, pool_scale=True), where)
        elif t['kind'] == 'norm':
            note('norm', normalise_ratio(t['data'], get(wire[i][0]), n_real), where)
            note('padding', _nonzero(t['data'][:, n_real:]), where)
    if outputs:
        pred_last = [i for i, t in enumerate(tensors) if t['kind'] == 'conv' and t['stage'] == 2]
        fin = tensors[pred_last[-1]]['data'] if pred_last else heads_from
        if 'pi' in outputs:
            note('head_policy', head_ratio(outputs['pi'], fin, sd, 'prediction_net.policy_net', 2, n_real), 'policy')
        note('head_value', head_ratio(outputs['value'], fin, sd, 'prediction_net.value_net', cfg['vkind'], n_real), 'value')
        if 'reward' in outputs:
            dyn_last = max((i for i, t in enumerate(tensors) if t['kind'] == 'conv' and t['stage'] == 1),
                           key=lambda i: tensors[i]['index'])
            note('head_reward', head_ratio(outputs['reward'], tensors[dyn_last]['data'], sd, 'dynamics_net.reward_head',
                                           cfg['rkind'], n_real), 'reward')
    return worst


# ---- the reference checked on the CPU against float64 runs of the oracle ---------------------------------------------
def _oracle_record(kind, onet, sd, cfg, obs=None, slots=None, action=None):
    """The tensors an engine call would record, from an eager float64 run of OracleNet's building blocks, with the
    conv weights set so that the fold is exact (w = W16 / s)."""
    tens = []
    add = lambda k, s, j, d: tens.append(dict(kind=k, stage=s, index=j, data=d))

    def cbr(p, x, stride=1, bn=True):
        y = onet._conv(p + ('.0' if bn else ''), x, stride, 1)
        return F.relu(onet._bn(p + '.1', y)) if bn else F.relu(y)

    def blocks(p, x, stage, j0, n):
        for i in range(n):
            o = F.relu(onet._bn(f'{p}.{i}.conv_block1.1', onet._conv(f'{p}.{i}.conv_block1.0', x)))
            add('conv', stage, j0 + 2 * i, o)
            x = F.relu(onet._bn(f'{p}.{i}.conv_block2.1', onet._conv(f'{p}.{i}.conv_block2.0', o)) + x)
            add('conv', stage, j0 + 2 * i + 1, x)
        return x
    if obs is not None:
        add('obs', 0, 0, obs)
        if kind == 'board':
            h = cbr('represent_net.conv_block', obs)
            add('conv', 0, 0, h)
            h = blocks('represent_net.res_blocks', h, 0, 1, cfg['blocks'])
            hn = onet_norm(h)
            add('norm', 0, 0, hn)
        else:
            h = cbr('represent_net.conv_1', obs, 2, False)
            add('conv', 0, 0, h)
            h = blocks('represent_net.res_blocks_1', h, 0, 1, 2)
            h = cbr('represent_net.conv_2', h, 2, False)
            add('conv', 0, 5, h)
            h = blocks('represent_net.res_blocks_2', h, 0, 6, 2)
            h = F.avg_pool2d(h, 3, 2, 1)
            add('pool', 0, 0, h)
            h = blocks('represent_net.res_blocks_3', h, 0, 10, 2)
            hn = onet_norm(F.avg_pool2d(h, 3, 2, 1))
            add('pool', 0, 1, hn)
    else:
        b = slots.shape[0]
        hh, ww = slots.shape[2], slots.shape[3]
        x = torch.cat([slots, comb_planes(action, cfg['actions'], hh, ww)], 1)
        h = cbr('dynamics_net.conv_block', x)
        add('conv', 1, 0, h)
        h = blocks('dynamics_net.res_blocks', h, 1, 1, cfg['blocks'])
        hn = onet_norm(h)
        add('norm', 1, 0, hn)
    f = blocks('prediction_net.res_blocks', hn, 2, 0, cfg['blocks'])
    pol, val = onet._head('prediction_net.policy_net', f), onet._head('prediction_net.value_net', f)
    out = {'pi': torch.softmax(pol, 1), 'value': _transform(val, cfg['vkind'])}
    if obs is None:
        out['reward'] = _transform(onet._head('dynamics_net.reward_head', h), cfg['rkind'])
    return tens, out


def onet_norm(h):
    from oracle.network_oracle import normalize_hidden_state
    return normalize_hidden_state(h)


def _transform(v, kind):
    if kind == 0:
        return v.view(-1)
    n = v.shape[1]
    hi = (n - 1) // 2
    x = (torch.softmax(v, 1) * torch.linspace(-hi, hi, n, dtype=v.dtype)).sum(1)
    return signed_parabolic(x)


def _exact_fold_sd(sd):
    """Conv weights w = W16 / s (float64): the fp32 fold of the test reproduces W16, and OracleNet in float64 multiplies
    back to W16 within 1e-16 -- the float64 run and the reference then use the same operand."""
    sd = {k: v.double() for k, v in sd.items()}
    for k in list(sd):
        if k.endswith('.0.weight') and k[:-len('.0.weight')] + '.1.running_var' in sd and sd[k].dim() == 4:
            p = k[:-len('.0.weight')]
            w16, _, _, s = fold(sd, p + '.0', p + '.1')
            s64 = sd[p + '.1.weight'] / torch.sqrt(sd[p + '.1.running_var'] + 1e-5)
            n_in = w16.shape[1]
            w = sd[k].clone()
            w[:, :n_in] = w16 / s64.view(-1, 1, 1, 1)
            sd[k] = w
        elif k.endswith(('conv_1.weight', 'conv_2.weight')):
            sd[k] = sd[k].float().half().double()
    return sd


def _cpu_net(kind, seed):
    import muzero_b200 as mz
    from oracle.network_oracle import OracleNet, randomize_batchnorm
    torch.manual_seed(seed)
    if kind == 'board':
        net = mz.MuZeroBoardGameNet((3, 5, 4), 7, 2, 16).eval()
        cfg = dict(planes=16, blocks=2, actions=7, vkind=0, rkind=0)
    else:
        net = mz.MuZeroAtariNet((4, 96, 96), 5, 1, 128, 7, 7).eval()
        cfg = dict(planes=128, blocks=1, actions=5, vkind=1, rkind=1)
    with torch.no_grad():
        randomize_batchnorm(net, seed)
    sd = _exact_fold_sd(net.state_dict())
    onet = OracleNet(kind, {}, cfg['actions'], 1 if kind == 'board' else 7, 1 if kind == 'board' else 7, cfg['blocks'])
    onet.sd = sd
    return sd, onet, cfg


@pytest.mark.parametrize('kind', ['board', 'atari'])
def test_reference_flags_planted_errors(kind):
    """Records filled from an eager float64 run of OracleNet (initial and recurrent) pass every check with wide margin,
    and each planted error is flagged at its layer: 3 fp16 ulps on the largest output element, one tap of one
    board-edge position taken across the edge, a residual from the wrong layer, a normalisation over the padded
    channels."""
    sd, onet, cfg = _cpu_net(kind, 5)
    g = torch.Generator().manual_seed(6)
    B = 3 if kind == 'board' else 1
    shape = (3, 5, 4) if kind == 'board' else (4, 96, 96)
    obs = torch.randint(0, 3 if kind == 'board' else 256, (B,) + shape, generator=g).double()
    with torch.no_grad():
        tens, out = _oracle_record(kind, onet, sd, cfg, obs=obs)
    worst = check_call(kind, sd, cfg, tens, outputs=out)
    assert max(v for v, _ in worst.values()) <= 1e-2, worst
    hid = [t for t in tens if t['kind'] in ('norm', 'pool') and t['index'] == (0 if kind == 'board' else 1)][-1]['data']
    slots = hid.half().double()
    action = torch.randint(0, cfg['actions'], (B,), generator=g)
    with torch.no_grad():
        rt, rout = _oracle_record(kind, onet, sd, cfg, slots=slots, action=action)
    worst = check_call(kind, sd, cfg, rt, slots_in=slots, action=action, outputs=rout)
    assert max(v for v, _ in worst.values()) <= 1e-2, worst
    assert {'conv', 'norm', 'head_policy', 'head_value', 'head_reward'} <= set(worst)

    def rec(recs, stage, index):
        return [t for t in recs if t['kind'] == 'conv' and t['stage'] == stage and t['index'] == index][0]

    def flagged(mutate, where):
        recs = [dict(t, data=t['data'].clone()) for t in rt]
        mutate(recs)
        per = {}
        check_call(kind, sd, cfg, recs, slots_in=slots, action=action, per=per)
        assert per[where] > 1.0, (where, per)

    def bump(recs):                   # 3 fp16 ulps on the largest element of the last dynamics conv
        d = rec(recs, 1, 2 * cfg['blocks'])['data'].view(-1)
        k = int(d.abs().argmax())
        d[k] += 3 * ulp16(d[k])
    flagged(bump, ('conv', f"conv 1.{2 * cfg['blocks']}"))

    def edge_tap(recs):               # board 0, position (1, 0) of dynamics conv 1: the tap (ky 1, kx 0) is not masked
        X = rec(recs, 1, 0)['data']  # and reads row P - 1, the last position (0, W - 1) of the row above
        w16, b, _, _ = fold(sd, *conv_names(kind, 1, 1, 0)[:2])
        R = conv3x3(X, w16) + b.view(1, -1, 1, 1)
        R[0, :, 1, 0] += w16[:, :, 1, 0] @ X[0, :, 0, -1]
        rec(recs, 1, 1)['data'] = R.clamp(0.0, 65504.0)
    flagged(edge_tap, ('conv', 'conv 1.1'))

    def wrong_residual(recs):         # the first prediction block adds its own first conv's output, not its input
        mid = rec(recs, 2, 0)['data']
        w16, b, _, _ = fold(sd, *conv_names(kind, 2, 1, 0)[:2])
        rec(recs, 2, 1)['data'] = (conv3x3(mid, w16) + b.view(1, -1, 1, 1) + mid).clamp(0.0, 65504.0)
    flagged(wrong_residual, ('conv', 'conv 2.1'))

    if kind == 'board':
        def padded_norm(recs):        # a 16-plane net normalised over its 32 padded channels (zeros past 16); the raw
            raw = rec(recs, 1, 2 * cfg['blocks'])['data']       # tensor moved off 0 so that the padding sets the minimum
            raw += 0.5
            [t for t in recs if t['kind'] == 'norm'][0]['data'] = onet_norm(torch.cat([raw, torch.zeros_like(raw)], 1))
        flagged(padded_norm, ('norm', 'norm 1.0'))


# ---- the engine (GPU) -----------------------------------------------------------------------------------------------
KINDS = {0: 'obs', 1: 'conv', 2: 'pool', 3: 'norm'}


def launch_forms(L):
    """The forms one launch record shows (names of FORMS)."""
    f = set()
    if L['n'] == 32:
        f.add('n32')
    if L['multi_pass']:
        f.add('multi_pass')
    if L['sub']:
        f.add('sub')
    elif L['num_layers'] == 1:
        f.add('single')
    elif L['resident']:
        f.add(f"resident{L['tile_rows']}")
        if L['khalf']:
            f.add('khalf')
    elif L['pair']:
        f.add('pair')
        if L['num_tiles'] % 2:
            f.add('pair_null_tile')
    elif L['tile_rows'] == 256:
        f.add('dataflow256')
    else:
        f.add('splitk128')
    return f


# name: (kind, input shape, actions, blocks, planes, support, batch, cta_limit, forced tile rows, forms it must show)
CASES = {
    'gomoku_bench_pair': ('board', (9, 9, 9), 81, 8, 128, 1, 1024, 144, None, {'pair'}),
    'gomoku_pair_null_tile': ('board', (9, 9, 9), 81, 8, 128, 1, 1000, 0, None, {'pair_null_tile'}),
    'gomoku_resident128': ('board', (9, 9, 9), 81, 8, 128, 1, 100, 0, None, {'resident128', 'single'}),
    'gomoku_resident256_khalf': ('board', (9, 9, 9), 81, 8, 128, 1, 300, 0, None, {'resident256', 'khalf'}),
    'gomoku_splitk128': ('board', (9, 9, 9), 81, 8, 128, 1, 600, 0, None, {'splitk128'}),
    'gomoku_single_cta_256': ('board', (9, 9, 9), 81, 8, 128, 1, 100, 1, 256, {'dataflow256'}),
    'board5_cg8_resident': ('board', (4, 5, 5), 25, 2, 64, 1, 37, 0, None, {'resident256'}),
    'board5_pair64': ('board', (4, 5, 5), 25, 2, 64, 1, 2000, 0, None, {'pair'}),
    'tictactoe_16_planes': ('board', (3, 3, 3), 9, 2, 16, 1, 1, 0, None, {'n32'}),
    'tictactoe_16_planes_1000': ('board', (3, 3, 3), 9, 2, 16, 1, 1000, 0, None, {'n32'}),
    'planes256_2blocks': ('board', (9, 9, 9), 82, 2, 256, 1, 7, 0, None, {'multi_pass'}),
    'planes256_16blocks_split': ('board', (9, 9, 9), 82, 16, 256, 1, 300, 0, None, {'multi_pass', 'split_in_block'}),
    'board19_never_resident': ('board', (17, 19, 19), 362, 2, 64, 1, 5, 0, None, {'pair'}),
    'board19_one': ('board', (17, 19, 19), 362, 2, 64, 1, 1, 0, None, set()),
    'board_1x9': ('board', (2, 1, 9), 9, 1, 32, 1, 5, 0, None, set()),
    'board_9x1': ('board', (2, 9, 1), 9, 1, 32, 1, 5, 0, None, set()),
    'board_2x2': ('board', (2, 2, 2), 4, 1, 32, 1, 3, 0, None, set()),
    'board_16x16_one_tile': ('board', (3, 16, 16), 256, 1, 64, 1, 4, 0, None, set()),
    'board_8x16_half_tile': ('board', (3, 8, 16), 128, 1, 64, 1, 4, 0, None, set()),
    'board_3x40_widest': ('board', (3, 3, 40), 120, 1, 128, 1, 6, 0, None, set()),
    'obs1_action1': ('board', (1, 4, 4), 1, 1, 32, 1, 5, 0, None, set()),
    'obs64_action226': ('board', (64, 6, 6), 226, 1, 64, 1, 5, 0, None, set()),
    'blocks0': ('board', (9, 9, 9), 81, 0, 128, 1, 1, 0, None, {'single'}),
    'blocks0_300': ('board', (9, 9, 9), 81, 0, 128, 1, 300, 0, None, {'single'}),
    'atari': ('atari', (16, 96, 96), 18, 8, 128, 61, 3, 0, None, {'sub'}),
    'atari_cta7': ('atari', (16, 96, 96), 18, 8, 128, 61, 8, 7, None, {'sub'}),
}


def _sample(batch, pb, seed):
    """Boards the reference runs on: first, last, every one straddling a 128-row (so also 256-row) tile boundary, and
    8 random ones."""
    s = {0, batch - 1}
    s.update(b for b in range(batch) if (b * pb) // 128 != ((b + 1) * pb - 1) // 128)
    s.update(np.random.RandomState(seed).choice(batch, min(batch, 8), replace=False).tolist())
    return torch.tensor(sorted(s))


# forms a case must NOT show (what its name promises)
NOT_FORMS = {'board19_never_resident': {'resident128', 'resident256'}, 'board19_one': {'resident128', 'resident256'},
             'gomoku_single_cta_256': {'pair', 'resident128', 'resident256'}, 'blocks0': set(FORMS[2:9]),
             'blocks0_300': set(FORMS[2:9])}


def _planes(buf_of, t, boards):
    """A recorded tensor as float64 [boards, groups*8, h, w] (the planes are [groups][plane rows][8] fp16)."""
    base, ten = buf_of(t.ptr)
    off = t.ptr - base
    raw = ten[off:off + t.plane_rows * t.groups * 16].view(torch.float16).view(t.groups, t.plane_rows, 8)
    pb = t.h * t.w
    x = raw[:, :t.batch * pb].view(t.groups, t.batch, t.h, t.w, 8)[:, boards.to(raw.device)]
    return x.permute(1, 0, 4, 2, 3).reshape(len(boards), t.groups * 8, t.h, t.w).double()


def _slots_nchw(slots, idx, cp, h, w):
    x = slots.view(torch.float16).reshape(slots.shape[0], cp // 8, h, w, 8)[idx]
    return x.permute(0, 1, 4, 2, 3).reshape(len(idx), cp, h, w).double()


def run_case(name, monkeypatch):
    import muzero_b200 as mz
    from muzero_b200 import _lib
    from oracle.network_oracle import randomize_batchnorm
    kind, shape, A, blocks, planes, support, batch, limit, rows, forms = CASES[name]
    torch.manual_seed(11)
    if kind == 'board':
        net = mz.MuZeroBoardGameNet(shape, A, blocks, planes).eval()
    else:
        net = mz.MuZeroAtariNet(shape, A, blocks, planes, support, support).eval()
    with torch.no_grad():
        randomize_batchnorm(net, 12)
    net = net.cuda()
    sd = {k: v.detach().clone() for k, v in net.state_dict().items()}
    kind1 = 0 if support == 1 else 1
    cfg = dict(planes=planes, blocks=blocks, actions=A, vkind=kind1, rkind=kind1)
    if rows:
        monkeypatch.setenv('MZ_CONV_TILE_ROWS', str(rows))
    else:
        monkeypatch.delenv('MZ_CONV_TILE_ROWS', raising=False)
    e = net.engine(batch)
    lib, h = _lib.lib(), e['handle']
    _lib.check(lib.mz_net_set_cta_limit(h, limit))
    gen = torch.Generator(device='cuda').manual_seed(13)
    obs = (torch.randint(0, 256 if kind == 'atari' else 3, (batch,) + shape, device='cuda', generator=gen)).float()
    nslots = 2 * batch + 3
    dst0 = torch.randperm(nslots, device='cuda', generator=gen)[:batch].int()
    src1 = dst0[torch.randperm(batch, device='cuda', generator=gen)]
    dst1 = torch.randperm(nslots, device='cuda', generator=gen)[:batch].int()
    act = torch.randint(0, A, (batch,), device='cuda', generator=gen).int()
    fill = torch.randint(0, 256, (nslots, net.hidden_bytes), dtype=torch.uint8, device='cuda', generator=gen)
    fill.view(torch.float16)[:] = fill.view(torch.float16).nan_to_num(0.5).clamp(-1, 1)   # finite, recognisable

    def calls():
        h0 = fill.clone()
        _, pi0, v0 = net.initial_inference_batch(obs, hidden_out=h0, dst_index=dst0)
        rec0 = capture_record()
        h1 = fill.clone()
        _, r1, pi1, v1 = net.recurrent_inference_batch(h0, act, src_index=src1, hidden_out=h1, dst_index=dst1)
        rec1 = capture_record()
        torch.cuda.synchronize()
        return (h0, pi0, v0, h1, r1, pi1, v1), rec0, rec1

    buf = None
    pb_lat = net.latent_hw[0] * net.latent_hw[1]
    boards = _sample(batch, pb_lat if kind == 'board' else 96 * 96, 14)
    cp = net.padded_planes

    def buf_of(p):
        for t in (buf, e['arena']):
            if t is not None and t.data_ptr() <= p < t.data_ptr() + t.numel():
                return t.data_ptr(), t
        raise AssertionError('tensor outside the capture buffer and the arena')

    def capture_record():
        if buf is None:
            return None
        n = C.c_int32()
        _lib.check(lib.mz_net_debug_tensor(h, -1, None, C.byref(n)))
        tens = []
        for i in range(n.value):
            t = _lib.DebugTensor()
            _lib.check(lib.mz_net_debug_tensor(h, i, C.byref(t), C.byref(n)))
            tens.append(dict(kind=KINDS[t.kind], stage=t.stage, index=t.index, src=t.src, residual=t.residual,
                             data=_planes(buf_of, t, boards)))
        _lib.check(lib.mz_net_debug_launch(h, -1, None, C.byref(n)))
        launches = []
        for i in range(n.value):
            L = _lib.DebugLaunch()
            _lib.check(lib.mz_net_debug_launch(h, i, C.byref(L), C.byref(n)))
            launches.append({k: (list(getattr(L, k)) if k in ('out', 'pass_', 'flags', 'dep0', 'res_layer', 'fwd')
                                 else getattr(L, k)) for k, _ in L._fields_})
        return tens, launches

    off, _, _ = calls()
    nb = C.c_size_t()
    _lib.check(lib.mz_net_debug_capture_bytes(h, batch, C.byref(nb)))
    buf = torch.empty(nb.value + 256, dtype=torch.uint8, device='cuda')
    base = (buf.data_ptr() + 255) // 256 * 256
    _lib.check(lib.mz_net_debug_capture(h, base, nb.value))
    try:
        on, rec0, rec1 = calls()
    finally:
        _lib.check(lib.mz_net_debug_capture(h, None, 0))
    bad, worst, seen = [], {}, set()
    for k, (a, b) in enumerate(zip(off, on)):
        if not torch.equal(a.view(torch.uint8), b.view(torch.uint8)):
            bad.append(f'output {k} differs between capture off and on')
    for call, (tens, launches), out in ((0, rec0, dict(pi=on[1], value=on[2])),
                                        (1, rec1, dict(pi=on[5], value=on[6], reward=on[4]))):
        for L in launches:
            seen |= launch_forms(L)
            for i in range(L['num_layers']):
                t = L['out'][i]
                if t >= 0 and tens[t]['residual'] >= 0 and L['dep0'][i] < 0:
                    seen.add('split_in_block')
        wire = wiring(kind, tens)
        for i, (src, res) in wire.items():
            got = (tens[i]['src'], tens[i]['residual'])
            want = (-1 if src == 'slots' else src, -1 if res is None else res)
            if tens[i]['kind'] != 'conv':
                got = got[0]
                want = want[0]
            if got != want:
                bad.append(f'call {call}: record wiring of tensor {i} {got}, structure says {want}')
        slots_in = _slots_nchw(on[0], src1[boards.cuda()].long(), cp, *net.latent_hw) if call else None
        outs = {k: v[boards.cuda()].double() for k, v in out.items()}
        w = check_call(kind, sd, cfg, tens, slots_in=slots_in, action=act[boards.cuda()].cpu() if call else None,
                       outputs=outs, heads_from=[t for t in tens if t['kind'] in ('norm', 'pool')][-1]['data'])
        for k, (v, where) in w.items():
            key = f'{k}'
            if key not in worst or not v <= worst[key][0]:
                worst[key] = (v, f'call {call} {where}')
            if not v <= 1.0:
                bad.append(f'call {call} {where}: {k} {v:.4g} > 1')
        # the normalised state: every written slot holds the bits of the normalised tensor, the others keep theirs
        norm = [t for t in tens if t['kind'] == 'norm' or (t['kind'] == 'pool' and t['index'] == 1)][-1]['data']
        hs = on[0] if call == 0 else on[3]
        di = (dst0 if call == 0 else dst1)
        if not torch.equal(_slots_nchw(hs, di[boards.cuda()].long(), cp, *net.latent_hw), norm):
            bad.append(f'call {call}: slots differ from the normalised tensor')
        keep = torch.ones(nslots, dtype=torch.bool, device='cuda')
        keep[di.long()] = False
        if not torch.equal(hs[keep], fill[keep]):
            bad.append(f'call {call}: a slot not named by dst_index changed')
    missing = forms - seen
    extra = NOT_FORMS.get(name, set()) & seen
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


def test_debug_launch_record_matches_the_header():
    """The Python mirror of mz_debug_launch holds MZ_DEBUG_MAX_LAYERS entries per layer field, as the header says
    (conv.cu ties that constant to kMaxLayers with a static_assert)."""
    import re
    from conftest import ROOT
    from muzero_b200 import _lib
    src = open(os.path.join(ROOT, 'include', 'muzero_b200.h')).read()
    assert int(re.search(r'#define MZ_DEBUG_MAX_LAYERS (\d+)', src).group(1)) == _lib.MZ_DEBUG_MAX_LAYERS
    assert C.sizeof(_lib.DebugLaunch) == 4 * (14 + 6 * _lib.MZ_DEBUG_MAX_LAYERS)
    assert C.sizeof(_lib.DebugTensor) == 8 + 4 * 10


@pytest.mark.gpu
def test_undersized_capture_buffer_fails_cleanly():
    """A capture buffer too small for a call: the call raises MemoryError and leaves nothing queued that points into
    that buffer -- after capture is turned off, the next calls give the same bytes as a net that never captured.  For
    a conv net and an MLP net."""
    import muzero_b200 as mz
    from muzero_b200 import _lib
    from oracle.network_oracle import randomize_batchnorm
    torch.manual_seed(21)
    nets = []
    for _ in range(2):
        torch.manual_seed(21)
        n = mz.MuZeroBoardGameNet((9, 9, 9), 81, 2, 128).eval()
        with torch.no_grad():
            randomize_batchnorm(n, 22)
        nets.append(n.cuda())
    B = 64
    gen = torch.Generator(device='cuda').manual_seed(23)
    obs = torch.randint(0, 3, (B, 9, 9, 9), device='cuda', generator=gen).float()
    act = torch.randint(0, 81, (B,), device='cuda', generator=gen).int()
    e = nets[0].engine(B)
    lib, h = _lib.lib(), e['handle']
    nb = C.c_size_t()
    _lib.check(lib.mz_net_debug_capture_bytes(h, B, C.byref(nb)))
    small = torch.empty(nb.value // 8, dtype=torch.uint8, device='cuda')
    base = (small.data_ptr() + 255) // 256 * 256
    _lib.check(lib.mz_net_debug_capture(h, base, small.numel() - 256))
    with pytest.raises(MemoryError):
        nets[0].initial_inference_batch(obs)
    with pytest.raises(MemoryError):
        nets[0].recurrent_inference_batch(nets[0].new_hidden(B), act)
    _lib.check(lib.mz_net_debug_capture(h, None, 0))
    del small
    torch.cuda.synchronize()
    outs = []
    for n in nets:
        hid, pi, v = n.initial_inference_batch(obs)
        hid2, r, pi2, v2 = n.recurrent_inference_batch(hid, act)
        torch.cuda.synchronize()
        outs.append([t.view(torch.uint8) for t in (hid, pi, v, hid2, r, pi2, v2)])
    for k, (a, b) in enumerate(zip(*outs)):
        assert torch.equal(a, b), k
    # the same for an MLP net: its SIMT initial call and its tcgen05 recurrent call
    torch.manual_seed(24)
    m = mz.MuZeroMLPNet((4, 5), 2, 512, 31, 31, 64).cuda().eval()
    mobs = torch.randn((B, 4, 5), device='cuda', generator=gen)
    mact = torch.randint(0, 2, (B,), device='cuda', generator=gen).int()
    ref = []
    for capture in (True, False):
        eh = m.engine(B)['handle']
        if capture:
            _lib.check(lib.mz_net_debug_capture_bytes(eh, B, C.byref(nb)))
            small = torch.empty(nb.value // 8, dtype=torch.uint8, device='cuda')
            base = (small.data_ptr() + 255) // 256 * 256
            _lib.check(lib.mz_net_debug_capture(eh, base, small.numel() - 256))
            with pytest.raises(MemoryError):
                m.initial_inference_batch(mobs)
            with pytest.raises(MemoryError):
                m.recurrent_inference_batch(m.new_hidden(B), mact)
            _lib.check(lib.mz_net_debug_capture(eh, None, 0))
            del small
            torch.cuda.synchronize()
        hid, pi, v = m.initial_inference_batch(mobs)
        hid2, r, pi2, v2 = m.recurrent_inference_batch(hid, mact)
        torch.cuda.synchronize()
        ref.append([t.view(torch.uint8) for t in (hid, pi, v, hid2, r, pi2, v2)])
        m.release_engine()
    for k, (a, b) in enumerate(zip(*ref)):
        assert torch.equal(a, b), f'mlp output {k}'
