"""Layer-by-layer tests of the training kernels (csrc/train.cu): every convolution, BatchNorm and ReLU of every tower
call of a training step against a float64 computation fed the kernels' OWN stored tensors (``mz_train_debug_view``).

Comparing whole towers with fp32 autograd (tests/test_train_gpu.py) has to be loose: a forward difference of 1e-3
flips one ReLU in a thousand and each flip moves that element's whole gradient, so a kernel that is wrong by a few
per cent still passes there.  Here each layer gets the kernel's own input, so the ReLU masks are identical and what
is left is rounding:

* forward, per layer l of every call, with X_l the layer's saved input and R_l = conv3x3_f64(X_l, fp16(W_l)):
  - raw conv output, every element: |Y_l - R_l| <= ulp16(R_l) + 2^-16 conv3x3_f64(|X_l|, |fp16(W_l)|);
  - saved batch mean within 1e-5 (|mean| + sigma) and 1/sqrt(var + eps) within 1e-4 relative of R_l's;
  - activated output A_l against relu(gamma (Y_l - mean) invstd + beta [+ residual]) in float64 from the kernel's own
    Y_l, statistics and residual: 1 fp16 ulp + 2^-20 of the magnitudes of the terms;
  - the halo, front and tail rows (and padding channels) of every saved plane are +0; the tower's float32 output is
    the last A exactly;
  - running mean / variance after the step: the float64 recursion over the calls in call order (momentum 0.1,
    unbiased variance) within 1e-5 (|mean| + sigma) / 1e-4 relative; num_batches_tracked counts every call.
  Measured worst over all cases, as error / bound (NVIDIA B200, 1000 W power limit): raw 0.49, mean 0.17, invstd 0.28,
  activation 0.50 (the fp16 rounding itself), running mean 0.12, running variance 0.033.
* backward: one float64 autograd graph per call, Z_l = BN_batchstats(conv_f64(A~_{l-1}, W_l)) [+ A~_{l-2}] with the
  fp32 parameters, and A~_l = A_l + (Z_l M_l - (Z_l M_l).detach()), M_l = (A_l > 0): the value is the kernel's
  activation, the derivative float64 with the kernel's masks.  What remains is bf16 storage of the gradients and of
  the dgrad weights.  Bound 2e-2 relative L2 per tensor for each of: grad_in of every dynamics and prediction call,
  every conv dW summed over the step's calls (the dynamics' first conv split into its hidden-state and action input
  channels), dgamma and dbeta.  Measured worst over all cases (NVIDIA B200, 1000 W power limit): grad_in 9.3e-3,
  dW 1.2e-2 (action channels 9.3e-3), dgamma 1.0e-2, dbeta 1.0e-2 -- all on the 8-block benchmarked step; the
  1- and 2-block cases stay below 7.2e-3.
  The kernels add into .grad: it is pre-filled with random values on the first step and keeps the first step's
  gradients on the second.

Every case runs two full steps (representation once, dynamics K times, prediction K times -- stacked where the
engine allows --, the backward in reverse, end_step) with the parameters changed in place between them, as an
optimizer would.  ``test_reference_equals_float64_autograd_of_the_modules`` checks the reference itself on the CPU."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

EPS, MOMENTUM = 1e-5, 0.1
GRAD_TOL = 2e-2                     # relative L2 per gradient tensor (module docstring)
TOWERS = ('representation', 'dynamics', 'prediction')


# ---- the float64 reference (device-agnostic) --------------------------------------------------------------------
def conv3x3(x, w):
    return F.conv2d(x, w, padding=1)


def ulp16(r):
    """Spacing of fp16 numbers at |r| (subnormal spacing 2^-24 below 2^-14)."""
    return torch.exp2(torch.floor(torch.log2(r.abs().clamp_min(2.0 ** -14))) - 10)


def fp16_weight(w):
    """The forward operand pack_weights_kernel makes of a conv weight, as float64."""
    return w.detach().float().clamp(-65504.0, 65504.0).half().double()


def residual_source(tower, layer):
    """The layer whose INPUT is added back after this layer's BatchNorm (second conv of a residual block), or None."""
    first = 0 if tower == 2 else 1
    return layer - 1 if layer >= first and (layer - first) % 2 == 1 else None


def layer_input(X, As, layer):
    return X if layer == 0 else As[layer - 1]


def _ch(t):
    return t.view(1, -1, 1, 1)


def forward_ratios(tower, X, Ys, As, stats, weights16, gammas, betas):
    """Error / bound of each forward check of one tower call, per layer, and the float64 (mean, biased variance) of
    every layer's exact conv output R_l.  X, Ys, As: float64 [B, C, H, W]; stats: [128, 2] (mean, invstd) per layer."""
    ratios, moments = [], []
    for l in range(len(Ys)):
        x, w = layer_input(X, As, l), weights16[l]
        R = conv3x3(x, w)
        raw = ((Ys[l] - R).abs() / (ulp16(R) + 2.0 ** -16 * conv3x3(x.abs(), w.abs()))).max()
        m, v = R.mean((0, 2, 3)), R.var((0, 2, 3), unbiased=False)
        del R
        mk, ik = stats[l][:, 0].double(), stats[l][:, 1].double()
        e_mean = ((mk - m).abs() / (1e-5 * (m.abs() + v.sqrt()) + 1e-300)).max()
        iref = (v + EPS).rsqrt()
        e_inv = ((ik - iref).abs() / (1e-4 * iref)).max()
        r = residual_source(tower, l)
        res = layer_input(X, As, r) if r is not None else torch.zeros_like(Ys[l])
        sc, beta = _ch(gammas[l].detach().double() * ik), _ch(betas[l].detach().double())
        ref = (sc * (Ys[l] - _ch(mk)) + beta + res).clamp_min(0.0)
        bound = ulp16(ref) + 2.0 ** -20 * ((sc * Ys[l]).abs() + (sc * _ch(mk)).abs() + beta.abs() + res.abs())
        e_act = ((As[l] - ref).abs() / bound).max()
        ratios.append({'raw': float(raw), 'mean': float(e_mean), 'invstd': float(e_inv), 'act': float(e_act)})
        moments.append((m, v))
    return ratios, moments


def reference_backward(tower, X, As, params, grad_out):
    """float64 autograd of one tower call over the kernel's activations As and their ReLU masks.  params: per layer
    (W, gamma, beta) float64 leaves, which accumulate their gradients.  Returns dL/dX."""
    x = X.detach().clone().requires_grad_(True)
    acts = []
    for l, (w, g, b) in enumerate(params):
        y = conv3x3(layer_input(x, acts, l), w)
        m = y.mean((0, 2, 3), keepdim=True)
        v = (y - m).square().mean((0, 2, 3), keepdim=True)
        z = (y - m) * torch.rsqrt(v + EPS) * _ch(g) + _ch(b)
        r = residual_source(tower, l)
        if r is not None:
            z = z + layer_input(x, acts, r)
        zm = z * (As[l] > 0)
        acts.append(As[l] + (zm - zm.detach()))
    acts[-1].backward(grad_out)
    return x.grad


def running_stats(rm, rv, moments, n):
    """BatchNorm2d's running-statistics update over the calls' (mean, biased variance), in call order."""
    for m, v in moments:
        rm = (1.0 - MOMENTUM) * rm + MOMENTUM * m
        rv = (1.0 - MOMENTUM) * rv + MOMENTUM * v * (n / (n - 1.0))
    return rm, rv


def rel(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float((a - b).norm() / (b.norm() + 1e-300))


# ---- the reference checked against plain float64 autograd of the modules (CPU) --------------------------------------
def test_reference_equals_float64_autograd_of_the_modules():
    """The "kernel tensors" filled from an eager float64 forward of the network's own modules (train mode): the
    reference's parameter and input gradients equal plain float64 autograd of those modules to 1e-10, its forward
    checks pass with room to spare and catch a 3-ulp error in one element, and the running-statistics recursion
    reproduces BatchNorm2d's buffers.  This covers the mask and residual wiring of every tower."""
    import muzero_b200 as mz
    from muzero_b200.network import action_planes
    from muzero_b200.train_engine import _tower_modules
    torch.manual_seed(3)
    B, h, w, c_in, A, calls = 3, 5, 5, 9, 26, 2
    net = mz.MuZeroBoardGameNet((c_in, h, w), A, 1, 128).double().train()
    mods = _tower_modules(net)
    with torch.no_grad():
        for conv, bn in mods:
            conv.weight.copy_(fp16_weight(conv.weight))     # fp16 values: the forward checks see no weight rounding
            bn.weight.uniform_(0.5, 1.5)
            bn.bias.uniform_(-0.3, 0.3)
            bn.running_mean.normal_(0.0, 0.5)
            bn.running_var.uniform_(0.5, 2.0)
    spans = [(0, 3), (3, 6), (6, 8)]
    for tower, tnet in enumerate((net.represent_net, net.dynamics_net, net.prediction_net)):
        tm = mods[spans[tower][0]:spans[tower][1]]
        a_mods = ([tnet.conv_block] if tower != 2 else []) + [m for blk in tnet.res_blocks for m in (blk.conv_block1, blk)]
        params = [p for conv, bn in tm for p in (conv.weight, bn.weight, bn.bias)]
        leaves = [tuple(p.detach().clone().requires_grad_(True) for p in (conv.weight, bn.weight, bn.bias)) for conv, bn in tm]
        want = [torch.zeros_like(p) for p in params]
        before = [(bn.running_mean.clone(), bn.running_var.clone()) for _, bn in tm]
        moments = [[] for _ in tm]
        for call in range(calls):
            x = (torch.rand((B, c_in, h, w), dtype=torch.float64) * 2 if tower == 0 else
                 torch.rand((B, 128, h, w), dtype=torch.float64)).requires_grad_(tower != 0)
            X = torch.cat([x, action_planes(torch.randint(0, A, (B, 1)), A, h, w).double()], dim=1) if tower == 1 else x
            ys, acts = {}, {}
            hooks = [conv.register_forward_hook(lambda mod, i, o, k=k: ys.__setitem__(k, o.detach())) for k, (conv, _) in enumerate(tm)]
            hooks += [m.register_forward_hook(lambda mod, i, o, k=k: acts.__setitem__(k, o.detach())) for k, m in enumerate(a_mods)]
            out = tnet.res_blocks(tnet.conv_block(X) if tower != 2 else X)
            for hk in hooks:
                hk.remove()
            gout = torch.randn_like(out) * (call + 0.5)
            got_plain = torch.autograd.grad(out, params + ([x] if tower else []), gout)
            for k, g in enumerate(got_plain[:len(params)]):
                want[k] += g
            Ys, As = [ys[k] for k in range(len(tm))], [acts[k] for k in range(len(tm))]
            stats = [torch.stack([y.mean((0, 2, 3)), (y.var((0, 2, 3), unbiased=False) + EPS).rsqrt()], dim=1) for y in Ys]
            w16 = [fp16_weight(conv.weight) for conv, _ in tm]
            gammas, betas = [bn.weight for _, bn in tm], [bn.bias for _, bn in tm]
            ratios, mom = forward_ratios(tower, X.detach(), Ys, As, stats, w16, gammas, betas)
            assert max(v for r in ratios for v in r.values()) <= 1e-3, ratios
            for k, mv in enumerate(mom):
                moments[k].append(mv)
            off = [y.clone() for y in Ys]
            big = off[-1].view(-1)                    # the largest output, where the accumulation allowance is < 1 ulp
            k = int(big.abs().argmax())
            big[k] += 3 * ulp16(big[k])
            assert forward_ratios(tower, X.detach(), off, As, stats, w16, gammas, betas)[0][-1]['raw'] > 1.0
            gi = reference_backward(tower, X, As, leaves, gout)
            if tower:
                assert rel(gi[:, :128], got_plain[-1]) <= 1e-10, (tower, call, rel(gi[:, :128], got_plain[-1]))
        got = [p.grad for lv in leaves for p in lv]
        for k, (a, b) in enumerate(zip(got, want)):
            assert rel(a, b) <= 1e-10, (tower, k, rel(a, b))
        for k, (_, bn) in enumerate(tm):
            rm, rv = running_stats(before[k][0], before[k][1], moments[k], B * h * w)
            assert rel(bn.running_mean, rm) <= 1e-12 and rel(bn.running_var, rv) <= 1e-12, (tower, k)


# ---- the kernels (GPU) ---------------------------------------------------------------------------------------------
def _raw_planes(eng, tower, call, layer, which):
    """A saved tensor as the 16-bit planes the kernels keep ([groups][plane rows][8], as int16) and its front row."""
    from muzero_b200 import _lib
    p, n, pr, fr = C.c_void_p(), C.c_size_t(), C.c_int32(), C.c_int32()
    _lib.check(_lib.lib().mz_train_debug_view(eng.handle, tower, call, layer, which, C.byref(p), C.byref(n), C.byref(pr),
                                              C.byref(fr)))
    off = p.value - eng.arena.data_ptr()
    return eng.arena[off:off + n.value].view(torch.int16).reshape(-1, pr.value, 8), fr.value


def _nonzero_padding(eng, raw, fr, calls, channels):
    """Elements of saved planes that are not +0 outside the real positions of `calls` consecutive calls from plane row
    fr and outside the first `channels` channels."""
    g, rows, _ = raw.shape
    _, h, w = eng.input_shape
    pb = (h + 1) * (w + 1)
    r = torch.arange(rows, device=raw.device) - fr
    q = torch.remainder(r, pb)
    real = (r >= 0) & (r < calls * eng.batch * pb) & (q // (w + 1) < h) & (q % (w + 1) < w)
    chan = (torch.arange(g * 8, device=raw.device) < channels).view(g, 1, 8)
    return int(((raw != 0) & ~(real.view(1, rows, 1) & chan)).sum())


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


# (board h, w), input planes, actions, residual blocks, batch (None: the smallest with more 128-row tiles than SMs),
# unroll K, prediction calls stacked
CASES = {
    'benchmarked_step': ((9, 9), 9, 82, 8, 128, 5, True),
    'unstacked_half_last_tile': ((9, 9), 9, 82, 2, 16, 5, False),
    'more_tiles_than_sms': ((9, 9), 9, 82, 1, None, 2, False),
    'one_row_last_tile': ((6, 6), 17, 37, 1, 81, 3, False),
    'single_plane_127_row_last_tile': ((6, 6), 1, 1, 1, 47, 1, False),
    'smallest_board': ((2, 2), 3, 5, 2, 2, 2, False),
    'non_square_board': ((6, 7), 3, 7, 1, 32, 4, True),
    'widest_board': ((3, 62), 128, 128, 1, 4, 2, False),
    'unroll_16': ((9, 9), 9, 82, 1, 32, 16, True),
}


def run_case(name, seed=0):
    """Two training steps of one case; returns ({check: (worst value, where)}, [failures])."""
    import muzero_b200 as mz
    from muzero_b200 import train_engine
    (h, w), in_planes, actions, blocks, batch, K, expect_stacked = CASES[name]
    if batch is None:
        batch = 128 * _sms() // ((h + 1) * (w + 1)) + 1
    torch.manual_seed(seed)
    net = mz.MuZeroBoardGameNet((in_planes, h, w), actions, blocks, 128).cuda().train()
    with torch.no_grad():
        for m in net.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.weight.uniform_(0.5, 1.5)
                m.bias.uniform_(-0.3, 0.3)
                m.running_mean.normal_(0.0, 0.5)
                m.running_var.uniform_(0.5, 2.0)
    eng = train_engine.engine_for(net, batch, K)
    assert eng is not None
    stacked = K > 1 and eng.max_stacked_calls >= K
    assert stacked == expect_stacked, (name, eng.max_stacked_calls)
    if name == 'more_tiles_than_sms':
        assert (batch * (h + 1) * (w + 1) + 127) // 128 > _sms() >= ((batch - 1) * (h + 1) * (w + 1) + 127) // 128
    mods = eng.modules
    nl = [1 + 2 * blocks, 1 + 2 * blocks, 2 * blocks]
    first = [0, nl[0], nl[0] + nl[1]]
    ncalls = [1, K, K]
    ci = [in_planes, 128 + actions, 128]
    tower_of = [t for t in range(3) for _ in range(nl[t])]
    n = batch * h * w
    gen = torch.Generator(device='cuda').manual_seed(seed + 1)
    rs = np.random.RandomState(seed + 2)
    worst, bad = {}, []

    def note(check, value, bound, where):
        if check not in worst or not value <= worst[check][0]:
            worst[check] = (value, where)
        if not value <= bound:
            bad.append(f'{where}: {check} {value:.4g} > {bound:.4g}')

    def randn(shape, scale=1.0):
        return torch.randn(shape, device='cuda', generator=gen) * scale

    def uniform(shape, lo, hi):
        return torch.rand(shape, device='cuda', generator=gen) * (hi - lo) + lo

    hshape = (batch, 128, h, w)
    for step in range(2):
        if step:
            with torch.no_grad():           # an optimizer step: new values in the same tensors, .grad not zeroed
                for conv, bn in mods:
                    conv.weight.add_(randn(conv.weight.shape, 0.1 * float(conv.weight.std())))
                    bn.weight.add_(uniform(128, -0.1, 0.1)).clamp_(0.5, 1.5)
                    bn.bias.add_(uniform(128, -0.05, 0.05)).clamp_(-0.3, 0.3)
        obs = uniform((batch, in_planes, h, w), 0.0, 2.0)
        xs_dyn = [uniform(hshape, 0.0, 1.0).requires_grad_(True) for _ in range(K)]
        acts = [torch.randint(0, actions, (batch, 1), device='cuda', generator=gen) for _ in range(K)]
        xs_pred = [uniform(hshape, 0.0, 1.0).requires_grad_(True) for _ in range(K)]
        scale = {(t, c): float(10.0 ** rs.uniform(-1.0, 1.0)) for t in range(3) for c in range(ncalls[t])}
        if name == 'unroll_16':             # both ends of the fixed-point gradient sums
            scale[(2, 2)], scale[(2, 9)] = 1e-4, 1e2
        gouts = {k: randn(hshape, s) for k, s in scale.items()}
        before = [(bn.running_mean.double(), bn.running_var.double(), int(bn.num_batches_tracked)) for _, bn in mods]

        rep = train_engine.tower(eng, 0, obs)
        dyn = [train_engine.tower(eng, 1, x, a) for x, a in zip(xs_dyn, acts)]
        pred = train_engine.prediction_calls(eng, xs_pred)
        assert eng.calls == [1, K, K]
        torch.cuda.synchronize()
        outs = {(0, 0): rep, **{(1, c): dyn[c] for c in range(K)}, **{(2, c): pred[c * batch:(c + 1) * batch] for c in range(K)}}

        leaves = [tuple(t.detach().double().requires_grad_(True) for t in (conv.weight, bn.weight, bn.bias)) for conv, bn in mods]
        w16 = [fp16_weight(conv.weight) for conv, _ in mods]
        moments = [[] for _ in mods]
        grad_in_ref = {}
        for tower in range(3):
            span = range(first[tower], first[tower] + nl[tower])
            for call in range(ncalls[tower]):
                where = f'step {step} {TOWERS[tower]} call {call}'
                X = eng.debug_view(tower, call, 0, 0)[:, :ci[tower]].double()
                Ys = [eng.debug_view(tower, call, l, 1).double() for l in range(nl[tower])]
                As = [eng.debug_view(tower, call, l, 2).double() for l in range(nl[tower])]
                stats = [eng.debug_view(tower, call, l, 3) for l in range(nl[tower])]
                if not torch.equal(outs[(tower, call)], As[-1].float()):
                    bad.append(f'{where}: the tower output is not its last saved activation')
                ratios, mom = forward_ratios(tower, X, Ys, As, stats, [w16[i] for i in span], [mods[i][1].weight for i in span],
                                             [mods[i][1].bias for i in span])
                for l, r in enumerate(ratios):
                    for k, v in r.items():
                        note('fwd_' + k, v, 1.0, f'{where} layer {l}')
                for l, mv in enumerate(mom):
                    moments[first[tower] + l].append(mv)
                gi = reference_backward(tower, X, As, [leaves[i] for i in span], gouts[(tower, call)].double())
                if tower:
                    grad_in_ref[(tower, call)] = gi[:, :128]
                del X, Ys, As, gi
                if tower == 2 and stacked and call > 0:
                    continue                # the stacked buffers are checked whole, through call 0
                calls_in_buf = K if tower == 2 and stacked else 1
                for layer, which, chans in [(0, 0, ci[tower])] + [(l, k, 128) for l in range(nl[tower]) for k in (1, 2)]:
                    raw, fr = _raw_planes(eng, tower, call, layer, which)
                    nz = _nonzero_padding(eng, raw, fr, calls_in_buf, chans)
                    if nz:
                        bad.append(f'{where} layer {layer} view {which}: {nz} nonzero halo / front / tail / padding elements')
        for i, (_, bn) in enumerate(mods):
            rm, rv = running_stats(before[i][0], before[i][1], moments[i], n)
            where = f'step {step} {TOWERS[tower_of[i]]} layer {i - first[tower_of[i]]}'
            note('running_mean', float(((bn.running_mean.double() - rm).abs() / (1e-5 * (rm.abs() + rv.sqrt()))).max()), 1.0, where)
            note('running_var', float(((bn.running_var.double() - rv).abs() / (1e-4 * rv)).max()), 1.0, where)
            if int(bn.num_batches_tracked) != before[i][2] + ncalls[tower_of[i]]:
                bad.append(f'{where}: num_batches_tracked {int(bn.num_batches_tracked)}, want {before[i][2] + ncalls[tower_of[i]]}')

        if step == 0:                       # the kernels add to .grad: start from random values of the gradients' size
            with torch.no_grad():
                for (conv, bn), lv in zip(mods, leaves):
                    for p, q in zip((conv.weight, bn.weight, bn.bias), lv):
                        p.grad.copy_(randn(p.shape, float(q.grad.square().mean().sqrt())))
        g0 = [tuple(p.grad.double() for p in (conv.weight, bn.weight, bn.bias)) for conv, bn in mods]
        pred.backward(torch.cat([gouts[(2, c)] for c in range(K)], dim=0))
        for c in reversed(range(K)):
            dyn[c].backward(gouts[(1, c)])
        rep.backward(gouts[(0, 0)])         # closes the step: the conv weight gradients are finalised
        torch.cuda.synchronize()

        for (tower, call), ref in grad_in_ref.items():
            got = (xs_dyn if tower == 1 else xs_pred)[call].grad
            note('grad_in', rel(got, ref), GRAD_TOL, f'step {step} {TOWERS[tower]} call {call}')
        for i, (conv, bn) in enumerate(mods):
            where = f'step {step} {TOWERS[tower_of[i]]} layer {i - first[tower_of[i]]}'
            dw, dg, db = (p.grad.double() - p0 for p, p0 in zip((conv.weight, bn.weight, bn.bias), g0[i]))
            rw, rg, rb = (q.grad for q in leaves[i])
            if i == first[1]:               # the dynamics' first conv: hidden-state and action input channels apart
                note('dW', rel(dw[:, :128], rw[:, :128]), GRAD_TOL, where)
                note('dW_action', rel(dw[:, 128:], rw[:, 128:]), GRAD_TOL, where)
            else:
                note('dW', rel(dw, rw), GRAD_TOL, where)
            note('dgamma', rel(dg, rg), GRAD_TOL, where)
            note('dbeta', rel(db, rb), GRAD_TOL, where)
        del rep, dyn, pred, outs, grad_in_ref, leaves
    del eng, net
    torch.cuda.empty_cache()
    return worst, bad


@pytest.mark.gpu
@pytest.mark.parametrize('case', list(CASES))
def test_every_layer_against_float64_on_the_kernels_own_tensors(case):
    worst, bad = run_case(case)
    print(f'\n{case}: ' + ', '.join(f'{k} {v:.3g} ({where})' for k, (v, where) in worst.items()))
    assert not bad, '\n'.join(bad[:40])


@pytest.mark.gpu
def test_stacked_debug_view_equals_separate_calls():
    """mz_train_debug_view of prediction calls that ran stacked returns the stacked buffers' rows of that call: the
    same bits (input, raw conv outputs, activations, batch statistics of every layer) a separate forward of the call
    stores."""
    import copy
    import muzero_b200 as mz
    from muzero_b200 import train_engine
    torch.manual_seed(7)
    K, B = 3, 32                                      # 32 * 100 rows per call: a multiple of 128
    net = mz.MuZeroBoardGameNet((9, 9, 9), 82, 2, 128).cuda().train()
    twin = copy.deepcopy(net)
    gen = torch.Generator(device='cuda').manual_seed(8)
    obs = torch.rand((B, 9, 9, 9), device='cuda', generator=gen)
    hids = [torch.rand((B, 128, 9, 9), device='cuda', generator=gen) * (k + 1) for k in range(K)]
    got = []
    for model, stacked in ((net, True), (twin, False)):
        eng = train_engine.engine_for(model, B, 5)
        assert eng.max_stacked_calls >= K
        rep = train_engine.tower(eng, 0, obs)
        if stacked:
            out = train_engine.prediction_calls(eng, hids)
            assert eng.calls[2] == K
        else:
            out = torch.cat([train_engine.tower(eng, 2, x) for x in hids], dim=0)
        torch.cuda.synchronize()
        got.append([[eng.debug_view(2, c, 0, 0)] + [eng.debug_view(2, c, l, k) for l in range(4) for k in (1, 2, 3)]
                    for c in range(K)])
        out.backward(torch.ones_like(out))
        rep.backward(torch.zeros_like(rep))           # closes the step
        torch.cuda.synchronize()
    for c in range(K):
        for k, (a, b) in enumerate(zip(got[0][c], got[1][c])):
            assert torch.equal(a, b), (c, k)
        assert float(got[0][c][2].abs().sum()) > 0    # not two empty buffers
