"""MuZero networks: the reference's constructors, state_dict keys and
``initial_inference`` / ``recurrent_inference`` signatures, with inference
running through the hand-written sm_100a kernels behind the C ABI.

Reference interface mirrored here (michaelnny/muzero):
  network.py:25-30    NetworkOutputs
  network.py:49-137   MuZeroNet (initial_inference / recurrent_inference)
  network.py:236-267  MuZeroMLPNet(input_shape, num_actions, num_planes, value_support_size,
                                   reward_support_size, hidden_dim)
  network.py:501-537  MuZeroAtariNet(input_shape, num_actions, num_res_blocks, num_planes,
                                     value_support_size, reward_support_size)
  network.py:540-574  MuZeroBoardGameNet(input_shape, num_actions, num_res_blocks, num_planes)

The torch modules below exist to (a) own the parameters under the reference's
state_dict key names, so its checkpoints load unchanged and autograd training
(``represent`` / ``dynamics`` / ``prediction``) works, and (b) be the source the
engine repacks its weights from.  Inference never runs through them: there is
no eager fallback — without CUDA and the built library the inference methods
raise.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import NamedTuple, Optional, Tuple

import numpy as np
import torch
import torch.nn.functional as F
from torch import nn

from . import _lib


class NetworkOutputs(NamedTuple):
    hidden_state: np.ndarray
    reward: float
    pi_probs: np.ndarray
    value: float


class StackedFrames(NamedTuple):
    """An Atari observation batch in the form it is born in (gym_env.py:306-313, StackFrameAndAction.observation):
    k uint8 frames and the values of the k constant action planes, instead of their float32 expansion [B, 2k, H, W]
    (which is what the reference uploads: 4x the bytes).  Accepted wherever a MuZeroAtariNet takes observations."""
    frames: 'torch.Tensor'          # uint8   [B, k, H, W]
    planes: 'torch.Tensor'          # float32 [B, k]   value of each broadcast action plane, (action + 1) / num_actions

    def expand(self) -> 'torch.Tensor':
        """The float32 observation [B, 2k, H, W] the reference would build."""
        f = torch.as_tensor(self.frames)
        p = torch.as_tensor(self.planes).to(torch.float32)
        return torch.cat([f.to(torch.float32), p[:, :, None, None].expand(-1, -1, f.shape[2], f.shape[3])], dim=1)


# ---------------------------------------------------------------------------
# parameter containers (attribute names == reference state_dict keys)
# ---------------------------------------------------------------------------
def _two_layer(i: int, h: int, o: int) -> nn.Sequential:
    return nn.Sequential(nn.Linear(i, h), nn.ReLU(), nn.Linear(h, o))


def _conv3(i: int, o: int, stride: int = 1) -> nn.Conv2d:
    return nn.Conv2d(i, o, kernel_size=3, stride=stride, padding=1, bias=False)


def _conv_bn_relu(i: int, o: int) -> nn.Sequential:
    return nn.Sequential(_conv3(i, o), nn.BatchNorm2d(o), nn.ReLU())


def _head(planes: int, mid: int, hw: int, out: int) -> nn.Sequential:
    return nn.Sequential(nn.Conv2d(planes, mid, kernel_size=1, stride=1, bias=False), nn.BatchNorm2d(mid),
                         nn.ReLU(), nn.Flatten(), nn.Linear(mid * hw, out))


class _Holder(nn.Module):
    """Plain namespace module; children are attached by the builders below."""


class ResNetBlock(nn.Module):
    def __init__(self, planes: int) -> None:
        super().__init__()
        self.conv_block1 = _conv_bn_relu(planes, planes)
        self.conv_block2 = nn.Sequential(_conv3(planes, planes), nn.BatchNorm2d(planes))

    def forward(self, x):
        return F.relu(self.conv_block2(self.conv_block1(x)) + x)


def _tower(planes: int, n: int) -> nn.Sequential:
    return nn.Sequential(*[ResNetBlock(planes) for _ in range(n)])


def _kaiming(net: nn.Module) -> None:
    """network.py:33-46, same module traversal order (so the same seed gives the same weights)."""
    for m in net.modules():
        if isinstance(m, (nn.Conv2d, nn.Linear)):
            nn.init.kaiming_normal_(m.weight, nonlinearity='relu')
            if m.bias is not None:
                nn.init.zeros_(m.bias)


def action_planes(action: torch.Tensor, num_actions: int, h: int, w: int) -> torch.Tensor:
    """The action encoding the reference's DynamicsConvNet actually feeds its first conv
    (network.py:440-444).  With the [B, 1] action every caller passes (mcts.py:383-384,
    pipeline.py:581) the one-hot is [B, 1, A]; ``repeat_interleave(h*w, dim=1)`` then ``reshape``
    to [B, A, h, w] yields a comb, not constant planes: flat element f of the A*h*w block is 1
    iff f % A == action.  Bit-for-bit the same tensor, built directly."""
    b = action.shape[0]
    f = torch.arange(num_actions * h * w, device=action.device)
    return ((f % num_actions)[None, :] == action.reshape(b, 1).long()).to(torch.float32).reshape(b, num_actions, h, w)


_MOMENTUM_WEIGHTS = {}


def _momentum_weights(calls: int, m: float, dtype, device) -> torch.Tensor:
    """[calls, 1] weights m (1 - m)^(calls - 1 - k) of the calls' statistics in the running average after `calls` updates.
    Cached per device: a CUDA-graph capture must not see the host-to-device copy that builds it (the learner runs three
    eager iterations before it captures)."""
    key = (calls, float(m), dtype, str(device))
    w = _MOMENTUM_WEIGHTS.get(key)
    if w is None:
        w = torch.tensor([m * (1.0 - m) ** (calls - 1 - k) for k in range(calls)], dtype=dtype, device=device)[:, None]
        _MOMENTUM_WEIGHTS[key] = w
    return w


class _HeadConv1x1(torch.autograd.Function):
    """y = conv2d(x, w) for a 1x1 kernel with at most four output channels on the kernels of csrc/optim.cu
    (mz_head_conv_forward / _backward): three passes over the input instead of cuDNN's transposes + split-K route."""

    @staticmethod
    def forward(ctx, x, w):
        n, c, h, wd = x.shape
        m = w.shape[0]
        x = x.contiguous()
        wm = w.reshape(m, c).contiguous()
        y = torch.empty((n, m, h, wd), dtype=torch.float32, device=x.device)
        _lib.check(_lib.lib().mz_head_conv_forward(x.data_ptr(), wm.data_ptr(), y.data_ptr(), n, c, h * wd, m, _lib.current_stream()))
        ctx.save_for_backward(x, wm)
        ctx.wshape = tuple(w.shape)
        return y

    @staticmethod
    def backward(ctx, dy):
        x, wm = ctx.saved_tensors
        n, c, h, wd = x.shape
        m = wm.shape[0]
        dy = dy.contiguous()
        dx = torch.empty_like(x)
        dw = torch.empty_like(wm)
        scratch = torch.empty(_lib.lib().mz_head_conv_scratch_bytes(n, c, m), dtype=torch.uint8, device=x.device)
        _lib.check(_lib.lib().mz_head_conv_backward(x.data_ptr(), wm.data_ptr(), dy.data_ptr(), dx.data_ptr(), dw.data_ptr(),
                                                    scratch.data_ptr(), n, c, h * wd, m, _lib.current_stream()))
        return dx, dw.view(ctx.wshape)


def _head_conv(x: torch.Tensor, weight: torch.Tensor) -> torch.Tensor:
    if (x.is_cuda and x.dtype == torch.float32 and weight.shape[0] <= 4 and weight.shape[1] <= 256
            and tuple(weight.shape[2:]) == (1, 1)):
        return _HeadConv1x1.apply(x, weight)
    return F.conv2d(x, weight)


class _HeadTail(torch.autograd.Function):
    """BatchNorm2d (train mode, per-call batch statistics) + ReLU + Flatten + Linear of a head over `calls` stacked calls on
    the kernels of csrc/optim.cu (mz_head_tail_forward / _backward): six launches instead of ~33 small PyTorch kernels."""

    @staticmethod
    def forward(ctx, y, gamma, beta, weight, bias, running_mean, running_var, calls, eps, momentum):
        tb, mid, h, w = y.shape
        o, j = weight.shape
        y = y.contiguous()
        dev = y.device
        saved = torch.empty((calls, mid, 3), dtype=torch.float32, device=dev)
        z = torch.empty((tb, j), dtype=torch.float32, device=dev)
        out = torch.empty((tb, o), dtype=torch.float32, device=dev)
        wc = weight.contiguous()
        _lib.check(_lib.lib().mz_head_tail_forward(y.data_ptr(), gamma.data_ptr(), beta.data_ptr(), wc.data_ptr(), bias.data_ptr(),
                                                   running_mean.data_ptr(), running_var.data_ptr(), saved.data_ptr(), z.data_ptr(),
                                                   out.data_ptr(), calls, tb // calls, mid, h * w, o, eps, momentum,
                                                   _lib.current_stream()))
        ctx.save_for_backward(y, gamma, wc, saved, z)
        ctx.calls = calls
        return out

    @staticmethod
    def backward(ctx, dout):
        y, gamma, wc, saved, z = ctx.saved_tensors
        tb, mid, h, w = y.shape
        o, j = wc.shape
        dev = y.device
        dout = dout.contiguous()
        dzr = torch.empty_like(z)
        sums = torch.empty((ctx.calls, mid, 2), dtype=torch.float32, device=dev)
        dy = torch.empty_like(y)
        dgamma = torch.empty_like(gamma)
        dbeta = torch.empty_like(gamma)
        _lib.check(_lib.lib().mz_head_tail_backward(dout.data_ptr(), y.data_ptr(), gamma.data_ptr(), wc.data_ptr(), saved.data_ptr(),
                                                    z.data_ptr(), dzr.data_ptr(), sums.data_ptr(), dy.data_ptr(), dgamma.data_ptr(),
                                                    dbeta.data_ptr(), ctx.calls, tb // ctx.calls, mid, h * w, o, _lib.current_stream()))
        # the Linear layer's own gradients: one small GEMM and one column sum
        return dy, dgamma, dbeta, dout.t().mm(z), dout.sum(0), None, None, None, None, None


def _head_after_conv(head: nn.Sequential, y: torch.Tensor, calls: int) -> torch.Tensor:
    """BatchNorm (per-call statistics) + ReLU + Flatten + Linear of a head on its 1x1 convolution's output for `calls`
    stacked calls."""
    _, bn, _, _, lin = head
    tb, mid, h, w = y.shape
    b = tb // calls
    if (y.is_cuda and bn.training and y.dtype == torch.float32 and mid <= 4 and mid * h * w <= 1024 and lin.out_features <= 128
            and b >= 2 and lin.bias is not None and bn.momentum is not None and os.environ.get('MZ_HEAD_TAIL', '1') != '0'):
        out = _HeadTail.apply(y, bn.weight, bn.bias, lin.weight, lin.bias, bn.running_mean, bn.running_var, calls, bn.eps, bn.momentum)
        with torch.no_grad():
            bn.num_batches_tracked += calls
        return out
    y = y.reshape(calls, b, mid, h * w).transpose(1, 2)                  # [calls, mid, B, hw] (a view for mid == 1)
    if bn.training:
        with torch.no_grad():
            var, mean = torch.var_mean(y, dim=(2, 3), unbiased=False)      # [calls, mid]
            n = b * h * w
            m = bn.momentum
            # running <- (1 - m) running + m stat, applied once per call in call order
            coef = _momentum_weights(calls, m, y.dtype, y.device)
            bn.running_mean.mul_((1.0 - m) ** calls).add_((coef * mean).sum(0))
            bn.running_var.mul_((1.0 - m) ** calls).add_((coef * var).sum(0) * (n / (n - 1.0)))
            bn.num_batches_tracked += calls
        z = F.instance_norm(y, None, None, bn.weight, bn.bias, True, 0.0, bn.eps)
    else:
        z = F.batch_norm(y.transpose(1, 2).reshape(tb, mid, h * w), bn.running_mean, bn.running_var, bn.weight, bn.bias, False,
                         0.0, bn.eps).view(calls, b, mid, h * w).transpose(1, 2)
    z = F.relu(z).transpose(1, 2).reshape(tb, mid * h * w)
    return lin(z)


def head_over_calls(head: nn.Sequential, x: torch.Tensor, calls: int) -> torch.Tensor:
    """One of the 1x1-conv heads (``_head``: conv, BatchNorm2d, ReLU, Flatten, Linear) applied to the inputs of ``calls``
    separate forward calls stacked along the batch axis (call-major, [calls * B, C, h, w]) -- the SAME arithmetic as
    ``calls`` invocations of ``head`` in train mode: every call keeps its own BatchNorm batch statistics (the stack is
    normalised per (call, channel) over that call's B * h * w values, which is what instance normalisation of the
    [calls, mid, B, h*w] view computes), and the running statistics receive the calls' updates in order.  One launch per
    layer instead of one per call: at batch 128 the K-step unroll is bound by kernel count, not by arithmetic."""
    return _head_after_conv(head, _head_conv(x, head[0].weight), calls)


def heads_over_calls(heads, x: torch.Tensor, calls: int):
    """Several heads that read the SAME stacked input (the policy and value heads on the prediction tower's output): their
    1x1 convolutions run as one convolution with the weights stacked along the output channels -- one pass over the
    input forward, one input gradient backward instead of one per head and an addition -- then each head continues on
    its own channels."""
    mids = [h[0].weight.shape[0] for h in heads]
    y = _head_conv(x, torch.cat([h[0].weight for h in heads], dim=0))
    outs, at = [], 0
    for h, mid in zip(heads, mids):
        outs.append(_head_after_conv(h, y[:, at:at + mid], calls))
        at += mid
    return outs


def normalize_hidden_state(h: torch.Tensor) -> torch.Tensor:
    """util.py:31-36 (torch, used by the autograd/training path only)."""
    lo = h.min(dim=1, keepdim=True)[0]
    hi = h.max(dim=1, keepdim=True)[0]
    return (h - lo) / (hi - lo + 1e-8)


# ---------------------------------------------------------------------------
# engine-backed base class
# ---------------------------------------------------------------------------
class MuZeroNet(nn.Module):
    kind = None            # _lib.MZ_NET_*
    hidden_shape: Tuple[int, ...] = ()

    def __init__(self, num_actions: int, value_support_size: int = 31, reward_support_size: int = 31) -> None:
        super().__init__()
        self.num_actions = num_actions
        self.value_support_size = value_support_size
        self.reward_support_size = reward_support_size
        self._engs = {}           # instance -> dict(handle, arena tensor, version stamp, device, max_batch)
        self._weight_epoch = 0    # bumped by mark_weights_updated(): updates the version counters cannot see

    @property
    def mse_loss_for_value(self):
        return self.value_support_size == 1

    @property
    def mse_loss_for_reward(self):
        return self.reward_support_size == 1

    # -- engine -------------------------------------------------------------
    def _net_config(self) -> _lib.NetConfig:
        raise NotImplementedError

    def mark_weights_updated(self) -> None:
        """Tell the engine that parameters / buffers changed behind autograd's back.

        ``_stamp`` reads the tensors' ``_version`` counters, which a CUDA-graph replay (the graphed training
        step of ``training.DataParallelLearner``) or a raw-pointer write never advances: without this call the
        next search would keep the engine (and the captured search graphs) packed from the old weights."""
        self._weight_epoch += 1

    def _stamp(self):
        return (tuple(p._version for p in self.parameters()), tuple(b._version for b in self.buffers()),
                self.training, self._weight_epoch)

    def engine(self, max_batch: int = 1, instance: int = 0):
        """The ``mz_net`` handle for the current weights (rebuilt when they changed).

        ``instance`` selects one of several independent engines over the same weights (each owns its
        activation buffers), so that two searches can be in flight at once (mcts.PipelinedSearchPlan)."""
        dev = next(self.parameters()).device
        if dev.type != 'cuda':
            raise RuntimeError('muzero_b200 inference runs on CUDA only (no CPU fallback): move the network to a '
                               'cuda device first')
        stamp = self._stamp()
        e = self._engs.get(instance)
        if e is not None and e['stamp'] == stamp and e['device'] == dev and e['max_batch'] >= max_batch:
            return e
        self.release_engine(instance)
        lib = _lib.lib()
        with torch.cuda.device(dev):
            _lib.check(lib.mz_device_check(dev.index or 0, None, None))
            cfg = self._net_config()
            nbytes = C.c_size_t()
            _lib.check(lib.mz_net_arena_bytes(C.byref(cfg), max_batch, C.byref(nbytes)))
            arena = torch.empty(nbytes.value + 256, dtype=torch.uint8, device=dev)
            base = (arena.data_ptr() + 255) // 256 * 256
            tensors = [t.detach().to(torch.float32).contiguous() for t in self._engine_tensors()]
            ptrs = (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])
            handle = C.c_void_p()
            torch.cuda.synchronize(dev)
            _lib.check(lib.mz_net_create(C.byref(cfg), ptrs, len(tensors), max_batch, base, nbytes.value,
                                         C.byref(handle)))
            hb = C.c_int32()
            _lib.check(lib.mz_net_hidden_bytes(C.byref(cfg), C.byref(hb)))
        self._engs[instance] = dict(handle=handle, arena=arena, stamp=stamp, device=dev, max_batch=max_batch,
                                    hidden_bytes=hb.value)
        return self._engs[instance]

    def release_engine(self, instance: Optional[int] = None) -> None:
        for k in ([instance] if instance is not None else list(self._engs)):
            e = self._engs.pop(k, None)
            if e is not None:
                _lib.lib().mz_net_destroy(e['handle'])

    def __del__(self):
        try:
            self.release_engine()
        except Exception:
            pass

    def _engine_tensors(self):
        """float32 tensors handed to mz_net_create, in state_dict order."""
        return [v for k, v in self.state_dict().items() if not k.endswith('num_batches_tracked')]

    @property
    def hidden_bytes(self) -> int:
        cfg = self._net_config()
        hb = C.c_int32()
        _lib.check(_lib.lib().mz_net_hidden_bytes(C.byref(cfg), C.byref(hb)))
        return hb.value

    # -- batched device API (additive) ---------------------------------------
    def new_hidden(self, n: int) -> torch.Tensor:
        """Uninitialised array of ``n`` hidden-state slots in the engine's layout."""
        dev = next(self.parameters()).device
        return torch.zeros((n, self.hidden_bytes), dtype=torch.uint8, device=dev)

    @torch.no_grad()
    def initial_inference_batch(self, obs: torch.Tensor, hidden_out: Optional[torch.Tensor] = None,
                                dst_index: Optional[torch.Tensor] = None):
        """``initial_inference`` for a batch, all outputs stay on the device.

        Returns (hidden slots [u8, engine layout], pi_probs f32[B,A], value f32[B])."""
        frames = isinstance(obs, StackedFrames)
        b = (obs.frames if frames else obs).shape[0]
        e = self.engine(b)
        dev = e['device']
        if hidden_out is None:
            hidden_out = self.new_hidden(b)
        pi = torch.empty((b, self.num_actions), dtype=torch.float32, device=dev)
        value = torch.empty((b,), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            if frames:
                f = torch.as_tensor(obs.frames).to(device=dev, dtype=torch.uint8).contiguous()
                pl = torch.as_tensor(obs.planes).to(device=dev, dtype=torch.float32).contiguous()
                _lib.check(_lib.lib().mz_net_initial_frames(e['handle'], b, _lib.ptr(f), _lib.ptr(pl),
                                                            _lib.ptr(hidden_out), _lib.ptr(dst_index), _lib.ptr(pi),
                                                            _lib.ptr(value), _lib.current_stream()))
            else:
                obs = obs.to(device=dev, dtype=torch.float32).reshape(b, -1).contiguous()
                _lib.check(_lib.lib().mz_net_initial(e['handle'], b, _lib.ptr(obs), _lib.ptr(hidden_out),
                                                     _lib.ptr(dst_index), _lib.ptr(pi), _lib.ptr(value),
                                                     _lib.current_stream()))
        return hidden_out, pi, value

    @torch.no_grad()
    def recurrent_inference_batch(self, hidden_in: torch.Tensor, action: torch.Tensor,
                                  src_index: Optional[torch.Tensor] = None,
                                  hidden_out: Optional[torch.Tensor] = None,
                                  dst_index: Optional[torch.Tensor] = None, want_policy: bool = True):
        """``recurrent_inference`` for a batch of (slot, action) pairs on the device.

        Returns (hidden slots, reward f32[B], pi_probs f32[B,A] or None, value f32[B])."""
        b = action.shape[0]
        e = self.engine(b)
        dev = e['device']
        action = action.to(device=dev, dtype=torch.int32).reshape(b).contiguous()
        if hidden_out is None:
            hidden_out = self.new_hidden(b)
        reward = torch.empty((b,), dtype=torch.float32, device=dev)
        value = torch.empty((b,), dtype=torch.float32, device=dev)
        pi = torch.empty((b, self.num_actions), dtype=torch.float32, device=dev) if want_policy else None
        with torch.cuda.device(dev):
            _lib.check(_lib.lib().mz_net_recurrent(e['handle'], b, _lib.ptr(hidden_in), _lib.ptr(src_index),
                                                   _lib.ptr(action), _lib.ptr(hidden_out), _lib.ptr(dst_index),
                                                   _lib.ptr(reward), _lib.ptr(value), _lib.ptr(pi),
                                                   _lib.current_stream()))
        return hidden_out, reward, pi, value

    # -- engine layout <-> reference layout ----------------------------------
    def hidden_to_reference(self, slots: torch.Tensor) -> torch.Tensor:
        """Engine slots [n, hidden_bytes] -> float32 [n, *hidden_shape] (reference layout)."""
        raise NotImplementedError

    def hidden_from_reference(self, h: torch.Tensor) -> torch.Tensor:
        raise NotImplementedError

    # -- the reference's single-observation API (network.py:62-111) ----------
    @torch.no_grad()
    def initial_inference(self, x: torch.Tensor) -> NetworkOutputs:
        hidden, pi, value = self.initial_inference_batch(x)
        h = self.hidden_to_reference(hidden)[0]
        return NetworkOutputs(hidden_state=h.cpu().numpy(), reward=0.0, pi_probs=pi[0].cpu().numpy(),
                              value=value[0].cpu().item())

    @torch.no_grad()
    def recurrent_inference(self, hidden_state: torch.Tensor, action: torch.Tensor) -> NetworkOutputs:
        dev = next(self.parameters()).device
        slots = self.hidden_from_reference(hidden_state.to(device=dev, dtype=torch.float32))
        hidden, reward, pi, value = self.recurrent_inference_batch(slots, action.reshape(-1))
        h = self.hidden_to_reference(hidden)[0]
        return NetworkOutputs(hidden_state=h.cpu().numpy(), reward=reward[0].cpu().item(),
                              pi_probs=pi[0].cpu().numpy(), value=value[0].cpu().item())

    # -- autograd path for training (network.py:113-124) ---------------------
    def represent(self, x: torch.Tensor) -> torch.Tensor:
        raise NotImplementedError

    def dynamics(self, hidden_state: torch.Tensor, action: torch.Tensor):
        raise NotImplementedError

    def prediction(self, hidden_state: torch.Tensor):
        raise NotImplementedError


# ---------------------------------------------------------------------------
# MLP family (network.py:140-267)
# ---------------------------------------------------------------------------
class MuZeroMLPNet(MuZeroNet):
    kind = _lib.MZ_NET_MLP

    def __init__(self, input_shape: Tuple, num_actions: int, num_planes: int = 256, value_support_size: int = 31,
                 reward_support_size: int = 31, hidden_dim: int = 64) -> None:
        super().__init__(num_actions, value_support_size, reward_support_size)
        self.input_shape = tuple(input_shape)
        self.num_planes, self.hidden_dim = num_planes, hidden_dim
        self.hidden_shape = (hidden_dim,)
        # construction order == network.py:249-253 so equal seeds give equal weights
        self.represent_net = _Holder()
        self.represent_net.net = _two_layer(math.prod(input_shape), num_planes, hidden_dim)
        self.dynamics_net = _Holder()
        self.dynamics_net.transition_net = _two_layer(hidden_dim + num_actions, num_planes, hidden_dim)
        self.dynamics_net.reward_net = _two_layer(hidden_dim, num_planes, reward_support_size)
        self.prediction_net = _Holder()
        self.prediction_net.policy_net = _two_layer(hidden_dim, num_planes, num_actions)
        self.prediction_net.value_net = _two_layer(hidden_dim, num_planes, value_support_size)

    def _net_config(self) -> _lib.NetConfig:
        return _lib.NetConfig(kind=self.kind, in_channels=math.prod(self.input_shape), in_h=1, in_w=1,
                              num_actions=self.num_actions, num_planes=self.num_planes, num_res_blocks=0,
                              hidden_dim=self.hidden_dim, value_support=self.value_support_size,
                              reward_support=self.reward_support_size)

    def hidden_to_reference(self, slots):
        return slots.view(torch.float32).reshape(slots.shape[0], self.hidden_dim)

    def hidden_from_reference(self, h):
        return h.reshape(-1, self.hidden_dim).contiguous().view(torch.uint8)

    def represent(self, x):
        return normalize_hidden_state(self.represent_net.net(x.reshape(x.shape[0], -1)))

    def dynamics(self, hidden_state, action):
        onehot = torch.zeros((hidden_state.shape[0], self.num_actions), dtype=torch.float32,
                             device=hidden_state.device).scatter_(1, action, 1.0)
        h = self.dynamics_net.transition_net(torch.cat([hidden_state, onehot], dim=1))
        return normalize_hidden_state(h), self.dynamics_net.reward_net(h)

    def prediction(self, hidden_state):
        return self.prediction_net.policy_net(hidden_state), self.prediction_net.value_net(hidden_state)


# ---------------------------------------------------------------------------
# ResNet families (network.py:273-574)
# ---------------------------------------------------------------------------
class _ConvNet(MuZeroNet):
    latent_hw: Tuple[int, int] = (0, 0)

    def _build_dyn_pred(self, planes, blocks, h, w, num_actions, reward_support, value_support):
        self.dynamics_net = _Holder()
        self.dynamics_net.num_actions = num_actions
        self.dynamics_net.conv_block = _conv_bn_relu(planes + num_actions, planes)
        self.dynamics_net.res_blocks = _tower(planes, blocks)
        self.dynamics_net.reward_head = _head(planes, 1, h * w, reward_support)
        self.prediction_net = _Holder()
        self.prediction_net.res_blocks = _tower(planes, blocks)
        self.prediction_net.policy_net = _head(planes, 2, h * w, num_actions)
        self.prediction_net.value_net = _head(planes, 1, h * w, value_support)

    def _net_config(self) -> _lib.NetConfig:
        c, h, w = self.input_shape
        return _lib.NetConfig(kind=self.kind, in_channels=c, in_h=h, in_w=w, num_actions=self.num_actions,
                              num_planes=self.num_planes, num_res_blocks=self.num_res_blocks, hidden_dim=0,
                              value_support=self.value_support_size, reward_support=self.reward_support_size)

    def _engine_tensors(self):
        if self.training:
            raise RuntimeError('engine inference folds BatchNorm running statistics: call .eval() first '
                               '(self-play always does, pipeline.py:79-80)')
        return super()._engine_tensors()

    # engine layout: fp16 planes of 8 channels, [Cp/8][(H+pad)*(W+pad)][8], pad = grid_pad, Cp = padded_planes
    # (see csrc/conv.cu)
    @property
    def padded_planes(self) -> int:
        """Channels of a hidden-state slot: num_planes rounded up to a multiple of 32 (the kernels' minimum tile
        width; the reference's ResNet Tic-Tac-Toe variant has 16 planes, config.py:126-127).  Extra channels are 0."""
        return max(32, (self.num_planes + 31) // 32 * 32)

    def hidden_to_reference(self, slots):
        h, w = self.latent_hw
        c, cp = self.num_planes, self.padded_planes
        pad = self.grid_pad
        x = slots.view(torch.float16).reshape(slots.shape[0], cp // 8, h + pad, w + pad, 8)[:, :, :h, :w, :]
        return x.permute(0, 1, 4, 2, 3).reshape(slots.shape[0], cp, h, w)[:, :c].to(torch.float32).contiguous()

    @property
    def grid_pad(self) -> int:
        """0: boards stored without halo (the conv kernel masks the edge taps); 1: the padded (H+1)x(W+1) layout
        (MZ_CONV_PAD=1).  Read off the engine's slot size so that this module never disagrees with the library."""
        h, w = self.latent_hw
        return 1 if self.hidden_bytes == (h + 1) * (w + 1) * self.padded_planes * 2 else 0

    def hidden_from_reference(self, hid):
        h, w = self.latent_hw
        c, cp = self.num_planes, self.padded_planes
        hid = hid.reshape(-1, c // 8, 8, h, w)
        pad = self.grid_pad
        out = torch.zeros((hid.shape[0], cp // 8, h + pad, w + pad, 8), dtype=torch.float16, device=hid.device)
        out[:, :c // 8, :h, :w, :] = hid.permute(0, 1, 3, 4, 2).to(torch.float16)
        return out.reshape(hid.shape[0], -1).view(torch.uint8)

    # -- training: the towers run on the hand-written kernels of csrc/train.cu where they apply (train_engine.py) ------
    unroll_hint = 5          # calc_loss tells the engine how many dynamics / prediction calls a step makes

    def _train_engine(self, x, begin: bool = False):
        if not (self.training and x.is_cuda):
            return None
        from . import train_engine
        eng = train_engine.engine_for(self, x.shape[0], self.unroll_hint)
        if eng is None or not (begin or eng.active):
            return None
        return eng

    def dynamics(self, hidden_state, action):
        eng = self._train_engine(hidden_state)
        if eng is not None:
            from . import train_engine
            hs, normalized = train_engine.tower(eng, 1, hidden_state, action, mode=2)
            return normalized, self.dynamics_net.reward_head(hs)
        b, c, h, w = hidden_state.shape
        planes = action_planes(action, self.num_actions, h, w).to(hidden_state.dtype)
        x = torch.cat([hidden_state, planes], dim=1)
        hs = self.dynamics_net.res_blocks(self.dynamics_net.conv_block(x))
        return normalize_hidden_state(hs), self.dynamics_net.reward_head(hs)

    def dynamics_tower(self, hidden_state, action):
        """The dynamics tower's raw output (before normalisation and the reward head) on the autograd modules."""
        b, c, h, w = hidden_state.shape
        planes = action_planes(action, self.num_actions, h, w).to(hidden_state.dtype)
        return self.dynamics_net.res_blocks(self.dynamics_net.conv_block(torch.cat([hidden_state, planes], dim=1)))

    def prediction_tower(self, hidden_state):
        return self.prediction_net.res_blocks(hidden_state)

    def prediction(self, hidden_state):
        eng = self._train_engine(hidden_state)
        if eng is not None:
            from . import train_engine
            f = train_engine.tower(eng, 2, hidden_state)
        else:
            f = self.prediction_net.res_blocks(hidden_state)
        return self.prediction_net.policy_net(f), self.prediction_net.value_net(f)


class MuZeroBoardGameNet(_ConvNet):
    kind = _lib.MZ_NET_BOARD

    def __init__(self, input_shape: tuple, num_actions: int, num_res_blocks: int = 16, num_planes: int = 256) -> None:
        super().__init__(num_actions, 1, 1)
        c, h, w = input_shape
        self.input_shape = tuple(input_shape)
        self.num_planes, self.num_res_blocks = num_planes, num_res_blocks
        self.latent_hw = (h, w)
        self.hidden_shape = (num_planes, h, w)
        self.represent_net = _Holder()
        self.represent_net.conv_block = _conv_bn_relu(c, num_planes)
        self.represent_net.res_blocks = _tower(num_planes, num_res_blocks)
        self._build_dyn_pred(num_planes, num_res_blocks, h, w, num_actions, 1, 1)
        _kaiming(self)

    def represent(self, x):
        eng = self._train_engine(x, begin=True)
        if eng is not None:
            from . import train_engine
            return train_engine.tower(eng, 0, x, mode=1)
        return normalize_hidden_state(self.represent_net.res_blocks(self.represent_net.conv_block(x)))


class MuZeroAtariNet(_ConvNet):
    kind = _lib.MZ_NET_ATARI

    def __init__(self, input_shape: tuple, num_actions: int, num_res_blocks: int = 16, num_planes: int = 256,
                 value_support_size: int = 601, reward_support_size: int = 601) -> None:
        super().__init__(num_actions, value_support_size, reward_support_size)
        c, h, w = input_shape
        self.input_shape = tuple(input_shape)
        self.num_planes, self.num_res_blocks = num_planes, num_res_blocks
        self.latent_hw = (6, 6)              # hard-wired downstream of the representation, network.py:516-519
        self.hidden_shape = (num_planes, 6, 6)
        r = self.represent_net = _Holder()
        r.conv_1 = _conv3(c, 128, stride=2)                       # 96 -> 48
        r.res_blocks_1 = _tower(128, 2)
        r.conv_2 = _conv3(128, num_planes, stride=2)              # 48 -> 24
        r.res_blocks_2 = _tower(num_planes, 2)
        r.avg_pool_1 = nn.AvgPool2d(kernel_size=3, stride=2, padding=1)   # 24 -> 12
        r.res_blocks_3 = _tower(num_planes, 2)
        r.avg_pool_2 = nn.AvgPool2d(kernel_size=3, stride=2, padding=1)   # 12 -> 6
        self._build_dyn_pred(num_planes, num_res_blocks, 6, 6, num_actions, reward_support_size, value_support_size)
        _kaiming(self)

    def represent(self, x):
        r = self.represent_net
        x = r.res_blocks_1(F.relu(r.conv_1(x)))
        x = r.res_blocks_2(F.relu(r.conv_2(x)))
        x = r.res_blocks_3(r.avg_pool_1(x))
        return normalize_hidden_state(r.avg_pool_2(x))
