"""Hand-written training path of the ResNet towers (csrc/train.cu) behind autograd (SURVEY.md 8 f-2).

The reference trains with plain PyTorch modules: ``calc_loss`` (pipeline.py:541-612) calls ``network.represent``,
``network.dynamics`` and ``network.prediction`` (network.py:113-124) and autograd + cuDNN do the rest.  Here the three
towers -- every 3x3 convolution with its train-mode BatchNorm, ReLU and residual connection, i.e. all but a rounding
error of the step's flops -- run as tcgen05 kernels forward AND backward; a tower is one ``torch.autograd.Function``
whose inputs / outputs are the float32 NCHW tensors the reference's modules exchange (optionally with the min-max
normalisation of ``normalize_hidden_state`` applied by the same pass, forward and backward), so ``calc_loss`` and
everything around it (the heads' BatchNorm / Linear, the losses, the 0.5 and 1/K gradient hooks) is unchanged.  The K
prediction calls of an unroll can run as ONE launch chain over the stacked hidden states (``prediction_calls``).

Parameter gradients are written by the kernels straight into ``p.grad`` (accumulated, like autograd's): BatchNorm
weights / biases during a tower's backward, convolution weights once per step after the representation tower's
backward -- the last tower backward of any step, since every other tower consumes its output.

Scope: ``MuZeroBoardGameNet`` with ``num_planes == 128`` on CUDA in train mode (BASELINE configs[2]/[4]); anything else
keeps the autograd modules.  ``MZ_TRAIN_NATIVE=0`` switches the kernels off.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref
from typing import Optional

import torch

from . import _lib


def _enabled() -> bool:
    return os.environ.get('MZ_TRAIN_NATIVE', '1') != '0'


def supported(network) -> bool:
    """The shapes csrc/train.cu is built for."""
    hw = getattr(network, 'latent_hw', (0, 0))
    return (getattr(network, 'kind', None) == _lib.MZ_NET_BOARD and getattr(network, 'num_planes', 0) == 128
            and 1 <= getattr(network, 'num_res_blocks', 0) <= 32 and network.num_actions <= 128
            and network.input_shape[0] <= 128 and 2 <= hw[0] and 2 <= hw[1] <= 62)


def _tower_modules(network):
    """(conv, bn) pairs in the order mz_train_bind expects."""
    out = []

    def block(seq):
        out.append((seq[0], seq[1]))

    r, d, p = network.represent_net, network.dynamics_net, network.prediction_net
    block(r.conv_block)
    for b in r.res_blocks:
        block(b.conv_block1)
        block(b.conv_block2)
    block(d.conv_block)
    for b in d.res_blocks:
        block(b.conv_block1)
        block(b.conv_block2)
    for b in p.res_blocks:
        block(b.conv_block1)
        block(b.conv_block2)
    return out


class TowerTrainEngine:
    """One ``mz_train`` handle: fixed batch size and unroll length, arena owned here."""

    def __init__(self, network, batch: int, unroll_steps: int) -> None:
        dev = next(network.parameters()).device
        assert dev.type == 'cuda', 'the training kernels need a CUDA device (there is no CPU fallback)'
        c, h, w = network.input_shape
        self.device, self.batch, self.unroll = dev, int(batch), int(unroll_steps)
        self.input_shape = (c, h, w)
        self.cfg = _lib.TrainConfig(in_channels=c, board_h=h, board_w=w, num_actions=network.num_actions,
                                    num_planes=network.num_planes, num_res_blocks=network.num_res_blocks,
                                    batch=self.batch, unroll_steps=self.unroll)
        nbytes = C.c_size_t()
        lib = _lib.lib()
        _lib.check(lib.mz_train_arena_bytes(C.byref(self.cfg), C.byref(nbytes)))
        with torch.cuda.device(dev):
            self.arena = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
            handle = C.c_void_p()
            _lib.check(lib.mz_train_create(C.byref(self.cfg), self.arena.data_ptr(), nbytes.value, C.byref(handle)))
        self.handle = handle
        self.modules = _tower_modules(network)
        nb = network.num_res_blocks
        n = [1 + 2 * nb, 1 + 2 * nb, 2 * nb]
        self.counters = [[bn.num_batches_tracked for _, bn in self.modules[sum(n[:k]):sum(n[:k + 1])]] for k in range(3)]
        mc = C.c_int32()
        _lib.check(lib.mz_train_stacked_calls(self.handle, C.byref(mc)))
        self.max_stacked_calls = int(mc.value)      # prediction-tower calls that may run as one launch chain
        self._bound = None
        self.calls = [0, 0, 0]
        self.active = False
        self.hidden_shape = (self.batch, network.num_planes, h, w)

    def __del__(self):
        try:
            if getattr(self, 'handle', None):
                _lib.lib().mz_train_destroy(self.handle)
                self.handle = None
        except Exception:       # noqa: BLE001 - interpreter shutdown
            pass

    # -- parameter pointers ---------------------------------------------------------------------------------------
    def _pointers(self):
        ptrs = []
        for conv, bn in self.modules:
            for p in (conv.weight, bn.weight, bn.bias):
                if p.grad is None:
                    p.grad = torch.zeros_like(p, memory_format=torch.contiguous_format)
            for t in (conv.weight, conv.weight.grad, bn.weight, bn.weight.grad, bn.bias, bn.bias.grad, bn.running_mean,
                      bn.running_var):
                if not t.is_contiguous():
                    raise RuntimeError('the training kernels take contiguous (NCHW) parameters and gradients; '
                                       'do not convert the network to channels_last')
                ptrs.append(t.data_ptr())
        return ptrs

    def bind_if_needed(self) -> None:
        ptrs = self._pointers()
        if ptrs != self._bound:
            arr = (C.c_void_p * len(ptrs))(*ptrs)
            _lib.check(_lib.lib().mz_train_bind(self.handle, arr, len(ptrs), _lib.current_stream()))
            self._bound = ptrs

    # -- one step ---------------------------------------------------------------------------------------------------
    def begin_step(self) -> None:
        if not torch.cuda.is_current_stream_capturing():
            self.bind_if_needed()
        _lib.check(_lib.lib().mz_train_begin_step(self.handle, _lib.current_stream()))
        self.calls = [0, 0, 0]
        self.active = True

    def end_step(self) -> None:
        _lib.check(_lib.lib().mz_train_end_step(self.handle, _lib.current_stream()))
        self.active = False

    def join(self) -> None:
        """The current stream waits for the handle's weight-gradient stream."""
        _lib.check(_lib.lib().mz_train_join(self.handle, _lib.current_stream()))

    def next_call(self, tower: int, n: int = 1) -> int:
        k = self.calls[tower]
        limit = 1 if tower == 0 else self.unroll
        if k + n > limit:
            raise RuntimeError(f'training engine built for {self.unroll} unroll steps: tower {tower} called {k + n} times '
                               'in one step')
        self.calls[tower] = k + n
        return k

    def forward(self, tower: int, call: int, x: torch.Tensor, action: Optional[torch.Tensor], raw: bool = True,
                norm: bool = False):
        """One tower call: the output [B, 128, H, W] (``raw``) and / or its min-max normalisation (``norm``, util.py:31-36)
        from the same pass.  Returns the tensor asked for, or the pair (raw, norm)."""
        out = torch.empty(self.hidden_shape, dtype=torch.float32, device=self.device) if raw else None
        out_n = torch.empty(self.hidden_shape, dtype=torch.float32, device=self.device) if norm else None
        _lib.check(_lib.lib().mz_train_tower_forward_calls(self.handle, tower, call, 1, _lib.ptr(x), _lib.ptr(action),
                                                           _lib.ptr(out), _lib.ptr(out_n), _lib.current_stream()))
        return (out, out_n) if (raw and norm) else (out if raw else out_n)

    def backward(self, tower: int, call: int, grad_out: Optional[torch.Tensor],
                 grad_norm: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        grad_in = torch.empty(self.hidden_shape, dtype=torch.float32, device=self.device) if tower != 0 else None
        _lib.check(_lib.lib().mz_train_tower_backward_calls(self.handle, tower, call, 1, _lib.ptr(grad_out), _lib.ptr(grad_norm),
                                                            _lib.ptr(grad_in), _lib.current_stream()))
        return grad_in

    def forward_calls(self, call: int, n: int, x: torch.Tensor) -> torch.Tensor:
        """n stacked prediction-tower calls (x [n * B, 128, H, W], call-major) as one launch chain."""
        out = torch.empty((n * self.batch,) + self.hidden_shape[1:], dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().mz_train_tower_forward_calls(self.handle, 2, call, n, _lib.ptr(x), None, _lib.ptr(out), None,
                                                           _lib.current_stream()))
        return out

    def backward_calls(self, call: int, n: int, grad_out: torch.Tensor) -> torch.Tensor:
        grad_in = torch.empty((n * self.batch,) + self.hidden_shape[1:], dtype=torch.float32, device=self.device)
        _lib.check(_lib.lib().mz_train_tower_backward_calls(self.handle, 2, call, n, _lib.ptr(grad_out), None, _lib.ptr(grad_in),
                                                            _lib.current_stream()))
        return grad_in

    def debug_view(self, tower: int, call: int, layer: int, which: int) -> torch.Tensor:
        """Float32 [B, C, H, W] copy of a saved tensor (which: 0 input, 1 raw conv output, 2 activated output) or the
        [128, 2] batch statistics (which = 3).  Parity tests only."""
        p, n, pr, fr = C.c_void_p(), C.c_size_t(), C.c_int32(), C.c_int32()
        _lib.check(_lib.lib().mz_train_debug_view(self.handle, tower, call, layer, which, C.byref(p), C.byref(n), C.byref(pr),
                                                  C.byref(fr)))
        off = p.value - self.arena.data_ptr()
        raw = self.arena[off:off + n.value]
        if which == 3:
            return raw.view(torch.float32).reshape(128, 2).clone()
        _, h, w = self.input_shape
        planes = raw.view(torch.float16).reshape(-1, pr.value, 8)[:, fr.value:fr.value + self.batch * (h + 1) * (w + 1)]
        g = planes.shape[0]
        x = planes.reshape(g, self.batch, h + 1, w + 1, 8)[:, :, :h, :w]
        return x.permute(1, 0, 4, 2, 3).reshape(self.batch, g * 8, h, w).float()


_ENGINES = weakref.WeakKeyDictionary()       # network -> {(batch, device): engine}; engines hold no reference to it


class _Tower(torch.autograd.Function):
    """y = tower(x[, action]); ``anchor`` (a tower parameter) makes the output require grad when x does not.
    mode 0: the raw output; 1: its min-max normalisation only (representation); 2: the pair (raw, normalised) (dynamics:
    the reward head reads the raw output, the next step the normalised one)."""

    @staticmethod
    def forward(ctx, x, anchor, eng, tower, call, action, mode):
        ctx.eng, ctx.tower, ctx.call, ctx.mode = eng, tower, call, mode
        ctx.set_materialize_grads(False)
        return eng.forward(tower, call, x, action, raw=mode != 1, norm=mode != 0)

    @staticmethod
    def backward(ctx, *grads):
        eng = ctx.eng
        if ctx.mode == 0:
            g_raw, g_norm = grads[0], None
        elif ctx.mode == 1:
            g_raw, g_norm = None, grads[0]
        else:
            g_raw, g_norm = grads
        if g_raw is None and g_norm is None:         # nothing downstream used this call: its gradient is zero
            g_raw = torch.zeros(eng.hidden_shape, dtype=torch.float32, device=eng.device)
        grad_in = eng.backward(ctx.tower, ctx.call, None if g_raw is None else g_raw.contiguous(),
                               None if g_norm is None else g_norm.contiguous())
        if ctx.tower == 0:
            eng.end_step()          # every other tower's backward has run: the conv weight gradients are complete
        return grad_in, None, None, None, None, None, None


class _PredictionCalls(torch.autograd.Function):
    """The prediction tower on n stacked hidden states (n forward calls of the reference) as one launch chain."""

    @staticmethod
    def forward(ctx, x, anchor, eng, call, n):
        ctx.eng, ctx.call, ctx.n = eng, call, n
        return eng.forward_calls(call, n, x)

    @staticmethod
    def backward(ctx, grad_out):
        return ctx.eng.backward_calls(ctx.call, ctx.n, grad_out.contiguous()), None, None, None, None


def prediction_calls(eng: TowerTrainEngine, hiddens) -> torch.Tensor:
    """The prediction tower on every hidden state of the list: [len * B, 128, H, W], call-major.  One launch chain where
    the engine can stack the calls (``max_stacked_calls``), else one chain per call."""
    n = len(hiddens)
    if n > 1 and eng.max_stacked_calls >= n and eng.calls[2] == 0:
        call = eng.next_call(2, n)
        x = torch.cat([h.to(dtype=torch.float32) for h in hiddens], dim=0)
        with torch.no_grad():
            torch._foreach_add_(eng.counters[2], n)
        return _PredictionCalls.apply(x, eng.modules[0][0].weight, eng, call, n)
    return torch.cat([tower(eng, 2, h) for h in hiddens], dim=0)


def tower(eng: TowerTrainEngine, which: int, x: torch.Tensor, action: Optional[torch.Tensor] = None, mode: int = 0):
    """The representation (0) / dynamics (1) / prediction (2) tower on the training kernels.  mode 0: the tower's output;
    1: its min-max normalisation (``normalize_hidden_state``) instead; 2: both, as a pair -- from the same kernel pass,
    forward and backward."""
    if which == 0:
        eng.begin_step()
    call = eng.next_call(which)
    x = x.to(dtype=torch.float32).contiguous()
    if action is not None:
        action = action.reshape(-1).to(dtype=torch.int64).contiguous()
    anchor = eng.modules[0][0].weight
    with torch.no_grad():           # BatchNorm2d.forward counts its train-mode calls
        torch._foreach_add_(eng.counters[which], 1)
    return _Tower.apply(x, anchor, eng, which, call, action, mode)


def engine_for(network, batch: int, unroll_steps: int = 5) -> Optional[TowerTrainEngine]:
    """The network's training engine for this batch size (created on first use), or None where the autograd modules
    are the training path (unsupported shape, CPU, eval mode, MZ_TRAIN_NATIVE=0)."""
    if not (_enabled() and network.training and supported(network)):
        return None
    p = next(network.parameters())
    if p.device.type != 'cuda':
        return None
    cache = _ENGINES.setdefault(network, {})
    key = (int(batch), p.device.index)
    eng = cache.get(key)
    if eng is None or eng.unroll < unroll_steps:
        cache.clear()               # one arena at a time (1-2 GB)
        eng = cache[key] = TowerTrainEngine(network, batch, max(int(unroll_steps), 5))
    return eng
