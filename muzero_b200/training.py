"""K-step-unroll training step, data-parallel over NCCL (BASELINE.json config 5).

Reference semantics mirrored here (michaelnny/muzero):
  pipeline.py:541-612  calc_loss(network, device, transitions, weights) -> (loss, priorities)
  pipeline.py:615-629  loss_func
  util.py:20-22,48-59,96-116  signed_hyperbolic, transform_to_2hot, scalar_to_categorical_probabilities
  pipeline.py:232-257  one learner iteration: zero_grad, calc_loss, backward, [clip], Adam step, LR step
  replay.py:27-32      Transition(state, action, pi_prob, value, reward)

The reference has ONE learner on one device; here every rank computes the loss of its shard of the replay batch and
the gradients are averaged with ONE flat-bucket all-reduce (the whole model, 29 MB fp32 for the Gomoku net, plus the
BatchNorm running statistics the inference engine folds into its weights: a single latency-bound NVLink transfer,
averaged inside NCCL), then every rank applies the identical Adam step (one launch of csrc/optim.cu on
torch.optim.Adam's own state), so weights stay in sync and the self-play engine on the same rank sees them without a
broadcast.  Forward / backward: for MuZeroBoardGameNet with 128 planes the three towers run on the tcgen05 kernels of
csrc/train.cu behind autograd Functions (train_engine.py; SURVEY.md 8 f-2), the prediction calls of an unroll stacked
into one launch chain, heads and losses once over the stacked calls; every other network trains through PyTorch autograd.

BatchNorm note: like the reference's `network.train()` (pipeline.py:218) each rank uses ITS shard's batch statistics;
DP therefore equals "mean of per-shard reference gradients", not the full-batch gradient, for the ResNets (MLP nets
have no BatchNorm and match the single-process full-batch step up to float reassociation).
"""
from __future__ import annotations

from typing import NamedTuple, Optional, Tuple

import os

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F

from .network import MuZeroNet, normalize_hidden_state


class _nullcontext:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


class Transition(NamedTuple):
    state: Optional[np.ndarray]
    action: Optional[np.ndarray]
    pi_prob: Optional[np.ndarray]
    value: Optional[np.ndarray]
    reward: Optional[np.ndarray]


def signed_hyperbolic(x: torch.Tensor, eps: float = 1e-3) -> torch.Tensor:
    return torch.sign(x) * (torch.sqrt(torch.abs(x) + 1) - 1) + eps * x


def signed_parabolic(x: torch.Tensor, eps: float = 1e-3) -> torch.Tensor:
    z = torch.sqrt(1 + 4 * eps * (eps + 1 + torch.abs(x))) / 2 / eps - 1 / 2 / eps
    return torch.sign(x) * (torch.square(z) - 1)


def transform_to_2hot(scalar: torch.Tensor, min_value: float, max_value: float, num_bins: int) -> torch.Tensor:
    """util.py:48-59."""
    scalar = torch.clamp(scalar, min_value, max_value)
    scalar_bin = (scalar - min_value) / (max_value - min_value) * (num_bins - 1)
    lower, upper = torch.floor(scalar_bin), torch.ceil(scalar_bin)
    lower_value = (lower / (num_bins - 1.0)) * (max_value - min_value) + min_value
    upper_value = (upper / (num_bins - 1.0)) * (max_value - min_value) + min_value
    p_lower = (upper_value - scalar) / (upper_value - lower_value + 1e-5)
    p_upper = 1 - p_lower
    return F.one_hot(lower.long(), num_bins) * p_lower.unsqueeze(-1) + F.one_hot(upper.long(), num_bins) * p_upper.unsqueeze(-1)


def scalar_to_categorical_probabilities(x: torch.Tensor, support_size: int) -> torch.Tensor:
    """util.py:96-116."""
    hi = (support_size - 1) // 2
    return transform_to_2hot(signed_hyperbolic(x), -hi, hi, support_size)


def logits_to_transformed_expected_value(logits: torch.Tensor, support_size: int) -> torch.Tensor:
    """util.py:70-93 (support created on the logits' device, unlike util.py:64)."""
    hi = (support_size - 1) // 2
    probs = torch.softmax(logits, dim=-1)
    support = torch.linspace(-hi, hi, support_size, device=logits.device).expand_as(probs)
    return signed_parabolic(torch.sum(probs * support, dim=-1, keepdim=True))


def _half_gradient(grad):
    """pipeline.py:583 ``register_hook(lambda grad: grad * 0.5)``; the last unrolled state feeds nothing, and a tower
    function that does not materialise unused gradients hands the hook None for it."""
    return None if grad is None else grad * 0.5


def loss_func(prediction: torch.Tensor, target: torch.Tensor, mse: bool = False) -> torch.Tensor:
    """pipeline.py:615-629."""
    assert prediction.shape == target.shape
    if mse:
        return F.mse_loss(prediction, target, reduction='none')
    assert prediction.dim() == 2
    return F.cross_entropy(prediction, target, reduction='none')


def calc_loss_tensors(network: MuZeroNet, state, action, target_value_scalar, target_reward_scalar, target_pi_prob,
                      weights):
    """pipeline.py:541-612 on device tensors, no host synchronisation (so a whole training step can be captured in a
    CUDA graph): representation, then T unrolled (prediction, dynamics) steps with the 0.5 gradient scale on the
    hidden state and the 1/T scale on the loss.  Returns (loss, priorities tensor [B])."""
    target_value = target_value_scalar if network.mse_loss_for_value else \
        scalar_to_categorical_probabilities(target_value_scalar, network.value_support_size)
    target_reward = target_reward_scalar if network.mse_loss_for_reward else \
        scalar_to_categorical_probabilities(target_reward_scalar, network.reward_support_size)

    B, T = action.shape
    reward_loss, value_loss, policy_loss = 0, 0, 0
    pred_values = []
    if hasattr(network, 'unroll_hint'):
        network.unroll_hint = T                      # sizes the training engine's activation slots (train_engine.py)
    hidden_state = network.represent(state)
    eng = network._train_engine(hidden_state) if hasattr(network, '_train_engine') else None
    mode = os.environ.get('MZ_TRAIN_BATCHED_HEADS', '1')    # 0: the reference's loop everywhere; 2: stacked heads for every conv net
    if eng is not None and mode != '0':
        from . import train_engine
        return _calc_loss_stacked(network, lambda h, a: train_engine.tower(eng, 1, h, a, mode=2),
                                  lambda hs: train_engine.prediction_calls(eng, hs), hidden_state, action, target_value, target_reward, target_pi_prob, target_value_scalar, weights)
    if mode == '2' and hasattr(network, 'dynamics_tower'):
        return _calc_loss_stacked(network, lambda h, a: (lambda raw: (raw, normalize_hidden_state(raw)))(network.dynamics_tower(h, a)),
                                  lambda hs: torch.cat([network.prediction_tower(h) for h in hs], dim=0), hidden_state, action, target_value,
                                  target_reward, target_pi_prob, target_value_scalar, weights)
    for t in range(T):
        pred_pi_logits, pred_value = network.prediction(hidden_state)
        hidden_state, pred_reward = network.dynamics(hidden_state, action[:, t].unsqueeze(1))
        hidden_state.register_hook(_half_gradient)
        value_loss = value_loss + loss_func(pred_value.squeeze(), target_value[:, t], network.mse_loss_for_value)
        reward_loss = reward_loss + loss_func(pred_reward.squeeze(), target_reward[:, t], network.mse_loss_for_reward)
        policy_loss = policy_loss + loss_func(pred_pi_logits, target_pi_prob[:, t])
        pred_values.append(pred_value.detach())
    loss = reward_loss + value_loss + policy_loss
    loss = torch.mean(loss * weights.detach())
    loss_scale = 1.0 / T
    loss.register_hook(lambda grad: grad * loss_scale)
    with torch.no_grad():
        pv = torch.stack(pred_values, dim=1)
        pv_scalar = pv.squeeze(-1) if network.mse_loss_for_value else \
            logits_to_transformed_expected_value(pv, network.value_support_size).squeeze(-1)
        priorities = (pv_scalar[:, 0] - target_value_scalar[:, 0]).abs()
    return loss, priorities


def _calc_loss_stacked(network, dyn_tower, pred_towers, hidden_state, action, target_value, target_reward, target_pi_prob,
                       target_value_scalar, weights):
    """The same loss with the work regrouped for the hand-written tower kernels (train_engine.py): the dynamics chain
    first (it is the only sequential part: h_0 -> h_1 -> ... ), then the prediction tower on h_0 .. h_{T-1}, then every
    head ONCE over the T calls' stacked inputs (``head_over_calls``: per-call BatchNorm statistics, running statistics
    updated in call order) and the losses over [T, B].  Same operands into the same operations as the loop of
    pipeline.py:579-600 -- only the launch count differs (the heads and losses were 60 % of the kernels of a step)."""
    from .network import head_over_calls, heads_over_calls
    B, T = action.shape
    hiddens, raws = [], []
    for t in range(T):
        hiddens.append(hidden_state)
        raw, hidden_state = dyn_tower(hidden_state, action[:, t].unsqueeze(1))     # the tower's output and its normalisation
        raws.append(raw)
        hidden_state.register_hook(_half_gradient)
    feats = pred_towers(hiddens)                                             # [T * B, C, h, w], call-major
    raws = torch.cat(raws, dim=0)
    pred_net, dyn_net = network.prediction_net, network.dynamics_net
    pi_logits, pred_value = heads_over_calls([pred_net.policy_net, pred_net.value_net], feats, T)   # [T * B, A], [T * B, S]
    pred_reward = head_over_calls(dyn_net.reward_head, raws, T)              # [T * B, S]

    def stacked(target):                                                      # [B, T, ...] -> [T * B, ...]
        return target.transpose(0, 1).reshape((T * B,) + tuple(target.shape[2:]))

    def per_call(pred, target, mse):
        if mse:
            return loss_func(pred.reshape(T * B), stacked(target), True).view(T, B).sum(0)
        return loss_func(pred, stacked(target), False).view(T, B).sum(0)

    value_loss = per_call(pred_value, target_value, network.mse_loss_for_value)
    reward_loss = per_call(pred_reward, target_reward, network.mse_loss_for_reward)
    policy_loss = per_call(pi_logits, target_pi_prob, False)
    loss = reward_loss + value_loss + policy_loss
    loss = torch.mean(loss * weights.detach())
    loss_scale = 1.0 / T
    loss.register_hook(lambda grad: grad * loss_scale)
    with torch.no_grad():
        pv0 = pred_value.detach()[:B]
        pv_scalar = pv0.squeeze(-1) if network.mse_loss_for_value else \
            logits_to_transformed_expected_value(pv0, network.value_support_size).squeeze(-1)
        priorities = (pv_scalar - target_value_scalar[:, 0]).abs()
    return loss, priorities


def _to_device(transitions: Transition, device):
    return (torch.as_tensor(transitions.state).to(device=device, dtype=torch.float32, non_blocking=True),
            torch.as_tensor(transitions.action).to(device=device, dtype=torch.long, non_blocking=True),
            torch.as_tensor(transitions.value).to(device=device, dtype=torch.float32, non_blocking=True),
            torch.as_tensor(transitions.reward).to(device=device, dtype=torch.float32, non_blocking=True),
            torch.as_tensor(transitions.pi_prob).to(device=device, dtype=torch.float32, non_blocking=True))


def calc_loss(network: MuZeroNet, device, transitions: Transition, weights: torch.Tensor):
    """pipeline.py:541-612 with the reference's signature: (loss, priorities as a host array)."""
    loss, priorities = calc_loss_tensors(network, *_to_device(transitions, device), weights)
    return loss, priorities.cpu().numpy()


class DataParallelLearner:
    """One learner iteration of pipeline.py:232-257 on every rank, gradients averaged by one all-reduce.

    On a CUDA device the whole iteration (zero grads, K-step unroll forward, backward, all-reduce, clip, Adam) is
    captured in ONE CUDA graph after three eager iterations and replayed from static input buffers: at batch 128 the
    ~3000 small kernels of the unroll are launch-bound when issued from Python.  ``use_graph=False`` keeps every
    iteration eager; a capture that fails (e.g. a collective backend that cannot be captured) falls back to eager."""

    def __init__(self, network: MuZeroNet, config, device, process_group=None, use_graph: bool = True,
                 data_parallel: bool = True) -> None:
        self.network, self.config, self.device = network, config, torch.device(device)
        # conv nets on CUDA train with NHWC weights / activations: same fp32 (TF32) cuDNN arithmetic without the layout
        # transposes around every convolution (24.8 -> 20.7 ms per 128 x K=5 Gomoku step).  state_dict shapes, the
        # engine's weight packing and checkpoints are unaffected (memory format only).
        # Networks the hand-written tower kernels cover (train_engine.py) keep NCHW parameters: the kernels read them.
        from . import train_engine
        self.native_towers = (self.device.type == 'cuda' and train_engine._enabled() and train_engine.supported(network))
        self.channels_last = (self.device.type == 'cuda' and getattr(network, 'latent_hw', (0, 0)) != (0, 0)
                              and not self.native_towers)
        if self.channels_last:
            network.to(memory_format=torch.channels_last)
        self.group = process_group
        self.world = dist.get_world_size(process_group) if dist.is_available() and dist.is_initialized() else 1
        if not data_parallel:                 # a learner of its own inside a multi-rank job (no collective)
            self.world = 1
        params = [p for p in network.parameters() if p.requires_grad]
        # ONE flat bucket: the gradients (every .grad is a view into it -> the all-reduce needs no packing copies) followed,
        # in a data-parallel job, by the BatchNorm running statistics -- a single collective per step
        n_grad = sum(p.numel() for p in params)
        pad = lambda n: (n + 63) // 64 * 64
        bufs = [b for b in network.buffers() if b.dtype.is_floating_point] if self.world > 1 else []
        n_buf = sum(pad(b.numel()) for b in bufs)
        self.flat_all = torch.zeros(pad(n_grad) + n_buf, dtype=torch.float32, device=self.device)
        self.flat_grad = self.flat_all[:n_grad]
        off = 0
        for p in params:
            # same strides as the parameter (NHWC conv weights are a dense permutation): autograd accumulates in place
            p.grad = self.flat_grad[off:off + p.numel()].as_strided(p.size(), p.stride())
            off += p.numel()
        self.params = params
        # BatchNorm running statistics are updated from each rank's shard: average them with a second flat bucket so that
        # every rank's actor folds the SAME statistics into its inference engine and any rank's checkpoint is the model
        # all ranks used (DDP broadcasts rank 0's buffers instead; the average uses every shard's data)
        self.flat_buf = None
        if bufs:
            # every buffer starts on a 256-byte boundary of the bucket: cuDNN's BatchNorm kernels take the running
            # statistics through vector loads and fault on the 4-byte-aligned views a dense packing would give the
            # buffers that follow a 1- or 2-channel head BatchNorm
            self.flat_buf = self.flat_all[pad(n_grad):]
            off = 0
            for b in bufs:
                view = self.flat_buf[off:off + b.numel()].view(b.shape)
                view.copy_(b)
                b.data = view
                off += pad(b.numel())
        self.use_graph = bool(use_graph) and self.device.type == 'cuda'
        # gomoku/run_training.py:110 / classic: Adam(lr_init, weight_decay), MultiStepLR(milestones, lr_decay_rate).
        # Graph mode: step counters and the learning rate live on the device so that a replay sees their updates.
        # (On CUDA the optimizer is the capturable flavour whether or not the graph is used, so that eager and
        # replayed iterations run the same arithmetic.)
        on_cuda = self.device.type == 'cuda'
        lr = torch.tensor(float(config.lr_init), device=self.device) if on_cuda else config.lr_init
        # fused=True: one multi-tensor kernel per step.  The capturable foreach flavour divides every parameter by two
        # 0-dim device scalars with one tiny kernel each -- 330 launches, 1.1 ms of a 14 ms Gomoku step.
        self.optimizer = torch.optim.Adam(params, lr=lr, weight_decay=config.weight_decay, capturable=on_cuda,
                                          **({'fused': True} if on_cuda else {}))
        self.lr_scheduler = torch.optim.lr_scheduler.MultiStepLR(self.optimizer, milestones=list(config.lr_milestones),
                                                                 gamma=config.lr_decay_rate)
        self._nccl = self.world > 1 and dist.get_backend(self.group) == 'nccl'
        self._fast_adam = None
        self.train_steps = 0
        self.last_allreduce_ms = None
        self._graph = None
        self._static = None
        self._eager_left = 3

    def _iteration(self, state, action, value, reward, pi, w, time_allreduce: bool = False):
        """zero grads -> loss -> backward -> all-reduce -> clip -> Adam; device tensors in and out."""
        self.flat_grad.zero_()                                  # optimizer.zero_grad() that keeps the views
        loss, priorities = calc_loss_tensors(self.network, state, action, value, reward, pi, w)
        loss.backward()
        if self.world > 1:
            if time_allreduce and self.device.type == 'cuda':
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            # gradients and running statistics in ONE collective; NCCL averages inside it (no division pass over 29 MB)
            if self._nccl:
                dist.all_reduce(self.flat_all, op=dist.ReduceOp.AVG, group=self.group)
            else:
                dist.all_reduce(self.flat_all, op=dist.ReduceOp.SUM, group=self.group)
                self.flat_all.div_(self.world)
            if time_allreduce and self.device.type == 'cuda':
                e1.record()
                torch.cuda.synchronize(self.device)
                self.last_allreduce_ms = e0.elapsed_time(e1)
        if self.config.clip_grad:
            torch.nn.utils.clip_grad_norm_(self.params, self.config.max_grad_norm)
        self._optimizer_step()
        return loss.detach(), priorities

    # -- optimizer step -----------------------------------------------------------------------------------------------
    def _optimizer_step(self) -> None:
        """torch.optim.Adam.step(), or -- once the optimizer's state exists (after its first step) -- the one-launch Adam of
        csrc/optim.cu on that very state (exp_avg, exp_avg_sq, step tensors of ``self.optimizer.state``, in place): same
        arithmetic, one kernel over a chunk table instead of five launches of 64 K-element chunks.  MZ_FAST_ADAM=0: torch's."""
        fast = self._fast_adam
        if fast is None:
            fast = self._fast_adam = self._build_fast_adam()
        if not fast:
            self.optimizer.step()
            return
        from . import _lib
        torch._foreach_add_(fast['steps'], 1)
        g = fast['group']
        _lib.check(_lib.lib().mz_adam_step(fast['tensors'].data_ptr(), fast['chunk_tensor'].data_ptr(), fast['chunk_start'].data_ptr(),
                                           fast['n_chunks'], fast['steps'][0].data_ptr(), g['lr'].data_ptr(), g['betas'][0],
                                           g['betas'][1], g['eps'], g['weight_decay'], _lib.current_stream()))

    def _build_fast_adam(self):
        """Pointer / chunk tables for mz_adam_step, or False where torch's step stays (CPU, no state yet this call, exotic
        layouts or options).  None is returned until the state exists, so the question is asked again next step."""
        if self.device.type != 'cuda' or os.environ.get('MZ_FAST_ADAM', '1') == '0' or len(self.optimizer.param_groups) != 1:
            return False
        g = self.optimizer.param_groups[0]
        if g.get('amsgrad') or g.get('maximize') or not torch.is_tensor(g['lr']) or torch.cuda.is_current_stream_capturing():
            return False if (g.get('amsgrad') or g.get('maximize') or not torch.is_tensor(g['lr'])) else None
        rows, steps = [], []
        for p in g['params']:
            st = self.optimizer.state.get(p)
            if not st:
                return None                      # state is created by the optimizer's first step
            m, v, step = st['exp_avg'], st['exp_avg_sq'], st['step']
            tensors = (p.data, p.grad, m, v)
            if any(t.dtype != torch.float32 or t.stride() != p.stride() or t.device != p.device for t in tensors) or \
                    not (p.is_contiguous() or p.is_contiguous(memory_format=torch.channels_last)) or \
                    step.dtype != torch.float32 or not step.is_cuda:
                return False
            rows.append((p.data_ptr(), p.grad.data_ptr(), m.data_ptr(), v.data_ptr(), p.numel()))
            steps.append(step)
        from . import _lib
        chunk = _lib.lib().mz_adam_chunk_elements()
        table = np.zeros((len(rows), 5), dtype=np.int64)
        chunk_tensor, chunk_start = [], []
        for k, r in enumerate(rows):
            table[k] = r
            for start in range(0, r[4], chunk):
                chunk_tensor.append(k)
                chunk_start.append(start)
        dev = self.device
        return {'group': g, 'steps': steps, 'n_chunks': len(chunk_tensor),
                'tensors': torch.from_numpy(table).to(dev),               # mz_adam_tensor records: four pointers + n
                'chunk_tensor': torch.tensor(chunk_tensor, dtype=torch.int32, device=dev),
                'chunk_start': torch.tensor(chunk_start, dtype=torch.int64, device=dev)}

    def _graphed(self, inputs):
        if self._static is None or any(a.shape != b.shape for a, b in zip(self._static, inputs)):
            self._static = [torch.empty_like(t) for t in inputs]
            self._graph = None
        for dst, src in zip(self._static, inputs):
            dst.copy_(src, non_blocking=True)
        if self._graph is None:
            try:
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    self._out = self._iteration(*self._static)
                self._graph = g
            except Exception as exc:                            # noqa: BLE001 - any capture failure -> eager for good
                import warnings
                warnings.warn(f'training-step graph capture failed ({exc!r}); continuing eagerly')
                self.use_graph = False
                torch.cuda.synchronize(self.device)
                self.flat_grad.zero_()
                return self._iteration(*inputs)
        self._graph.replay()
        return self._out

    def step(self, transitions: Transition, weights, time_allreduce: bool = False) -> Tuple[float, np.ndarray]:
        self.network.train()
        with torch.cuda.device(self.device) if self.device.type == 'cuda' else _nullcontext():
            w = torch.as_tensor(weights).to(device=self.device, dtype=torch.float32)
            inputs = _to_device(transitions, self.device) + (w,)
            if self.channels_last and inputs[0].dim() == 4:
                inputs = (inputs[0].contiguous(memory_format=torch.channels_last),) + inputs[1:]
            if self.use_graph and not time_allreduce and self._eager_left <= 0:
                loss, priorities = self._graphed(inputs)
            else:
                self._eager_left -= 1
                loss, priorities = self._iteration(*inputs, time_allreduce=time_allreduce)
        self.lr_scheduler.step()
        self.train_steps += 1
        # a graph replay does not advance the parameters' version counters: tell the inference engine explicitly
        if hasattr(self.network, 'mark_weights_updated'):
            self.network.mark_weights_updated()
        return float(loss), priorities.cpu().numpy()

    def state_dict(self):
        """Same keys as the reference's checkpoints (pipeline.py:224-230)."""
        return {'network': self.network.state_dict(), 'optimizer': self.optimizer.state_dict(),
                'lr_scheduler': self.lr_scheduler.state_dict(), 'train_steps': self.train_steps}


def synthetic_transitions(network: MuZeroNet, batch: int, unroll: int, seed: int) -> Tuple[Transition, np.ndarray]:
    """A replay batch of config 5's shapes (SURVEY.md §8d): state int8/float32 [B,*obs], action [B,T],
    value/reward float32 [B,T], pi float32 [B,T,A], importance weights float32 [B]."""
    gen = np.random.RandomState(seed)
    A = network.num_actions
    shape = tuple(network.input_shape)
    state = gen.randint(0, 2, size=(batch,) + shape).astype(np.float32)
    action = gen.randint(0, A, size=(batch, unroll)).astype(np.int64)
    value = gen.choice([-1.0, 0.0, 1.0], size=(batch, unroll)).astype(np.float32)
    reward = (gen.standard_normal((batch, unroll)) * 0.1).astype(np.float32)
    pi = gen.dirichlet(np.ones(A), size=(batch, unroll)).astype(np.float32)
    weights = gen.uniform(0.5, 1.0, size=batch).astype(np.float32)
    return Transition(state=state, action=action, pi_prob=pi, value=value, reward=reward), weights
