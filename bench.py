#!/usr/bin/env python
"""Benchmark of the self-play hot path: MCTS simulations/sec, network evaluation included.

    python bench.py --gpus N --steps K --warmup W [--workload tictactoe|cartpole|gomoku|atari] [--dump-outputs DIR]
    python bench.py --impl reference ...        # the CPU arm (oracle port of the reference path)

--dump-outputs DIR writes what the last timed search returned (action, pi, root_value of rank 0's trees) and the
last timed training step's loss / priorities as DIR/<name>.npy (float64), so that two builds run with the same
arguments, hence the same inputs, weights and RNG seeds, can be compared output for output.

A "step" is ONE batched search: B trees x S simulations, from observations to
(action, pi, root value): initial inference, Dirichlet noise, S x (select, recurrent
inference, expand+backup), visit policy and action sampling all inside the timed region.
`value` keeps the inputs resident in HBM; `e2e` goes through the public
``uct_search_batch`` with HOST (pinned) observations/masks and reads the results back.
Under torchrun (N > 1) every rank searches its own B trees (games shard across GPUs with no
collective, weak scaling), time is the max over ranks, value the whole-job aggregate.
One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')

METRIC = 'mcts_simulations_per_sec_net_eval_incl'
UNIT = 'simulations/s'


# ---------------------------------------------------------------------------
# workloads (SURVEY.md section 8d)
# ---------------------------------------------------------------------------
def workload_spec(name: str, trees: int | None):
    import muzero_b200 as mz
    if name == 'tictactoe':       # BASELINE.json configs[1]
        cfg = mz.make_tictactoe_config(use_tensorboard=False)
        spec = dict(kind='mlp', ckpt='tictactoe', net_kw=dict(input_shape=(9, 3, 3), num_actions=10, num_planes=256,
                    value_support_size=1, reward_support_size=1, hidden_dim=64), trees=4096, board=True,
                    label='Tic-Tac-Toe 3x3 MLP MuZero from checkpoint TicTacToe_train_steps_35000')
    elif name == 'cartpole':      # configs[0]
        cfg = mz.make_classic_config(use_tensorboard=False)
        spec = dict(kind='mlp', ckpt='cartpole', net_kw=dict(input_shape=(4, 5), num_actions=2, num_planes=512,
                    value_support_size=31, reward_support_size=31, hidden_dim=64), trees=16384, board=False,
                    label='CartPole-v1 MLP MuZero from checkpoint CartPole-v1_train_steps_44800')
    elif name == 'gomoku':        # configs[2]
        cfg = mz.make_gomoku_config(use_tensorboard=False)
        spec = dict(kind='board', ckpt=None, net_kw=dict(input_shape=(9, 9, 9), num_actions=82, num_res_blocks=8,
                    num_planes=128), trees=2048, board=True, label='Gomoku 9x9 ResNet(128x8) MuZero, random init seed 0')
    elif name == 'atari':         # configs[3]
        cfg = mz.make_atari_config(use_tensorboard=False)
        cfg.num_simulations = 50
        spec = dict(kind='atari', ckpt=None, net_kw=dict(input_shape=(16, 96, 96), num_actions=18, num_res_blocks=8,
                    num_planes=128, value_support_size=61, reward_support_size=61), trees=1024, board=False,
                    label='Atari-shaped 16x96x96 ResNet(128x8) MuZero, random init seed 0, 50 sims')
    else:
        raise SystemExit(f'unknown workload {name}')
    if trees:
        spec['trees'] = trees
    spec['name'], spec['cfg'] = name, cfg
    return spec


def state_dict_for(spec):
    import torch
    import muzero_b200 as mz
    if spec['ckpt']:
        return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, f"ckpt_{spec['ckpt']}.npz")).items()}
    torch.manual_seed(0)
    cls = mz.MuZeroBoardGameNet if spec['kind'] == 'board' else mz.MuZeroAtariNet
    return cls(**spec['net_kw']).eval().state_dict()


def synthetic_inputs(spec, B: int, seed: int):
    """Observations / masks / players of each config's shape (no envs, no ROMs)."""
    gen = np.random.RandomState(seed)
    shape, A = spec['net_kw']['input_shape'], spec['net_kw']['num_actions']
    if spec['name'] in ('tictactoe', 'gomoku'):
        c, h, w = shape
        n_hist = (c - 1) // 2
        obs = np.zeros((B, c, h, w), dtype=np.int8)
        mask = np.ones((B, A), dtype=bool)
        max_moves = 6 if spec['name'] == 'tictactoe' else 40
        cur = np.ones(B, dtype=np.int32)
        for b in range(B):
            k = gen.randint(0, max_moves + 1)
            cells = gen.permutation(h * w)[:k]
            boards = np.zeros((k + 1, 2, h * w), dtype=np.int8)
            for i, cell in enumerate(cells):
                boards[i + 1] = boards[i]
                boards[i + 1, i % 2, cell] = 1
            me = k % 2                                # side to move
            for t in range(n_hist):                   # most recent first: [mine_t, theirs_t] * history, then colour
                bd = boards[max(k - t, 0)]
                obs[b, 2 * t] = bd[me].reshape(h, w)
                obs[b, 2 * t + 1] = bd[1 - me].reshape(h, w)
            obs[b, c - 1] = 1 if me == 0 else 0
            mask[b, :h * w] = boards[k].sum(0) == 0
            mask[b, h * w:] = True                    # resign
            cur[b] = 1 + me
        return obs, mask, cur, (3 - cur).astype(np.int32)
    if spec['name'] == 'cartpole':
        obs = gen.standard_normal((B,) + shape).astype(np.float32)
        obs[:, :, -1] = (gen.randint(0, 2, size=(B, shape[0])) + 1) / 2.0
    else:
        # the Atari observation as the environment produces it (gym_env.py:306-313): k uint8 frames + k constant action
        # planes (action + 1) / A.  Kept in that compact form (muzero_b200.StackedFrames); .expand() gives the float32
        # [B, 2k, H, W] tensor the reference builds from it.
        import torch
        from muzero_b200 import StackedFrames
        half = shape[0] // 2
        frames = gen.randint(0, 256, size=(B, half) + shape[1:]).astype(np.uint8)
        planes = ((gen.randint(0, A, size=(B, shape[0] - half)) + 1) / A).astype(np.float32)
        obs = StackedFrames(torch.from_numpy(frames), torch.from_numpy(planes))
    one = np.ones(B, dtype=np.int32)
    return obs, np.ones((B, A), dtype=bool), one, one


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, uuid: str):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', uuid, f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, power, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            f = [x.strip() for x in r.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); power.append(float(f[2]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['no samples']}
        busy = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
        return {'sm_mhz': statistics.median(busy), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons),
                'samples': len(sm), 'power_w_max': max(power)}


# ---------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path, one tree per process at a time
# ---------------------------------------------------------------------------
_W = {}


def _cpu_worker_init(name, trees):
    import torch
    torch.set_num_threads(1)
    from oracle.network_oracle import OracleNet
    spec = workload_spec(name, trees)
    sd = state_dict_for(spec)
    kw = spec['net_kw']
    _W['spec'] = spec
    _W['net'] = OracleNet(spec['kind'], sd, kw['num_actions'], kw.get('value_support_size', 1),
                          kw.get('reward_support_size', 1), kw.get('num_res_blocks', 0))


def _cpu_worker_run(args):
    """Run `n` single-tree searches (reference structure: batch-1 network call per simulation)."""
    wid, n, seed = args
    from oracle import mcts_oracle as orc
    spec = _W['spec']
    obs, mask, cur, opp = synthetic_inputs(spec, n, seed + wid)
    if hasattr(obs, 'expand'):
        obs = obs.expand().numpy()
    rs = np.random.RandomState(1234 + wid)
    t0 = time.perf_counter()
    for i in range(n):
        orc.uct_search(obs[i], _W['net'], 'cpu', spec['cfg'], 1.0, mask[i], int(cur[i]), int(opp[i]), False, rng=rs)
    return n * spec['cfg'].num_simulations, time.perf_counter() - t0


class CpuArm:
    def __init__(self, name, trees, procs):
        import multiprocessing as mp
        self.procs = procs
        self.pool = mp.get_context('spawn').Pool(procs, initializer=_cpu_worker_init, initargs=(name, trees))

    def step(self, searches_per_proc, seed):
        t0 = time.perf_counter()
        out = self.pool.map(_cpu_worker_run, [(w, searches_per_proc, seed) for w in range(self.procs)])
        wall = time.perf_counter() - t0
        return sum(o[0] for o in out), wall

    def close(self):
        self.pool.close()
        self.pool.join()


def cpu_searches_per_step(name):
    return {'tictactoe': 40, 'cartpole': 12, 'gomoku': 1, 'atari': 2}[name]


def bench_config(spec, trees_per_gpu, world, strong):
    """The `config` object of the JSON line: ONE definition for both arms, so that the driver's same_config check
    compares like with like.  Engine-side scheduling detail lives under `schedule`, not here."""
    return {'workload': spec['label'], 'trees_per_gpu': int(trees_per_gpu), 'simulations': int(spec['cfg'].num_simulations),
            'num_actions': int(spec['net_kw']['num_actions']),
            'l2': 'flushed between timed iterations (256 MiB write)',
            'parallelism': ('2048 games split over' if strong else 'games sharded over') + f' {world} GPU(s), no collective'}


def run_reference_arm(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    spec = workload_spec(args.workload, args.trees)
    if args.strong:
        spec['trees'] = max(1, spec['trees'] // max(1, args.gpus))
    procs = min(os.cpu_count() or 1, args.cpu_procs)
    arm = CpuArm(args.workload, args.trees, procs)
    n = cpu_searches_per_step(args.workload)
    for w in range(args.warmup):
        arm.step(max(1, n // 4), 10_000 + w)
    sims, wall = 0, 0.0
    for k in range(args.steps):
        s, t = arm.step(n, 20_000 + k)
        sims += s; wall += t
    arm.close()
    value = sims / wall
    sample = f'{procs} processes x {n} single-tree searches x {spec["cfg"].num_simulations} sims per step, {args.steps} steps'
    emit({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1000.0 * wall / args.steps, 'higher_is_better': True,
        'scaling': 'strong' if args.strong else 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': bench_config(spec, spec['trees'], args.gpus, bool(args.strong)),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': procs, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    })


# ---------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------
def algorithmic_bytes_per_launch(kernel, spec, B, A, S, mean_depth, hidden_bytes, noise):
    """SURVEY.md section 8(d) per-tree-per-simulation figures x B trees (one launch = one simulation of B trees)."""
    d = mean_depth
    if kernel == 'select':
        per = d * (16 * A + 4) + (8 if noise else 4) * A
    elif kernel == 'expand_backup':
        per = 32 * (d + 1) + 16 * A + 32
    else:   # recurrent inference: read parent state once, write child state once, + action
        per = 2 * hidden_bytes + 4
    return per * B


def initial_flops(spec):
    """Multiply-add flops (x2) of ONE initial_inference of the reference graph: representation + prediction nets."""
    kw = spec['net_kw']
    A = kw['num_actions']
    if spec['kind'] == 'mlp':
        ind = int(np.prod(kw['input_shape'])); P, H = kw['num_planes'], kw['hidden_dim']
        return 2 * (ind * P + P * H + H * P + P * A + H * P + P * kw['value_support_size'])
    c, h, w = kw['input_shape']
    C_, nb = kw['num_planes'], kw['num_res_blocks']
    conv = lambda ci, co, hh, ww: 2 * 9 * ci * co * hh * ww
    if spec['kind'] == 'board':
        rep = conv(c, C_, h, w) + 2 * nb * conv(C_, C_, h, w)
        lh, lw = h, w
    else:       # network.py:312-353: conv_1 s2, 2 blocks @48, conv_2 s2, 2 blocks @24, pool, 2 blocks @12, pool
        rep = conv(c, 128, h // 2, w // 2) + 4 * conv(128, 128, h // 2, w // 2) + conv(128, C_, h // 4, w // 4) + \
            4 * conv(C_, C_, h // 4, w // 4) + 4 * conv(C_, C_, h // 8, w // 8)
        lh, lw = 6, 6
    pred = 2 * nb * conv(C_, C_, lh, lw)
    heads = 2 * lh * lw * (C_ * 2 + C_ * 1) + 2 * lh * lw * (2 * A + kw.get('value_support_size', 1))
    return rep + pred + heads


def build_search(spec, dev, rank=0, parts=0, cta_limit=0):
    """Network, search plan and synthetic inputs exactly as the bench runs them (tests/test_bench_parity_gpu.py builds
    its plan through this function, so what is parity-checked IS what is timed)."""
    import torch
    import muzero_b200 as mz
    from muzero_b200.mcts import PipelinedSearchPlan, SearchPlan, pipeline_shape
    cfg, B = spec['cfg'], spec['trees']
    cls = {'mlp': mz.MuZeroMLPNet, 'board': mz.MuZeroBoardGameNet, 'atari': mz.MuZeroAtariNet}[spec['kind']]
    net = cls(**spec['net_kw'])
    net.load_state_dict(state_dict_for(spec))
    net = net.to(dev).eval()
    # conv nets with enough rows: two half-batches interleaved on two streams (tree kernels of one overlap the tower
    # of the other)
    auto_parts, auto_limit = pipeline_shape(net, B)
    if not parts:
        parts, cta_limit = auto_parts, auto_limit
    plan = PipelinedSearchPlan(net, cfg, B, parts, cta_limit) if parts > 1 else SearchPlan(net, cfg, B)
    seeds = 1234 + rank * B + np.arange(B)
    plan.pool.seed(seeds)
    obs, mask, cur, opp = synthetic_inputs(spec, B, 99 + rank)
    mask_h = torch.from_numpy(mask).pin_memory()
    # inputs resident in HBM for `value`
    if isinstance(obs, mz.StackedFrames):
        obs_h = mz.StackedFrames(obs.frames.pin_memory(), obs.planes.pin_memory())
        plan.use_frames()
        plan.frames.copy_(obs_h.frames); plan.planes.copy_(obs_h.planes)
    else:
        obs_h = torch.from_numpy(obs).pin_memory()
        plan.obs.copy_(obs_h.reshape(B, -1))
    plan.mask.copy_(mask_h)
    plan.players.copy_(torch.from_numpy(np.stack([cur, opp], 1)))
    plan.temps.fill_(1.0)
    return dict(net=net, plan=plan, parts=parts, cta_limit=cta_limit, obs=obs, mask=mask, cur=cur, opp=opp,
                obs_h=obs_h, mask_h=mask_h, seeds=seeds)


def measure_workload(spec, args, dev, world, rank, steps, warmup, min_seconds=0.0, parts=0, cta_limit=0,
                     kernel_timing=True):
    """One workload on this rank's GPU: device-timed `value`, `e2e` through uct_search_batch with host buffers,
    clocks sampled during the timed region, per-kernel roofline (eager launches bracketed by CUDA events)."""
    import torch
    import torch.distributed as dist
    import muzero_b200 as mz
    from muzero_b200 import _lib

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg, B, A, S = spec['cfg'], spec['trees'], spec['net_kw']['num_actions'], spec['cfg'].num_simulations
    built = build_search(spec, dev, rank, parts, cta_limit)
    net, plan, parts, cta_limit = built['net'], built['plan'], built['parts'], built['cta_limit']
    obs_h, mask_h, cur, opp = built['obs_h'], built['mask_h'], built['cur'], built['opp']
    pool = plan.pool
    read_stats = (lambda: pool.stats()) if parts > 1 else (lambda: pool.view('STATS').cpu().numpy().copy())
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)      # > 126 MB L2

    def step_device():
        plan.run('device', True, False)

    out_h = [torch.empty(B, dtype=torch.int32).pin_memory(), torch.empty((B, A), dtype=torch.float64).pin_memory(),
             torch.empty(B, dtype=torch.float64).pin_memory()]

    def step_e2e():
        a, pi, q = mz.uct_search_batch(obs_h, net, cfg, 1.0, mask_h, cur, opp, plan=plan)
        out_h[0].copy_(a, non_blocking=True); out_h[1].copy_(pi, non_blocking=True); out_h[2].copy_(q, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def timed(fn, steps):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        for e0, e1 in ev:
            flush.zero_()                      # L2 flush between timed iterations (not timed)
            e0.record(); fn(); e1.record()
        barrier()
        ms = sum(e0.elapsed_time(e1) for e0, e1 in ev) / steps
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    warmup = max(warmup, 3)
    t0 = time.perf_counter()
    for _ in range(warmup):
        step_device()
    torch.cuda.synchronize()
    for _ in range(2):
        step_e2e()
    torch.cuda.synchronize()
    pool.check_errors()
    if min_seconds > 0:
        # short workloads (a Tic-Tac-Toe search lasts a millisecond): enough steps that nvidia-smi, sampling every
        # 100 ms, sees the timed region at least ten times.  Same count on every rank.
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); step_device(); step_device(); e1.record()
        torch.cuda.synchronize()
        est = max(1e-4, e0.elapsed_time(e1) / 2e3 + 1e-3)            # + the L2 flush between steps
        steps = int(min(5000, max(steps, min_seconds / est)))
    stats0 = read_stats()

    uuid = str(torch.cuda.get_device_properties(dev).uuid)
    sampler = ClockSampler(uuid if uuid.startswith('GPU-') else 'GPU-' + uuid) if rank == 0 else None
    ms_dev = timed(step_device, steps)
    # what the last timed search returned, read before the e2e steps below overwrite the plan's output buffers
    built['outputs'] = {'action': plan.action.cpu().numpy(), 'pi': plan.pi.cpu().numpy(),
                        'root_value': plan.root_value.cpu().numpy()}
    stats1 = read_stats()
    ms_e2e = timed(step_e2e, steps)
    clocks = sampler.stop() if rank == 0 else None
    pool.check_errors()

    mean_depth = float(stats1[0] - stats0[0]) / max(1.0, float(stats1[1] - stats0[1]))
    value = world * B * S / (ms_dev / 1000.0)
    e2e_value = world * B * S / (ms_e2e / 1000.0)
    obs_bytes = sum(t.numel() * t.element_size() for t in (obs_h if isinstance(obs_h, tuple) else (obs_h,)))
    h2d = obs_bytes + mask_h.numel() + 2 * 4 * B + 8 * B
    d2h = sum(t.numel() * t.element_size() for t in out_h)

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    hbm_peak = float(peaks.get('hbm_gbs', 6650.0))
    tf_peak = float(peaks.get('bf16_tflops', 1590.0))
    tf_sustained = float(peaks.get('bf16_tflops_sustained', tf_peak))
    peak_src = 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback (B200_PROFILING.md)'
    pplan = plan.parts[0] if parts > 1 else plan
    Bp = pplan.B
    result = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': steps, 'warmup': warmup,
        'ms_per_step': ms_dev, 'higher_is_better': True, 'scaling': 'strong' if args.strong else 'weak',
        'vs_baseline': None,
        'dtype': 'f64 tree statistics / f32 scores; network fp16 x fp16 -> f32 (tcgen05)' +
                 (' for recurrent inference, f32 SIMT for the root inference' if spec['kind'] == 'mlp' else ''),
        'data': 'synthetic',
        'config': bench_config(spec, B, world, bool(args.strong)),
        'schedule': {'pipeline_parts': parts, 'trees_per_kernel_launch': Bp,
                     'ctas_per_tower_launch': getattr(plan, 'cta_limit', 0) or cta_limit or 148,
                     'ctas_per_tree_kernel_launch': getattr(plan, 'tree_ctas', 0) or 'one warp per tree, all SMs',
                     'mean_select_depth': mean_depth},
        'e2e': {'value': e2e_value, 'unit': UNIT, 'ms_per_step': ms_e2e, 'h2d_bytes_per_step': int(h2d),
                'd2h_bytes_per_step': int(d2h)},
        'gpu_launches': int(plan.launches_per_search * steps * 2),
        'clocks': clocks,
    }
    if not kernel_timing:
        return result, built

    # ---- per-kernel timing (eager launches, CUDA events on the launching stream) -> roofline.
    # With a pipelined plan the kernels run on sub-batches of B / parts trees: part 0 is timed as it runs there.
    lib = _lib.lib()
    ppool = pplan.pool
    eng = net.engine(Bp, pplan.instance)
    hidden = ppool.hidden.data_ptr() if ppool.hidden_bytes else None
    names = ['select', 'recurrent', 'expand_backup']
    tot = {n: 0.0 for n in names}
    reps = max(1, min(steps, 3))
    import ctypes as C
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream().cuda_stream
        use_frames = pplan.obs_mode == 'u8'
        prof_ms, prof_n = [0.0] * 5, [0] * 5
        init_ms = []
        init_prof = None
        for _ in range(reps):
            # root part eagerly (initial inference with the root preparation fused into its policy epilogue), timed
            # on its own; then the instrumented simulation loop
            _lib.check(lib.mz_net_profile_begin(eng['handle']))
            i0, i1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            i0.record()
            _lib.check(lib.mz_net_initial_search(
                eng['handle'], ppool.handle, Bp, None if use_frames else pplan.obs.data_ptr(),
                pplan.frames.data_ptr() if use_frames else None, pplan.planes.data_ptr() if use_frames else None, hidden,
                pplan.root_slots.data_ptr(), pplan.pi0.data_ptr(), pplan.v0.data_ptr(), 2, pplan.noise.data_ptr(),
                float(np.float32(cfg.root_dirichlet_alpha)), float(cfg.root_exploration_eps), pplan.mask.data_ptr(),
                pplan.players.data_ptr(), stream))
            i1.record()
            ip_ms, ip_n = (C.c_double * 5)(), (C.c_int64 * 5)()
            _lib.check(lib.mz_net_profile_end(eng['handle'], ip_ms, ip_n))
            init_ms.append(i0.elapsed_time(i1))
            init_prof = (list(ip_ms), list(ip_n))
            _lib.check(lib.mz_net_profile_begin(eng['handle']))
            evs = []
            for _s in range(S):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
                e[0].record()
                _lib.check(lib.mz_select(ppool.handle, stream)); e[1].record()
                _lib.check(lib.mz_net_recurrent(eng['handle'], Bp, hidden, ppool.view('SRC_SLOT').data_ptr(),
                                                ppool.view('LEAF_ACTION').data_ptr(), hidden,
                                                ppool.view('DST_SLOT').data_ptr(), ppool.view('REWARD').data_ptr(),
                                                ppool.view('VALUE').data_ptr(), None, stream)); e[2].record()
                _lib.check(lib.mz_expand_backup(ppool.handle, None, None, stream)); e[3].record()
                evs.append(e)
            torch.cuda.synchronize()
            for e in evs:
                for i, n in enumerate(names):
                    tot[n] += e[i].elapsed_time(e[i + 1])
            r_ms, r_n = (C.c_double * 5)(), (C.c_int64 * 5)()
            _lib.check(lib.mz_net_profile_end(eng['handle'], r_ms, r_n))
            for i in range(5):
                prof_ms[i] += r_ms[i]; prof_n[i] += r_n[i]
    launches = reps * S
    avg_ms = {n: tot[n] / launches for n in names}
    share = {n: tot[n] / sum(tot.values()) for n in names}
    dominant = max(names, key=lambda n: tot[n])
    roof = {}
    for n in names:
        ab = algorithmic_bytes_per_launch(n, spec, Bp, A, S, mean_depth, pool.hidden_bytes, True)
        roof[n] = {'bound': 'hbm', 'achieved': ab / (avg_ms[n] * 1e-3) / 1e9, 'peak': hbm_peak, 'unit': 'GB/s',
                   'avg_launch_us': avg_ms[n] * 1e3, 'share_of_sim_loop': share[n], 'algorithmic_bytes': ab}
        roof[n]['frac'] = roof[n]['achieved'] / hbm_peak
    flops = {'tictactoe': 175104, 'cartpole': 395264, 'gomoku': 803712780, 'atari': 351896688}[spec['name']]
    ach = flops * Bp / (avg_ms['recurrent'] * 1e-3) / 1e12        # every family runs recurrent inference on tcgen05
    roof['recurrent'].update({'bound': 'tensor', 'achieved': ach, 'peak': tf_peak, 'unit': 'TFLOP/s',
                              'frac': ach / tf_peak, 'reference_graph_flops': flops * Bp})
    roofline = dict(roof[dominant])
    roofline.update({'kernel': dominant, 'traffic': None, 'peak_source': peak_src})
    if spec['kind'] == 'mlp':
        # where mz_search_run runs ONE persistent kernel for all S simulations (configuration 2: the warp-per-tree
        # kernel), that launch is what a search executes; the three kernels above are the per-simulation launch chain it
        # replaces, kept as a diagnostic.  Timed eagerly with CUDA events around the launch.
        sm = []
        with torch.cuda.device(dev):
            for _ in range(max(3, reps)):
                _lib.check(lib.mz_net_initial_search(eng['handle'], ppool.handle, Bp, pplan.obs.data_ptr(), None, None,
                                                     hidden, pplan.root_slots.data_ptr(), pplan.pi0.data_ptr(),
                                                     pplan.v0.data_ptr(), 2, pplan.noise.data_ptr(),
                                                     float(np.float32(cfg.root_dirichlet_alpha)),
                                                     float(cfg.root_exploration_eps), pplan.mask.data_ptr(),
                                                     pplan.players.data_ptr(), stream))
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                n0 = lib.mz_launch_count()
                e0.record()
                _lib.check(lib.mz_search_run(eng['handle'], ppool.handle, stream))
                e1.record()
                n_launch = int(lib.mz_launch_count() - n0)
                torch.cuda.synchronize()
                sm.append(e0.elapsed_time(e1))
        search_ms = min(sm)
        if n_launch == 1:
            ab = sum(algorithmic_bytes_per_launch(n, spec, Bp, A, S, mean_depth, pool.hidden_bytes, True) for n in names) * S
            ach = flops * Bp * S / (search_ms * 1e-3) / 1e12
            roofline = {'kernel': 'mlp_search32_kernel / mlp_tc_kernel<search>: one persistent launch per search (select / '
                                  'backup around the tcgen05 MLP chain, trees owned by their CTA for all simulations)',
                        'bound': 'tensor', 'achieved': ach, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': ach / tf_peak,
                        'traffic': None, 'avg_launch_us': search_ms * 1e3, 'us_per_simulation': search_ms * 1e3 / S,
                        'algorithmic_bytes_per_launch': ab, 'hbm_achieved_gbs': ab / (search_ms * 1e-3) / 1e9,
                        'hbm_frac': ab / (search_ms * 1e-3) / 1e9 / hbm_peak,
                        'note': 'latency-bound: 0.18-0.40 MFLOP and a few hundred bytes per row and simulation',
                        'peak_source': peak_src}
            roof = {'search_kernel': dict(roofline), 'launch_chain_diagnostic': roof}
    if spec['kind'] != 'mlp' and prof_n[0] > 0:
        # the dominant KERNEL is the tcgen05 3x3 convolution.  One launch runs a whole tower pair as a dataflow
        # of layers (33 convs for a recurrent inference): algorithmic flops per layer = the reference graph's
        # CxC 3x3 conv over the H*W real positions of the boards of one launch.  Launch duration: CUDA events around
        # every eager launch.
        c, h, w = spec['net_kw']['input_shape']
        hh, ww = (h, w) if spec['kind'] == 'board' else (6, 6)
        planes = spec['net_kw']['num_planes']
        per_pos = 2.0 * planes * planes * 9
        layers_per_launch = prof_n[0] / max(1, prof_n[4])
        launch_ms = prof_ms[0] / max(1, prof_n[4])
        alg = per_pos * hh * ww * Bp * layers_per_launch
        pad = net.grid_pad          # 0: no halo rows (edge taps masked in the MMA), 1: padded (H+1)(W+1) grid
        exe = per_pos * (hh + pad) * (ww + pad) * Bp * layers_per_launch
        ach = alg / (launch_ms * 1e-3) / 1e12
        traffic = None
        try:     # dram bytes of one launch from the committed ncu --set full capture of the same kernel
            tj = json.load(open(os.path.join(ROOT, 'profiles', 'conv_traffic.json')))
            if tj.get('workload') == spec['name'] and tj.get('trees_per_launch') == Bp:
                traffic = tj['dram_bytes_per_launch']
        except Exception:
            pass
        roofline = {'kernel': 'conv3x3_kernel (tcgen05.mma M128 N128 K16, TMEM accumulators, TMA tile loads)',
                    'bound': 'tensor', 'achieved': ach, 'peak': tf_peak, 'unit': 'TFLOP/s', 'frac': ach / tf_peak,
                    'peak_regime': 'burst (cuBLAS bf16 8192^3 best of 10); the kernel is timed inside the eager '
                                   'simulation loop of a long step, where the sustained figure applies',
                    'frac_of_sustained_peak': ach / tf_sustained, 'sustained_peak': tf_sustained,
                    'traffic': traffic, 'avg_launch_us': launch_ms * 1e3, 'launches_timed': int(prof_n[4]),
                    'conv_layers_per_launch': layers_per_launch,
                    'algorithmic_flops_per_launch': alg, 'executed_flops_per_launch': exe,
                    'executed_tflops': exe / (launch_ms * 1e-3) / 1e12,
                    'share_of_recurrent_inference': prof_ms[0] / max(1e-9, prof_ms[0] + prof_ms[1] + prof_ms[2]),
                    'share_of_sim_loop': prof_ms[0] / max(1e-9, sum(tot.values())), 'peak_source': peak_src}
        roof['head_kernel'] = {'avg_launch_us': 1e3 * prof_ms[1] / max(1, prof_n[1]), 'launches_timed': int(prof_n[1])}
    # the once-per-search root inference (representation + prediction, root preparation fused into the policy epilogue)
    fl0 = initial_flops(spec)
    im = min(init_ms)
    roof['initial_inference'] = {'avg_launch_us': im * 1e3, 'share_of_search': im / max(1e-9, im + sum(tot.values()) / reps),
                                 'reference_graph_flops': fl0 * Bp, 'bound': 'tensor',
                                 'achieved': fl0 * Bp / (im * 1e-3) / 1e12, 'peak': tf_peak, 'unit': 'TFLOP/s',
                                 'frac': fl0 * Bp / (im * 1e-3) / 1e12 / tf_peak,
                                 'conv_ms': init_prof[0][0], 'conv_layers': init_prof[1][0], 'pack_pool_ms': init_prof[0][2],
                                 'head_ms': init_prof[0][1], 'mlp_ms': init_prof[0][3]}
    result['roofline'] = roofline
    result['kernels'] = roof
    del flush
    return result, built


def release(built):
    """Drop a workload's plan, pools and engines before the next one is built."""
    import gc
    import torch
    import muzero_b200 as mz
    built['net'].release_engine()
    built.clear()
    mz.mcts._PLANS.clear()
    gc.collect()
    torch.cuda.empty_cache()


def run_engine_arm(args):
    import torch
    import torch.distributed as dist

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)

    spec = workload_spec(args.workload, args.trees)
    if args.strong:                       # SURVEY 8d: the configuration's trees in TOTAL, split over the ranks
        spec['trees'] = max(1, spec['trees'] // world)
    result, built = measure_workload(spec, args, dev, world, rank, args.steps, args.warmup, parts=args.parts,
                                     cta_limit=args.cta_limit)
    net = built['net']
    outputs = dict(built['outputs'])
    if not args.no_train_step:
        try:
            result['train_step'] = train_step_sample(net, spec, dev, world, outputs=outputs)
        except Exception as exc:                      # never lose the search line to the secondary measurement
            result['train_step'] = {'error': repr(exc)[:200]}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    if spec['name'] in ('gomoku', 'tictactoe') and not args.no_self_play:
        try:
            result['self_play'] = self_play_sample(net, spec, dev, rank)
        except Exception as exc:
            result['self_play'] = {'error': repr(exc)[:200]}
    release(built)
    if world > 1 and not args.strong and not args.no_configs and spec['name'] == 'gomoku':
        # the same configuration split over the ranks (SURVEY 8d "2048 total"): the latency regime of the design
        try:
            s2 = workload_spec(args.workload, max(1, spec['trees'] // world))
            r2, b2 = measure_workload(s2, args, dev, world, rank, max(3, args.steps // 2), 3, kernel_timing=False)
            result['strong_scaling'] = {'trees_total': s2['trees'] * world, 'trees_per_gpu': s2['trees'],
                                        'value': r2['value'], 'ms_per_step': r2['ms_per_step'], 'unit': UNIT,
                                        'e2e': r2['e2e'], 'schedule': r2['schedule'],
                                        'speedup_vs_one_gpu_weak_step': result['ms_per_step'] / r2['ms_per_step']}
            release(b2)
        except Exception as exc:
            result['strong_scaling'] = {'error': repr(exc)[:200]}
    if not args.no_configs and spec['name'] == 'gomoku' and not args.strong:
        # short sub-runs of the other BASELINE.json configurations, so that the driver's line carries every config
        # (each with its own clocks record of >= 10 samples, e2e and per-kernel roofline)
        result['configs'] = {}
        for name in ('cartpole', 'tictactoe', 'atari'):
            try:
                s_i = workload_spec(name, None)
                r_i, b_i = measure_workload(s_i, args, dev, world, rank, 5, 3, min_seconds=1.5)
                release(b_i)
                for k in ('metric', 'unit', 'higher_is_better', 'vs_baseline', 'data'):
                    r_i.pop(k, None)
                result['configs'][name] = r_i
            except Exception as exc:
                result['configs'][name] = {'error': repr(exc)[:300]}
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        result['cpu_baseline'] = cpu_baseline_sample(args, spec)
    if rank == 0:
        emit(result)
    if world > 1:
        dist.destroy_process_group()


def train_step_sample(net, spec, dev, world, batch=128, unroll=5, warmup=6, steps=20, outputs=None):
    """BASELINE.json config 5's second half: the K=5-unroll training step, data-parallel, one flat
    NCCL all-reduce of the gradients; the towers' forward / dgrad / wgrad and train-mode BatchNorm run on the
    hand-written tcgen05 kernels of csrc/train.cu (SURVEY.md section 8 e / f-2).  The last timed step's loss and
    priorities go into `outputs` when it is given."""
    import copy
    import torch
    import torch.distributed as dist
    import muzero_b200 as mz
    from muzero_b200.training import DataParallelLearner, synthetic_transitions
    cls = type(net)
    rank = dist.get_rank() if world > 1 else 0
    local_ms = None
    if world > 1:
        # the same step WITHOUT the collective (what one GPU does on its own), on this box, right before the
        # data-parallel one: ms_local / ms_dp is the step's own weak-scaling efficiency
        twin0 = cls(**spec['net_kw']).to(dev)
        twin0.load_state_dict(net.state_dict())
        solo = DataParallelLearner(twin0, spec['cfg'], dev, data_parallel=False)
        tr0, w0 = synthetic_transitions(twin0, batch, unroll, seed=400 + rank)
        for _ in range(warmup):
            solo.step(tr0, w0)
        torch.cuda.synchronize(dev)
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        l0.record()
        for _ in range(steps):
            solo.step(tr0, w0)
        l1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([l0.elapsed_time(l1) / steps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        local_ms = float(t.item())
        del solo, twin0
        torch.cuda.empty_cache()
    twin = cls(**spec['net_kw']).to(dev)
    twin.load_state_dict(net.state_dict())
    learner = DataParallelLearner(twin, spec['cfg'], dev)
    # batches come out of the device-resident replay (SURVEY 8f f-4): 64 batches' worth of synthetic transitions,
    # uniform sampling like every run_training.py of the reference, sample + gather inside the timed step
    from muzero_b200.replay import DeviceReplay
    replay = DeviceReplay(64 * batch, 0.0, 0.0, np.random.RandomState(900 + rank), device=dev)
    for k in range(64):
        tr_k, _ = synthetic_transitions(twin, batch, unroll, seed=500 + 64 * rank + k)
        replay.add_batch(tr_k, np.ones(batch, np.float32))
    for _ in range(warmup):
        tr, idx, w = replay.sample(batch)
        learner.step(tr, w)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ar = []
    if world > 1:
        dist.barrier()
    e0.record()
    for _ in range(steps):
        s0.record()
        tr, idx, w = replay.sample(batch)
        s1.record()
        loss, prio = learner.step(tr, w)
        replay.update_priorities(idx, prio)
    e1.record()
    torch.cuda.synchronize(dev)
    if outputs is not None:
        outputs['train_loss'], outputs['train_priorities'] = np.array([loss]), prio
    sample_ms = s0.elapsed_time(s1)
    dp_only_ms = None
    if world > 1:                        # the data-parallel learner step on its own (fixed batch, no replay calls)
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        dist.barrier()
        d0.record()
        for _ in range(steps):
            learner.step(tr, w)
        d1.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([d0.elapsed_time(d1) / steps], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dp_only_ms = float(t.item())
    if world > 1:                        # the gradient all-reduce on its own (inside the step it is part of the graph)
        for i in range(8):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            dist.all_reduce(learner.flat_grad, op=dist.ReduceOp.SUM)
            a1.record()
            torch.cuda.synchronize(dev)
            if i >= 3:
                ar.append(a0.elapsed_time(a1))
    ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    nbytes = learner.flat_grad.numel() * 4
    out = {'ms_per_step': float(ms.item()), 'batch_per_gpu': batch, 'unroll_steps': unroll, 'loss': loss,
           'samples_per_s': world * batch / (float(ms.item()) / 1e3), 'grad_bytes': nbytes,
           'replay_sample_ms': sample_ms, 'replay_items': replay.size,
           'cuda_graph': bool(learner.use_graph and learner._graph is not None),
           'native_towers': bool(learner.native_towers),
           'impl': ('DeviceReplay.sample (sampling + gather kernels) -> ONE CUDA graph of: the towers forward / dgrad / wgrad + '
                    'train-mode BatchNorm on the tcgen05 kernels of csrc/train.cu (fp16 activations, bf16 gradients, fp32 '
                    'accumulation; the K prediction calls stacked into one launch chain), heads / losses in PyTorch over the '
                    'stacked calls, the flat NCCL all-reduce and fused Adam -> update_priorities') if learner.native_towers else
                   ('DeviceReplay.sample (sampling + gather kernels) -> ONE CUDA graph of the PyTorch autograd fwd/bwd, the flat '
                    'NCCL all-reduce and Adam -> update_priorities')}
    if learner.native_towers:
        out['towers'] = tower_chain_sample(twin, batch, unroll)
        # roofline of the step's tensor-core work: every 3x3 convolution of the K-step unroll forward, dgrad and wgrad
        # (algorithmic flops, the padded halo rows the kernels also multiply are not counted) against the measured peak
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            peaks = {}
        tf_peak = float(peaks.get('bf16_tflops', 1590.0))
        c, h, w = spec['net_kw']['input_shape']
        nb, planes, A = twin.num_res_blocks, twin.num_planes, twin.num_actions
        px = batch * h * w
        conv = lambda cin: px * 2.0 * 9 * cin * planes
        rep = conv(c) + 2 * nb * conv(planes)
        dyn = conv(planes + A) + 2 * nb * conv(planes)
        pred = 2 * nb * conv(planes)
        fwd = rep + unroll * (dyn + pred)
        # backward: dgrad for every convolution whose input needs a gradient (not the representation's first), wgrad for all
        bwd = 2 * fwd - conv(c)
        step_s = float(ms.item()) / 1e3
        out['roofline'] = {'kernel': 'tconv_kernel / twgrad_kernel (tcgen05.mma M128 N128 K16; csrc/train.cu)', 'bound': 'tensor',
                           'algorithmic_flops_per_step': fwd + bwd, 'achieved': (fwd + bwd) / step_s / 1e12, 'peak': tf_peak,
                           'unit': 'TFLOP/s', 'frac': (fwd + bwd) / step_s / 1e12 / tf_peak,
                           'peak_source': 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback (B200_PROFILING.md)',
                           'note': 'latency-bound: 182 layer-calls of 100 tiles on 148 SMs per direction, each waiting for the '
                                   'one before it (DESIGN.md section 4, Training towers); the stacked prediction calls run at the '
                                   'rates under towers.prediction_x%d' % unroll}
    if local_ms is not None:
        out['ms_per_learner_step_no_collective'] = local_ms
        out['ms_per_learner_step_data_parallel'] = dp_only_ms
        out['efficiency'] = local_ms / dp_only_ms
    if ar:
        a = sum(ar) / len(ar)
        out['allreduce_ms'] = a
        out['allreduce_bus_gbs'] = 2.0 * (world - 1) / world * nbytes / (a * 1e-3) / 1e9
    del learner, twin, replay
    torch.cuda.empty_cache()
    return out


def tower_chain_sample(net, batch, unroll, reps=10):
    """The training towers on their own (CUDA events around graph replays of one launch chain): the prediction tower's
    forward and backward for one call and for the K stacked calls, with the convolution flops they execute."""
    import torch
    from muzero_b200 import train_engine
    eng = train_engine.engine_for(net.train(), batch, unroll)
    if eng is None:
        return None
    c, h, w = eng.hidden_shape[1:]
    dev = eng.device
    layers = 2 * net.num_res_blocks
    flops = lambda calls: calls * batch * h * w * 2.0 * 9 * c * c * layers

    def graphed(fn):
        s = torch.cuda.Stream(device=dev)
        with torch.cuda.stream(s):
            fn()
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fn()
        return g

    def timed(g):
        for _ in range(3):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / reps * 1e3

    out = {'layers': layers, 'batch': batch}
    with torch.cuda.device(dev):
        for calls in (1, unroll) if eng.max_stacked_calls >= unroll else (1,):
            x = torch.rand((calls * batch, c, h, w), device=dev)
            gr = torch.randn((calls * batch, c, h, w), device=dev)

            def fwd():
                return eng.forward(2, 0, x, None) if calls == 1 else eng.forward_calls(0, calls, x)

            def bwd():
                if calls == 1:
                    eng.backward(2, 0, gr)
                else:
                    eng.backward_calls(0, calls, gr)
                eng.join()
            eng.begin_step()                 # (weight packing and the statistics reset are not part of a tower's chain)
            gf = graphed(fwd)
            tf = timed(gf)
            gb = graphed(bwd)
            tb = timed(gb)
            out['prediction_x%d' % calls] = {
                'forward_us': tf, 'backward_us': tb, 'forward_tflops': flops(calls) / (tf * 1e-6) / 1e12,
                'backward_tflops': 2.0 * flops(calls) / (tb * 1e-6) / 1e12,
                'us_per_layer_forward': tf / layers, 'us_per_layer_backward': tb / layers}
        eng.begin_step()
        eng.active = False
    return out


def self_play_sample(net, spec, dev, rank, moves=3):
    """SURVEY 8f rows f-1/f-3 on top of the search: B concurrent games on the device (batched env step, trajectory
    buffers, MC-return targets + unroll windows for finished games), a few moves timed end to end."""
    import torch
    import muzero_b200 as mz
    c, h, w = spec['net_kw']['input_shape']
    num_to_win = 3 if spec['name'] == 'tictactoe' else 5
    env = mz.BatchedBoardEnv(spec['trees'], h, num_to_win, (c - 1) // 2, device=dev)
    loop = mz.BoardSelfPlay(net, spec['cfg'], env, seed=777 + rank)
    loop.play_move()                                   # plan creation + graph capture
    loop.play_move()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    samples = 0
    for _ in range(moves):
        out = loop.play_move()
        samples += 0 if out is None else int(out.state.shape[0])
    e1.record()
    torch.cuda.synchronize(dev)
    env.check_errors()
    ms = e0.elapsed_time(e1) / moves
    S = spec['cfg'].num_simulations
    res = {'ms_per_move': ms, 'games_in_flight': spec['trees'], 'moves_per_s': spec['trees'] / (ms / 1e3),
           'simulations_per_s': spec['trees'] * S / (ms / 1e3), 'samples_emitted': samples,
           'impl': 'uct_search_batch + env_step_kernel + target/unroll kernels, one D2H flag read per move'}
    del loop, env
    mz.mcts._PLANS.clear()
    torch.cuda.empty_cache()
    return res


def cpu_baseline_sample(args, spec):
    procs = min(os.cpu_count() or 1, args.cpu_procs)
    arm = CpuArm(args.workload, args.trees, procs)
    n = cpu_searches_per_step(args.workload)
    arm.step(max(1, n // 4), 1)
    sims, wall = arm.step(n, 2)
    arm.close()
    return {'value': sims / wall, 'unit': UNIT, 'cores': procs, 'kind': 'port',
            'sample': f'{procs} processes x {n} single-tree searches x {spec["cfg"].num_simulations} sims '
                      f'(oracle port of uct_search + fp32 torch network, 1 thread per process)'}


DUMP_LIMIT_BYTES = 60 << 20         # under 64 MB in all, .npy headers included


def dump_outputs(dirname: str, outputs: dict, limit: int = DUMP_LIMIT_BYTES) -> None:
    """`outputs` as float64 arrays DIR/<name>.npy.  Past `limit` bytes in all, the per-tree arrays keep a fixed sample of
    trees (seed 0; the tree indices go to DIR/sampled_trees.npy) so that the files stay small enough to keep and diff."""
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in outputs.items()}
    per_tree = ('action', 'pi', 'root_value')
    B = len(arrays['action'])
    total = sum(a.nbytes for a in arrays.values())
    if total > limit:
        tree_bytes = sum(arrays[k].nbytes for k in per_tree)
        keep = max(1, int(B * (limit - (total - tree_bytes) - 8 * B) / tree_bytes))
        rows = np.sort(np.random.RandomState(0).choice(B, size=keep, replace=False))
        arrays = {k: (a[rows] if k in per_tree else a) for k, a in arrays.items()}
        arrays['sampled_trees'] = rows.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(dirname, f'{k}.npy'), a)


_REAL_STDOUT = None


def emit(obj) -> None:
    """The ONE JSON line goes to the real stdout; everything else any library prints (NCCL's version
    banner goes to fd 1) was diverted to stderr by main()."""
    line = json.dumps(obj) + '\n'
    if _REAL_STDOUT is None:
        sys.stdout.write(line)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line.encode())


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10, help='timed steps (searches) of the workload')
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--workload', default=os.environ.get('MZ_BENCH_WORKLOAD', 'gomoku'))
    ap.add_argument('--trees', type=int, default=None, help='trees per GPU (default: the config size)')
    ap.add_argument('--impl', default='engine', choices=['engine', 'reference'])
    ap.add_argument('--cpu-procs', type=int, default=int(os.environ.get('MZ_BENCH_CPU_PROCS', '64')))
    ap.add_argument('--parts', type=int, default=0, help='sub-batches in flight per GPU (0: 2 for conv nets, 1 for MLPs)')
    ap.add_argument('--cta-limit', type=int, default=0, help='with --parts: SMs per tower launch (0: all)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-train-step', action='store_true')
    ap.add_argument('--no-self-play', action='store_true')
    ap.add_argument('--no-configs', action='store_true', help='skip the sub-runs of the other configurations')
    ap.add_argument('--strong', action='store_true',
                    help="strong scaling: the configuration's trees in total, split over the ranks")
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help="write the last timed step's outputs to DIR/<name>.npy (engine arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs applies to the engine arm')
    if args.impl == 'reference':
        run_reference_arm(args)
    else:
        run_engine_arm(args)


if __name__ == '__main__':
    main()
