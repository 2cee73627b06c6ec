#!/usr/bin/env python
"""bench.py -- view-tuples/sec of the hot path on synthetic 5-view x 1024-keypoint tuples.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg3|cfg2|cfg4|cfg5] [--tuples B]
                    [--dump-outputs DIR]

A *step* is one pass of the hot path over one batch of B synthetic units per GPU.  Default = BASELINE.json
configs[2] (cfg3: ScanNet-shape 5-tuple, 1024 kpts, 28-layer matcher, confidence head, 10 x {w8pt + two-view BA},
spanning tree, rotation averaging + LUD, global LM BA); --config cfg2 / cfg4 are the two-view workloads
(configs[1] / [3]: pairs/sec at 1024 / 2048 kpts, w8pt_ba).  One JSON line on rank 0; see DESIGN.md §measurement
for every field.  `--impl reference` times the CPU port of the reference path (oracle/) on the host cores; the
reference project itself is not needed.

`--dump-outputs DIR` writes what the last timed step of rank 0 returned (see dump_outputs) as DIR/<name>.npy.  Weights
and inputs are seeded, so two builds of the project run with the same arguments can be compared array for array.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

if int(os.environ.get('WORLD_SIZE', '1')) > 1:
    # multi-rank launch: NCCL's communicator lines ("comm ... rank R nranks N ... Init COMPLETE") go to the job log, so
    # that whoever launched it can count the ranks that really joined.  Must be in the environment before torch loads
    # NCCL (the debug level is latched at NCCL's first call); caller-set values win.
    # (the GPU boxes of this project export NCCL_DEBUG=VERSION: the "NCCL version ..." line of the log is kept as is)
    if 'NCCL_DEBUG' not in os.environ:
        os.environ['NCCL_DEBUG'] = 'INFO'
        os.environ.setdefault('NCCL_DEBUG_SUBSYS', 'INIT')

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GAIN = 12.0          # final_proj gain of the seeded weights: gives the assignment real structure
D = 256

# BASELINE.json `configs`: [2] is the headline (view-tuples/sec, the default), [1] and [3] are the two-view
# (eval_pairs.py) workloads.  `batch` = units (tuples / pairs) per step per GPU.
CONFIGS = {
    'cfg3': dict(workload='scannet_5tuple_1024kpts_28layers_mvba', kind='tuple', views=5, kpts=1024,
                 layers=(['self'] + ['cross'] * 3) * 7, batch=14, width=640, height=480, f=577.87, seed_base=1000,
                 metric='view-tuples/sec @1024 kpts 5-view', unit='tuples/s', parity_kpts=192,
                 pose='10x(w8pt+10it 2-view BA) + spanning tree + rotation averaging/LUD + global LM BA (<=50 it)'),
    'cfg2': dict(workload='scannet_2view_1024kpts_18layers_w8pt_ba', kind='pair', views=2, kpts=1024,
                 layers=['self', 'cross'] * 9, batch=32, width=720, height=537, f=650.0, seed_base=2000,
                 metric='pairs/sec @1024 kpts 2-view w8pt_ba', unit='pairs/s', parity_kpts=256,
                 pose='w8pt + 10it 2-view BA (eval_pairs.py w8pt_ba)'),
    'cfg4': dict(workload='megadepth_2view_2048kpts_18layers_w8pt_ba', kind='pair', views=2, kpts=2048,
                 layers=['self', 'cross'] * 9, batch=8, width=1600, height=1200, f=1400.0, seed_base=4000,
                 metric='pairs/sec @2048 kpts 2-view w8pt_ba', unit='pairs/s', parity_kpts=256,
                 pose='w8pt + 10it 2-view BA (eval_pairs.py w8pt_ba)'),
    # BASELINE.json configs[4], STAGE 1 of it (match loss; the pose-loss gradients of stage 2 are not built): one training
    # iteration per step -- train-mode forward, match loss, backward through the kernels, gradient all-reduce, Adam
    'cfg5': dict(workload='train_stage1_5tuple_400kpts_28layers_matchloss', kind='train', views=5, kpts=400,
                 layers=(['self'] + ['cross'] * 3) * 7, batch=8, width=640, height=480, f=577.87, seed_base=5000,
                 metric='training steps/sec, tuple_size 5, 8 tuples per GPU, 400 kpts (stage 1: match loss)', unit='steps/s',
                 pose='none (stage 1 of train.py: match loss only)'),
}


def attention_flops(cfg):
    """Algorithmic QK^T + PV FLOPs of one unit (SURVEY.md §8d): per layer 4 N M D per view, M = N (self) or (T-1) N."""
    T, N = cfg['views'], cfg['kpts']
    n_self, n_cross = cfg['layers'].count('self'), cfg['layers'].count('cross')
    return n_self * 4 * N * N * D * T + n_cross * 4 * N * (T - 1) * N * D * T


def sinkhorn_bytes_per_problem(cfg, iters=100):
    """The reference's formulation: 2 full passes over the (N+1)^2 fp32 matrix per iteration + one read + one write."""
    return (iters * 2 + 2) * (cfg['kpts'] + 1) ** 2 * 4


def n_pairs(cfg):
    return cfg['views'] * (cfg['views'] - 1) // 2


def workload_config(cfg):
    """The `config` object of the JSON line: what defines the workload (identical for both arms)."""
    return {'workload': cfg['workload'], 'views': cfg['views'], 'kpts': cfg['kpts'], 'gnn_layers': len(cfg['layers']),
            'sinkhorn_iters': 100, 'pose': cfg['pose']}


def make_weights(cfg):
    from e2e_multi_view_matching_b200.synthetic import make_state_dict
    return make_state_dict(len(cfg['layers']), seed=0, final_proj_gain=GAIN, conf_head='score')


def make_inputs(cfg, seed, batch, kpts=None):
    from e2e_multi_view_matching_b200.synthetic import make_scene_tuple_inputs
    return make_scene_tuple_inputs(seed, cfg['views'], kpts or cfg['kpts'], batch=batch, width=cfg['width'],
                                   height=cfg['height'], f=cfg['f'])


TF32_PEAK_TFLOPS = 148 * 4096 * 1.965e9 / 1e12      # tcgen05 kind::tf32 issue floor x SMs x max SM clock


def emit(line):
    """The one JSON line, on a line of its own even if another writer (NCCL_DEBUG=INFO, a warning) left stdout mid-line."""
    sys.stdout.flush()
    sys.stdout.write('\n' + json.dumps(line) + '\n')
    sys.stdout.flush()


DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(out_dir, arrays, budget=DUMP_BYTES):
    """--dump-outputs: every numeric array of `arrays` (torch tensors or numpy) as <out_dir>/<name>.npy, float64 for
    float64 and integer results, float32 for the rest (both exact).  To stay within `budget` bytes in all, an array
    of more than `cap` elements is replaced by its elements at `cap` fixed positions (flat, C order, increasing),
    drawn from a seeded generator: runs with the same arguments dump the same positions.  `cap` is the largest
    halving of the biggest array's size that fits the budget.  -> {name: stored element count}."""
    import torch
    host = {}
    for name, v in arrays.items():
        if isinstance(v, torch.Tensor):
            v = v.detach().cpu().numpy()
        if isinstance(v, np.ndarray) and v.dtype.kind in 'biuf':
            host[name] = v.astype(np.float64 if v.dtype.kind in 'iu' or v.dtype == np.float64 else np.float32)
    cap = max([v.size for v in host.values()] + [1])
    while cap > 1 and sum(min(v.size, cap) * v.itemsize for v in host.values()) > budget:
        cap //= 2
    os.makedirs(out_dir, exist_ok=True)
    stored = {}
    for name, v in host.items():
        if v.size > cap:
            v = v.reshape(-1)[np.sort(np.random.default_rng(0).choice(v.size, cap, replace=False))]
        np.save(os.path.join(out_dir, name + '.npy'), v)
        stored[name] = v.size
    return stored


def load_traffic(workload, batch):
    """Per-launch DRAM traffic of the dominant kernels from the committed ncu capture (profiles/ncu_traffic.json),
    valid for the workload / batch size it was captured at."""
    try:
        t = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'profiles', 'ncu_traffic.json')))
        if t.get('tuples_per_step') == batch and t.get('workload', 'scannet_5tuple_1024kpts_28layers_mvba') == workload:
            return t['attention']['avg_bytes_per_launch'], t['sinkhorn']['avg_bytes_per_launch']
    except Exception:
        pass
    return None, None


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d['hbm_gbs'], 'tflops': d.get('bf16_tflops_sustained', d['bf16_tflops']),
                'source': 'measured (MEASURED_PEAKS.json, bf16 sustained / copy)'}
    return {'hbm_gbs': 6650.0, 'tflops': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler(threading.Thread):
    """SM clock / throttle reasons sampled DURING the timed region.  In-process NVML (a few microseconds
    per query) -- an `nvidia-smi` subprocess takes ~0.5 s per sample and stalls kernel launches while it
    holds the driver lock, which showed up as a 100 ms hiccup inside the e2e timing; it is only the
    fallback when NVML cannot be loaded."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples = []
        self.stop_flag = False
        self.nvml = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            try:
                self.handle = pynvml.nvmlDeviceGetHandleByUUID('GPU-' + str(torch.cuda.get_device_properties(gpu_index).uuid))
            except Exception:
                self.handle = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _sample_nvml(self):
        n, h = self.nvml, self.handle
        sm = n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(h, n.NVML_CLOCK_SM)
        try:
            r = n.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = n.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        act = lambda bit: 'Active' if (r & bit) else 'Not Active'
        # NVML reason bits: SwPowerCap 0x4, HwSlowdown 0x8, SwThermalSlowdown 0x20, HwThermalSlowdown 0x40
        return [str(sm), str(mx), '', act(0x8), act(0x40), act(0x20), act(0x4)]

    def run(self):
        q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
             'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
             'clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    self.samples.append(self._sample_nvml())
                    time.sleep(0.02)
                    continue
                o = subprocess.run(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + q,
                                    '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
                f = [x.strip() for x in o.stdout.strip().split(',')]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        sm = sorted(float(s[0]) for s in self.samples)
        reasons = []
        for i, name in ((3, 'hw_slowdown'), (4, 'hw_thermal_slowdown'), (5, 'sw_thermal_slowdown'), (6, 'sw_power_cap')):
            if any(s[i].lower().startswith('active') for s in self.samples):
                reasons.append(name)
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.samples[0][1]), 'reasons': reasons,
                'samples': len(self.samples), 'source': 'nvml' if self.nvml is not None else 'nvidia-smi'}


# ---------------------------------------------------------------------------------------------
# CPU port of the reference path (oracle) -- cpu_baseline leg and the --impl reference arm
# ---------------------------------------------------------------------------------------------
def cpu_reference_unit(cfg, sd, data_np, b=0, cap2=128):
    """One unit (tuple / pair) through the CPU restatement of the reference: full-size matcher (100 Sinkhorn
    iterations, confidence head), then the pose stage.  The reference's two-view BA is a dense (6+3n)^2 LU
    (minutes per pair at n ~ 900), so it runs on the first `cap2` valid matches of a pair; the weighted
    eight-point and the global BA (Schur complement, like Ceres' DENSE_SCHUR) run on all matches.
    Returns (matcher seconds, pose seconds)."""
    from oracle.matcher_torch import matcher_forward
    from oracle import pose as P, mvba as M
    T = cfg['views']
    one = {k: (v[b:b + 1] if isinstance(v, np.ndarray) and not k.startswith('image') else v) for k, v in data_np.items()}
    t0 = time.time()
    res = matcher_forward(sd, {'GNN_layers': cfg['layers'], 'multi_frame_matching': cfg['kind'] == 'tuple'}, one)
    t1 = time.time()
    K = one['intr0'].astype(np.float64)
    rel, weight, pm, inl = {}, {}, {}, {}
    for j in range(T):
        for i in range(j):
            m = res['matches%d_%d_%d' % (i, i, j)][0]
            c = res['conf_scores_%d_%d' % (i, j)][0, :, 0].astype(np.float64)
            valid = np.nonzero((m >= 0) & (c > 0))[0]
            if valid.size < 8:
                continue
            k0 = one['keypoints%d' % i][0][valid].astype(np.float64)[None]
            k1 = one['keypoints%d' % j][0][m[valid]].astype(np.float64)[None]
            Tw, info = P.estimate_relative_pose_w8pt(k0, k1, K, K, c[valid][None, :, None], determine_inliers=True)
            cn = info['confidence'].copy()
            cn[~info['pos_depth_mask']] = 0
            ext, vb = P.run_bundle_adjust_2_view(info['kpts0_norm'][:, :cap2], info['kpts1_norm'][:, :cap2], cn[:, :cap2], Tw, 10)
            rel[(i, j)], weight[(i, j)] = (ext[0] if vb[0] else Tw[0]), int(valid.size)
            pm[(i, j)] = (info['kpts0_norm'][0], info['kpts1_norm'][0], c[valid])
            inl[(i, j)] = int(info['inliers'].sum())
    if cfg['kind'] == 'tuple' and rel:
        from oracle.ba_init import ba_initialize
        extr0, tree = M.spanning_tree_extrinsics(T, rel, weight)
        keep = {k: v for k, v in rel.items() if inl[k] >= 20 or k in tree}
        extr0 = ba_initialize(T, extr0, keep)
        M.solve_schur(M.build_problem(T, pm, extr0))
    return t1 - t0, time.time() - t1


def cpu_threads():
    """The torch port scales badly beyond ~32 threads on the many small ops of the matcher (128 host threads were
    2.5x slower than 8 on the same tuple): use at most 32, and say so in `cores`."""
    return max(1, min(os.cpu_count() or 1, 32))


def pose_auc_parity(cfg, model, sd, dev, n_units=32):
    """Engine and CPU oracle on the SAME n_units synthetic units (reduced keypoint count so that the oracle's dense
    two-view BA stays tractable; full layer stack, same weights): AUC@5/10/20 of both, eval_multi_view.py:53-87 /
    eval_pairs.py:262-277."""
    import torch
    from oracle import pipeline as OP
    from e2e_multi_view_matching_b200.pipeline import MultiViewPipeline, PairPipeline, pose_auc, compute_pose_error_np
    N = cfg['parity_kpts']
    data = make_inputs(cfg, cfg['seed_base'] + 500, n_units, kpts=N)
    tdata = {k: (torch.from_numpy(v).to(dev) if isinstance(v, np.ndarray) and not k.startswith('image') else
                 (torch.empty(v.shape, device='meta') if isinstance(v, np.ndarray) else v)) for k, v in data.items()}
    t0 = time.time()
    if cfg['kind'] == 'tuple':
        _, pose = MultiViewPipeline(model)(tdata)
        eng = [e[0] for e in MultiViewPipeline.pair_errors(tdata, pose, cfg['views'])]
        ora = [e[0] for b in range(n_units) for e in OP.tuple_errors(sd, cfg['layers'], data, b)]
    else:
        _, pose = PairPipeline(model, eval_mode='w8pt_ba')(tdata)
        Tp, ok = pose['T_021'].double().cpu().numpy(), pose['success'].cpu().numpy()
        eng, ora = [], []
        for b in range(n_units):
            gt = np.linalg.inv(data['pose1'][b].astype(np.float64)) @ data['pose0'][b].astype(np.float64)
            eng.append(max(compute_pose_error_np(gt, Tp[b, :3, :3], Tp[b, :3, 3])) if ok[b] else np.inf)
            ora.append(OP.pair_error(sd, cfg['layers'], data, b))
    eng, ora = np.array(eng), np.array(ora)
    ae = [100 * a for a in pose_auc(eng, [5, 10, 20])]
    ao = [100 * a for a in pose_auc(ora, [5, 10, 20])]
    fin = np.isfinite(eng) & np.isfinite(ora)
    return {'workload': '%d x (%d views x %d kpts, %d layers)' % (n_units, cfg['views'], N, len(cfg['layers'])),
            'engine': [round(x, 3) for x in ae], 'oracle': [round(x, 3) for x in ao],
            'max_abs_diff_pt': round(max(abs(x - y) for x, y in zip(ae, ao)), 4),
            'median_abs_pose_error_diff_deg': float(np.median(np.abs(eng[fin] - ora[fin]))) if fin.any() else None,
            'n_errors': int(eng.size), 'seconds': round(time.time() - t0, 1)}


def torch_gpu_port(cfg, sd, data_np, dev, B, stage_ms):
    import torch
    from oracle.matcher_torch import matcher_forward
    nb = min(B, 4)                                      # the port materialises prob[B,4,N,4N]: keep the batch small
    data = {k: (v[:nb] if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[0] == B else v) for k, v in data_np.items()
            if not k.startswith(('landmark', 'pose', 'extr'))}
    data = {k: (torch.empty(v.shape, device='meta') if k.startswith('image') else torch.from_numpy(v).to(dev))
            if isinstance(v, np.ndarray) else v for k, v in data.items()}
    mcfg = {'GNN_layers': cfg['layers'], 'multi_frame_matching': cfg['kind'] == 'tuple'}
    out = {}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for name, tf32 in (('tf32_allowed', True), ('fp32', False)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(2):
                matcher_forward(sd, mcfg, data, device=dev, to_numpy=False)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(3):
                matcher_forward(sd, mcfg, data, device=dev, to_numpy=False)
            e1.record()
            torch.cuda.synchronize()
            out['matcher_units_per_s_' + name] = 3 * nb / (e0.elapsed_time(e1) * 1e-3)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    ours = sum(stage_ms.get(k, 0.0) for k in ('gemm', 'attention', 'sinkhorn', 'score_gemm', 'match', 'conf', 'kenc'))
    out['ours_matcher_units_per_s'] = B / (ours * 1e-3)
    out['note'] = ('torch port of the reference matcher (oracle/matcher_torch.py) in eager stock PyTorch on the same GPU, '
                   'batch %d; matcher only; tf32_allowed = torch 1.10 defaults' % nb)
    return out


def run_reference_arm(args, cfg, rank, world):
    """`--impl reference`: the CPU port of the reference path on the host cores, honouring --steps / --warmup; a step
    is ONE unit of the same workload (the GPU arm's step is `batch` units; both report units per second)."""
    if rank != 0:
        return
    import torch
    torch.set_num_threads(cpu_threads())
    sd = make_weights(cfg)
    data = make_inputs(cfg, cfg['seed_base'], 1)
    for _ in range(args.warmup):
        cpu_reference_unit(cfg, sd, data)
    t0 = time.time()
    tm = tp = 0.0
    for _ in range(args.steps):
        a, b_ = cpu_reference_unit(cfg, sd, data)
        tm, tp = tm + a, tp + b_
    dt = time.time() - t0
    val = args.steps / dt
    sample = ('1 %s/step: matcher full size (%dx%d kpts, %d layers, 100 Sinkhorn iters, conf head) %.1f s + pose stage %.1f s '
              '(w8pt and global BA on all matches; the dense (6+3n)^2 two-view BA of the reference on the first 128 '
              'matches of a pair)' % (cfg['kind'], cfg['views'], cfg['kpts'], len(cfg['layers']), tm / args.steps, tp / args.steps))
    line = {'impl': 'reference', 'metric': cfg['metric'], 'value': val, 'unit': cfg['unit'], 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * dt / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32 (matcher) / f64 (pose)', 'data': 'synthetic',
            'config': workload_config(cfg), 'units_per_step': 1,
            'cpu_baseline': {'value': val, 'unit': cfg['unit'], 'cores': cpu_threads(), 'kind': 'port', 'sample': sample},
            'e2e': {'value': val, 'unit': cfg['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    emit(line)


def run_train_arm(args, cfg, rank, world, local):
    """--config cfg5: training iterations per second (training.train_step: train-mode forward with batch-statistics
    BatchNorm, CUDA match loss, MatcherTrainFn backward on the kernels, bucketed gradient all-reduce over NCCL when
    world > 1, torch.optim.Adam like train.py:360).  Data parallel: every rank trains on its own tuples (weak scaling:
    the global batch grows with the ranks, steps/s should stay flat); `tuples_per_s` is the whole-job rate."""
    if args.impl == 'reference':
        if rank == 0:
            emit({'impl': 'reference', 'unavailable': 'cfg5 reference arm: the reference\'s training step needs its own '
                  'autograd on the host CPU (minutes per step at this size); the gradients are pinned by the committed '
                  'reference goldens instead (tests/golden/train_backward_*.npz)'})
        return
    import types
    import torch
    import torch.distributed as dist
    from e2e_multi_view_matching_b200 import _lib, sharding, training
    from e2e_multi_view_matching_b200.models.multi_view_matcher import MultiViewMatcher
    from e2e_multi_view_matching_b200.synthetic import landmark_gt_matches
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.lib()
    B, T = args.tuples or cfg['batch'], cfg['views']
    P = n_pairs(cfg)
    sd = make_weights(cfg)
    model = MultiViewMatcher({'GNN_layers': cfg['layers'], 'multi_frame_matching': True, 'conf_mlp': False, 'full_output': False})
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items() if not k.startswith('conf_mlp')})
    model = model.to(dev).train()
    opt = types.SimpleNamespace(pose_loss=False, rot_weight=0.0, trans_weight=0.0)
    optimizer = torch.optim.Adam(model.parameters(), lr=1e-4)
    data_np = make_inputs(cfg, sharding.tuple_shard(rank, world, B, base=cfg['seed_base'])[0], B)
    for b_ in range(T):
        for a_ in range(b_):
            data_np['gt_indices_%d_%d' % (a_, b_)], data_np['gt_weights_%d_%d' % (a_, b_)] = \
                landmark_gt_matches(data_np['landmark%d' % a_], data_np['landmark%d' % b_])
    keys = [k for k, v in data_np.items() if isinstance(v, np.ndarray) and k.startswith(('keypoints', 'scores', 'descriptors', 'gt_'))]
    host = {k: torch.from_numpy(data_np[k]).pin_memory() for k in keys}
    meta = {k: torch.empty(v.shape, device='meta') for k, v in data_np.items() if k.startswith('image')}
    fixed = dict(meta, ids=data_np['ids'], pose0=torch.zeros(1, device=dev))
    data_dev = dict({k: v.to(dev) for k, v in host.items()}, **fixed)
    h2d_bytes = sum(v.numel() * v.element_size() for v in host.values())
    loss_host = torch.zeros(1).pin_memory()
    last = {}

    def step_device():
        last['loss'], last['losses'] = training.train_step(opt, dict(data_dev), model, optimizer, P)
        return last['loss']

    def step_e2e():
        d = dict({k: v.to(dev, non_blocking=True) for k, v in host.items()}, **fixed)
        loss = training.train_step(opt, d, model, optimizer, P)[0]
        loss_host.copy_(loss.reshape(1), non_blocking=True)
        return loss

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for a, b in evs:
            flush.zero_()
            a.record()
            fn()
            b.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return sharding.max_over_ranks(sum(a.elapsed_time(b) for a, b in evs), dev)

    losses = []
    for _ in range(args.warmup):
        losses.append(float(step_device()))
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.mvm_launch_count()
    ms_dev = timed(step_device, args.steps)
    launches = lib.mvm_launch_count() - n0
    if args.dump_outputs and rank == 0:
        # a training step returns its losses and leaves the gradients and the updated weights in the model
        named = list(model.named_parameters())
        dump_outputs(args.dump_outputs, dict(last['losses'], loss=last['loss'],
                                             **{'grad.' + k: p.grad for k, p in named if p.grad is not None},
                                             **{'param.' + k: p for k, p in named}))
    ms_e2e = timed(step_e2e, args.steps)
    sampler.stop_flag = True
    losses.append(float(step_device()))
    # stage split (CUDA events around forward / backward / optimiser of two more steps) and the kernel-class timers
    lib.mvm_profile_enable(1)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    split = np.zeros(3)
    for _ in range(2):
        d = dict(data_dev)
        ev[0].record()
        ls, _ = training.run_matcher(opt, d, model)
        loss, _ = training.combine_losses(ls, P, 0.0, 0.0, 0.0)
        ev[1].record()
        optimizer.zero_grad(set_to_none=True)
        loss.backward()
        ev[2].record()
        sharding.all_reduce_gradients(list(model.parameters()))
        optimizer.step()
        ev[3].record()
        torch.cuda.synchronize()
        split += [ev[i].elapsed_time(ev[i + 1]) / 2 for i in range(3)]
    prof = _lib.profile_collect()
    lib.mvm_profile_enable(0)
    if rank == 0:
        peaks = load_peaks()
        att_ms, att_n = prof['attention']
        # algorithmic work: forward QK^T + PV (4 N M D per view and layer) + the five products of a memory-efficient
        # backward (S recomputed once, dP = dO V^T, dQ = dS K, dK = dS^T Q, dV = P^T dO: 10 N M D) = 14 N M D.  The two
        # backward kernels EXECUTE eight (S three times, dP twice); the lines committed as profiles/bench_r02_cfg5_*.json
        # were taken with 18 N M D in this place.
        att_flops = attention_flops(cfg) * B * 2 * (14.0 / 4.0)
        att_tflops = att_flops / (att_ms * 1e-3) / 1e12 if att_ms > 0 else 0.0
        line = {'metric': cfg['metric'], 'value': args.steps / (ms_dev * 1e-3), 'unit': cfg['unit'], 'n_gpus': world,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms_dev / args.steps, 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None,
                'dtype': 'f32 via split operands on the tensor cores (fp16x3 forward, tf32x3 backward GEMMs and attention backward), f32 CUDA cores (Sinkhorn, BatchNorm)',
                'data': 'synthetic', 'config': workload_config(cfg), 'units_per_step': B * world,
                'tuples_per_s': B * world * args.steps / (ms_dev * 1e-3),
                'run': {'tuples_per_step_per_gpu': B, 'l2': 'flushed between timed steps (256 MB write)', 'parallelism': 'dp%d' % world,
                        'optimizer': 'torch.optim.Adam (train.py:360)', 'collective': 'bucketed gradient all-reduce (sharding.all_reduce_gradients)' if world > 1 else 'none',
                        'stage': 'stage 1 of cfg5 (match loss); stage 2 (--pose_loss) is not built'},
                'e2e': {'value': args.steps / (ms_e2e * 1e-3), 'unit': cfg['unit'], 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': 4,
                        'ms_per_step': ms_e2e / args.steps},
                'gpu_launches': int(launches), 'clocks': sampler.summary(),
                'roofline': {'kernel': 'attention forward (tcgen05 fp16x3) + backward (mma.sync TF32 x 3 split passes, flash-style recomputation)',
                             'bound': 'tensor', 'achieved': att_tflops, 'peak': peaks['tflops'], 'unit': 'TFLOP/s',
                             'frac': att_tflops / peaks['tflops'], 'traffic': None, 'launches_timed': att_n, 'peak_source': peaks['source'],
                             'note': 'the backward runs on the legacy mma.sync path with register fragments; its tcgen05 port is the next step'},
                'step_split_ms': {'forward+loss': round(float(split[0]), 3), 'backward': round(float(split[1]), 3),
                                  'allreduce+optimizer': round(float(split[2]), 3)},
                'stage_ms_per_step': {k: round(v[0] / 2, 4) for k, v in prof.items() if v[1] > 0},
                'loss_first_last': [losses[0], losses[-1]], 'cpu_baseline': None}
        if world == 1:
            emit(line)
    if world > 1:       # the JSON line last: the other ranks tear their communicators down (and NCCL logs that) first
        dist.barrier()
        if rank != 0:
            dist.destroy_process_group()
        else:
            time.sleep(2.0)
            dist.destroy_process_group()
            emit(line)
            if os.environ.get('NCCL_DEBUG', '').upper() in ('INFO', 'TRACE'):
                os._exit(0)


# ---------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='cfg3', choices=sorted(CONFIGS),
                    help='BASELINE.json configs: cfg3 = 5-view tuples (headline, default), cfg2 / cfg4 = two-view pairs')
    ap.add_argument('--tuples', type=int, default=0, help='units (tuples / pairs) per step per GPU (0 = the config default)')
    ap.add_argument('--no-cpu-baseline', action='store_true', help='skip the CPU legs (cpu_baseline, AUC parity)')
    ap.add_argument('--no-torch-gpu', action='store_true', help='skip the informational stock-PyTorch-on-GPU matcher line')
    ap.add_argument('--gemm-tile', type=int, default=256, choices=[128, 256])
    ap.add_argument('--gemm-kernel', default='persistent', choices=['persistent', 'tile'],
                    help='3xTF32 GEMM kernel: persistent (default) or the one-tile-per-CTA kernel (A/B comparison)')
    ap.add_argument('--attn-split', type=int, default=-1, choices=[-1, 0, 1],
                    help='operand planes of the mode-3 attention: 0 = tf32 hi/lo, 1 = fp16 hi/lo, -1 = library default')
    ap.add_argument('--gemm-split', type=int, default=-1, choices=[-1, 0, 1],
                    help='operand planes of the mode-3 layer GEMMs (persistent kernel): 0 = tf32 hi/lo, 1 = fp16 hi/lo')
    ap.add_argument('--math-mode', type=int, default=3, choices=[0, 1, 3],
                    help='3 = tcgen05 3xTF32 (fp32-faithful, default), 1 = tcgen05 single-pass TF32, 0 = fp32 CUDA cores')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the arrays the last timed step returned as DIR/<name>.npy (float32 / float64, '
                         'at most 64 MB in all: larger outputs are stored as a fixed, seeded sample)')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs records the outputs of --impl ours')
    cfg = CONFIGS[args.config]
    args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if cfg['kind'] == 'train':
        run_train_arm(args, cfg, rank, world, local)
        return
    if args.impl == 'reference':
        run_reference_arm(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist
    from e2e_multi_view_matching_b200 import _lib
    from e2e_multi_view_matching_b200.models.multi_view_matcher import MultiViewMatcher
    from e2e_multi_view_matching_b200.pipeline import MultiViewPipeline, PairPipeline, pose_auc, compute_pose_error_np
    from e2e_multi_view_matching_b200 import sharding

    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    lib = _lib.lib()
    lib.mvm_set_math_mode(args.math_mode)
    lib.mvm_debug_set_gemm_tile(args.gemm_tile)
    lib.mvm_debug_set_gemm_kernel(1 if args.gemm_kernel == 'persistent' else 0)
    if args.attn_split >= 0:
        lib.mvm_debug_set_attention_split(args.attn_split)
    if args.gemm_split >= 0:
        lib.mvm_debug_set_gemm_split(args.gemm_split)
    opt = _lib.MatcherOptions()
    lib.mvm_matcher_options_default(opt)
    B = args.tuples or cfg['batch']
    T_VIEWS, N_KPTS, LAYERS = cfg['views'], cfg['kpts'], cfg['layers']
    is_tuple = cfg['kind'] == 'tuple'
    P = n_pairs(cfg)

    sd = make_weights(cfg)
    model = MultiViewMatcher({'GNN_layers': LAYERS, 'multi_frame_matching': is_tuple}).eval()
    model.load_state_dict({k: torch.from_numpy(np.asarray(v)) for k, v in sd.items()})
    model = model.to(dev)
    pipe = MultiViewPipeline(model) if is_tuple else PairPipeline(model, eval_mode='w8pt_ba')

    # units base + (rank*B + k): every rank works on its own shard (weak scaling, no data-path collective)
    data_np = make_inputs(cfg, sharding.tuple_shard(rank, world, B, base=cfg['seed_base'])[0], B)
    keys = [k for k, v in data_np.items() if isinstance(v, np.ndarray) and not k.startswith(('image', 'landmark'))]
    host = {k: torch.from_numpy(data_np[k]).pin_memory() for k in keys}
    meta = {k: torch.empty(v.shape, device='meta') for k, v in data_np.items() if k.startswith('image')}
    data_dev = {k: v.to(dev) for k, v in host.items()}
    data_dev.update(meta)
    data_dev['ids'] = data_np['ids']
    h2d_keys = [k for k in keys if not k.startswith(('pose', 'extr'))]
    h2d_bytes = sum(host[k].numel() * host[k].element_size() for k in h2d_keys)
    if is_tuple:
        out_host = {'extrinsics': torch.empty(B, T_VIEWS, 4, 4).pin_memory(), 'T_pair': torch.empty(B, P, 4, 4).pin_memory()}
    else:
        out_host = {'T_021': torch.empty(B, 4, 4).pin_memory()}
    d2h_bytes = sum(v.numel() * v.element_size() for v in out_host.values())
    loss = torch.zeros(1, device=dev)

    last = {}

    def step_loss(pose):
        return (pose['ba_cost'][:, 1].sum() if is_tuple else pose['T_021'].sum()).float().reshape(1)

    def step_device():
        res, pose = pipe(data_dev)
        last['res'], last['pose'] = res, pose
        if world > 1:   # the per-rank loss is accumulated on the device; ONE all-reduce closes the timed region
            loss.add_(step_loss(pose))
        return pose

    # End-to-end step through the public API.  Every step's inputs come from pinned host memory into one of two
    # PERSISTENT device input sets (allocated once: a per-step allocation on the copy stream made the caching
    # allocator grow and synchronise, 30-70 ms hiccups in the cfg2 / cfg4 e2e steps of r02_v10): the copy of step
    # k+1 is issued on a copy stream right after step k's kernels are enqueued, so it overlaps step k's compute; a
    # set is overwritten only after the step that read it has finished (event on the compute stream); the step's
    # result (poses) is read back to pinned host memory.
    copy_stream = torch.cuda.Stream(device=dev)
    dev_in = [{k: torch.empty_like(host[k], device=dev) for k in h2d_keys} for _ in range(2)]
    consumed = [None, None]          # compute-stream event: the last step that read this set has been enqueued
    staged = {}
    e2e_count = [0]

    def stage_inputs(slot):
        with torch.cuda.stream(copy_stream):
            if consumed[slot] is not None:
                copy_stream.wait_event(consumed[slot])
            for k in h2d_keys:
                dev_in[slot][k].copy_(host[k], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        staged[slot] = ev

    def step_e2e():
        slot = e2e_count[0] % 2
        e2e_count[0] += 1
        if slot not in staged:
            stage_inputs(slot)
        torch.cuda.current_stream().wait_event(staged.pop(slot))
        d = dict(dev_in[slot])
        d.update(meta)
        d['ids'] = data_np['ids']
        res, pose = pipe(d)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream())
        consumed[slot] = done
        stage_inputs(1 - slot)                       # next step's H2D, overlapped with this step's kernels
        for k, v in out_host.items():
            v.copy_(pose[k], non_blocking=True)
        if world > 1:
            loss.add_(step_loss(pose))
        return pose

    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def timed(fn, steps):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.time()
        if world > 1:
            loss.zero_()
        for a, b in evs:
            flush.zero_()                      # L2 flush between timed iterations (outside the events)
            a.record()
            fn()
            b.record()
        if world > 1:
            # the path shards by tuple with no data-path exchange; the one collective is the scalar loss all-reduce
            # after the loop, as the reference's validation pass does (train.py:104-106) -- not once per step, which
            # would couple every step to the slowest rank
            sharding.all_reduce_step_loss(loss)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        wall = time.time() - t0
        per_step = [a.elapsed_time(b) for a, b in evs]
        last['per_step_ms'] = per_step
        ms = sum(per_step)
        return sharding.max_over_ranks(ms, dev), wall

    for _ in range(args.warmup):
        step_device()
        step_e2e()
    torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    n0 = lib.mvm_launch_count()
    ms_dev, wall_dev = timed(step_device, args.steps)
    launches = lib.mvm_launch_count() - n0
    if args.dump_outputs and rank == 0:
        # pose is None when fewer than two views have keypoints (pipeline.py); its arrays carry a 'pose.' prefix
        dump_outputs(args.dump_outputs, dict(last['res'], **{'pose.' + k: v for k, v in (last['pose'] or {}).items()}))
    staged.clear()                 # the first timed step stages its own inputs inside the timed region
    ms_e2e, wall_e2e = timed(step_e2e, args.steps)
    e2e_steps = [round(x, 2) for x in last['per_step_ms']]
    sampler.stop_flag = True

    # secondary line: the same steps in single-pass TF32 (what torch 1.10 ran on Ampere by default)
    tf32 = None
    if args.math_mode == 3:
        lib.mvm_set_math_mode(1)
        for _ in range(2):
            step_device()
        ms_tf32, _ = timed(step_device, args.steps)
        staged.clear()
        ms_tf32_e2e, _ = timed(step_e2e, args.steps)
        lib.mvm_set_math_mode(3)
        tf32 = (ms_tf32, ms_tf32_e2e)

    # live per-kernel-class timing (CUDA events on the launching stream) over two more steps
    lib.mvm_profile_enable(1)
    prof_steps = 2
    for _ in range(prof_steps):
        flush.zero_()
        pose = step_device()
    torch.cuda.synchronize()
    prof = _lib.profile_collect()
    lib.mvm_profile_enable(0)

    if rank == 0:
        peaks = load_peaks()
        clocks = sampler.summary()
        total_units = B * args.steps * world
        value = sharding.whole_job_throughput(B, args.steps, world, ms_dev)
        e2e = total_units / (ms_e2e * 1e-3)
        traffic_att, traffic_sink = load_traffic(cfg['workload'], B)
        att_ms, att_n = prof['attention']
        att_flops = attention_flops(cfg) * B * prof_steps                  # over the profiled steps
        att_tflops = att_flops / (att_ms * 1e-3) / 1e12 if att_ms > 0 else 0.0
        sk_ms, sk_n = prof['sinkhorn']
        n_prob = P * B * prof_steps
        sk_gbs = sinkhorn_bytes_per_problem(cfg) * n_prob / (sk_ms * 1e-3) / 1e9 if sk_ms > 0 else 0.0
        # what the production kernel really streams: K~ is resident ON CHIP (registers + shared memory), two passes
        # over it per iteration; peak = SMs x 128 B/clk x SM clock (shared-memory datapath)
        onchip_gbs = 100 * 2 * N_KPTS * N_KPTS * 4 * n_prob / (sk_ms * 1e-3) / 1e9 if sk_ms > 0 else 0.0
        sm_mhz = clocks.get('sm_mhz') or 1965.0
        smem_peak_gbs = 148 * 128 * sm_mhz * 1e6 / 1e9
        stage_ms = {k: round(v[0] / prof_steps, 4) for k, v in prof.items() if v[1] > 0}
        # pose AUC of the engine on the bench units (informational; engine-vs-oracle parity below and in tests/)
        if is_tuple:
            errs = [e[0] for e in MultiViewPipeline.pair_errors({k: v for k, v in data_dev.items() if k.startswith('pose')}, pose, T_VIEWS)]
        else:
            Tp, ok = pose['T_021'].double().cpu().numpy(), pose['success'].cpu().numpy()
            errs = []
            for i in range(B):
                gt = np.linalg.inv(data_np['pose1'][i].astype(np.float64)) @ data_np['pose0'][i].astype(np.float64)
                errs.append(max(compute_pose_error_np(gt, Tp[i, :3, :3], Tp[i, :3, 3])) if ok[i] else np.inf)
        auc = pose_auc(np.array(errs), [5, 10, 20])
        last_res = last['res']
        # issue-rate ceiling of the arithmetic the attention kernel really runs: kind::tf32 = 4096 FLOP/clk/SM, kind::f16
        # twice that; the fp32-faithful modes spend three MMAs per product
        if args.math_mode == 3:
            ceiling = (2.0 if opt.attention_split == 1 else 1.0) * TF32_PEAK_TFLOPS / 3.0
            ceiling_name = 'fp16x3' if opt.attention_split == 1 else 'tf32x3'
        else:
            ceiling, ceiling_name = TF32_PEAK_TFLOPS, 'tf32'

        line = {
            'metric': cfg['metric'], 'value': value, 'unit': cfg['unit'], 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': {3: 'f32 via split operands on tcgen05 (fp16x3 / tf32x3, fp32-faithful) / f64 pose kernels', 1: 'tf32 on tcgen05 / f64 pose kernels',
                      0: 'f32 CUDA cores / f64 pose kernels'}[args.math_mode], 'data': 'synthetic',
            'config': workload_config(cfg), 'units_per_step': B * world,
            'run': {'units_per_step_per_gpu': B, 'l2': 'flushed between timed steps (256 MB write)',
                    'math_mode': args.math_mode, 'attention_split': {0: 'tf32 hi/lo', 1: 'fp16 hi/lo'}[opt.attention_split],
                    'gemm_split': {0: 'tf32 hi/lo', 1: 'fp16 hi/lo'}[opt.gemm_split],
                    'parallelism': 'dp%d' % world,
                    'weights': 'seeded random GNN (final_proj gain 12) + score-driven confidence head (synthetic.py)'},
            'e2e': {'value': e2e, 'unit': cfg['unit'], 'h2d_bytes_per_step': h2d_bytes, 'd2h_bytes_per_step': d2h_bytes,
                    'ms_per_step': ms_e2e / args.steps, 'ms_steps': e2e_steps,
                    'h2d': 'pinned host -> device on a copy stream, step k+1 staged under step k'},
            'gpu_launches': int(launches),
            'clocks': clocks,
            'roofline': {'kernel': 'attention (QK^T + PV, all views of one GNN layer per launch)', 'bound': 'tensor',
                         'achieved': att_tflops, 'peak': peaks['tflops'], 'unit': 'TFLOP/s',
                         'frac': att_tflops / peaks['tflops'], 'traffic': traffic_att, 'launches_timed': att_n,
                         'peak_source': peaks['source'],
                         # the path computes in tf32 (half the bf16 rate: M128.N.K8 every N/2 cycles = 4096 FLOP/clk/SM)
                         # and needs three passes to stay fp32-faithful: the reachable algorithmic ceiling
                         'ceiling': ceiling, 'ceiling_arithmetic': ceiling_name, 'frac_of_ceiling': att_tflops / ceiling},
            'roofline_sinkhorn': {'kernel': 'sinkhorn (%d pairs x %d problems per launch)' % (P, B),
                                  'bound': 'on-chip (K~ resident in registers + shared memory; not HBM)',
                                  'achieved': onchip_gbs, 'peak': smem_peak_gbs, 'unit': 'GB/s',
                                  'frac': onchip_gbs / smem_peak_gbs, 'launches_timed': sk_n,
                                  'peak_source': '148 SMs x 128 B/clk x sampled SM clock (shared-memory datapath)',
                                  # SURVEY.md 8(d)'s per-unit figure (the reference's HBM passes) over the same time
                                  'hbm_equivalent': {'achieved': sk_gbs, 'peak': peaks['hbm_gbs'], 'frac': sk_gbs / peaks['hbm_gbs'],
                                                     'unit': 'GB/s', 'traffic': traffic_sink}},
            'stage_ms_per_step': stage_ms,
            'wall_s': {'device_resident': wall_dev, 'e2e': wall_e2e},
            'pose_auc_5_10_20': [round(100 * a, 2) for a in auc],
        }
        if tf32 is not None:
            line['tf32_single_pass'] = {'value': total_units / (tf32[0] * 1e-3), 'e2e': total_units / (tf32[1] * 1e-3),
                                        'unit': cfg['unit'], 'note': 'math mode 1 (tcgen05 kind::tf32, one pass)'}
        # quality of the synthetic assignment: fraction of returned matches that join the same landmark
        hits = tot = 0
        for b_ in range(T_VIEWS):
            for a_ in range(b_):
                m = last_res['matches%d_%d_%d' % (a_, a_, b_)].cpu().numpy()
                la, lb = data_np['landmark%d' % a_], data_np['landmark%d' % b_]
                for i in range(B):
                    v = m[i] >= 0
                    hits += int((la[i][v] == lb[i][m[i][v]]).sum()); tot += int(v.sum())
        line['match_precision'] = round(hits / max(tot, 1), 4)
        if world == 1 and not args.no_torch_gpu:
            # informational: the op-for-op torch port of the reference matcher run by stock PyTorch (cuBLAS / cuDNN
            # eager) on the same GPU -- what a user of the reference gets by moving its model to the B200.  Matcher
            # only (the reference's pose stage is CPU code); our matcher-only rate from the stage timers beside it.
            try:
                line['torch_gpu_port'] = torch_gpu_port(cfg, sd, data_np, dev, B, stage_ms)
            except Exception as e:                                  # never let the extra line break the bench
                line['torch_gpu_port'] = {'error': repr(e)[:200]}
        if world == 1 and not args.no_cpu_baseline:
            torch.set_num_threads(cpu_threads())
            t_m, t_p = cpu_reference_unit(cfg, sd, data_np)
            line['cpu_baseline'] = {
                'value': 1.0 / (t_m + t_p), 'unit': cfg['unit'], 'cores': cpu_threads(), 'kind': 'port',
                'sample': '1 %s: matcher full size %.1f s + pose stage %.1f s (w8pt and global BA on all matches, the '
                          'dense two-view BA on the first 128 matches of a pair)' % (cfg['kind'], t_m, t_p)}
            try:
                line['pose_auc_parity'] = pose_auc_parity(cfg, model, sd, dev)
            except Exception as e:
                line['pose_auc_parity'] = {'error': repr(e)[:300]}
        if world == 1:
            emit(line)
    if world > 1:
        # the JSON line must be the LAST line of the job's output: every other rank tears its communicator down (and
        # NCCL logs that) first, rank 0 follows and prints
        dist.barrier()
        if rank != 0:
            dist.destroy_process_group()
        else:
            time.sleep(2.0)
            dist.destroy_process_group()
            emit(line)
            if os.environ.get('NCCL_DEBUG', '').upper() in ('INFO', 'TRACE'):
                os._exit(0)          # NCCL logs its unload at interpreter exit: keep the JSON line last


if __name__ == '__main__':
    main()
