#!/usr/bin/env python
"""Benchmark of the SM3Det sparse-MoE backbone hot path (BASELINE.json metric: backbone images/s @1024^2, bs = 32).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--config t_e8|b_e16|lsk_s] [--global-batch G | --batch B] [--expert-parallel] [--dump-outputs DIR]

One "step" = forward + backward of the backbone over the GLOBAL batch of synthetic 1024^2 tiles:
  t_e8  (default) BASELINE configs[1]/[2]: ConvNeXt-T, E = 8 top-2, MoE in the last two stages every other block.
        Global batch 32 at every N (the batch the metric is quoted on) -> strong scaling: 32 / 16 / 8 / 4 images per GPU at
        N = 1 / 2 / 4 / 8, each GPU's share in ONE forward/backward pass (61 GB of activations at 32 images; `--micro-batch 8`
        splits it with gradient accumulation, measured 4 % slower; `--global-batch 8` is configs[1] literally).  N > 1: one
        process per GPU (torchrun), one flat gradient all-reduce per step over NCCL, captured in the step's CUDA graph
        (`--cuda-graph off` = eager launches under DistributedDataParallel).  Gating is the reference constructor's default
        (noisy top-k while training); `--noisy-gating off` = deterministic routing.
  b_e16 BASELINE configs[3]: ConvNeXt-B, E = 16, all 36 blocks MoE; experts sharded over the ranks when N > 1.
  lsk_s BASELINE configs[4]: LSKNet-S MoE, SyncBN, global batch 16 (4 GPUs -> 4 per GPU).
The timed region is bracketed by barrier + synchronize and the max over ranks is reported.  `--impl reference` times the
reference's own CPU implementation of the same path (the oracle port: identical torch CPU ops in the reference's order)
on the box's host cores.
"""
import argparse
import contextlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'backbone images/sec @1024^2 (fwd+bwd)'
NOISY_DEFAULT = 'config'
CONFIGS = {
    't_e8': dict(family='convnext', global_batch=32, micro=32,
                 kw=dict(arch='tiny', MoE_Block_inds=[[], [], [0, 2, 4, 6, 8], [0, 2]], num_experts=8, top_k=2,
                         noisy_gating=True, drop_path_rate=0.0),
                 name='SM3Det ConvNeXt-T e8t2 last-2-blocks MoE backbone (BASELINE configs[1]/[2])'),
    'b_e16': dict(family='convnext', global_batch=8, micro=2,
                  kw=dict(arch='base', MoE_Block_inds=[[0, 1, 2], [0, 1, 2], list(range(27)), [0, 1, 2]], num_experts=16,
                          top_k=2, noisy_gating=True, drop_path_rate=0.0),
                  name='SM3Det ConvNeXt-B e16t2 all-blocks MoE backbone (BASELINE configs[3])'),
    'lsk_s': dict(family='lsk', global_batch=16, micro=4,
                  kw=dict(MoE_Block_inds_fc1=[[], [0], [0, 2], [0]], MoE_Block_inds_fc2=[[], [0], [0, 2], [0]], num_experts=4,
                          top_k=2, embed_dims=[64, 128, 320, 512], depths=[2, 2, 4, 2], drop_rate=0.1, drop_path_rate=0.,
                          norm_cfg=dict(type='SyncBN', requires_grad=True)),
                  name='SM3Det LSKNet-S MoE backbone, SyncBN, noisy gating + dropout as configured (BASELINE configs[4])'),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=6)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--config', default='t_e8', choices=sorted(CONFIGS))
    ap.add_argument('--global-batch', type=int, default=None, help='images per step over all GPUs (strong scaling)')
    ap.add_argument('--batch', type=int, default=None, help='images per GPU per step (weak scaling; overrides --global-batch)')
    ap.add_argument('--micro-batch', type=int, default=None, help='images per forward/backward pass (gradient accumulation)')
    ap.add_argument('--size', type=int, default=1024)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-gpu-eager', action='store_true')
    ap.add_argument('--amp', action='store_true', help='NOT the headline: run the mixed-precision recipe (single-pass bf16 GEMMs)')
    ap.add_argument('--expert-parallel', action='store_true',
                    help='N > 1: shard the experts over the ranks (NVLink peer-memory dispatch); default for --config b_e16')
    ap.add_argument('--no-expert-parallel', action='store_true')
    ap.add_argument('--cpu-images', type=int, default=1, help='images in the bounded CPU sample')
    ap.add_argument('--noisy-gating', choices=['config', 'off'], default=NOISY_DEFAULT,
                    help="ConvNeXt configs: 'config' = the reference constructor's default (noisy top-k gating while training, "
                         "what configs/SM3Det/*.py run), 'off' = deterministic routing")
    ap.add_argument('--cuda-graph', choices=['auto', 'on', 'off'], default='auto',
                    help='capture the whole step (fwd+bwd over all micro-batches, gradient all-reduce included) in a CUDA graph; '
                         'auto = on except for AMP and expert parallelism')
    ap.add_argument('--grad-sync', choices=['auto', 'ddp', 'flat'], default='auto',
                    help='N > 1: DistributedDataParallel bucket hooks, or one flat all-reduce at the end of the step (capturable); '
                         'auto = flat when the step is graph-captured')
    ap.add_argument('--no-grad-sync', action='store_true',
                    help='DIAGNOSTIC, N > 1: never all-reduce gradients (isolates the exposed cost of the DDP collective)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write what the last step returned (rank 0: feature maps, gate losses, step loss, '
                         'parameter gradients) as DIR/<name>.npy; inputs, weights and gating noise are seeded, so two builds '
                         'run with the same arguments can be compared file by file')
    a = ap.parse_args()
    if a.steps < 1:
        ap.error('--steps must be at least 1')
    if a.dump_outputs and a.impl != 'ours':
        ap.error('--dump-outputs writes the outputs of --impl ours')
    for c in CONFIGS.values():            # applies to both arms (ours and --impl reference) and to the oracle baselines
        if c['family'] == 'convnext':
            c['kw']['noisy_gating'] = a.noisy_gating == 'config'
    return a


def resolve(args, world):
    """-> (cfg entry, per-GPU batch, micro-batch, scaling)."""
    c = CONFIGS[args.config]
    if args.batch is not None:
        per, scaling = args.batch, 'weak'
    else:
        g = args.global_batch if args.global_batch is not None else c['global_batch']
        if g % world:
            raise SystemExit(f'global batch {g} is not divisible by {world} GPUs')
        per, scaling = g // world, 'strong'
    micro = min(per, args.micro_batch or c['micro'])
    while per % micro:
        micro -= 1
    ep = world > 1 and c['family'] == 'convnext' and not args.no_expert_parallel and \
        (args.expert_parallel or args.config == 'b_e16') and c['kw']['num_experts'] % world == 0
    return c, per, micro, scaling, ep


def workload_config(args, world):
    c, per, micro, scaling, ep = resolve(args, world)
    kw = c['kw']
    return {'workload': f'{c["name"]}, fwd+bwd, global batch {per * world} = {per}/GPU x {world} GPU in micro-batches of '
                        f'{micro}, {args.size}x{args.size}x3 synthetic SAR/RGB/IR 2:1:1, fp32',
            'config': args.config, 'num_experts': kw['num_experts'], 'top_k': kw['top_k'],
            'noisy_gating': bool(kw.get('noisy_gating', True)),
            'per_gpu_batch': per, 'micro_batch': micro, 'global_batch': per * world, 'image': args.size,
            'parallelism': f'dp{world}' + ('+ep' if ep else ''),
            'l2': 'inputs and activations exceed L2 (>= 100 MB per tensor); no flush needed'}


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-i', str(self.index), '-lms', '200'], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace('.', '').isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace('.', '').isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows if len(r) >= 7 for n, v in zip(names, r[3:7]) if v.lower().startswith('active')})
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': reasons, 'samples': len(sm)}


# ---- the reference's own implementation (oracle port): CPU baseline, --impl reference, GPU-eager comparator ----------
def oracle_model(config):
    """(forward(x, train) -> (outs, loss), state_dict on CPU) of the oracle port for a bench config -- test infrastructure,
    used only as a *baseline that is timed*, never on the product path."""
    from sm3det_b200.synth import make_state_dict
    c = CONFIGS[config]
    if c['family'] == 'convnext':
        from oracle.convnext_moe_oracle import OracleConfig, backbone_forward, param_shapes
        kw = dict(c['kw'])
        cfg = OracleConfig(**kw)
        sd = make_state_dict(param_shapes(cfg), 0, True)
        return (lambda s, x, train: backbone_forward(s, cfg, x, train=train)), sd
    from oracle.lsk_moe_oracle import LskConfig, lsk_backbone_forward, lsk_param_shapes
    kw = {k: v for k, v in c['kw'].items() if k != 'norm_cfg'}
    cfg = LskConfig(**kw)
    sd = make_state_dict(lsk_param_shapes(cfg), 0, True)
    return (lambda s, x, train: lsk_backbone_forward(s, cfg, x, train=train, bn_state={})), sd


def _grad_sd(sd):
    skip = ('ffn.mean', 'ffn.std', 'running_', 'num_batches', '.mean', '.std')
    return {k: (v.clone().requires_grad_(True) if v.is_floating_point() and not any(t in k for t in skip) else v) for k, v in sd.items()}


def oracle_step(fwd, sd, x):
    outs, loss = fwd(_grad_sd(sd), x, True)
    (sum(o.mean() for o in outs) + loss).backward()


def time_cpu_reference(args, images, steps, warmup):
    """fwd+bwd (the bench metric) and eval forward (what north_star names as the CPU baseline) of the oracle port."""
    from sm3det_b200.synth import make_images
    # torch's CPU kernels stop scaling (and then collapse: 143 s/img at 128 threads vs 1.5 s at 16 on the 128-thread
    # B200 host, profiles/r01_cpu_threads.txt) long before the box runs out of cores: use the best-performing count.
    threads = int(os.environ.get('SM3_CPU_THREADS', min(16, os.cpu_count() or 1)))
    torch.set_num_threads(threads)
    fwd, sd = oracle_model(args.config)
    x = make_images(images, args.size, args.size, seed=1234)
    oracle_step(fwd, sd, make_images(1, 128, 128, seed=1))     # thread-pool / allocator warm-up, not timed
    for _ in range(warmup):
        oracle_step(fwd, sd, x)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle_step(fwd, sd, x)
    dt = (time.perf_counter() - t0) / max(steps, 1)
    with torch.no_grad():
        t1 = time.perf_counter()
        fwd(sd, x, False)
        dt_fwd = time.perf_counter() - t1
    return images / dt, dt, threads, images / dt_fwd


def cpu_baseline_entry(args, ips, dt, threads, fwd_ips):
    return {'value': ips, 'unit': 'img/s', 'cores': threads, 'kind': 'port', 'host_cpus': os.cpu_count(),
            'eval_forward_img_s': fwd_ips,
            'sample': f'fwd+bwd of {args.cpu_images} workload image(s) per step (oracle port = the reference\'s torch CPU fp32 '
                      f'ops in its order), {threads} of {os.cpu_count()} host threads (torch CPU stops scaling beyond, '
                      f'profiles/r01_cpu_threads.txt), {dt:.1f} s/step; eval_forward_img_s = one eval forward of the same images'}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    ips, dt, threads, fwd_ips = time_cpu_reference(args, args.cpu_images, steps, warmup)
    _, _, _, scaling, _ = resolve(args, args.gpus)
    line = {'impl': 'reference', 'metric': METRIC, 'value': ips, 'unit': 'img/s', 'n_gpus': args.gpus, 'steps': steps,
            'warmup': warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None,
            'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args, args.gpus),
            'cpu_baseline': cpu_baseline_entry(args, ips, dt, threads, fwd_ips),
            'e2e': {'value': ips, 'unit': 'img/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


def time_gpu_eager(args, micro):
    """The GPU-side comparator (SURVEY 8d, BASELINE.md 3): the reference's own module graph -- here its oracle port, the same
    torch ops -- run in eager PyTorch on this B200 (cuBLAS / cuDNN / ATen kernels), fp32 and with TF32 allowed, timed with
    CUDA events like tools/analysis_tools/benchmark.py:118-146.  Not the product: the number our kernels have to beat."""
    from sm3det_b200.synth import make_images
    fwd, sd = oracle_model(args.config)
    torch.cuda.reset_peak_memory_stats()
    sd = {k: v.cuda() for k, v in sd.items()}
    x = make_images(micro, args.size, args.size, seed=1234).cuda()
    out = {'kind': 'oracle port (the reference\'s torch ops) in eager PyTorch on cuda:0', 'micro_batch': micro, 'unit': 'img/s'}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    try:
        for name, tf32 in (('fp32', False), ('tf32', True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(2):
                oracle_step(fwd, sd, x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n = 5
            e0.record()
            for _ in range(n):
                oracle_step(fwd, sd, x)
            e1.record()
            torch.cuda.synchronize()
            out[name] = micro * n / (e0.elapsed_time(e1) * 1e-3)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    out['peak_mem_gb'] = torch.cuda.max_memory_allocated() / 2 ** 30
    return out


# ------------------------------------------------------------------------------------------------
TENSOR_OPS = ('gemm', 'ffn_fused_fwd', 'ffn_fused_bwd')     # ops.* entry points that launch tcgen05 kernels


def gemm_roofline(step_fn, peaks):
    """Instrumented pass: CUDA-event time of every tensor-core launch in one fwd+bwd micro-batch and its algorithmic FLOPs
    (2*M*N*K per GEMM; the fused FFN kernels report the FLOPs of the GEMMs the algorithm needs, not their recomputation)."""
    from sm3det_b200 import ops
    rec = []
    orig = {n: getattr(ops, n) for n in TENSOR_OPS if hasattr(ops, n)}

    def wrap(name, fn):
        def timed(*a, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r = fn(*a, **kw)
            e1.record()
            if name == 'gemm':
                rows = kw['M']
                flops = 2.0 * rows * kw['N'] * kw['K']
                byts = 4.0 * (rows * kw['K'] + kw['N'] * kw['K'] + rows * kw['N'])
                shape = (kw['M'], kw['N'], kw['K'], kw.get('sched', 0))
            else:
                flops, byts, shape = ops.fused_cost(name, *a, **kw)
            rec.append((e0, e1, flops, byts, name, shape))
            return r
        return timed

    for n, f in orig.items():
        setattr(ops, n, wrap(n, f))
    try:
        step_fn()
        torch.cuda.synchronize()
    finally:
        for n, f in orig.items():
            setattr(ops, n, f)
    tot_ms = sum(a.elapsed_time(b) for a, b, *_ in rec)
    if os.environ.get('SM3_GEMM_TABLE'):
        with open(os.environ['SM3_GEMM_TABLE'], 'w') as f:
            for a, b, fl, _, name, shape in rec:
                ms = a.elapsed_time(b)
                f.write(f'{name} shape={shape} ms={ms:.4f} tflops={fl / ms * 1e-9:.1f}\n')
    tot_flops = sum(r[2] for r in rec)
    peak = peaks.get('bf16_tflops_sustained') or peaks.get('bf16_tflops') or 1590.0
    ach = tot_flops / (tot_ms * 1e-3) / 1e12 if tot_ms > 0 else 0.0
    return {'bound': 'tensor', 'kernel': 'tcgen05 kernels (gemm_bf16x3 + fused FFN), all launches of one fwd+bwd micro-batch',
            'achieved': ach, 'peak': peak, 'unit': 'TFLOP/s', 'frac': ach / peak, 'traffic': None, 'launches': len(rec),
            'algorithmic_bytes_per_launch': sum(r[3] for r in rec) / max(len(rec), 1),
            'tensor_ms_per_micro_batch': tot_ms, 'algorithmic_tflop_per_micro_batch': tot_flops / 1e12,
            'note': 'algorithmic fp32 FLOPs; each costs 3 bf16 tensor-core MACs (hi*hi+hi*lo+lo*hi), so the tensor pipe '
                    'runs at 3x this rate (ceiling of frac = 1/3); peak = measured cuBLAS bf16 (sustained) from MEASURED_PEAKS.json'
                    if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else 'peak = fallback 1.59 PFLOP/s'}


def moe_roofline(net, x, peaks):
    """BASELINE metric (2): achieved HBM GB/s of the MoE dispatch(+expert) path of one forward, against the measured copy
    bandwidth.  Timed with CUDA events around (a) the whole 3-kernel-sequence the north star names -- dispatch gather
    (fused into the operand pack), grouped expert GEMM pair, combine scatter -- and (b) the dispatch kernels alone
    (gather-pack + combine).  Algorithmic bytes: SURVEY.md 8(d): (5k+1)*T*C*4 + E*(8C^2+5C)*4 + 8kT for the sequence,
    (3k+1)*T*C*4 for gather + scatter."""
    from sm3det_b200 import ops
    seq, disp = [], []
    o_assign, o_combine, o_pack = ops.moe_assign, ops.moe_combine, ops.pack_act
    state = {}

    def ev():
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def assign(top_idx, plan, *, T, E, k):
        r = o_assign(top_idx, plan, T=T, E=E, k=k)
        state.update(t0=ev(), T=T, E=E, k=k)
        return r

    def pack(x_, **kw):
        if kw.get('row_index') is not None and 't0' in state:
            a = ev(); r = o_pack(x_, **kw); b = ev()
            state['gather'] = (a, b)
            return r
        return o_pack(x_, **kw)

    def combine(o, slot_of, top_idx, gate, gamma, resid, row_scale, *, T, Cc, k, want_y=False):
        a = ev()
        r = o_combine(o, slot_of, top_idx, gate, gamma, resid, row_scale, T=T, Cc=Cc, k=k, want_y=want_y)
        b = ev()
        E = state['E']
        seq.append((state.pop('t0'), b, ((5 * k + 1) * T * Cc * 4 + E * (8 * Cc * Cc + 5 * Cc) * 4 + 8 * k * T), 16.0 * k * T * Cc * Cc))
        g = state.pop('gather', None)
        if g is not None:
            disp.append((g[0], g[1], a, b, (3 * k + 1) * T * Cc * 4))
        return r

    ops.moe_assign, ops.moe_combine, ops.pack_act = assign, combine, pack
    try:
        with torch.no_grad():
            net(x)
        torch.cuda.synchronize()
    finally:
        ops.moe_assign, ops.moe_combine, ops.pack_act = o_assign, o_combine, o_pack
    peak = peaks.get('hbm_gbs') or 6550.0
    ms = sum(a.elapsed_time(b) for a, b, *_ in seq)
    by = sum(r[2] for r in seq)
    fl = sum(r[3] for r in seq)
    dms = sum(a.elapsed_time(b) + c.elapsed_time(d) for a, b, c, d, _ in disp)
    dby = sum(r[4] for r in disp)
    out = {'bound': 'hbm', 'kernel': 'MoE dispatch+expert path (gather-pack -> grouped GEMM x2 -> combine), all MoE layers of one forward',
           'layers': len(seq), 'achieved': by / (ms * 1e-3) / 1e9 if ms else 0.0, 'peak': peak, 'unit': 'GB/s',
           'ms': ms, 'algorithmic_bytes': by, 'expert_tflops': fl / (ms * 1e-3) / 1e12 if ms else 0.0,
           'note': 'the expert GEMM pair is tensor-bound (16kTC^2 FLOP on 3-pass split-bf16), so the sequence cannot reach the '
                   'HBM roofline (the north-star 60 % target is NOT met on the sequence as written); dispatch_only isolates '
                   'the HBM-bound gather + scatter kernels'}
    out['frac'] = out['achieved'] / peak
    if dms:
        out['dispatch_only'] = {'achieved': dby / (dms * 1e-3) / 1e9, 'frac': dby / (dms * 1e-3) / 1e9 / peak, 'ms': dms,
                                'algorithmic_bytes': dby}
    return out


DUMP_FEATURE_SAMPLES = 1 << 20     # elements kept of each feature level (float32: 4 MB)
DUMP_GRAD_SAMPLES = 1 << 23        # elements kept of all parameter gradients together (32 MB)


def dump_outputs(path, kept):
    """--dump-outputs: the last step's results as .npy files, 48 MB and a few kB at most.  Tensors above their budget are
    reduced to a fixed-seed sample of elements (same shapes -> same positions), plus the float64 L2 norm of every full tensor:
      features_<i>   level i of the backbone output over the per-GPU batch (micro-batches concatenated), float32
      feature_l2     L2 norm of each full level, float64
      gate_loss      load-balance loss of each micro-batch, float32
      step_loss      the value the step returns (sum of the levels' means + gate loss, over the micro-batches), float32
      grads          samples of every parameter gradient, in named_parameters() order, concatenated, float32
      grad_l2        L2 norm of each full parameter gradient, float64"""
    import numpy as np
    os.makedirs(path, exist_ok=True)

    def sample(t, n, seed):
        t = t.detach().reshape(-1)
        if t.numel() > n:
            idx = torch.randint(0, t.numel(), (n,), generator=torch.Generator().manual_seed(seed)).sort().values
            t = t[idx.to(t.device)]
        return t.float().cpu().numpy()

    def l2(ts):
        return np.array([torch.linalg.vector_norm(t.detach(), dtype=torch.float64).item() for t in ts])

    levels = [torch.cat(per_micro) for per_micro in zip(*kept['outs'])]
    grads = [g for g in kept['grads'] if g is not None]
    per_grad = max(1, DUMP_GRAD_SAMPLES // len(grads))
    files = {f'features_{i}': sample(f, DUMP_FEATURE_SAMPLES, i) for i, f in enumerate(levels)}
    files.update(feature_l2=l2(levels), gate_loss=torch.stack(kept['gate_loss']).float().cpu().numpy(),
                 step_loss=kept['loss'].float().cpu().numpy(),
                 grads=np.concatenate([sample(g, per_grad, 1000 + j) for j, g in enumerate(grads)]), grad_l2=l2(grads))
    for name, a in files.items():
        np.save(os.path.join(path, name + '.npy'), a)


def build_model(args, world, ep, ddp=True):
    import torch.distributed as dist
    from sm3det_b200.synth import make_state_dict
    c = CONFIGS[args.config]
    if c['family'] == 'convnext':
        from sm3det_b200 import ConvNeXt_moe_MultiInput
        net = ConvNeXt_moe_MultiInput(**c['kw'])
    else:
        from sm3det_b200 import LSKNet_moe_MultiInput
        net = LSKNet_moe_MultiInput(**c['kw'])
    # seeded "trained-like" weights keyed by state_dict name (the product leg never touches oracle/)
    sd = make_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0, True)
    net.load_state_dict(sd, strict=True)
    del sd
    net = net.cuda().train()
    model = net
    if ep:
        from sm3det_b200.expert_parallel import ddp_ignored_parameters, enable_expert_parallel
        enable_expert_parallel(net, dist.new_group(list(range(world))))
        # expert parameters never enter a gradient bucket: each rank keeps the gradients of the experts it owns
        torch.nn.parallel.DistributedDataParallel._set_params_and_buffers_to_ignore_for_model(net, ddp_ignored_parameters(net))
    if world > 1 and ddp:
        local = int(os.environ.get('LOCAL_RANK', '0'))
        model = torch.nn.parallel.DistributedDataParallel(net, device_ids=[local], broadcast_buffers=False,
                                                          gradient_as_bucket_view=True)
    return net, model


def run_ours(args):
    global T0
    T0 = time.time()
    import torch.distributed as dist
    from sm3det_b200 import _lib
    from sm3det_b200.graphed import GraphedStep, allreduce_gradients
    from sm3det_b200.synth import make_images

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    # the gating noise and LSKNet's dropout seeds come from torch's default generators; unseeded, CUDA's starts from a
    # different seed in every process, so repeated runs would not compute the same step
    torch.manual_seed(rank)
    if world > 1:
        dist.init_process_group('nccl')
    lib = _lib.load()
    assert lib.sm3_device_supported() == 1, 'bench.py needs an sm_100 (B200) device'
    c, B, MB, scaling, ep = resolve(args, world)
    # gradient sync: DDP's bucketed all-reduce hooks (eager launches), or ONE flat all-reduce at the end of the step, which
    # is capturable in the CUDA graph together with the whole forward+backward (sm3det_b200/graphed.py)
    want_graph = args.cuda_graph == 'on' or (args.cuda_graph == 'auto' and not args.amp and not ep)
    flat_sync = world > 1 and (args.grad_sync == 'flat' or (args.grad_sync == 'auto' and want_graph))
    net, model = build_model(args, world, ep, ddp=not flat_sync)
    named_params = list(net.named_parameters())
    ignored = set()
    if ep:
        from sm3det_b200.expert_parallel import ddp_ignored_parameters
        ignored = set(ddp_ignored_parameters(net))
    S = args.size
    n_micro = B // MB
    host_x = make_images(B, S, S, seed=1234 + rank).pin_memory()
    dev_x = host_x.cuda()
    # --dump-outputs: references to what the latest step returned.  Under graph capture these are the graph's static
    # tensors, which every replay rewrites.
    kept = {}

    def micro_step(x):
        with torch.autocast('cuda', dtype=torch.bfloat16, enabled=args.amp):
            outs, loss = model(x)
        if args.dump_outputs:
            kept['outs'].append([o.detach() for o in outs])
            kept['gate_loss'].append(loss.detach())
        tot = (sum(o.float().mean() for o in outs) + loss) / n_micro
        tot.backward()
        return tot.detach()

    def step(x):
        """one optimizer step's worth of work: fwd+bwd over the per-GPU batch, gradients accumulated over the micro-batches,
        all-reduced (DDP) once, during the last micro-batch's backward"""
        if args.dump_outputs:
            kept.update(outs=[], gate_loss=[])
        tot = None
        for i in range(n_micro):
            sync_ctx = model.no_sync() if (world > 1 and not flat_sync and (i + 1 < n_micro or args.no_grad_sync)) else contextlib.nullcontext()
            with sync_ctx:
                t = micro_step(x[i * MB:(i + 1) * MB])
            tot = t if tot is None else tot + t
        if flat_sync and not args.no_grad_sync:
            allreduce_gradients(None, named=named_params, skip=ignored)
        if args.dump_outputs:
            kept.update(loss=tot, grads=[p.grad for _, p in named_params])
        return tot

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step(dev_x)
        model.zero_grad(set_to_none=True)
    # ---- CUDA graph of the whole step (all micro-batches, forward + backward): one replay per step instead of thousands of
    # launches.  On several GPUs the gradient all-reduce is the flat one above and is part of the graph.
    graphed, graph_note = None, 'off'
    if want_graph:
        try:
            graphed = GraphedStep(step, [dev_x], net.parameters(), warmup=2,
                                  invalidate=[m._packs for m in net.modules() if hasattr(m, '_packs')],
                                  capture_error_mode='global' if world == 1 else 'thread_local')
            graph_note = f'whole step captured: {graphed.launches_per_replay} C-ABI launches per replay'
        except Exception as e:       # noqa: BLE001 -- report and fall back to eager launches
            if args.cuda_graph == 'on':
                raise
            graphed, graph_note = None, f'capture failed, eager launches: {type(e).__name__}: {e}'[:300]
            torch.cuda.synchronize()
            model.zero_grad(set_to_none=True)

    def run(x):
        if graphed is not None:
            return graphed(x)            # gradients are replaced by the replay (no zero_grad between steps)
        t = step(x)
        return t

    def after_step():
        if graphed is None:
            model.zero_grad(set_to_none=True)

    sampler = ClockSampler(local)
    # ---- device-resident timing -------------------------------------------------------------------
    _lib.LAUNCHES = 0
    sync()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        run(dev_x)
        after_step()
    e1.record()
    sync()
    launches = _lib.LAUNCHES + (graphed.launches_per_replay * args.steps if graphed is not None else 0)
    ms = e0.elapsed_time(e1) / args.steps
    # ---- end to end: pinned host input -> device, result scalar back to the host, every step --------
    # Every step's batch is copied from pinned host memory inside the timed region; the copy of step i+1 is issued on
    # a side stream before step i computes (double-buffered), the way a data loader feeds the reference's train loop.
    h2d = host_x.numel() * 4
    copy_stream = torch.cuda.Stream()
    bufs = [torch.empty_like(dev_x), torch.empty_like(dev_x)]
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    freed = [torch.cuda.Event(), torch.cuda.Event()]
    main = torch.cuda.current_stream()

    def prefetch(slot, first_use):
        with torch.cuda.stream(copy_stream):
            if not first_use:
                copy_stream.wait_event(freed[slot])        # the step that last read this buffer has finished
            bufs[slot].copy_(host_x, non_blocking=True)
            ready[slot].record(copy_stream)

    sync()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    acc = 0.0
    # the 4-byte result of every step is copied to pinned host memory asynchronously and read one step later, so the
    # host keeps enqueueing step i+1 while step i runs (a blocking .item() per step drains the launch queue: ~1.5 ms/step)
    host_res = [torch.empty((), dtype=torch.float32).pin_memory() for _ in range(2)]
    res_ready = [torch.cuda.Event(), torch.cuda.Event()]
    prefetch(0, True)
    for i in range(args.steps):
        cur = i & 1
        if i + 1 < args.steps:
            prefetch(cur ^ 1, i == 0)
        main.wait_event(ready[cur])
        tot = run(bufs[cur])
        freed[cur].record(main)
        host_res[cur].copy_(tot, non_blocking=True)      # D2H read of the step result (4 bytes)
        res_ready[cur].record(main)
        if i > 0:
            res_ready[cur ^ 1].synchronize()
            acc += float(host_res[cur ^ 1])
        after_step()
    res_ready[(args.steps - 1) & 1].synchronize()
    acc += float(host_res[(args.steps - 1) & 1])
    e3.record()
    sync()
    clocks = sampler.stop() if rank == 0 else None
    if ep:
        net._ep_ctx.check()                      # expert-side capacity was never exceeded (reads a device flag; off the clock)
    ms_e2e = e2.elapsed_time(e3) / args.steps
    grad_l1 = None
    if graphed is not None:       # the last replay's gradients are still in .grad: a checksum to cross-check micro-batch splits
        grad_l1 = float(sum(p.grad.double().abs().sum() for p in net.parameters() if p.grad is not None))
    peak_mem = torch.cuda.max_memory_allocated() / 2 ** 30
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, kept)     # before the instrumented passes below accumulate into .grad
    kept.clear()
    t = torch.tensor([ms, ms_e2e], device='cuda', dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = t.tolist()
    del bufs
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:
            pass
        roof = roof_moe = None
        # the instrumented extra passes are rank-0 only: expert parallelism and SyncBN (LSKNet) need every rank in each layer
        if not ep and not args.amp and (world == 1 or c['family'] == 'convnext'):
            xm = dev_x[:MB]

            def one():
                outs, loss = net(xm)
                (sum(o.mean() for o in outs) + loss).backward()
            if graphed is not None:
                # torch.cuda.graph() empties the caching allocator before capture: re-grow the eager pool off the clock so
                # that no cudaMalloc lands between the CUDA events of the instrumented pass
                one()
                net.zero_grad(set_to_none=True)
                torch.cuda.synchronize()
            roof = gemm_roofline(one, peaks)
            net.zero_grad(set_to_none=True)
            try:   # measured DRAM traffic of the tensor-core launches of one micro-batch (ncu dram__bytes_read+write, profiles/)
                tr = json.load(open(os.path.join(ROOT, 'profiles', 'r02_gemm_traffic.json')))
                roof['traffic'] = tr['bytes_per_launch']
                roof['traffic_note'] = tr['note']
            except Exception:
                pass
            if c['family'] == 'convnext':
                roof_moe = moe_roofline(net, xm, peaks)
        line = {'metric': METRIC, 'value': B * world / (ms * 1e-3), 'unit': 'img/s', 'n_gpus': world, 'steps': args.steps,
                'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': scaling, 'vs_baseline': None,
                'dtype': ('bf16 GEMM operands (single pass), fp32 accumulate and fp32 elsewhere -- optional AMP recipe, not the headline'
                          if args.amp else 'f32 (bf16 hi+lo split operands on tcgen05, fp32 accumulate; SIMT fp32 elsewhere)'),
                'data': 'synthetic', 'config': workload_config(args, world), 'clocks': clocks,
                'e2e': {'value': B * world / (ms_e2e * 1e-3), 'unit': 'img/s', 'h2d_bytes_per_step': h2d,
                        'd2h_bytes_per_step': 4, 'ms_per_step': ms_e2e},
                'gpu_launches': launches, 'peak_mem_gb': peak_mem, 'roofline': roof, 'roofline_moe': roof_moe}
        line['cuda_graph'] = graph_note
        line['grad_l1'] = grad_l1
        line['step_scalar'] = acc / max(args.steps, 1)      # mean of the per-step result read back in the e2e loop (sanity cross-check)
        if world > 1:
            line['grad_sync'] = 'one flat all-reduce at the end of the step' if flat_sync else 'DDP bucket hooks'
        if args.no_grad_sync:
            line['diagnostic'] = 'gradients NOT all-reduced (--no-grad-sync): not a valid training step, comm-cost isolation only'
        if os.environ.get('SM3_RESERVE_SMS'):
            line['config']['reserved_sms_for_nccl'] = int(os.environ['SM3_RESERVE_SMS'])
        if world == 1 and not args.no_gpu_eager:
            graphed = None                       # release the step graph's memory pool before the comparator allocates
            del model, net
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            try:
                line['gpu_eager'] = time_gpu_eager(args, min(MB, 8))
                line['gpu_eager']['ours_over_eager_fp32'] = line['value'] / line['gpu_eager']['fp32']
                line['gpu_eager']['ours_over_eager_tf32'] = line['value'] / line['gpu_eager']['tf32']
            except Exception as e:                      # a comparator failure must not lose the bench line
                line['gpu_eager'] = {'error': f'{type(e).__name__}: {e}'[:300]}
        if world == 1 and not args.no_cpu_baseline:
            ips, dt, threads, fwd_ips = time_cpu_reference(args, args.cpu_images, 1, 0)
            line['cpu_baseline'] = cpu_baseline_entry(args, ips, dt, threads, fwd_ips)
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear-down order matters when the step was graph-captured: NCCL keeps a communicator alive (and ncclCommDestroy
        # blocks) while a CUDA graph that captured collectives on it exists -- measured as a hang at exit after the JSON line
        # on 4 GPUs (profiles/r02_multi_gpu.txt).  Destroy the graph first, then leave without tearing the group down.
        def stamp(msg):
            print(f'[bench rank {rank}] {msg} t={time.time() - T0:.1f}s', file=sys.stderr, flush=True)
        stamp('result printed' if rank == 0 else 'timed region done')
        graphed = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        stamp('graph released')
        dist.barrier()
        stamp('barrier passed, exiting')
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
