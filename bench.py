#!/usr/bin/env python
"""Benchmark of the pix2pix3D render hot path (BASELINE.json metric: rendered images/s at 512^2 output, 128^2
neural-rendering resolution, 48+48 samples per ray).

    python bench.py --gpus 1 --steps K --warmup W                     # this repository (CUDA, libp3d.so)
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...          # the UNMODIFIED reference (baseline/_ref) on the host cores, same config
    python bench.py --impl reference-cuda ...     # the UNMODIFIED reference on the GPU through its own JIT-built plugins
    python bench.py --workload {seg2cat_smoke,seg2cat_512,seg2face_512,edge2car_128}     # BASELINE.json configs 1-4
    python bench.py ... --dump-outputs DIR        # also write the outputs of the last timed step as DIR/<name>.npy

A step is one `G.synthesis(ws, c, noise_mode='const', neural_rendering_resolution=128)` of
TriPlaneSemanticEntangleGenerator on a batch of 4 (BASELINE configs[1]); weights are seeded random, inputs synthetic.
`value` is timed with CUDA events with inputs resident in HBM; `e2e` repeats the measurement through the same public
call with pinned-host inputs copied in and the two 512^2 outputs copied back inside the timed region.
One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = 'seg2cat_512'           # BASELINE.json configs[1], the configuration the metric is quoted on
METRIC = 'rendered images/sec (512^2, 128^2 NeRF res, 96 samples/ray)'
sys.path.insert(0, os.path.join(ROOT, 'baseline'))


def metric_name(workload):
    from pix2pix3d_b200 import configs
    w = configs.WORKLOADS[workload]
    rk = configs.generator_kwargs(workload)['rendering_kwargs']
    if workload == 'seg2cat_512':
        return METRIC
    return (f"rendered images/sec ({w['img_resolution']}^2, {w['nrr']}^2 NeRF res, "
            f"{rk['depth_resolution'] + rk['depth_resolution_importance']} samples/ray)")


def workload_config(workload, B, world, extra=None):
    """`config` object shared by every arm so that the driver can tell the arms ran the same thing."""
    from pix2pix3d_b200 import configs
    w = configs.WORKLOADS[workload]
    rk = configs.generator_kwargs(workload)['rendering_kwargs']
    cfg = {'workload': workload, 'batch_per_gpu': B, 'global_batch': B * world, 'neural_rendering_resolution': w['nrr'],
           'samples_per_ray': rk['depth_resolution'] + rk['depth_resolution_importance'], 'img_resolution': w['img_resolution'],
           'parallelism': f'dp{world} (batch-sharded, no collective)'}
    cfg.update(extra or {})
    return cfg


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi sampling of SM clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    FIELDS = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
              'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
              'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(',')]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2])); pw.append(float(parts[3]))
            except ValueError:
                continue
            for n, v in zip(names, parts[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(n)
        if not sm:
            return None
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': max(mx), 'power_w_max': max(pw), 'samples': len(sm),
                'reasons': sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        try:
            with open(path) as fh:
                return json.load(fh), 'measured (MEASURED_PEAKS.json)'
        except (OSError, ValueError):
            pass
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}, 'fallback (B200_PROFILING.md)'


# ---------------------------------------------------------------------------------------------
def cpu_port_step(state, n_images=1):
    """One pass of the oracle (CPU port of the reference path, oracle/p3d_oracle) over `n_images` config-2 images."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import p3d_oracle as O
    sd, ws, c, cfg, jitter, u = state
    for i in range(n_images):
        O.networks.generator_synthesis(ws[i:i + 1], c[i:i + 1], sd, cfg, jitter[i:i + 1], u[i * cfg['nrr'] ** 2:(i + 1) * cfg['nrr'] ** 2])


def cpu_port_state(batch):
    import numpy as np
    import torch
    from pix2pix3d_b200 import configs
    torch.set_num_threads(os.cpu_count())
    G = configs.build_generator(WORKLOAD, seed=0, device='cpu', with_mapping=False)
    sd = {k: v.numpy() for k, v in G.state_dict().items()}
    rk = dict(G.rendering_kwargs)
    w = configs.WORKLOADS[WORKLOAD]
    nrr = w['nrr']
    ws = configs.synthetic_ws(batch, G.backbone.num_ws, 1).numpy()
    c = configs.camera_labels(batch, 2).numpy()
    rng = np.random.RandomState(1234)
    jitter = rng.rand(batch, nrr * nrr, rk['depth_resolution'], 1).astype(np.float32)
    u = rng.rand(batch * nrr * nrr, rk['depth_resolution_importance']).astype(np.float32)
    cfg = dict(nrr=nrr, rendering_kwargs=rk, semantic_channels=w['semantic_channels'], sr_kind='SuperresolutionHybrid8XDC',
               sr_kind_semantic='SuperresolutionHybrid8XDC_semantic', sr_fp16=True)
    return sd, ws, c, cfg, jitter, u


def run_reference_arm(args):
    """`--impl reference`: the UNMODIFIED reference (baseline/_ref, byte-identical copy of /root/reference) on the host
    cores -- `G.synthesis` of its own TriPlaneSemanticEntangleGenerator, custom ops on their `_ref` branch, fp32, all host
    threads, same workload / batch / seeds / inputs as the product arm. Steps are capped by a time budget so the run ends
    within a few minutes. Falls back to the oracle port only if baseline/_ref is absent."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import ref_harness as rh
    from pix2pix3d_b200 import configs
    w = configs.WORKLOADS[args.workload]
    B = args.batch or w['batch']
    cores = os.cpu_count()
    if rh.available():
        r = rh.time_synthesis(args.workload, 'cpu', B, args.steps, args.warmup, budget_s=float(os.environ.get('P3D_REF_BUDGET_S', '200')),
                              log=lambda m: print(m, file=sys.stderr))
        value, ms_step, steps, warm = r['images_per_s'], r['ms_per_step'], r['steps'], r['warmup']
        kind = 'reference'
        sample = (f"{steps} steps x G.synthesis of {B} images ({args.workload}) through the unmodified reference on CPU "
                  f"(_ref ops, fp32; {r['threads']} torch threads = the fastest of a sweep up to the {rh.usable_cores()} usable of "
                  f"{cores} host cores), after {warm} warm-up steps")
        cores = r['threads']
        stages = r['stage_ms_per_step']
    else:
        state = cpu_port_state(1)
        cpu_port_step(state)
        t0 = time.perf_counter()
        cpu_port_step(state)
        dt = time.perf_counter() - t0
        value, ms_step, steps, warm, kind, stages = 1.0 / dt, 1000 * dt, 1, 1, 'port', None
        sample = '1 image through oracle/p3d_oracle (baseline/_ref missing)'
    line = {
        'impl': 'reference', 'metric': metric_name(args.workload), 'value': value, 'unit': 'images/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': warm, 'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args.workload, B, 1, {'device': 'cpu', 'launch': 'reference G.synthesis, eager'}),
        'cpu_baseline': {'value': value, 'unit': 'images/s', 'cores': cores, 'kind': kind, 'sample': sample,
                         'stage_ms_per_step': stages},
        'e2e': {'value': value, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


def run_reference_cuda_arm(args):
    """`--impl reference-cuda`: the reference's stock CUDA path on one B200 (BASELINE.md plan item 2, the ">= 5x" baseline):
    its plugins are JIT-built on first use by its own torch_utils/custom_ops.py:61, convolutions are cuDNN, SR runs in fp16 as
    shipped; a second measurement uses force_fp32. CUDA events, inputs resident."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    import ref_harness as rh
    from pix2pix3d_b200 import configs
    if not rh.available():
        print(json.dumps({'impl': 'reference-cuda', 'unavailable': 'baseline/_ref missing (run baseline/vendor_reference.py)'}), flush=True)
        return
    if not torch.cuda.is_available():
        print(json.dumps({'impl': 'reference-cuda', 'unavailable': 'no CUDA device'}), flush=True)
        return
    w = configs.WORKLOADS[args.workload]
    B = args.batch or w['batch']
    sampler = ClockSampler(0)
    sampler.start()
    r = rh.time_synthesis(args.workload, 'cuda', B, args.steps, max(args.warmup, 5), log=lambda m: print(m, file=sys.stderr))
    clocks = sampler.stop()
    r32 = rh.time_synthesis(args.workload, 'cuda', B, args.steps, max(args.warmup, 5), force_fp32=True, stage_split=False)
    line = {
        'impl': 'reference-cuda', 'metric': metric_name(args.workload), 'value': r['images_per_s'], 'unit': 'images/s',
        'n_gpus': 1, 'steps': r['steps'], 'warmup': r['warmup'], 'ms_per_step': r['ms_per_step'], 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': r['dtype'], 'data': 'synthetic',
        'config': workload_config(args.workload, B, 1, {'device': 'cuda', 'launch': 'reference G.synthesis, eager, stock plugins + cuDNN'}),
        'stage_ms_per_step': r['stage_ms_per_step'], 'first_step_s': r['first_step_s'],
        'force_fp32': {'value': r32['images_per_s'], 'ms_per_step': r32['ms_per_step']},
        'rays_per_s': r['images_per_s'] * w['nrr'] ** 2, 'clocks': clocks,
    }
    print(json.dumps(line), flush=True)


def run_train_step_arm(args):
    """`--workload train_step`: BASELINE.json configs[4] -- one `train.py` iteration of the afhq_seg recipe at 4 images per GPU
    (G main [+ density reg every 4], D main [+ R1 every 16], D_semantic main [+ R1 every 16], one flat NCCL all-reduce per phase,
    Adam, G_ema), pix2pix3d_b200/train_step.py. `--impl ours`: the reference's loss class driving this package's modules and
    kernels through `install()`; `--impl reference-cuda`: the unmodified reference end to end. Weak scaling (4 images per GPU)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    import ref_harness as rh
    if args.impl == 'ours':
        import pix2pix3d_b200
        from pix2pix3d_b200 import _lib
        _lib.lib()
        pix2pix3d_b200.install(reference_root=rh.REF_ROOT)       # training.loss etc. come from the reference checkout
    else:
        rh.import_reference()
    from pix2pix3d_b200 import train_step as ts
    cfg = dict(ts.AFHQ_TRAIN)
    if args.batch:
        cfg['batch_gpu'] = args.batch
        cfg['mbstd_group'] = min(cfg['mbstd_group'], args.batch)
    st = ts.build(cfg, dev, rank=rank, num_gpus=world, seed=0)
    batch = ts.synthetic_batch(cfg, dev, 100 + rank)
    steps = args.steps
    warm = max(args.warmup, 3)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    launches0 = 0
    if args.impl == 'ours':
        from pix2pix3d_b200 import _lib
    for _ in range(warm):
        ts.run_iteration(st, batch)
    st.batch_idx = 0                                               # timed region starts on a regularisation iteration
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    if args.impl == 'ours':
        launches0 = _lib.launch_count
    timers = {}
    torch.cuda.reset_peak_memory_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        ts.run_iteration(st, batch, timers if rank == 0 else None)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        phases = {k: {'calls': len(v), 'ms_per_call': sum(a.elapsed_time(b) for a, b in v) / len(v)} for k, v in timers.items()}
        b = cfg['batch_gpu']
        value = world * b * steps / (ms / 1000.0)
        line = {
            'metric': 'train.py step images/sec (afhq_seg 512^2 / 128^2 rays: G fwd + dual discriminator + R1, 4 images per GPU)',
            'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': steps, 'warmup': warm, 'ms_per_step': ms / steps,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32 (G backbone, renderer) + f16 (super-resolution, top-4 D resolutions), as train.py', 'data': 'synthetic',
            'impl': args.impl,
            'config': {'workload': 'train_step', 'batch_per_gpu': b, 'global_batch': b * world, 'neural_rendering_resolution': cfg['nrr'],
                       'img_resolution': cfg['img_resolution'], 'parallelism': f'dp{world}: one flat fp32 all-reduce per phase (NCCL)',
                       'phases': 'Gmain Dmain D_semanticmain every iteration, Greg every 4, Dreg / D_semanticreg every 16',
                       'l2_policy': 'no flush: activations of a step exceed L2 by orders of magnitude'},
            'phase_ms': phases, 'allreduce_bytes_per_phase': st.flat_bytes,
            'peak_mem_gb': torch.cuda.max_memory_allocated() / 2 ** 30, 'clocks': clocks,
            'gpu_launches': ((_lib.launch_count - launches0) / steps) if args.impl == 'ours' else None,
            'params_digest': ts.grads_digest(st),
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def stock_cuda_leg(args, B, timeout_s=900):
    """Run `--impl reference-cuda` in a child process (its module names `training.*` stay out of this process and a JIT
    failure cannot take the product measurement down) and return its JSON line."""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference-cuda', '--workload', args.workload, '--steps', str(args.steps),
           '--warmup', str(args.warmup), '--batch', str(B)]
    env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')}
    try:
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout_s, env=env)
    except subprocess.TimeoutExpired:
        return {'unavailable': f'reference-cuda child exceeded {timeout_s} s'}
    for ln in reversed(r.stdout.strip().splitlines()):
        if ln.startswith('{'):
            try:
                return json.loads(ln)
            except ValueError:
                pass
    return {'unavailable': 'reference-cuda child printed no JSON line', 'rc': r.returncode, 'stderr_tail': r.stderr[-1500:]}


def render_traffic(workload, B):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the fused render kernel, from the committed ncu --set full
    summary (profiles/render_traffic.json, written by tools/ncu_traffic.py from the .ncu-rep)."""
    path = os.path.join(ROOT, 'profiles', 'render_traffic.json')
    try:
        with open(path) as fh:
            t = json.load(fh)
        for e in t['captures']:
            if e['workload'] == workload and e['batch'] == B:
                return e['dram_bytes_per_launch'], e.get('source')
    except (OSError, ValueError, KeyError):
        pass
    return None, None


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, outputs, limit=DUMP_LIMIT_BYTES):
    """Write each output as out_dir/<name>.npy in float32. Above `limit` bytes in all, every output is cut to a share of
    the limit proportional to its size: a sorted sample of its flattened elements drawn with a fixed seed, so two runs of
    the same workload keep the same elements."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.numpy().astype(np.float32) for k, v in outputs.items()}
    total = sum(a.size for a in arrays.values())
    budget = (limit - 4096 * len(arrays)) // 4          # 4 KiB per file covers the .npy header
    for k, a in arrays.items():
        if total > budget:
            keep = a.size * budget // total
            a = a.reshape(-1)[np.sort(np.random.RandomState(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, k + '.npy'), a)


# ---------------------------------------------------------------------------------------------
def main():
    global WORKLOAD
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None,
                    help='timed steps (default: 20; 16 for train_step, one full lazy-regularisation period)')
    ap.add_argument('--warmup', type=int, default=None, help='untimed steps before the timed ones (default: 5; 3 for train_step)')
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'reference-cuda'])
    ap.add_argument('--workload', default=WORKLOAD, choices=['seg2cat_smoke', 'seg2cat_512', 'seg2face_512', 'edge2car_128', 'train_step'],
                    help='BASELINE.json configs 1-4 (default: configs[1], the metric\'s configuration)')
    ap.add_argument('--no-stock-cuda', action='store_true', help='skip the reference stock-CUDA leg (child process, ~1-2 min incl. plugin JIT)')
    ap.add_argument('--batch', type=int, default=None, help='images per GPU per step (default: the workload batch, 4)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--force-fp32', action='store_true', help='run the SR stacks in fp32 (reference default is fp16)')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel from Python instead of replaying a CUDA graph')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the outputs of the last timed step as DIR/<name>.npy (float32); when they exceed 64 MB in all, '
                         'each is replaced by the same fixed-seed sample of its flattened elements')
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 16 if args.workload == 'train_step' else 20
    if args.warmup is None:
        args.warmup = 3 if args.workload == 'train_step' else 5
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.workload == 'train_step' or args.impl != 'ours'):
        ap.error('--dump-outputs applies to the G.synthesis benchmark of this repository (--impl ours, not train_step)')
    if args.workload == 'train_step':
        if args.impl == 'reference':
            raise SystemExit('--workload train_step has the arms `ours` and `reference-cuda` (a CPU train step takes minutes per image)')
        run_train_step_arm(args)
        return
    if args.impl == 'reference':
        run_reference_arm(args)
        return
    if args.impl == 'reference-cuda':
        run_reference_cuda_arm(args)
        return
    WORKLOAD = args.workload
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    from pix2pix3d_b200 import _lib, configs, native

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (there is no CPU fallback of the product path)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    _lib.lib()   # fail loudly if the native library is missing

    w = configs.WORKLOADS[WORKLOAD]
    B = args.batch or w['batch']
    nrr = w['nrr']
    G = configs.build_generator(WORKLOAD, seed=0, device=dev, with_mapping=False)
    rk = G.rendering_kwargs
    S = rk['depth_resolution'] + rk['depth_resolution_importance']
    # every rank renders its own batch (weak scaling, no collective on the render path)
    ws_host = configs.synthetic_ws(B, G.backbone.num_ws, 1 + rank).pin_memory()
    c_host = configs.camera_labels(B, 2 + rank, w['preset']).pin_memory()
    ws, c = ws_host.to(dev), c_host.to(dev)
    syn_kw = dict(noise_mode='const', neural_rendering_resolution=nrr)
    if args.force_fp32:
        syn_kw['force_fp32'] = True

    graphed = None
    if not args.no_graph:
        from pix2pix3d_b200.graphs import GraphedSynthesis
        graphed = GraphedSynthesis(G, ws, c, **syn_kw)      # public serving entry point: capture once, replay per step

    def step(ws_, c_):
        if graphed is not None:
            return graphed(ws_, c_)
        with torch.no_grad():
            return G.synthesis(ws_, c_, **syn_kw)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        out = step(ws, c)
    barrier()

    # ---- device-resident timing -------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    native.kernel_events = []
    launches0 = _lib.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        out = step(ws, c)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    # graph replay reuses its output tensors, so the last timed step's outputs are copied out before anything else runs
    dumped = {k: v.detach().float().cpu() for k, v in out.items()} if args.dump_outputs and rank == 0 else None
    launches = graphed.native_launches if graphed is not None else (_lib.launch_count - launches0) / args.steps
    kev = native.kernel_events
    native.kernel_events = None
    render_ms = [e[1].elapsed_time(e[2]) for e in kev if e[0] == 'render_fwd']
    conv_ev = [e for e in kev if e[0] == 'conv_gemm']
    if not render_ms:
        # graph replay hides individual launches: time the render kernel inside eager steps of the same workload
        native.kernel_events = []
        with torch.no_grad():
            for _ in range(max(3, args.steps)):
                G.synthesis(ws, c, **syn_kw)
        torch.cuda.synchronize()
        render_ms = [e[1].elapsed_time(e[2]) for e in native.kernel_events if e[0] == 'render_fwd'][1:]
        conv_ev = [e for e in native.kernel_events if e[0] == 'conv_gemm']
        native.kernel_events = None
    clocks = sampler.stop() if rank == 0 else None
    value = world * B * args.steps / (ms / 1000.0)

    # ---- end-to-end: pinned host inputs in, 512^2 outputs back, every step ---------------------
    img_host = torch.empty(B, 3, w['img_resolution'], w['img_resolution'], dtype=torch.float32).pin_memory()
    sem_host = torch.empty(B, w['semantic_channels'], w['img_resolution'], w['img_resolution'], dtype=torch.float32).pin_memory()
    ws_d, c_d = torch.empty_like(ws), torch.empty_like(c)

    # Serving-style pipeline: inputs go in on the compute stream; outputs are staged device-side (two buffers) and read
    # back on a copy stream, so the device->host copy of step i runs under the compute of step i+1. Every step still
    # copies its own inputs in and its own outputs out, and the timed region ends after the last read-back has landed.
    copy_stream = torch.cuda.Stream()
    stage = [(torch.empty(img_host.shape, device=dev), torch.empty(sem_host.shape, device=dev)) for _ in range(2)]
    staged_ev = [torch.cuda.Event() for _ in range(2)]      # outputs of a step are in stage[k]
    drained_ev = [torch.cuda.Event() for _ in range(2)]     # stage[k] has been read back
    for ev in drained_ev:
        ev.record()
    step_no = [0]

    def e2e_step():
        k = step_no[0] & 1
        step_no[0] += 1
        cur = torch.cuda.current_stream()
        ws_d.copy_(ws_host, non_blocking=True)
        c_d.copy_(c_host, non_blocking=True)
        o = step(ws_d, c_d)
        cur.wait_event(drained_ev[k])
        stage[k][0].copy_(o['image'], non_blocking=True)
        stage[k][1].copy_(o['semantic'], non_blocking=True)
        staged_ev[k].record(cur)
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(staged_ev[k])
            img_host.copy_(stage[k][0], non_blocking=True)
            sem_host.copy_(stage[k][1], non_blocking=True)
            drained_ev[k].record(copy_stream)

    def e2e_drain():
        torch.cuda.current_stream().wait_stream(copy_stream)

    for _ in range(3):
        e2e_step()
    e2e_drain()
    barrier()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e2e_drain()
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))
    e2e_value = world * B * args.steps / (ms_e2e / 1000.0)
    h2d = ws_host.numel() * 4 + c_host.numel() * 4
    d2h = img_host.numel() * 4 + sem_host.numel() * 4

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (fused render) ---------------------------------------
    peaks, peak_src = measured_peaks()
    alg_bytes = configs.render_algorithmic_bytes(B, nrr * nrr, S)
    roofline = None
    traffic, traffic_src = render_traffic(WORKLOAD, B)
    if render_ms:
        t_k = sum(render_ms) / len(render_ms) / 1000.0
        achieved = alg_bytes / t_k / 1e9
        roofline = {'kernel': 'render_fwd_tc_kernel' if native.render_impl in ('auto', 'tc') else 'render_fwd_kernel', 'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                    'frac': achieved / peaks['hbm_gbs'],
                    # dram__bytes_read + write per launch of this kernel at this workload, read from the committed ncu --set full
                    # summary (profiles/render_traffic.json); null when no capture of this workload/batch exists
                    'traffic': traffic, 'traffic_source': traffic_src, 'peak_source': peak_src,
                    'kernel_ms': t_k * 1000, 'algorithmic_bytes': alg_bytes, 'share_of_step': t_k * 1000 / (ms / args.steps),
                    'rays_per_s': B * nrr * nrr / t_k}

    # second bound: the tensor-core convolutions (62 launches per step), algorithmic FLOPs / summed launch time
    roofline_tensor = None
    if conv_ev:
        per_step = len(conv_ev) // max(1, len(render_ms) + 1)
        use = conv_ev[per_step:] if per_step and len(conv_ev) > per_step else conv_ev      # drop the first (cold) step
        t_c = sum(e[1].elapsed_time(e[2]) for e in use) / 1000.0
        fl_alg, fl_exec = sum(e[3] for e in use), sum(e[4] for e in use)
        n_steps = max(1, len(use) // max(1, per_step))
        roofline_tensor = {'kernel': 'conv_gemm_kernel', 'bound': 'tensor', 'achieved': fl_alg / t_c / 1e12, 'peak': peaks['bf16_tflops'],
                           'unit': 'TFLOP/s', 'frac': fl_alg / t_c / 1e12 / peaks['bf16_tflops'],
                           'executed_tflops': fl_exec / t_c / 1e12, 'launches_per_step': per_step,
                           'ms_per_step': t_c * 1000 / n_steps,
                           'note': 'fp32 backbone layers execute 3 fp16 passes per algorithmic FLOP (hi/lo split); '
                                   'event pairs around single launches in eager steps'}

    # ---- CPU baseline: the unmodified reference on the host cores, same batch, bounded sample ------
    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        import ref_harness as rh
        if rh.available():
            r = rh.time_synthesis(WORKLOAD, 'cpu', B, steps=2, warmup=2, budget_s=30)
            cpu_baseline = {'value': r['images_per_s'], 'unit': 'images/s', 'cores': r['threads'], 'kind': 'reference',
                            'sample': f"{r['steps']} steps x G.synthesis of {B} images through the unmodified reference on CPU "
                                      f"(baseline/_ref, _ref ops, fp32, {r['threads']} torch threads = fastest of a sweep, "
                                      f"{os.cpu_count()} host cores) after {r['warmup']} warm-up steps, "
                                      f"{r['ms_per_step'] / 1000:.1f} s per step",
                            'stage_ms_per_step': r['stage_ms_per_step']}
        else:
            state = cpu_port_state(1)
            t0 = time.perf_counter()
            cpu_port_step(state)
            dt = time.perf_counter() - t0
            cpu_baseline = {'value': 1.0 / dt, 'unit': 'images/s', 'cores': os.cpu_count(), 'kind': 'port',
                            'sample': f'1 image through oracle/p3d_oracle (baseline/_ref missing), {dt:.1f} s'}

    # ---- reference stock CUDA path on this GPU (child process) ---------------------------------------
    stock_cuda, vs_stock = None, None
    if world == 1 and not args.no_stock_cuda:
        torch.cuda.empty_cache()
        sc = stock_cuda_leg(args, B)
        stock_cuda = {k: sc.get(k) for k in ('value', 'unit', 'ms_per_step', 'steps', 'warmup', 'dtype', 'stage_ms_per_step',
                                             'force_fp32', 'first_step_s', 'unavailable', 'stderr_tail', 'clocks') if k in sc}
        if sc.get('value'):
            vs_stock = {'device_timed': value / sc['value'], 'e2e_over_stock_device_timed': e2e_value / sc['value'],
                        'vs_force_fp32': value / sc['force_fp32']['value'] if sc.get('force_fp32') else None}

    line = {
        'metric': metric_name(WORKLOAD), 'value': value, 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f32' if args.force_fp32 else 'f32 (backbone, renderer) + f16 (super-resolution, as the reference)',
        'data': 'synthetic',
        'config': workload_config(WORKLOAD, B, world, {
                   'launch': 'CUDA graph replay of G.synthesis (pix2pix3d_b200.graphs.GraphedSynthesis)' if graphed is not None else 'eager',
                   'l2_policy': 'no flush: per-step working set (planes 100 MB + SR activations > 2 GB) exceeds the 126 MB L2'}),
        'rays_per_s': world * B * nrr * nrr * args.steps / (ms / 1000.0),
        'gpu_launches': launches,
        'e2e': {'value': e2e_value, 'unit': 'images/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'ms_per_step': ms_e2e / args.steps,
                'pipeline': 'pinned-host ws/c in and image+semantic out every step; read-back of step i overlaps step i+1 '
                            '(two staging buffers, copy stream); timed region ends after the last read-back'},
        'clocks': clocks, 'roofline': roofline, 'roofline_tensor': roofline_tensor, 'cpu_baseline': cpu_baseline,
        'stock_cuda': stock_cuda, 'vs_stock_cuda': vs_stock,
    }
    print(json.dumps(line), flush=True)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
