#!/usr/bin/env python
"""Benchmark of the OctFusion denoising U-Net hot path (BASELINE.json: "U-Net denoise steps/sec
(depth-6, B=32) at 1/2/4/8 B200").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload unet|cond|vae]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A step = one pass of the hot path over one batch: the stage-2 ("hr") U-Net forward on B=32 synthetic depth-6
ShapeNet-shaped octrees (uncond yaml: model_channels [64,128], channel_mult [[1,2,4],[1,2,4]], num_res_blocks
[[1,1,1],[1,1,0]], 4 heads, LR middle block included, 8 latent channels) + the eps-DDIM update, exactly what reference
sample_loop does per time step (models/octfusion_model_union.py:313-350).  bf16 activations, fp32 accumulation /
statistics / latent.  Random-init weights (no checkpoint is reachable), synthetic octrees (no dataset is reachable).

One JSON line on stdout (rank 0):
  value        whole-job steps/s, inputs resident in HBM (CUDA-graph replay, CUDA events, max over ranks)
  e2e          the same metric through the public sampler API (HRStepper) with the latent arriving from pinned host
               memory and the result returning to the host every step (copies inside the timed region)
  roofline     the tcgen05 tap-gather GEMM aggregated over all its launches of one step (per-launch CUDA events)
  cpu_baseline the reference's own modules (build container) or the oracle port (GPU box: the reference tree does
               not travel) on the host cores: bounded sample, thread-count sweep, best reported
  library_baseline  the reference op sequence (oracle port = the same ATen calls) on the SAME B200 in fp32 through
               ATen / cuBLAS -- the "same-box library" bar of BASELINE.md section 3
Multi-GPU (BASELINE.json configs[2]): the B=32 shapes are SHARDED over the ranks (32/N per GPU, `scaling: strong`);
no collective in the step loop (SURVEY.md 8e); one ragged all-gather of the final latents after the timed region.
`--weak` keeps 32 shapes per GPU instead.  --workload cond = the class-conditional config (configs[4]);
--workload vae = GraphVAE encode + decode at depth 8 (configs[3], HBM-bound regime).
Weights, shapes and noise are seeded, so the same arguments give the same inputs on every run; --dump-outputs DIR
writes what the last timed step returned (unet / cond: latent.npy = the updated latent, eps.npy = the U-Net output,
all ranks' rows; vae: the decoder's logits and regression values per depth) as float32, at most 64 MB in all.
"""
from __future__ import annotations
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNCOND = dict(
    image_size=[16, 64], input_depth=[4, 6], unet_type=['lr', 'hr'], df_type=['x0', 'eps'], full_depth=4,
    input_channels=[8, 3], out_channels=[8, 3], model_channels=[64, 128], num_res_blocks=[[1, 1, 1], [1, 1, 0]],
    attention_resolutions=[2, 4], channel_mult=[[1, 2, 4], [1, 2, 4]], num_heads=4, use_checkpoint=False, dims=3)
COND = dict(UNCOND, num_res_blocks=[[1, 1, 1], [2, 2, 0]], attention_resolutions=[2, 4, 8],
            channel_mult=[[1, 2, 4, 8], [1, 2, 4]], num_classes=5)
METRICS = {'unet': 'unet_denoise_steps_per_sec_depth6_B32', 'cond': 'unet_cond_denoise_steps_per_sec_depth6_B32',
           'vae': 'graphvae_encode_decode_per_sec_depth8'}
UNIT = 'steps/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default='unet', choices=['unet', 'cond', 'vae'])
    ap.add_argument('--batch', type=int, default=32, help='shapes per step of the WHOLE job (sharded over the GPUs)')
    ap.add_argument('--weak', action='store_true', help='weak scaling: --batch shapes on EVERY GPU')
    ap.add_argument('--code-channels', type=int, default=8,
                    help='feature channels of the latent (BASELINE.json: 8; the shipped snet yaml uses 3)')
    ap.add_argument('--dtype', default='bf16', choices=['bf16', 'fp32'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-library-baseline', action='store_true')
    ap.add_argument('--no-roofline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step returned as DIR/<name>.npy (float32), to compare two builds')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be >= 1 and --warmup >= 0')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes what --impl ours computed')
    return args


def config_for(args):
    cfg = dict(COND if args.workload == 'cond' else UNCOND)
    if args.workload != 'cond':
        cfg['input_channels'] = [8, args.code_channels]
        cfg['out_channels'] = [8, args.code_channels]
    return cfg


def latent_channels(args):
    return 3 if args.workload == 'cond' else args.code_channels


def randomise_(net, seed):
    """default init + N(0, 1/fan_in) for the reference's zero-initialised tensors (modules.py:719,525,499;
    graph_unet_hr.py:209), which would otherwise make the whole net output 0 and let kernels skip nothing
    but also prove nothing."""
    g = torch.Generator().manual_seed(seed)
    for _, p in net.named_parameters():
        if float(p.detach().abs().max()) == 0.0 and p.dim() > 1:
            fan = p[..., 0].numel() if p.dim() == 2 and p.shape[0] > p.shape[1] else p[0].numel()
            p.data.copy_(torch.randn(p.shape, generator=g) / max(fan, 1) ** 0.5)
    return net


DUMP_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: each tensor as path/<name>.npy in float32.  Above DUMP_BYTES in all, every array keeps the same
    share of its rows, chosen by a fixed seed (sorted), so that two builds with the same arguments stay comparable."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    total = sum(t.numel() * 4 for t in arrays.values())
    for name, t in arrays.items():
        t = t.detach().float()
        if total > DUMP_BYTES:
            keep = max(1, int(t.shape[0] * DUMP_BYTES // total))
            rows = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            t = t[rows.to(t.device)]
        np.save(os.path.join(path, name + '.npy'), t.cpu().numpy())


def _synth():
    """octfusion_b200/synth.py loaded by path: the input generator is pure torch-CPU and must be usable by the
    baseline legs WITHOUT importing the product package (which would map liboctfusion_b200.so into the process)."""
    if 'of_synth' not in sys.modules:
        spec = importlib.util.spec_from_file_location('of_synth', os.path.join(ROOT, 'octfusion_b200', 'synth.py'))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        sys.modules['of_synth'] = m
    return sys.modules['of_synth']


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return None
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for t, line in self.samples:
            f = [s.strip() for s in line.split(',')]
            if len(f) < 6 or not (t0 - 0.05 <= t <= t1 + 0.15):
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[2:6]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return None
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': mx, 'reasons': sorted(reasons), 'samples': len(sm)}


# --------------------------------------------------------------------------------------------------
# baseline legs (the ONLY place bench.py touches oracle/): the reference path on the host cores, and the same ATen
# op sequence on the GPU.  Nothing here imports octfusion_b200.
# --------------------------------------------------------------------------------------------------
def _state_shapes(cfg, name):
    with open(os.path.join(ROOT, 'tests', 'golden', 'state_shapes.json')) as f:
        table = json.load(f)
    key = name if name in table else 'uncond'
    shapes = {k: tuple(v) for k, v in table[key].items()}
    cc = cfg['input_channels'][1]
    if key == 'uncond' and cc != 3:                       # only the first / last GraphConv depend on the latent width
        nt = cfg['input_depth'][1] - 1
        shapes['unet_hr.input_blocks.0.weights'] = (7 * (cc + nt), shapes['unet_hr.input_blocks.0.weights'][1])
        shapes['unet_hr.out.weights'] = (shapes['unet_hr.out.weights'][0], cc)
    return shapes


def _move_graph(dg, dev):
    """the oracle's DualGraph with its index tensors on `dev` (library leg)"""
    import copy
    g2 = copy.copy(dg)
    g2.graph = [{k: v.to(dev) for k, v in g.items()} for g in dg.graph]
    g2._bid = {k: v.to(dev) for k, v in dg._bid.items()}
    g2._child = {k: v.to(dev) for k, v in dg._child.items()}
    oc = copy.copy(dg.octree)
    cache = {}

    def xyzb(depth, nempty=False, _o=dg.octree):
        if (depth, nempty) not in cache:
            cache[(depth, nempty)] = tuple(t.to(dev) for t in _o.xyzb(depth, nempty))
        return cache[(depth, nempty)]
    oc.xyzb = xyzb
    g2.octree = oc
    return g2


def baseline_step_fn(cfg, cfg_name, batch, device, use_reference):
    """returns (step callable, kind): one U-Net forward + eps-DDIM update on `batch` of the synthetic shapes in fp32,
    by the unmodified reference modules (when /root/reference is present and device is the CPU) or the oracle port."""
    from oracle import restate as R
    from oracle.octree_util import octree_from_splits
    from oracle import ref_import
    l4, l5 = _synth().synth_splits(batch, 0)
    octree = octree_from_splits(l4, l5, batch)
    cc = cfg['input_channels'][1]
    g = torch.Generator().manual_seed(1)
    ts = torch.full((batch,), 1.5)
    label = (torch.arange(batch) % cfg['num_classes']) if cfg.get('num_classes') else None
    ls, lsn = torch.tensor(1.5), torch.tensor(1.9)
    if use_reference and ref_import.available() and device == 'cpu':
        ref = ref_import.load()
        net = ref.union.UNet3DModel('hr', **cfg).eval()
        sd = R.seeded_state_dict({k: tuple(v.shape) for k, v in net.state_dict().items()}, 0)
        net.load_state_dict(sd)
        doc = ref.dual_octree.DualOctree(octree)
        doc.post_processing_for_docnn()
        x = torch.randn(doc.total_num, cc, generator=g)

        def step():
            eps = net(unet_type='hr', x=x, doctree=doc, timesteps=ts, unet_lr=net.unet_lr, label=label)
            return R.ddim_eps_update(x, eps, ls, lsn)
        return step, 'reference'
    sd = R.seeded_state_dict(_state_shapes(cfg, cfg_name), 0)
    dg = R.DualGraph(octree)
    lr_cfg, hr_cfg = R.split_cfg(cfg)
    x = torch.randn(dg.total_num, cc, generator=g)
    if device != 'cpu':
        dev = torch.device(device)
        sd = {k: v.to(dev) for k, v in sd.items()}
        dg = _move_graph(dg, dev)
        x, ts, ls, lsn = x.to(dev), ts.to(dev), ls.to(dev), lsn.to(dev)
        label = label.to(dev) if label is not None else None

        def step():
            with torch.device(dev):
                eps = R.hr_forward(x, dg, ts, sd, hr_cfg, lr_cfg, label=label)
                return R.ddim_eps_update(x, eps, ls, lsn)
        return step, 'port'

    def step():
        eps = R.hr_forward(x, dg, ts, sd, hr_cfg, lr_cfg, label=label)
        return R.ddim_eps_update(x, eps, ls, lsn)
    return step, 'port'


def cpu_baseline(cfg, cfg_name, batch_full, sample_batch=4, timed=2, budget_s=150.0):
    """reference path on the host cores: B = sample_batch of the shapes, thread sweep {8,16,32,64,cores} with one
    timed forward each (after one warm-up at the first setting), then `timed` forwards at the best setting."""
    cores = os.cpu_count() or 1
    step, kind = baseline_step_fn(cfg, cfg_name, sample_batch, 'cpu', True)
    sweep = sorted({t for t in (8, 16, 32, 64, cores) if t <= cores}) or [cores]
    t_start = time.perf_counter()
    results = {}
    with torch.no_grad():
        torch.set_num_threads(sweep[0])
        step()                                                  # warm-up (allocator, lazy inits)
        for th in sweep:
            torch.set_num_threads(th)
            t0 = time.perf_counter(); step(); results[th] = time.perf_counter() - t0
            # stop when the budget is spent or more threads have clearly stopped helping (oversubscribed hosts get
            # 10x slower at the full core count: 100 s for one B=4 step on the 128-core GPU box)
            if (time.perf_counter() - t_start > budget_s and len(results) >= 2) or results[th] > 1.25 * min(results.values()):
                break
        best = min(results, key=results.get)
        torch.set_num_threads(best)
        ts = []
        for _ in range(timed):
            t0 = time.perf_counter(); step(); ts.append(time.perf_counter() - t0)
    dt = min(min(ts), results[best])
    value = 1.0 / (dt * batch_full / sample_batch)
    return {'value': value, 'unit': UNIT, 'cores': best, 'kind': kind, 'host_cores': cores,
            'sweep_s_per_step': {str(k): round(v, 3) for k, v in results.items()},
            'sample': '%s U-Net step (fp32, torch CPU) on B=%d of the %d shapes; thread sweep %s, best %d threads: %.2f s '
                      'per B=%d step (best of %d timed), scaled linearly to B=%d'
                      % ('unmodified reference modules under the ocnn shim' if kind == 'reference' else 'oracle port of the reference',
                         sample_batch, batch_full, sweep, best, dt, sample_batch, timed + 1, batch_full)}


def library_baseline(cfg, cfg_name, batch, dev, timed=3):
    """the reference op sequence through ATen / cuBLAS on this GPU (fp32, as the reference computes)"""
    step, kind = baseline_step_fn(cfg, cfg_name, batch, str(dev), False)
    with torch.no_grad():
        step(); step()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(timed):
            step()
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / timed
    return {'value': 1000.0 / ms, 'unit': UNIT, 'ms_per_step': ms, 'batch': batch, 'dtype': 'fp32',
            'kind': 'oracle port of the reference op sequence (index / index_add_ / mm / conv3d / softmax) with '
                    'device=cuda: ATen + cuBLAS + cuDNN, torch %s, %d timed steps' % (torch.__version__, timed)}


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path, timed on the host cores."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    if args.workload == 'vae':
        print(json.dumps({'impl': 'reference', 'unavailable': 'the vae workload has no CPU arm (unet / cond only)'}))
        return
    cfg = config_for(args)
    name = 'cond' if args.workload == 'cond' else ('uncond8' if args.code_channels == 8 else 'uncond')
    base = cpu_baseline(cfg, name, args.batch, 4, max(2, min(args.steps, 3)))
    line = {'impl': 'reference', 'metric': METRICS[args.workload], 'value': base['value'], 'unit': UNIT,
            'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1000.0 / base['value'],
            'higher_is_better': True, 'scaling': 'weak' if args.weak else 'strong', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': workload_config(args, None, args.batch), 'cpu_baseline': base,
            'e2e': {'value': base['value'], 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


def workload_config(args, nodes, per_gpu):
    what = {'unet': 'uncond snet yaml, %d latent channels' % args.code_channels,
            'cond': 'class-conditional snet yaml (num_classes 5, LR channel_mult [1,2,4,8], attention at 8^3/4^3/2^3, '
                    'HR num_res_blocks [2,2,0])',
            'vae': 'GraphVAE (vae_snet_train.yaml) encoder + decoder at depth 8'}[args.workload]
    c = {'workload': 'OctFusion stage-2 (hr) denoising U-Net step: %s, depth-6 synthetic ShapeNet-shaped octrees, '
                     'full_depth 4, LR middle block + attention included, eps-DDIM update' % what
         if args.workload != 'vae' else what,
         'global_batch': args.batch * (args.gpus if args.weak else 1), 'batch_per_gpu': per_gpu,
         'code_channels': latent_channels(args),
         'parallelism': 'dp%d (batch shard, no collective in the step loop)' % args.gpus,
         'l2': 'no flush: one step streams several GB of activations (>> 126 MB L2)'}
    if nodes:
        c['nodes_per_gpu'] = nodes
    return c


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    # exactly ONE line may reach stdout (the JSON): NCCL / torch banners are sent to stderr for the whole run
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py --impl ours needs a CUDA device: octfusion_b200 has no CPU path')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    torch.manual_seed(0)            # the nets' default init draws from the global generator: same weights every run
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    if args.workload == 'vae':
        return run_vae(args, dev, rank, world, real_stdout)
    from octfusion_b200 import graph_unet_union, octree_from_splits, DualOctree, ops, _lib, shard
    from octfusion_b200.synth import synth_splits, slice_splits
    from octfusion_b200.sampler import HRStepper, sampling_log_snr

    cfg = config_for(args)
    act = torch.bfloat16 if args.dtype == 'bf16' else torch.float32
    net = randomise_(graph_unet_union.UNet3DModel('hr', **cfg), 0).to(dev).eval()
    # the job's shapes: every rank generates the same `batch` shapes; strong scaling keeps a contiguous block of them
    # (BASELINE.json configs[2]: "batch 32 sharded over 8xB200"), weak scaling keeps them all
    l4, l5 = synth_splits(args.batch, seed=0)
    if args.weak or world == 1:
        per_gpu = args.batch
    else:
        lo, hi = shard.shard_range(args.batch, rank, world)
        per_gpu = hi - lo
        l4, l5 = slice_splits(l4, l5, lo, hi)
    if per_gpu == 0:
        raise SystemExit('bench.py: more ranks than shapes')
    doc = DualOctree(octree_from_splits(l4, l5, per_gpu, device=dev))
    nodes = {d: doc.plan[d].rows for d in range(4, 7)}
    # stage-1 -> stage-2 handoff (SURVEY.md 8f-2), once per batch of shapes, outside the timed step: device split tensor
    # -> octree -> dual graph with its tap tables and statistics plans (second build: kernels and allocator are warm)
    build_ms = None
    if rank == 0:
        try:
            from octfusion_b200 import split2octree_small, octree2split_small
            import time as _time
            split = octree2split_small(doc.octree, 4)
            torch.cuda.synchronize(); t_a = _time.perf_counter()
            oc2 = split2octree_small(split, 6, 4)
            torch.cuda.synchronize(); t_b = _time.perf_counter()
            doc2 = DualOctree(oc2)
            torch.cuda.synchronize(); t_c = _time.perf_counter()
            build_ms = {'split2octree_small': (t_b - t_a) * 1e3, 'dual_octree': (t_c - t_b) * 1e3,
                        'shapes': per_gpu, 'depth6_rows': int(doc2.plan[6].rows),
                        'note': 'once per batch of shapes (not per step): wall clock incl. its two host synchronisations'}
            del doc2, oc2, split
        except Exception as e:  # noqa: BLE001
            build_ms = {'error': repr(e)}
    n6, cc = doc.total_num, latent_channels(args)
    label = (torch.arange(per_gpu, device=dev) % cfg['num_classes']) if cfg.get('num_classes') else None
    total_steps = args.warmup + args.steps
    ls = sampling_log_snr(max(total_steps, 50))
    g = torch.Generator(device=dev).manual_seed(rank)
    noise = torch.randn((n6, cc), generator=g, device=dev)

    st = HRStepper(net.unet_hr, net.unet_lr, doc, act, label, use_cuda_graph=True)
    st.set_latent(noise)
    for i in range(args.warmup):                                   # includes the eager pass + graph capture
        st.step(ls[i], ls[i + 1])
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
        time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.time()
    e0.record()
    for i in range(args.warmup, total_steps):
        st.step(ls[i], ls[i + 1])
    e1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    clk = clocks.stop(t0, t1) if rank == 0 else None
    # strong scaling: one step of the job = all ranks' shards done; weak: every rank does a full batch per step
    value = (world if args.weak else 1) * args.steps / (ms_total / 1000.0)
    kernels_per_step = int(st.kernels_per_step)
    if args.dump_outputs:            # the last timed step's latent and U-Net output, all ranks' rows (the e2e legs reuse st)
        out = {name: torch.cat(shard.all_gather_latents(t)) for name, t in (('latent', st.x), ('eps', st.eps))}
        if rank == 0:
            dump_outputs(args.dump_outputs, out)
        del out

    # ---- e2e: public sampler API (HRStepper, CUDA-graph step), host buffers, H2D + D2H inside the timed region ----
    x_host = torch.randn((n6, cc)).pin_memory()
    y_host = torch.empty((n6, cc)).pin_memory()

    def e2e_serial(i):                                            # everything on one stream: copy, step, copy
        st.set_latent(x_host.to(dev, non_blocking=True))          # H2D of this step's latent (+ bf16 copy kernel)
        st.step(ls[i], ls[i + 1])
        y_host.copy_(st.x, non_blocking=True)                     # D2H of the step's result

    def e2e_piped(i):                                             # the public host-latent call: copies overlap the neighbours' compute
        st.step_host(x_host, ls[i], ls[i + 1], y_host)

    def run_e2e(fn, k):
        for i in range(2):
            fn(i)
        st.sync_host()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0.record()
        for i in range(k):
            fn(i)
        st.sync_host()                                            # the timed region ends when the last result is on the host
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return (world if args.weak else 1) * k / (float(ms.item()) / 1000.0)
    e2e_serial_v = run_e2e(e2e_serial, args.steps)
    e2e_v = run_e2e(e2e_piped, args.steps)
    e2e = {'value': e2e_v, 'unit': UNIT,
           'h2d_bytes_per_step': n6 * cc * 4 + 8, 'd2h_bytes_per_step': n6 * cc * 4,
           'steps': args.steps, 'serial_value': e2e_serial_v,
           'path': 'sampler.HRStepper.step_host(pinned host latent, ..., pinned host result), per rank: H2D + [CUDA-graph replay of '
                   'U-Net forward + DDIM update] + D2H every step; double-buffered, the copies of step i run on copy streams '
                   'beside the compute of steps i-1 / i+1 (independent latents).  serial_value = the same with copy, step, '
                   'copy on one stream'}

    # ---- roofline of the dominant kernel (per-launch CUDA events, eager pass) -----------------------
    roofline, per_layer = None, None
    if rank == 0 and not args.no_roofline and act == torch.bfloat16:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:  # noqa: BLE001
            pass
        # burst figure unless the timed region is long enough (>= 2 s) for the power cap to set the clocks
        long_run = ms_total >= 2000.0
        key = 'bf16_tflops_sustained' if long_run else 'bf16_tflops'
        peak_tf = float(peaks.get(key, 1400.0 if long_run else 1590.0))
        peak_src = ('MEASURED_PEAKS.json %s (of measured)' % key) if peaks else \
            ('%.0f TF/s (of fallback)' % peak_tf)
        agg = {}
        reps = 3
        for rep in range(reps + 1):
            sink = []
            ops.set_profile(sink)
            st.use_cuda_graph = False
            st.step(ls[0], ls[1])
            ops.set_profile(None)
            torch.cuda.synchronize()
            if rep == 0:
                continue
            for r in sink:
                if r['kind'] != 'tc':
                    continue
                key = (r['M'], r['K'], r['N'], r['taps'])
                a = agg.setdefault(key, {'ms': 0.0, 'flops': 0.0, 'bytes': 0.0, 'launches': 0})
                a['ms'] += r['start'].elapsed_time(r['end']); a['flops'] += r['flops']; a['bytes'] += r['bytes']
                a['launches'] += 1
        st.use_cuda_graph = True
        tot_ms = sum(a['ms'] for a in agg.values()); tot_fl = sum(a['flops'] for a in agg.values())
        tot_by = sum(a['bytes'] for a in agg.values())
        if tot_ms > 0:
            ach = tot_fl / (tot_ms * 1e-3) / 1e12
            traffic, traffic_src = None, None
            for cand in ('tc_traffic_r02.json', 'tc_traffic_r01.json'):   # DRAM bytes of the same launches (ncu capture)
                try:
                    tj = json.load(open(os.path.join(ROOT, 'profiles', cand)))
                    traffic = tj['dram_bytes_per_step'] / tj['launches_per_step']
                    traffic_src = 'profiles/' + cand
                    break
                except Exception:  # noqa: BLE001
                    pass
            nl = sum(a['launches'] for a in agg.values()) / reps
            roofline = {'kernel': 'gather_gemm_tc_kernel (all launches of one step)', 'bound': 'tensor',
                        'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf, 'traffic': traffic,
                        'traffic_unit': 'DRAM bytes per launch (ncu dram__bytes_read+write, mean over the step; %s)' % traffic_src,
                        'launches_per_step': nl, 'algorithmic_bytes_per_launch': tot_by / reps / max(nl, 1),
                        'peak_source': peak_src, 'frac_of_sustained': ach / float(peaks.get('bf16_tflops_sustained', 1400.0)),
                        'ms_per_step_in_kernel': tot_ms / reps,
                        'algorithmic_gflop_per_step': tot_fl / reps / 1e9, 'algorithmic_gb_per_step': tot_by / reps / 1e9}
            per_layer = []
            for (m, k, n, taps), a in sorted(agg.items(), key=lambda kv: -kv[1]['ms']):
                per_layer.append({'M': m, 'K': k, 'N': n, 'taps': taps, 'launches_per_step': a['launches'] // reps,
                                  'us': 1000.0 * a['ms'] / a['launches'],
                                  'tflops': a['flops'] / (a['ms'] * 1e-3) / 1e12,
                                  'frac': a['flops'] / (a['ms'] * 1e-3) / 1e12 / peak_tf,
                                  'gbps_algorithmic': a['bytes'] / (a['ms'] * 1e-3) / 1e9})

    # ---- the one collective of the path: ragged all-gather of the final latents ---------------------
    gathered = shard.all_gather_latents(st.x)
    if rank != 0:
        if world > 1:
            dist.barrier(); dist.destroy_process_group()
        return
    # ---- baselines (rank 0, N = 1): free this arm's GPU memory first --------------------------------
    cfg_name = 'cond' if args.workload == 'cond' else ('uncond8' if args.code_channels == 8 else 'uncond')
    cpu, library = None, None
    if world == 1:
        del st
        torch.cuda.empty_cache()
        if not args.no_library_baseline:
            try:
                library = library_baseline(cfg, cfg_name, per_gpu, dev)
            except Exception as e:  # noqa: BLE001
                library = {'value': None, 'unit': UNIT, 'kind': 'failed: %r' % (e,)}
            torch.cuda.empty_cache()
        if not args.no_cpu_baseline:
            try:
                cpu = cpu_baseline(cfg, cfg_name, args.batch, 4, 2)
            except Exception as e:  # noqa: BLE001
                cpu = {'value': None, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': 'port', 'sample': 'failed: %r' % (e,)}
    line = {'metric': METRICS[args.workload], 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms_total / args.steps, 'higher_is_better': True,
            'scaling': 'weak' if args.weak else 'strong', 'vs_baseline': None,
            'dtype': args.dtype, 'data': 'synthetic', 'config': workload_config(args, nodes, per_gpu), 'clocks': clk,
            'e2e': e2e, 'gpu_launches': kernels_per_step * args.steps, 'kernels_per_step': kernels_per_step,
            'graph_build_ms': build_ms,
            'roofline': roofline, 'cpu_baseline': cpu, 'library_baseline': library,
            'gathered_latent_rows': [int(t.shape[0]) for t in gathered]}
    if per_layer:
        line['roofline_per_layer'] = per_layer[:40]
    os.write(real_stdout, (json.dumps(line) + '\n').encode())
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def run_vae(args, dev, rank, world, real_stdout):
    """BASELINE.json configs[3]: GraphVAE encoder (`extract_code` network on caller-provided input features) + decoder
    (`decode_code`, octree kept) on depth-8 octrees -- the sparse-conv-only, HBM-bound regime (C = 24..32)."""
    import torch.distributed as dist
    from octfusion_b200 import _lib
    from tools.prof_vae import build_case
    case = build_case(args.batch if args.weak or world == 1 else max(1, args.batch // world), dev,
                      torch.bfloat16 if args.dtype == 'bf16' else torch.float32)
    for _ in range(args.warmup):
        case['step']()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    c0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = case['step']()
    e1.record()
    torch.cuda.synchronize()
    launches = _lib.launch_count() - c0
    if args.dump_outputs and rank == 0:       # every rank decodes the same shapes
        dump_outputs(args.dump_outputs, {'%s_d%d' % (k, d): t for k in ('logits', 'reg_voxs') for d, t in out[k].items()})
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank == 0:
        per = float(ms.item()) / args.steps
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
        except Exception:  # noqa: BLE001
            pass
        hbm = float(peaks.get('hbm_gbs', 6650.0))
        gbs = case['algorithmic_bytes'] / (per * 1e-3) / 1e9
        line = {'metric': METRICS['vae'], 'value': (world if args.weak else 1) * 1000.0 / per, 'unit': 'passes/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': per, 'higher_is_better': True,
                'scaling': 'weak' if args.weak else 'strong', 'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
                'config': dict(workload_config(args, case['nodes'], case['batch']), note=case['note']),
                'gpu_launches': int(launches), 'kernels_per_step': int(launches // max(args.steps, 1)),
                'roofline': {'kernel': 'whole encode+decode pass', 'bound': 'hbm', 'achieved': gbs, 'peak': hbm,
                             'unit': 'GB/s', 'frac': gbs / hbm, 'traffic': None,
                             'algorithmic_bytes_per_pass': case['algorithmic_bytes'],
                             'peak_source': 'MEASURED_PEAKS.json hbm_gbs (of measured)' if peaks else '6650 GB/s (of fallback)'}}
        os.write(real_stdout, (json.dumps(line) + '\n').encode())
    if world > 1:
        dist.barrier(); dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
