#!/usr/bin/env python
"""bench.py — RVT hot-path throughput on B200 (contract: task statement §④ + base contract).

Workload (BASELINE.json configs[1]): RVT-Base 1Mpx, event tensor 8 x 20 x 360 x 640 (uint8, zero
padding to the model's 384x640 folded into the stem), seq_len 21, states carried, inference.
One *step* = one 21-timestep sequence for the local batch (8 samples/GPU) = 168 frames/GPU.
Batch-sharded over N GPUs with no data-path collective (weak scaling).

  value : frames/s, whole job, inputs resident in HBM (774 MB of uint8 sequences > L2)
  e2e   : frames/s through rvt_b200.RNNDetector.forward with HOST (pinned) uint8 inputs copied
          H2D every timestep and the stage-4 feature map read back D2H every timestep
  --impl reference : the reference's CPU path (oracle port, torch fp32, all host threads) on a
          bounded sample of the same workload.
  --dump-outputs DIR : also write what the last timed step computed (dump_outputs); the inputs and
          weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'RVT-B 1Mpx seq_len=21 backbone frames/sec'
B_PER_GPU, SEQ_LEN, IN_C, IN_H, IN_W, PAD_H, PAD_W = 8, 21, 20, 360, 640, 384, 640
# per timestep: S1 s2d+conv, 4 fused attn/mlp, lstm; S2 conv, 4 fused, lstm; S3/S4 conv+ln, 2 x (ln,qkv,core,proj,ln,fc1,fc2), lstm
LAUNCHES_PER_TIMESTEP = (2 + 4 + 1) + (1 + 4 + 1) + 2 * (2 + 2 * 7 + 1)
TRAIN_METRIC = 'RVT-B 1Mpx seq_len=21 backbone training frames/sec'
LOSS_SCALE = 65536.0      # static stand-in for the harness' GradScaler (precision 16, config/general.yaml:6)
GFLOP_PER_FRAME = 20.62                                 # BASELINE.md §3 (algorithmic, MAC = 2 FLOP)


_REAL_STDOUT = None


def protect_stdout():
    """stdout must carry exactly ONE JSON line, but NCCL prints its version banner to fd 1 (at NCCL_DEBUG=VERSION, the
    image default, and at WARN too) and other libraries may chat as well: keep a private copy of the real stdout for the
    result line and point fd 1 at stderr for everything else."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')


def emit(obj):
    data = (json.dumps(obj) + '\n').encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def rvt_b_spec():
    """oracle-side description of RVT-Base 1Mpx (reference arms only)."""
    from oracle import backbone_oracle as bo
    return bo.BackboneSpec(embed_dim=64, dim_head=32, partition_size=(6, 10))


def rvt_b_cfg():
    """RVT-Base 1Mpx `mdl_config` (config/model/maxvit_yolox/default.yaml + base.yaml, partition size as
    config/modifier.py:36-41 derives it for 384x640) as a plain dict — what the reference hands to the backbone."""
    return dict(
        name='MaxViTRNN', compile=dict(enable=False, args=dict(mode='reduce-overhead')),
        input_channels=IN_C, enable_masking=False, partition_split_32=2, embed_dim=64, dim_multiplier=[1, 2, 4, 8],
        num_blocks=[1, 1, 1, 1], T_max_chrono_init=[4, 8, 16, 32], stem=dict(patch_size=4),
        stage=dict(downsample=dict(type='patch', overlap=True, norm_affine=True),
                   attention=dict(use_torch_mha=False, partition_size=(6, 10), dim_head=32, attention_bias=True,
                                  mlp_activation='gelu', mlp_gated=False, mlp_bias=True, mlp_ratio=4, drop_mlp=0, drop_path=0,
                                  ls_init_value=1e-5, norm_eps=1e-5),
                   lstm=dict(dws_conv=False, dws_conv_only_hidden=True, dws_conv_kernel_size=3, drop_cell_update=0)))


def build_model(seed=0):
    """rvt_b200.RNNDetector with random-init weights of the RVT-Base architecture: N(0, 1/fan_in) weights, N(0, 0.1) biases,
    LayerNorm weights and LayerScale gammas ~ U(0.5, 1.5) (so no branch is numerically dead, SURVEY.md D10).  Nothing of
    oracle/ is touched on the product arm."""
    import rvt_b200
    model = rvt_b200.RNNDetector(rvt_b_cfg())
    g = torch.Generator(device='cpu').manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith('gamma') or ('norm' in name and name.endswith('weight')):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
            elif name.endswith('bias'):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
            elif name.endswith('mask_token'):
                p.copy_(torch.randn(p.shape, generator=g) * 0.5)
            else:
                fan_in = p[0].numel()
                p.copy_(torch.randn(p.shape, generator=g) / fan_in ** 0.5)
    return model


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [v.strip() for v in ln.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


def cpu_reference_fps(n_timesteps, batch, threads):
    """The reference's CPU implementation of the path (oracle port: torch fp32 eager ops, the same
    ATen kernels the reference dispatches to), states carried; returns frames/s."""
    from oracle import backbone_oracle as bo
    spec = rvt_b_spec()
    torch.set_num_threads(threads)
    params = bo.synth_params(spec, 0)
    xs = [torch.nn.functional.pad(bo.synth_events_tensor(i, batch, IN_C, IN_H, IN_W).float(),
                                  (0, PAD_W - IN_W, 0, PAD_H - IN_H)) for i in range(n_timesteps + 1)]
    st = None
    with torch.inference_mode():
        _, st = bo.backbone_forward(xs[0], st, params, spec)      # warm-up timestep
        t0 = time.perf_counter()
        for i in range(n_timesteps):
            _, st = bo.backbone_forward(xs[1 + i], st, params, spec)
        dt = time.perf_counter() - t0
    return batch * n_timesteps / dt


def best_cpu_threads():
    """torch's intra-op pool at os.cpu_count() threads is far slower than a moderate pool on big hosts
    (measured 0.56 frames/s at 128 threads vs ~10 at 8-32): calibrate on one bs=1 timestep."""
    cores = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64, cores) if c <= cores})
    best, best_fps = cands[0], 0.0
    for c in cands:
        fps = cpu_reference_fps(1, 1, c)
        if fps > best_fps:
            best, best_fps = c, fps
    return best


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port) on the host cores.  A step is one full 21-timestep, bs-8
    sequence (the product arm's own config) whenever K + W of them fit in ~4 minutes of CPU time; otherwise a bounded sample
    (fewer timesteps per step) and the line says so."""
    if rank != 0:
        return
    cores = best_cpu_threads()
    t0 = time.perf_counter()
    fps1 = cpu_reference_fps(2, B_PER_GPU, cores)                       # probe (also the warm-up)
    est_seq_s = B_PER_GPU * SEQ_LEN / fps1
    budget_s = 240.0 - (time.perf_counter() - t0)
    steps = max(1, args.steps)
    n_ts = SEQ_LEN
    if steps * est_seq_s > budget_s:
        n_ts = max(2, min(SEQ_LEN, int(SEQ_LEN * budget_s / (steps * est_seq_s))))
    vals = [cpu_reference_fps(n_ts, B_PER_GPU, cores) for _ in range(steps)]
    v = sum(vals) / len(vals)
    full = n_ts == SEQ_LEN
    sample = ((f'full sequences: {SEQ_LEN} timesteps x batch {B_PER_GPU} per step' if full else
               f'{n_ts} of the {SEQ_LEN} timesteps x batch {B_PER_GPU} per step (bounded to ~4 min of CPU time)') +
              f', states carried, fp32; {cores} torch threads (best of a sweep up to os.cpu_count()={os.cpu_count()})')
    emit({
        'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': 1, 'ms_per_step': 1e3 * B_PER_GPU * n_ts / v,     # what was actually timed per step
        'timed_timesteps_per_step': n_ts, 'same_config': full,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'RVT-Base 1Mpx 8x20x360x640 uint8 (model res 384x640) seq_len=21 bs=8/GPU '
                               'inference, states carried', 'frames_per_step': B_PER_GPU * SEQ_LEN, 'device': 'CPU'},
        'cpu_baseline': {'value': v, 'unit': 'frames/s', 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': v, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    })


def make_uint8_sequence(seed, length, batch):
    g = torch.Generator(device='cpu').manual_seed(seed)
    shape = (length, batch, IN_C, IN_H, IN_W)
    seq = torch.randint(1, 11, shape, generator=g, dtype=torch.uint8)            # counts 1..10 ...
    seq.mul_(torch.randint(0, 10, shape, generator=g, dtype=torch.uint8) == 0)   # ... on ~10 % of the bins
    return seq


def run_reference_gpu(args, rank, world, local_rank):
    """Informational arm (the denominator of north_star's '>= 10x PyTorch-eager on one B200'): the reference's
    op-by-op PyTorch path (oracle port = the same ATen/cuDNN/cuBLAS calls) on the GPU under fp16 autocast and
    inference_mode, same workload, inputs resident.  Not the driver's reference arm (that is --impl reference, CPU)."""
    if rank != 0:
        return
    from oracle import backbone_oracle as bo
    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    spec = rvt_b_spec()
    params = {k: v.to(dev) for k, v in bo.synth_params(spec, 0).items()}
    if args.mode == 'train':
        # the same training step as run_train (fwd 21 timesteps + loss + bwd + unscale + fused Adam), PyTorch eager + autograd
        B = args.train_batch
        plist = [v.requires_grad_(True) for v in params.values()]
        opt = torch.optim.Adam(plist, lr=2e-4, fused=True)
        seq = make_uint8_sequence(4321, SEQ_LEN, B).to(dev)

        def tstep():
            opt.zero_grad(set_to_none=True)
            st, out = None, None
            with torch.autocast('cuda', dtype=torch.float16):
                for t in range(SEQ_LEN):
                    x = torch.nn.functional.pad(seq[t].float(), (0, PAD_W - IN_W, 0, PAD_H - IN_H))
                    out, st = bo.backbone_forward(x, st, params, spec)
            loss = sum((out[s].float() ** 2).mean() for s in (1, 2, 3, 4)) * LOSS_SCALE
            loss.backward()
            torch._foreach_mul_([p.grad for p in plist], 1.0 / LOSS_SCALE)
            opt.step()

        for _ in range(max(args.warmup, 3)):
            tstep()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            tstep()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1)
        emit({
            'impl': 'reference-gpu', 'metric': TRAIN_METRIC, 'value': B * SEQ_LEN * args.steps / (ms * 1e-3), 'unit': 'frames/s',
            'n_gpus': 1, 'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps,
            'higher_is_better': True, 'dtype': 'f16 autocast', 'data': 'synthetic',
            'config': {'workload': f'RVT-Base 1Mpx bs={B} TBPTT seq_len=21 training step, PyTorch eager + autograd on the GPU '
                                   '(oracle port of the reference op sequence), fp16 autocast'}})
        return
    seq = make_uint8_sequence(1234, SEQ_LEN, B_PER_GPU).to(dev)

    def step():
        st = None
        for t in range(SEQ_LEN):
            x = torch.nn.functional.pad(seq[t].float(), (0, PAD_W - IN_W, 0, PAD_H - IN_H))   # modules/detection.py:133-134
            _, st = bo.backbone_forward(x, st, params, spec)
        return st

    with torch.inference_mode(), torch.autocast('cuda', dtype=torch.float16):
        for _ in range(max(args.warmup, 3)):
            step()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            step()
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1)
    v = B_PER_GPU * SEQ_LEN * args.steps / (ms * 1e-3)
    emit({
        'impl': 'reference-gpu', 'metric': METRIC, 'value': v, 'unit': 'frames/s', 'n_gpus': 1, 'steps': args.steps,
        'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f16 autocast', 'data': 'synthetic',
        'config': {'workload': 'RVT-Base 1Mpx 360x640 (padded 384x640) seq_len=21 bs=8 inference, PyTorch eager on the GPU '
                               '(oracle port of the reference op sequence), fp16 autocast, inputs resident'}})




def train_leg(args, rank, world, local_rank, steps, warmup):
    """BASELINE configs[2]: RVT-Base 1Mpx training step, TBPTT over seq_len 21, 3 samples per GPU, batch-sharded,
    ONE NCCL all-reduce over the flat gradient buffer, fused Adam on the backbone parameters.  A step = forward of
    21 timesteps (states carried) + synthetic loss on the last step's four feature maps + backward through all 21
    timesteps + gradient all-reduce + unscale + optimizer step."""
    import torch.distributed as dist
    import rvt_b200  # noqa: F401
    from rvt_b200 import sharding

    dev = torch.device('cuda', local_rank)
    B = args.train_batch
    model = build_model(0).to(dev).train()
    model.pad_to_hw = (PAD_H, PAD_W)
    model.train_wavefront = args.train_wavefront      # stage-per-stream schedule (measured slower in training: off by default)
    lo, hi = sharding.batch_slice(B * world, rank, world)
    n_seq = 4                                                        # rotate sequences: 4 x 290 MB of uint8 inputs > L2
    seqs = [make_uint8_sequence(4321 + lo * 10 + i, SEQ_LEN, B).to(dev) for i in range(n_seq)]
    params = [p for p in model.parameters() if p.requires_grad]
    opt = torch.optim.Adam(params, lr=2e-4, fused=True)
    ev = {k: [torch.cuda.Event(enable_timing=True) for _ in range(2)] for k in ('fwd', 'bwd', 'ar', 'opt')}
    acc_ms = {k: 0.0 for k in ev}
    counter = [0]

    cpu_ms = {'fwd': 0.0, 'bwd': 0.0}
    graphed = {}

    def fwd_bwd(seq, record=False):
        if record:
            ev['fwd'][0].record()
        t0 = time.perf_counter()
        st, out = None, None
        for t in range(SEQ_LEN):
            out, st = model(seq[t], st)
        loss = sum((out[s].float() ** 2).mean() for s in (1, 2, 3, 4)) * LOSS_SCALE
        t1 = time.perf_counter()
        if record:
            ev['fwd'][1].record(); ev['bwd'][0].record()
        loss.backward()
        t2 = time.perf_counter()
        if record:
            ev['bwd'][1].record()
            cpu_ms['fwd'] += (t1 - t0) * 500; cpu_ms['bwd'] += (t2 - t1) * 500    # mean of the 2 recorded steps, ms
        return loss

    def capture():
        # ONE CUDA graph of forward (21 timesteps) + loss + backward (rvt_b200.graph.capture_training_step): the weight
        # re-packing, every kernel and the gradient hand-over are replayed without Python; the all-reduce and the optimizer
        # stay outside.  p.grad become static tensors that each replay overwrites.
        from rvt_b200.graph import capture_training_step
        static_seq = torch.empty_like(seqs[0])
        graphed['seq'] = static_seq
        graphed['run'] = capture_training_step(model, lambda: fwd_bwd(static_seq), params)

    def step(record=False):
        seq = seqs[counter[0] % n_seq]
        counter[0] += 1
        if graphed:
            graphed['seq'].copy_(seq, non_blocking=True)
            if record:
                ev['fwd'][0].record(); ev['fwd'][1].record(); ev['bwd'][0].record()
            loss = graphed['run']()
            if record:
                ev['bwd'][1].record()
        else:
            opt.zero_grad(set_to_none=True)
            loss = fwd_bwd(seq, record)
        if record:
            ev['ar'][0].record()
        n_coll = sharding.allreduce_gradients(params)
        if record:
            ev['ar'][1].record(); ev['opt'][0].record()
        torch._foreach_mul_([p.grad for p in params if p.grad is not None], 1.0 / LOSS_SCALE)
        opt.step()
        if record:
            ev['opt'][1].record()
        return loss, n_coll

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    if not args.train_eager:
        capture()            # (no eager step before this: AccumulateGrad nodes must first be created on the capture stream)
    for _ in range(max(warmup, 3)):
        loss, n_coll = step()
    assert torch.isfinite(loss.detach()).item(), 'non-finite training loss'
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        loss, n_coll = step()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = sharding.max_over_ranks(e0.elapsed_time(e1), dev)
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    for _ in range(2):                                               # phase breakdown (separate, event-instrumented steps)
        step(record=True)
        torch.cuda.synchronize(dev)
        for k in ev:
            acc_ms[k] += ev[k][0].elapsed_time(ev[k][1]) / 2
    grad_ok = all(p.grad is not None and bool(torch.isfinite(p.grad).all()) for p in params)
    ar_ms = sharding.max_over_ranks(acc_ms['ar'], dev)
    frames = B * SEQ_LEN * steps * world
    n_par = sum(p.numel() for p in params)
    return {
        'metric': TRAIN_METRIC, 'value': frames / (ms * 1e-3), 'unit': 'frames/s', 'n_gpus': world, 'steps': steps,
        'warmup': max(warmup, 3), 'ms_per_step': ms / steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
        'config': {'workload': f'RVT-Base 1Mpx {B}x20x360x640 uint8 per GPU (model res 384x640) TBPTT seq_len=21 training step: '
                               'fwd + bwd through 21 timesteps + grad all-reduce + fused Adam (backbone only)',
                   'global_batch': B * world, 'frames_per_step': B * SEQ_LEN,
                   'l2_policy': f'{n_seq} rotating input sequences ({n_seq * seqs[0].numel() >> 20} MB) > L2',
                   'parallelism': f'batch-sharded x{world}; {n_coll} NCCL all-reduce of {n_par * 4 >> 20} MB fp32 gradients per step',
                   'loss_scale': LOSS_SCALE},
        'schedule': ('eager launches' if args.train_eager else 'fwd+bwd replayed as one CUDA graph; all-reduce + Adam eager') +
                    ('; stage-per-stream wavefront (4 streams)' if args.train_wavefront else ''),
        'clocks': clocks, 'phases_ms': acc_ms, 'allreduce_ms_max_over_ranks': ar_ms, 'n_collectives': n_coll,
        'allreduce_bytes': n_par * 4, 'cpu_issue_ms': cpu_ms if args.train_eager else None,
        'final_loss': float(loss.detach()) / LOSS_SCALE, 'grads_finite': grad_ok,
    }


def run_train(args, rank, world, local_rank):
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    line = train_leg(args, rank, world, local_rank, args.steps, args.warmup)
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_MAX_ELEMS = 1 << 21      # per array (8 MB of float32): the eight state arrays of RVT-B stay below 64 MB in all


def dump_outputs(out_dir, states):
    """Write what one timed step returns -- the final (h, c) of every stage, NCHW float32 -- as
    out_dir/stage<s>_h.npy and out_dir/stage<s>_c.npy (s = 1..4).  An array of more than DUMP_MAX_ELEMS
    elements is written as a fixed sample: the values at DUMP_MAX_ELEMS ascending flat NCHW positions
    drawn with seed 0, the same positions on every run, so two builds can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for s, (h, c) in enumerate(states, 1):
        for name, t in (('h', h), ('c', c)):
            a = t.float().contiguous().cpu().numpy()
            if a.size > DUMP_MAX_ELEMS:
                idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))
                a = a.reshape(-1)[idx]
            np.save(os.path.join(out_dir, f'stage{s}_{name}.npy'), a)


def count_kernel_launches(fn, dev):
    """MEASURED number of GPU kernels one call of `fn` launches (CUPTI activity records through torch.profiler; kernels
    launched by CUDA-graph replay and through the ctypes C-ABI are included).  Returns (count, {name: count})."""
    try:
        from torch.profiler import profile, ProfilerActivity
        torch.cuda.synchronize(dev)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize(dev)
        names = {}
        for e in prof.events():
            if getattr(e, 'device_type', None) is not None and 'cuda' in str(e.device_type).lower():
                n = e.name
                if n.startswith('Memcpy') or n.startswith('Memset'):
                    continue
                names[n] = names.get(n, 0) + 1
        return sum(names.values()), names
    except Exception as ex:            # profiler unavailable: fall back to the analytic count, and say so
        return None, {'error': repr(ex)}


def voxel_leg(dev, peak_gbs):
    """BASELINE configs[4]: 50 M synthetic (x, y, t, p) events -> StackedHistogram 2 x 10 x 720 x 1280 (uint8)."""
    import rvt_b200
    n, H, W, bins = 50_000_000, 720, 1280, 10
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randint(0, W, (n,), generator=g, device=dev, dtype=torch.int64)
    y = torch.randint(0, H, (n,), generator=g, device=dev, dtype=torch.int64)
    p = torch.randint(0, 2, (n,), generator=g, device=dev, dtype=torch.int64)
    t = torch.sort(torch.randint(0, 50000, (n,), generator=g, device=dev, dtype=torch.int64)).values
    sh = rvt_b200.StackedHistogram(bins, H, W, 10, fastmode=True, validate=False)
    out = torch.empty(sh.get_shape(), dtype=torch.uint8, device=dev)
    for _ in range(3):
        sh.construct(x, y, p, t, out=out)
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    e0.record()
    for _ in range(reps):
        sh.construct(x, y, p, t, out=out)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    total = int(out.sum(dtype=torch.int64).item())
    algo_bytes = 32 * n + out.numel()                       # SURVEY 8(d): 32 B/event (int64 x, y, p, t) + 1 B per output bin
    del x, y, p, t
    return {'events': n, 'ms': ms, 'events_per_s': n / (ms * 1e-3), 'algorithmic_bytes': algo_bytes,
            'gbs': algo_bytes / ms / 1e6, 'frac_of_hbm_peak': algo_bytes / ms / 1e6 / peak_gbs, 'out_sum': total,
            'workload': '50 M uniform events, sorted timestamps, 2x10x720x1280 uint8, count_cutoff 10, fastmode; 1.6 GB of int64 inputs > L2'}


def eager_gpu_leg(dev, steps=2):
    """The reference's op-by-op PyTorch path on the SAME GPU (oracle port = the same ATen / cuDNN / cuBLAS calls) under fp16
    autocast + inference_mode, inputs resident: the denominator of north_star's '>= 10x PyTorch-eager'."""
    from oracle import backbone_oracle as bo
    spec = rvt_b_spec()
    params = {k: v.to(dev) for k, v in bo.synth_params(spec, 0).items()}
    seq = make_uint8_sequence(1234, SEQ_LEN, B_PER_GPU).to(dev)

    def step():
        st = None
        for t in range(SEQ_LEN):
            x = torch.nn.functional.pad(seq[t].float(), (0, PAD_W - IN_W, 0, PAD_H - IN_H))   # modules/detection.py:133-134
            _, st = bo.backbone_forward(x, st, params, spec)

    with torch.inference_mode(), torch.autocast('cuda', dtype=torch.float16):
        step()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {'frames_per_s': B_PER_GPU * SEQ_LEN / (ms * 1e-3), 'ms_per_step': ms, 'steps': steps,
            'what': 'oracle port of the reference op sequence, PyTorch eager, fp16 autocast, inference_mode, inputs resident'}


def dropin_leg(model, seq_dev, dev, steps=3):
    """Exactly what the UNMODIFIED harness does (modules/detection.py:131-148): a Python loop over the timesteps, every
    timestep uint8 -> float32 + zero pad to the model resolution, then forward(x, prev_states) -- eager launches, one
    stream, no graph, no wavefront."""
    model.pad_to_hw = None

    def step():
        st = None
        for t in range(SEQ_LEN):
            x = torch.nn.functional.pad(seq_dev[t].to(torch.float32), (0, PAD_W - IN_W, 0, PAD_H - IN_H))
            _, st = model(x, st)

    with torch.inference_mode():
        step()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize(dev)
    model.pad_to_hw = (PAD_H, PAD_W)
    ms = e0.elapsed_time(e1) / steps
    return {'frames_per_s': B_PER_GPU * SEQ_LEN / (ms * 1e-3), 'ms_per_step': ms, 'steps': steps,
            'what': 'per-timestep RNNDetector.forward() from a Python loop, fp32 padded input, eager launches (reference harness call pattern)'}


def rvt_s_gen1_leg(dev, steps=5):
    """BASELINE configs[3]: RVT-Small Gen1 (240x304 -> 256x320, dim_head 24, P = 80) eval, batch 64."""
    import rvt_b200
    cfg = rvt_b_cfg()
    cfg['embed_dim'] = 48
    cfg['partition_split_32'] = 1
    cfg['stage']['attention']['dim_head'] = 24
    cfg['stage']['attention']['partition_size'] = (8, 10)
    model = rvt_b200.RNNDetector(cfg)
    g = torch.Generator(device='cpu').manual_seed(3)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.endswith('gamma') or ('norm' in name and name.endswith('weight')):
                p.copy_(torch.rand(p.shape, generator=g) + 0.5)
            elif name.endswith('bias'):
                p.copy_(torch.randn(p.shape, generator=g) * 0.1)
            else:
                p.copy_(torch.randn(p.shape, generator=g) / p[0].numel() ** 0.5)
    model = model.to(dev).eval()
    model.pad_to_hw = (256, 320)
    L, B = 5, 64
    gg = torch.Generator(device=dev).manual_seed(9)
    seq = torch.randint(1, 11, (L, B, IN_C, 240, 304), generator=gg, device=dev, dtype=torch.uint8)
    seq = seq * (torch.randint(0, 10, seq.shape, generator=gg, device=dev, dtype=torch.uint8) == 0)
    with torch.inference_mode():
        run = rvt_b200.GraphedCallable(lambda: model.forward_sequence(seq, None, wavefront=True)[1], warmup=2)
        for _ in range(3):
            run()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            run()
        e1.record()
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {'frames_per_s': L * B / (ms * 1e-3), 'ms_per_step': ms, 'steps': steps,
            'workload': f'RVT-Small Gen1 {B}x20x240x304 uint8 (model res 256x320), {L} timesteps, states carried, graph replay'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference', 'reference-gpu'])
    ap.add_argument('--mode', default='infer', choices=['infer', 'train'],
                    help="infer: BASELINE configs[1] (the headline metric) + the extra legs; train: configs[2] alone")
    ap.add_argument('--train-batch', type=int, default=3, help='samples per GPU of the training step (BASELINE configs[2]: 3)')
    ap.add_argument('--train-wavefront', action='store_true', help='training step: stage-per-stream schedule (fwd and bwd)')
    ap.add_argument('--train-eager', action='store_true',
                    help='training step: launch forward+backward eagerly instead of replaying one CUDA graph of them')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch eagerly instead of replaying CUDA graphs')
    ap.add_argument('--no-wavefront', action='store_true', help='run the four stages strictly one after the other')
    ap.add_argument('--extras', default='train,voxel,eager_gpu,dropin,rvt_s_gen1_bs64',
                    help='comma list of the extra legs reported under "extra" (empty string: none)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the final states of the last timed step (rank 0) to DIR/*.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or args.mode != 'infer'):
        ap.error('--dump-outputs applies to the inference benchmark (--impl ours --mode infer)')

    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    protect_stdout()

    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if args.impl == 'reference-gpu':
        run_reference_gpu(args, rank, world, local_rank)
        return
    if args.mode == 'train':
        run_train(args, rank, world, local_rank)
        return

    import torch.distributed as dist
    import rvt_b200
    from rvt_b200 import sharding

    extras_wanted = [e for e in args.extras.split(',') if e]
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        # NCCL prints its version banner to STDOUT at NCCL_DEBUG=VERSION (the image default); stdout must carry
        # exactly one JSON line, so keep NCCL at WARN unless the user asked for more.
        if os.environ.get('NCCL_DEBUG', '').upper() in ('', 'VERSION'):
            os.environ['NCCL_DEBUG'] = 'WARN'
        dist.init_process_group('nccl', device_id=dev)

    model = build_model(0).to(dev).eval()
    model.pad_to_hw = (PAD_H, PAD_W)

    # weak scaling: the global batch is 8*N samples; this rank owns [lo, hi) and its states (no exchange)
    lo, hi = sharding.batch_slice(B_PER_GPU * world, rank, world)
    assert hi - lo == B_PER_GPU
    # synthetic uint8 event tensors: SEQ_LEN timesteps, resident on the device (37 MB each)
    g = torch.Generator(device='cpu').manual_seed(1234 + lo)
    shape = (SEQ_LEN, B_PER_GPU, IN_C, IN_H, IN_W)
    seq_host = torch.randint(1, 11, shape, generator=g, dtype=torch.uint8)         # counts 1..10 ...
    seq_host.mul_(torch.randint(0, 10, shape, generator=g, dtype=torch.uint8) == 0)  # ... on ~10 % of the bins
    seq_host = seq_host.pin_memory()
    seq_dev = seq_host.to(dev)

    wavefront = not args.no_wavefront

    def run_sequence_resident():
        _, st = model.forward_sequence(seq_dev, None, wavefront=wavefront)
        return st

    feat_host = torch.empty((B_PER_GPU, 512, PAD_H // 32, PAD_W // 32), dtype=torch.float32).pin_memory()
    copy_stream = torch.cuda.Stream(dev)

    seq_stage = torch.empty_like(seq_dev)        # device landing buffers of the per-timestep H2D copies
    d2h_stream = torch.cuda.Stream(dev)

    def run_sequence_e2e():
        """Public API with HOST buffers: every timestep's uint8 event tensor is copied H2D from pinned
        memory (copy stream, overlapping compute), the sequence runs through
        RNNDetector.forward_sequence, and every timestep's stage-4 feature map is read back D2H."""
        main_s = torch.cuda.current_stream(dev)
        copy_stream.wait_stream(main_s)
        ready = []
        with torch.cuda.stream(copy_stream):
            for tstep in range(SEQ_LEN):
                seq_stage[tstep].copy_(seq_host[tstep], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
                ready.append(ev)
        outs, st = model.forward_sequence(seq_stage, None, wavefront=wavefront, input_ready=ready)
        with torch.cuda.stream(d2h_stream):
            for tstep in range(SEQ_LEN):
                d2h_stream.wait_event(model.last_step_events[tstep])
                feat_host.copy_(outs[tstep][4], non_blocking=True)
        main_s.wait_stream(d2h_stream)
        main_s.wait_stream(copy_stream)
        return st

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(fn, steps):
        """(device ms of `steps` calls of fn, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = sharding.max_over_ranks(e0.elapsed_time(e1), dev)     # device time, max over ranks
        barrier()
        return ms, out

    with torch.inference_mode():
        if args.no_graph:
            step_resident, step_e2e = run_sequence_resident, run_sequence_e2e
        else:
            # whole-sequence CUDA graphs (rvt_b200.graph): kernels + H2D/D2H copies of all 4+2 streams
            step_resident = rvt_b200.GraphedCallable(run_sequence_resident, warmup=2)
            step_e2e = rvt_b200.GraphedCallable(run_sequence_e2e, warmup=2)
        for _ in range(max(args.warmup, 3)):
            step_resident()
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        ms, last_states = timed(step_resident, args.steps)
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, last_states)
        for _ in range(3):
            step_e2e()
        ms_e2e, _ = timed(step_e2e, args.steps)
        launches_per_step, launch_names = (None, {})
        if rank == 0:
            launches_per_step, launch_names = count_kernel_launches(step_resident, dev)

    # ---- roofline of the dominant kernel, timed live with CUDA events on its launch stream ----
    # fused attention, stage-1 instance (largest single-kernel share of the step): one launch = the attention half of one
    # PartitionAttentionCl block over 8 x 96 x 160 tokens, C = 64.
    roof = None
    if rank == 0:
        from rvt_b200 import ops
        with torch.inference_mode():
            pk = model._ensure_packed(dev)[0]
            blk = pk['blocks'][0]
            n_tok, c, P = B_PER_GPU * 96 * 160, 64, 60
            bufs = [torch.randn(B_PER_GPU, 96, 160, c, device=dev) for _ in range(10)]   # 315 MB > L2: cold x every launch
            dummy = torch.empty(1, dtype=torch.float16, device=dev)
            for xb in bufs[:3]:
                ops.partition_attention_(xb, blk, dummy, dummy, dummy)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 3
            e0.record()
            for _ in range(reps):
                for xb in bufs:
                    ops.partition_attention_(xb, blk, dummy, dummy, dummy)
            e1.record()
            torch.cuda.synchronize(dev)
            us = e0.elapsed_time(e1) * 1e3 / (reps * len(bufs))
            del bufs
        algo_bytes = 2 * n_tok * c * 4                               # x read + x written, fp32 (SURVEY §8d)
        algo_flops = 8 * n_tok * c * c + 4 * n_tok * P * c           # qkv + proj + QK^T + PV
        kname = next((k for k in launch_names if 'attn' in k), 'attn kernel')
        roof = {'kernel': f'{kname.split("(")[0]} (stage 1 window block, C=64, 122880 tokens)', 'us_per_launch': us,
                'algorithmic_bytes': algo_bytes, 'algorithmic_flops': algo_flops}

    # ---- extra legs (all inside this one driver-run line) ----
    extra = {}
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak_gbs = peaks.get('hbm_gbs', 6650.0)
    if 'train' in extras_wanted:
        del step_resident, step_e2e
        torch.cuda.empty_cache()
        tr = train_leg(args, rank, world, local_rank, steps=min(args.steps, 5), warmup=3)
        extra['train'] = {k: tr[k] for k in ('value', 'unit', 'ms_per_step', 'steps', 'n_gpus', 'phases_ms',
                                             'allreduce_ms_max_over_ranks', 'n_collectives', 'allreduce_bytes', 'schedule',
                                             'grads_finite')}
        extra['train']['config'] = tr['config']
        torch.cuda.empty_cache()
    if rank == 0:
        def guarded(name, fn):
            if name not in extras_wanted:
                return
            try:
                extra[name] = fn()
            except Exception as ex:
                extra[name] = {'error': repr(ex)}
            torch.cuda.empty_cache()
        guarded('dropin', lambda: dropin_leg(model, seq_dev, dev))
        guarded('voxel', lambda: voxel_leg(dev, peak_gbs))
        guarded('rvt_s_gen1_bs64', lambda: rvt_s_gen1_leg(dev))
        guarded('eager_gpu', lambda: eager_gpu_leg(dev))

    frames = B_PER_GPU * SEQ_LEN * args.steps * world
    value = frames / (ms * 1e-3)
    e2e = frames / (ms_e2e * 1e-3)
    if rank == 0:
        peak_tf = peaks.get('bf16_tflops_sustained', 1400.0)
        peak_src = 'measured (MEASURED_PEAKS.json)' if peaks else 'fallback (B200_PROFILING.md)'
        ach_tf = value / world * GFLOP_PER_FRAME / 1e3
        ach_gbs = roof['algorithmic_bytes'] / roof['us_per_launch'] / 1e3
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, 'profiles', 'traffic_r02.json'))).get('attn_s1_dram_bytes')
        except Exception:
            pass
        if 'eager_gpu' in extra and 'frames_per_s' in extra['eager_gpu']:
            extra['eager_gpu']['ours_over_eager'] = value / world / extra['eager_gpu']['frames_per_s']
        line = {
            'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f16', 'data': 'synthetic',
            'config': {'workload': 'RVT-Base 1Mpx 8x20x360x640 uint8 (model res 384x640) seq_len=21 bs=8/GPU '
                                   'inference, states carried', 'frames_per_step': B_PER_GPU * SEQ_LEN,
                       'l2_policy': 'inputs larger than L2 (774 MB of uint8 sequences per GPU)',
                       'parallelism': f'batch-sharded x{world}, no collective',
                       'schedule': ('wavefront over 4 streams' if wavefront else 'sequential') +
                                   (', eager launches' if args.no_graph else ', CUDA-graph replay')},
            'e2e': {'value': e2e, 'unit': 'frames/s',
                    'h2d_bytes_per_step': SEQ_LEN * B_PER_GPU * IN_C * IN_H * IN_W,
                    'd2h_bytes_per_step': SEQ_LEN * feat_host.numel() * 4},
            'gpu_launches': (launches_per_step if launches_per_step is not None else LAUNCHES_PER_TIMESTEP * SEQ_LEN) * args.steps,
            'gpu_launches_how': ('measured: CUPTI kernel records of one replayed step x steps' if launches_per_step is not None
                                 else 'analytic (profiler unavailable)'),
            'kernels_per_step': launch_names,
            'clocks': clocks,
            # C = 64: 94 FLOP/B algorithmic intensity, below the 263 FLOP/B ridge -> HBM is the bounding roof
            'roofline': {'bound': 'hbm', 'achieved': ach_gbs, 'peak': peak_gbs, 'unit': 'GB/s',
                         'frac': ach_gbs / peak_gbs, 'traffic': traffic, 'kernel': roof['kernel'],
                         'us_per_launch': roof['us_per_launch'], 'peak_source': peak_src,
                         'tensor_tflops': roof['algorithmic_flops'] / roof['us_per_launch'] / 1e6,
                         'note': 'algorithmic bytes = x read + written (fp32) = 62.9 MB per launch; see DESIGN.md §6'},
            'whole_step': {'algorithmic_tflops': ach_tf, 'frac_of_sustained_bf16_peak': ach_tf / peak_tf,
                           'gflop_per_frame': GFLOP_PER_FRAME},
            'extra': extra,
        }
        if not args.no_cpu_baseline:
            cores = best_cpu_threads()
            v = cpu_reference_fps(SEQ_LEN, B_PER_GPU, cores)
            line['cpu_baseline'] = {'value': v, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                                    'sample': f'one full sequence: {SEQ_LEN} timesteps x batch {B_PER_GPU} (after 1 warm-up timestep), '
                                              f'fp32 torch CPU ops; {cores} threads = best of a sweep up to os.cpu_count()={os.cpu_count()}'}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
