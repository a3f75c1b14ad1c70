"""Benchmark of the PASTA-GAN++ 512 px generator on this repo's sm_100a kernels (BASELINE.json configs[1]).

    python bench.py --gpus 1 --steps 10 --warmup 3                 # this repo's kernels, full generator, batch 32 per GPU
    python bench.py --impl reference --steps 3 --warmup 1          # the CPU ref path (oracle port) on the host cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port P bench.py --gpus 8 ...
    python bench.py --workload chain                               # only the modulated-conv synthesis chain (round-1 early workload)
    python bench.py --steps 10 --warmup 3 --dump-outputs DIR       # also write what the last timed step returned, as DIR/<name>.npy

One "step" = one batch (default 32 images per GPU) through `GeneratorFull_v20.forward` (pgpp_b200.training.generator, same
state-dict as the reference): const / style encoders, mapping, synthesis blocks b8..b512, SPADE blocks and the texture branch --
per image 24 modulated_conv2d + 76 plain convolutions (all on the tcgen05 implicit-GEMM kernel), the FIR resamplers and the
bias_act calls; instance norm / nearest resize / masks / per-pixel Linear stay PyTorch library ops as in the reference.

Prints ONE JSON line (rank 0).  `value` is device-resident throughput over all GPUs in the fp32-parity mode (bf16x2 split
MMAs); `e2e` goes through the pipeline API with uint8 pinned-host inputs and the try-on image read back to the host inside the
timed region; `bf16_mode` reports the single-product bf16 mode separately; `roofline` describes the dominant kernel launch.
"""
import argparse
import importlib
import importlib.util
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W_DIM = 512
RES = 512
DUMP_BYTES = 64 * 2 ** 20


def dump_outputs(out_dir, outputs):
    """Write `outputs` (name -> tensor, what the timed step returned) as out_dir/<name>.npy, float64 as float64 and every other dtype
    as float32.  Above DUMP_BYTES in all, every output keeps the same rows of its leading (batch) dimension, drawn with a fixed seed, so
    that two builds run with the same arguments can be compared output for output."""
    arrays = {name.replace('/', '_'): t.detach().to(torch.float64 if t.dtype == torch.float64 else torch.float32) for name, t in outputs.items()}
    total = sum(a.numel() * a.element_size() for a in arrays.values())
    if total > DUMP_BYTES:
        batch = {a.shape[0] for a in arrays.values()}
        assert len(batch) == 1, f'outputs of {total} bytes without a common batch dimension to sample: {sorted(batch)}'
        batch = batch.pop()
        keep = DUMP_BYTES * batch // total
        assert keep >= 1, f'one batch row of the outputs is larger than {DUMP_BYTES} bytes'
        rows = torch.randperm(batch, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        arrays = {name: a.index_select(0, rows.to(a.device)) for name, a in arrays.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f'{name}.npy'), a.cpu().numpy())


def build_chain(device, resolution=RES):
    from __graft_entry__ import load_pkg
    load_pkg()
    synthesis = importlib.import_module('pgpp_b200.training.synthesis')
    torch.manual_seed(0)
    net = synthesis.SynthesisChain(w_dim=W_DIM, img_resolution=resolution).eval()
    # random init like the reference (weights N(0,1), biases 0, affine bias 1); non-zero noise strength so the
    # noise path is exercised (the reference initialises it to 0)
    for name, p in net.named_parameters():
        if name.endswith('noise_strength'):
            p.data.fill_(0.1)
    return net.to(device).requires_grad_(False)


def build_generator(device):
    """GeneratorFull_v20 with the reference's configuration, name-seeded random weights (same recipe as the golden fixture)"""
    from __graft_entry__ import load_pkg
    load_pkg()
    gen = importlib.import_module('pgpp_b200.training.generator')
    G = gen.build_generator().eval()
    import zlib
    with torch.no_grad():
        for name, t in list(G.named_parameters()) + list(G.named_buffers()):
            if not torch.is_floating_point(t) or name.endswith('resample_filter') or name.endswith('w_avg'):
                continue
            g = torch.Generator().manual_seed(zlib.crc32(name.encode()) & 0x7FFFFFFF)
            v = torch.randn(t.shape, generator=g)
            if name.endswith('noise_strength'):
                v = torch.full(t.shape, 0.1)
            elif name.endswith('affine.bias'):
                v = 1.0 + 0.1 * v
            elif name.endswith('bias') or name.endswith('m_bias1'):
                v = 0.1 * v
            elif name.endswith('linear.weight'):
                v = v / (t.shape[1] ** 0.5)
            elif name.startswith('mapping.fc'):
                v = v * 100.0
            t.copy_(v)
    return G.to(device).requires_grad_(False)


def make_generator_inputs_u8(batch, seed):
    """synthetic 512x320 try-on inputs as the dataset delivers them: uint8 host tensors (test.py:126-147 converts on the GPU).
    Signal in columns 96..415, constant side bands (SURVEY 8d)."""
    g = torch.Generator().manual_seed(seed)
    band = torch.zeros(1, 1, 1, 512, dtype=torch.bool); band[..., 96:416] = True

    def img(ch, fill):
        t = torch.randint(0, 256, (batch, ch, 512, 512), generator=g, dtype=torch.uint8)
        return torch.where(band, t, torch.full_like(t, fill))
    return dict(c=torch.randint(0, 256, (batch, 45, 128, 128), generator=g, dtype=torch.uint8),
                retain=img(6, 255), pose=img(5, 0), denorm_upper=img(3, 255), denorm_lower=img(3, 255),
                denorm_upper_mask=(torch.rand(batch, 1, 512, 512, generator=g) > 0.5).to(torch.uint8) * band,
                denorm_lower_mask=(torch.rand(batch, 1, 512, 512, generator=g) > 0.5).to(torch.uint8) * band)


def to_device_f32(u8, device):
    """H2D of the uint8 batch + the /127.5 - 1 conversion of test.py:126-147 on the device (pgpp_u8_to_f32; masks: plain cast)"""
    io = importlib.import_module('pgpp_b200.torch_utils.custom_ops').get_plugin('io_edge_plugin')
    out = {}
    for k, v in u8.items():
        d = v.to(device, non_blocking=True)
        out[k] = io.u8_to_f32(d, torch.empty(d.shape, dtype=torch.float32, device=device), normalize=not k.endswith('mask'))
    return out


def run_generator(G, x, gt_parsing=None):
    with torch.no_grad():
        return G(torch.zeros(x['c'].shape[0], 0, device=x['c'].device), x['c'], x['retain'], x['pose'], x['denorm_upper'], x['denorm_lower'],
                 x['denorm_upper_mask'], x['denorm_lower_mask'], gt_parsing=gt_parsing, noise_mode='const')


def make_inputs(net, batch, seed, device='cpu', pin=False):
    g = torch.Generator().manual_seed(seed)
    ws = torch.randn(batch, net.num_ws, W_DIM, generator=g)
    pose = torch.randn(batch, net.channels[8], 8, 8, generator=g)
    if pin:
        ws, pose = ws.pin_memory(), pose.pin_memory()
    return ws.to(device) if device != 'cpu' else ws, pose.to(device) if device != 'cpu' else pose


def make_cat_feats(net, batch, device):
    # warped garment features: produced on-GPU by the style encoder in the full generator -> device-resident here
    g = torch.Generator().manual_seed(1)
    return {str(r): torch.randn(batch, 64, r, r, generator=g).clamp_(-1, 1).to(device) for r in net.block_resolutions if r > 32}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                                          '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            self.thread.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [v.strip() for v in l.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': statistics.median(sm), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons), 'samples': len(sm)}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        p = json.load(open(path))
        return {'tflops': p['bf16_tflops_sustained'], 'gbs': p['hbm_gbs'], 'source': 'MEASURED_PEAKS.json (bf16 sustained, HBM copy)'}
    return {'tflops': 1400.0, 'gbs': 6650.0, 'source': 'fallback of B200_PROFILING.md (1.4 PF sustained, 6.65 TB/s)'}


def host_threads():
    """all host threads this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm must not inherit that)"""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_reference_rate(net_sd, num_ws, c8, batch, reps, threads=None):
    """images/s of the CPU ref path (oracle port of the reference's impl='ref' ops) on the host cores."""
    from oracle import ref_chain
    torch.set_num_threads(threads or host_threads())
    g = torch.Generator().manual_seed(7)
    ws = torch.randn(batch, num_ws, W_DIM, generator=g)
    pose = torch.randn(batch, c8, 8, 8, generator=g)
    cat = {str(r): torch.randn(batch, 64, r, r, generator=g).clamp_(-1, 1) for r in (64, 128, 256, 512)}
    times = []
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            ref_chain.synthesis_chain(net_sd, ws, pose, cat, img_resolution=RES)
            times.append(time.perf_counter() - t0)
    return batch / min(times), times


GEN_DESC = ('PASTA-GAN++ GeneratorFull_v20 512px inference (train.py:191-202 config, 43.1 M params, random weights): encoders + mapping + '
            'synthesis b8..b512 + SPADE blocks + texture branch = 24 modulated_conv2d + 76 plain convs + upfirdn2d + bias_act per image')
CHAIN_DESC = ('PASTA-GAN++ 512px generator synthesis chain only: 24 modulated_conv2d (+bias_act, noise, ToRGB accumulate), 5 merge 1x1 convs, '
              '6 image-skip upfirdn2d; SPADE blocks/encoders not included')


def generator_cpu_rate(reps, threads):
    """images/s of the full generator on the CPU ref path (oracle/ref_generator.py over torch CPU ops), batch 1 per rep"""
    from oracle import ref_generator
    torch.set_num_threads(threads)
    G = build_generator('cpu')
    sd = {k: v.detach() for k, v in G.state_dict().items()}
    inp = ref_generator.synthetic_inputs(1, seed=3)
    times = []
    with torch.no_grad():
        for _ in range(reps):
            t0 = time.perf_counter()
            ref_generator.generator(sd, inp['c'], inp['retain'], inp['pose'], inp['denorm_upper'], inp['denorm_lower'],
                                    inp['denorm_upper_mask'], inp['denorm_lower_mask'], None)
            times.append(time.perf_counter() - t0)
    return times


def run_reference(args):
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    cores = host_threads()
    torch.set_num_threads(cores)
    batch = 1
    if args.workload == 'generator':
        if args.warmup:
            generator_cpu_rate(1, cores)
        times = generator_cpu_rate(args.steps, cores)
        metric, desc, src = 'generator_512px_images_per_sec', GEN_DESC, 'oracle/ref_generator.py'
    else:
        net = build_chain('cpu')
        sd = {k: v.detach() for k, v in net.state_dict().items()}
        for _ in range(args.warmup):
            cpu_reference_rate(sd, net.num_ws, net.channels[8], batch, 1)
        _, times = cpu_reference_rate(sd, net.num_ws, net.channels[8], batch, args.steps)
        metric, desc, src = 'synthesis_hot_path_images_per_sec', CHAIN_DESC, 'oracle/ref_chain.py'
    value = batch * args.steps / sum(times)
    line = {
        'impl': 'reference', 'metric': metric, 'value': value, 'unit': 'images/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * sum(times) / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': desc + '; CPU ref path, bounded sample of batch 1 per step', 'resolution': RES},
        'cpu_baseline': {'value': value, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{args.steps} steps of batch {batch} through {src} (torch CPU ops, {cores} threads)'},
        'e2e': {'value': value, 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


class SynthesisPipeline:
    """The public end-to-end call: pinned host inputs -> device -> synthesis chain -> image back in pinned host memory.
    Copies run on a side stream so the read-back of batch i overlaps the compute of batch i+1."""

    def __init__(self, net, cat_feats, batch, device):
        self.net, self.cat, self.device = net, cat_feats, device
        self.copy_stream = torch.cuda.Stream(device)
        self.out_host = [torch.empty(batch, RES, RES, 3, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.io = importlib.import_module('pgpp_b200.torch_utils.custom_ops').get_plugin('io_edge_plugin')
        self.slot = 0
        self.pending = None

    def __call__(self, ws_host, pose_host):
        cur = torch.cuda.current_stream(self.device)
        ws = ws_host.to(self.device, non_blocking=True)
        pose = pose_host.to(self.device, non_blocking=True)
        with torch.no_grad():
            img, parsing, tex = self.net(ws, pose, self.cat, noise_mode='const')
        done = torch.cuda.Event()
        done.record(cur)
        self.copy_stream.wait_event(done)
        with torch.cuda.stream(self.copy_stream):
            host = self.out_host[self.slot]
            host.copy_(img, non_blocking=True)
            img.record_stream(self.copy_stream)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        prev, self.pending = self.pending, (ev, host)
        self.slot ^= 1
        if prev is not None:
            prev[0].synchronize()       # the previous batch is now readable on the host
        return prev[1] if prev is not None else None

    def flush(self):
        if self.pending is not None:
            self.pending[0].synchronize()
            host, self.pending = self.pending[1], None
            return host
        return None


class GeneratorPipeline:
    """End-to-end call for the full generator: uint8 pinned-host try-on inputs -> device (+ /127.5-1 conversion, test.py:126-147)
    -> GeneratorFull_v20 -> uint8 BGR HWC try-on image (pgpp_image_to_u8, test.py:162-166) back in pinned host memory.  The upload of
    batch i + 1 (own stream, two staging sets) and the read-back of batch i - 1 (own stream) overlap the compute of batch i."""

    def __init__(self, G, batch, device, graphed=None):
        self.G, self.device, self.graphed = G, device, graphed
        self.copy_stream = torch.cuda.Stream(device)
        # uploads run on their own stream into one of two uint8 staging sets, so the H2D copy of batch i overlaps the compute of batch i - 1
        self.up_stream = torch.cuda.Stream(device)
        self.stage, self.stage_free, self.in_slot = [None, None], [None, None], 0
        self.out_host = [torch.empty(batch, RES, RES, 3, dtype=torch.uint8).pin_memory() for _ in range(2)]
        self.io = importlib.import_module('pgpp_b200.torch_utils.custom_ops').get_plugin('io_edge_plugin')
        self.slot, self.pending = 0, None

    def __call__(self, host_u8):
        cur = torch.cuda.current_stream(self.device)
        slot = self.in_slot
        self.in_slot ^= 1
        if self.stage[slot] is None:
            self.stage[slot] = {k: torch.empty(v.shape, dtype=torch.uint8, device=self.device) for k, v in host_u8.items()}
        with torch.cuda.stream(self.up_stream):
            if self.stage_free[slot] is not None:
                self.up_stream.wait_event(self.stage_free[slot])        # the conversion that last read this staging set has run
            for k, v in host_u8.items():
                self.stage[slot][k].copy_(v, non_blocking=True)
            uploaded = torch.cuda.Event(); uploaded.record(self.up_stream)
        cur.wait_event(uploaded)
        # uint8 -> float32 (/127.5 - 1, test.py:126-147) straight into the graph's static inputs (or fresh tensors on the eager path)
        x = {}
        for k, d in self.stage[slot].items():
            dst = self.graphed.static_in[k] if self.graphed is not None else torch.empty(d.shape, dtype=torch.float32, device=self.device)
            x[k] = self.io.u8_to_f32(d, dst, normalize=not k.endswith('mask'))
        self.stage_free[slot] = torch.cuda.Event(); self.stage_free[slot].record(cur)
        _, finetune, _ = self.graphed.replay() if self.graphed is not None else run_generator(self.G, x)
        finetune = self.io.image_to_u8(finetune.contiguous(), reverse_channels=True)
        done = torch.cuda.Event(); done.record(cur)
        self.copy_stream.wait_event(done)
        with torch.cuda.stream(self.copy_stream):
            host = self.out_host[self.slot]
            host.copy_(finetune, non_blocking=True)
            finetune.record_stream(self.copy_stream)
            ev = torch.cuda.Event(); ev.record(self.copy_stream)
        prev, self.pending = self.pending, (ev, host)
        self.slot ^= 1
        if prev is not None:
            prev[0].synchronize()
        return prev[1] if prev is not None else None

    def flush(self):
        if self.pending is not None:
            self.pending[0].synchronize()
            host, self.pending = self.pending[1], None
            return host
        return None


TRAIN_DESC = ('PASTA-GAN++ 512px training iteration (training_loop_fullbody.py:603-650, loss_fullbody.py:115-330): phases Gboth, Dboth, '
              'D_parsingboth x2 (the reference lists D_parsing twice) = G forward/backward through D and D_parsing, D and D_parsing steps on '
              'generated + real batches with the R1 penalty (conv2d_gradfix double backward) EVERY iteration (lazy regularisation off), '
              'Adam, G_ema; GeneratorFull_v20 43.1 M + 2 x Discriminator (channel_base 32768, c_dim 512, fp16 blocks at >= 128 px as '
              'train.py:196); l1 10, mask 30, r1_gamma 10, vgg / contextual 0 (checkpoints not shipped), aug=noaug')


def make_train_inputs_u8(batch, seed):
    """what the data loader delivers per iteration (training_loop_fullbody.py:540-590): uint8 host tensors"""
    d = make_generator_inputs_u8(batch, seed)
    g = torch.Generator().manual_seed(seed + 7)
    band = torch.zeros(1, 1, 1, 512, dtype=torch.bool); band[..., 96:416] = True
    real = torch.randint(0, 256, (batch, 3, 512, 512), generator=g, dtype=torch.uint8)
    d['real_img'] = torch.where(band, real, torch.full_like(real, 255))
    d['gt_parsing'] = torch.randint(0, 7, (batch, 1, 512, 512), generator=g, dtype=torch.uint8)
    return d


def train_inputs_to_device(u8, device):
    x = to_device_f32({k: v for k, v in u8.items() if k != 'gt_parsing'}, device)
    return dict(real_img=x['real_img'], style_input=x['c'], retain=x['retain'], pose=x['pose'], denorm_upper_input=x['denorm_upper'],
                denorm_lower_input=x['denorm_lower'], denorm_upper_mask=x['denorm_upper_mask'], denorm_lower_mask=x['denorm_lower_mask'],
                gt_parsing=u8['gt_parsing'].to(device, non_blocking=True).float())


def train_leg(steps, warmup, batch, precision, device, rank, world, fp16_res=3, dump_dir=None):
    """BASELINE configs[4]: the G + D + D_parsing training iteration with R1, data-parallel (DDP gradient all-reduce over NCCL when
    world > 1).  Returns the per-rank measurement dict (times already max-reduced over ranks).  With `dump_dir`, rank 0 writes the
    statistics the last timed iteration returned there (dump_outputs)."""
    import torch.distributed as dist
    ts = importlib.import_module('pgpp_b200.training.training_step')
    cg = importlib.import_module('pgpp_b200.torch_utils.ops.conv2d_gradfix')
    custom_ops = importlib.import_module('pgpp_b200.torch_utils.custom_ops')
    cg.fp32_precision = precision
    torch.manual_seed(0)
    G, D, DP = ts.build_networks(device, num_fp16_res=fp16_res)
    step = ts.TrainingStep(G, D, DP, device, batch_size=batch * world)
    host = {k: v.pin_memory() for k, v in make_train_inputs_u8(batch, 200 + rank).items()}
    data = train_inputs_to_device(host, device)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, n):
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        barrier()
        t = torch.tensor([a.elapsed_time(b)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0]) / n

    for _ in range(max(warmup, 3)):
        step(data)
    torch.cuda.reset_peak_memory_stats(device)
    l0 = custom_ops.launch_count()
    last = {}
    ms = timed(lambda: last.update(step(data)), steps)
    launches = (custom_ops.launch_count() - l0) // steps
    if dump_dir is not None and rank == 0:
        dump_outputs(dump_dir, last)
    # per-phase split on rank 0 (CUDA events around each phase of one more iteration)
    phase_ms = {}
    for ph in dict.fromkeys(p['name'] for p in step.phases):
        phase_ms[ph] = timed(lambda: step(data, phases=[ph]), 2)
    # end to end: uint8 pinned-host batch in, loss scalar back, every iteration
    def e2e_step():
        d = train_inputs_to_device(host, device)
        st = step(d)
        return float(st['Loss/scores/real'].item())
    e2e_step()
    e2e_ms = timed(e2e_step, steps)
    # the exchange step alone: the same iteration on the same networks WITHOUT the DistributedDataParallel wrappers (no bucketing, no
    # all-reduce) -> compute-only time per rank; ms - compute-only = exposed all-reduce.  (DDP.no_sync cannot be used for this: the loss
    # runs G_style_encoding under a synchronising forward in phases that never back-propagate into it, as the reference does, and a
    # no_sync forward after such an unfinished reduction trips the reducer.)  Measured last: the replicas' weights diverge from here on.
    nosync_ms = None
    if world > 1:
        import gc
        step.loss = step.ddp_modules = None     # drop the DDP wrappers: their reducers take their autograd hooks off the parameters
        gc.collect()
        local = ts.TrainingStep(G, D, DP, device, batch_size=batch * world, distributed=False)
        local(data)
        nosync_ms = timed(lambda: local(data), steps)
    grad_bytes = {n: 4 * sum(p.numel() for p in m.parameters()) for n, m in (('G', G), ('D', D), ('D_parsing', DP))}
    return {'ms_per_step': ms, 'images_per_sec': batch * world / (ms * 1e-3), 'e2e_ms_per_step': e2e_ms,
            'e2e_images_per_sec': batch * world / (e2e_ms * 1e-3), 'h2d_bytes_per_step': sum(v.numel() for v in host.values()),
            'd2h_bytes_per_step': 4, 'gpu_launches_per_step': launches, 'phase_ms': phase_ms,
            'no_allreduce_ms_per_step': nosync_ms, 'exposed_allreduce_ms': None if nosync_ms is None else ms - nosync_ms,
            'allreduce_bytes_per_step': grad_bytes['G'] + grad_bytes['D'] + 2 * grad_bytes['D_parsing'], 'grad_bytes': grad_bytes,
            'collective': f'DDP bucketed gradient all-reduce (NCCL, {world} ranks) per phase' if world > 1 else 'none (1 GPU)',
            'peak_mem_gb': torch.cuda.max_memory_allocated(device) / 2 ** 30, 'batch_per_gpu': batch, 'global_batch': batch * world,
            'precision': precision, 'fp16_blocks': fp16_res}


def run_train(args):
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1)); local = int(os.environ.get('LOCAL_RANK', 0))
    assert torch.cuda.is_available(), 'bench.py needs a GPU'
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        torch.distributed.init_process_group('nccl', device_id=device)
    from __graft_entry__ import load_pkg
    load_pkg()
    importlib.import_module('pgpp_b200.torch_utils.custom_ops').load_library()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    batch = args.batch if args.batch != 32 else 8
    with ClockSampler(local) as clocks:
        r = train_leg(args.steps, args.warmup, batch, args.precision, device, rank, world, fp16_res=args.fp16_res, dump_dir=args.dump_outputs)
    if rank == 0:
        line = {'metric': 'training_512px_images_per_sec', 'value': r['images_per_sec'], 'unit': 'images/s', 'n_gpus': world,
                'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': r['ms_per_step'], 'higher_is_better': True,
                'scaling': 'weak', 'vs_baseline': None,
                'dtype': f'f32 tensors ({args.precision} split tcgen05 MMAs); D blocks >= 128 px in fp16 (native f16 MMA)' if args.fp16_res else
                         f'f32 tensors ({args.precision} split tcgen05 MMAs)',
                'data': 'synthetic',
                'config': {'workload': TRAIN_DESC, 'batch_per_gpu': batch, 'global_batch': batch * world, 'resolution': RES,
                           'parallelism': f'data-parallel x{world}, DDP gradient all-reduce over NCCL', 'precision': args.precision,
                           'l2': 'per-step working set (tens of GB of saved activations) exceeds the 126 MB L2; no flush needed'},
                'clocks': clocks.summary(), 'gpu_launches': r['gpu_launches_per_step'] * args.steps,
                'e2e': {'value': r['e2e_images_per_sec'], 'unit': 'images/s', 'h2d_bytes_per_step': r['h2d_bytes_per_step'],
                        'd2h_bytes_per_step': r['d2h_bytes_per_step'],
                        'note': 'uint8 pinned-host batch in (+ on-device /127.5-1), one loss scalar read back, every iteration'},
                'train': r}
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def run_ours(args):
    rank = int(os.environ.get('RANK', 0)); world = int(os.environ.get('WORLD_SIZE', 1)); local = int(os.environ.get('LOCAL_RANK', 0))
    assert torch.cuda.is_available(), 'bench.py needs a GPU (there is no CPU fallback; use --impl reference for the CPU ref path)'
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=device)
    from __graft_entry__ import load_pkg
    load_pkg()
    custom_ops = importlib.import_module('pgpp_b200.torch_utils.custom_ops')
    cg = importlib.import_module('pgpp_b200.torch_utils.ops.conv2d_gradfix')
    custom_ops.load_library()
    cg.fp32_precision = args.precision
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False

    batch = args.batch
    gen_mode = args.workload == 'generator'
    gen = importlib.import_module('pgpp_b200.training.generator')
    if gen_mode:
        net = build_generator(device)
        host_u8 = {k: v.pin_memory() for k, v in make_generator_inputs_u8(batch, 100 + rank).items()}
        dev_in = to_device_f32(host_u8, device)

        def step_eager():
            return run_generator(net, dev_in)
        step = step_eager
    else:
        net = build_chain(device)
        cat = make_cat_feats(net, batch, device)
        ws_h, pose_h = make_inputs(net, batch, 100 + rank, pin=True)
        ws_d, pose_d = ws_h.to(device), pose_h.to(device)

        def step_eager():
            with torch.no_grad():
                return net(ws_d, pose_d, cat, noise_mode='const')
        step = step_eager

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ----
    # The public inference entry for fixed shapes is `GraphedGenerator`: the whole forward (about 400 launches) captured once into a CUDA
    # graph and replayed - same kernels, same order, bit-identical output, no per-launch host work.  `--no-graph` times eager launches.
    eager_step_ms = None
    graphed = None
    launches_per_step = None
    if gen_mode and not args.no_graph:
        for _ in range(3):
            step_eager()
        barrier()
        l0 = custom_ops.launch_count()
        step_eager()
        launches_per_step = custom_ops.launch_count() - l0         # graph replays do not pass through the C ABI: count one eager pass
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); a0.record()
        for _ in range(args.steps):
            step_eager()
        a1.record(); barrier()
        eager_step_ms = a0.elapsed_time(a1) / args.steps
        graphed = gen.GraphedGenerator(net, dev_in)
        step = graphed.replay
    for _ in range(max(args.warmup, 3)):
        out = step()
    barrier()
    launches0 = custom_ops.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        barrier()
        e0.record()
        for _ in range(args.steps):
            out = step()
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1)
    launches = custom_ops.launch_count() - launches0
    if graphed is not None:
        launches = launches_per_step * args.steps
    if args.dump_outputs and rank == 0:
        names = ('img', 'finetune_img', 'pred_parsing') if gen_mode else ('img', 'pred_parsing', 'tex')
        dump_outputs(args.dump_outputs, dict(zip(names, out)))

    # ---- end to end through the pipeline API (pinned host in, image back to host) ----
    if gen_mode:
        pipe = GeneratorPipeline(net, batch, device, graphed=graphed)
        call = lambda: pipe(host_u8)
        h2d = sum(v.numel() for v in host_u8.values())
    else:
        pipe = SynthesisPipeline(net, cat, batch, device)
        call = lambda: pipe(ws_h, pose_h)
        h2d = ws_h.numel() * 4 + pose_h.numel() * 4
    for _ in range(3):
        call()
    pipe.flush()
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for _ in range(args.steps):
        host_img = call()
    host_img = pipe.flush()
    f1.record()
    barrier()
    e2e_ms = f0.elapsed_time(f1)        # device clock; f1 is recorded after the last read-back completed
    d2h = batch * 3 * RES * RES * (1 if gen_mode else 4)

    # ---- max over ranks ----
    times = torch.tensor([ms, e2e_ms, eager_step_ms or 0.0], device=device, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(times, op=torch.distributed.ReduceOp.MAX)
    ms, e2e_ms = float(times[0]), float(times[1])
    if eager_step_ms is not None:
        eager_step_ms = float(times[2])

    # ---- bf16 mode (reported separately, north star): same step with single-product bf16 MMAs ----
    cg.fp32_precision = 'bf16'
    if graphed is not None:
        del pipe
        graphed = None
        torch.cuda.empty_cache()
        graphed_bf16 = gen.GraphedGenerator(net, dev_in)          # the captured launches carry the precision they were captured with
        step = graphed_bf16.replay
    for _ in range(3):
        step()
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(args.steps):
        step()
    g1.record()
    barrier()
    bf16_ms = g0.elapsed_time(g1)
    times = torch.tensor([bf16_ms], device=device, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(times, op=torch.distributed.ReduceOp.MAX)
    bf16_ms = float(times[0])
    if gen_mode and not args.no_graph:
        step = step_eager
        graphed_bf16 = None
        torch.cuda.empty_cache()

    # ---- BASELINE configs[4] beside the headline: a few training iterations (G + D + D_parsing with R1, DDP all-reduce when world > 1) ----
    train = None
    if gen_mode and args.train_steps > 0:
        try:
            # 5 untimed iterations first: the caching allocator still re-shapes its pools after the generator legs (73 GB peak here)
            train = train_leg(args.train_steps, 5, 8, args.precision, device, rank, world, fp16_res=args.fp16_res)
        except Exception as e:      # noqa: BLE001 - the extra measurement must never break the contract line
            train = {'error': f'{type(e).__name__}: {str(e)[:300]}'}
        cg.fp32_precision = args.precision
        torch.cuda.empty_cache()

    if rank == 0:
        pk = peaks()

        def traced(precision):
            """per-launch CUDA-event times of every igemm launch of one step (after one untimed traced pass)"""
            cg.fp32_precision = precision
            for _ in range(2):
                cg.trace = []
                step(); torch.cuda.synchronize()
            tr, cg.trace = cg.trace, None
            return [(t[0], t[1], t[2].elapsed_time(t[3])) for t in tr]

        def roofline(tr, step_ms, precision):
            flops = sum(t[1] for t in tr); kms = sum(t[2] for t in tr)
            # dominant launch shape = largest total time
            by = {}
            for name, fl, ms_ in tr:
                e = by.setdefault(name, [0.0, 0.0, 0]); e[0] += fl; e[1] += ms_; e[2] += 1
            top_name, (tfl, tms, tcnt) = max(by.items(), key=lambda kv: kv[1][1])
            achieved = tfl / (tms * 1e-3) / 1e12
            traffic = None
            # DRAM bytes of that launch shape from a committed ncu --set full capture (newest round first); the key is the
            # launch label without its operand-format suffix
            shape_key = ' '.join(top_name.split(' ')[:6])
            for tfile in ('r02_traffic.json', 'r01_traffic.json'):
                tpath = os.path.join(ROOT, 'profiles', tfile)
                if traffic is None and os.path.isfile(tpath):
                    traffic = json.load(open(tpath)).get(shape_key)
            return {'bound': 'tensor', 'kernel': 'pgpp::igemm_kernel', 'launch': top_name, 'launches_per_step': tcnt,
                    'achieved': achieved, 'peak': pk['tflops'], 'unit': 'TFLOP/s', 'frac': achieved / pk['tflops'], 'traffic': traffic,
                    'peak_source': pk['source'], 'avg_launch_ms': tms / tcnt, 'algorithmic_flops_per_launch': tfl / tcnt,
                    'mma_products_per_flop': {'bf16': 1, 'bf16x2': 3, 'bf16x3': 6}[precision],
                    'all_igemm_launches': {'achieved': flops / (kms * 1e-3) / 1e12, 'frac': flops / (kms * 1e-3) / 1e12 / pk['tflops'],
                                           'share_of_step': kms / step_ms, 'algorithmic_flops_per_step': flops, 'launches': len(tr)},
                    'top_launches': [{'launch': t[0], 'ms': t[2], 'tflops': t[1] / t[2] / 1e9} for t in sorted(tr, key=lambda t: -t[2])[:3]]}

        roof = roofline(traced(args.precision), ms / args.steps, args.precision)
        roof_bf16 = roofline(traced('bf16'), bf16_ms / args.steps, 'bf16')
        cg.fp32_precision = args.precision
        # parity of this very step against the CPU oracle on a bounded sample (batch 1), reported with the number
        parity = parity_bf16 = None
        cpu = None
        if not args.skip_cpu and gen_mode:
            from oracle import ref_generator
            sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
            one = {k: v[:1] for k, v in dev_in.items()}
            cpu_in = {k: v.cpu() for k, v in one.items()}
            rel = lambda a, b: float((a.cpu().double() - b.double()).norm() / b.double().norm())
            gt = torch.randint(0, 7, (1, 1, RES, RES), generator=torch.Generator().manual_seed(5)).float()
            cores = host_threads()
            torch.set_num_threads(cores)
            with torch.no_grad():
                # parity with gt_parsing fixed (no discrete decision depends on rounding, SURVEY section 7)
                t0 = time.perf_counter()
                r_img, r_fin, r_par = ref_generator.generator(sd, cpu_in['c'], cpu_in['retain'], cpu_in['pose'], cpu_in['denorm_upper'],
                                                              cpu_in['denorm_lower'], cpu_in['denorm_upper_mask'], cpu_in['denorm_lower_mask'], gt)
                t_first = time.perf_counter() - t0
                g_img, g_fin, g_par = run_generator(net, one, gt_parsing=gt.to(device))
                parity = {'img_rel_l2': rel(g_img, r_img), 'finetune_rel_l2': rel(g_fin, r_fin), 'parsing_rel_l2': rel(g_par, r_par),
                          'finetune_max_abs': float((g_fin.cpu() - r_fin).abs().max()), 'finetune_abs_scale': float(r_fin.abs().max())}
                cg.fp32_precision = 'bf16'
                b_img, b_fin, b_par = run_generator(net, one, gt_parsing=gt.to(device))
                cg.fp32_precision = args.precision
                parity_bf16 = {'img_rel_l2': rel(b_img, r_img), 'finetune_rel_l2': rel(b_fin, r_fin), 'parsing_rel_l2': rel(b_par, r_par),
                               'finetune_max_abs': float((b_fin.cpu() - r_fin).abs().max())}
                ctimes = [t_first]
                for _ in range(2):
                    t0 = time.perf_counter()
                    ref_generator.generator(sd, cpu_in['c'], cpu_in['retain'], cpu_in['pose'], cpu_in['denorm_upper'], cpu_in['denorm_lower'],
                                            cpu_in['denorm_upper_mask'], cpu_in['denorm_lower_mask'], None)
                    ctimes.append(time.perf_counter() - t0)
            cpu = {'value': 1.0 / min(ctimes), 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                   'sample': f'best of 3 x batch 1 through oracle/ref_generator.py (torch CPU ops, {cores} threads; {sum(ctimes):.1f} s total)'}
        elif not args.skip_cpu:
            from oracle import ref_chain
            sd = {k: v.detach().cpu() for k, v in net.state_dict().items()}
            cat1 = {k: v[:1] for k, v in cat.items()}
            rel = lambda a, b: float((a.cpu().double() - b.double()).norm() / b.double().norm())
            with torch.no_grad():
                r_img, r_par, r_tex = ref_chain.synthesis_chain(sd, ws_h[:1], pose_h[:1], {k: v.cpu() for k, v in cat1.items()}, img_resolution=RES)
                g_img, g_par, g_tex = net(ws_d[:1], pose_d[:1], cat1, noise_mode='const')
                parity = {'img_rel_l2': rel(g_img, r_img), 'parsing_rel_l2': rel(g_par, r_par), 'texture_rel_l2': rel(g_tex, r_tex),
                          'img_max_abs': float((g_img.cpu() - r_img).abs().max()), 'img_abs_scale': float(r_img.abs().max())}
                cg.fp32_precision = 'bf16'
                b_img, b_par, b_tex = net(ws_d[:1], pose_d[:1], cat1, noise_mode='const')
                cg.fp32_precision = args.precision
                parity_bf16 = {'img_rel_l2': rel(b_img, r_img), 'parsing_rel_l2': rel(b_par, r_par), 'texture_rel_l2': rel(b_tex, r_tex),
                               'img_max_abs': float((b_img.cpu() - r_img).abs().max())}
            cores = host_threads()
            rate, ctimes = cpu_reference_rate(sd, net.num_ws, net.channels[8], 1, 3, threads=cores)
            cpu = {'value': rate, 'unit': 'images/s', 'cores': cores, 'kind': 'port',
                   'sample': f'best of 3 x batch 1 through oracle/ref_chain.py (torch CPU ops, {cores} threads; {sum(ctimes):.1f} s total)'}
        batch1 = None
        if gen_mode:
            # BASELINE configs[0] shape (batch 1): eager launches vs CUDA-graph replay of the same forward
            try:
                gen = importlib.import_module('pgpp_b200.training.generator')
                one = {k: v[:1].contiguous() for k, v in dev_in.items()}
                for _ in range(3):
                    run_generator(net, one)
                def lat(fn, iters=20):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize(); a.record()
                    for _ in range(iters):
                        fn()
                    b.record(); torch.cuda.synchronize()
                    return a.elapsed_time(b) / iters
                eager_ms = lat(lambda: run_generator(net, one))
                gg = gen.GraphedGenerator(net, one)
                graph_ms = lat(lambda: gg(one))
                batch1 = {'eager_ms': eager_ms, 'cuda_graph_ms': graph_ms, 'images_per_sec_cuda_graph': 1e3 / graph_ms,
                          'note': 'batch-1 latency of the full generator (fp32-parity mode); graph replay is bit-identical to eager'}
            except Exception as e:      # noqa: BLE001 - the extra measurement must never break the contract line
                batch1 = {'error': f'{type(e).__name__}: {str(e)[:200]}'}
        # BASELINE configs[3] / the metric's "modconv TFLOPS and upfirdn2d GB/s": the op sweep of this very build (tools/op_bench.py)
        ops = None
        if gen_mode and not args.no_ops:
            try:
                del net
                torch.cuda.empty_cache()
                spec = importlib.util.spec_from_file_location('pgpp_op_bench', os.path.join(ROOT, 'tools', 'op_bench.py'))
                op_bench = importlib.util.module_from_spec(spec)
                spec.loader.exec_module(op_bench)
                ops = op_bench.run_ops(device=device, n=32)
            except Exception as e:      # noqa: BLE001 - the extra measurement must never break the contract line
                ops = {'error': f'{type(e).__name__}: {str(e)[:300]}'}
            cg.fp32_precision = args.precision
        imgs = batch * world * args.steps
        line = {
            'metric': 'generator_512px_images_per_sec' if gen_mode else 'synthesis_hot_path_images_per_sec',
            'value': imgs / (ms * 1e-3), 'unit': 'images/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'f32 tensors; bf16x2-split tcgen05 MMAs (3 bf16 products per multiply), fp32 accumulation' if args.precision != 'bf16'
                     else 'bf16 MMA, fp32 accumulate, f32 tensors',
            'data': 'synthetic',
            'config': {'workload': GEN_DESC if gen_mode else CHAIN_DESC,
                       'batch_per_gpu': batch, 'global_batch': batch * world, 'resolution': RES, 'precision': args.precision,
                       'parallelism': f'batch-sharded x{world}, no collective',
                       'launch': ('CUDA-graph replay of the whole forward (GraphedGenerator, the inference entry for fixed shapes; same kernels as the '
                                  'eager pass, bit-identical output)') if eager_step_ms is not None else 'eager launches',
                       'l2': 'per-step working set (several GB of activations) exceeds the 126 MB L2; no flush needed'},
            'clocks': clocks.summary(),
            'gpu_launches': launches,
            'eager': None if eager_step_ms is None else {'ms_per_step': eager_step_ms, 'value': imgs / args.steps / (eager_step_ms * 1e-3), 'unit': 'images/s',
                                                     'note': 'the same step issued launch by launch through Python / ctypes (device-resident inputs)'},
            'e2e': {'value': imgs / (e2e_ms * 1e-3), 'unit': 'images/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'note': ('uint8 pinned-host try-on inputs in (+ on-device /127.5-1, test.py:126-147), uint8 BGR try-on image read back (test.py:162-166); '
                             'upload of batch i+1 and read-back of batch i-1 overlap the compute of batch i (separate streams, double-buffered staging)') if gen_mode else
                            'pinned-host ws + pose features in, fp32 image read back; copy of batch i overlaps compute of i+1'},
            'roofline': roof,
            'cpu_baseline': cpu,
            'parity_vs_cpu_oracle': parity,
            'batch1': batch1,
            'ops': ops,
            'train': train,
            'bf16_mode': {'value': imgs / (bf16_ms * 1e-3), 'unit': 'images/s', 'ms_per_step': bf16_ms / args.steps, 'roofline': roof_bf16,
                          'parity_vs_cpu_oracle': parity_bf16,
                          'note': 'same step with single-product bf16 MMAs (per-layer rel error ~3e-3); reported separately, not the headline'},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=32, help='images per GPU per step')
    ap.add_argument('--precision', default='bf16x2', choices=['bf16', 'bf16x2', 'bf16x3'])
    ap.add_argument('--workload', default='generator', choices=['generator', 'chain', 'train'],
                    help='generator: the full GeneratorFull_v20 forward (BASELINE configs[1]); chain: the modulated-conv synthesis chain only; '
                         'train: the G + D training iteration with R1 under DDP (BASELINE configs[4], batch 8 per GPU)')
    ap.add_argument('--train-steps', type=int, default=3, help='generator workload: also time this many training iterations (0 = skip)')
    ap.add_argument('--fp16-res', type=int, default=3, help='train workload: number of highest-resolution D blocks in fp16 (train.py:196)')
    ap.add_argument('--skip-cpu', action='store_true', help='skip the CPU baseline / parity leg')
    ap.add_argument('--no-graph', action='store_true', help='generator workload: time eager launches instead of CUDA-graph replay (GraphedGenerator)')
    ap.add_argument('--no-ops', action='store_true', help='generator workload: skip the op microbench sweep (the `ops` key, BASELINE configs[3])')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned as DIR/<name>.npy (float32 / float64; at most 64 MB in all, a fixed '
                         'seeded choice of batch rows when the outputs are larger)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of this package\'s kernels (--impl ours)')
    if args.impl == 'reference':
        run_reference(args)
    elif args.workload == 'train':
        run_train(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
