"""fp8 (e4m3) against bf16x2 / bf16 on the dominant implicit-GEMM shapes of the generator, batch 32, one box, one run.

Per layer, shape and precision: the convolution alone (operands packed once, outside the timed window), 20 launches captured in a CUDA
graph (no host work in the window), 5 repeats of 10 replays each (200 launches) timed with CUDA events; median and spread of the repeats,
algorithmic TFLOP/s = 2 N O I kh kw H W / median time; and the fp8 output's rel-L2 / max-abs against bf16x2 on the same inputs.  The
SPADE row runs the real gamma|beta launch (instance-norm modulation in the epilogue, bf16 operand-format output).
Generator: GeneratorFull_v20 at batch 32 under CUDA-graph replay (GraphedGenerator) in each precision, 5 repeats of 10 replays; the fp8
images against bf16x2 on the same inputs.  The card name and power limit are read in the same run, the SM clock is sampled by nvidia-smi
DURING the timed windows (bench.ClockSampler).  The working sets exceed the 126 MB L2 except for the 512-channel layer.

    python tools/fp8_bench.py [--out profiles/r03_fp8_bench.txt]
"""
import argparse
import importlib
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as entry  # noqa: E402
import bench  # noqa: E402

entry.load_pkg()
cg = importlib.import_module('pgpp_b200.torch_utils.ops.conv2d_gradfix')
gen = importlib.import_module('pgpp_b200.training.generator')

# (label, in channels, out channels, kernel, resolution): 64->64 @512^2, 128->128 @256^2, 512->512 @32^2, the 128->256 SPADE gamma|beta GEMM @256^2
SHAPES = [('64->64 k3 @512', 64, 64, 3, 512), ('128->128 k3 @256', 128, 128, 3, 256), ('512->512 k3 @32', 512, 512, 3, 32),
          ('128->256 k3 @256 (SPADE gamma|beta)', 128, 256, 3, 256)]
MODES = ('bf16x2', 'bf16', 'fp8')


def smi(query):
    try:
        return subprocess.run(['nvidia-smi', f'--query-gpu={query}', '--format=csv,noheader', '-i', '0'], capture_output=True, text=True,
                              timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return f'unavailable ({e})'


def time_replays(fn, per_graph, replays=10, repeats=5, clocks=None):
    """ms per call of fn (captured per_graph times into one CUDA graph): (median, min, max) over the repeats"""
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(per_graph):
            out = fn()
    g.replay()
    torch.cuda.synchronize()
    ts = []
    with bench.ClockSampler(0) as cs:
        for _ in range(repeats):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(replays):
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / (replays * per_graph))
    if clocks is not None:
        clocks.extend(cs.lines)
    ts.sort()
    return (ts[len(ts) // 2], ts[0], ts[-1]), out


def clock_summary(lines):
    sm = []
    for l in lines:
        try:
            sm.append(float(l.split(',')[0]))
        except ValueError:
            pass
    return f'{min(sm):.0f}-{max(sm):.0f} MHz over {len(sm)} samples' if sm else 'not sampled'


def layer_rows(label, flops, run, lines, clocks):
    outs = {}
    for mode in MODES:
        t, y = run(mode, clocks)
        outs[mode] = y.to(torch.float32) if not isinstance(y, cg.PackedAct) else y.data[0].to(torch.float32)
        extra = ''
        if mode == 'fp8':
            ref = outs['bf16x2'].double()
            d = outs['fp8'].double() - ref
            extra = f'rel-L2 {float(d.norm() / ref.norm()):.3e}  max-abs {float(d.abs().max()):.3e}  (max |ref| {float(ref.abs().max()):.3e})'
        lines.append(f'{label:44s} {mode:7s} {t[0]:8.4f} [{t[1]:.4f}-{t[2]:.4f}] {flops / t[0] / 1e9:8.1f}  {extra}')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--batch', type=int, default=32)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'fp8_bench measures on the GPU'
    cg._init()
    lines = [f'card: {smi("name,power.limit,clocks.max.sm")}  (name, power limit, max SM clock)',
             f'batch {args.batch}; ms per launch: median [min-max] of 5 repeats of 200 graph-replayed launches']
    lines.append(f'{"layer":44s} {"mode":7s} {"ms":>8s} {"spread":>17s} {"TFLOP/s":>8s}  fp8 vs bf16x2')
    clocks = []
    g = torch.Generator(device='cuda').manual_seed(0)
    n = args.batch
    for label, ic, oc, k, res in SHAPES:
        x = torch.randn(n, ic, res, res, device='cuda', generator=g)
        w = torch.randn(oc, ic, k, k, device='cuda', generator=g) / (ic * k * k) ** 0.5
        flops = 2.0 * n * oc * ic * k * k * res * res
        spade = label.startswith('128->256')
        if spade:       # the SPADE gamma|beta launch: x_norm (C = 128 channels), its statistics, the modulated operand-format output
            xs = torch.randn(n, oc // 2, res, res, device='cuda', generator=g)
            var, mean = torch.var_mean(xs, dim=(2, 3), unbiased=False)
            rstd = (var + 1e-5).rsqrt()

        def run(mode, clocks, x=x, w=w, ic=ic, oc=oc, k=k, spade=spade):
            cg.fp32_precision = mode
            parts = cg._PRODUCTS[mode][1]
            pw = cg.pack_weights_native(w, k, k, parts, k // 2, k // 2, e4m3=mode == 'fp8')
            with torch.no_grad():
                xp = cg.pack_operand(x, mode)
                if spade:
                    out = cg.PackedAct(cg.PackedAct.empty(n, res, res, oc // 2, parts, x.device), oc // 2)
                    fn = lambda: cg.igemm_conv(xp, pw, precision=mode, out_packed=out, spade=(xs, mean, rstd, 1.0))
                else:
                    fn = lambda: cg.igemm_conv(xp, pw, precision=mode, out_dtype=torch.float32)
                return time_replays(fn, 20, clocks=clocks)
        layer_rows(label + (' SPADE launch' if spade else ''), flops, run, lines, clocks)
        del x
        torch.cuda.empty_cache()
    # the generator step under graph replay
    net = bench.build_generator(torch.device('cuda:0'))
    dev_in = bench.to_device_f32(bench.make_generator_inputs_u8(n, 100), torch.device('cuda:0'))
    imgs = {}
    for mode in MODES:
        cg.fp32_precision = mode
        with torch.no_grad():
            gg = gen.GraphedGenerator(net, dev_in)
            ts = []
            for _ in range(3):
                gg.replay()
            torch.cuda.synchronize()
            with bench.ClockSampler(0) as cs:
                for _ in range(5):
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(10):
                        out = gg.replay()
                    e1.record()
                    torch.cuda.synchronize()
                    ts.append(e0.elapsed_time(e1) / 10)
            clocks.extend(cs.lines)
            imgs[mode] = [t.detach().double().clone() for t in out]
        ts.sort()
        extra = ''
        if mode == 'fp8':
            parts_ = []
            for name, a, b in zip(('img', 'finetune', 'parsing'), imgs['fp8'], imgs['bf16x2']):
                d = a - b
                parts_.append(f'{name} rel-L2 {float(d.norm() / b.norm()):.3e} max-abs {float(d.abs().max()):.3e} (max |ref| {float(b.abs().max()):.2f})')
            extra = '; '.join(parts_)
        lines.append(f'{"generator step, batch " + str(n) + ", graph replay":44s} {mode:7s} {ts[len(ts) // 2]:8.3f} [{ts[0]:.3f}-{ts[-1]:.3f}] '
                     f'{n * 1000.0 / ts[len(ts) // 2]:7.1f} img/s  {extra}')
        del gg
        torch.cuda.empty_cache()
    lines.append(f'SM clock sampled during the timed windows: {clock_summary(clocks)}')
    lines.append('dense FP8 data-sheet rate of one B200 (1,000 W): 4,500 TFLOP/s; BF16: 2,250 TFLOP/s - not reached here')
    text = '\n'.join(lines)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
