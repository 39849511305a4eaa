"""MobileNetV3 large / small and MobileNetV2 (cocokp heads, 641x641) on the compiled forward, next to stock
PyTorch / cuDNN on the same Shell.  Prints one JSON document (and writes it to --out):
  - images/s at 64 and 8 images per batch: forward only, and forward + decode of planted poses
    (Predictor.decode_fields_override, as bench.py does);
  - per-op-kind milliseconds of one 64-image forward (CompiledNet.forward_timed) with the algorithmic bytes and the
    achieved TB/s against MEASURED_PEAKS.json (or the data-sheet 7.7 TB/s when that file is absent);
  - PyTorch eval forward of the same architecture: bf16 channels_last and fp32 (TF32 off);
  - the card's name and power limit (nvidia-smi, read-only query).
Random-init weights (heads calibrated as bench.py does); torchvision is called with weights=None."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]

from openpifpaf_b200 import constants, network, predictor as pred_mod, synth   # noqa: E402
import mobilenet_oracle                                                         # noqa: E402

KIND = {0: 'input_conv', 1: 'gemm', 2: 'depthwise', 3: 'fused_dw_gemm', 4: 'squeeze_excitation'}


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return out[0] if out else 'unknown'
    except (OSError, subprocess.SubprocessError):
        return 'unknown'


def peak_hbm_gbs():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)['hbm_gbs']), 'MEASURED_PEAKS.json'
    return 7700.0, 'data sheet (not measured)'


def time_ms(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def bench_one(name, size, batches, steps, warmup):
    res = {}
    plan = network.random_mobilenet_plan(name, seed=0, confidence_bias=-2.5)
    network.calibrate_random_heads(plan, size=min(size, 321), batch=2)
    stride = plan['heads'][0]['stride']
    side = (size - 1) // stride + 1
    for B in batches:
        net = network.CompiledNet(plan, size, size, B)
        x = torch.randn(B, 3, size, size, generator=torch.Generator().manual_seed(B)).cuda()
        fwd = time_ms(lambda: net.forward(x), steps, warmup)
        pred = pred_mod.Predictor(net, constants.COCO_N_KEYPOINTS, constants.COCO_PERSON_SKELETON)
        items = [synth.make_fields('cocokp', side, side, None, 77 * 1000 + b) for b in range(B)]
        cif = torch.from_numpy(np.stack([it['cif'] for it in items])).cuda()
        caf = torch.from_numpy(np.stack([it['caf'] for it in items])).cuda()
        pred.decode_fields_override = (cif, stride, caf, stride)

        def step():
            pred.batch_device(x)
            pred.join()
        e2e = time_ms(step, steps, warmup)
        res[f'b{B}'] = {'forward_ms': round(fwd, 4), 'forward_images_per_s': round(B / fwd * 1e3, 1),
                        'forward_decode_ms': round(e2e, 4), 'forward_decode_images_per_s': round(B / e2e * 1e3, 1),
                        'planted_people': int(sum(it['n_planted'] for it in items))}
        if B == max(batches):
            ms, kind, flops, nbytes = net.forward_timed(x)
            ms, kind, flops, nbytes = net.forward_timed(x)
            peak, src = peak_hbm_gbs()
            split = {}
            for k in sorted(set(int(v) for v in kind)):
                sel = kind == k
                t, b = float(ms[sel].sum()), float(nbytes[sel].sum())
                split[KIND[k]] = {'ms': round(t, 4), 'launches': int(sel.sum()), 'algorithmic_GB': round(b / 1e9, 4),
                                  'TB_per_s': round(b / t / 1e9, 3) if t > 0 else None,
                                  'share_of_hbm_peak': round(b / t / 1e6 / peak, 3) if t > 0 else None}
            res['per_op_kind'] = {'batch': B, 'sum_ms': round(float(ms.sum()), 4), 'hbm_peak_gbs': peak,
                                  'hbm_peak_source': src, 'kinds': split}
        pred.close()
    # stock PyTorch on the oracle Shell (same architecture, torchvision modules)
    shell = mobilenet_oracle.make_shell(name, seed=0).cuda()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.benchmark = True
    for B in batches:
        x = torch.randn(B, 3, size, size, generator=torch.Generator().manual_seed(B)).cuda()
        with torch.no_grad():
            f32 = time_ms(lambda: shell(x), max(steps // 2, 3), warmup)
            sb = shell.to(torch.bfloat16).to(memory_format=torch.channels_last)
            xb = x.to(torch.bfloat16).to(memory_format=torch.channels_last)
            bf = time_ms(lambda: sb(xb), max(steps // 2, 3), warmup)
            shell = sb.float().to(memory_format=torch.contiguous_format)
        res[f'b{B}']['pytorch_fp32_images_per_s'] = round(B / f32 * 1e3, 1)
        res[f'b{B}']['pytorch_bf16_channels_last_images_per_s'] = round(B / bf * 1e3, 1)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--size', type=int, default=641)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--batches', default='64,8')
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    batches = [int(v) for v in args.batches.split(',')]
    doc = {'card': card(), 'size': args.size, 'steps': args.steps, 'warmup': args.warmup,
           'weights': 'random init, heads calibrated; planted poses for the decode', 'results': {}}
    for name in mobilenet_oracle.MOBILENETS:
        doc['results'][name] = bench_one(name, args.size, batches, args.steps, args.warmup)
        print(name, json.dumps(doc['results'][name]), flush=True)
    text = json.dumps(doc, indent=1)
    print(text)
    if args.out:
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
