#!/usr/bin/env python
"""bench.py -- images/sec end-to-end (backbone + heads + CifCaf decode), shufflenetv2k16 641 px, total batch 64.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference --gpus N ...            # the reference's own CPU path on the host cores
  python bench.py ... --dump-outputs DIR                   # + what the last timed step computed, as DIR/*.npy

One "step" = one pass of the hot path over one batch of synthetic input (BASELINE.json config C0):
  images [64,3,641,641] f32 -> shufflenetv2k16 backbone + CIF/CAF heads -> batched CifCaf decode.
A random-init network emits no poses, so the decode inside every timed step runs on planted fields of the same
batch (Poisson(4)+1 people per image, SURVEY.md 8d) -- in both arms.
`value` : images/s, image batch resident in HBM (CUDA events on the launching stream, max over ranks).
`e2e`   : the same through Predictor.batches() with pinned HOST images: H2D + forward + decode + D2H per step.
--gpus N (under torchrun): the 64 images are sharded over the ranks, 64/N each, no data-path collective
(SURVEY.md 8d/8e) -> `scaling: "strong"`; `weak_scaling` reports 64 images per GPU beside it.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOTAL_BATCH = 64
SIZE = 641
METRIC = 'images/sec end-to-end (backbone+heads+decode) 641px bs64; decoder-only ms/img'

# BASELINE.json configs (SURVEY.md 8d).  C0 is the headline; the others are bounded extra measurements.
CONFIGS = {
    'C0': dict(base='shufflenetv2k16', workload='cocokp', size=641, batch=64, people=None),
    'C2': dict(base='shufflenetv2k16', workload='cocokp', size=641, batch=32, people=None),
    'C3': dict(base='shufflenetv2k30', workload='wholebody', size=641, batch=16, people=None),
    'C4': dict(base='resnet50', workload='cocokp', size=801, batch=8, people=None),      # 8 per GPU (x8 GPUs = 64)
    'C5': dict(base='shufflenetv2k16', workload='cocokp', size=641, batch=8, people=30),
}
ALGO_GFLOP_PER_IMAGE = {'C0': 73.2, 'C2': 73.2, 'C3': 266.6, 'C4': 417.9, 'C5': 73.2}     # SURVEY.md 8d


def workload_name(n_per_gpu, world):
    return (f'C0: shufflenetv2k16 cocokp(17kp/19caf) 641x641, total batch {TOTAL_BATCH} '
            f'({n_per_gpu} images per GPU x {world})')


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {'hbm_gbs': p['hbm_gbs'], 'bf16_tflops': p.get('bf16_tflops_sustained', p['bf16_tflops']),
                'source': 'measured (MEASURED_PEAKS.json, sustained)'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1400.0, 'source': 'fallback (B200_PROFILING.md)'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--id={self.gpu}', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '20'],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:       # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:       # noqa: BLE001
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.lines:
            parts = [p.strip() for p in line.split(',')]
            if len(parts) < 8:
                continue
            try:
                sm.append(float(parts[1]))
                smax = float(parts[2])
            except ValueError:
                continue
            for nm, v in zip(names, parts[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': smax,
                'reasons': sorted(reasons), 'samples': len(sm)}


def dist_setup():
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(value, world, device):
    if world > 1:
        import torch.distributed as dist
        t = torch.tensor([value], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return value


def measured_traffic(kernels, launches_per_step):
    """DRAM bytes per launch of the GEMM kernels (`kernels`: the names that together make up the launches of one step)
    from the committed ncu capture of this same command (profiles/), or None.  Only accepted if the capture holds a
    whole number of steps of their launches -- a capture of an older build (other kernel mix) is not quoted."""
    for name in ('r2_dram_traffic_bench_step.json', 'r1_dram_traffic_bench_step.json'):
        path = os.path.join(ROOT, 'profiles', name)
        try:
            table = json.load(open(path))['kernels']
        except (OSError, KeyError, ValueError):
            continue
        found = [table[k] for k in kernels if k in table]
        if name.startswith('r2') and len(found) != len(kernels):
            continue
        launches = sum(k['launches'] for k in found)
        if not found or launches % launches_per_step != 0 or (name.startswith('r1') and len(kernels) > 1):
            continue
        total = sum(k['dram_read_bytes'] + k['dram_write_bytes'] for k in found)
        return round(total / launches), f'profiles/{name} (ncu, one bs64 step)'
    return None, 'no ncu capture of this build committed'


# ----------------------------------------------------------------------------- workload construction
def make_plan(cfg, seed=0):
    from openpifpaf_b200 import network, synth
    K = synth.WORKLOADS[cfg['workload']][0]
    C = len(synth.skeleton_for(cfg['workload']))
    heads = ((K, 1, 1, 1), (C, 1, 2, 2))
    if cfg['base'].startswith('resnet'):
        return network.random_resnet_plan(cfg['base'], heads=heads, seed=seed, confidence_bias=-2.5)
    return network.random_plan(cfg['base'], heads=heads, seed=seed, confidence_bias=-2.5)


def planted_fields(cfg, n_images, first_image=0):
    """The planted decoder input of images [first_image, first_image + n_images) of the config's global batch."""
    from openpifpaf_b200 import synth
    h = w = (cfg['size'] - 1) // 16 + 1
    items = [synth.make_fields(cfg['workload'], h, w, cfg['people'], 77 * 1000 + first_image + b) for b in range(n_images)]
    return {'cif': np.stack([it['cif'] for it in items]), 'caf': np.stack([it['caf'] for it in items]),
            'n_planted': [it['n_planted'] for it in items]}


def build_predictor(cfg, batch, local, overlap, calibrate_size=None):
    """random-init weights; heads centred and rescaled on the bench resolution (~N(0,1) pre-activations with a
    sparse-confidence bias), compiled for `batch` images"""
    from openpifpaf_b200 import network, predictor as pred_mod, synth
    plan = make_plan(cfg)
    network.calibrate_random_heads(plan, device=local, size=calibrate_size or min(cfg['size'], 641), batch=2)
    net = network.CompiledNet(plan, cfg['size'], cfg['size'], batch, device=local)
    K = synth.WORKLOADS[cfg['workload']][0]
    pred = pred_mod.Predictor(net, K, synth.skeleton_for(cfg['workload']), device=local, overlap_decode=overlap)
    return plan, net, pred


def timed_steps(pred, dev_images, steps, warmup, world, device):
    """W untimed + K timed passes of forward+decode on device-resident images; ms per step (max over ranks)."""
    stream = torch.cuda.current_stream(device)
    for _ in range(warmup):
        pred.batch_device(dev_images)
    pred.join()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        pred.batch_device(dev_images)
    pred.join()
    e1.record(stream)
    barrier(world)
    return max_over_ranks(e0.elapsed_time(e1), world, device) / steps


def timed_e2e(pred, host_pool, steps, warmup, world, device):
    for _ in pred.batches(host_pool[i % 2] for i in range(max(2, warmup))):
        pass
    barrier(world)
    t0 = time.perf_counter()
    n_ann = 0
    for res in pred.batches(host_pool[i % 2] for i in range(steps)):
        n_ann = sum(len(a) for a, _ in res)
    torch.cuda.synchronize()
    return max_over_ranks(time.perf_counter() - t0, world, device), n_ann


def forward_profile(net, images, pk):
    """per-launch CUDA events inside one forward: the tcgen05 GEMMs' achieved bytes/s and FLOP/s (ALGORITHMIC
    bytes and FLOPs: padding columns are not counted, net.cu emit_gemm)"""
    ms_op, kind, flops, nbytes = net.forward_timed(images)
    sel = kind == 1
    gemm_ms = float(ms_op[sel].sum())
    # every tcgen05 GEMM launch against ITS OWN bound: the slower of (algorithmic bytes / measured HBM peak) and
    # (algorithmic FLOPs / measured bf16 peak).  Stage-4 / conv5 launches (K, N >= 696) are tensor bound, the rest
    # HBM bound; `frac` below = sum of the bound times / sum of the measured times.
    t_hbm = nbytes[sel] / (pk['hbm_gbs'] * 1e9) * 1e3
    t_ten = flops[sel] / (pk['bf16_tflops'] * 1e12) * 1e3
    is_hbm = t_hbm >= t_ten
    ms_g = ms_op[sel]

    def cls(mask, bound_ms, unit_scale, work, unit, peak):
        if not mask.any():
            return None
        t = float(ms_g[mask].sum())
        return {'launches': int(mask.sum()), 'ms': round(t, 3), 'achieved': round(float(work[mask].sum()) / (t * 1e-3) / unit_scale, 1),
                'peak': peak, 'unit': unit, 'frac': round(float(bound_ms[mask].sum()) / t, 4)}
    per_bound = {
        'hbm_bound': cls(is_hbm, t_hbm, 1e9, nbytes[sel], 'GB/s', pk['hbm_gbs']),
        'tensor_bound': cls(~is_hbm, t_ten, 1e12, flops[sel], 'TFLOP/s', pk['bf16_tflops']),
        'frac_of_own_bound': round(float(np.maximum(t_hbm, t_ten).sum()) / gemm_ms, 4),
    }
    return ms_op, kind, flops, nbytes, {
        'per_bound': per_bound,
        'forward_ms': round(float(ms_op.sum()), 3),
        'by_kind_ms': {'input_conv': round(float(ms_op[kind == 0].sum()), 3), 'gemm_tc': round(gemm_ms, 3),
                       'dwconv': round(float(ms_op[kind == 2].sum()), 3),
                       'fused_dw_gemm': round(float(ms_op[kind == 3].sum()), 3)},
        'gemm_gbs': round(float(nbytes[sel].sum()) / (gemm_ms * 1e-3) / 1e9, 1),
        'gemm_tflops': round(float(flops[sel].sum()) / (gemm_ms * 1e-3) / 1e12, 1),
        'forward_gbs': round(float(nbytes.sum()) / (float(ms_op.sum()) * 1e-3) / 1e9, 1),
        'forward_tflops': round(float(flops.sum()) / (float(ms_op.sum()) * 1e-3) / 1e12, 1),
    }


def decoder_only(pred, cfg, fields_dev, pk, reps=10):
    """decode alone on device-resident planted fields: ms per image, and where that sits against HBM"""
    cif, caf = fields_dev
    nb = int(cif.shape[0])
    dec = pred.decoder
    stream = torch.cuda.current_stream(pred.device)
    for _ in range(3):
        dec.decode_batch(cif, 16, caf, 16)
    torch.cuda.synchronize()
    d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    d0.record(stream)
    for _ in range(reps):
        dec.decode_batch_async(cif, 16, caf, 16)
    d1.record(stream)
    torch.cuda.synchronize()
    ms_batch = d0.elapsed_time(d1) / reps
    n_dec = sum(len(a) for a, _ in dec.fetch())
    st = dec.last_stats()
    F, C = int(cif.shape[1]), int(caf.shape[1])
    hw = int(cif.shape[3] * cif.shape[4])
    side = cfg['size']
    field_bytes = (F * 5 + C * 8) * hw * 4
    dense = field_bytes + F * side * side * 4                       # SURVEY 8d A_dec: fields once + one pass over CifHr
    sparse = field_bytes + 8.0 * st['cifhr_pixels_written'] / nb     # SURVEY 8d sparse lower bound
    t_img = ms_batch * 1e-3 / nb
    return {
        'ms_per_img': round(ms_batch / nb, 4), 'ms_per_batch': round(ms_batch, 3), 'batch': nb, 'annotations': n_dec,
        'fields': f"planted poses ({'Poisson(4)+1' if cfg['people'] is None else cfg['people']} people/img), "
                  f"{int(cif.shape[3])}x{int(cif.shape[4])} cells", 'work': st,
        'roofline': {
            'bound': 'hbm', 'unit': 'GB/s', 'peak': pk['hbm_gbs'],
            'dense_bytes_per_img': int(dense), 'achieved_dense': round(dense / t_img / 1e9, 1),
            'frac_dense': round(dense / t_img / 1e9 / pk['hbm_gbs'], 4),
            'sparse_bytes_per_img': int(sparse), 'achieved_sparse': round(sparse / t_img / 1e9, 1),
            'frac_sparse': round(sparse / t_img / 1e9 / pk['hbm_gbs'], 4),
            'note': 'the decode is latency bound (one CTA per image walks the frontier), not HBM bound: the sparse '
                    'map touches a few % of the dense bytes; frac_dense is the figure SURVEY 8d asks for'},
    }


def extra_config(name, local, pk, steps=5, warmup=3):
    """bounded measurement of another BASELINE config at N=1: forward + planted decode per step"""
    cfg = CONFIGS[name]
    device = torch.device('cuda', local)
    B = cfg['batch']
    try:
        plan, net, pred = build_predictor(cfg, B, local, overlap=False)
        fields = planted_fields(cfg, B)
        cif = torch.from_numpy(fields['cif']).to(device)
        caf = torch.from_numpy(fields['caf']).to(device)
        pred.decode_fields_override = (cif, 16, caf, 16)
        images = torch.randn((B, 3, cfg['size'], cfg['size']), generator=torch.Generator().manual_seed(5)).to(device)
        ms_step = timed_steps(pred, images, steps, warmup, 1, device)
        n_ann = sum(len(a) for a, _ in pred.decoder.fetch())
        _, _, _, _, prof = forward_profile(net, images, pk)
        dec = decoder_only(pred, cfg, (cif, caf), pk, reps=5)
        img_s = B / (ms_step * 1e-3)
        out = {'network': cfg['base'], 'workload': cfg['workload'], 'input': [B, 3, cfg['size'], cfg['size']],
               'images_per_s': round(img_s, 1), 'ms_per_step': round(ms_step, 3), 'annotations_per_step': n_ann,
               'planted_people': int(sum(fields['n_planted'])),
               'forward_ms': prof['forward_ms'], 'by_kind_ms': prof['by_kind_ms'],
               'decode_ms_per_batch': dec['ms_per_batch'],
               'algorithmic_gflop_per_image': round(net.flops_per_image / 1e9, 1),
               'survey_gflop_per_image': ALGO_GFLOP_PER_IMAGE[name],
               'tensor_frac_of_measured_bf16': round(net.flops_per_image * B / (prof['forward_ms'] * 1e-3) / 1e12 / pk['bf16_tflops'], 4),
               'forward_hbm_frac': round(prof['forward_gbs'] / pk['hbm_gbs'], 4),
               'gemm_hbm_frac': round(prof['gemm_gbs'] / pk['hbm_gbs'], 4)}
        pred.close()
        return out
    except Exception as e:      # noqa: BLE001  (a failing extra config must not take the headline down)
        return {'error': f'{type(e).__name__}: {e}'[:300]}


DUMP_HEAD_IMAGES = 16       # cif + caf of 16 images of 641 px: 25.5 MB of float32


def dump_outputs(out_dir, results, heads):
    """What the last timed step computed, as .npy files a second build's dump can be compared with: the decoded
    annotations of every image (concatenated, with per-image counts and ids) and the two head outputs of a fixed,
    seeded sample of DUMP_HEAD_IMAGES images (all heads of a 64-image batch would be 100 MB)."""
    os.makedirs(out_dir, exist_ok=True)
    cif, caf = heads
    b = int(cif.shape[0])
    pick = np.sort(np.random.default_rng(0).choice(b, min(b, DUMP_HEAD_IMAGES), replace=False))
    arrays = {
        'annotations': np.concatenate([a.numpy() for a, _ in results]).astype(np.float32),
        'annotation_counts': np.array([len(a) for a, _ in results], dtype=np.float64),
        'annotation_ids': np.concatenate([i.numpy() for _, i in results]).astype(np.float64),
        'head_images': pick.astype(np.float64),
        'cif': cif[torch.from_numpy(pick).to(cif.device)].cpu().numpy().astype(np.float32),
        'caf': caf[torch.from_numpy(pick).to(caf.device)].cpu().numpy().astype(np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def load_committed(name):
    try:
        with open(os.path.join(ROOT, 'profiles', name)) as f:
            return json.load(f)
    except (OSError, ValueError):
        return None


# ----------------------------------------------------------------------------- this repo's arm
def run_b200(args):
    from openpifpaf_b200 import _lib
    rank, world, local = dist_setup()
    device = torch.device('cuda', local)
    torch.cuda.set_device(device)
    assert TOTAL_BATCH % world == 0, 'the 64 images shard evenly over 1, 2, 4 or 8 ranks'
    B = args.batch if args.batch else TOTAL_BATCH // world
    first = rank * B
    cfg = dict(CONFIGS['C0'], batch=B)
    pk = peaks()

    plan, net, pred = build_predictor(cfg, B, local, overlap=bool(args.overlap))
    fields = planted_fields(cfg, B, first_image=first)
    cif = torch.from_numpy(fields['cif']).to(device)
    caf = torch.from_numpy(fields['caf']).to(device)
    pred.decode_fields_override = (cif, 16, caf, 16)

    g = torch.Generator().manual_seed(1234 + rank)
    if args.raw_input:      # raw uint8 HWC images; ToTensor + Normalize run inside the stem kernel (not the default:
        # the reference's Predictor.batch takes the normalised float batch, and so does the headline number)
        host_images = torch.randint(0, 256, (B, SIZE, SIZE, 3), generator=g, dtype=torch.uint8).pin_memory()
    else:
        host_images = torch.randn((B, 3, SIZE, SIZE), generator=g, dtype=torch.float32).pin_memory()
    dev_images = host_images.to(device)

    # ---- device-resident throughput (value): forward + decode of the planted batch, every step
    sampler = ClockSampler(local)
    for _ in range(args.warmup):
        pred.batch_device(dev_images)
    pred.join()
    barrier(world)
    sampler.start()
    launches0 = _lib.lib().pifpaf_launch_count()
    ms_per_step = timed_steps(pred, dev_images, args.steps, 0, world, device)
    launches = int(_lib.lib().pifpaf_launch_count() - launches0)
    clocks = sampler.stop()
    results = pred.decoder.fetch(stream=pred.result_stream())
    n_ann_value = sum(len(a) for a, _ in results)
    torch.cuda.synchronize()
    value = world * B / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, results, net._head_views(B))

    # ---- end to end through the public API with host buffers: Predictor.batches() is the pipelined
    # iterator (H2D of batch i+1 under the compute of batch i), like the reference's Predictor.dataloader()
    host_pool = [host_images, host_images.clone().pin_memory()]
    t_e2e, n_ann_e2e = timed_e2e(pred, host_pool, args.steps, args.warmup, world, device)
    e2e_value = world * B * args.steps / t_e2e
    hdr = ((3 * B + 1) * 4 + 15) // 16 * 16
    d2h_bytes = min(hdr + 512 * 1024, hdr + B * 512 * 18 * 16)       # one fixed-size async copy per step

    # ---- N > 1: the weak-scaled point (64 images per GPU) beside the strong-scaled headline
    weak = None
    if world > 1 and not args.no_weak:
        cfg_w = dict(CONFIGS['C0'], batch=TOTAL_BATCH)
        _, _, pred_w = build_predictor(cfg_w, TOTAL_BATCH, local, overlap=bool(args.overlap))
        fw = planted_fields(cfg_w, TOTAL_BATCH, first_image=0)
        pred_w.decode_fields_override = (torch.from_numpy(fw['cif']).to(device), 16, torch.from_numpy(fw['caf']).to(device), 16)
        imgs_w = torch.randn((TOTAL_BATCH, 3, SIZE, SIZE), generator=g).to(device)
        ms_w = timed_steps(pred_w, imgs_w, max(3, args.steps // 2), 3, world, device)
        weak = {'images_per_gpu': TOTAL_BATCH, 'value': round(world * TOTAL_BATCH / (ms_w * 1e-3), 2),
                'ms_per_step': round(ms_w, 3), 'unit': 'images/s'}
        pred_w.close()

    out = None
    if rank == 0:
        # ---- roofline of the dominant kernels (the tcgen05 GEMMs k_gemm_tc / k_gemm_tc2), measured live with CUDA events per launch
        prof_images = dev_images if not args.raw_input else torch.randn((B, 3, SIZE, SIZE), device=device)
        ms_op, kind, flops, nbytes, prof = forward_profile(net, prof_images, pk)
        sel = kind == 1
        n_gemm = int(sel.sum())
        gemm_ms = float(ms_op[sel].sum())
        traffic, traffic_src = measured_traffic(('k_gemm_tc', 'k_gemm_tc2'), n_gemm)
        roofline = {
            'kernel': 'k_gemm_tc + k_gemm_tc2 (tcgen05 1x1-conv GEMMs: one CTA M=128 / CTA pairs cta_group::2 M=256; '
                      '%d launches/step)' % n_gemm,
            'bound': 'hbm', 'achieved': prof['gemm_gbs'], 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
            'frac': round(prof['gemm_gbs'] / pk['hbm_gbs'], 4), 'traffic': traffic,
            'traffic_unit': 'bytes/launch (dram read+write)', 'traffic_source': traffic_src,
            'algorithmic_bytes_per_launch': round(float(nbytes[sel].sum()) / n_gemm),
            'bytes_basis': 'algorithmic: real input channels read once + real output channels written once + '
                           'non-zero weights, bf16 (padding columns of the NHWC layout not counted)',
            'peak_source': pk['source'],
            'tensor_tflops': prof['gemm_tflops'],
            'tensor_frac_of_measured_bf16': round(prof['gemm_tflops'] / pk['bf16_tflops'], 4),
            'share_of_forward': round(gemm_ms / float(ms_op.sum()), 3),
            'forward_ms': prof['forward_ms'], 'by_kind_ms': prof['by_kind_ms'],
            'forward_tflops': prof['forward_tflops'],
            'forward_tensor_frac_of_measured_bf16': round(prof['forward_tflops'] / pk['bf16_tflops'], 4),
            'forward_hbm_frac': round(prof['forward_gbs'] / pk['hbm_gbs'], 4),
            'per_bound': prof['per_bound'],
        }
        # ---- decoder-only on the planted fields
        pred.decode_fields_override = None
        dec_only = decoder_only(pred, cfg, (cif[:min(B, 64)], caf[:min(B, 64)]), pk)
        if args.dump_ops:
            table = []
            for i, o in enumerate(net.op_desc):
                hh, ww, _ = net.tensor_shapes[o['out']] if 'out' in o else net.tensor_shapes[o['in']]
                table.append({'op': i, 'kind': o['kind'], 'out_hw': [hh, ww], 'k_cols': o.get('k_cols'),
                              'n_out': o.get('n_out', o.get('channels')), 'stride': o.get('stride'),
                              'ms': round(float(ms_op[i]), 4), 'gflops': round(float(flops[i]) / 1e9, 2),
                              'gbytes': round(float(nbytes[i]) / 1e9, 4),
                              'tflops': round(float(flops[i]) / float(ms_op[i]) / 1e9, 1),
                              'gbs': round(float(nbytes[i]) / float(ms_op[i]) / 1e6, 0)})
            with open(args.dump_ops, 'w') as f:
                json.dump({'batch': B, 'ops': table}, f, indent=1)
        pred.close()
        extra, library, cpu = {}, None, None
        if world == 1 and not args.quick:
            for name in ('C2', 'C3', 'C4', 'C5'):
                extra[name] = extra_config(name, local, pk)
            library = library_baseline(plan, dev_images if not args.raw_input else prof_images, ms_op)
            cpu = cpu_baseline(args)
        elif world == 8 and not args.quick:
            extra['C4'] = extra_config('C4', local, pk)      # 8 images per GPU: the per-GPU share of the 64-image C4
        out = {
            'metric': METRIC, 'value': round(value, 2), 'unit': 'images/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': round(ms_per_step, 3), 'higher_is_better': True,
            'scaling': 'strong' if not args.batch else 'weak',
            'vs_baseline': None, 'dtype': 'bf16 (f32 accumulate; decoder f32/f64)', 'data': 'synthetic',
            'config': {'workload': workload_name(B, world), 'total_batch': B * world, 'batch_per_gpu': B,
                       'input': ('raw uint8 HWC images (normalisation fused into the stem), ' if args.raw_input else 'randn images, ') +
                                'random-init weights (He), head pre-activations centred and rescaled to N(0,1) '
                                'with confidence bias -2.5',
                       'decoder_input': 'planted poses, Poisson(4)+1 people per image (SURVEY 8d), decoded inside every '
                                        'timed step in place of the random network\'s own (pose-free) fields',
                       'parallelism': f'{world} rank(s), the 64 images sharded by rank, no data-path collective',
                       'decode_overlap': 'decode of step i on a second stream under the forward of step i+1 '
                                         '(double-buffered head outputs)' if args.overlap else 'same stream, sequential',
                       'l2': f'inputs {int(host_images.numel() * host_images.element_size() / 1e6)} MB/step'
                             + (' > 126 MB L2 (no explicit flush)' if host_images.numel() * host_images.element_size() > 126e6
                                else '; activations of one forward (>= 3 GB at 8 images) stream through the 126 MB L2 between steps')},
            'impl': 'b200', 'gpu_launches': launches,
            'e2e': {'value': round(e2e_value, 2), 'unit': 'images/s',
                    'h2d_bytes_per_step': int(host_images.numel() * host_images.element_size()), 'd2h_bytes_per_step': int(d2h_bytes),
                    'api': 'openpifpaf_b200.predictor.Predictor.batches(iterable of pinned host image batches)'},
            'annotations_last_step': int(n_ann_value), 'annotations_last_step_e2e': int(n_ann_e2e),
            'planted_people_per_step': int(sum(fields['n_planted'])),
            'decoder_only': {k: v for k, v in dec_only.items() if k != 'roofline'},
            'decoder_roofline': dec_only['roofline'],
            'roofline': roofline, 'clocks': clocks, 'cpu_baseline': cpu, 'library_baseline': library,
            'extra_configs': extra, 'weak_scaling': weak,
            'net_gflop_per_image': round(net.flops_per_image / 1e9, 2),
            'net_gflop_per_image_survey': ALGO_GFLOP_PER_IMAGE['C0'],
            'bf16_accuracy': load_committed('r2_bf16_accuracy.json'),
        }
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
        dist.destroy_process_group()
    if out is not None:
        print(json.dumps(out), flush=True)


# ----------------------------------------------------------------------------- baselines (the only users of oracle/)
def library_baseline(plan, dev_images, ms_op):
    """BASELINE.md 4: stock PyTorch / cuDNN forward of the reference's own Shell (same weights, same GPU, same
    batch), forward only.  Needs the staged reference package (oracle/_ref_pkg)."""
    try:
        from oracle import ref_arm
        if not ref_arm.available():
            return {'unavailable': 'oracle/_ref_pkg not staged'}
        res = ref_arm.run_library_gpu(plan, 'shufflenetv2k16', 'cocokp', dev_images)
        ours = float(ms_op.sum())
        return {'what': "forward of the reference's own Shell through stock PyTorch/cuDNN on this GPU, same weights and batch",
                'fp32_ms': round(res['fp32_ms'], 2), 'bf16_channels_last_ms': round(res['bf16_channels_last_ms'], 2),
                'this_repo_forward_ms': round(ours, 3),
                'speedup_vs_fp32': round(res['fp32_ms'] / ours, 2),
                'speedup_vs_bf16_channels_last': round(res['bf16_channels_last_ms'] / ours, 2)}
    except Exception as e:      # noqa: BLE001
        return {'unavailable': f'{type(e).__name__}: {e}'[:300]}


def reference_step_setup(cpu_sample):
    """The CPU arm's workload: the same random plan with its heads calibrated the same way on the same calibration
    input (statistics from this arm's own fp32 features instead of the CUDA arm's bf16 ones), `cpu_sample` images of
    the batch, the planted fields of those images."""
    from oracle import ref_arm
    cfg = CONFIGS['C0']
    plan = make_plan(cfg)
    images = torch.randn((cpu_sample, 3, SIZE, SIZE), generator=torch.Generator().manual_seed(1234))
    # head calibration like network.calibrate_random_heads, on the CPU arm's own features
    shell = ref_arm.cpu_shell(plan, cfg['base'], cfg['workload'])
    with torch.no_grad():     # the input network.calibrate_random_heads draws on the GPU side
        feat = shell.base_net(torch.randn((2, 3, SIZE, SIZE), generator=torch.Generator().manual_seed(0)))
    f = feat.permute(0, 2, 3, 1).reshape(-1, feat.shape[1]).double().numpy()
    mu = f.mean(0)
    std = float(np.sqrt(np.mean(np.square(f - mu))))
    for hd in plan['heads']:
        w = hd['w'].astype(np.float64) / max(std, 1e-6)
        hd['b'] = (hd['b'].astype(np.float64) - w @ mu).astype(np.float32)
        hd['w'] = w.astype(np.float32)
    return ref_arm, plan, cfg, images, planted_fields(cfg, cpu_sample)


def cpu_baseline(args):
    """bounded sample of the reference arm, run as its own process (its torch thread settings and the reference
    package's plugin registry stay out of this one)"""
    cmd = [sys.executable, os.path.abspath(__file__), '--impl', 'reference', '--steps', '1', '--warmup', '1',
           '--cpu-sample', str(args.cpu_sample)]
    try:
        env = {k: v for k, v in os.environ.items() if k not in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK')}
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=env)
        line = [ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1]
        return json.loads(line)['cpu_baseline']
    except Exception as e:      # noqa: BLE001
        return {'unavailable': f'{type(e).__name__}: {e}'[:300]}


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    base = {'metric': METRIC, 'unit': 'images/s', 'n_gpus': args.gpus, 'higher_is_better': True, 'scaling': 'strong',
            'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'impl': 'reference', 'gpu_launches': 0}
    sample = args.cpu_sample
    ref_arm_mod, plan, cfg, images, planted = reference_step_setup(sample)
    steps, warmup = max(1, args.steps), max(0, min(args.warmup, 2))
    # keep the whole run within a few minutes: one probe step decides how many of the K steps fit
    probe = ref_arm_mod.run_cpu(plan, cfg['base'], cfg['workload'], images, planted, 1, warmup)
    budget_s = 150.0
    steps_run = int(max(1, min(steps, budget_s // max(probe['seconds'], 1e-3))))
    res = ref_arm_mod.run_cpu(plan, cfg['base'], cfg['workload'], images, planted, steps_run, 0)
    value = res['images'] / res['seconds']
    if res['kind'] == 'reference':
        what = ("the reference's own Shell (network.Factory, same weights as the CUDA arm) on PyTorch-CPU fp32, "
                "{threads}, + its Decoder.batch with the C++ CifCaf decoding the planted fields of the same images, "
                "serial per image (decoder/decoder.py:33-34)")
    else:
        what = ("the port (the reference package is not staged): oracle/net_oracle.py's Shell (same weights as the "
                "CUDA arm) on PyTorch-CPU fp32, {threads}, + the plain-C oracle CifCaf decoding the planted fields of "
                "the same images, serial per image")
    threads = (f"{res['cores']} threads = the fastest of all / half / quarter / eighth of the {os.cpu_count()} "
               f"host cores")
    desc = (f"{sample} images of the C0 batch per step, {steps_run} of {steps} steps (150 s budget): "
            + what.format(threads=threads)
            + f"; forward {res['nn_seconds'] / steps_run:.2f} s + decode {res['decoder_seconds'] / steps_run * 1e3:.1f} ms per step")
    cpu = {'value': round(value, 3), 'unit': 'images/s', 'cores': res['cores'], 'kind': res['kind'], 'sample': desc,
           'annotations_last_step': res['annotations_last_step']}
    out = dict(base, value=round(value, 3), steps=steps_run, warmup=warmup,
               ms_per_step=round(res['seconds'] / steps_run * 1e3, 2),
               config={'workload': workload_name(TOTAL_BATCH // max(1, args.gpus), max(1, args.gpus)), 'sample': desc,
                       'decoder_input': 'planted poses, Poisson(4)+1 people per image (same fields as the CUDA arm)'},
               cpu_baseline=cpu,
               e2e={'value': round(value, 3), 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
               annotations_last_step=res['annotations_last_step'])
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--batch', type=int, default=0,
                    help='images per GPU per step (default: 64 / n_gpus, the strong-scaled C0; setting it makes the run weak-scaled)')
    ap.add_argument('--cpu-sample', type=int, default=4, help='images per step of the bounded CPU arm')
    ap.add_argument('--overlap', type=int, default=1, help='decode on a second stream under the next forward (0/1)')
    ap.add_argument('--quick', action='store_true', help='headline only: no extra configs, library or CPU baselines')
    ap.add_argument('--no-weak', action='store_true', help='N > 1: skip the weak-scaled (64 per GPU) point')
    ap.add_argument('--raw-input', action='store_true',
                    help='feed raw uint8 [B,H,W,3] images (normalisation fused into the stem) instead of float32 [B,3,H,W]')
    ap.add_argument('--dump-ops', default=None, help='write the per-op timing table (profiling pass) to this JSON file')
    ap.add_argument('--dump-outputs', default=None, metavar='DIR',
                    help='write what the last timed step computed (annotations, sampled head outputs) as DIR/<name>.npy')
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == 'b200' else args.warmup
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
