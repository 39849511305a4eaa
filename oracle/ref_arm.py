"""oracle/ref_arm.py -- TEST / BASELINE INFRASTRUCTURE, NOT PRODUCT CODE.

Runs the UNMODIFIED reference (the staged package oracle/_ref_pkg, see build_ref.stage_package) on the bench
workload: its own ``Shell`` built by its own ``network.Factory`` and its own ``Decoder.batch`` with the CPU C++
``CifCaf`` (decoder/decoder.py:114-137, decoder/cifcaf.py:224-277).  Used only by bench.py's reference legs
(`--impl reference`, `cpu_baseline`, `library_baseline`) and by tests; the product never imports it.  Where the package is not staged,
the CPU legs run the port instead: oracle/net_oracle.py's Shell and the plain-C oracle decoder (`run_port_cpu`).

Same workload as the CUDA arm:
  * same weights: the folded plan of openpifpaf_b200.network.random_plan (+ calibrated heads) is written into the
    reference Shell (conv <- folded weight, BatchNorm <- identity scale with the folded bias), so both arms compute
    the same function;
  * same decoder input: a random-init network emits no poses, so both arms decode the planted Poisson(4)+1 fields
    of the same images (the CUDA arm through Predictor.decode_fields_override, here by substituting the fields
    that Decoder.fields_batch returns AFTER it has run the model and moved its output to the host -- the stock
    code path runs in full, only the tensors handed to the per-image decode are replaced).
"""
import os
import sys
import time

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PKG_DIR = os.path.join(HERE, '_ref_pkg')


def available():
    return os.path.exists(os.path.join(PKG_DIR, 'openpifpaf', '_cpp.so'))


def import_reference():
    """import the staged reference package (never a pip-installed one)"""
    if not available():
        raise RuntimeError('oracle/_ref_pkg is not staged: run `python oracle/build_ref.py` where /root/reference exists')
    if PKG_DIR not in sys.path:
        sys.path.insert(0, PKG_DIR)
    if ROOT not in sys.path:
        sys.path.insert(1, ROOT)
    import warnings
    warnings.filterwarnings('ignore')
    import openpifpaf
    torch.ops.openpifpaf.set_quiet(True)
    return openpifpaf


def head_metas(openpifpaf, workload):
    if workload == 'wholebody':
        return openpifpaf.plugins.wholebody.Wholebody().head_metas
    return openpifpaf.plugins.coco.CocoKp().head_metas


def _set_conv_bn(conv, bn, wb):
    w, b = wb
    with torch.no_grad():
        conv.weight.copy_(torch.from_numpy(np.ascontiguousarray(w)).view_as(conv.weight))
        bn.weight.fill_(1.0)
        bn.bias.copy_(torch.from_numpy(np.ascontiguousarray(b)))
        bn.running_mean.zero_()
        bn.running_var.fill_(1.0 - bn.eps)          # (x - 0) / sqrt(var + eps) == x


def shell_from_plan(openpifpaf, plan, base_name, workload='cocokp'):
    """The reference's own Shell (network/factory.py:182-199, from scratch) carrying the weights of a folded plan
    (inverse of openpifpaf_b200.network.plan_from_shell)."""
    f = openpifpaf.network.Factory()
    f.base_name, f.checkpoint = base_name, None
    openpifpaf.network.basenetworks.Resnet.pretrained = False
    shell, _ = f.factory(head_metas=head_metas(openpifpaf, workload))
    return _load_plan(shell, plan)


def port_shell_from_plan(plan, base_name, workload='cocokp'):
    """oracle/net_oracle.py's restatement of the same Shell (same module and parameter names) carrying the weights
    of a folded plan: the CPU arm's network when the reference package is not staged."""
    from oracle import net_oracle
    from openpifpaf_b200 import synth
    shell = net_oracle.make_shell(base_name, n_keypoints=synth.WORKLOADS[workload][0],
                                  n_connections=len(synth.skeleton_for(workload)), randomize_bn=False)
    return _load_plan(shell, plan)


def _load_plan(shell, plan):
    base = shell.base_net
    if plan['kind'] == 'shufflenetv2k':
        _set_conv_bn(base.input_block[0][0], base.input_block[0][1], (plan['input']['w'], plan['input']['b']))
        for stage, blocks in zip((base.stage2, base.stage3, base.stage4), plan['stages']):
            for blk, e in zip(stage, blocks):
                b2 = blk.branch2
                _set_conv_bn(b2[0], b2[1], e['b2_pw1'])
                _set_conv_bn(b2[3], b2[4], e['b2_dw'])
                _set_conv_bn(b2[5], b2[6], e['b2_pw2'])
                if e['first']:
                    _set_conv_bn(blk.branch1[0], blk.branch1[1], e['b1_dw'])
                    _set_conv_bn(blk.branch1[2], blk.branch1[3], e['b1_pw'])
        _set_conv_bn(base.conv5[0], base.conv5[1], plan['conv5'])
    elif plan['kind'] == 'resnet':
        _set_conv_bn(base.input_block[0], base.input_block[1], (plan['input']['w'], plan['input']['b']))
        blocks = [blk for stage in (base.block2, base.block3, base.block4, base.block5) for blk in stage]
        for blk, e in zip(blocks, plan['blocks']):
            pairs = [(blk.conv1, blk.bn1), (blk.conv2, blk.bn2)] + ([(blk.conv3, blk.bn3)] if hasattr(blk, 'conv3') else [])
            for (c, n), ce in zip(pairs, e['convs']):
                _set_conv_bn(c, n, (ce['w'], ce['b']))
            if e['downsample'] is not None:
                _set_conv_bn(blk.downsample[0], blk.downsample[1], (e['downsample']['w'], e['downsample']['b']))
    else:
        raise ValueError(plan['kind'])
    with torch.no_grad():
        for hn, hd in zip(shell.head_nets, plan['heads']):
            hn.conv.weight.copy_(torch.from_numpy(np.ascontiguousarray(hd['w'])).view_as(hn.conv.weight))
            hn.conv.bias.copy_(torch.from_numpy(np.ascontiguousarray(hd['b'])))
    shell.eval()
    return shell


class SubstitutedFields:
    """Context manager: Decoder.fields_batch (decoder/decoder.py:76-112) runs as it is -- model forward, `.cpu()` of
    every head -- and then hands the planted fields of the same images to the per-image decode."""

    def __init__(self, openpifpaf, planted_cif, planted_caf):
        self.cls = openpifpaf.decoder.Decoder
        self.cif = torch.from_numpy(planted_cif)
        self.caf = torch.from_numpy(planted_caf)
        self.cursor = 0

    def __enter__(self):
        self.original = self.cls.__dict__['fields_batch']
        orig = self.original.__func__
        outer = self

        def fields_batch(cls, model, image_batch, *, device=None):
            heads = orig(cls, model, image_batch, device=device)
            out = []
            for i in range(len(heads)):
                k = (outer.cursor + i) % outer.cif.shape[0]
                out.append([outer.cif[k], outer.caf[k]])
            outer.cursor += len(heads)
            return out

        self.cls.fields_batch = classmethod(fields_batch)
        return self

    def __exit__(self, *exc):
        self.cls.fields_batch = self.original


def pick_threads(shell, size=321):
    """PyTorch-CPU convolutions need not scale to every core of a many-core host (round 1: 0.15 images/s with all
    128 threads of the GPU box, 0.66 with 8): probe all / half / quarter / eighth of the cores, keep the fastest."""
    cores = os.cpu_count() or 1
    candidates = sorted({max(1, cores // d) for d in (1, 2, 4, 8)}, reverse=True)
    probe = torch.randn((1, 3, size, size), generator=torch.Generator().manual_seed(7))
    best, best_dt = cores, None
    for n in candidates:
        torch.set_num_threads(n)
        with torch.no_grad():
            shell(probe)
            t0 = time.perf_counter()
            shell(probe)
            dt = time.perf_counter() - t0
        if best_dt is None or dt < best_dt:
            best, best_dt = n, dt
    torch.set_num_threads(best)
    return best


def cpu_shell(plan, base_name, workload='cocokp'):
    """The CPU arm's network: the reference's own Shell when the reference package is staged, else the port's."""
    if available():
        return shell_from_plan(import_reference(), plan, base_name, workload)
    return port_shell_from_plan(plan, base_name, workload)


def run_cpu(plan, base_name, workload, images, planted, steps, warmup, decoder_workers=0):
    """`steps` timed passes of Decoder.batch(model, images) on the host cores.  Returns a dict with the timing where
    the reference measures it (decoder/decoder.py:116-118,129-132).  Without the staged reference package the same
    step runs on the port (`run_port_cpu`); `kind` says which of the two ran."""
    if not available():
        return run_port_cpu(plan, base_name, workload, images, planted, steps, warmup)
    openpifpaf = import_reference()
    shell = shell_from_plan(openpifpaf, plan, base_name, workload)
    cores = pick_threads(shell)
    metas = shell.head_metas
    if decoder_workers:
        openpifpaf.decoder.Decoder.default_worker_pool = int(decoder_workers)
    dec = openpifpaf.decoder.CifCaf([metas[0]], [metas[1]])        # the CPU decoder, not the plugin
    device = torch.device('cpu')
    n_ann, nn_t, dec_t = 0, 0.0, 0.0
    with SubstitutedFields(openpifpaf, planted['cif'], planted['caf']) as sub:
        for _ in range(warmup):
            dec.batch(shell, images[:1], device=device)
        sub.cursor = 0
        t0 = time.perf_counter()
        for _ in range(steps):
            sub.cursor = 0
            res = dec.batch(shell, images, device=device)
            nn_t += dec.last_nn_time
            dec_t += dec.last_decoder_time
            n_ann = sum(len(r) for r in res)
        dt = time.perf_counter() - t0
    return {'seconds': dt, 'images': int(images.shape[0]) * steps, 'cores': cores, 'annotations_last_step': n_ann,
            'nn_seconds': nn_t, 'decoder_seconds': dec_t, 'decoder_workers': int(decoder_workers), 'kind': 'reference'}


def run_port_cpu(plan, base_name, workload, images, planted, steps, warmup):
    """The step of `run_cpu` on the port: net_oracle's Shell forward on PyTorch-CPU fp32, then the plain-C oracle
    (a bit-exact restatement of the reference's C++ CifCaf, tests/test_oracle.py) decoding the planted fields of
    each image in turn."""
    from oracle import cifcaf as oc
    from openpifpaf_b200 import synth
    shell = port_shell_from_plan(plan, base_name, workload)
    cores = pick_threads(shell)
    n_kp = synth.WORKLOADS[workload][0]
    skeleton = np.asarray(synth.skeleton_for(workload), dtype=np.int64) - 1
    stride = shell.base_net.stride
    params = oc.default_params()

    def step(batch):
        t0 = time.perf_counter()
        with torch.no_grad():
            [h.cpu() for h in shell(batch)]
        t1 = time.perf_counter()
        anns = [oc.decode(planted['cif'][k], stride, planted['caf'][k], stride, skeleton, n_kp, params=params)[0]
                for k in range(int(batch.shape[0]))]
        return t1 - t0, time.perf_counter() - t1, sum(len(a) for a in anns)

    for _ in range(warmup):
        step(images[:1])
    n_ann, nn_t, dec_t = 0, 0.0, 0.0
    t0 = time.perf_counter()
    for _ in range(steps):
        dn, dd, n_ann = step(images)
        nn_t += dn
        dec_t += dd
    dt = time.perf_counter() - t0
    return {'seconds': dt, 'images': int(images.shape[0]) * steps, 'cores': cores, 'annotations_last_step': n_ann,
            'nn_seconds': nn_t, 'decoder_seconds': dec_t, 'decoder_workers': 0, 'kind': 'port'}


def run_library_gpu(plan, base_name, workload, images_dev, reps=3):
    """Stock PyTorch / cuDNN forward of the reference's own Shell with the same weights on the same GPU
    (BASELINE.md 4: the library bar): fp32 as the reference runs it (TF32 allowed, torch default for convolutions)
    and bf16 channels_last.  ms per forward of the whole batch, CUDA events."""
    openpifpaf = import_reference()
    shell = shell_from_plan(openpifpaf, plan, base_name, workload).to(images_dev.device)
    out = {}
    for name in ('fp32', 'bf16_channels_last'):
        m, x = shell, images_dev
        if name == 'bf16_channels_last':
            m = shell.to(memory_format=torch.channels_last).to(torch.bfloat16)
            x = images_dev.to(torch.bfloat16).contiguous(memory_format=torch.channels_last)
        with torch.no_grad():
            for _ in range(2):
                m(x)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                m(x)
            e1.record()
            torch.cuda.synchronize()
        out[name + '_ms'] = e0.elapsed_time(e1) / reps
    del shell
    torch.cuda.empty_cache()
    return out
