"""GPU: MobileNetV2 / MobileNetV3 backbones with CompositeField4 heads on the sm_100a kernels -- every op against the
bf16 emulation (tcgen05 and SIMT debug GEMMs), fields against fp32 PyTorch at 641x641, batch independence of the
squeeze-excitation path, the raw uint8 input path, and the reference's own Predictor through the plugin."""
import os
import subprocess
import sys
import textwrap

import numpy as np
import pytest
import torch

import mobilenet_emulator
import mobilenet_oracle
from openpifpaf_b200 import network

pytestmark = pytest.mark.gpu

FIELD_TOL_REL = 3e-2      # tests/test_network_gpu.py: 3e-2 * std + 1e-3 against fp32 PyTorch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'oracle', '_ref_pkg')


@pytest.mark.parametrize('name', mobilenet_oracle.MOBILENETS)
def test_every_op_matches_bf16_emulation(name):
    shell = mobilenet_oracle.make_shell(name, seed=3)
    plan = network.plan_from_shell(shell)
    h, w, B = 97, 129, 2
    x = torch.randn(B, 3, h, w, generator=torch.Generator().manual_seed(0))
    tensors, ops, _ = network.build_ops(plan, h, w)
    emu_heads, emu_acts = mobilenet_emulator.run_ops(tensors, ops, x, bf16=True)
    net = network.CompiledNet(plan, h, w, B)
    for impl in (1, 0):
        heads = net.forward(x.cuda(), gemm_impl=impl)
        torch.cuda.synchronize()
        for o in ops:
            if o['kind'] == 'heads':
                continue
            got = net.tap(o['out'], B)
            ref = emu_acts[o['out']].numpy()
            scale = max(float(np.abs(ref).max()), 1e-6)
            assert float(np.abs(got - ref).max()) / scale < 3e-2, (impl, o['kind'], o['out'])
        for hg, he in zip(heads, emu_heads):
            assert float((hg.cpu() - he).abs().max()) < 5e-2 * max(1.0, float(he.std()))
    net.close()


@pytest.mark.parametrize('name', mobilenet_oracle.MOBILENETS)
def test_fields_match_fp32_pytorch_full_size(name):
    """641x641, batch 4, vs fp32 PyTorch (no TF32) on the same GPU"""
    shell = mobilenet_oracle.make_shell(name, seed=2)
    plan = network.plan_from_shell(shell)
    net = network.CompiledNet(plan, 641, 641, 4)
    x = torch.randn(4, 3, 641, 641, generator=torch.Generator().manual_seed(1)).cuda()
    heads = [t.clone() for t in net.forward(x)]
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        ref = shell.cuda()(x)
    side = 21 if name == 'mobilenetv2' else 41
    for hg, hr in zip(heads, ref):
        assert hg.shape == hr.shape == (4, hr.shape[1], hr.shape[2], side, side)
        err = float((hg - hr).abs().max())
        assert err < FIELD_TOL_REL * float(hr.std()) + 1e-3, err
    net.close()


@pytest.mark.parametrize('name', mobilenet_oracle.MOBILENETS)
def test_batch_of_different_images_equals_each_image_alone(name):
    """the squeeze-excitation pools and per-image projection weights never mix images: each image of a batch of three
    different images gives the fields it gives alone, bit for bit"""
    plan = network.random_mobilenet_plan(name, seed=4)
    net = network.CompiledNet(plan, 161, 193, 3)
    g = torch.Generator().manual_seed(9)
    x = torch.cat([torch.randn(1, 3, 161, 193, generator=g) * s + m for s, m in ((1.0, 0.0), (0.3, 1.0), (2.0, -0.5))])
    x = x.cuda()
    full = [t.clone() for t in net.forward(x)]
    for b in range(3):
        one = net.forward(x[b:b + 1].contiguous())
        for hf, ho in zip(full, one):
            assert torch.isfinite(ho).all()
            assert torch.equal(hf[b], ho[0]), (b, float((hf[b] - ho[0]).abs().max()))
    assert not torch.equal(full[0][0], full[0][1])
    net.close()


@pytest.mark.parametrize('name', mobilenet_oracle.MOBILENETS)
def test_uint8_input_equals_float_path(name):
    plan = network.random_mobilenet_plan(name, seed=6)
    net = network.CompiledNet(plan, 129, 161, 2)
    raw = torch.randint(0, 256, (2, 129, 161, 3), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
    mean = torch.tensor(network.CompiledNet.IMAGE_MEAN).view(1, 3, 1, 1)
    std = torch.tensor(network.CompiledNet.IMAGE_STD).view(1, 3, 1, 1)
    flt = ((raw.permute(0, 3, 1, 2).float() / 255.0) - mean) / std
    a = [t.clone() for t in net.forward(flt.contiguous().cuda())]
    b = [t.clone() for t in net.forward_uint8(raw.cuda())]
    for ta, tb in zip(a, b):
        assert torch.equal(ta, tb)
    net.close()


SCRIPT = textwrap.dedent('''
    import json, sys, warnings
    warnings.filterwarnings('ignore')
    import numpy as np
    import torch
    import openpifpaf
    from openpifpaf.network import basenetworks
    basenetworks.MobileNetV2.pretrained = basenetworks.MobileNetV3.pretrained = False     # never download
    torch.ops.openpifpaf.set_quiet(True)
    assert 'openpifpaf_b200' in openpifpaf.plugin.REGISTERED
    report = {}
    for base_name in ('mobilenetv3large', 'mobilenetv3small'):
        torch.manual_seed(0)
        openpifpaf.network.Factory.base_name = base_name
        openpifpaf.network.Factory.checkpoint = None
        datamodule = openpifpaf.plugins.coco.CocoKp()
        predictor = openpifpaf.Predictor(head_metas=datamodule.head_metas)
        multi = predictor.processor
        top = multi.decoders[0]
        assert type(top).__name__ == 'CifCafB200', type(top).__name__
        cif_meta, caf_meta = predictor.model_cpu.head_metas
        model = predictor.model
        with torch.no_grad():        # trained-network-like head statistics (tests/test_plugin_gpu.py)
            probe = torch.randn(2, 3, 161, 193, generator=torch.Generator().manual_seed(7)).to(predictor.device)
            feat = model.base_net(probe)
            mu = feat.mean((0, 2, 3))
            std = (feat - mu[None, :, None, None]).pow(2).mean().sqrt()
            for head in model.head_nets:
                w = head.conv.weight / std
                head.conv.bias.copy_(head.conv.bias - w[:, :, 0, 0] @ mu)
                head.conv.weight.copy_(w)
                head.conv.bias.view(head.meta.n_fields, head.n_components)[:, 1] += -1.0
        ref_cpu = openpifpaf.decoder.CifCaf([cif_meta], [caf_meta])
        import argparse
        parser = argparse.ArgumentParser()
        openpifpaf.decoder.cli(parser)
        openpifpaf.decoder.configure(parser.parse_args(['--force-complete-pose', '--seed-threshold=0.1']))
        g = torch.Generator().manual_seed(1)
        images = torch.randn(3, 3, 161, 193, generator=g)
        pred_batch = multi.batch(model, images, device=predictor.device)
        compiled = [p for (_, _, p) in top._compiled.values() if (p.net.in_h, p.net.in_w) == (161, 193)][0]
        fields = [t.cpu() for t in compiled.net.forward(images.cuda())]
        n = 0
        for i in range(3):
            want = ref_cpu([f[i] for f in fields])
            got = pred_batch[i]
            assert len(got) == len(want), (base_name, i, len(got), len(want))
            for a, b in zip(got, want):
                assert float(np.abs(a.data[:, :2] - b.data[:, :2]).max()) <= 1e-4
                assert float(np.abs(a.data[:, 2] - b.data[:, 2]).max()) <= 1e-5
            n += len(want)
        openpifpaf.decoder.configure(parser.parse_args([]))
        report[base_name] = n
    assert all(v > 0 for v in report.values()), report
    print('MOBILENET_PLUGIN_OK', json.dumps(report))
''')


@pytest.mark.skipif(not os.path.exists(os.path.join(PKG, 'openpifpaf', '_cpp.so')),
                    reason='oracle/_ref_pkg not staged (python oracle/build_ref.py in the build container)')
def test_reference_predictor_runs_mobilenets_through_the_plugin(tmp_path):
    env = dict(os.environ, PYTHONPATH=f'{PKG}:{ROOT}')
    r = subprocess.run([sys.executable, '-c', SCRIPT], capture_output=True, text=True, env=env, cwd=str(tmp_path),
                       timeout=900)
    assert 'MOBILENET_PLUGIN_OK' in r.stdout, r.stdout[-3000:] + r.stderr[-5000:]
