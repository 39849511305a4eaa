"""CPU: the MobileNetV2 / MobileNetV3 lowering.  (1) tests/mobilenet_oracle.py equals the reference's own
basenetworks.MobileNetV2 / V3 (tests/golden/reference_mobilenet.npz); (2) build_ops + tests/mobilenet_emulator.py reproduce the
oracle Shell in fp32; (3) the op list has the architecture's work and 32-byte aligned rows; (4) modules the kernels
cannot fuse are refused."""
import importlib.util
import os

import numpy as np
import pytest
import torch

import helpers
import mobilenet_emulator
import mobilenet_oracle
from openpifpaf_b200 import network
from oracle import make_golden as mg

_spec = importlib.util.spec_from_file_location(
    'make_mobilenet_golden', os.path.join(os.path.dirname(helpers.GOLDEN_DIR), '..', 'tools', 'make_mobilenet_golden.py'))
golden_gen = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(golden_gen)

# per image at 641x641 (forward hooks on torchvision's constructors): dense (non-depthwise) backbone convs and
# depthwise convs, GMAC
GMAC_641 = {'mobilenetv3large': (6.50, 0.61), 'mobilenetv3small': (1.58, 0.25), 'mobilenetv2': (2.39, 0.17)}


@pytest.mark.parametrize('name', mobilenet_oracle.MOBILENETS)
def test_oracle_mobilenet_equals_reference_module(name):
    g = np.load(os.path.join(helpers.GOLDEN_DIR, 'reference_mobilenet.npz'))
    oracle = mobilenet_oracle.make_shell(name, seed=5).base_net
    assert golden_gen.weights_sha(oracle) == str(g[f'{name}_weights_sha256'])
    x = golden_gen.net_input()
    assert mg.sha(x.numpy()) == str(g['input_sha256'])
    with torch.no_grad():
        out = oracle(x)
    assert int(g[f'{name}_stride']) == oracle.stride
    assert tuple(out.shape) == tuple(g[f'{name}_shape'])
    torch.testing.assert_close(out.reshape(-1)[torch.from_numpy(golden_gen.sample_index(out.numel()))],
                               torch.from_numpy(g[f'{name}_sample']), rtol=0, atol=1e-5)
    torch.testing.assert_close(out[0].mean((1, 2)), torch.from_numpy(g[f'{name}_channel_mean']), rtol=0, atol=1e-5)


@pytest.mark.parametrize('shape', [(97, 129), (65, 81)])
@pytest.mark.parametrize('name', mobilenet_oracle.MOBILENETS)
def test_mobilenet_lowering_reproduces_oracle_net(name, shape):
    h, w = shape
    shell = mobilenet_oracle.make_shell(name, seed=1)
    x = torch.randn(2, 3, h, w, generator=torch.Generator().manual_seed(2))
    with torch.no_grad():
        want = shell(x)
    plan = network.plan_from_shell(shell)
    assert plan['kind'] == 'mobilenet'
    tensors, ops, _ = network.build_ops(plan, h, w)
    got, _ = mobilenet_emulator.run_ops(tensors, ops, x)
    for g, wnt in zip(got, want):
        assert g.shape == wnt.shape
        assert float((g - wnt).abs().max()) < 1e-5 * max(1.0, float(wnt.abs().max()))
    assert all(c % 16 == 0 for (_, _, c) in tensors)
    n_se = sum(o['kind'] == 'se_conv1x1' for o in ops)
    assert n_se == {'mobilenetv3large': 8, 'mobilenetv3small': 9, 'mobilenetv2': 0}[name]


@pytest.mark.parametrize('name', mobilenet_oracle.MOBILENETS)
def test_random_mobilenet_plan_has_reference_architecture(name):
    """random_mobilenet_plan has the layout plan_from_shell extracts, and the work of the table in GMAC_641"""
    plan = network.random_mobilenet_plan(name)
    ref = network.plan_from_shell(mobilenet_oracle.make_shell(name))
    assert len(plan['blocks']) == len(ref['blocks'])
    for a, b in zip(plan['blocks'], ref['blocks']):
        for key in ('expand', 'dw', 'project'):
            assert (a[key] is None) == (b[key] is None)
            if a[key] is not None:
                assert a[key]['w'].shape == b[key]['w'].shape
                assert (a[key]['kernel'], a[key]['stride'], a[key]['pad'], a[key]['act']) == \
                    (b[key]['kernel'], b[key]['stride'], b[key]['pad'], b[key]['act'])
        assert (a['se'] is None) == (b['se'] is None) and a['residual'] == b['residual']
        if a['se'] is not None:
            assert a['se']['w1'].shape == b['se']['w1'].shape
    assert plan['input']['stride'] == ref['input']['stride'] and plan['input']['act'] == ref['input']['act']
    assert plan['last']['w'].shape == ref['last']['w'].shape and plan['last']['act'] == ref['last']['act']
    tensors, ops, info = network.build_ops(plan, 641, 641)
    dense = dw = 0.0
    for o in ops:
        if o['kind'] in ('input_conv', 'conv1x1', 'conv', 'se_conv1x1'):
            hh, ww, _ = tensors[o['out']]
            dense += hh * ww * o['w'].size / 1e9
        elif o['kind'] == 'dwconv':
            hh, ww, _ = tensors[o['out']]
            dw += hh * ww * o['w'].size / 1e9
    want_dense, want_dw = GMAC_641[name]
    assert abs(dense / want_dense - 1) < 0.01, dense
    assert abs(dw / want_dw - 1) < 0.01 + 0.005 / want_dw, dw        # the table rounds to 0.01 GMAC
    stride = 32 if name == 'mobilenetv2' else 16
    assert tensors[info['feature'][0]][:2] == ((641 - 1) // stride + 1,) * 2


def _shell_with(name, module_path, module):
    shell = mobilenet_oracle.make_shell(name)
    parent = shell.base_net.backbone
    for p in module_path[:-1]:
        parent = parent[p] if isinstance(p, int) else getattr(parent, p)
    parent[module_path[-1]] = module
    return shell


@pytest.mark.parametrize('name,path,module,msg', [
    ('mobilenetv3large', (4, 'block', 1, 2), torch.nn.LeakyReLU(), 'LeakyReLU'),
    ('mobilenetv2', (3, 'conv', 0, 2), torch.nn.SiLU(), 'SiLU'),
    ('mobilenetv3small', (1, 'block', 0, 2), torch.nn.GELU(), 'GELU'),
    ('mobilenetv3small', (0, 2), torch.nn.ELU(), 'ELU'),
])
def test_unsupported_module_is_rejected(name, path, module, msg):
    shell = _shell_with(name, path, module)
    with pytest.raises(RuntimeError, match=f'unsupported module in the MobileNet backbone: {msg}'):
        network.plan_from_shell(shell)


def test_squeeze_excitation_with_other_activations_is_rejected():
    shell = mobilenet_oracle.make_shell('mobilenetv3small')
    shell.base_net.backbone[1].block[1].scale_activation = torch.nn.Sigmoid()
    with pytest.raises(RuntimeError, match='squeeze-excitation'):
        network.plan_from_shell(shell)


def test_hardswish_still_rejected_outside_mobilenets():
    """the up-front module scan keeps refusing Hardswish & co. in ShuffleNetV2K and ResNet backbones"""
    from oracle import net_oracle
    shell = net_oracle.make_shell('shufflenetv2k16')
    shell.base_net.conv5[2] = torch.nn.Hardswish()
    with pytest.raises(RuntimeError, match='Hardswish'):
        network.plan_from_shell(shell)
