"""CPU: (1) the oracle network equals the reference's own PyTorch modules (their outputs stored by
oracle/make_golden.py); (2) the product's host lowering (BN folding, physical channel placement, fused
cat+channel_shuffle, head epilogue) reproduces the oracle network when its op list is interpreted on the CPU."""
import os

import numpy as np
import pytest
import torch

import helpers
import ops_emulator
from openpifpaf_b200 import network
from oracle import make_golden as mg
from oracle import net_oracle


def reference_networks():
    """the reference's own modules on oracle/make_golden.py's inputs (python -m oracle.make_golden reference)"""
    return np.load(os.path.join(helpers.GOLDEN_DIR, 'reference_networks.npz'))


def test_oracle_net_equals_reference_modules():
    """net_oracle's shufflenetv2k16 + CompositeField4 heads == the reference's basenetworks.ShuffleNetV2K and
    heads.CompositeField4 carrying the same (randomised) weights"""
    g = reference_networks()
    oracle = net_oracle.make_shell('shufflenetv2k16', seed=3)
    x = mg.net_input('shufflenetv2k16')
    assert mg.sha(x.numpy()) == str(g['shufflenetv2k16_input_sha256'])
    with torch.no_grad():
        got = oracle(x)
    for name, gt in zip(('cif', 'caf'), got):
        want = torch.from_numpy(g['shufflenetv2k16_' + name])
        assert want.shape == gt.shape
        torch.testing.assert_close(gt, want, rtol=0, atol=1e-5)


@pytest.mark.parametrize('layout', ['bins', 'shuffle'])
@pytest.mark.parametrize('shape', [(97, 129), (65, 65)])
def test_lowering_reproduces_oracle_net(shape, layout):
    h, w = shape
    shell = net_oracle.make_shell('shufflenetv2k16', seed=1)
    x = torch.randn(2, 3, h, w)
    with torch.no_grad():
        want = shell(x)
    plan = network.plan_from_shell(shell)
    tensors, ops, _ = network.build_ops(plan, h, w, layout=layout)
    got, _ = ops_emulator.run_ops(tensors, ops, x)
    for g, wnt in zip(got, want):
        assert g.shape == wnt.shape
        assert float((g - wnt).abs().max()) < 2e-5
    # rows start on 32-byte boundaries (256-bit stores); TMA views start on 16-byte boundaries
    assert all(c % 16 == 0 for (_, _, c) in tensors)
    for o in ops:
        if o['kind'] in ('conv1x1', 'dwconv'):
            assert o['in_off'] % 8 == 0
    if layout == 'shuffle':
        for o in ops:
            if o['kind'] in ('conv1x1', 'dwconv'):
                assert o['out_off'] % 16 == 0
        # x.chunk(2) of 348 channels: the view starts at or below column 174 on a multiple of 8, the leading
        # columns carry zero weights
        a0 = network._view_start(174)
        assert a0 % 8 == 0 and 174 - 64 < a0 <= 174
        views = [o for o in ops if o['kind'] == 'conv1x1' and o['in_off'] == a0]
        assert views and all(not o['w'][:, :174 - a0].any() for o in views)
    else:
        # no fused shuffle, no column views: every 1x1 reads a whole tensor and the scatter pieces tile its columns
        assert all(o['shuffle_src'] < 0 and o['in_off'] == 0 for o in ops if o['kind'] == 'conv1x1')
        scat = [o for o in ops if 'pieces' in o]
        assert len(scat) == 2 * 3 + (3 + 7 + 3)          # two producers per first block + one per later block
        for o in scat:
            cols = 0
            for (c0, cnt, t_id, t_col) in o['pieces']:
                assert c0 == cols and cnt % 16 == 0 and t_col % 16 == 0 and t_col + cnt <= tensors[t_id][2]
                cols += cnt
            assert cols == o['n_out'] == o['w'].shape[0]


def _simulate_stage(bf, T):
    """cat + channel_shuffle + chunk of basenetworks.py:233-242 on channel labels (producer, channel)."""
    vec = [lab for n in range(bf) for lab in ((0, n), (1, n))]
    consumed = {}
    for t in range(1, T):
        x1, x2 = vec[:bf], vec[bf:]
        consumed[t] = x2
        vec = [lab for n in range(bf) for lab in (x1[n], (t + 1, n))]
    return consumed, vec


@pytest.mark.parametrize('seed', range(4))
def test_stage_bins_random_sizes(seed):
    """any branch width / block count: every bin holds exactly the inputs of its block, pieces are 16-aligned"""
    rng = np.random.default_rng(seed)
    bf, T = int(rng.integers(1, 90)) * 2, int(rng.integers(1, 10))
    producers, bins, final = network._plan_stage_bins(bf, T)
    consumed, vec = _simulate_stage(bf, T)
    where = {}
    for k, pr in enumerate(producers):
        assert len(pr['order']) % 16 == 0
        for (c0, cnt, d, dc) in pr['pieces']:
            assert cnt % 16 == 0 and dc % 16 == 0
            for i in range(cnt):
                if pr['order'][c0 + i] >= 0:
                    where[(k, int(pr['order'][c0 + i]))] = (d, dc + i)
    for t in range(1, T):
        assert [bins[t]['wcol'][where[lab][1]] for lab in consumed[t]] == list(range(bf))
        assert all(where[lab][0] == t for lab in consumed[t])
    assert [final['logical'][where[lab][1]] for lab in vec] == list(range(2 * bf))
    assert all(where[lab][0] == 'final' for lab in vec)


def test_stage_bins_route_every_channel_once():
    """_plan_stage_bins against a direct simulation of cat + channel_shuffle + chunk on channel labels."""
    for bf, T in ((174, 4), (348, 8), (6, 3), (10, 5), (256, 8)):
        producers, bins, final = network._plan_stage_bins(bf, T)
        # labels: (producer, channel); block 0 interleaves producers 0 and 1; block t interleaves x1 with producer t+1
        vec = [lab for n in range(bf) for lab in ((0, n), (1, n))]
        consumed = {}
        for t in range(1, T):
            x1, x2 = vec[:bf], vec[bf:]
            consumed[t] = x2
            vec = [lab for n in range(bf) for lab in (x1[n], (t + 1, n))]
        where = {}                                         # label -> (dest, slot)
        for k, pr in enumerate(producers):
            for (c0, cnt, d, dc) in pr['pieces']:
                for i in range(cnt):
                    n = int(pr['order'][c0 + i])
                    if n >= 0:
                        assert (k, n) not in where
                        where[(k, n)] = (d, dc + i)
        assert len(where) == (T + 1) * bf
        for t in range(1, T):
            for wc, lab in enumerate(consumed[t]):
                d, slot = where[lab]
                assert d == t and bins[t]['wcol'][slot] == wc
        for c, lab in enumerate(vec):
            d, slot = where[lab]
            assert d == 'final' and final['logical'][slot] == c


def test_k30_wholebody_lowering_reproduces_oracle_net():
    """BASELINE configs[3]: shufflenetv2k30 with the wholebody heads (133 keypoints, 160 connections)."""
    shell = net_oracle.make_shell('shufflenetv2k30', n_keypoints=133, n_connections=160, seed=3)
    x = torch.randn(1, 3, 65, 81)
    with torch.no_grad():
        want = shell(x)
    plan = network.plan_from_shell(shell)
    assert [len(st) for st in plan['stages']] == [8, 16, 6]
    tensors, ops, _ = network.build_ops(plan, 65, 81)
    got, _ = ops_emulator.run_ops(tensors, ops, x)
    assert [tuple(g.shape) for g in got] == [(1, 133, 5, 5, 6), (1, 160, 8, 5, 6)]
    for g, wnt in zip(got, want):
        assert float((g - wnt).abs().max()) < 2e-5
    head = ops[-1]
    assert head['kind'] == 'heads' and head['w'].shape == (133 * 5 + 160 * 8, 2048)


@pytest.mark.parametrize('fuse', [False, True])
def test_random_plan_has_reference_architecture(fuse):
    plan = network.random_plan('shufflenetv2k16')
    assert [len(s) for s in plan['stages']] == [4, 8, 4]
    assert plan['conv5'][0].shape[:2] == (1392, 1392)
    assert [h['w'].shape[0] for h in plan['heads']] == [85, 152]
    tensors, ops, _ = network.build_ops(plan, 641, 641, fuse_dw=fuse)
    gmac = 0.0
    for o in ops:
        hh, ww, _ = tensors[o['out']] if 'out' in o else tensors[o['in']]
        if o['kind'] == 'conv1x1':
            gmac += hh * ww * np.count_nonzero(o['w']) / 1e9
        elif o['kind'] == 'heads':
            gmac += hh * ww * o['w'].size / 1e9
        elif o['kind'] == 'dwconv':
            gmac += hh * ww * np.count_nonzero(o['w']) / 1e9
        elif o['kind'] == 'dw_conv1x1':         # fused depthwise -> 1x1 (k_dw_gemm)
            gmac += hh * ww * (np.count_nonzero(o['w']) + np.count_nonzero(o['dw_w'])) / 1e9
        elif o['kind'] == 'input_conv':
            gmac += hh * ww * o['w'].size / 1e9
    assert abs(gmac - 36.58) < 0.2, gmac       # SURVEY.md 8d: 36.58 GMAC / image @641
    # fused schedule: the stride-1 blocks of stages 2 and 3 (N <= 512)
    assert sum(o['kind'] == 'dw_conv1x1' for o in ops) == ((3 + 7) if fuse else 0)


@pytest.mark.parametrize('fuse', [True, False])
def test_fused_and_unfused_lowerings_compute_the_same_network(fuse):
    """the fused depthwise -> 1x1 op is a pure scheduling change: the op list with and without it reproduces the
    oracle network (fp32 emulation)"""
    shell = net_oracle.make_shell('shufflenetv2k16', seed=3)
    x = torch.randn(1, 3, 97, 129)
    with torch.no_grad():
        want = shell(x)
    plan = network.plan_from_shell(shell)
    tensors, ops, _ = network.build_ops(plan, 97, 129, fuse_dw=fuse)
    assert any(o['kind'] == 'dw_conv1x1' for o in ops) == fuse
    got, _ = ops_emulator.run_ops(tensors, ops, x)
    for g, wnt in zip(got, want):
        assert float((g - wnt).abs().max()) < 2e-5 * max(1.0, float(wnt.abs().max()))


def test_oracle_resnet_equals_reference_module():
    """SURVEY 8a row a3: the oracle Resnet wrapper == reference basenetworks.Resnet (max-pool removed, stride 16), on a
    seeded sample of the output elements and on every channel's mean"""
    g = reference_networks()
    torch.manual_seed(0)
    oracle = net_oracle.make_base('resnet18')
    oracle.eval()
    assert mg.sha(np.concatenate([p.detach().numpy().ravel() for p in oracle.parameters()])) == \
        str(g['resnet18_weights_sha256'])
    x = mg.net_input('resnet18')
    assert mg.sha(x.numpy()) == str(g['resnet18_input_sha256'])
    with torch.no_grad():
        out = oracle(x)
    assert int(g['resnet18_stride']) == oracle.stride == 16
    assert tuple(out.shape) == tuple(g['resnet18_shape']) == (1, 512, 11, 11)
    torch.testing.assert_close(out.reshape(-1)[torch.from_numpy(mg.resnet_sample_index())],
                               torch.from_numpy(g['resnet18_sample']), rtol=0, atol=1e-5)
    torch.testing.assert_close(out[0].mean((1, 2)), torch.from_numpy(g['resnet18_channel_mean']), rtol=0, atol=1e-5)


@pytest.mark.parametrize('name,shape', [('resnet18', (161, 161)), ('resnet50', (97, 113))])
def test_resnet_lowering_reproduces_oracle_net(name, shape):
    h, w = shape
    shell = net_oracle.make_shell(name, seed=1)
    x = torch.randn(2, 3, h, w)
    with torch.no_grad():
        want = shell(x)
    plan = network.plan_from_shell(shell)
    assert plan['kind'] == 'resnet'
    tensors, ops, _ = network.build_ops(plan, h, w)
    got, _ = ops_emulator.run_ops(tensors, ops, x)
    for g, wnt in zip(got, want):
        assert g.shape == wnt.shape
        assert float((g - wnt).abs().max()) < 1e-5 * max(1.0, float(wnt.abs().max()))
    n_conv = sum(o['kind'] == 'conv' for o in ops)
    assert n_conv == (20 if name == 'resnet18' else 53) - 1       # all convs but the stem (SURVEY appendix A)


def test_stride2_depthwise_inputs_have_128_byte_pixels():
    """network._dw_in_pitch: the tensor in front of the stride-2 depthwise conv of a stage's first block is padded to a
    multiple of 64 channels (DRAM serves the depthwise TMA reads in aligned 128-byte lines: 1.96x over-read with 352-byte
    pixels, profiles/r2_history.md), every other branch-internal tensor keeps the 16-channel pitch, and the depthwise op
    still covers the real channels only."""
    plan = network.random_plan('shufflenetv2k16', seed=3)
    tensors, ops, _ = network.build_ops(plan, 161, 161, layout='bins', fuse_dw=False)
    s2 = [o for o in ops if o['kind'] == 'dwconv' and o['stride'] == 2]
    s1 = [o for o in ops if o['kind'] == 'dwconv' and o['stride'] == 1]
    assert len(s2) == 6 and len(s1) == 13
    for o in s2:
        c_phys = tensors[o['in']][2]
        assert (c_phys * 2) % 128 == 0 or c_phys <= 32, (o['in'], c_phys)       # (the 24-channel stem output: 64-byte pixels)
        assert o['channels'] <= c_phys and o['channels'] % 16 == 0
    assert {tensors[o['in']][2] for o in s1} == {176, 352, 704}
