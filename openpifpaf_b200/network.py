"""Host-side mirror of the reference network modules for the inference hot path.

Reference (paths relative to /root/reference/src/openpifpaf/):
  Shell.forward                       network/nets.py:35-48
  ShuffleNetV2K / InvertedResidualK   network/basenetworks.py:186-355
  MobileNetV2 / MobileNetV3           network/basenetworks.py:407-458 (torchvision `features`)
  CompositeField4 (eval)              network/heads.py:330-378

`plan_from_shell(shell)` walks a reference-style ``Shell`` (duck-typed: the
reference's own ``openpifpaf.network.nets.Shell`` or any module tree with the
same attribute names), folds every eval-mode BatchNorm into its convolution and
returns a plain "plan" of float32 numpy arrays.  `CompiledNet` turns a plan into
a fused op list of libpifpaf_b200 (tcgen05 GEMMs for the 1x1 convolutions) and
replays it.  torch.cat / chunk / channel_shuffle never run as kernels: they are
folded into the physical channel placement computed here.

  'bins' layout (default): every channel of a stage is written once, by the GEMM
  that produces it, into the buffer of the block that consumes it; pass-through
  channels are never copied (see _plan_stage_bins).

  'shuffle' layout: activations in logical channel order; the last GEMM of a block
  writes logical channel 2n <- pass-through[n], 2n+1 <- conv[n] (== cat +
  channel_shuffle(groups=2), basenetworks.py:233-242) with aligned 256-bit stores,
  and the next block's x.chunk(2) is the TMA start coordinate _view_start(half) of
  its A operand (the leading pass-through columns meet zero weight columns).
"""
import ctypes
import os

import numpy as np
import torch

from . import _lib

OP_RAW, OP_SIGMOID, OP_ADD_X, OP_ADD_Y, OP_SOFTPLUS = 0, 1, 2, 3, 4

SHUFFLENETV2K_CONFIGS = {     # network/factory.py:68-79
    'shufflenetv2k16': ([4, 8, 4], [24, 348, 696, 1392, 1392]),
    'shufflenetv2k20': ([5, 10, 5], [32, 512, 1024, 2048, 2048]),
    'shufflenetv2k30': ([8, 16, 6], [32, 512, 1024, 2048, 2048]),
}


def pad8(v):
    return (v + 7) // 8 * 8


def pad16(v):
    return (v + 15) // 16 * 16


# ----------------------------------------------------------------------------- plans

def _fold(conv, bn):
    """conv (bias-free) followed by eval BatchNorm -> (weight, bias) float32 numpy."""
    w = conv.weight.detach().double()
    scale = bn.weight.detach().double() / torch.sqrt(bn.running_var.detach().double() + bn.eps)
    b = bn.bias.detach().double() - bn.running_mean.detach().double() * scale
    if conv.bias is not None:
        b = b + conv.bias.detach().double() * scale
    w = w * scale.view(-1, 1, 1, 1)
    return w.float().cpu().numpy(), b.float().cpu().numpy()


def head_ops(n_confidences, n_vectors, n_scales, vector_offsets):
    """Per-component epilogue of CompositeField4.forward in eval mode (heads.py:360-378)."""
    ops = [OP_RAW] + [OP_SIGMOID] * n_confidences
    for i in range(n_vectors):
        ops += [OP_ADD_X, OP_ADD_Y] if vector_offsets[i] else [OP_RAW, OP_RAW]
    ops += [OP_SOFTPLUS] * n_scales
    return ops


def _heads_plan(shell, base):
    heads = []
    for hn in shell.head_nets:
        m = hn.meta
        up = int(getattr(m, 'upsample_stride', 1))
        ncomp = 1 + m.n_confidences + m.n_vectors * 2 + m.n_scales
        heads.append({
            # upsample_stride > 1 (heads.py:307-343): the conv has n_fields * n_comp * up^2 channels, PixelShuffle(up)
            # and the crop run in the GEMM epilogue (pifpaf_net_heads_upsampled)
            'w': hn.conv.weight.detach().float().cpu().numpy().reshape(m.n_fields * ncomp * up * up, -1),
            'b': hn.conv.bias.detach().float().cpu().numpy(),
            'n_fields': int(m.n_fields), 'n_comp': int(ncomp), 'upsample': up,
            'ops': head_ops(m.n_confidences, m.n_vectors, m.n_scales, tuple(m.vector_offsets)),
            'stride': int(base.stride) // up})
    if len({hd['upsample'] for hd in heads}) > 1:
        raise RuntimeError('heads with different upsample_stride values are not supported')
    return heads


def _plan_from_resnet(shell):
    """basenetworks.py:71-150: torchvision ResNet without the max-pool (input_block = conv1, bn1, relu;
    block2..block5 = layer1..layer4 of BasicBlock / Bottleneck)."""
    base = shell.base_net
    if len(base.input_block) != 3:
        raise RuntimeError('only the default Resnet input block (conv, bn, relu; pool0_stride=0) is supported')
    conv, bn = base.input_block[0], base.input_block[1]
    w, b = _fold(conv, bn)
    plan = {'kind': 'resnet',
            'input': {'w': w, 'b': b, 'stride': int(conv.stride[0]), 'pad': int(conv.padding[0])},
            'blocks': [], 'heads': _heads_plan(shell, base)}

    def conv_entry(c, n):
        if c.dilation[0] != 1 or c.groups != 1:
            raise RuntimeError('dilated / grouped ResNet convolutions are not supported')
        w_, b_ = _fold(c, n)
        return {'w': w_, 'b': b_, 'kernel': int(c.kernel_size[0]), 'stride': int(c.stride[0]), 'pad': int(c.padding[0])}

    for stage in (base.block2, base.block3, base.block4, base.block5):
        for blk in stage:
            e = {'convs': [conv_entry(blk.conv1, blk.bn1), conv_entry(blk.conv2, blk.bn2)]}
            if hasattr(blk, 'conv3'):
                e['convs'].append(conv_entry(blk.conv3, blk.bn3))
            e['downsample'] = None if blk.downsample is None else conv_entry(blk.downsample[0], blk.downsample[1])
            plan['blocks'].append(e)
    return plan


# fused activation codes of the C ABI (include/pifpaf_b200.h)
ACT_NONE, ACT_RELU, ACT_RELU6, ACT_HARDSWISH = 0, 1, 2, 3


def _act_code(m):
    for cls, code in ((torch.nn.ReLU, ACT_RELU), (torch.nn.ReLU6, ACT_RELU6), (torch.nn.Hardswish, ACT_HARDSWISH)):
        if type(m) is cls:
            return code
    raise RuntimeError(f'unsupported module in the MobileNet backbone: {type(m).__name__} '
                       '(only ReLU, ReLU6, Hardswish and squeeze-excitation with ReLU / Hardsigmoid)')


def _conv_bn_act(seq):
    """torchvision Conv2dNormActivation: Conv2d (bias-free), BatchNorm2d, optional activation."""
    mods = list(seq.children())
    if not (2 <= len(mods) <= 3 and isinstance(mods[0], torch.nn.Conv2d) and type(mods[1]) is torch.nn.BatchNorm2d):
        raise RuntimeError('unsupported module in the MobileNet backbone: expected Conv2d, BatchNorm2d[, activation], '
                           f'got {[type(m).__name__ for m in mods]}')
    return mods[0], mods[1], (_act_code(mods[2]) if len(mods) == 3 else ACT_NONE)


def _conv_entry(conv, bn, act):
    if conv.dilation[0] != 1 or conv.dilation[1] != 1 or conv.kernel_size[0] != conv.kernel_size[1] or \
            conv.stride[0] != conv.stride[1] or conv.padding[0] != conv.padding[1]:
        raise RuntimeError('dilated / non-square MobileNet convolutions are not supported')
    w, b = _fold(conv, bn)
    return {'w': w, 'b': b, 'kernel': int(conv.kernel_size[0]), 'stride': int(conv.stride[0]),
            'pad': int(conv.padding[0]), 'groups': int(conv.groups), 'act': act}


def _plan_from_mobilenet(shell):
    """basenetworks.py:407-458: `backbone` = torchvision MobileNetV2 / V3 `features` (the V3 stem stride set to 1 by
    the reference is read from the module).  Stem Conv2dNormActivation, InvertedResidual blocks ([expand 1x1],
    depthwise kxk, [SqueezeExcitation], linear 1x1 projection, residual when use_res_connect), last 1x1 conv."""
    base = shell.base_net
    feats = list(base.backbone.children())
    if len(feats) < 3:
        raise RuntimeError('unsupported MobileNet backbone: too few layers')
    stem = _conv_entry(*_conv_bn_act(feats[0]))
    if stem['groups'] != 1:
        raise RuntimeError('unsupported MobileNet stem')
    last = _conv_entry(*_conv_bn_act(feats[-1]))
    if last['kernel'] != 1 or last['stride'] != 1 or last['groups'] != 1:
        raise RuntimeError('unsupported MobileNet last layer: expected a 1x1 conv')
    blocks = []
    for blk in feats[1:-1]:
        inner = getattr(blk, 'block', None)
        if inner is None:
            inner = getattr(blk, 'conv', None)              # torchvision MobileNetV2's InvertedResidual
        if inner is None or not hasattr(blk, 'use_res_connect'):
            raise RuntimeError(f'unsupported module in the MobileNet backbone: {type(blk).__name__}')
        mods, units = list(inner.children()), []
        i = 0
        while i < len(mods):
            m = mods[i]
            if isinstance(m, torch.nn.Conv2d):             # MobileNetV2's projection: Conv2d, BatchNorm2d
                if i + 1 >= len(mods) or type(mods[i + 1]) is not torch.nn.BatchNorm2d:
                    raise RuntimeError('unsupported MobileNet block: a Conv2d without its BatchNorm2d')
                units.append(_conv_entry(m, mods[i + 1], ACT_NONE))
                i += 2
            elif isinstance(m, torch.nn.Sequential):
                units.append(_conv_entry(*_conv_bn_act(m)))
                i += 1
            elif hasattr(m, 'fc1') and hasattr(m, 'fc2'):  # torchvision SqueezeExcitation
                if type(getattr(m, 'activation', None)) is not torch.nn.ReLU or \
                        type(getattr(m, 'scale_activation', None)) is not torch.nn.Hardsigmoid:
                    raise RuntimeError('unsupported module in the MobileNet backbone: squeeze-excitation '
                                       'activations other than ReLU / Hardsigmoid')
                units.append({'se': {'w1': m.fc1.weight.detach().float().cpu().numpy()[:, :, 0, 0],
                                     'b1': m.fc1.bias.detach().float().cpu().numpy(),
                                     'w2': m.fc2.weight.detach().float().cpu().numpy()[:, :, 0, 0],
                                     'b2': m.fc2.bias.detach().float().cpu().numpy()}})
                i += 1
            else:
                _act_code(m)                               # raises with the module's name
                raise RuntimeError(f'unsupported module in the MobileNet backbone: {type(m).__name__}')
        dw_i = [k for k, u in enumerate(units) if 'se' not in u and u['groups'] > 1]
        if len(dw_i) != 1:
            raise RuntimeError('unsupported MobileNet block: expected exactly one depthwise conv')
        k = dw_i[0]
        pre, dw, post = units[:k], units[k], units[k + 1:]
        se = post.pop(0)['se'] if post and 'se' in post[0] else None
        c_dw = dw['w'].shape[0]
        if dw['groups'] != c_dw or dw['w'].shape[1] != 1 or dw['kernel'] not in (3, 5) or dw['stride'] not in (1, 2):
            raise RuntimeError('unsupported MobileNet depthwise conv (3x3 / 5x5, stride 1 / 2 only)')
        if len(pre) > 1 or len(post) != 1 or any(u['kernel'] != 1 or u['stride'] != 1 or u['groups'] != 1
                                                 for u in pre + post) or post[0]['act'] != ACT_NONE:
            raise RuntimeError('unsupported MobileNet block: expected [1x1], depthwise, [SE], linear 1x1')
        blocks.append({'expand': pre[0] if pre else None, 'dw': dw, 'se': se, 'project': post[0],
                       'residual': bool(blk.use_res_connect)})
    return {'kind': 'mobilenet', 'input': stem, 'blocks': blocks, 'last': last, 'heads': _heads_plan(shell, base)}


def plan_from_shell(shell):
    """Extract a folded plan from a reference-style Shell (ShuffleNetV2K, Resnet, MobileNetV2 or MobileNetV3 base
    net)."""
    base = shell.base_net
    if shell.training:
        raise RuntimeError('the Shell must be in eval() mode (BatchNorm is folded)')
    # network/nets.py:12-13,36-46: optional pre/post-processing hooks -- not lowered, so refuse them loudly
    if getattr(shell, 'process_input', None) is not None or getattr(shell, 'process_heads', None) is not None:
        raise RuntimeError('Shell.process_input / process_heads are not supported by the compiled forward')
    if hasattr(base, 'backbone'):
        return _plan_from_mobilenet(shell)
    for m in base.modules():
        # the kernels fuse max(x, 0); --shufflenetv2k-leaky-relu etc. would be folded wrongly
        if isinstance(m, (torch.nn.LeakyReLU, torch.nn.ELU, torch.nn.PReLU, torch.nn.SiLU, torch.nn.GELU,
                          torch.nn.Hardswish, torch.nn.InstanceNorm2d, torch.nn.GroupNorm)):
            raise RuntimeError(f'unsupported module in the base network: {type(m).__name__} (only ReLU + BatchNorm)')
    if all(hasattr(base, a) for a in ('input_block', 'block2', 'block3', 'block4', 'block5')):
        return _plan_from_resnet(shell)
    if not all(hasattr(base, a) for a in ('input_block', 'stage2', 'stage3', 'stage4', 'conv5')):
        raise RuntimeError(f'unsupported base network {type(base).__name__}: expected ShuffleNetV2K or Resnet')
    if len(base.input_block) != 1:
        raise RuntimeError('input_conv2 variants are not supported')
    conv, bn = base.input_block[0][0], base.input_block[0][1]
    w, b = _fold(conv, bn)
    plan = {'kind': 'shufflenetv2k',
            'input': {'w': w, 'b': b, 'stride': int(conv.stride[0]), 'pad': int(conv.padding[0])},
            'stages': [], 'heads': []}
    for stage in (base.stage2, base.stage3, base.stage4):
        blocks = []
        for blk in stage:
            b2 = blk.branch2
            dw = b2[3]
            if dw.dilation[0] != 1:
                raise RuntimeError('dilated stages are not supported')
            entry = {'first': blk.branch1 is not None, 'stride': int(dw.stride[0]),
                     'kernel': int(dw.kernel_size[0]), 'pad': int(dw.padding[0])}
            entry['b2_pw1'] = _fold(b2[0], b2[1])
            entry['b2_dw'] = _fold(b2[3], b2[4])
            entry['b2_pw2'] = _fold(b2[5], b2[6])
            if blk.branch1 is not None:
                entry['b1_dw'] = _fold(blk.branch1[0], blk.branch1[1])
                entry['b1_pw'] = _fold(blk.branch1[2], blk.branch1[3])
            blocks.append(entry)
        plan['stages'].append(blocks)
    if not isinstance(base.conv5[0], torch.nn.Conv2d):
        raise RuntimeError('conv5_as_stage is not supported')
    plan['conv5'] = _fold(base.conv5[0], base.conv5[1])
    plan['heads'] = _heads_plan(shell, base)
    return plan


def heads_only_plan(plan, c_in=None):
    """The heads of `plan` as a net of their own (one GEMM with the CompositeField4 eval epilogue); compile it with
    the FEATURE map size as in_h, in_w and run it with CompiledNet.forward_features."""
    c = int(plan['heads'][0]['w'].shape[1]) if c_in is None else int(c_in)
    return {'kind': 'heads_only', 'c_in': c, 'heads': plan['heads']}


def random_plan(base_name='shufflenetv2k16', heads=((17, 1, 1, 1), (19, 1, 2, 2)), seed=0, confidence_bias=-4.0):
    """Random-init folded plan of the named architecture (no checkpoint can be downloaded here).
    heads: (n_fields, n_confidences, n_vectors, n_scales) per head; vector offsets all True.
    confidence_bias is added to the bias of the confidence channels so that a random-init head emits a
    sparse confidence map (sigmoid(-4) ~ 0.02) like a trained network's background; with a zero bias every
    cell sits near 0.5 and passes every decoder threshold, which no trained model produces."""
    repeats, ch = SHUFFLENETV2K_CONFIGS[base_name]
    rng = np.random.Generator(np.random.PCG64(seed))

    def conv(cout, cin, k=1, dw=False):
        fan_in = (1 if dw else cin) * k * k
        w = rng.standard_normal((cout, 1 if dw else cin, k, k)).astype(np.float32) * np.float32(np.sqrt(2.0 / fan_in))
        b = (rng.standard_normal(cout) * 0.05).astype(np.float32)
        return w, b

    w, b = conv(ch[0], 3, 3)
    plan = {'kind': 'shufflenetv2k', 'input': {'w': w, 'b': b, 'stride': 2, 'pad': 1}, 'stages': [], 'heads': []}
    cin = ch[0]
    for rep, cout in zip(repeats, ch[1:4]):
        bf = cout // 2
        blocks = []
        for i in range(rep):
            first = i == 0
            e = {'first': first, 'stride': 2 if first else 1, 'kernel': 5, 'pad': 2}
            e['b2_pw1'] = conv(bf, cin if first else bf)
            e['b2_dw'] = conv(bf, bf, 5, dw=True)
            e['b2_pw2'] = conv(bf, bf)
            if first:
                e['b1_dw'] = conv(cin, cin, 5, dw=True)
                e['b1_pw'] = conv(bf, cin)
            blocks.append(e)
        plan['stages'].append(blocks)
        cin = cout
    plan['conv5'] = conv(ch[4], cin)
    for (nf, nconf, nvec, nsc) in heads:
        ncomp = 1 + nconf + 2 * nvec + nsc
        w = (rng.standard_normal((nf * ncomp, ch[4])) * np.sqrt(1.0 / ch[4])).astype(np.float32)
        b = (rng.standard_normal(nf * ncomp) * 0.1).astype(np.float32)
        b.reshape(nf, ncomp)[:, 1:1 + nconf] += np.float32(confidence_bias)
        plan['heads'].append({'w': w, 'b': b, 'n_fields': nf, 'n_comp': ncomp,
                              'ops': head_ops(nconf, nvec, nsc, (True,) * nvec), 'stride': 16})
    return plan


RESNET_CONFIGS = {      # torchvision.models.resnet: (block, layers); network/factory.py:57-58
    'resnet18': ('basic', [2, 2, 2, 2]),
    'resnet50': ('bottleneck', [3, 4, 6, 3]),
}


def random_resnet_plan(base_name='resnet50', heads=((17, 1, 1, 1), (19, 1, 2, 2)), seed=0, confidence_bias=-4.0):
    """Random-init folded plan of the reference's Resnet base network (basenetworks.py:71-150: torchvision ResNet,
    max-pool removed, stride 16; BasicBlock 3x3-3x3 / Bottleneck 1x1-3x3(stride)-1x1 with expansion 4, 1x1
    downsample on the first block of a stage) -- the same dict layout `_plan_from_resnet` extracts from a Shell.
    The last conv of a block and the downsample conv get half the He variance so that the residual sum keeps the
    activation scale over 16 blocks."""
    kind, layers = RESNET_CONFIGS[base_name]
    rng = np.random.Generator(np.random.PCG64(seed))

    def conv(cout, cin, k, stride, gain=2.0):
        w = rng.standard_normal((cout, cin, k, k)).astype(np.float32) * np.float32(np.sqrt(gain / (cin * k * k)))
        b = (rng.standard_normal(cout) * 0.05).astype(np.float32)
        return {'w': w, 'b': b, 'kernel': k, 'stride': stride, 'pad': (k - 1) // 2}

    stem = conv(64, 3, 7, 2)
    plan = {'kind': 'resnet', 'input': {'w': stem['w'], 'b': stem['b'], 'stride': 2, 'pad': 3}, 'blocks': [], 'heads': []}
    expansion = 1 if kind == 'basic' else 4
    cin = 64
    for si, (planes, n) in enumerate(zip((64, 128, 256, 512), layers)):
        for bi in range(n):
            stride = 2 if (bi == 0 and si > 0) else 1
            cout = planes * expansion
            if kind == 'basic':
                convs = [conv(planes, cin, 3, stride), conv(planes, planes, 3, 1, gain=1.0)]
            else:
                convs = [conv(planes, cin, 1, 1), conv(planes, planes, 3, stride), conv(cout, planes, 1, 1, gain=1.0)]
            down = conv(cout, cin, 1, stride, gain=1.0) if (stride != 1 or cin != cout) else None
            plan['blocks'].append({'convs': convs, 'downsample': down})
            cin = cout
    for (nf, nconf, nvec, nsc) in heads:
        ncomp = 1 + nconf + 2 * nvec + nsc
        w = (rng.standard_normal((nf * ncomp, cin)) * np.sqrt(1.0 / cin)).astype(np.float32)
        b = (rng.standard_normal(nf * ncomp) * 0.1).astype(np.float32)
        b.reshape(nf, ncomp)[:, 1:1 + nconf] += np.float32(confidence_bias)
        plan['heads'].append({'w': w, 'b': b, 'n_fields': nf, 'n_comp': ncomp,
                              'ops': head_ops(nconf, nvec, nsc, (True,) * nvec), 'stride': 16})
    return plan


# torchvision.models.mobilenetv3._mobilenet_v3_conf / mobilenetv2 inverted_residual_setting (width 1.0):
# (kernel, expanded channels, out channels, SE, activation code, stride) per block; stem channels, last conv channels
MOBILENET_CONFIGS = {
    'mobilenetv3large': (16, ACT_HARDSWISH, 960, 16, [
        (3, 16, 16, False, 1, 1), (3, 64, 24, False, 1, 2), (3, 72, 24, False, 1, 1), (5, 72, 40, True, 1, 2),
        (5, 120, 40, True, 1, 1), (5, 120, 40, True, 1, 1), (3, 240, 80, False, 3, 2), (3, 200, 80, False, 3, 1),
        (3, 184, 80, False, 3, 1), (3, 184, 80, False, 3, 1), (3, 480, 112, True, 3, 1), (3, 672, 112, True, 3, 1),
        (5, 672, 160, True, 3, 2), (5, 960, 160, True, 3, 1), (5, 960, 160, True, 3, 1)]),
    'mobilenetv3small': (16, ACT_HARDSWISH, 576, 16, [
        (3, 16, 16, True, 1, 2), (3, 72, 24, False, 1, 2), (3, 88, 24, False, 1, 1), (5, 96, 40, True, 3, 2),
        (5, 240, 40, True, 3, 1), (5, 240, 40, True, 3, 1), (5, 120, 48, True, 3, 1), (5, 144, 48, True, 3, 1),
        (5, 288, 96, True, 3, 2), (5, 576, 96, True, 3, 1), (5, 576, 96, True, 3, 1)]),
}


def _mobilenet_v2_blocks():
    """(kernel, expanded, out, SE, act, stride) of torchvision's MobileNetV2 (expand ratio t of the block's INPUT)"""
    out, cin = [], 32
    for t, c, n, s in [(1, 16, 1, 1), (6, 24, 2, 2), (6, 32, 3, 2), (6, 64, 4, 2), (6, 96, 3, 1), (6, 160, 3, 2),
                       (6, 320, 1, 1)]:
        for i in range(n):
            out.append((3, cin * t, c, False, ACT_RELU6, s if i == 0 else 1))
            cin = c
    return out


MOBILENET_CONFIGS['mobilenetv2'] = (32, ACT_RELU6, 1280, 32, _mobilenet_v2_blocks())


def _make_divisible(v, divisor=8):
    """torchvision.models._utils._make_divisible (the squeeze channels of SqueezeExcitation)"""
    new_v = max(divisor, int(v + divisor / 2) // divisor * divisor)
    return new_v + divisor if new_v < 0.9 * v else new_v


def random_mobilenet_plan(base_name='mobilenetv3large', heads=((17, 1, 1, 1), (19, 1, 2, 2)), seed=0,
                          confidence_bias=-4.0):
    """Random-init folded plan of the reference's MobileNetV2 / MobileNetV3 base networks (basenetworks.py:407-458;
    V3 with the stem stride 1 the reference sets: output stride 16, V2: 32) -- the same dict layout
    `_plan_from_mobilenet` extracts from a Shell.  He-scaled weights; the projection of a residual block gets half the
    variance so that the sums keep the activation scale."""
    c0, stem_act, c_last, stride, cfg = MOBILENET_CONFIGS[base_name]
    rng = np.random.Generator(np.random.PCG64(seed))

    def conv(cout, cin, k, stride_, act, groups=1, gain=2.0):
        fan_in = cin // groups * k * k
        w = rng.standard_normal((cout, cin // groups, k, k)).astype(np.float32) * np.float32(np.sqrt(gain / fan_in))
        b = (rng.standard_normal(cout) * 0.05).astype(np.float32)
        return {'w': w, 'b': b, 'kernel': k, 'stride': stride_, 'pad': (k - 1) // 2, 'groups': groups, 'act': act}

    v3 = base_name.startswith('mobilenetv3')
    plan = {'kind': 'mobilenet', 'input': conv(c0, 3, 3, 1 if v3 else 2, stem_act), 'blocks': [], 'heads': []}
    cin = c0
    for (k, ce, co, se, act, st) in cfg:
        sq = _make_divisible(ce // 4)
        blk = {'expand': conv(ce, cin, 1, 1, act) if ce != cin else None,
               'dw': conv(ce, ce, k, st, act, groups=ce),
               'se': None if not se else {
                   'w1': (rng.standard_normal((sq, ce)) * np.sqrt(2.0 / ce)).astype(np.float32),
                   'b1': (rng.standard_normal(sq) * 0.05).astype(np.float32),
                   'w2': (rng.standard_normal((ce, sq)) * np.sqrt(1.0 / sq)).astype(np.float32),
                   'b2': (rng.standard_normal(ce) * 0.05).astype(np.float32)},
               'residual': st == 1 and cin == co}
        blk['project'] = conv(co, ce, 1, 1, ACT_NONE, gain=1.0 if blk['residual'] else 2.0)
        plan['blocks'].append(blk)
        cin = co
    plan['last'] = conv(c_last, cin, 1, 1, stem_act if v3 else ACT_RELU6)
    for (nf, nconf, nvec, nsc) in heads:
        ncomp = 1 + nconf + 2 * nvec + nsc
        w = (rng.standard_normal((nf * ncomp, c_last)) * np.sqrt(1.0 / c_last)).astype(np.float32)
        b = (rng.standard_normal(nf * ncomp) * 0.1).astype(np.float32)
        b.reshape(nf, ncomp)[:, 1:1 + nconf] += np.float32(confidence_bias)
        plan['heads'].append({'w': w, 'b': b, 'n_fields': nf, 'n_comp': ncomp,
                              'ops': head_ops(nconf, nvec, nsc, (True,) * nvec), 'stride': stride})
    return plan


def calibrate_random_heads(plan, device=0, seed=0, size=161, batch=2):
    """Give a random-init plan trained-network-like head statistics: measure mean and spread of the backbone
    features on a small random batch (on the GPU, through the product kernels), then centre and rescale the head
    so that every head channel's pre-activation is ~N(0, 1) over positions: w' = w / std, b' = b - w' . mean.
    (Post-ReLU features have a large common mean; without centring every head channel gets its own random DC
    offset and whole confidence maps saturate.)  Together with random_plan's confidence bias this yields
    confidence maps with isolated cells above the decoder thresholds instead of saturated noise.
    Returns (feature std, feature mean norm)."""
    net = CompiledNet(plan, size, size, batch, device=device)
    x = torch.randn((batch, 3, size, size), generator=torch.Generator().manual_seed(seed)).to(f'cuda:{device}')
    net.forward(x)
    torch.cuda.synchronize()
    t, lay = net.info['feature']
    feat = net.tap(t, batch)[..., lay.cols()].astype(np.float64)
    mu = feat.reshape(-1, feat.shape[-1]).mean(axis=0)
    std = float(np.sqrt(np.mean(np.square(feat - mu))))
    for hd in plan['heads']:
        w = hd['w'].astype(np.float64) / max(std, 1e-6)
        hd['b'] = (hd['b'].astype(np.float64) - w @ mu).astype(np.float32)
        hd['w'] = w.astype(np.float32)
    return std, float(np.linalg.norm(mu))


# ----------------------------------------------------------------------------- compiled net

class _DevArray:
    """Expose a raw device pointer to torch through __cuda_array_interface__ (no copy)."""

    def __init__(self, ptr, shape, typestr='<f4'):
        self.__cuda_array_interface__ = {'shape': tuple(shape), 'typestr': typestr, 'data': (int(ptr), False),
                                         'version': 2}


class _Layout:
    """Physical column placement of a logical channel vector; rows padded to a multiple of 16 channels (32-byte
    aligned rows for 256-bit stores).  Default: physical == logical order.  `split` marks tensors of the
    'shuffle' layout whose two logical halves are consumed separately (x.chunk(2)): the second half starts at
    column `half`; its TMA view starts at _view_start(half) with zero weights on the leading columns.
    `phys` (int array [channels]) places logical channel c at physical column phys[c] of a `width`-wide row (the
    'bins' layout's stage outputs, whose rows hold the channels in order of production)."""

    def __init__(self, channels, split, phys=None, width=None):
        self.channels = channels
        self.split = split
        self.half = channels // 2 if split else None
        self.width = pad16(channels) if width is None else width
        self.phys = None if phys is None else np.asarray(phys, dtype=np.int64)

    def cols(self):
        return np.arange(self.channels) if self.phys is None else self.phys


def _view_start(half):
    """First column of the x.chunk(2)[1] view: a multiple of 8 channels (16 bytes, the TMA requirement), aligned
    further down (to 64 / 32 / 16 channels) as long as the GEMM keeps its number of 64-channel K blocks -- a box
    row that starts on a 128-byte line costs one L2 request instead of two."""
    align = os.environ.get('PIFPAF_VIEW_ALIGN', 'auto')
    if align != 'auto':
        return half // int(align) * int(align)
    k_blocks = (half - half // 8 * 8 + half + 63) // 64
    for al in (64, 32, 16, 8):
        a0 = half // al * al
        if (half - a0 + half + 63) // 64 == k_blocks:
            return a0
    return half // 8 * 8


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _plan_stage_bins(bf, n_blocks):
    """Channel routing of one ShuffleNetV2K stage for the 'bins' layout, in which no pass-through channel is ever
    copied.  The reference (basenetworks.py:233-242) computes, for block t >= 1 with input vector L_t (2*bf
    channels), L_{t+1}[2n] = L_t[n] (pass-through) and L_{t+1}[2n+1] = branch2(L_t[bf:])[n]; block 0 gives
    L_1[2n] = branch1[n], L_1[2n+1] = branch2[n].  So a channel born at position p of L_v sits at position
    p * 2^(t-v) of L_t until that position reaches bf: then it is an input of block t's branch2 (weight column
    position - bf) and dies; channels that never reach bf live on into L_T, the stage output.
    Every channel is therefore WRITTEN ONCE, by its producer GEMM, straight into the buffer of the block that
    consumes it ("bin" t = the bf inputs of block t, or the stage output), and never moved: the producer GEMM's
    columns are ordered by destination, each destination piece padded to a multiple of 16 channels (32 bytes:
    whole sectors, one 256-bit store per lane and 16 columns).

    Producers: 0 = branch1 of block 0, 1 = branch2 of block 0, t + 1 = branch2 of block t (1 <= t < n_blocks).
    Returns (producers, bins, final):
      producers[k] = {'order': int[n_total] (GEMM column -> producer output channel, -1 padding),
                      'pieces': [(col0, count, dest, dest_col)], dest = block index t or 'final'}
      bins[t]      = {'width': W (multiple of 16), 'wcol': int[W] (slot -> weight column of block t's first 1x1, -1 padding)}
      final        = {'width': W, 'logical': int[W] (slot -> channel index of the stage output, -1 padding)}"""
    T = n_blocks
    # piece granularity in channels (16 = 32 bytes: whole sectors).  PIFPAF_BIN_PAD=32 makes every piece a whole number of
    # 64-byte DRAM bursts (more padding columns: experiment of session v)
    G = int(os.environ.get('PIFPAF_BIN_PAD', '16'))

    def route(v, p):
        for t in range(max(v, 1), T):
            pos = p << (t - v)
            if pos >= bf:
                return t, pos - bf
        return 'final', p << (T - v)

    births = [(1, [2 * n for n in range(bf)]), (1, [2 * n + 1 for n in range(bf)])]
    births += [(t + 1, [2 * n + 1 for n in range(bf)]) for t in range(1, T)]
    dest_fill = {t: 0 for t in range(1, T)}
    dest_fill['final'] = 0
    slots = {d: [] for d in dest_fill}              # dest -> list of (dest_col, values) pieces
    producers = []
    for v, positions in births:
        routed = [route(v, p) for p in positions]
        order, pieces = [], []
        for d in list(range(1, T)) + ['final']:
            members = [n for n in range(bf) if routed[n][0] == d]
            if not members:
                continue
            padded = (len(members) + G - 1) // G * G
            pieces.append((len(order), padded, d, dest_fill[d]))
            slots[d].append((dest_fill[d], [routed[n][1] for n in members] + [-1] * (padded - len(members))))
            order += members + [-1] * (padded - len(members))
            dest_fill[d] += padded
        producers.append({'order': np.asarray(order, dtype=np.int64), 'pieces': pieces})

    def flat(d):
        out = np.full((dest_fill[d],), -1, dtype=np.int64)
        for col, vals in slots[d]:
            out[col:col + len(vals)] = vals
        return out

    bins = {t: {'width': dest_fill[t], 'wcol': flat(t)} for t in range(1, T)}
    final = {'width': dest_fill['final'], 'logical': flat('final')}
    for t in range(1, T):
        assert sorted(int(c) for c in bins[t]['wcol'] if c >= 0) == list(range(bf))
    assert sorted(int(c) for c in final['logical'] if c >= 0) == list(range(2 * bf))
    return producers, bins, final


def _branch_pitch(bf):
    """Physical channel count of the branch-internal tensors (1x1 -> depthwise -> 1x1).  The depthwise kernels fetch
    one 64-channel block (128 bytes) per pixel and CTA; with a pitch that is a multiple of 64 channels every block is
    one aligned 128-byte line instead of straddling two 64-byte DRAM atoms.  PIFPAF_BRANCH_PAD selects the multiple
    (16: the round-1 layout)."""
    mult = int(os.environ.get('PIFPAF_BRANCH_PAD', '16'))
    return (bf + mult - 1) // mult * mult


def _dw_in_pitch(bf):
    """Physical channel count of the tensor BETWEEN the first 1x1 of a branch and its depthwise conv.  DRAM serves the
    depthwise kernels' TMA reads (one 128-byte 64-channel block per pixel) in aligned 128-byte lines: with 352- / 704-byte
    pixels (176 / 352 channels) a block straddles two lines and the launch reads 1.96x / 1.55x the tensor
    (profiles/r2_history.md, "analysis"); tensors whose pixels are a multiple of 128 bytes read 1.00x.  Only this tensor
    is padded (to 64 channels): its producer writes the real channels with the same stores as before, and the tensor
    behind the depthwise conv -- the A operand of a GEMM, which would read the padding -- keeps the 16-channel pitch.
    PIFPAF_DWIN_PAD selects the multiple (16 = the old layout)."""
    mult = int(os.environ.get('PIFPAF_DWIN_PAD', '64'))
    return max(_branch_pitch(bf), (bf + mult - 1) // mult * mult)


def default_layout():
    """'bins' (no pass-through copies, see _plan_stage_bins) or 'shuffle' (every block writes the interleaved
    2*bf-channel tensor through the fused cat+shuffle epilogue); PIFPAF_LAYOUT overrides."""
    return os.environ.get('PIFPAF_LAYOUT', 'bins')


def default_fuse_dw():
    """Fuse depthwise 5x5 (stride 1) with the 1x1 conv that follows it into one kernel (k_dw_gemm)?  Off by default:
    the fused kernel is bit-identical to the two-kernel schedule but measured SLOWER on B200 (round 2: 0.91 ms against
    0.42 + 0.22 ms per stage-2 block, 0.58 against 0.27 + 0.14 ms per stage-3 block -- one CTA per SM leaves only 8
    depthwise warps per SM where the stand-alone depthwise kernel runs 16, and the depthwise FMA loop is issue bound;
    profiles/r2_history.md).  PIFPAF_FUSE_DW=1 turns it on."""
    return os.environ.get('PIFPAF_FUSE_DW', '0') == '1'


def build_ops(plan, in_h, in_w, layout=None, fuse_dw=None):
    """Lower a plan to the op list of libpifpaf_b200 (pure Python; no GPU needed).

    Returns (tensors, ops): tensors[i] = (h, w, c_phys); ops are dicts with a 'kind' in
    {'input_conv', 'conv1x1', 'dwconv', 'heads'} whose fields are the C ABI arguments."""
    if plan.get('kind') == 'resnet':
        return _build_ops_resnet(plan, in_h, in_w)
    if plan.get('kind') == 'mobilenet':
        return _build_ops_mobilenet(plan, in_h, in_w)
    if plan.get('kind') == 'heads_only':
        # in_h x in_w is the FEATURE map here; the feature tensor is filled through CompiledNet.forward_features
        c_in = int(plan['c_in'])
        return [(in_h, in_w, pad16(c_in))], [_heads_op(plan['heads'], 0, c_in)], \
            {'block_outputs': [], 'feature': (0, _Layout(c_in, split=False))}
    if plan.get('kind') != 'shufflenetv2k':
        raise RuntimeError('unsupported plan kind')
    layout = default_layout() if layout is None else layout
    if layout not in ('bins', 'shuffle'):
        raise RuntimeError("layout must be 'bins' or 'shuffle'")
    fuse_dw = default_fuse_dw() if fuse_dw is None else bool(fuse_dw)
    tensors, ops = [], []

    def tensor(h, w, c):
        tensors.append((h, w, c))
        return len(tensors) - 1

    def conv1x1(tin, in_off, in_cols, k_cols, wb, relu, tout, shuffle=None):
        w, b = wb
        w = w.reshape(w.shape[0], -1)
        n, cin = w.shape
        assert len(in_cols) == cin
        wp = np.zeros((n, k_cols), dtype=np.float32)
        wp[:, in_cols] = w
        s_t, s_off = (-1, 0) if shuffle is None else shuffle
        ops.append({'kind': 'conv1x1', 'in': tin, 'in_off': in_off, 'k_cols': k_cols, 'n_out': n,
                    'w': wp, 'b': _f32(b), 'relu': int(relu), 'out': tout, 'out_off': 0,
                    'shuffle_src': s_t, 'shuffle_off': s_off})

    def conv1x1_scatter(tin, in_cols, k_cols, wb, relu, order, pieces):
        """1x1 conv whose GEMM columns are the producer's output channels in `order` (-1: padding column, zero
        weights) and whose column pieces (col0, count, tensor, tensor_col) go to different tensors."""
        w, b = wb
        w = w.reshape(w.shape[0], -1)
        assert len(in_cols) == w.shape[1]
        real = order >= 0
        wp = np.zeros((len(order), k_cols), dtype=np.float32)
        wp[np.ix_(np.nonzero(real)[0], in_cols)] = w[order[real]]
        bp = np.zeros((len(order),), dtype=np.float32)
        bp[real] = b[order[real]]
        ops.append({'kind': 'conv1x1', 'in': tin, 'in_off': 0, 'k_cols': k_cols, 'n_out': len(order),
                    'w': wp, 'b': bp, 'relu': int(relu), 'out': pieces[0][2], 'out_off': pieces[0][3],
                    'shuffle_src': -1, 'shuffle_off': 0, 'pieces': [tuple(int(v) for v in pc) for pc in pieces]})

    def dw_conv1x1_scatter(tin, width, dw_wb, kernel, stride, pad, wb, relu, order, pieces):
        """depthwise kxk on the first len(dw) channels of tin, then the scatter 1x1 conv of conv1x1_scatter on its
        output -- one fused kernel, no intermediate tensor"""
        dw_w, dw_b = dw_wb
        c = dw_w.shape[0]
        dwp = np.zeros((width, kernel * kernel), dtype=np.float32)
        dbp = np.zeros((width,), dtype=np.float32)
        dwp[:c] = dw_w.reshape(c, kernel * kernel)
        dbp[:c] = dw_b
        w, b = wb
        w = w.reshape(w.shape[0], -1)
        assert w.shape[1] == c
        real = order >= 0
        wp = np.zeros((len(order), width), dtype=np.float32)
        wp[np.ix_(np.nonzero(real)[0], np.arange(c))] = w[order[real]]
        bp = np.zeros((len(order),), dtype=np.float32)
        bp[real] = b[order[real]]
        ops.append({'kind': 'dw_conv1x1', 'in': tin, 'in_off': 0, 'channels': width, 'kernel': kernel,
                    'stride': stride, 'pad': pad, 'dw_w': dwp, 'dw_b': dbp, 'dw_relu': 0, 'n_out': len(order),
                    'w': wp, 'b': bp, 'relu': int(relu), 'out': pieces[0][2],
                    'pieces': [tuple(int(v) for v in pc) for pc in pieces]})

    def dwconv(tin, cols, width, wb, kernel, stride, pad, tout):
        w, b = wb
        w = w.reshape(w.shape[0], kernel * kernel)
        wp = np.zeros((width, kernel * kernel), dtype=np.float32)
        bp = np.zeros((width,), dtype=np.float32)
        wp[cols] = w
        bp[cols] = b
        ops.append({'kind': 'dwconv', 'in': tin, 'in_off': 0, 'channels': width, 'kernel': kernel,
                    'stride': stride, 'pad': pad, 'w': wp, 'b': bp, 'relu': 0, 'out': tout, 'out_off': 0})

    inp = plan['input']
    k = inp['w'].shape[-1]
    h = (in_h + 2 * inp['pad'] - k) // inp['stride'] + 1
    w = (in_w + 2 * inp['pad'] - k) // inp['stride'] + 1
    c0 = inp['w'].shape[0]
    cur = tensor(h, w, pad16(c0))
    ops.append({'kind': 'input_conv', 'in_h': in_h, 'in_w': in_w, 'kernel': k, 'stride': inp['stride'],
                'pad': inp['pad'], 'c_out': c0, 'w': _f32(inp['w']), 'b': _f32(inp['b']), 'relu': 1, 'out': cur})
    lay = _Layout(c0, split=False)
    block_outputs = []
    for blocks in plan['stages'] if layout == 'bins' else []:
        # ---- 'bins' layout: every channel is written once, into the buffer of the block that consumes it
        bf = blocks[0]['b2_pw2'][0].shape[0]
        hp = _branch_pitch(bf)
        e0 = blocks[0]
        kk, st, pd = e0['kernel'], e0['stride'], e0['pad']
        ho, wo = (h + 2 * pd - kk) // st + 1, (w + 2 * pd - kk) // st + 1
        producers, bins, final = _plan_stage_bins(bf, len(blocks))
        t_bin = {t: tensor(ho, wo, pad16(bins[t]['width'])) for t in bins}
        t_bin['final'] = tensor(ho, wo, pad16(final['width']))

        def pieces_of(k):
            return [(c0_, cnt, t_bin[d], dc) for (c0_, cnt, d, dc) in producers[k]['pieces']]

        cols = lay.cols()
        # block 0, branch1: dw (stride) -> 1x1; branch2: 1x1 -> dw (stride) -> 1x1   (basenetworks.py:200-226)
        t_a = tensor(ho, wo, lay.width)
        dwconv(cur, cols, lay.width, e0['b1_dw'], kk, st, pd, t_a)
        conv1x1_scatter(t_a, cols, lay.width, e0['b1_pw'], True, producers[0]['order'], pieces_of(0))
        # the tensor in front of the STRIDE-2 depthwise conv gets 128-byte pixels (_dw_in_pitch).  (Measured, session s:
        # letting its producer write the padding channels too -- whole rows instead of rows with a 32-byte hole -- costs
        # that GEMM more (0.53 -> 0.69 ms at 321 x 321) than the hole does (0.53 -> 0.64).)
        t_c = tensor(h, w, _dw_in_pitch(bf))
        conv1x1(cur, 0, cols, lay.width, e0['b2_pw1'], True, t_c)
        t_d = tensor(ho, wo, hp)
        dwconv(t_c, np.arange(bf), hp, e0['b2_dw'], kk, st, pd, t_d)
        conv1x1_scatter(t_d, np.arange(bf), hp, e0['b2_pw2'], True, producers[1]['order'], pieces_of(1))
        h, w = ho, wo
        for t, e in enumerate(blocks[1:], start=1):
            assert not e['first'] and e['stride'] == 1 and e['b2_pw2'][0].shape[0] == bf
            # x2 = the bin of block t: slot j holds the channel that meets weight column wcol[j] of the first 1x1
            wcol = bins[t]['wcol']
            in_cols = np.empty((bf,), dtype=np.int64)
            in_cols[wcol[wcol >= 0]] = np.nonzero(wcol >= 0)[0]
            width = tensors[t_bin[t]][2]
            t_c = tensor(h, w, hp)          # stride-1 depthwise launches are issue bound: the padding buys nothing there
            conv1x1(t_bin[t], 0, in_cols, width, e['b2_pw1'], True, t_c)
            order = producers[t + 1]['order']
            if fuse_dw and e['kernel'] == 5 and e['pad'] == 2 and len(order) <= 512:
                dw_conv1x1_scatter(t_c, hp, e['b2_dw'], 5, 1, 2, e['b2_pw2'], True, order, pieces_of(t + 1))
                continue
            t_d = tensor(h, w, hp)
            dwconv(t_c, np.arange(bf), hp, e['b2_dw'], e['kernel'], 1, e['pad'], t_d)
            conv1x1_scatter(t_d, np.arange(bf), hp, e['b2_pw2'], True, order, pieces_of(t + 1))
        logical = final['logical']
        phys = np.empty((2 * bf,), dtype=np.int64)
        phys[logical[logical >= 0]] = np.nonzero(logical >= 0)[0]
        cur, lay = t_bin['final'], _Layout(2 * bf, split=False, phys=phys, width=tensors[t_bin['final']][2])
        block_outputs.append((cur, lay))
    for blocks in plan['stages'] if layout == 'shuffle' else []:
        for e in blocks:
            bf = e['b2_pw2'][0].shape[0]
            hp = pad16(bf)
            kk, st, pd = e['kernel'], e['stride'], e['pad']
            ho, wo = (h + 2 * pd - kk) // st + 1, (w + 2 * pd - kk) // st + 1
            out_lay = _Layout(2 * bf, split=True)
            t_out = tensor(ho, wo, out_lay.width)
            if e['first']:
                cols = lay.cols()
                # branch1: dw (stride) -> 1x1   (basenetworks.py:200-212)
                t_a = tensor(ho, wo, lay.width)
                dwconv(cur, cols, lay.width, e['b1_dw'], kk, st, pd, t_a)
                t_b = tensor(ho, wo, hp)
                conv1x1(t_a, 0, cols, lay.width, e['b1_pw'], True, t_b)
                # branch2: 1x1 -> dw (stride) -> 1x1   (basenetworks.py:214-226)
                t_c = tensor(h, w, hp)
                conv1x1(cur, 0, cols, lay.width, e['b2_pw1'], True, t_c)
                t_d = tensor(ho, wo, hp)
                dwconv(t_c, np.arange(bf), hp, e['b2_dw'], kk, st, pd, t_d)
                conv1x1(t_d, 0, np.arange(bf), hp, e['b2_pw2'], True, t_out, shuffle=(t_b, 0))
            else:
                assert lay.split and lay.half == bf
                # x1, x2 = x.chunk(2): x2 is the column window [bf, 2*bf) (basenetworks.py:234-236).  TMA needs a
                # 16-byte aligned start (32 bytes or more is faster), so the view begins at _view_start(bf) <= bf;
                # the leading columns are pass-through channels and get zero weights.
                a0 = _view_start(bf)
                lead = bf - a0
                t_c = tensor(h, w, hp)
                conv1x1(cur, a0, lead + np.arange(bf), lead + bf, e['b2_pw1'], True, t_c)
                t_d = tensor(ho, wo, hp)
                dwconv(t_c, np.arange(bf), hp, e['b2_dw'], kk, st, pd, t_d)
                conv1x1(t_d, 0, np.arange(bf), hp, e['b2_pw2'], True, t_out, shuffle=(cur, 0))
            cur, lay, h, w = t_out, out_lay, ho, wo
            block_outputs.append((cur, lay))
    w5, b5 = plan['conv5']
    c5 = w5.shape[0]
    t5 = tensor(h, w, pad16(c5))
    conv1x1(cur, 0, lay.cols(), lay.width, (w5, b5), True, t5)
    ops.append(_heads_op(plan['heads'], t5, c5))
    return tensors, ops, {'block_outputs': block_outputs, 'feature': (t5, _Layout(c5, split=False))}


def _heads_op(heads, t_in, k_cols):
    return {'kind': 'heads', 'in': t_in, 'k_cols': k_cols, 'upsample': int(heads[0].get('upsample', 1)),
            'n_fields': [hd['n_fields'] for hd in heads], 'n_comp': [hd['n_comp'] for hd in heads],
            'ops': [o for hd in heads for o in hd['ops']],
            'w': _f32(np.concatenate([_f32(hd['w']) for hd in heads], axis=0)),
            'b': _f32(np.concatenate([_f32(hd['b']) for hd in heads], axis=0))}


def _build_ops_resnet(plan, in_h, in_w):
    """torchvision BasicBlock / Bottleneck (eval): every conv+BN is one implicit-GEMM conv op; the residual
    add and the final ReLU of a block are fused into the epilogue of its last conv."""
    tensors, ops = [], []

    def tensor(h, w, c):
        tensors.append((h, w, c))
        return len(tensors) - 1

    def conv(tin, e, relu, tout, residual=-1):
        ops.append({'kind': 'conv', 'in': tin, 'in_off': 0, 'c_in': e['w'].shape[1], 'kernel': e['kernel'],
                    'stride': e['stride'], 'pad': e['pad'], 'n_out': e['w'].shape[0], 'w': _f32(e['w']),
                    'b': _f32(e['b']), 'relu': int(relu), 'out': tout, 'out_off': 0,
                    'residual': residual, 'residual_off': 0})

    def out_hw(h, w, e):
        return ((h + 2 * e['pad'] - e['kernel']) // e['stride'] + 1, (w + 2 * e['pad'] - e['kernel']) // e['stride'] + 1)

    inp = plan['input']
    k = inp['w'].shape[-1]
    h = (in_h + 2 * inp['pad'] - k) // inp['stride'] + 1
    w = (in_w + 2 * inp['pad'] - k) // inp['stride'] + 1
    c0 = inp['w'].shape[0]
    cur = tensor(h, w, pad16(c0))
    ops.append({'kind': 'input_conv', 'in_h': in_h, 'in_w': in_w, 'kernel': k, 'stride': inp['stride'],
                'pad': inp['pad'], 'c_out': c0, 'w': _f32(inp['w']), 'b': _f32(inp['b']), 'relu': 1, 'out': cur})
    c_cur = c0
    block_outputs = []
    for e in plan['blocks']:
        identity = cur
        hh, ww = h, w
        t_in = cur
        if e['downsample'] is not None:
            ds = e['downsample']
            dh, dw_ = out_hw(h, w, ds)
            identity = tensor(dh, dw_, pad16(ds['w'].shape[0]))
            conv(cur, ds, False, identity)
        n_convs = len(e['convs'])
        for ci, ce in enumerate(e['convs']):
            oh, ow = out_hw(hh, ww, ce)
            t_out = tensor(oh, ow, pad16(ce['w'].shape[0]))
            last = ci == n_convs - 1
            conv(t_in, ce, True, t_out, residual=identity if last else -1)
            t_in, hh, ww = t_out, oh, ow
        cur, h, w, c_cur = t_in, hh, ww, e['convs'][-1]['w'].shape[0]
        block_outputs.append((cur, _Layout(c_cur, split=False)))
    ops.append(_heads_op(plan['heads'], cur, c_cur))
    return tensors, ops, {'block_outputs': block_outputs, 'feature': (cur, _Layout(c_cur, split=False))}


def _build_ops_mobilenet(plan, in_h, in_w):
    """torchvision InvertedResidual (eval): expand 1x1 GEMM (+ activation), depthwise kxk (+ activation), then the
    linear projection -- a plain GEMM, a GEMM with the residual add fused (use_res_connect), or, behind a
    squeeze-excitation, the 'se_conv1x1' op (pooled sums from the depthwise kernel, per-image projection weights)."""
    tensors, ops = [], []

    def tensor(h, w, c):
        tensors.append((h, w, c))
        return len(tensors) - 1

    def out_hw(h, w, e):
        return ((h + 2 * e['pad'] - e['kernel']) // e['stride'] + 1, (w + 2 * e['pad'] - e['kernel']) // e['stride'] + 1)

    def conv1x1(tin, c_in, e, tout):
        ops.append({'kind': 'conv1x1', 'in': tin, 'in_off': 0, 'k_cols': c_in, 'n_out': e['w'].shape[0],
                    'w': _f32(e['w'].reshape(e['w'].shape[0], -1)), 'b': _f32(e['b']), 'relu': int(e['act']),
                    'out': tout, 'out_off': 0, 'shuffle_src': -1, 'shuffle_off': 0})

    inp = plan['input']
    h, w = out_hw(in_h, in_w, inp)
    c_cur = inp['w'].shape[0]
    cur = tensor(h, w, pad16(c_cur))
    ops.append({'kind': 'input_conv', 'in_h': in_h, 'in_w': in_w, 'kernel': inp['kernel'], 'stride': inp['stride'],
                'pad': inp['pad'], 'c_out': c_cur, 'w': _f32(inp['w']), 'b': _f32(inp['b']), 'relu': int(inp['act']),
                'out': cur})
    block_outputs = []
    for blk in plan['blocks']:
        x_in, t_in, c_in = cur, cur, c_cur
        if blk['expand'] is not None:
            c_in = blk['expand']['w'].shape[0]
            t_in = tensor(h, w, pad16(c_in))
            conv1x1(cur, c_cur, blk['expand'], t_in)
        dw = blk['dw']
        ho, wo = out_hw(h, w, dw)
        t_d = tensor(ho, wo, pad16(c_in))
        k = dw['kernel']
        ops.append({'kind': 'dwconv', 'in': t_in, 'in_off': 0, 'channels': c_in, 'kernel': k, 'stride': dw['stride'],
                    'pad': dw['pad'], 'w': _f32(dw['w'].reshape(c_in, k * k)), 'b': _f32(dw['b']),
                    'relu': int(dw['act']), 'out': t_d, 'out_off': 0})
        pr = blk['project']
        c_out = pr['w'].shape[0]
        t_o = tensor(ho, wo, pad16(c_out))
        res = x_in if blk['residual'] else -1
        wp = _f32(pr['w'].reshape(c_out, c_in))
        if blk['se'] is not None:
            se = blk['se']
            ops.append({'kind': 'se_conv1x1', 'in': t_d, 'channels': c_in, 'squeeze': se['w1'].shape[0],
                        'fc1_w': _f32(se['w1']), 'fc1_b': _f32(se['b1']), 'fc2_w': _f32(se['w2']),
                        'fc2_b': _f32(se['b2']), 'n_out': c_out, 'w': wp, 'b': _f32(pr['b']), 'out': t_o,
                        'residual': res})
        elif res >= 0:
            ops.append({'kind': 'conv', 'in': t_d, 'in_off': 0, 'c_in': c_in, 'kernel': 1, 'stride': 1, 'pad': 0,
                        'n_out': c_out, 'w': wp.reshape(c_out, c_in, 1, 1), 'b': _f32(pr['b']), 'relu': 0,
                        'out': t_o, 'out_off': 0, 'residual': res, 'residual_off': 0})
        else:
            conv1x1(t_d, c_in, pr, t_o)
        cur, c_cur, h, w = t_o, c_out, ho, wo
        block_outputs.append((cur, _Layout(c_cur, split=False)))
    last = plan['last']
    c_last = last['w'].shape[0]
    t_f = tensor(h, w, pad16(c_last))
    conv1x1(cur, c_cur, last, t_f)
    ops.append(_heads_op(plan['heads'], t_f, c_last))
    return tensors, ops, {'block_outputs': block_outputs, 'feature': (t_f, _Layout(c_last, split=False))}


class CompiledNet:
    """A plan compiled to libpifpaf_b200 ops for a fixed input size and maximum batch."""

    def __init__(self, plan, in_h, in_w, max_batch, device=0, layout=None, fuse_dw=None):
        self.lib = _lib.lib()
        self.device = int(device)
        self.max_batch = int(max_batch)
        self.in_h, self.in_w = int(in_h), int(in_w)
        if plan.get('kind') == 'shufflenetv2k':
            self.tensor_shapes, ops, self.info = build_ops(plan, self.in_h, self.in_w, layout=layout, fuse_dw=fuse_dw)
        else:
            self.tensor_shapes, ops, self.info = build_ops(plan, self.in_h, self.in_w)
        self.op_desc = [{k: v for k, v in o.items() if not isinstance(v, np.ndarray)} for o in ops]
        self.handle = ctypes.c_void_p()
        _lib.check(self.lib.pifpaf_net_create(ctypes.byref(self.handle), self.device, self.max_batch))
        self._emit(ops)
        self.flops_per_image = float(self.lib.pifpaf_net_flops_per_image(self.handle))
        self.num_ops = int(self.lib.pifpaf_net_num_ops(self.handle))
        self.heads = []
        for i, h in enumerate(plan['heads']):
            ptr = ctypes.c_void_p()
            nf, nc, hh, ww = (ctypes.c_int32() for _ in range(4))
            _lib.check(self.lib.pifpaf_net_head_output(self.handle, i, ctypes.byref(ptr), ctypes.byref(nf),
                                                       ctypes.byref(nc), ctypes.byref(hh), ctypes.byref(ww)))
            self.heads.append({'ptr': ptr.value, 'n_fields': nf.value, 'n_comp': nc.value,
                               'h': hh.value, 'w': ww.value, 'stride': h['stride']})

    def __del__(self):
        self.close()

    def close(self):
        """Free every device buffer of the net (idempotent)."""
        h, self.handle = getattr(self, 'handle', None), None
        if h:
            try:
                self.lib.pifpaf_net_destroy(h)
            except Exception:
                pass

    def set_head_buffers(self, n):
        """1: head outputs are valid until the next forward (default); 2: successive forwards alternate between two
        sets, so a decode of forward i may run concurrently with forward i+1."""
        _lib.check(self.lib.pifpaf_net_set_head_buffers(self.handle, int(n)))

    def set_sm_limit(self, n_sm):
        """Cap the persistent grids of the forward at n_sm SMs (0: all of them)."""
        _lib.check(self.lib.pifpaf_net_set_sm_limit(self.handle, int(n_sm)))

    def _emit(self, ops):
        L, H = self.lib, self.handle
        for (h, w, c) in self.tensor_shapes:
            tid = ctypes.c_int32(-1)
            _lib.check(L.pifpaf_net_tensor(H, h, w, c, ctypes.byref(tid)))
        for o in ops:
            if o['kind'] == 'input_conv':
                _lib.check(L.pifpaf_net_input_conv(H, o['in_h'], o['in_w'], o['kernel'], o['stride'], o['pad'],
                                                   o['c_out'], _ptr(o['w']), _ptr(o['b']), o['relu'], o['out']))
            elif o['kind'] == 'dw_conv1x1':
                pcs = np.ascontiguousarray(np.asarray(o['pieces'], dtype=np.int32).T)
                _lib.check(L.pifpaf_net_dw_conv1x1_scatter(
                    H, o['in'], o['in_off'], o['channels'], o['kernel'], o['stride'], o['pad'], _ptr(o['dw_w']),
                    _ptr(o['dw_b']), o['dw_relu'], o['n_out'], _ptr(o['w']), _ptr(o['b']), o['relu'], pcs.shape[1],
                    _ptr(pcs[0]), _ptr(pcs[1]), _ptr(pcs[2]), _ptr(pcs[3])))
            elif o['kind'] == 'conv1x1' and 'pieces' in o:
                pcs = np.ascontiguousarray(np.asarray(o['pieces'], dtype=np.int32).T)     # rows: col0, count, tensor, col
                _lib.check(L.pifpaf_net_conv1x1_scatter(H, o['in'], o['in_off'], o['k_cols'], o['n_out'],
                                                        _ptr(o['w']), _ptr(o['b']), o['relu'], pcs.shape[1],
                                                        _ptr(pcs[0]), _ptr(pcs[1]), _ptr(pcs[2]), _ptr(pcs[3])))
            elif o['kind'] == 'conv1x1':
                _lib.check(L.pifpaf_net_conv1x1(H, o['in'], o['in_off'], o['k_cols'], o['n_out'], _ptr(o['w']),
                                                _ptr(o['b']), o['relu'], o['out'], o['out_off'],
                                                o['shuffle_src'], o['shuffle_off']))
            elif o['kind'] == 'conv':
                _lib.check(L.pifpaf_net_conv(H, o['in'], o['in_off'], o['c_in'], o['kernel'], o['stride'], o['pad'],
                                             o['n_out'], _ptr(o['w']), _ptr(o['b']), o['relu'], o['out'],
                                             o['out_off'], o['residual'], o['residual_off']))
            elif o['kind'] == 'se_conv1x1':
                _lib.check(L.pifpaf_net_se_conv1x1(H, o['in'], o['channels'], o['squeeze'], _ptr(o['fc1_w']),
                                                   _ptr(o['fc1_b']), _ptr(o['fc2_w']), _ptr(o['fc2_b']), o['n_out'],
                                                   _ptr(o['w']), _ptr(o['b']), o['out'], o['residual']))
            elif o['kind'] == 'dwconv':
                _lib.check(L.pifpaf_net_dwconv(H, o['in'], o['in_off'], o['channels'], o['kernel'], o['stride'],
                                               o['pad'], _ptr(o['w']), _ptr(o['b']), o['relu'], o['out'], o['out_off']))
            elif o['kind'] == 'heads':
                n = len(o['n_fields'])
                nf = (ctypes.c_int32 * n)(*o['n_fields'])
                nc = (ctypes.c_int32 * n)(*o['n_comp'])
                ops_c = (ctypes.c_int32 * len(o['ops']))(*o['ops'])
                _lib.check(L.pifpaf_net_heads_upsampled(H, o['in'], o['k_cols'], n, nf, nc, ops_c, int(o.get('upsample', 1)),
                                                        _ptr(o['w']), _ptr(o['b'])))
            else:
                raise RuntimeError(o['kind'])

    # --- execution -----------------------------------------------------------
    def forward(self, image_batch, *, gemm_impl=0, stream=None):
        """Shell.forward: image_batch [B,3,H,W] float32 CUDA -> tuple of [B,F,comp,h,w] float32 CUDA views
        (valid until the next forward)."""
        if not image_batch.is_cuda or image_batch.dtype != torch.float32:
            raise RuntimeError('image_batch must be a float32 CUDA tensor')
        if image_batch.dim() != 4 or image_batch.shape[1] != 3 or tuple(image_batch.shape[2:]) != (self.in_h, self.in_w):
            raise RuntimeError(f'expected [B,3,{self.in_h},{self.in_w}]')
        b = int(image_batch.shape[0])
        if b > self.max_batch:
            raise RuntimeError('batch exceeds max_batch')
        image_batch = image_batch.contiguous()
        st = stream if stream is not None else torch.cuda.current_stream(image_batch.device)
        _lib.check(self.lib.pifpaf_net_forward(self.handle, image_batch.data_ptr(), b, int(gemm_impl),
                                               ctypes.c_void_p(st.cuda_stream)))
        self._keepalive = image_batch
        return self._head_views(b)

    def _head_views(self, b):
        outs = []
        for i, hd in enumerate(self.heads):
            ptr = ctypes.c_void_p()       # the buffer set the last forward wrote (set_head_buffers)
            _lib.check(self.lib.pifpaf_net_head_output(self.handle, i, ctypes.byref(ptr), None, None, None, None))
            arr = _DevArray(ptr.value, (b, hd['n_fields'], hd['n_comp'], hd['h'], hd['w']))
            outs.append(torch.as_tensor(arr, device=f'cuda:{self.device}'))
        return tuple(outs)

    def forward_features(self, features, *, gemm_impl=0, stream=None):
        """CompositeField4 heads alone (heads.py:330-378) on a given feature map: features [B,h,w,C] float32
        (host numpy or tensor; rounded to bf16 on upload) -> head outputs.  For plans of kind 'heads_only'
        (`heads_only_plan`): parity / accuracy tests feed the heads GEMM with controlled activations."""
        if self.op_desc[0]['kind'] != 'heads':
            raise RuntimeError('forward_features needs a heads_only plan')
        f = np.ascontiguousarray(features.cpu().numpy() if isinstance(features, torch.Tensor) else features,
                                 dtype=np.float32)
        b = int(f.shape[0])
        h, w, c = self.tensor_shapes[0]
        if f.shape[1:3] != (h, w) or f.shape[3] > c or b > self.max_batch:
            raise RuntimeError(f'expected features [B<={self.max_batch},{h},{w},<={c}]')
        padded = np.zeros((b, h, w, c), dtype=np.float32)
        padded[..., :f.shape[3]] = f
        _lib.check(self.lib.pifpaf_net_set_tensor(self.handle, 0, b, _ptr(padded), padded.size))
        st = stream if stream is not None else torch.cuda.current_stream(self.device)
        _lib.check(self.lib.pifpaf_net_forward(self.handle, None, b, int(gemm_impl), ctypes.c_void_p(st.cuda_stream)))
        return self._head_views(b)

    # the reference's eval preprocessing constants (transforms/__init__.py:26-33)
    IMAGE_MEAN = (0.485, 0.456, 0.406)
    IMAGE_STD = (0.229, 0.224, 0.225)

    def forward_uint8(self, image_batch, *, mean=IMAGE_MEAN, std=IMAGE_STD, gemm_impl=0, stream=None):
        """Shell.forward on raw images: image_batch [B,H,W,3] uint8 CUDA (HWC, as PIL / numpy hold them).  ToTensor
        and Normalize(mean, std) of the reference's EVAL_TRANSFORM are applied inside the stem kernel; the result
        equals forward() on the normalised float batch bit for bit."""
        if not image_batch.is_cuda or image_batch.dtype != torch.uint8:
            raise RuntimeError('image_batch must be a uint8 CUDA tensor')
        if image_batch.dim() != 4 or image_batch.shape[3] != 3 or tuple(image_batch.shape[1:3]) != (self.in_h, self.in_w):
            raise RuntimeError(f'expected [B,{self.in_h},{self.in_w},3]')
        b = int(image_batch.shape[0])
        if b > self.max_batch:
            raise RuntimeError('batch exceeds max_batch')
        image_batch = image_batch.contiguous()
        st = stream if stream is not None else torch.cuda.current_stream(image_batch.device)
        m = (ctypes.c_float * 3)(*[float(v) for v in mean])
        s = (ctypes.c_float * 3)(*[float(v) for v in std])
        _lib.check(self.lib.pifpaf_net_forward_u8(self.handle, image_batch.data_ptr(), b, m, s, int(gemm_impl),
                                                  ctypes.c_void_p(st.cuda_stream)))
        self._keepalive = image_batch
        return self._head_views(b)

    def forward_timed(self, image_batch, *, gemm_impl=0):
        """Profiling pass: per library op (ms, kind, flops, bytes); kind 0 input conv, 1 tcgen05 GEMM, 2 depthwise,
        3 fused depthwise -> GEMM, 4 squeeze-excitation (an 'se_conv1x1' op is two library ops: 4, then its GEMM)."""
        b, n = int(image_batch.shape[0]), self.num_ops
        ms = np.zeros((n,), dtype=np.float32)
        kind = np.zeros((n,), dtype=np.int32)
        flops = np.zeros((n,), dtype=np.float64)
        nbytes = np.zeros((n,), dtype=np.float64)
        st = torch.cuda.current_stream(image_batch.device)
        _lib.check(self.lib.pifpaf_net_forward_timed(self.handle, image_batch.contiguous().data_ptr(), b,
                                                     int(gemm_impl), ctypes.c_void_p(st.cuda_stream),
                                                     _ptr(ms), _ptr(kind), _ptr(flops), _ptr(nbytes)))
        return ms, kind, flops, nbytes

    def tap(self, tensor_id, batch):
        """Debug: activation tensor as float32 numpy [B,h,w,c_phys]."""
        h, w, c = self.tensor_shapes[tensor_id]
        out = np.empty((batch, h, w, c), dtype=np.float32)
        _lib.check(self.lib.pifpaf_net_tap_tensor(self.handle, tensor_id, batch, _ptr(out), out.size))
        return out
