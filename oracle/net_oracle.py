"""oracle/net_oracle.py -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Plain PyTorch fp32 restatement of the reference's network forward for the hot
path (paths relative to /root/reference/src/openpifpaf/):

  Shell.forward                       network/nets.py:35-48
  ShuffleNetV2K / InvertedResidualK   network/basenetworks.py:186-355
  factory configs                     network/factory.py:68-79
  CompositeField4 (eval, in-place)    network/heads.py:272-378
  index_field_torch                   network/heads.py:16-28
  model_defaults (BN eps >= 1e-3)     network/nets.py:63-78

Attribute names and state_dict keys equal the reference's, so a reference
`Shell` state_dict loads here unchanged; tests/test_network_lowering.py
(test_oracle_net_equals_reference_modules, test_oracle_resnet_equals_reference_module) checks the
two produce identical fields, against the reference modules' outputs stored by
oracle/make_golden.py.  It is the fp32
numerics reference for the CUDA kernels and the "port" CPU baseline of bench.py.
"""
import torch

SHUFFLENETV2K_CONFIGS = {
    # network/factory.py:68-79
    'shufflenetv2k16': ([4, 8, 4], [24, 348, 696, 1392, 1392]),
    'shufflenetv2k20': ([5, 10, 5], [32, 512, 1024, 2048, 2048]),
    'shufflenetv2k30': ([8, 16, 6], [32, 512, 1024, 2048, 2048]),
}


def channel_shuffle(x, groups):
    """torchvision.models.shufflenetv2.channel_shuffle (called at basenetworks.py:240)."""
    b, c, h, w = x.shape
    x = x.view(b, groups, c // groups, h, w)
    x = torch.transpose(x, 1, 2).contiguous()
    return x.view(b, c, h, w)


class InvertedResidualK(torch.nn.Module):
    """basenetworks.py:186-242"""

    def __init__(self, inp, oup, first_in_stage, *, stride=1, kernel_size=5):
        super().__init__()
        self.first_in_stage = first_in_stage
        bf = oup // 2
        pad = (kernel_size - 1) // 2
        bn, relu, conv = torch.nn.BatchNorm2d, (lambda: torch.nn.ReLU(inplace=True)), torch.nn.Conv2d
        self.branch1 = None
        if first_in_stage:
            self.branch1 = torch.nn.Sequential(
                conv(inp, inp, kernel_size, stride, pad, bias=False, groups=inp), bn(inp),
                conv(inp, bf, 1, 1, 0, bias=False), bn(bf), relu())
        self.branch2 = torch.nn.Sequential(
            conv(inp if first_in_stage else bf, bf, 1, 1, 0, bias=False), bn(bf), relu(),
            conv(bf, bf, kernel_size, stride, pad, bias=False, groups=bf), bn(bf),
            conv(bf, bf, 1, 1, 0, bias=False), bn(bf), relu())

    def forward(self, x):
        if self.branch1 is None:
            x1, x2 = x.chunk(2, dim=1)
            out = torch.cat((x1, self.branch2(x2)), dim=1)
        else:
            out = torch.cat((self.branch1(x), self.branch2(x)), dim=1)
        return channel_shuffle(out, 2)


class ShuffleNetV2K(torch.nn.Module):
    """basenetworks.py:245-355 (default configuration: no input_conv2, no dilation, conv5 as conv)."""

    def __init__(self, name, stages_repeats, stages_out_channels):
        super().__init__()
        self.name = name
        self.stride = 16
        self.out_features = stages_out_channels[-1]
        c0 = stages_out_channels[0]
        self.input_block = torch.nn.Sequential(torch.nn.Sequential(
            torch.nn.Conv2d(3, c0, 3, 2, 1, bias=False), torch.nn.BatchNorm2d(c0), torch.nn.ReLU(inplace=True)))
        stages = []
        cin = c0
        for repeats, cout in zip(stages_repeats, stages_out_channels[1:4]):
            seq = [InvertedResidualK(cin, cout, True, stride=2)]
            seq += [InvertedResidualK(cout, cout, False) for _ in range(repeats - 1)]
            stages.append(torch.nn.Sequential(*seq))
            cin = cout
        self.stage2, self.stage3, self.stage4 = stages
        cl = stages_out_channels[-1]
        self.conv5 = torch.nn.Sequential(
            torch.nn.Conv2d(cin, cl, 1, 1, 0, bias=False), torch.nn.BatchNorm2d(cl), torch.nn.ReLU(inplace=True))

    def forward(self, x):
        x = self.input_block(x)
        x = self.stage2(x)
        x = self.stage3(x)
        x = self.stage4(x)
        return self.conv5(x)


class Resnet(torch.nn.Module):
    """basenetworks.py:71-150 in its default configuration: torchvision ResNet with the max-pool removed
    (pool0_stride = 0 -> stride 16), no dilation, all four blocks."""

    def __init__(self, name, torchvision_resnet, out_features=2048):
        super().__init__()
        modules = list(torchvision_resnet(weights=None).children())
        self.name = name
        self.stride = 16
        self.out_features = out_features
        self.input_block = torch.nn.Sequential(*modules[:3])       # conv1, bn1, relu (max-pool popped, :86-93)
        self.block2, self.block3, self.block4, self.block5 = modules[4], modules[5], modules[6], modules[7]

    def forward(self, x):
        x = self.input_block(x)
        x = self.block2(x)
        x = self.block3(x)
        x = self.block4(x)
        return self.block5(x)


def make_base(base_name):
    import torchvision
    if base_name in SHUFFLENETV2K_CONFIGS:
        repeats, channels = SHUFFLENETV2K_CONFIGS[base_name]
        return ShuffleNetV2K(base_name, repeats, channels)
    if base_name == 'resnet18':
        return Resnet('resnet18', torchvision.models.resnet18, 512)          # network/factory.py:57
    if base_name == 'resnet50':
        return Resnet('resnet50', torchvision.models.resnet50)               # network/factory.py:58
    raise ValueError(base_name)


class HeadMeta:
    """The subset of headmeta.Cif / headmeta.Caf (headmeta.py:12-113) the forward pass needs."""

    def __init__(self, name, n_fields, n_confidences, n_vectors, n_scales, vector_offsets):
        self.name = name
        self.n_fields = n_fields
        self.n_confidences = n_confidences
        self.n_vectors = n_vectors
        self.n_scales = n_scales
        self.vector_offsets = tuple(vector_offsets)
        self.upsample_stride = 1
        self.head_index = None
        self.base_stride = None

    @property
    def stride(self):
        return self.base_stride // self.upsample_stride

    @staticmethod
    def cif(n_keypoints):
        return HeadMeta('cif', n_keypoints, 1, 1, 1, [True])                # headmeta.py:44-47

    @staticmethod
    def caf(n_connections):
        return HeadMeta('caf', n_connections, 1, 2, 2, [True, True])         # headmeta.py:74-77


class CompositeField4(torch.nn.Module):
    """heads.py:272-378, eval + inplace_ops branch, upsample_stride 1."""

    def __init__(self, meta, in_features):
        super().__init__()
        self.meta = meta
        self.n_components = 1 + meta.n_confidences + meta.n_vectors * 2 + meta.n_scales
        self.conv = torch.nn.Conv2d(in_features, meta.n_fields * self.n_components, 1)

    def forward(self, x):
        m = self.meta
        x = self.conv(x)
        b, _, h, w = x.shape
        x = x.view(b, m.n_fields, self.n_components, h, w)
        torch.sigmoid_(x[:, :, 1:1 + m.n_confidences])
        index_field = torch.empty((2, h, w), device=x.device, dtype=x.dtype)
        index_field[0] = torch.arange(w, device=x.device)
        index_field[1] = torch.arange(h, device=x.device).unsqueeze(1)
        first_reg = 1 + m.n_confidences
        for i, do_offset in enumerate(m.vector_offsets):
            if do_offset:
                x[:, :, first_reg + i * 2:first_reg + (i + 1) * 2].add_(index_field)
        first_scale = 1 + m.n_confidences + m.n_vectors * 2
        scales = x[:, :, first_scale:first_scale + m.n_scales]
        scales[:] = torch.nn.functional.softplus(scales)
        return x


class Shell(torch.nn.Module):
    """network/nets.py:7-48"""

    def __init__(self, base_net, head_nets):
        super().__init__()
        self.base_net = base_net
        self.head_nets = torch.nn.ModuleList(head_nets)
        for i, hn in enumerate(self.head_nets):
            hn.meta.head_index = i
            hn.meta.base_stride = base_net.stride

    @property
    def head_metas(self):
        return [hn.meta for hn in self.head_nets]

    def forward(self, image_batch):
        x = self.base_net(image_batch)
        return tuple(hn(x) for hn in self.head_nets)


def model_defaults(net):
    """network/nets.py:63-89"""
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.eps = max(m.eps, 1e-3)
            m.momentum = 0.01


def make_shell(base_name='shufflenetv2k16', n_keypoints=17, n_connections=19, seed=0, randomize_bn=True,
               he_init=False):
    """From-scratch Shell like network/factory.py:276-295 (eval mode).  randomize_bn gives the BatchNorm
    layers non-trivial running statistics/affine parameters so that BN folding is actually exercised.
    he_init re-draws every backbone convolution with std sqrt(2 / fan_in): with torch's default init (gain
    1/sqrt(3)) and eval-mode BatchNorm the signal of a 58-layer ShuffleNetV2K dies out -- its features are the same
    for any input to 7 digits (measured) -- whereas the variance-preserving init keeps them input dependent
    (std over positions ~ 0.45 of the rms, effective rank ~230 at 21x21), like a trained network's."""
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    base = make_base(base_name)
    heads = [CompositeField4(HeadMeta.cif(n_keypoints), base.out_features),
             CompositeField4(HeadMeta.caf(n_connections), base.out_features)]
    shell = Shell(base, heads)
    model_defaults(shell)
    if randomize_bn:
        for m in shell.modules():
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
                m.running_var.copy_(torch.rand(m.num_features, generator=g) * 0.5 + 0.75)
                m.weight.data.copy_(torch.rand(m.num_features, generator=g) * 0.5 + 0.75)
                m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)
    if he_init:
        with torch.no_grad():
            for m in shell.base_net.modules():
                if isinstance(m, torch.nn.Conv2d):
                    fan_in = m.weight.shape[1] * m.weight.shape[2] * m.weight.shape[3]
                    m.weight.copy_(torch.randn(m.weight.shape, generator=g) * (2.0 / fan_in) ** 0.5)
    shell.eval()
    return shell
