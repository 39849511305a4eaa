"""Plain PyTorch fp32 restatement of the reference's MobileNet base networks (test infrastructure, not product code).

  MobileNetV2                          network/basenetworks.py:407-429   (stride 32, 1280 features)
  MobileNetV3 (large / small)          network/basenetworks.py:432-458   (stem stride set to 1: stride 16)
  factory entries                      network/factory.py:52-56

torchvision's constructors with weights=None (no download is ever attempted); the Shell and the CompositeField4 heads
are oracle/net_oracle.py's.  tests/test_mobilenet.py checks these against the reference's own classes through
tests/golden/reference_mobilenet.npz (tools/make_mobilenet_golden.py)."""
import torch

from oracle import net_oracle

MOBILENETS = ('mobilenetv3large', 'mobilenetv3small', 'mobilenetv2')


class MobileNetV2(torch.nn.Module):
    """basenetworks.py:407-429"""

    def __init__(self, name, torchvision_mobilenetv2, out_features=1280):
        super().__init__()
        self.name, self.stride, self.out_features = name, 32, out_features
        self.backbone = list(torchvision_mobilenetv2(weights=None).children())[0]    # classifier removed

    def forward(self, x):
        return self.backbone(x)


class MobileNetV3(torch.nn.Module):
    """basenetworks.py:432-458"""

    def __init__(self, name, torchvision_mobilenetv3, out_features=960):
        super().__init__()
        self.name, self.stride, self.out_features = name, 16, out_features
        self.backbone = list(torchvision_mobilenetv3(weights=None).children())[0]
        self.backbone[0][0].stride = torch.nn.modules.utils._pair(1)               # stem stride 1

    def forward(self, x):
        return self.backbone(x)


def make_base(base_name):
    import torchvision
    if base_name == 'mobilenetv2':
        return MobileNetV2('mobilenetv2', torchvision.models.mobilenet_v2)
    if base_name == 'mobilenetv3large':
        return MobileNetV3('mobilenetv3large', torchvision.models.mobilenet_v3_large)
    if base_name == 'mobilenetv3small':
        return MobileNetV3('mobilenetv3small', torchvision.models.mobilenet_v3_small, 576)
    raise ValueError(base_name)


def make_shell(base_name, n_keypoints=17, n_connections=19, seed=0, randomize_bn=True):
    """From-scratch eval Shell like oracle/net_oracle.make_shell: torchvision's init after torch.manual_seed(seed),
    randomised BatchNorm statistics so that BN folding is exercised, and random squeeze-excitation biases."""
    g = torch.Generator().manual_seed(seed)
    torch.manual_seed(seed)
    base = make_base(base_name)
    heads = [net_oracle.CompositeField4(net_oracle.HeadMeta.cif(n_keypoints), base.out_features),
             net_oracle.CompositeField4(net_oracle.HeadMeta.caf(n_connections), base.out_features)]
    shell = net_oracle.Shell(base, heads)
    net_oracle.model_defaults(shell)
    with torch.no_grad():
        if randomize_bn:
            for m in shell.modules():
                if isinstance(m, torch.nn.BatchNorm2d):
                    m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.1)
                    m.running_var.copy_(torch.rand(m.num_features, generator=g) * 0.5 + 0.75)
                    m.weight.data.copy_(torch.rand(m.num_features, generator=g) * 0.5 + 0.75)
                    m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.1)
        for m in base.modules():
            if hasattr(m, 'fc1') and hasattr(m, 'fc2'):          # torchvision initialises the SE biases to 0
                m.fc1.bias.copy_(torch.randn(m.fc1.bias.shape, generator=g) * 0.1)
                m.fc2.bias.copy_(torch.randn(m.fc2.bias.shape, generator=g) * 0.5)
    shell.eval()
    return shell
