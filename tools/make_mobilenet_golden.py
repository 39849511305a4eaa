"""Writes tests/golden/reference_mobilenet.npz: the reference's own basenetworks.MobileNetV2 / MobileNetV3 (pretrained
off, torchvision weights=None) carrying tests/mobilenet_oracle.py's seeded weights and randomised BatchNorm
statistics, on a seeded input: input and weight hashes, a seeded sample of the output elements and every channel's
mean (as oracle/make_golden.py stores them for resnet18).  Needs the reference sources:

    python tools/make_mobilenet_golden.py /path/to/openpifpaf/src/openpifpaf
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, 'tests')]

INPUT = (1, 3, 97, 129)          # the input image: torch.randn with seed 11
SAMPLE = 4096                    # output elements kept, seeded choice


def net_input():
    import torch
    return torch.randn(INPUT, generator=torch.Generator().manual_seed(11))


def sample_index(n_elems):
    return np.sort(np.random.default_rng(0).choice(n_elems, min(SAMPLE, n_elems), replace=False))


def weights_sha(module):
    from oracle import make_golden as mg
    return mg.sha(np.concatenate([t.detach().numpy().ravel() for t in module.state_dict().values()
                                  if t.dtype.is_floating_point]))


def main(src):
    import torch
    import torchvision
    import mobilenet_oracle
    from oracle import make_golden as mg, net_oracle
    _, base, _ = mg._reference_modules(src)
    # never let torchvision reach for pretrained weights
    base.MobileNetV2.pretrained = False
    base.MobileNetV3.pretrained = False
    ctors = {'mobilenetv2': lambda: base.MobileNetV2('mobilenetv2', torchvision.models.mobilenet_v2),
             'mobilenetv3large': lambda: base.MobileNetV3('mobilenetv3large', torchvision.models.mobilenet_v3_large),
             'mobilenetv3small': lambda: base.MobileNetV3('mobilenetv3small', torchvision.models.mobilenet_v3_small, 576)}
    data = {}
    x = net_input()
    for name in mobilenet_oracle.MOBILENETS:
        oracle = mobilenet_oracle.make_shell(name, seed=5).base_net
        ref = ctors[name]()
        ref.load_state_dict(oracle.state_dict())
        net_oracle.model_defaults(ref)           # network/nets.py:63-78, as the reference's factory applies it
        ref.eval()
        with torch.no_grad():
            out = ref(x).numpy()
        data.update({f'{name}_stride': ref.stride, f'{name}_shape': np.array(out.shape),
                     f'{name}_weights_sha256': weights_sha(oracle),
                     f'{name}_sample': out.reshape(-1)[sample_index(out.size)],
                     f'{name}_channel_mean': out[0].mean((1, 2))})
    data['input_sha256'] = mg.sha(x.numpy())
    path = os.path.join(ROOT, 'tests', 'golden', 'reference_mobilenet.npz')
    np.savez_compressed(path, **data)
    print(path, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
    main(sys.argv[1])
