"""Generate tests/golden/* from the UNMODIFIED reference (oracle/_ref, oracle/_ref_pkg).

Run where the reference sources exist (oracle/build_ref.py builds and stages them):
    python -m oracle.make_golden              # decoder_*.npz, cifdet_*.npz
    python -m oracle.make_golden reference    # reference_*.npz / .json
Each decoder fixture stores the generator arguments, the sha256 of the generated float32 fields
(openpifpaf_b200.synth is bit-reproducible, so inputs need not be stored), and the reference's
outputs on a FRESH CifCaf instance: annotations, ids, sorted seeds, per-connection CafScored
counts and a sha256 of the CifHr map.  The smallest case also stores the raw fields.
The reference_* fixtures hold what the reference computes in the cases tests/test_oracle.py,
test_network_lowering.py, test_preprocess.py and test_constants.py compare against.
TEST INFRASTRUCTURE."""
import hashlib
import importlib.util
import json
import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from openpifpaf_b200 import synth      # noqa: E402
from oracle import cifcaf as oc        # noqa: E402

CASES = [
    # name, workload, h, w, n_people, seed, n_distractors, stride, reference statics
    ('coco11_1p', 'cocokp', 11, 11, 1, 5, 0, 16, {}),
    ('coco11_2p_d3', 'cocokp', 11, 11, 2, 6, 3, 16, {}),
    ('coco41_poisson_s0', 'cocokp', 41, 41, None, 0, 10, 16, {}),
    ('coco41_poisson_s1', 'cocokp', 41, 41, None, 1, 10, 16, {}),
    ('coco31x41_3p', 'cocokp', 31, 41, 3, 12, 0, 16, {}),
    ('coco51_5p_stride8', 'cocokp', 51, 51, 5, 14, 4, 8, {}),
    ('crowd30', 'cocokp', 41, 41, 30, 7, 20, 16, {}),
    ('greedy_4p', 'cocokp', 41, 41, 4, 13, 0, 16, {'greedy': True}),
    ('force_complete_3p', 'cocokp', 41, 41, 3, 11, 5, 16,
     {'force_complete': True, 'keypoint_threshold': 0.0, 'keypoint_threshold_rel': 0.0,
      'nms_keypoint_threshold': 0.0, 'nms_instance_threshold': 0.0}),
    ('wholebody_1p', 'wholebody', 41, 41, 1, 21, 0, 16, {}),
    ('wholebody_4p', 'wholebody', 41, 41, 4, 22, 0, 16, {}),
]


DET_CASES = [
    # name, n_categories, h, w, n_objects, seed, n_distractors, stride
    ('det11_3cat_1', 3, 11, 11, 1, 2, 2, 16),
    ('det41_80cat_6', 80, 41, 41, 6, 0, 4, 16),
    ('det21x33_80cat_3', 80, 21, 33, 3, 1, 4, 16),
    ('det51_80cat_150', 80, 51, 51, 150, 4, 10, 8),         # hits max_detections_before_nms = 120
]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def main():
    out_dir = os.path.join(ROOT, 'tests', 'golden')
    os.makedirs(out_dir, exist_ok=True)
    for name, workload, h, w, n_people, seed, n_dis, stride, statics in CASES:
        f = synth.make_fields(workload, h, w, n_people, seed, n_dis)
        oc.ref_configure(**statics)
        ann, ids, taps = oc.ref_decode(f['cif'], stride, f['caf'], stride, f['skeleton'], f['n_keypoints'], taps=True)
        data = dict(
            workload=workload, h=h, w=w, n_people=-1 if n_people is None else n_people, seed=seed,
            n_distractors=n_dis, stride=stride,
            statics_keys=np.array(list(statics.keys()), dtype='U64'),
            statics_vals=np.array([float(v) for v in statics.values()], dtype=np.float64),
            fields_sha256=synth.fields_digest(f['cif'], f['caf']),
            annotations=ann, ids=ids,
            seeds_f=taps['seeds_f'], seeds_vxys=taps['seeds_vxys'],
            n_fwd=np.array([len(x) for x in taps['fwd']], dtype=np.int64),
            n_bwd=np.array([len(x) for x in taps['bwd']], dtype=np.int64),
            fwd_sha256=sha(np.concatenate([x.reshape(-1, 7) for x in taps['fwd']])),
            bwd_sha256=sha(np.concatenate([x.reshape(-1, 7) for x in taps['bwd']])),
            cifhr_sha256=sha(taps['cifhr']), cifhr_sum=float(taps['cifhr'].astype(np.float64).sum()),
        )
        if name == 'coco11_1p':
            data['cif'] = f['cif']
            data['caf'] = f['caf']
        path = os.path.join(out_dir, f'decoder_{name}.npz')
        np.savez_compressed(path, **data)
        print(name, 'N =', len(ann), 'seeds =', len(taps['seeds_f']), os.path.getsize(path), 'bytes')
    oc.ref_configure()
    # CifDet (csrc/src/cifdet.cpp): raw output of a FRESH torch.classes.openpifpaf_decoder.CifDet instance
    for name, n_cat, h, w, n_obj, seed, n_dis, stride in DET_CASES:
        f = synth.make_det_fields(n_cat, h, w, n_obj, seed, n_dis)
        cats, scores, boxes = oc.ref_decode_det(f['field'], stride)
        path = os.path.join(out_dir, f'cifdet_{name}.npz')
        np.savez_compressed(path, n_categories=n_cat, h=h, w=w, n_objects=n_obj, seed=seed, n_distractors=n_dis,
                            stride=stride, field_sha256=sha(f['field']), categories=cats, scores=scores, boxes=boxes)
        print(name, 'N =', len(cats), os.path.getsize(path), 'bytes')


# ---------------------------------------------------------------- reference_* fixtures
# inputs of the cases (the tests draw the same ones)
LIVE_CIFCAF_SEEDS = range(4)            # make_fields('cocokp', 21, 27, None, 100 + s, n_distractors=4)
LIVE_CIFDET_SEEDS = range(3)            # make_det_fields(80, 27, 21, 5 + 20 * s, 200 + s, n_distractors=6)
NET_INPUT = dict(shufflenetv2k16=(97, 113, 3), resnet18=(161, 161, 4))      # h, w, seed of the input image
RESNET_SAMPLE = 4096                    # output elements of resnet18 kept (of 61952), seeded choice


def live_cifcaf_fields(s):
    return synth.make_fields('cocokp', 21, 27, None, 100 + s, n_distractors=4)


def live_cifdet_field(s):
    return synth.make_det_fields(80, 27, 21, 5 + 20 * s, 200 + s, n_distractors=6)['field']


def net_input(name):
    import torch
    h, w, seed = NET_INPUT[name]
    return torch.randn(1, 3, h, w, generator=torch.Generator().manual_seed(seed))


def resnet_sample_index():
    return np.sort(np.random.default_rng(0).choice(512 * 11 * 11, RESNET_SAMPLE, replace=False))


def initial_annotations_fields():
    return synth.make_fields('cocokp', 41, 41, 3, 31)


def blend_caf():
    rng = np.random.default_rng(0)
    return rng.random((50, 7)).astype(np.float32) * np.array([1, 40, 40, 40, 40, 8, 8], dtype=np.float32)


def _reference_modules(src):
    """basenetworks / heads / headmeta of the reference loaded by path, without running the package __init__."""
    top = types.ModuleType('refpifpaf')
    top.__path__ = [src]
    sys.modules['refpifpaf'] = top
    net_pkg = types.ModuleType('refpifpaf.network')
    net_pkg.__path__ = [os.path.join(src, 'network')]
    sys.modules['refpifpaf.network'] = net_pkg

    def load(name, path):
        spec = importlib.util.spec_from_file_location(name, path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
        return mod

    headmeta = load('refpifpaf.headmeta', os.path.join(src, 'headmeta.py'))
    base = load('refpifpaf.network.basenetworks', os.path.join(src, 'network', 'basenetworks.py'))
    heads = load('refpifpaf.network.heads', os.path.join(src, 'network', 'heads.py'))
    return headmeta, base, heads


def reference_oracle_cases(out_dir):
    """the reference decoder on the cases of the oracle's live comparisons (tests/test_oracle.py)"""
    import torch
    data = {}
    oc.ref_configure()
    for s in LIVE_CIFCAF_SEEDS:
        f = live_cifcaf_fields(s)
        ann, ids, t = oc.ref_decode(f['cif'], 16, f['caf'], 16, f['skeleton'], 17, taps=True)
        data.update({f'cifcaf{s}_fields_sha256': synth.fields_digest(f['cif'], f['caf']),
                     f'cifcaf{s}_cifhr_sha256': sha(t['cifhr']), f'cifcaf{s}_seeds_vxys': t['seeds_vxys'],
                     f'cifcaf{s}_n_fwd': np.array([len(x) for x in t['fwd']], dtype=np.int64),
                     f'cifcaf{s}_n_bwd': np.array([len(x) for x in t['bwd']], dtype=np.int64),
                     f'cifcaf{s}_fwd_sha256': sha(np.concatenate([x.reshape(-1, 7) for x in t['fwd']])),
                     f'cifcaf{s}_bwd_sha256': sha(np.concatenate([x.reshape(-1, 7) for x in t['bwd']])),
                     f'cifcaf{s}_annotations': ann, f'cifcaf{s}_ids': ids})
    f = initial_annotations_fields()
    base, _ = oc.ref_decode(f['cif'], 16, f['caf'], 16, f['skeleton'], 17)
    init = base[:1].copy()
    init[0, 5:] = 0.0          # keep a few joints of the first person, let the decoder regrow the rest
    init_ids = np.array([42], dtype=np.int64)
    ann, ids = oc.ref_decode(f['cif'], 16, f['caf'], 16, f['skeleton'], 17, initial_annotations=init, initial_ids=init_ids)
    data.update(init_fields_sha256=synth.fields_digest(f['cif'], f['caf']), init_annotations=init, init_ids=init_ids,
                init_result_annotations=ann, init_result_ids=ids)
    caf = blend_caf()
    for only_max in (False, True):
        want = torch.ops.openpifpaf_decoder.grow_connection_blend(torch.from_numpy(caf), 20.0, 20.0, 30.0, 1.0, only_max)
        data[f'blend_only_max{int(only_max)}'] = np.array(list(want), dtype=np.float64)
    for s in LIVE_CIFDET_SEEDS:
        field = live_cifdet_field(s)
        cats, scores, boxes = oc.ref_decode_det(field, 16)
        data.update({f'cifdet{s}_field_sha256': sha(field), f'cifdet{s}_categories': cats,
                     f'cifdet{s}_scores': scores, f'cifdet{s}_boxes': boxes})
    np.savez_compressed(os.path.join(out_dir, 'reference_oracle_cases.npz'), **data)


def reference_networks(out_dir, src):
    """the reference's own modules carrying oracle/net_oracle.py's weights (tests/test_network_lowering.py)"""
    import torch
    import torchvision
    from oracle import net_oracle
    headmeta, base, heads = _reference_modules(src)
    data = {}
    # shufflenetv2k16 + CompositeField4 heads, the oracle's randomised weights (make_shell seed 3)
    ref_base = base.ShuffleNetV2K('shufflenetv2k16', [4, 8, 4], [24, 348, 696, 1392, 1392])
    kps = [str(i) for i in range(17)]
    cif = headmeta.Cif('cif', 'cocokp', keypoints=kps, sigmas=[0.1] * 17)
    caf = headmeta.Caf('caf', 'cocokp', keypoints=kps, sigmas=[0.1] * 17, skeleton=[(1, 2)] * 19)
    ref_heads = [heads.CompositeField4(cif, 1392), heads.CompositeField4(caf, 1392)]
    oracle = net_oracle.make_shell('shufflenetv2k16', seed=3)
    ref_base.load_state_dict(oracle.base_net.state_dict())
    for rh, oh in zip(ref_heads, oracle.head_nets):
        rh.load_state_dict(oh.state_dict())
        rh.eval()
    net_oracle.model_defaults(ref_base)
    ref_base.eval()
    x = net_input('shufflenetv2k16')
    with torch.no_grad():
        feat = ref_base(x)
        data['shufflenetv2k16_cif'], data['shufflenetv2k16_caf'] = [rh(feat).numpy() for rh in ref_heads]
    data['shufflenetv2k16_input_sha256'] = sha(x.numpy())
    # resnet18 backbone (max-pool removed, stride 16), torchvision's init drawn after torch.manual_seed(0)
    base.Resnet.pretrained = False
    ref = base.Resnet('resnet18', lambda pretrained: torchvision.models.resnet18(weights=None), 512)
    torch.manual_seed(0)
    oracle = net_oracle.make_base('resnet18')
    ref.load_state_dict(oracle.state_dict())
    ref.eval()
    x = net_input('resnet18')
    with torch.no_grad():
        out = ref(x).numpy()
    data.update(resnet18_stride=ref.stride, resnet18_shape=np.array(out.shape), resnet18_input_sha256=sha(x.numpy()),
                resnet18_sample=out.reshape(-1)[resnet_sample_index()], resnet18_channel_mean=out[0].mean((1, 2)),
                resnet18_weights_sha256=sha(np.concatenate([p.detach().numpy().ravel() for p in oracle.parameters()])))
    np.savez_compressed(os.path.join(out_dir, 'reference_networks.npz'), **data)


TRANSFORM_CASES = ((427, 640, 641, True), (480, 360, 321, True), (333, 500, 385, False), (200, 300, None, False))


def reference_transforms(out_dir):
    """the reference's own Predictor preprocessing (Pillow path) and Annotation methods (tests/test_preprocess.py)"""
    import torch
    import PIL.Image
    from oracle import ref_arm
    openpifpaf = ref_arm.import_reference()
    from openpifpaf import transforms
    import openpifpaf.transforms.scale as scale_mod
    scale_mod.cv2 = None                         # the documented Pillow path (transforms/scale.py:56-59)
    from openpifpaf.plugins.coco.constants import COCO_KEYPOINTS, COCO_PERSON_SKELETON, COCO_PERSON_SCORE_WEIGHTS
    rng = np.random.default_rng(0)
    cases = []
    for (h, w, long_edge, batched) in TRANSFORM_CASES:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        pre = [transforms.NormalizeAnnotations()]
        if long_edge:
            pre.append(transforms.RescaleAbsolute(long_edge, fast=True))
        pre.append(transforms.CenterPad(long_edge) if batched else transforms.CenterPadTight(16))
        torch.manual_seed(3)
        image, _, meta = transforms.Compose(pre)(PIL.Image.fromarray(img), [], None)
        image = np.asarray(image)
        ch, cw = image.shape[:2]
        dec = rng.random((4, 17, 4)).astype(np.float32) * np.array([1, cw, ch, 9], dtype=np.float32)
        dec[1, 5:11, 0] = 0.0
        anns = []
        for i in range(4):
            a = openpifpaf.Annotation(COCO_KEYPOINTS, COCO_PERSON_SKELETON, score_weights=COCO_PERSON_SCORE_WEIGHTS)
            a.data[:, :2] = dec[i, :, 1:3]
            a.data[:, 2] = dec[i, :, 0]
            a.joint_scales[:] = dec[i, :, 3]
            b = a.inverse_transform(meta)
            anns.append({'data': b.data.astype(np.float64).tolist(),
                         'joint_scales': np.asarray(b.joint_scales, dtype=np.float64).tolist(),
                         'json_data': b.json_data()})
        cases.append({'h': h, 'w': w, 'long_edge': long_edge, 'batched': batched,
                      'image_shape': list(image.shape), 'image_sha256': sha(image),
                      'meta': {k: np.asarray(meta[k], dtype=np.float64).tolist()
                               for k in ('offset', 'scale', 'valid_area', 'width_height')},
                      'annotations': anns})
    with open(os.path.join(out_dir, 'reference_transforms.json'), 'w') as f:
        json.dump({'score_weights': list(COCO_PERSON_SCORE_WEIGHTS), 'cases': cases}, f)


def reference_skeletons(out_dir):
    """the skeletons of the reference's coco and wholebody plugins (tests/test_constants.py)"""
    from oracle import ref_arm
    ref_arm.import_reference()
    from openpifpaf.plugins.coco.constants import COCO_PERSON_SKELETON
    from openpifpaf.plugins.wholebody.constants import WHOLEBODY_SKELETON
    with open(os.path.join(out_dir, 'reference_skeletons.json'), 'w') as f:
        json.dump({'COCO_PERSON_SKELETON': [list(e) for e in COCO_PERSON_SKELETON],
                   'WHOLEBODY_SKELETON': [list(e) for e in WHOLEBODY_SKELETON]}, f)


def main_reference():
    import subprocess
    from oracle import build_ref
    out_dir = os.path.join(ROOT, 'tests', 'golden')
    build_ref.stage_package()
    reference_oracle_cases(out_dir)
    reference_networks(out_dir, build_ref.REF_PY)
    # the staged package loads the same extension under another path: torch refuses a second registration of its
    # operators in one process
    subprocess.check_call([sys.executable, '-m', 'oracle.make_golden', 'reference-package'], cwd=ROOT)
    for name in sorted(os.listdir(out_dir)):
        if name.startswith('reference_'):
            print(name, os.path.getsize(os.path.join(out_dir, name)), 'bytes')


if __name__ == '__main__':
    if sys.argv[1:] == ['reference']:
        main_reference()
    elif sys.argv[1:] == ['reference-package']:
        reference_transforms(os.path.join(ROOT, 'tests', 'golden'))
        reference_skeletons(os.path.join(ROOT, 'tests', 'golden'))
    else:
        main()
