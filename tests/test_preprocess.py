"""Image preprocessing (SURVEY.md 8f rank 2).

CPU: the restatement of Pillow's ImagingResample (coefficient tables + integer arithmetic) against PIL.Image.resize
itself -- Pillow is the third-party dependency the reference resizes with (transforms/scale.py:56-59); the meta dicts
and the batched inverse_transform / json_data against the reference's own transforms / Annotation (their results
stored by oracle/make_golden.py).  GPU: the kernels against PIL + torchvision's pad, and the whole raw-image path."""
import json
import os

import numpy as np
import pytest
import torch

from helpers import GOLDEN_DIR
from openpifpaf_b200 import preprocess as pp
from oracle import make_golden as mg

SIZES = [(480, 640, 641, 481), (375, 500, 321, 241), (100, 37, 161, 435), (600, 800, 400, 300), (33, 33, 33, 65),
         (720, 1280, 641, 360), (50, 50, 50, 50), (427, 640, 640, 427), (2, 3, 7, 5), (1080, 1920, 321, 180)]


@pytest.mark.parametrize('h,w,tw,th', SIZES)
def test_pillow_bilinear_restatement_is_bit_exact(h, w, tw, th):
    PIL = pytest.importorskip('PIL.Image')
    img = np.random.default_rng(h * 7 + w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    want = np.asarray(PIL.fromarray(img).resize((tw, th), PIL.BILINEAR))
    np.testing.assert_array_equal(pp.resize_bilinear_reference(img, tw, th), want)


def test_coefficient_tables_are_normalised():
    for n_in, n_out in ((640, 641), (1280, 321), (37, 161)):
        bounds, kk = pp.pil_bilinear_coeffs(n_in, n_out)
        assert bounds.shape == (n_out, 2) and (bounds[:, 0] >= 0).all() and (bounds[:, 0] + bounds[:, 1] <= n_in).all()
        assert np.abs(kk.sum(axis=1) - (1 << pp.PRECISION_BITS)).max() <= kk.shape[1]      # rounding of each tap


def test_inverse_transform_and_json_batch_forms():
    """array forms == per-annotation arithmetic of annotation.py:121-214, written out (numpy-2 roundings)"""
    rng = np.random.default_rng(1)
    ann = rng.random((5, 17, 4)).astype(np.float32) * np.array([1, 600, 400, 9], dtype=np.float32)
    ann[2, 3:9, 0] = 0.0
    meta = pp.reference_meta(640, 427, 641, 428, np.asarray(pp.center_pad_ltrb(641, 428, 641, 641)))
    data, scales = pp.inverse_transform_batch(ann, meta)
    for i in range(5):
        d = np.stack([ann[i, :, 1], ann[i, :, 2], ann[i, :, 0]], axis=1).astype(np.float32)
        d[:, 0] += meta['offset'][0]
        d[:, 1] += meta['offset'][1]
        d[:, 0] = d[:, 0] / meta['scale'][0]
        d[:, 1] = d[:, 1] / meta['scale'][1]
        s = ann[i, :, 3].copy()
        s /= meta['scale'][0]
        np.testing.assert_array_equal(data[i], d)
        np.testing.assert_array_equal(scales[i], s)
    js = pp.json_data_batch(data, scales)
    assert len(js) == 5 and len(js[0]['keypoints']) == 51 and js[0]['score'] >= 0.001


def test_meta_and_annotations_equal_reference_transforms():
    """the reference's own Predictor preprocessing (PIL path) and Annotation methods, stored by oracle/make_golden.py"""
    import hashlib
    with open(os.path.join(GOLDEN_DIR, 'reference_transforms.json')) as f:
        golden = json.load(f)
    cases, score_weights = golden['cases'], golden['score_weights']
    assert [(c['h'], c['w'], c['long_edge'], c['batched']) for c in cases] == list(mg.TRANSFORM_CASES)
    rng = np.random.default_rng(0)
    for (h, w, long_edge, batched), ref in zip(mg.TRANSFORM_CASES, cases):
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        torch.manual_seed(3)
        fill = int(torch.randint(0, 255, (1,)).item())
        g = pp.GpuPreprocess.__new__(pp.GpuPreprocess)          # host logic only (no GPU here)
        g.long_edge, g.batched, g.multiple = long_edge, batched, 16
        (tw, th, ltrb, (cw, ch)), = g.plan([(w, h)])[0]
        assert ref['image_shape'] == [ch, cw, 3], (ref['image_shape'], cw, ch)
        canvas = np.empty((ch, cw, 3), dtype=np.uint8)
        canvas[:] = (fill, fill, fill) if batched else pp.TIGHT_PAD_FILL
        canvas[ltrb[1]:ltrb[1] + th, ltrb[0]:ltrb[0] + tw] = pp.resize_bilinear_reference(img, tw, th)
        assert hashlib.sha256(canvas.tobytes()).hexdigest() == ref['image_sha256'], 'resized + padded image differs'
        mine = pp.reference_meta(w, h, tw, th, np.asarray(ltrb))
        for k in ('offset', 'scale', 'valid_area', 'width_height'):
            assert np.array_equal(np.asarray(ref['meta'][k], dtype=np.float64), np.asarray(mine[k], dtype=np.float64)), \
                (k, ref['meta'][k], mine[k])
        # annotations: inverse_transform + json_data
        dec = rng.random((4, 17, 4)).astype(np.float32) * np.array([1, cw, ch, 9], dtype=np.float32)
        dec[1, 5:11, 0] = 0.0
        data, scales = pp.inverse_transform_batch(dec, mine)
        js = pp.json_data_batch(data, scales, score_weights=score_weights)
        for i, b in enumerate(ref['annotations']):
            assert np.array_equal(np.asarray(b['data'], dtype=np.float32), data[i])
            assert np.array_equal(np.asarray(b['joint_scales'], dtype=np.float32), scales[i])
            assert b['json_data'] == js[i], (b['json_data'], js[i])


@pytest.mark.gpu
def test_gpu_resize_pad_equals_pillow_and_torchvision_pad():
    PIL = pytest.importorskip('PIL.Image')
    rng = np.random.default_rng(5)
    raw = [rng.integers(0, 256, s, dtype=np.uint8) for s in ((427, 640, 3), (640, 480, 3), (641, 641, 3), (90, 1000, 3), (641, 300, 3))]
    fills = [7, 200, 0, 33, 255]
    g = pp.GpuPreprocess(641, batched=True)
    canvas, metas = g(raw, fill=fills)
    assert tuple(canvas.shape) == (5, 641, 641, 3)
    got = canvas.cpu().numpy()
    for i, (img, fill) in enumerate(zip(raw, fills)):
        h, w = img.shape[:2]
        tw, th = pp.rescale_target(w, h, 641)
        l, t, _, _ = pp.center_pad_ltrb(tw, th, 641, 641)
        want = np.full((641, 641, 3), fill, dtype=np.uint8)
        want[t:t + th, l:l + tw] = np.asarray(PIL.fromarray(img).resize((tw, th), PIL.BILINEAR))
        np.testing.assert_array_equal(got[i], want)
        assert metas[i]['offset'][0] == -l + 0.0 and metas[i]['scale'][0] == (tw - 1) / (w - 1)
    # batch size 1: CenterPadTight(16)
    g1 = pp.GpuPreprocess(385, batched=False)
    canvas, metas = g1([raw[0]])
    tw, th = pp.rescale_target(640, 427, 385)
    assert tuple(canvas.shape) == (1, (th - 1 + 15) // 16 * 16 + 1, 385, 3)
    l, t, _, _ = pp.center_pad_ltrb(tw, th, 385, canvas.shape[1])
    want = np.empty(tuple(canvas.shape[1:]), dtype=np.uint8)
    want[:] = pp.TIGHT_PAD_FILL                                      # transforms/pad.py:100-101
    want[t:t + th, l:l + tw] = np.asarray(PIL.fromarray(raw[0]).resize((tw, th), PIL.BILINEAR))
    np.testing.assert_array_equal(canvas[0].cpu().numpy(), want)


@pytest.mark.gpu
def test_raw_images_through_preprocess_stem_and_decoder():
    """raw uint8 images -> GPU resize / pad -> uint8 stem -> heads == the reference's PIL + float pipeline fed to the
    float stem, bit for bit; annotations inverse-transformed in one batch"""
    PIL = pytest.importorskip('PIL.Image')
    from openpifpaf_b200 import constants, network, predictor
    rng = np.random.default_rng(11)
    raw = [rng.integers(0, 256, s, dtype=np.uint8) for s in ((120, 161, 3), (161, 100, 3))]
    g = pp.GpuPreprocess(161, batched=True)
    canvas, metas = g(raw, fill=[5, 6])
    plan = network.random_plan('shufflenetv2k16', seed=2, confidence_bias=0.0)
    net = network.CompiledNet(plan, 161, 161, 2)
    heads_u8 = [t.clone() for t in net.forward_uint8(canvas)]
    mean = torch.tensor(network.CompiledNet.IMAGE_MEAN).view(1, 3, 1, 1)
    std = torch.tensor(network.CompiledNet.IMAGE_STD).view(1, 3, 1, 1)
    ref_imgs = []
    for img, fill in zip(raw, (5, 6)):
        h, w = img.shape[:2]
        tw, th = pp.rescale_target(w, h, 161)
        l, t, _, _ = pp.center_pad_ltrb(tw, th, 161, 161)
        c = np.full((161, 161, 3), fill, dtype=np.uint8)
        c[t:t + th, l:l + tw] = np.asarray(PIL.fromarray(img).resize((tw, th), PIL.BILINEAR))
        ref_imgs.append(torch.from_numpy(c).permute(2, 0, 1).float().div(255.0))
    x = ((torch.stack(ref_imgs) - mean) / std).cuda()
    for a, b in zip(heads_u8, net.forward(x)):
        assert torch.equal(a, b)
    pred = predictor.Predictor(net, constants.COCO_N_KEYPOINTS, constants.COCO_PERSON_SKELETON)
    res = pred.batch(canvas.cpu().pin_memory())
    via_api = pred.raw_images(raw, fill=[5, 6])
    for (ann, _), meta, (data2, scales2, meta2) in zip(res, metas, via_api):
        data, scales = pp.inverse_transform_batch(ann.numpy(), meta)
        assert data.shape == (ann.shape[0], 17, 3) and np.isfinite(data).all()
        np.testing.assert_array_equal(data, data2)
        np.testing.assert_array_equal(scales, scales2)
    js = pred.raw_images(raw, fill=[5, 6], json_data=True)
    assert len(js) == 2 and all(isinstance(j, list) for j, _ in js)
