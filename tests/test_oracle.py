"""CPU: the plain-C oracle against the reference's outputs: golden vectors dumped from the unmodified reference
build (oracle/make_golden.py), bit for bit at every stage."""
import hashlib
import os

import numpy as np
import pytest

import helpers
from openpifpaf_b200 import synth
from oracle import cifcaf as oc
from oracle import make_golden as mg


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def reference_cases():
    """the reference decoder's outputs on the cases below (python -m oracle.make_golden reference)"""
    return np.load(os.path.join(helpers.GOLDEN_DIR, 'reference_oracle_cases.npz'))


@pytest.mark.parametrize('path', helpers.golden_cases(), ids=lambda p: p.split('decoder_')[-1][:-4])
def test_oracle_matches_golden(path):
    g, f, statics, digest_ok = helpers.load_golden(path)
    assert digest_ok, 'synthetic field generator is not bit-reproducible on this machine'
    p = oc.default_params(**helpers.statics_to_params(statics))
    ann, ids, taps = oc.decode(f['cif'], int(g['stride']), f['caf'], int(g['stride']), f['skeleton'],
                               f['n_keypoints'], params=p, taps=True)
    # bit-exact, every stage (the oracle restates libstdc++'s sort/heap tie order too)
    assert sha(taps['cifhr']) == str(g['cifhr_sha256'])
    np.testing.assert_array_equal(taps['seeds_f'], g['seeds_f'])
    np.testing.assert_array_equal(taps['seeds_vxys'], g['seeds_vxys'])
    assert [len(x) for x in taps['fwd']] == list(g['n_fwd'])
    if not statics.get('force_complete'):
        assert sha(np.concatenate([x.reshape(-1, 7) for x in taps['fwd']])) == str(g['fwd_sha256'])
        assert sha(np.concatenate([x.reshape(-1, 7) for x in taps['bwd']])) == str(g['bwd_sha256'])
    np.testing.assert_array_equal(ann, g['annotations'])
    np.testing.assert_array_equal(ids, g['ids'])


def test_golden_stored_fields_roundtrip():
    g = np.load([p for p in helpers.golden_cases() if 'coco11_1p' in p][0])
    ann, ids = oc.decode(g['cif'], 16, g['caf'], 16, synth.make_fields('cocokp', 11, 11, 1, 5)['skeleton'], 17)
    np.testing.assert_array_equal(ann, g['annotations'])


@pytest.mark.parametrize('seed', mg.LIVE_CIFCAF_SEEDS)
def test_oracle_matches_live_reference(seed):
    g = reference_cases()
    f = mg.live_cifcaf_fields(seed)
    assert synth.fields_digest(f['cif'], f['caf']) == str(g[f'cifcaf{seed}_fields_sha256'])
    oa, oi, ot = oc.decode(f['cif'], 16, f['caf'], 16, f['skeleton'], 17, taps=True)
    assert sha(ot['cifhr']) == str(g[f'cifcaf{seed}_cifhr_sha256'])
    np.testing.assert_array_equal(ot['seeds_vxys'], g[f'cifcaf{seed}_seeds_vxys'])
    for side in ('fwd', 'bwd'):
        assert [len(x) for x in ot[side]] == list(g[f'cifcaf{seed}_n_{side}'])
        assert sha(np.concatenate([x.reshape(-1, 7) for x in ot[side]])) == str(g[f'cifcaf{seed}_{side}_sha256'])
    np.testing.assert_array_equal(oa, g[f'cifcaf{seed}_annotations'])
    np.testing.assert_array_equal(oi, g[f'cifcaf{seed}_ids'])


def test_oracle_initial_annotations_match_reference():
    g = reference_cases()
    f = mg.initial_annotations_fields()
    assert synth.fields_digest(f['cif'], f['caf']) == str(g['init_fields_sha256'])
    init, ids = g['init_annotations'], g['init_ids']
    oa, oi = oc.decode(f['cif'], 16, f['caf'], 16, f['skeleton'], 17, initial_annotations=init, initial_ids=ids)
    np.testing.assert_array_equal(oa, g['init_result_annotations'])
    np.testing.assert_array_equal(oi, g['init_result_ids'])
    assert 42 in oi


def test_oracle_grow_connection_blend_matches_reference():
    g = reference_cases()
    caf = mg.blend_caf()
    for only_max in (False, True):
        got = oc.grow_connection_blend(caf, 20.0, 20.0, 30.0, 1.0, only_max)
        assert list(g[f'blend_only_max{int(only_max)}']) == got


def test_empty_and_degenerate_fields():
    sk = synth.make_fields('cocokp', 3, 3, 0, 0)['skeleton']
    cif = np.zeros((17, 5, 3, 3), dtype=np.float32)
    caf = np.zeros((19, 8, 3, 3), dtype=np.float32)
    ann, ids = oc.decode(cif, 16, caf, 16, sk, 17)
    assert ann.shape == (0, 17, 4)
    f = synth.make_fields('cocokp', 1, 1, 0, 0)
    ann, _ = oc.decode(f['cif'], 16, f['caf'], 16, f['skeleton'], 17)
    assert ann.shape[0] == 0


# ---------------------------------------------------------------- CifDet (csrc/src/cifdet.cpp)
@pytest.mark.parametrize('path', helpers.golden_det_cases(), ids=lambda p: p.split('cifdet_')[-1][:-4])
def test_oracle_cifdet_matches_golden(path):
    g, f, digest_ok = helpers.load_golden_det(path)
    assert digest_ok, 'synthetic field generator is not bit-reproducible on this machine'
    cats, scores, boxes = oc.decode_det(f['field'], int(g['stride']))
    np.testing.assert_array_equal(cats, g['categories'])
    np.testing.assert_array_equal(scores, g['scores'])
    np.testing.assert_array_equal(boxes, g['boxes'])
    assert len(cats) <= 120


@pytest.mark.parametrize('seed', mg.LIVE_CIFDET_SEEDS)
def test_oracle_cifdet_matches_live_reference(seed):
    g = reference_cases()
    field = mg.live_cifdet_field(seed)
    assert sha(field) == str(g[f'cifdet{seed}_field_sha256'])
    got = oc.decode_det(field, 16)
    for a, key in zip(got, ('categories', 'scores', 'boxes')):
        np.testing.assert_array_equal(a, g[f'cifdet{seed}_{key}'])
    assert len(got[0]) >= 3


def test_oracle_cifdet_empty_field():
    cats, scores, boxes = oc.decode_det(np.zeros((5, 6, 4, 7), dtype=np.float32), 16)
    assert cats.shape == (0,) and boxes.shape == (0, 4)
