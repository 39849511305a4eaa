"""CPU: dataset topology tables equal the reference plugin constants (stored from the reference by
oracle/make_golden.py)."""
import json
import os

import helpers
from openpifpaf_b200 import constants


def test_skeletons_equal_reference():
    with open(os.path.join(helpers.GOLDEN_DIR, 'reference_skeletons.json')) as f:
        ref = json.load(f)
    assert [tuple(e) for e in ref['COCO_PERSON_SKELETON']] == list(constants.COCO_PERSON_SKELETON)
    assert [tuple(e) for e in ref['WHOLEBODY_SKELETON']] == list(constants.wholebody_skeleton())
