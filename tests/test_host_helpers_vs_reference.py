"""Host-side helpers of the drop-in `pose_detector` module (SURVEY.md 8a row a14: get_unit_length, crop_face,
crop_hands, crop_image, crop_around_keypoint, crop_person, draw_person_pose) against the reference's own methods on
seeded random poses.  The reference results are committed as digests (tests/golden/host_helpers_ref.json, produced by
oracle/make_goldens.py host_helper_goldens from the reference's files executed verbatim).  CPU only."""
import json
import os

import pytest

from conftest import GOLDEN, pkg
from oracle import make_goldens as MG

with open(os.path.join(GOLDEN, "host_helpers_ref.json")) as _f:
    REF = json.load(_f)


def _det():
    PD = pkg("pose_detector").PoseDetector
    return PD.__new__(PD)


@pytest.mark.parametrize("seed", range(12))
def test_unit_length_and_crops_match_reference(seed):
    assert MG.unit_length_and_crops(_det(), seed) == REF["unit_length_and_crops"][seed]


@pytest.mark.parametrize("seed", range(6))
def test_draw_person_pose_matches_reference(seed):
    assert MG.draw_person_pose_cases(pkg("pose_detector").draw_person_pose, seed) == REF["draw_person_pose"][seed]


@pytest.mark.parametrize("seed", range(8))
def test_crop_person_matches_reference(seed):
    """pose_detector.py:311-352 (the reference method needs the `sys` it never imports, :1-12).  Degenerate poses (no
    joint right of the first one) make both raise -- AttributeError (`.astype` on an int, :346-349) in the reference,
    ValueError (negative crop size) here."""
    assert MG.crop_person_cases(_det(), seed) == REF["crop_person"][seed]
