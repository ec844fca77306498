"""GPU test of the device-side visualisation extraction (SURVEY.md 8(f) next #2) against the REFERENCE's own
GetPointCloud / GetSliceMarker: their results on the same frames are stored in tests/golden/reference_golden.json
(vis_replay, generated with oracle/_ref by tests/golden/make_golden.py)."""
import json
import os

import pytest

from tests.golden import make_golden

pytestmark = pytest.mark.gpu

GOLD = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_golden.json")))


def test_point_cloud_and_slice_marker():
    import fiesta_b200
    gold = GOLD["vis_replay"]
    assert gold["point_cloud_0_31"]["n"] > 50 and gold["local_slice_14_1.0"]["n"] > 0
    dev = fiesta_b200.ESDFMap(*make_golden.VIS_MAP, mode="exact")
    got = make_golden.vis_replay(dev)
    for key in gold:
        assert got[key] == gold[key], key
