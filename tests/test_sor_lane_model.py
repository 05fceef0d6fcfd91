"""The synchronisation protocol and the index arithmetic of sor_lane_kernel, replayed on the CPU
(tools/sor_lane_model.py): random warp interleavings, early and late landing of the asynchronous copies --
no stale ring slot is ever read, no deadlock, result bitwise equal to a raster-scan SOR."""
import os
import sys

import pytest

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "..", "tools"))
import sor_lane_model  # noqa: E402


@pytest.mark.parametrize("w,h,K", [(20, 14, 3), (33, 28, 3), (40, 56, 3), (17, 70, 2), (64, 33, 1), (9, 100, 3), (50, 64, 4), (5, 40, 3), (3, 64, 3), (2, 33, 2), (1, 96, 3)])
@pytest.mark.parametrize("late", [True, False])
def test_lane_wavefront_protocol(w, h, K, late):
    for seed in range(3):
        ok, checked = sor_lane_model.one_case(w, h, K, seed, late)
        assert ok and checked == w * h * K


def test_model_constants_match_the_kernel():
    src = open(os.path.join(os.path.dirname(__file__), "..", "of_dis_b200", "csrc", "sor_lane_kernel.cuh")).read()
    for name, val in (("SL_C", sor_lane_model.C), ("SL_R", sor_lane_model.R), ("SL_D", sor_lane_model.D),
                      ("SL_DS", sor_lane_model.DS), ("SL_DP", sor_lane_model.DP), ("SL_P", sor_lane_model.P)):
        assert "constexpr int %s = %d;" % (name, val) in src
