"""The UNMODIFIED reference class (VisualOdometryPipeLine.py of ManuelWendl/Monocular_Visual_Odometry_VA4MR) running
on the CUDA path through `cv2_compat.install()` -- what "drop-in" means.  The reference is not part of this
repository, so the test needs a B200 and a checkout of the reference named by B200VO_REFERENCE_DIR, and skips
without one.  The free-running GPU tests in test_free_running_gpu.py drive the same data flow through
tests/mini_vo.py (a restatement that is itself pinned to the recorded reference run by test_oracle_free_running.py)."""
import os
import sys

import numpy as np
import pytest

from monocular_visual_odometry_va4mr_b200 import cv2_compat, synth

pytestmark = pytest.mark.gpu
REF = os.environ.get("B200VO_REFERENCE_DIR", "")


@pytest.mark.skipif(not REF or not os.path.exists(os.path.join(REF, "VisualOdometryPipeLine.py")),
                    reason="B200VO_REFERENCE_DIR does not name a checkout of the reference project")
def test_unmodified_reference_class_runs_on_the_cuda_path():
    cv2 = pytest.importorskip("cv2")
    sys.path.insert(0, REF)
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_reference_trace import OPTIONS, RENDER          # the reference's KITTI options (main.py:20-44)
    if not hasattr(np, "bool"):
        np.bool = bool                                          # the reference uses np.bool (:346)
    s = synth.render_sequence(RENDER["shape"], RENDER["n_frames"], seed=RENDER["seed"])
    frames = [s["frames"][i] for i in range(RENDER["n_frames"])]
    from VisualOdometryPipeLine import VisualOdometryPipeLine

    def run():
        vo = VisualOdometryPipeLine(s["K"], OPTIONS)
        b0, b1 = RENDER["bootstrap"]
        vo.initialization(frames[b0], frames[b1])
        counts, poses = [len(vo.matched_keypoints)], []
        for i in range(b1 + 1, len(frames)):
            vo.continuous_operation(frames[i])
            counts.append(len(vo.matched_keypoints))
            R, t = vo.transforms[-1]
            poses.append(np.hstack([np.ravel(R), np.ravel(t)]))
        return counts, np.array(poses)

    want_counts, want_poses = run()                              # real cv2
    cv2_compat.install()
    try:
        got_counts, got_poses = run()                            # the six call sites on libb200vo.so
    finally:
        cv2_compat.uninstall()
    assert got_counts == want_counts
    # SURVEY 8c tier (ii): first frames of a free run, <= 0.5 % of the path length
    path = np.linalg.norm(np.diff(want_poses[:, 9:], axis=0), axis=1).sum() + 1e-9
    assert np.linalg.norm(got_poses[:, 9:] - want_poses[:, 9:], axis=1).max() <= 5e-3 * path
