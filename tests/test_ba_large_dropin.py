"""The drop-in Optimizer::looseBA / fullBA (host/optimizer_localba_gpu.cpp) hands long keyframe ranges to ov2_localba_solve
whole: only the gauge keyframes are constant, none is held constant for capacity below OV2_BA_MAX_OPT_KEYFRAMES.  Runs the
self-test driver under the tests/helpers/ba_dump.c recorder (LD_PRELOAD), which writes the window the drop-in would solve
instead of solving it - no GPU needed."""
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest

from ov2slam_b200 import api, build, synth

ROOT = Path(__file__).resolve().parents[1]


def _write_window(path, pb):
    import struct
    ncam, npts, nobs = len(pb["pose"]), len(pb["lm_invdepth"]), len(pb["obs_cam"])
    with open(path, "wb") as f:
        f.write(struct.pack("4i", ncam, npts, nobs, 0))
        f.write(np.asarray(pb["K"], np.float64).tobytes())
        f.write(np.asarray(pb["K"], np.float64).tobytes())
        f.write(np.asarray([0, 0, 0, 0, 0, 0, 1], np.float64).tobytes())
        for k, dt in (("pose", np.float64), ("pose_const", np.uint8), ("lm_anchor_cam", np.int32), ("lm_anchor_px", np.float64),
                      ("lm_invdepth", np.float64), ("obs_cam", np.int32), ("obs_lm", np.int32), ("obs_px", np.float64)):
            f.write(np.ascontiguousarray(pb[k], dt).tobytes())
        f.write(np.zeros(nobs, np.uint8).tobytes())


def _record(tmp_path, pb, mode):
    exe = build.build_optimizer_shim()
    rec = tmp_path / "librec.so"
    subprocess.check_call(["gcc", "-shared", "-fPIC", "-O1", "-o", str(rec), str(ROOT / "tests" / "helpers" / "ba_dump.c")])
    _write_window(tmp_path / "w.bin", pb)
    env = dict(os.environ, LD_PRELOAD=str(rec), OV2_BA_DUMP=str(tmp_path / "d.bin"))
    out = subprocess.run([str(exe), str(tmp_path / "w.bin"), str(tmp_path / "r.bin"), mode], capture_output=True, text=True,
                         timeout=600, env=env)
    assert out.returncode == 0, out.stdout + out.stderr
    raw = np.fromfile(tmp_path / "d.bin", np.uint8)
    dcam = int(raw[:12].view(np.int32)[0])
    return dcam, raw[12 + 56 * dcam:12 + 57 * dcam].astype(bool), out.stderr


def test_dropin_fullba_beyond_the_total_keyframe_cap_keeps_a_solvable_window(tmp_path):
    """fullBA over a map of more than OV2_BA_MAX_KEYFRAMES keyframes: the large-window solve cannot take any window of that
    size, so the drop-in keeps OV2_BA_SMALL_MAX_OPT_KEYFRAMES optimised keyframes (the newest; the window ov2_localba_solve
    takes at any total size) instead of handing over a window the solve refuses."""
    nkf = api.OV2_BA_MAX_KEYFRAMES + 24
    pb = synth.make_loop_ba_problem(32, nkf, 30000)
    dcam, dconst, err = _record(tmp_path, pb, "full")
    assert dcam == nkf > api.OV2_BA_MAX_KEYFRAMES
    assert int((~dconst).sum()) == api.OV2_BA_SMALL_MAX_OPT_KEYFRAMES
    assert not dconst[-api.OV2_BA_SMALL_MAX_OPT_KEYFRAMES:].any()      # the newest keyframes are the optimised ones
    assert "held constant" in err


@pytest.mark.parametrize("mode", ["loose", "full"])
def test_dropin_hands_over_a_150_keyframe_range_with_only_the_gauge_constant(tmp_path, mode):
    assert api.OV2_BA_MAX_OPT_KEYFRAMES >= 150
    pb = synth.make_loop_ba_problem(31, 150, 3000)
    dcam, dconst, err = _record(tmp_path, pb, mode)
    assert "held constant" not in err
    assert dcam == 150
    assert int(dconst.sum()) == 2                      # the mono gauge: the first two keyframes of the range
    assert int((~dconst).sum()) == 148
