"""Statistical calibration of the pose covariance on the CPU oracle (oracle/dpr_cov_oracle.py: calibration).

For each camera, 4 seeded working-volume poses, 40 noise seeds each: the seed-to-seed scatter of the refined pose
against sigma_noise^2 H^-1 and against s^2 H^-1.  tests/test_cpu_pose_cov.py asserts the band [0.15, 5] on the same
sweep; this script prints every number.  Usage: python scripts/pose_cov_calibration.py [--out profiles/r03_pose_cov_calibration.log]
"""
import argparse
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from accurate_aprilgroup_tracking_b200 import synth  # noqa: E402
from oracle import dpr_cov_oracle, dpr_pin  # noqa: E402

def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    lines = []
    mdl = dpr_pin.model()
    for cam_name, cam in dpr_pin.CAMERAS.items():
        for k, truth in enumerate(dpr_cov_oracle.calibration_poses(cam_name)):
            t0 = time.time()
            r = dpr_cov_oracle.calibration(cam, mdl, truth, dpr_cov_oracle.CALIBRATION_SEEDS, np.random.default_rng(k))
            line = (f"{cam_name} pose {k} z={truth[5]:.3f} m, level {r['level']}: n {r['n']:.0f}, residual sigma {r['sigma_res']:.1f} "
                    f"(pixel noise {synth.NOISE_SIGMA}, at the level {dpr_cov_oracle.level_noise_var(r['level'], synth.NOISE_SIGMA) ** 0.5:.2f}), "
                    f"eig(scatter / sigma_level^2 H^-1) {r['eig'].min():.2f} .. {r['eig'].max():.2f}, NEES of s^2 H^-1 {r['nees']:.2f} (6 expected), "
                    f"|bias| / sd max {r['bias_over_sd'].max():.1f}  [{time.time() - t0:.0f} s]")
            print(line, flush=True)
            lines.append(line)
    if a.out:
        Path(a.out).write_text("# python scripts/pose_cov_calibration.py (CPU oracle; numbers do not depend on the machine)\n" + "\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
