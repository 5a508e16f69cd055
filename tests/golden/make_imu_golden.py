"""Generates tests/golden/imu_pose_vel_10s.npz from the reference fixture test/data/imu_pose_vel.txt
(layout per include/utils/LoadVirtual.h:84-106: t, qw qx qy qz, tx ty tz, vx vy vz, gx gy gz,
ax ay az, ba x3, bg x3), given the path of that file in a lio-mapping checkout:
    python tests/golden/make_imu_golden.py <lio-mapping>/test/data/imu_pose_vel.txt
The first 10 s (2001 rows) are kept; the clean file's bias columns are uninitialised denormals and
are stored as zeros (SURVEY.md §4)."""
import os
import sys

import numpy as np

DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "imu_pose_vel_10s.npz")

if __name__ == "__main__":
    rows = []
    with open(sys.argv[1]) as f:
        for line in f:
            v = line.split()
            if len(v) >= 17:
                rows.append([float(x) for x in v[:17]])
    a = np.array(rows[:2001])
    np.savez_compressed(DST, t=a[:, 0], q_wxyz=a[:, 1:5], p=a[:, 5:8], v=a[:, 8:11], gyro=a[:, 11:14], acc=a[:, 14:17])
    print("wrote", DST, a.shape)
