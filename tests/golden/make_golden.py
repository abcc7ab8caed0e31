"""Generates tests/golden/<log>_<kind>.txt.xz from the reference's bundled logs (needs the reference's dataset tree; the
committed files are all the tests read).

    python tests/golden/make_golden.py REFERENCE_DATASET_DIR

Contents (parsed from the 6-significant-digit text logs with numpy.loadtxt, float64):
  water_corners [1062,18]  t id + 16 undistorted normalised stereo corner coords  (vision.cpp:111-119)
  water_image   [1062,9]   t id p(3) q(wxyz): logged output of RefractionTriangulation+ComputeMarkerPose
  land_corners  [1257,14]  t id + 4 triangulated 3-D corners                    (vision.cpp:120-124)
  land_image    [1257,9]   logged output of ComputeMarkerPose
  land_imu / water_imu     [n,7] t accel(3) gyro(3) raw IMU log                  (filter.cpp:31-32)
  land_fusion / water_fusion [n,17] logged filter output of an OLDER reference revision: shape-only pin
Source: REFERENCE_DATASET_DIR/{landdata/dataset-02,waterdata/dataset-06}.

Each log is stored as text the way the reference's `ofstream <<` writes it ("%g", the marker id as an integer; LF line
ends), xz-compressed: numpy.loadtxt gives back exactly the parsed rows, at a fraction of the size of binary doubles.

Also writes log_heads.json: the first 4 text lines of every log verbatim (without the line ends), the format pin of
fbus_ekf_b200/logio.py (`ofstream <<` at default precision, SURVEY A.7).
"""
import io
import json
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LOGS = (("land", "landdata/dataset-02"), ("water", "waterdata/dataset-06"))
KINDS = ("corners", "image", "imu", "fusion")
ID_COLUMN = {"corners": 1, "image": 1, "imu": None, "fusion": None}


def save_log(path, rows, id_column):
    text = "".join(" ".join(("%d" % int(v)) if i == id_column else ("%g" % v) for i, v in enumerate(r)) + "\n" for r in rows)
    assert np.array_equal(np.loadtxt(io.StringIO(text), ndmin=2), rows), path
    with lzma.open(path, "wt", preset=9 | lzma.PRESET_EXTREME) as fh:
        fh.write(text)


def main(src):
    for key, sub in LOGS:
        for kind in KINDS:
            rows = np.loadtxt(os.path.join(src, sub, kind + ".txt"), ndmin=2)
            save_log(os.path.join(HERE, f"{key}_{kind}.txt.xz"), rows, ID_COLUMN[kind])
            print(key, kind, rows.shape)
    heads = {}
    for key, sub in LOGS:
        for kind in KINDS:
            with open(os.path.join(src, sub, kind + ".txt"), newline="") as fh:
                heads[f"{key}_{kind}"] = [fh.readline().rstrip("\r\n") for _ in range(4)]
    json.dump(heads, open(os.path.join(HERE, "log_heads.json"), "w"), indent=1)


if __name__ == "__main__":
    main(sys.argv[1])
