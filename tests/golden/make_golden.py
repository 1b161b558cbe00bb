"""Generates the golden fixtures under tests/golden/ from a checkout of the reference (rust-cv/cv):

    python tests/golden/make_golden.py <reference checkout>

The tests read only the stored fixtures, never the reference checkout.

 - kitti_0000000000.npz / kitti_0000000014.npz : the two reference fixture frames
   (res/*.png of the reference, 1392x512 8-bit gray) as uint8 arrays -- inputs of the reference's
   own golden test akaze/tests/estimate_pose.rs:24-76.
 - akaze_goldens.json : the counts that test asserts (399 / 343 descriptors, 11 Lowe-0.5 matches,
   estimate_pose.rs:41-42,59) plus secondary counts produced by the oracle at Akaze::default().
 - oracle_kitti_sparse.npz : oracle keypoints + descriptors for both frames at Akaze::sparse();
   lets the GPU parity test run against committed vectors as well as the live oracle.
"""
import json
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import pyoracle as O  # noqa: E402


def main(ref_root):
    frames = {}
    for name in ("0000000000", "0000000014"):
        im = cv2.imread(os.path.join(ref_root, "res", name + ".png"), cv2.IMREAD_UNCHANGED)
        assert im.dtype == np.uint8 and im.ndim == 2
        np.savez_compressed(os.path.join(HERE, f"kitti_{name}.npz"), image=im)
        frames[name] = im.astype(np.float32) / np.float32(255)  # GrayFloatImage::from_dynamic, image.rs:53-55
    out = {"reference_asserted": {"descriptors_0": 399, "descriptors_14": 343, "lowe_0.5_matches": 11,
                                  "source": "akaze/tests/estimate_pose.rs:41-42,59"}}
    res = {}
    for thr, tag in ((0.01, "sparse"), (0.001, "default")):
        stages = {}
        descs = {}
        for name, img in frames.items():
            ak = O.Akaze(detector_threshold=thr)
            kps, d = ak.extract(img)
            stages[name] = {s: int(len(ak.stage(s))) for s in O.STAGES}
            descs[name] = (kps, d)
        idx, dist = O.hamming_knn(descs["0000000000"][1], descs["0000000014"][1], 2)
        lowe = int((dist[:, 0].astype(np.float32) < dist[:, 1].astype(np.float32) * np.float32(0.5)).sum())
        res[tag] = {"stages": stages, "lowe_0.5_matches": lowe}
        if tag == "sparse":
            np.savez_compressed(os.path.join(HERE, "oracle_kitti_sparse.npz"),
                                kps0=descs["0000000000"][0], desc0=descs["0000000000"][1],
                                kps14=descs["0000000014"][0], desc14=descs["0000000014"][1],
                                knn_idx=idx, knn_dist=dist)
    out["oracle_derived"] = res
    with open(os.path.join(HERE, "akaze_goldens.json"), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main(sys.argv[1])
