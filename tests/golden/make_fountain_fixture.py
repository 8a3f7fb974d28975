"""Generates tests/golden/fountain11_ir.npz from the reference's own fixtures
  data/sfm/fountain11.bin      (a reconstruction saved by Theia after ITS OWN bundle adjustment)
  data/sfm/gt_fountain11.bin   (ground-truth cameras of Strecha fountain-P11)
used by incremental_reconstruction_estimator_test.cc:52-160.  The reference cannot run here (C++ needing Ceres), but its
saved OUTPUT travels: the flattened IR of that reconstruction pins our cost function against a state the reference's
BA produced (tests/test_fountain_fixture.py).    Run:  python tests/golden/make_fountain_fixture.py <TheiaSfM>/data/sfm

The file is stored compacted, losslessly, to stay small: pixel coordinates as float32 (every one of them is exactly
representable, asserted below), pt and obs_xy as the byte planes of their column-major data (the sign / exponent bytes
then compress well), obs_pt as differences of consecutive entries.  tests/helpers.py:fountain_problem() undoes it.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import theia_cereal  # noqa: E402


def byte_planes(a):
    """[n, k] -> uint8 [itemsize, n * k]: byte j of every element of the column-major data in row j."""
    a = np.ascontiguousarray(np.asarray(a).T)
    return np.ascontiguousarray(a.view(np.uint8).reshape(-1, a.dtype.itemsize).T)


def main(data):
    rec = theia_cereal.reconstruction(open(os.path.join(data, "fountain11.bin"), "rb").read())
    gt = theia_cereal.reconstruction(open(os.path.join(data, "gt_fountain11.bin"), "rb").read())
    assert rec["consumed"] == rec["total"] and gt["consumed"] == gt["total"]
    vids = sorted(rec["views"])
    tids = sorted(t for t in rec["tracks"] if rec["tracks"][t]["est"])
    assert all(rec["views"][v]["est"] for v in vids)
    cam_of = {v: i for i, v in enumerate(vids)}
    pt_of = {t: i for i, t in enumerate(tids)}
    names = [rec["views"][v]["name"] for v in vids]
    ext = np.array([rec["views"][v]["camera"]["ext"] for v in vids])
    assert len({rec["views"][v]["camera"]["intr_id"] for v in vids}) == 1  # one shared PinholeCameraModel
    intr = np.zeros((1, 10))
    intr[0, :7] = rec["views"][vids[0]]["camera"]["intr"]
    pt = np.array([rec["tracks"][t]["pt"] for t in tids])
    oc, op, oxy = [], [], []
    for v in vids:
        for t, f in sorted(rec["views"][v]["features"].items()):
            if t in pt_of:
                oc.append(cam_of[v]); op.append(pt_of[t]); oxy.append(f)
    gt_by_name = {gt["views"][v]["name"]: gt["views"][v]["camera"] for v in gt["views"]}
    gt_ext = np.array([gt_by_name[n]["ext"] for n in names])
    gt_intr = np.array([gt_by_name[n]["intr"] for n in names])
    out = os.path.join(HERE, "fountain11_ir.npz")
    oxy = np.array(oxy)
    assert np.array_equal(oxy.astype(np.float32), oxy) and len(vids) < 256 and len(tids) < 2 ** 15
    np.savez_compressed(out, names=np.array(names), ext=ext, intr=intr, pt=byte_planes(pt), obs_cam=np.array(oc, np.uint8),
                        obs_pt=np.diff(np.array(op), prepend=0).astype(np.int16), obs_xy=byte_planes(oxy.astype(np.float32)),
                        gt_ext=gt_ext, gt_intr=gt_intr)
    print("wrote", out, "cams", len(vids), "points", len(tids), "obs", len(oc), "bytes", os.path.getsize(out))


if __name__ == "__main__":
    main(sys.argv[1])
