"""Run HERE (the container that has /root/reference): packs one dataset pair into
tests/golden/inputs_<name>.npz so that GPU-box runs never need /root/reference.

ref: src/main.cpp:93 (imread colour), :160-170 (annotation: gray read, 32 = unannotated).
"""
import os
import sys

import cv2
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
REF = "/root/reference/dataset"


def main(names):
    for name in names:
        bgr = cv2.imread(os.path.join(REF, "images", name + ".jpg"))
        ann = cv2.imread(os.path.join(REF, "annotations", name + ".png"), 0)
        assert bgr is not None and ann is not None and bgr.shape[:2] == ann.shape
        out = os.path.join(ROOT, "tests", "golden", "inputs_%s.npz" % name.lower())
        np.savez_compressed(out, bgr=bgr, annotation=ann)
        print(out, bgr.shape, os.path.getsize(out))


def pack_all():
    """All 12 pairs, one file each under tests/golden/dataset/ (0.1 - 0.45 MB): the JPEG bytes as they are (decoded by cv2 at
    test time, like main.cpp's imread) and the annotation as the gray plane main.cpp reads."""
    import glob
    outdir = os.path.join(ROOT, "tests", "golden", "dataset")
    os.makedirs(outdir, exist_ok=True)
    for f in sorted(glob.glob(os.path.join(REF, "images", "*.jpg"))):
        name = os.path.basename(f)[:-4]
        raw = np.fromfile(f, np.uint8)
        assert np.array_equal(cv2.imread(f), cv2.imdecode(raw, cv2.IMREAD_COLOR))
        ann = cv2.imread(os.path.join(REF, "annotations", name + ".png"), 0)
        assert ann is not None
        out = os.path.join(outdir, name.lower() + ".npz")
        np.savez_compressed(out, jpg=raw, ann=ann)
        print(out, os.path.getsize(out))


if __name__ == "__main__":
    if "--pack" in sys.argv:
        pack_all()
    else:
        main(sys.argv[1:] or ["Dog"])
