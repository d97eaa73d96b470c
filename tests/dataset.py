"""The reference's 12 dataset pairs as test fixtures (BASELINE configs[0]).

tests/golden/dataset/<name>.npz holds, per pair, the JPEG file's bytes ("jpg") and the annotation read as gray ("ann"; what
main.cpp reads: src/main.cpp:93 imread colour, :160-162 imread gray); written by tests/golden/make_golden_inputs.py --pack
from the reference's dataset directory, so that the tests need nothing outside this repository.
"""
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PAIRS = os.path.join(GOLD, "dataset")
NAMES = ["arara", "archespark", "dog", "flower", "heidelberg", "hills", "pigs", "rock", "straw", "streetart", "vintagegirl", "womanparasol"]


def have_pack():
    return all(os.path.exists(os.path.join(PAIRS, name + ".npz")) for name in NAMES)


def annotation_to_planes(bgr, ann):
    """ref: src/main.cpp:163-168 -- every annotation pixel != 32: edited BGR := that value, scribble := 255."""
    scribble = np.where(ann != 32, 255, 0).astype(np.uint8)
    edited = bgr.copy()
    edited[ann != 32] = ann[ann != 32][:, None]
    return scribble, edited


def load_pair(name):
    """-> (bgr, scribble, edited, annotation) of one dataset pair, decoded with the same cv2 the rest of the tests use."""
    import cv2
    z = np.load(os.path.join(PAIRS, name + ".npz"))
    bgr = cv2.imdecode(z["jpg"], cv2.IMREAD_COLOR)
    ann = z["ann"]
    assert bgr is not None and bgr.shape[:2] == ann.shape
    scribble, edited = annotation_to_planes(bgr, ann)
    return bgr, scribble, edited, ann
