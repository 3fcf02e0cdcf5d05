"""Loader for the committed slice of the reference's fixture scene (tests/golden/scene000, written by
oracle/make_golden.py) and for the shipped weights (NOT committed: 133 MB; copied from a checkout of the
original project into the git-ignored tests/golden/_ref_data/ by tools/fetch_fixtures.py)."""
import os

import numpy as np

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENE = os.path.join(REPO, "tests", "golden", "scene000")
REF_DATA = os.path.join(REPO, "tests", "golden", "_ref_data")
MODULE_FILES = {"fusionnet": ["0_feature_extractor", "1_feature_pyramid", "2_encoder", "3_lstm_fusion", "4_decoder"],
                "pairnet": ["0_feature_extractor", "1_feature_pyramid", "2_encoder", "3_decoder"]}
TAGS = {"fusionnet": ["fe", "fpn", "cve", "lstm", "cvd"], "pairnet": ["fe", "fpn", "cve", "cvd"]}


def shipped_weights_dir(net="fusionnet"):
    d = os.path.join(REF_DATA, "weights", net)
    return d if all(os.path.isfile(os.path.join(d, f)) for f in MODULE_FILES[net]) else None


def load_shipped_weights(net="fusionnet"):
    import torch
    d = shipped_weights_dir(net)
    if d is None:
        return None
    return {tag: torch.load(os.path.join(d, f), map_location="cpu", weights_only=True)
            for tag, f in zip(TAGS[net], MODULE_FILES[net])}


def preprocess_rgb(path, new_w, new_h):
    """dataset_loader.py:260-263 load_image + :325-336 PreprocessImage.apply_rgb (perform_crop=False)."""
    import cv2
    img = cv2.cvtColor(cv2.imread(path, cv2.IMREAD_COLOR).astype(np.float32), cv2.COLOR_BGR2RGB)
    old_h, old_w = img.shape[:2]
    img = cv2.resize(img, (new_w, new_h), interpolation=cv2.INTER_LINEAR) / 255.0
    for c, (m, s) in enumerate(zip((0.485, 0.456, 0.406), (0.229, 0.224, 0.225))):
        img[:, :, c] = (img[:, :, c] - m) / s
    return np.transpose(img, (2, 0, 1)).astype(np.float32), old_w, old_h


def load_scene(new_w=320, new_h=256):
    """Returns list of keyframes: dict(reference_image, reference_pose, measurement_images, measurement_poses),
    the rescaled full-res K (dataset_loader.py:312-323, perform_crop=False) and golden predictions."""
    meta = np.load(os.path.join(SCENE, "poses_subset.npz"))
    names = [str(n) for n in meta["names"]]
    poses = meta["poses"]
    K = meta["K"].astype(np.float32)
    with open(os.path.join(SCENE, "keyframe+hololens-dataset+000+nmeas+3")) as fh:
        lines = fh.read().splitlines()
    frames = []
    cache = {}
    old = None
    for line in lines:
        ids = line.split(" ")
        for n in ids:
            if n not in cache:
                cache[n], ow, oh = preprocess_rgb(os.path.join(SCENE, "images", n), new_w, new_h)
                old = (ow, oh)
        frames.append(dict(reference_image=cache[ids[0]], reference_pose=poses[names.index(ids[0])].astype(np.float32),
                           measurement_images=[cache[n] for n in ids[1:]],
                           measurement_poses=[poses[names.index(n)].astype(np.float32) for n in ids[1:]]))
    fx, fy = new_w / float(old[0]), new_h / float(old[1])
    full_K = np.array([[K[0, 0] * fx, 0, K[0, 2] * fx], [0, K[1, 1] * fy, K[1, 2] * fy], [0, 0, 1]], dtype=np.float64)
    from oracle import npz_parts
    gold = npz_parts.load(os.path.join(SCENE, "golden_predictions_first10.npz"))["predictions"]
    return frames, full_K.astype(np.float32), gold
