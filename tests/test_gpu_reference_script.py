"""SURVEY section 8 row b: the reference's OWN test driver, the unmodified file dvmvs/fusionnet/run-testing.py, executed as a
script against this package (drop-in `dvmvs`), with the environment overlay in compat/ (NumPy-2 `loadtxt` newline
delimiter, the un-installed `path` package) and `Config` set through environment variables.  Its saved predictions are
compared with the reference's shipped golden predictions.

The script file is copied verbatim from a checkout of the original project by tools/fetch_fixtures.py into the git-ignored
tests/golden/_ref_data/scripts/ (it is never imported by the product); without it the test skips.  The
sample-data tree it reads is staged here from the committed fixture subset of scene 000: the images the first 10 keyframes
touch, their poses in sorted-file order (the script indexes poses by the position of the image in the sorted directory,
run-testing.py:75-82,104-109), K.txt, the first 10 lines of the shipped index file, and placeholder depth maps (ground truth
only feeds the error metrics, not the predictions)."""
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENE = os.path.join(REPO, "tests", "golden", "scene000")
REF_DATA = os.path.join(REPO, "tests", "golden", "_ref_data")


def _stage_sample_data(root):
    import cv2
    meta = np.load(os.path.join(SCENE, "poses_subset.npz"))
    names = [str(n) for n in meta["names"]]
    order = np.argsort(names)
    scene = os.path.join(root, "hololens-dataset", "000")
    os.makedirs(os.path.join(scene, "images"))
    os.makedirs(os.path.join(scene, "depth"))
    os.makedirs(os.path.join(root, "indices"))
    np.savetxt(os.path.join(scene, "K.txt"), meta["K"].astype(np.float64), fmt="%.18e")
    np.savetxt(os.path.join(scene, "poses.txt"), meta["poses"][order].reshape(-1, 16).astype(np.float64), fmt="%.18e")
    for i in order:
        src = os.path.join(SCENE, "images", names[i])
        shutil.copyfile(src, os.path.join(scene, "images", names[i]))
        h, w = cv2.imread(src, -1).shape[:2]
        cv2.imwrite(os.path.join(scene, "depth", names[i]), np.zeros((h, w), dtype=np.uint16))
    shutil.copyfile(os.path.join(SCENE, "keyframe+hololens-dataset+000+nmeas+3"),
                    os.path.join(root, "indices", "keyframe+hololens-dataset+000+nmeas+3"))


@pytest.mark.parametrize("backend,terms,bound", [("tc", "3", 1e-4), ("tc", "1", 3.3e-4)])
def test_reference_run_testing_script_runs_unchanged(tmp_path, backend, terms, bound):
    script = os.path.join(REF_DATA, "scripts", "fusionnet", "run-testing.py")
    weights = os.path.join(REF_DATA, "weights", "fusionnet")
    if not os.path.isfile(script) or not os.path.isdir(weights):
        pytest.skip("the original project's run-testing.py / shipped weights are not in tests/golden/_ref_data (python tools/fetch_fixtures.py <deep-video-mvs checkout>)")
    data = str(tmp_path / "sample-data")
    _stage_sample_data(data)
    cwd = tmp_path / "fusionnet"          # the script loads sorted(Path("weights").files()) relative to its working directory
    cwd.mkdir()
    os.symlink(weights, str(cwd / "weights"))
    results = str(tmp_path / "results")
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join([os.path.join(REPO, "compat"), os.path.join(REPO, "deep-video-mvs_b200")])
    env.update(DVMVS_DATA=data, DVMVS_RESULTS=results, DVMVS_CONV_BACKEND=backend, DVMVS_TC_TERMS=terms)
    run = subprocess.run([sys.executable, script], cwd=str(cwd), env=env, capture_output=True, text=True, timeout=900)
    assert run.returncode == 0, run.stdout[-3000:] + "\n" + run.stderr[-3000:]
    assert "Loaded weights for" in run.stdout
    out = os.path.join(results, "keyframe_hololens-dataset_320_256_3_dvmvs_fusionnet_predictions_000.npz")
    assert os.path.isfile(out), os.listdir(results)
    pred = np.load(out)["arr_0"]
    from oracle import npz_parts
    gold = npz_parts.load(os.path.join(SCENE, "golden_predictions_first10.npz"))["predictions"]
    assert pred.shape == gold[:len(pred)].shape and len(pred) == 10
    errs = [float(np.abs(1.0 / p - 1.0 / g).sum() / np.abs(1.0 / g).sum()) for p, g in zip(pred, gold)]
    print("run-testing.py (unmodified) + drop-in dvmvs, %s terms=%s: rel-L1(inverse depth) vs shipped golden per keyframe:" % (backend, terms),
          ["%.2e" % e for e in errs])
    assert max(errs) <= bound, errs
