"""Copies the reference's shipped weight files (parity fixtures, SURVEY.md section 2 row 7) and its test-driver scripts from
a checkout of the original project into tests/golden/_ref_data/ (git-ignored; 133 MB, too large for the repository).

    python tools/fetch_fixtures.py <deep-video-mvs checkout>      # or DVMVS_REFERENCE_ROOT=<checkout>

The tests that need these files skip without them."""
import os
import shutil
import sys

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def fetch(ref, verbose=True):
    if not os.path.isdir(os.path.join(ref, "dvmvs")):
        if verbose:
            print("fetch_fixtures: no reference tree at", ref, "- nothing fetched")
        return False
    for net in ("fusionnet", "pairnet"):
        src = os.path.join(ref, "dvmvs", net, "weights")
        dst = os.path.join(REPO, "tests", "golden", "_ref_data", "weights", net)
        os.makedirs(dst, exist_ok=True)
        for f in sorted(os.listdir(src)):
            s, d = os.path.join(src, f), os.path.join(dst, f)
            if not os.path.isfile(d) or os.path.getsize(d) != os.path.getsize(s):
                shutil.copyfile(s, d)
                if verbose:
                    print("fetched", net, f)
    # the reference's test drivers, verbatim, for the "runs unchanged" test (tests/test_gpu_reference_script.py): git-ignored like
    # the weights, never imported by the product
    for net in ("fusionnet", "pairnet"):
        dst = os.path.join(REPO, "tests", "golden", "_ref_data", "scripts", net)
        os.makedirs(dst, exist_ok=True)
        for f in ("run-testing.py", "run-testing-online.py"):
            s = os.path.join(ref, "dvmvs", net, f)
            if os.path.isfile(s):
                shutil.copyfile(s, os.path.join(dst, f))
                if verbose:
                    print("fetched script", net, f)
    return True


if __name__ == "__main__":
    root = sys.argv[1] if len(sys.argv) > 1 else os.environ.get("DVMVS_REFERENCE_ROOT")
    if not root:
        sys.exit("usage: python tools/fetch_fixtures.py <deep-video-mvs checkout>")
    sys.exit(0 if fetch(root) else 1)
