"""Generates tests/golden/dropin_calls.npz: renderer calls of the REFERENCE's own examples and convention tests, run
here with the reference's own Cython extension (built in a scratch copy, see below) through tests/dropin/runner.py,
together with what that extension returned for them (tests/dropin/dropin_calls.py describes what is kept).

    D=<scratch dir>; mkdir $D; cp -r <reference checkout>/{deodr,C++,setup.py,readme.md,tests} $D; chmod -R u+w $D
    (cd $D && python setup.py build_ext --inplace)
    DEODR_STAGED_REFERENCE=$D python tests/golden/make_dropin_calls.py

Kept calls: every call of the three convention tests; the soup fits' first two iterations and their last (the example
renders its target first, so its forward ordinals are shifted by one); the hand fits' first and last iterations.
The GPU acceptance test (tests/test_dropin_reference.py) replays them through deodr_b200.differentiable_renderer_cython.
"""
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
RUNNER = os.path.join(os.path.dirname(HERE), "dropin", "runner.py")
ITERATIONS = 50


sys.path.insert(0, os.path.dirname(RUNNER))
from dropin_calls import load, save  # noqa: E402

MANIFEST, ARRAYS = {}, {}


def record(tag, calls, *args):
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "calls.npz")
        env = dict(os.environ, DEODR_RECORD_OUT=out)
        if calls is not None:
            env["DEODR_RECORD_CALLS"] = ",".join(str(c) for c in calls)
        subprocess.run([sys.executable, RUNNER, *[str(a) for a in args]], env=env, check=True,
                       capture_output=True)
        manifest, arrays = load(out)
    MANIFEST[tag] = manifest["calls"]
    ARRAYS.update(arrays)


def main():
    staged = os.environ.get("DEODR_STAGED_REFERENCE")
    if not staged or not os.path.isdir(os.path.join(staged, "deodr")):
        sys.exit("DEODR_STAGED_REFERENCE must name a copy of the reference with its extension built:\n" + __doc__)
    tests = os.path.join(staged, "tests")
    record("conventions", None, "pytest", os.path.join(tests, "test_pixel_center_coordinates.py"),
           os.path.join(tests, "test_texture_coordinates.py"),
           os.path.join(tests, "test_render_mesh.py") + "::test_render_mesh_triangle_soup")
    for clockwise in (0, 1):
        for antialiase_error in (0, 1):
            record(f"soup_cw{clockwise}_err{antialiase_error}", [0, 1, 2, ITERATIONS], "soup", clockwise,
                   antialiase_error, ITERATIONS)
    fits = [0, ITERATIONS - 1]
    for lib in ("none", "pytorch"):
        record(f"hand_depth_{lib}", fits, "hand_depth", lib, ITERATIONS)
    record("hand_rgb_none", fits, "hand_rgb", "none", ITERATIONS)
    out = os.path.join(HERE, "dropin_calls.npz")
    save(out, MANIFEST, ARRAYS)
    print(out, os.path.getsize(out), "bytes")


if __name__ == "__main__":
    main()
