"""TEST INFRASTRUCTURE: records the renderer calls of the REFERENCE package's own tests / examples.

    DEODR_STAGED_REFERENCE=<copy of the reference with its Cython extension built> DEODR_RECORD_OUT=<file.npz> \
    [DEODR_RECORD_CALLS=<forward-call ordinals, comma-separated; all when unset>] \
    python tests/dropin/runner.py pytest <pytest args ...>     # the reference's test files, unmodified
    python tests/dropin/runner.py soup <clockwise 0|1> <antialiase_error 0|1> <iterations>
    python tests/dropin/runner.py hand_depth <none|pytorch> <iterations>
    python tests/dropin/runner.py hand_rgb <none|pytorch> <iterations>

The reference's code runs unchanged with its own extension; ``dropin_calls.Recorder`` wraps the extension's two entry
points and stores the selected calls with the reference's results (tests/golden/make_dropin_calls.py drives this, and
tests/test_dropin_reference.py replays the result through deodr_b200).
"""
import atexit
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def main():
    mode, args = sys.argv[1], sys.argv[2:]
    staged = os.environ["DEODR_STAGED_REFERENCE"]
    sys.path[:0] = [os.path.join(HERE, "stubs"), staged]
    import cv2

    cv2.waitKey = lambda *a, **k: -1
    cv2.imshow = lambda *a, **k: None
    import deodr  # the staged reference package
    from deodr import differentiable_renderer_cython as ffi
    from dropin_calls import Recorder

    assert os.path.abspath(deodr.__file__).startswith(os.path.abspath(staged)), deodr.__file__
    keep = os.environ.get("DEODR_RECORD_CALLS")
    rec = Recorder(ffi.renderSceneCpp, ffi.renderSceneBCpp, None if not keep else {int(i) for i in keep.split(",")})
    ffi.renderSceneCpp, ffi.renderSceneBCpp = rec.render, rec.render_b
    atexit.register(rec.save, os.environ["DEODR_RECORD_OUT"])
    if mode == "pytest":
        import pytest

        sys.exit(pytest.main(["-q", "-x", "-p", "no:cacheprovider", "--rootdir", staged] + args))
    if mode == "soup":
        from deodr.examples.triangle_soup_fitting import run

        run(nb_max_iter=int(args[2]), display=False, clockwise=bool(int(args[0])), antialiase_error=bool(int(args[1])))
        return
    if mode in ("hand_depth", "hand_rgb"):
        if mode == "hand_depth":
            from deodr.examples.depth_image_hand_fitting import run
        else:
            from deodr.examples.rgb_image_hand_fitting import run
        run(dl_library=args[0], plot_curves=False, display=False, save_images=False, max_iter=int(args[1]))
        return
    raise SystemExit(f"unknown mode {mode}")


if __name__ == "__main__":
    main()
