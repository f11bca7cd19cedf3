import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
for p in (ROOT, HERE):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(HERE, "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def texture():
    return np.load(os.path.join(GOLDEN, "trefle_texture_u8.npy")).astype(np.float64) / 255


@pytest.fixture(scope="session")
def build_native():
    """Compiles liboracle.so / libdeodr_b200.so if missing (nvcc cross-compiles without a GPU)."""
    import __graft_entry__ as entry

    entry.build()
    return True


@pytest.fixture(scope="session")
def port_oracle(build_native):
    from oracle.oracle import Oracle

    return Oracle("port")


@pytest.fixture(scope="session")
def ref_oracle(build_native):
    """The compiled reference itself (oracle/_ref); prebuilt in the build container, travels to the GPU box."""
    from oracle.oracle import Oracle, available

    if not available("reference"):
        pytest.skip("oracle/_ref not built (no /root/reference here)")
    return Oracle("reference")


@pytest.fixture(scope="session")
def checker(build_native):
    """Best available checker for gradients with the summed texture adjoint: _ref(texfix) else the port(texfix)."""
    from oracle.oracle import Oracle, available

    if available("reference", texfix=True):
        return Oracle("reference", texfix=True)
    return Oracle("port", texfix=True)


def load_small(tag):
    """Scene + expected outputs of tests/golden/small_<tag>.npz."""
    from deodr_b200.scenes import SceneArrays

    d = np.load(os.path.join(GOLDEN, f"small_{tag}.npz"))
    f = d["flags"]
    scene = SceneArrays(
        faces=d["in_faces"], faces_uv=d["in_faces_uv"], ij=d["in_ij"], depths=d["in_depths"],
        textured=d["in_textured"], uv=d["in_uv"], shade=d["in_shade"], colors=d["in_colors"],
        shaded=d["in_shaded"], edgeflags=d["in_edgeflags"], height=int(f[0]), width=int(f[1]), nb_colors=int(f[2]),
        texture=d["in_texture"].astype(np.float64),
        background_image=d["in_background_image"] if "in_background_image" in d else None,
        background_color=d["in_background_color"] if "in_background_color" in d else None,
        clockwise=bool(f[3]), backface_culling=bool(f[4]), strict_edge=bool(f[5]), perspective_correct=bool(f[6]),
        integer_pixel_centers=bool(f[7]),
    )
    return scene, d


SMALL_TAGS = ["soup_s1", "soup_nonstrict_halfpix_s2", "soup_persp", "torus", "torus_tex"]
