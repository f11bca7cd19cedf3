"""CPU: the parts of bench.py's contract that need no GPU - the algorithmic byte budget of SURVEY.md section 8(d) that
`roofline.achieved` divides, and the JSON line of the reference arm (`--impl reference`, the compiled reference on the
host cores) with the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np
from conftest import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402


class Dims:
    """Only what the byte budget looks at."""

    def __init__(self, T, V, U, H, W, C, textured=False, tex=(2, 2)):
        self.faces, self.depths, self.uv = np.zeros((T, 3), np.uint32), np.zeros(V), np.zeros((U, 2))
        self.height, self.width, self.nb_colors = H, W, C
        self.textured = np.full(T, textured)
        self.texture = np.zeros(tex + (C,))


def test_algorithmic_bytes_are_the_contract_figures():
    # c5 (SURVEY.md 8d): 100.66 + 17.04 + 18.05 = 135.8 MB forward, + 10.03 = 145.8 MB adjoint, 281.5 MB per step
    c5 = Dims(T=1002528, V=501264, U=1, H=2048, W=2048, C=3)
    fwd, bwd = bench.algorithmic_bytes(c5)
    assert fwd == 4194304 * 24 + 1002528 * 17 + 501264 * 36 == 135751776
    assert bwd == fwd + 501264 * 20 == 145777056
    # textured term: T 12 + Nuv 8 + V 4 + Ht Wt C 4 read once per direction, Nuv 8 + V 4 + Ht Wt C 4 of gradients
    c3 = Dims(T=49928, V=24964, U=24964, H=1024, W=1024, C=3, textured=True, tex=(512, 512))
    fwd_t, bwd_t = bench.algorithmic_bytes(c3)
    plain = 1048576 * 24 + 49928 * 17 + 24964 * 36
    tex = 49928 * 12 + 24964 * 8 + 24964 * 4 + 512 * 512 * 3 * 4
    assert fwd_t == plain + tex
    assert bwd_t == plain + 24964 * 20 + tex + 24964 * 8 + 24964 * 4 + 512 * 512 * 3 * 4
    # per-kernel shares: the fused z pass owns the framebuffer planes and the colours, the binning pass the geometry
    k = bench.kernel_algorithmic_bytes(c5)
    assert k["bin"] == 1002528 * 17 + 501264 * 24
    assert k["tile_z"] + k["shade"] == fwd


def test_reference_arm_line(build_native):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c2",
                          "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600, check=True)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "fwd+bwd Mpixels/s" and line["unit"] == "Mpixels/s"
    assert line["higher_is_better"] is True and line["n_gpus"] == 1 and line["gpu_launches"] == 0
    assert line["steps"] == 2 == line["steps_requested"] and line["value"] > 0 and line["ms_per_step"] > 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 == line["e2e"]["d2h_bytes_per_step"]
    assert line["config"]["workload"].startswith("c2")


def test_dump_outputs_refused_beyond_one_process(tmp_path):
    """The shared gradients of a multi-process step are cleared after their all-reduce: nothing to dump there."""
    dump = tmp_path / "dump"
    for extra, env in ((["--impl", "reference"], {}), ([], {"WORLD_SIZE": "2"})):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(dump), *extra],
                             capture_output=True, text=True, timeout=120, env=dict(os.environ, **env))
        assert out.returncode == 2 and "--dump-outputs needs" in out.stderr, out.stderr
        assert not dump.exists()
