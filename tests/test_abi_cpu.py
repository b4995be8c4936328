"""CPU-side checks of the C-ABI library: it loads, exports every symbol include/b200tag.h declares,
its pure-host entry points agree with the oracle, and without a GPU it fails loudly (no fallback)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    from ros_vision_b200 import build, detector
    build.build_native()
    return detector.load_library()


def test_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "b200tag.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(b200tag_[a-z_0-9]+)\s*\(", hdr))
    assert len(names) >= 20
    for n in sorted(names):
        assert hasattr(lib, n), f"libb200tag.so does not export {n}"
    assert lib.b200tag_version() == 2


def test_struct_layouts_match_header(tmp_path):
    """numpy / ctypes mirrors in ros_vision_b200/detector.py against sizeof() from the C header."""
    import subprocess
    from ros_vision_b200 import detector as D
    names = ["b200tag_detection", "b200tag_quad", "b200tag_blob", "b200tag_lfp", "b200tag_moments", "b200tag_fit_quad",
             "b200tag_point", "b200tag_config", "b200tag_frame_info"]
    src = tmp_path / "sz.c"
    src.write_text('#include "b200tag.h"\n#include <stdio.h>\nint main(void){' +
                   "".join(f'printf("%zu\\n", sizeof({n}));' for n in names) + "return 0;}")
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    mirrors = [D.DETECTION_DT.itemsize, D.QUAD_DT.itemsize, D.BLOB_DT.itemsize, D.LFP_DT.itemsize, D.MOMENTS_DT.itemsize,
               D.FIT_QUAD_DT.itemsize, D.POINT_DT.itemsize, C.sizeof(D.Config), C.sizeof(D.FrameInfo)]
    assert sizes == mirrors


def test_default_config_matches_node_settings(lib):
    """apriltags_cuda_detector.cu:142-147 + apriltag_detector_create() defaults."""
    from ros_vision_b200 import detector as D
    cfg = D.default_config(1280, 800, "yuyv")
    assert (cfg.quad_decimate, cfg.quad_sigma, cfg.refine_edges, cfg.max_nmaxima) == (2, 0.0, 1, 10)
    assert cfg.min_white_black_diff == 5 and cfg.min_cluster_pixels == 5 and cfg.decode_sharpening == 0.25
    assert abs(cfg.cos_critical_rad - np.cos(np.deg2rad(10))) < 1e-6 and cfg.max_line_fit_mse == 10.0


def test_undistort_matches_oracle(lib, oracle):
    from ros_vision_b200 import detector as D
    cam = (905.495617, 609.916016, 907.909470, 352.682645)
    dist = (0.059238, -0.075154, -0.003801, 0.001113, 0.0)
    cfg = oracle.make_config(1920, 1080, camera=cam, dist=dist)
    for u0, v0 in [(10.5, 20.25), (960.0, 540.0), (1300.0, 777.0), (1800.0, 1000.0)]:
        u, v, ok = D.GpuDetector.UnDistort(u0, v0, cam, dist)
        cu, cv = C.c_double(u0), C.c_double(v0)
        ok2 = oracle.lib().orc_undistort(C.byref(cu), C.byref(cv), C.byref(cfg))
        assert (u, v, ok) == (cu.value, cv.value, bool(ok2))


def test_no_gpu_means_loud_failure(lib):
    """The product path must not degrade to a CPU implementation.  The detector is created in a child process that
    sees no CUDA device (CUDA_VISIBLE_DEVICES=""), so the check runs on machines with a GPU as well."""
    import subprocess
    import sys
    child = "\n".join([
        "import sys, pytest",
        f"sys.path.insert(0, {ROOT!r})",
        "from ros_vision_b200 import detector as D",
        "with pytest.raises(D.B200TagError, match='CUDA|device'):",
        "    D.GpuDetector(640, 480, 'gray')",
    ])
    r = subprocess.run([sys.executable, "-c", child], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_does_not_touch_the_oracle():
    """Nothing under ros_vision_b200/ may import, link or execute oracle/."""
    for dirpath, _, files in os.walk(os.path.join(ROOT, "ros_vision_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".h", ".cc", ".cpp")):
                src = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "pyoracle" not in src and "liboracle" not in src and "apriltag_oracle" not in src, f
                for line in src.splitlines():
                    s = line.strip()
                    if s.startswith(("import ", "from ", "#include")):
                        assert "oracle" not in s, (f, line)
