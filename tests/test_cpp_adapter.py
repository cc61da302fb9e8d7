"""The C++ drop-in adapter (include/CPhotoconsistencyOdometryCuda.h), compiled against the reference's
abstract class and matrix types (its own phovo/include/CPhotoconsistencyOdometry.h + Matrix.h when
REF names a checkout of the original project, else the stand-in tests/cpp/shim/CPhotoconsistencyOdometry.h;
OpenCV / Eigen are the stand-ins of oracle/shim), checked against the CPU oracle:

  * tests/cpp/frame_alignment_app.cpp -- headless mirror of both apps' main() (strided cv::Mat_ inputs,
    the VO loop, warpImage through the adapter);
  * the reference's apps/PhotoconsistencyFrameAlignment/PhotoconsistencyFrameAlignment.cpp and
    apps/PhotoconsistencyVisualOdometry/PhotoconsistencyVisualOdometry.cpp THEMSELVES with exactly the
    INTEGRATION.md patch applied (USE_PHOTOCONSISTENCY_ODOMETRY_METHOD == 3), built by
    tests/cpp/build_adapter_test.sh into tests/cpp/_build/ (git-ignored) from the checkout REF names;
    their tests skip without one.
"""
import os
import subprocess

import numpy as np
import pytest

from helpers import assert_pose_close
from test_gpu_parity import conv_cfg

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
APP = os.path.join(ROOT, "tests", "cpp", "_build", "frame_alignment_app")
REF_APP = os.path.join(ROOT, "tests", "cpp", "_build", "reference_frame_alignment")
REF_VO_APP = os.path.join(ROOT, "tests", "cpp", "_build", "reference_visual_odometry")


def build_app():
    subprocess.check_call(["bash", os.path.join(ROOT, "tests", "cpp", "build_adapter_test.sh")], stdout=subprocess.DEVNULL)
    return APP


def build_reference_apps():
    build_app()
    if not os.environ.get("REF"):
        pytest.skip("the reference apps are built from a checkout of the original project: set REF to one")


def test_adapter_compiles_and_fails_loudly_without_gpu(phovo, tmp_path):
    """No CPU fallback behind the C++ surface either: without a device the constructor throws."""
    app = build_app()
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    cfg = phovo.configs.write_yaml("config_4_level_optimization_analytic", str(tmp_path))
    args = [app, "align", cfg, "4", "4", "1", "1", "1", "1", "a", "b", "c", "d"]
    r = subprocess.run(args, capture_output=True, text=True)
    assert r.returncode == 3 and "phovo_create" in r.stderr and "no CPU path" in r.stderr, (r.returncode, r.stderr)


def write_pgm(path, img):
    """Binary PGM, 8 bit or 16 bit big endian: the one format the stand-in cv::imread reads."""
    img = np.ascontiguousarray(img)
    maxval = 255 if img.dtype == np.uint8 else 65535
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n%d\n" % (img.shape[1], img.shape[0], maxval))
        f.write(img.tobytes() if img.dtype == np.uint8 else img.astype(">u2").tobytes())


def reference_app_inputs(phovo, tmp_path, seed):
    """Frames for the reference app's own main(): 8-bit gray + 16-bit depth in millimetres, which it
    scales with `img * 1. / 1000.` (FrameAlignment.cpp:74-81).  Returns the doubles it ends up with."""
    K = phovo.synth.K_FRAME_ALIGNMENT                       # hard-coded in the app (FrameAlignment.cpp:69-71)
    g0, d0, g1, d1 = phovo.synth.make_pair(480, 640, K=K, seed=seed)
    mm0, mm1 = np.rint(d0 * 1000.).astype(np.uint16), np.rint(d1 * 1000.).astype(np.uint16)
    paths = [str(tmp_path / n) for n in ("gray0.pgm", "depth0.pgm", "gray1.pgm", "depth1.pgm")]
    for p, img in zip(paths, (g0, mm0, g1, mm1)):
        write_pgm(p, img)
    return K, g0, mm0.astype(np.float64) * (1. / 1000.), g1, paths


def test_reference_app_with_the_integration_patch_builds_and_fails_loudly_without_gpu(phovo, tmp_path):
    """The reference's own FrameAlignment main() + the METHOD == 3 branch compiles against the real
    CPhotoconsistencyOdometry.h / Matrix.h; without a device the adapter's constructor throws (the app
    has no handler: it terminates, it does not fall back to anything)."""
    build_reference_apps()
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present: covered by the gpu tests")
    K, g0, d0, g1, paths = reference_app_inputs(phovo, tmp_path, 22)
    yml = phovo.configs.write_yaml("config_4_level_optimization_analytic", str(tmp_path))
    r = subprocess.run([REF_APP, yml] + paths, capture_output=True, text=True)
    assert r.returncode != 0 and "phovo_create" in r.stderr, (r.returncode, r.stderr)


@pytest.mark.gpu
def test_reference_frame_alignment_app_method_3_matches_oracle(phovo, oracle, tmp_path):
    """apps/PhotoconsistencyFrameAlignment/PhotoconsistencyFrameAlignment.cpp, unmodified but for the
    INTEGRATION.md patch, run on the GPU: the Rt it prints (:109-110) equals the oracle's."""
    build_reference_apps()
    K, g0, d0, g1, paths = reference_app_inputs(phovo, tmp_path, 22)
    name = "config_4_level_optimization_analytic"
    yml = phovo.configs.write_yaml(name, str(tmp_path))
    r = subprocess.run([REF_APP, yml] + paths, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    at = lines.index("main::Rt eigen:")
    Rt = np.array([[float(x) for x in ln.split()] for ln in lines[at + 1:at + 5]])
    assert any(ln.startswith("Time = ") for ln in lines)
    cfg = phovo.configs.to_config(name, phovo.capi)
    o = oracle.Oracle(conv_cfg(oracle, cfg), K)
    o.set_source(g0, d0)
    o.set_target(g1)
    o.set_initial_state(np.zeros(6))
    o.optimize()
    assert len(o.iter_stats()) > 0
    assert np.max(np.abs(Rt - o.rt())) < 1e-10
    assert np.max(np.abs(Rt[:3, 3] - o.state()[:3])) < 1e-10


@pytest.mark.gpu
def test_frame_alignment_app_matches_oracle(phovo, oracle, tmp_path):
    """PhotoconsistencyFrameAlignment.cpp:90-105 through the adapter, strided cv::Mat_ inputs."""
    app = build_app()
    K = phovo.synth.K_FRAME_ALIGNMENT
    g0, d0, g1, _ = phovo.synth.make_pair(480, 640, K=K, seed=21)
    name = "config_4_level_optimization_analytic"
    yml = phovo.configs.write_yaml(name, str(tmp_path))
    paths = {}
    for nm, arr in (("g0", g0), ("d0", d0.astype(np.float64)), ("g1", g1), ("d1", np.zeros_like(d0, dtype=np.float64))):
        paths[nm] = str(tmp_path / (nm + ".bin"))
        arr.tofile(paths[nm])
    args = [app, "align", yml, "480", "640", repr(float(K[0, 0])), repr(float(K[1, 1])), repr(float(K[0, 2])), repr(float(K[1, 2])),
            paths["g0"], paths["d0"], paths["g1"], paths["d1"], "24"]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    out = {ln.split()[0]: ln.split()[1:] for ln in r.stdout.splitlines() if ln.strip()}
    state = np.array([float(x) for x in out["state"]])
    Rt = np.array([float(x) for x in out["Rt"]]).reshape(4, 4)
    cfg = phovo.configs.to_config(name, phovo.capi)
    o = oracle.Oracle(conv_cfg(oracle, cfg), K)
    o.set_source(g0, d0)
    o.set_target(g1)
    o.set_initial_state(np.zeros(6))
    o.optimize()
    assert int(out["iterations"][0]) == len(o.iter_stats())
    assert_pose_close(state, o.state(), "C++ adapter")
    assert np.max(np.abs(state - o.state())) < 1e-10
    assert np.max(np.abs(Rt - o.rt())) < 1e-10
    # the app's warpImage step through the adapter: same image as the Python binding produces
    odo = phovo.CPhotoconsistencyOdometryCuda()
    w = odo.WarpImage(g0, d0.astype(np.float64), Rt, K)
    mask = w > 0
    assert int(out["warped"][0]) == int(mask.sum())
    assert int(out["warped"][1]) == int(np.abs(w.astype(np.int64) - g1.astype(np.int64))[mask].sum())


@pytest.mark.gpu
def test_visual_odometry_app_trajectory_matches_oracle(phovo, oracle, tmp_path):
    """PhotoconsistencyVisualOdometry.cpp:212-259: zero initial state every frame, pose *= Rt^-1,
    TUM line `ts tx ty tz qx qy qz qw`; source pyramid reused on the device between frames."""
    app = build_app()
    K = phovo.synth.K_VISUAL_ODOMETRY
    n = 5
    frames = [phovo.synth.make_sequence_frame(k, 240, 320, K=K) for k in range(n)]
    for k, (g, d) in enumerate(frames):
        g.tofile(str(tmp_path / ("gray_%d.bin" % k)))
        d.astype(np.float64).tofile(str(tmp_path / ("depth_%d.bin" % k)))
    name = "config_5_level_optimization_analytic"
    yml = phovo.configs.write_yaml(name, str(tmp_path))
    traj = str(tmp_path / "trajectory.txt")
    args = [app, "vo", yml, "240", "320", repr(float(K[0, 0])), repr(float(K[1, 1])), repr(float(K[0, 2])), repr(float(K[1, 2])), str(n),
            str(tmp_path / "gray_%d.bin"), str(tmp_path / "depth_%d.bin"), traj]
    r = subprocess.run(args, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.loadtxt(traj)
    assert got.shape == (n - 1, 8)
    cfg = phovo.configs.to_config(name, phovo.capi)
    pose = np.eye(4)
    for k in range(1, n):
        o = oracle.Oracle(conv_cfg(oracle, cfg), K)
        o.set_source(*frames[k - 1])
        o.set_target(frames[k][0])
        o.set_initial_state(np.zeros(6))
        o.optimize()
        pose = pose @ np.linalg.inv(o.rt())
        assert np.max(np.abs(got[k - 1, 1:4] - pose[:3, 3])) < 1e-9
        q = got[k - 1, 4:8]
        x, y, z, w = q
        R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                      [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                      [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
        assert abs(np.linalg.norm(q) - 1) < 1e-12 and np.max(np.abs(R - pose[:3, :3])) < 1e-9


@pytest.mark.gpu
def test_reference_visual_odometry_app_method_3_trajectory_matches_oracle(phovo, oracle, tmp_path):
    """apps/PhotoconsistencyVisualOdometry/PhotoconsistencyVisualOdometry.cpp, unmodified but for the INTEGRATION.md
    patch, on a recorded sequence (rgb.txt / depth.txt + image files read by the reference's own CCameraRecord /
    CImageReader): the TUM trajectory it writes (:240-243) equals the oracle's frame-by-frame loop."""
    build_reference_apps()
    K = phovo.synth.K_VISUAL_ODOMETRY                      # hard-coded in the app (VisualOdometry.cpp:171-173)
    n = 5
    os.makedirs(tmp_path / "rgb"); os.makedirs(tmp_path / "depth")
    frames, stamps = [], []
    with open(tmp_path / "rgb.txt", "w") as fr, open(tmp_path / "depth.txt", "w") as fd:
        fr.write("# color images\n# timestamp filename\n"); fd.write("# depth maps\n# timestamp filename\n")
        for k in range(n):
            g, d = phovo.synth.make_sequence_frame(k, 480, 640, K=K)
            raw = np.rint(d * 5000.).astype(np.uint16)                     # the app scales by 1/5000 (:163)
            write_pgm(str(tmp_path / "rgb" / ("%04d.pgm" % k)), g)
            write_pgm(str(tmp_path / "depth" / ("%04d.pgm" % k)), raw)
            stamp = 1305031102.175304 + 0.033 * k
            fr.write("%.6f rgb/%04d.pgm\n" % (stamp, k)); fd.write("%.6f depth/%04d.pgm\n" % (stamp, k))
            frames.append((g, raw.astype(np.float64) * (1. / 5000.))); stamps.append(stamp)
    name = "config_5_level_optimization_analytic"
    yml = phovo.configs.write_yaml(name, str(tmp_path))
    traj = str(tmp_path / "out" / "trajectory.txt")                       # the app creates the directory (:109-116)
    r = subprocess.run([REF_VO_APP, yml, str(tmp_path), traj], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = np.loadtxt(traj)
    assert got.shape == (n - 1, 8)
    cfg = phovo.configs.to_config(name, phovo.capi)
    pose = np.eye(4)
    for k in range(1, n):
        o = oracle.Oracle(conv_cfg(oracle, cfg), K)
        o.set_source(*frames[k - 1])
        o.set_target(frames[k][0])
        o.set_initial_state(np.zeros(6))
        o.optimize()
        pose = pose @ np.linalg.inv(o.rt())
        assert abs(got[k - 1, 0] - stamps[k]) < 1e-5
        assert np.max(np.abs(got[k - 1, 1:4] - pose[:3, 3])) < 1e-9
        x, y, z, w = got[k - 1, 4:8]
        R = np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                      [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                      [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])
        assert np.max(np.abs(R - pose[:3, :3])) < 1e-9
