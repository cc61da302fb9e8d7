"""Host-side logic that runs without a GPU: the YAML reader (ReadConfigurationFile,
AN:581-607 / CE:526-576), constructor defaults (AN:430-443), eigenPose (BASE:47-71), and the
C-ABI surface: the library loads and exports every symbol include/phovo_b200.h declares."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from conftest import REF_CONFIG_DIR, ROOT


def test_library_exports_every_declared_symbol(phovo):
    header = open(os.path.join(ROOT, "include", "phovo_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(phovo_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 40
    lib = C.CDLL(phovo.capi.LIB_PATH)
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing
    # and the ctypes table covers the same set
    assert declared == set(phovo.capi.SIGNATURES), declared ^ set(phovo.capi.SIGNATURES)


def test_struct_layout_matches_c(phovo, oracle):
    # the oracle is compiled from the same header: sizes must agree with the ctypes mirrors
    assert C.sizeof(phovo.capi.Config) == C.sizeof(oracle.Config) == 8 + 4 * 10 * 2 + 8 * 10 * 3 + 16 + 8 + 8 * 10 * 7 + 16
    assert C.sizeof(phovo.capi.IterStats) == C.sizeof(oracle.IterStats) == 16 + 8 * (21 + 6 + 3 + 12)


def test_constructor_defaults(phovo):
    cfg = phovo.default_config()          # AN:430-443
    assert cfg.mode == 0 and cfg.num_levels == 5
    assert list(cfg.max_num_iterations)[:5] == [0, 0, 5, 20, 50]
    assert all(v == 0.0625 for v in list(cfg.grad_scale)[:5])
    assert all(v == 1.0 for v in list(cfg.lambda_step)[:5])
    assert all(v == 300.0 for v in list(cfg.min_gradient_norm)[:5])
    assert (cfg.min_depth, cfg.max_depth) == (0.3, 5.0)


@pytest.mark.parametrize("name", ["config_4_level_optimization_analytic", "config_5_level_optimization_analytic",
                                  "config_6_level_optimization_analytic", "config_only_level_0_analytic",
                                  "config_5_level_optimization_ceres", "config_3_level_optimization_ceres",
                                  "config_only_level_1_ceres"])
def test_yaml_reader(phovo, tmp_path, name):
    path = phovo.configs.write_yaml(name, str(tmp_path))
    cfg = phovo.parse_config_yaml(path)
    want = phovo.configs.REFERENCE_CONFIGS[name]
    n = want[phovo.configs.K_LEVELS]
    assert cfg.num_levels == n
    assert list(cfg.max_num_iterations)[:n] == list(want[phovo.configs.K_ITERS])[:n]
    assert all(cfg.max_num_iterations[l] == 0 for l in range(n, phovo.MAXL))
    assert list(cfg.blur_filter_size)[:n] == list(want[phovo.configs.K_BLUR])[:n]
    assert list(cfg.grad_scale)[:n] == [float(v) for v in want[phovo.configs.K_GRAD][:n]]
    if phovo.configs.K_MINGRAD in want:
        assert list(cfg.min_gradient_norm)[:n] == [float(v) for v in want[phovo.configs.K_MINGRAD][:n]]
        assert cfg.visualize_iterations == want["visualizeIterations"]
    if phovo.configs.K_RMIN in want:
        # ragged vector (SURVEY H8): missing entries repeat the last one
        given = want[phovo.configs.K_RMIN]
        got = list(cfg.min_trust_region_radius)[:n]
        assert got == [float(given[i] if i < len(given) else given[-1]) for i in range(n)]
        assert list(cfg.min_relative_decrease)[:n] == [float(v) for v in want[phovo.configs.K_ETA][:n]]
        assert cfg.num_threads == want["num_threads"]


@pytest.mark.skipif(not os.path.isdir(REF_CONFIG_DIR), reason="needs the original project's config_files: set REF to a checkout of it")
def test_config_table_matches_reference_files(phovo, tmp_path):
    """The table in configs.py against the reference's own files, read by our parser AND by
    OpenCV's FileStorage (what the reference itself uses)."""
    cv2 = pytest.importorskip("cv2")
    for name, want in phovo.configs.REFERENCE_CONFIGS.items():
        ref_path = os.path.join(REF_CONFIG_DIR, name + ".yml")
        assert os.path.exists(ref_path), ref_path
        a = phovo.parse_config_yaml(ref_path)
        b = phovo.parse_config_yaml(phovo.configs.write_yaml(name, str(tmp_path)))
        assert bytes(a) == bytes(b), name
        fs = cv2.FileStorage(ref_path, cv2.FILE_STORAGE_READ)
        assert int(fs.getNode("numOptimizationLevels").real()) == a.num_levels
        node = fs.getNode("max_num_iterations (at each level)")
        vals = [int(node.at(i).real()) for i in range(node.size())]
        assert vals[:a.num_levels] == list(a.max_num_iterations)[:a.num_levels]
        node = fs.getNode("imageGradientsScalingFactor (at each level)")
        vals = [node.at(i).real() for i in range(node.size())]
        assert vals[:a.num_levels] == list(a.grad_scale)[:a.num_levels]


def test_yaml_errors(phovo, tmp_path):
    with pytest.raises(phovo.PhovoError) as e:
        phovo.parse_config_yaml(str(tmp_path / "does_not_exist.yml"))
    assert e.value.code == phovo.capi.E_CONFIG
    p = tmp_path / "bad.yml"
    p.write_text("%YAML:1.0\nnumOptimizationLevels: 3\nmax_num_iterations (at each level): [1, x, 3]\n")
    with pytest.raises(phovo.PhovoError):
        phovo.parse_config_yaml(str(p))
    p.write_text("%YAML:1.0\nmax_num_iterations (at each level): [1, 2, 3]\n")
    with pytest.raises(phovo.PhovoError):
        phovo.parse_config_yaml(str(p))
    p.write_text("%YAML:1.0\nnumOptimizationLevels: 2\nblurFilterSize (at each level): [0, 4]\n")
    with pytest.raises(phovo.PhovoError):
        phovo.parse_config_yaml(str(p))      # cv::GaussianBlur needs an odd size
    # multi-line flow sequence and comments
    p.write_text("%YAML:1.0\n# comment\nnumOptimizationLevels: 2\nmax_num_iterations (at each level): [7,\n   9]\n")
    cfg = phovo.parse_config_yaml(str(p))
    assert list(cfg.max_num_iterations)[:2] == [7, 9]


def test_state_to_rt_is_eigenpose(phovo, oracle):
    rng = np.random.default_rng(0)
    for _ in range(20):
        s = rng.uniform(-1, 1, 6)
        Rt = phovo.state_to_rt(s)
        want = phovo.synth.state_to_rt(s)
        assert np.max(np.abs(Rt - want)) < 1e-15
        assert abs(np.linalg.det(Rt[:3, :3]) - 1) < 1e-14
        o = np.zeros(16)
        oracle.lib().pho_state_to_rt(s.ctypes.data_as(C.POINTER(C.c_double)), o.ctypes.data_as(C.POINTER(C.c_double)))
        assert np.array_equal(o.reshape(4, 4), Rt)


def test_no_cpu_fallback_without_gpu(phovo):
    """The product fails loudly when no CUDA device can be opened (there is no CPU path)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    with pytest.raises(phovo.PhovoError) as e:
        phovo.CPhotoconsistencyOdometryCuda()
    assert e.value.code == phovo.capi.E_CUDA
    assert "no CPU path" in str(e.value)


def test_product_does_not_reference_oracle():
    """Nothing under the product package or include/ may import, link or name the oracle."""
    pkg = os.path.join(ROOT, "photoconsistency-visual-odometry_b200")
    for base in (pkg, os.path.join(ROOT, "include")):
        for dp, _, files in os.walk(base):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                    txt = open(os.path.join(dp, f), errors="ignore").read()
                    assert "phovo_oracle" not in txt and "oracle_py" not in txt and "np_restatement" not in txt, f
