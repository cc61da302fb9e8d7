"""Each numerical decision of the general path's solver loops is defined once: the Levenberg-Marquardt decision of Ceres
mode is shared by the host loop and the device loop (csrc/phovo_lm.h), the Gauss-Newton update by every device driver,
the level's LM options come out of the configuration in one builder, and the analytic Jacobian row has one body."""
import os
import re

import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    "photoconsistency-visual-odometry_b200", "csrc")
SOURCES = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h", ".cpp")))
LM_FUNCTIONS = ["expand_sym", "chol_solve6", "lm_log", "lm_start", "lm_propose", "lm_judge", "lm_update_radius"]
QUALIFIERS = r"(?:(?:static|inline|__host__|__device__|__global__|__forceinline__|__noinline__)\s+)*"


def _code(name):
    """The source without comments and string literals."""
    with open(os.path.join(CSRC, name)) as f:
        text = re.sub(r"//[^\n]*|/\*.*?\*/", "", f.read(), flags=re.S)
    return re.sub(r'"(?:\\.|[^"\\])*"', '""', text)


def _definitions(name, code):
    """Start offsets of the definitions of function `name` (return type, name, parameter list, body)."""
    pattern = (r"^[ \t]*(?:template\s*<[^>]*>\s*)?" + QUALIFIERS + r"[\w:<>]+[\s*&]+" + QUALIFIERS +
               r"%s\s*\([^;{]*\)\s*(?:const\s*)?\{" % name)
    return [m.start() for m in re.finditer(pattern, code, flags=re.M)]


def _defined_in(name):
    return [f for f in SOURCES for _ in _definitions(name, _code(f))]


def _function_bodies(code):
    """(name, start, end) of every function defined at namespace scope (its header starts in column 0)."""
    out = []
    header = re.compile(r"^(?:template\s*<[^>]*>\s*)?(?!namespace\b|struct\b|enum\b|#)[A-Za-z_]"
                        r"(?:__launch_bounds__\s*\([^)]*\)|[^;{}()])*?\b(?!__launch_bounds__)(\w+)\s*\([^;{]*\)\s*(?:const\s*)?\{", flags=re.M)
    for m in header.finditer(code):
        depth, i = 1, m.end()
        while depth:
            depth += {"{": 1, "}": -1}.get(code[i], 0)
            i += 1
        out.append((m.group(1), m.start(), i))
    return out


def _enclosing(code, pos):
    names = [n for n, a, b in _function_bodies(code) if a <= pos < b]
    assert names, "no function encloses offset %d" % pos
    return names[-1]


@pytest.mark.parametrize("name", LM_FUNCTIONS)
def test_lm_step_defined_once_for_host_and_device(name):
    assert _defined_in(name) == ["phovo_lm.h"], "%s is defined in %s" % (name, _defined_in(name) or "no file")
    twins = [f for f in SOURCES if re.search(r"\b%s_dev\b" % name, _code(f))]
    assert twins == [], "%s has a device twin in %s" % (name, twins)


@pytest.mark.parametrize("name", ["phovo_api.cu", "kernels_align.cu"])
def test_both_lm_drivers_include_the_shared_header(name):
    with open(os.path.join(CSRC, name)) as f:
        assert re.search(r'^#include\s+"phovo_lm\.h"', f.read(), flags=re.M), name


def test_gauss_newton_solve_in_one_function():
    code = _code("kernels_align.cu")
    callers = {_enclosing(code, m.start()) for m in re.finditer(r"\bsolve6_ldlt\s*\(", code)}
    assert len(callers) == 1, "solve6_ldlt is called from %s" % (sorted(callers) or "no function")


def test_analytic_jacobian_defined_once():
    assert _defined_in("analytic_jacobian") == ["phovo_device.cuh"]
    for f in SOURCES:
        assert not re.search(r"\banalytic_jacobian_(core|row)\b", _code(f)), f


@pytest.mark.parametrize("field", ["initial_trust_region_radius", "max_trust_region_radius", "min_relative_decrease"])
def test_lm_options_read_only_by_the_builder(field):
    readers = []
    for f in SOURCES:
        if f == "yaml_config.cpp":   # the parser fills the configuration
            continue
        code = _code(f)
        readers += [(f, _enclosing(code, m.start())) for m in re.finditer(r"\b%s\s*\[" % field, code)]
    assert readers and set(readers) == {("phovo_lm.h", "lm_params")}, readers
