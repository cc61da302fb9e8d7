"""Every driver of Optimize() runs through the same host code: one coarse-to-fine level walk (for_each_level in
csrc/phovo_ctx.h), one upload of the initial state for the drivers, one function that records a launch the device
refused, and one record of the paths that failed on a context (no per-driver flags beside phovo_ctx::execution)."""
import os
import re

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    "photoconsistency-visual-odometry_b200", "csrc")
SOURCES = sorted(f for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h", ".cpp")))


def _code(name):
    """The source without comments and string literals."""
    with open(os.path.join(CSRC, name)) as f:
        text = re.sub(r"//[^\n]*|/\*.*?\*/", "", f.read(), flags=re.S)
    return re.sub(r'"(?:\\.|[^"\\])*"', '""', text)


def _block_end(code, i):
    """Offset just past the brace that closes the block whose opening brace ends at offset i."""
    depth = 1
    while depth:
        depth += {"{": 1, "}": -1}.get(code[i], 0)
        i += 1
    return i


def _function_bodies(code):
    """(name, start, end) of every function defined at namespace scope (its header starts in column 0)."""
    header = re.compile(r"^(?:template\s*<[^>]*>\s*)?(?!namespace\b|struct\b|enum\b|#)[A-Za-z_]"
                        r"(?:__launch_bounds__\s*\([^)]*\)|[^;{}()])*?\b(?!__launch_bounds__)(\w+)\s*\([^;{]*\)\s*(?:const\s*)?\{", flags=re.M)
    return [(m.group(1), m.start(), _block_end(code, m.end())) for m in header.finditer(code)]


def _enclosing(code, pos):
    names = [n for n, a, b in _function_bodies(code) if a <= pos < b]
    assert names, "no function encloses offset %d" % pos
    return names[-1]


def test_one_coarse_to_fine_walk():
    walk = re.compile(r"\bfor\s*\(\s*int\s+(\w+)\s*=\s*[\w.>-]*num_levels\s*-\s*1\s*;\s*\1\s*>=\s*0\s*;\s*(?:--\s*\1|\1\s*--)\s*\)")
    found = [f for f in SOURCES for _ in walk.finditer(_code(f))]
    assert found == ["phovo_ctx.h"], "level loops counting down from num_levels - 1 in %s; use for_each_level" % (found or "no file")


def test_initial_state_uploaded_from_three_functions():
    # the drivers' shared upload, the graph capture (it uploads from a device copy), and eval_at (a state, no log)
    code = _code("phovo_api.cu")
    callers = {_enclosing(code, m.start()) for m in re.finditer(r"\blaunch_set_state\s*\(", code)}
    assert len(callers) <= 3, "launch_set_state is called from %s" % sorted(callers)


def test_refused_launch_recorded_in_one_function():
    # a fallback keeps the CUDA error text in a context field other than the error of the call (err)
    code = _code("phovo_api.cu")
    writers = {_enclosing(code, m.start()) for m in re.finditer(r"\bctx->(\w+)\s*=[^;]*\bcudaGetErrorString\s*\(", code)
               if m.group(1) != "err"}
    assert len(writers) == 1, "path fallbacks keep their reason in %s" % (sorted(writers) or "no function")


def test_context_keeps_no_per_driver_flags():
    code = _code("phovo_ctx.h")
    m = re.search(r"\bstruct\s+phovo_ctx\s*\{", code)
    body = code[m.end():_block_end(code, m.end())]
    fields = re.findall(r"\b(use_graph|last_used_graph|\w+_broken)\b", body)
    assert fields == [], "phovo_ctx keeps %s beside execution / failed_paths / last_path" % sorted(set(fields))
