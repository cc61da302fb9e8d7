"""The host layer's CUDA resources have owners: only csrc/phovo_host.h allocates or frees device / pinned memory and
destroys streams and events, no hand-kept capacity field is left in the context or the batch state, and the helpers
both host translation units use are defined once."""
import os
import re

import pytest

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                    "photoconsistency-visual-odometry_b200", "csrc")
HOST_FILES = ["phovo_api.cu", "phovo_batch.cu", "phovo_ctx.h", "phovo_host.h"]


def _read(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _code(name):
    """The source without comments and string literals."""
    text = re.sub(r"//[^\n]*|/\*.*?\*/", "", _read(name), flags=re.S)
    return re.sub(r'"(?:\\.|[^"\\])*"', '""', text)


def _struct_body(text, name):
    m = re.search(r"\bstruct\s+%s\s*\{" % name, text)
    assert m, name
    depth, i = 1, m.end()
    while depth:
        depth += {"{": 1, "}": -1}.get(text[i], 0)
        i += 1
    return text[m.end():i - 1]


@pytest.mark.parametrize("name", ["phovo_api.cu", "phovo_batch.cu", "phovo_ctx.h"])
def test_no_raw_allocation_outside_host_header(name):
    calls = re.findall(r"\b(cudaMalloc|cudaMallocHost|cudaFree|cudaFreeHost|cudaStreamDestroy|cudaEventDestroy)\s*\(",
                       _code(name))
    assert calls == [], "%s calls %s; allocate through phovo_host.h's owners" % (name, sorted(set(calls)))


@pytest.mark.parametrize("struct, name", [("phovo_ctx", "phovo_ctx.h"), ("phovo_batch_state", "phovo_batch.cu")])
def test_no_capacity_fields(struct, name):
    body = _struct_body(_code(name), struct)
    fields = re.findall(r"\b(\w*_cap|lcap|bcap)\b(?!\s*\()", body)
    assert fields == [], "%s keeps capacity fields %s" % (struct, sorted(set(fields)))


@pytest.mark.parametrize("helper", ["CK", "ensure", "level_size", "depth_elt", "is_device_pointer"])
def test_shared_helpers_defined_once(helper):
    defs = []
    for name in HOST_FILES:
        code = _code(name)
        if helper == "CK":
            n = len(re.findall(r"#\s*define\s+CK\s*\(", code))
        else:
            # a function definition: return type, name, parameter list, body
            n = len(re.findall(r"^[ \t]*(?:template\s*<[^>]*>\s*)?(?:static\s+|inline\s+)*[\w:<>]+[\s*&]+%s\s*\([^;{)]*\)\s*"
                               r"(?:const\s*)?\{" % helper, code, flags=re.M))
        defs += [name] * n
    assert len(defs) == 1, "%s is defined in %s" % (helper, defs or "no file")
