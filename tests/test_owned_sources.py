"""Every CUDA buffer, event and stream of the product is held by an owner of csrc/owned.h, which
releases it on every return path.  A direct allocation, free, or handle creation or destruction
anywhere else would be one more thing to keep in step by hand."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "oxli_b200", "csrc")

CALL = re.compile(r"\b(cudaMalloc\w*|cudaFree\w*|cudaEventCreate\w*|cudaEventDestroy|cudaStreamCreate\w*|cudaStreamDestroy)\s*\(")
# top-level function definitions (a line that starts in column 0 and names a function)
DEFINITION = re.compile(r"^[A-Za-z][^\n;]*?\b(\w+)\s*\(", re.M)
# the ABI's own memory helpers allocate for the caller, who owns and frees what they return
PASS_THROUGH = {"oxg_pinned_alloc", "oxg_pinned_free", "oxg_device_alloc", "oxg_device_free"}


def strip_comments(text: str) -> str:
    text = re.sub(r"/\*.*?\*/", lambda m: re.sub(r"[^\n]", " ", m.group()), text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def unowned_calls(text: str) -> list[str]:
    code = strip_comments(text)
    found = []
    for m in CALL.finditer(code):
        defs = [d.group(1) for d in DEFINITION.finditer(code, 0, m.start())]
        if defs and defs[-1] in PASS_THROUGH:
            continue
        found.append(f"line {code.count(chr(10), 0, m.start()) + 1}: {m.group(1)}")
    return found


def test_resources_are_created_and_released_by_owners_only():
    sources = [f for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h", ".inc", ".cpp"))]
    assert "owned.h" in sources and "capi.cu" in sources
    bad = {f: calls for f in sources if f != "owned.h"
           for calls in [unowned_calls(open(os.path.join(CSRC, f)).read())] if calls}
    assert not bad, bad


def test_the_scan_sees_calls_and_skips_comments_and_pass_throughs():
    text = """
oxg_status oxg_device_alloc(int device, uint64_t bytes, void **d_out) {
    CU(cudaMalloc(d_out, bytes));
}
// cudaFree(p) in a comment
/* cudaEventCreate(&e) in a block comment */
oxg_status other(void) {
    CU(cudaStreamCreateWithFlags(&s, 0));
}
"""
    assert [c.split(": ")[1] for c in unowned_calls(text)] == ["cudaStreamCreateWithFlags"]
