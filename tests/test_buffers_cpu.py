"""CPU test of device-memory ownership in the native library: every cudaMalloc / cudaFree goes through disn::DevBuf
(disn_b200/csrc/common.cuh), whose destructor frees what it owns, so no buffer is freed twice or left out of a teardown."""
import collections
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "disn_b200", "csrc")
RAW_CALL = re.compile(r"\b(cudaMalloc|cudaFree|cudaMallocHost|cudaFreeHost)\s*\(")
# a definition starting in column 0: `class X {`, `struct X {` or the line that names a function, `int disn::f(`
DEFINITION = re.compile(r"^(?:class|struct)\s+(\w+)|^[A-Za-z_][^;{}()]*?\b([\w:]+)\s*\(")

# (file, enclosing definition, call) -> count of the raw calls that are allowed to remain
ALLOWED = {
    ("common.cuh", "DevBuf", "cudaMalloc"): 1,
    ("common.cuh", "DevBuf", "cudaFree"): 1,
    # CUDA IPC buffer for the multi-GPU gather: its lifetime belongs to the caller
    ("api.cu", "disn_shared_alloc", "cudaMalloc"): 1,
    ("api.cu", "disn_shared_alloc", "cudaFree"): 1,
    ("api.cu", "disn_shared_close", "cudaFree"): 1,
    # the two pinned host words: h_status (disn_create) and mc_totals_host (mc_run), both freed in disn_destroy
    ("api.cu", "disn_create", "cudaMallocHost"): 1,
    ("mc.cu", "mc_run", "cudaMallocHost"): 1,
    ("api.cu", "disn_destroy", "cudaFreeHost"): 2,
}


def _raw_calls():
    found, where = collections.Counter(), collections.defaultdict(list)
    for fn in sorted(os.listdir(CSRC)):
        if not fn.endswith((".cu", ".cuh", ".h")):
            continue
        owner = None
        with open(os.path.join(CSRC, fn)) as f:
            for lineno, line in enumerate(f, 1):
                code = line.split("//")[0]
                m = DEFINITION.match(code)
                if m:
                    owner = (m.group(1) or m.group(2)).split("::")[-1]
                for call in RAW_CALL.findall(code):
                    found[(fn, owner, call)] += 1
                    where[(fn, owner, call)].append("%s:%d" % (fn, lineno))
    return found, where


def test_device_memory_is_owned_by_devbuf():
    found, where = _raw_calls()
    extra = {k: where[k] for k in found if found[k] > ALLOWED.get(k, 0)}
    assert not extra, "raw CUDA allocation calls outside disn::DevBuf (use a DevBuf member or local): %s" % extra
    assert found == collections.Counter(ALLOWED), "an allowed raw call moved or disappeared: %s" % dict(found)
