"""The C-ABI library builds, loads without a GPU and exports exactly what include/coper.h declares."""
import os
import re

from coper_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    src = open(os.path.join(ROOT, "include", "coper.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(coper_[A-Za-z0-9_]+)\s*\(", src)))


def test_builds_and_loads():
    build.build()
    lib = _lib.load()
    assert lib.coper_version() >= 100
    assert lib.coper_status_string(-3) == b"unsupported configuration"


def test_every_declared_symbol_is_exported_and_bound():
    build.build()
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), "declared in coper.h but not exported: " + n
        assert n in _lib.SIGNATURES, "declared in coper.h but not bound in _lib.SIGNATURES: " + n
    for n in _lib.SIGNATURES:
        assert n in names, "bound but not declared in coper.h: " + n


def test_python_constants_mirror_the_header():
    """The limits and flags _lib repeats for its callers equal the values include/coper.h defines."""
    src = open(os.path.join(ROOT, "include", "coper.h")).read()
    defs = {k: int(v) for k, v in re.findall(r"#define (COPER_\w+) (\d+)", src)}
    for name in ("TOPK_MAX", "SEGSCATTER_SMALL_M", "SUMSQ_BLOCKS", "MT_CHUNK", "CPG_BWD_REUSE_FWD",
                 "CPG_BWD_INPUT_GRADS_ONLY", "CPG_BWD_WEIGHT_GRADS_ONLY", "CPG_BWD_DCB_ACCUMULATE"):
        assert defs["COPER_" + name] == getattr(_lib, name), name


def test_workspace_queries_run_without_gpu():
    lib = _lib.load()
    assert lib.coper_colstats_chunks(1000) == 16
    assert lib.coper_cpg_fc_fwd_workspace_bytes(512, 8, 4608, 200, 0) > 0
    assert lib.coper_score1n_bce_workspace_bytes(512, 40943, 200, 0) > 0


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "coper_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt, f


def test_integration_doc_names_every_entry_point():
    """INTEGRATION.md is the map from the C ABI to the reference call sites: every function of include/coper.h must be
    named in it."""
    import os
    import re
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    header = open(os.path.join(root, "include", "coper.h")).read()
    doc = open(os.path.join(root, "INTEGRATION.md")).read()
    syms = sorted(set(re.findall(r"\b(coper_[A-Za-z0-9_]+)\s*\(", header)))
    # `coper_bn_*`-style wildcards and `coper_conv_fwd`, `coper_conv_bwd` lists both count
    # (a bare `coper_*...` would match everything: only wildcards that name a family count)
    wild = [w[:-1] for w in re.findall(r"`(coper_[a-z0-9_]*\*)", doc) if len(w) > len("coper_*") + 1]
    missing = [s for s in syms if s not in doc and not any(s.startswith(w) for w in wild)]
    assert not missing, missing


def test_every_kernel_waits_for_its_programmatic_predecessor():
    """Programmatic dependent launch (DESIGN 4.6): every kernel of the library is launched through launch_pdl, i.e. it may
    be scheduled before its stream predecessor has finished - so every __global__ function must execute
    griddepcontrol.wait (pdl_enter() first thing, or pdl_trigger() ... pdl_wait() around a prologue that touches no
    global memory) and no launch may bypass launch_pdl."""
    import re
    csrc = os.path.join(ROOT, "coper_b200", "csrc")
    pat = re.compile(r"__global__\s+void\s+(?:__launch_bounds__\([^)]*\)\s*)?(\w+)\s*\(")
    n_kernels = 0
    for f in sorted(os.listdir(csrc)):
        if not f.endswith((".cu", ".cuh")):
            continue
        src = open(os.path.join(csrc, f)).read()
        code = re.sub(r"//[^\n]*", "", src)
        assert "<<<" not in code, "%s launches a kernel without launch_pdl" % f
        for m in pat.finditer(src):
            depth, i = 0, m.end() - 1
            while True:                       # end of the parameter list
                depth += src[i] == "("
                depth -= src[i] == ")"
                if depth == 0:
                    break
                i += 1
            b = src.find("{", i)
            if src[i + 1:b].strip():
                continue                      # a declaration
            depth, j = 0, b
            while True:                       # end of the body
                depth += src[j] == "{"
                depth -= src[j] == "}"
                if depth == 0:
                    break
                j += 1
            body = src[b:j]
            head = body[:200]
            ok = "pdl_enter();" in head or ("pdl_trigger();" in head and "pdl_wait();" in body)
            assert ok, "%s: kernel %s does not wait for its programmatic predecessor" % (f, m.group(1))
            n_kernels += 1
    assert n_kernels >= 60
