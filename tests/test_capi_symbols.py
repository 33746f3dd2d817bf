"""CPU-side checks of the drop-in boundary: the library loads and exports every
symbol include/bhsparse_b200.h declares; without a GPU the entry points fail
loudly instead of falling back to a CPU path."""
import ctypes
import os
import re

import pytest

from benchmark_spgemm_using_csr_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "bhsparse_b200.h")).read()
    return sorted(set(re.findall(r"BHB200_API[^;(]*?\b(bhb200_\w+)\s*\(", text)))


def test_header_and_binding_agree():
    assert _declared() == sorted(capi.EXPORTED)


def test_library_exports_every_declared_symbol():
    lib = capi.load(build_if_missing=True)
    for name in _declared():
        assert hasattr(lib, name), f"{name} missing from {capi.LIB_PATH}"
    assert b"sm_100a" in lib.bhb200_version()


def test_stats_struct_matches_header():
    text = open(os.path.join(ROOT, "include", "bhsparse_b200.h")).read()
    body = re.search(r"typedef struct bhb200_stats \{(.*?)\} bhb200_stats;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        for part in decl.split(None, 1)[1].split(","):
            names.append(re.sub(r"\[.*\]", "", part).strip())
    assert names == [f[0] for f in capi.Stats._fields_]


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = capi.load(build_if_missing=True)
    ctx = ctypes.c_void_p(None)
    assert lib.bhb200_create(ctypes.byref(ctx), 0) == capi.ERR_NO_DEVICE
    assert not ctx
    from benchmark_spgemm_using_csr_b200 import generators as gen, spgemm
    A = gen.poisson5pt(4, 4)
    with pytest.raises(capi.BhsparseError):
        spgemm(A, A)


def test_context_without_gpu_raises():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    capi.load(build_if_missing=True)
    with pytest.raises(capi.BhsparseError) as e:
        capi.Context()
    assert e.value.code == capi.ERR_NO_DEVICE


@pytest.mark.parametrize("op", [capi.OP_N, capi.OP_T, capi.OP_C])
def test_op_dims(op):
    """op(X) of a stored rows x cols X is rows x cols for OP_N and cols x rows for OP_T and OP_C."""
    from benchmark_spgemm_using_csr_b200.generators import CSR
    A, B = CSR(3, 5, None, None, None), CSR(7, 11, None, None, None)
    m, k = (3, 5) if op == capi.OP_N else (5, 3)
    assert capi.op_dims(A, B, op, capi.OP_N) == (m, k, 11)
    assert capi.op_dims(A, B, capi.OP_N, op) == (3, 5, 11 if op == capi.OP_N else 7)
    assert capi.op_shape(*capi.op_shape(3, 5, op), op) == (3, 5)


def test_header_is_plain_c_and_links(tmp_path):
    """The boundary is a C ABI: the header must compile as C99 and a C caller must link
    against the shared library (no compute call: there is no GPU here)."""
    import shutil
    import subprocess
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    if not cc:
        pytest.skip("no C compiler")
    capi.load(build_if_missing=True)
    src = tmp_path / "caller.c"
    src.write_text('#include <stdio.h>\n#include "bhsparse_b200.h"\n'
                   'int main(void) {\n'
                   '    bhb200_ctx *ctx = NULL;\n'
                   '    printf("%s\\n", bhb200_version());\n'
                   '    int rc = bhb200_create(&ctx, 0);\n'
                   '    if (rc == BHB200_SUCCESS) bhb200_destroy(ctx);\n'
                   '    return (rc == BHB200_SUCCESS || rc == BHB200_ERR_NO_DEVICE) ? 0 : 1;\n'
                   '}\n')
    exe = tmp_path / "caller"
    libdir = os.path.dirname(capi.LIB_PATH)
    r = subprocess.run([cc, "-std=c99", "-Wall", "-Wextra", "-pedantic", "-Werror", "-I", os.path.join(ROOT, "include"),
                        str(src), "-o", str(exe), "-L", libdir, "-lbhsparse_b200", f"-Wl,-rpath,{libdir}"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0 and "sm_100a" in r.stdout, (r.stdout, r.stderr)
