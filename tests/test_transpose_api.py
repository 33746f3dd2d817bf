"""CPU check of the transpose flags of the C++ forwarder: a caller of include/bhsparse.h that uses
both the reference's initData form and the one with transA / transB compiles warning-free and links
against the library (no compute call: no GPU is needed)."""
import os
import shutil
import subprocess

import pytest

from benchmark_spgemm_using_csr_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

CALLER = r'''
#include "bhsparse.h"

int main()
{
    bool platforms[NUM_PLATFORMS] = {false};
    platforms[BHSPARSE_CUDA] = true;
    bhsparse bh;
    bh.set_verbose(false);
    if (bh.initPlatform(platforms) != BHSPARSE_SUCCESS) return 0;   /* no device: nothing to run */
    /* A = [[1, 2, 0], [0, 3, 4]] (2 x 3) */
    index_type rowptr[3] = {0, 2, 4}, col[4] = {0, 1, 1, 2};
    value_type val[4] = {1, 2, 3, 4};
    index_type rowptrC[4];
    int rc = bh.initData(2, 3, 2, 4, val, rowptr, col, 4, val, rowptr, col, rowptrC, false, true);     /* A * A^T */
    rc |= bh.initData(3, 2, 3, 4, val, rowptr, col, 4, val, rowptr, col, rowptrC, true, false);        /* A^T * A */
    rc |= bh.initData(2, 3, 3, 4, val, rowptr, col, 4, val, rowptr, col, rowptrC, false);              /* A * (3 x 3) */
    rc |= bh.initData(2, 3, 3, 4, val, rowptr, col, 4, val, rowptr, col, rowptrC);                     /* reference form */
    return rc == BHSPARSE_SUCCESS ? 0 : 1;
}
'''


@pytest.mark.parametrize("value", ["double", "float"])
def test_initdata_old_and_transposed_forms_compile(tmp_path, value):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if not cxx:
        pytest.skip("no C++ compiler")
    capi.load(build_if_missing=True)
    src = tmp_path / "caller.cpp"
    src.write_text(CALLER)
    exe = tmp_path / "caller"
    libdir = os.path.dirname(capi.LIB_PATH)
    defs = ["-DBHSPARSE_VALUE_FLOAT"] if value == "float" else []
    r = subprocess.run([cxx, "-std=c++17", "-Wall", "-Wextra", "-Werror", *defs, "-I", os.path.join(ROOT, "include"),
                        str(src), "-o", str(exe), "-L", libdir, "-lbhsparse_b200", f"-Wl,-rpath,{libdir}"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    header = open(os.path.join(ROOT, "include", "bhsparse_b200.h")).read()
    assert "#define BHB200_OP_N 0" in header and "#define BHB200_OP_T 1" in header
