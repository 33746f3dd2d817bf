"""CPU check of the structure-only interface: a C99 caller of bhsparse_b200.h and a C++ caller of bhsparse.h that
use bhb200_init_data_structure, bhb200_get_C_structure, BHB200_DTYPE_NONE and initDataStructure compile
warning-free and link against the library (the calls return early without a device), and the Python binding
knows the new type."""
import os
import shutil
import subprocess

import pytest

from benchmark_spgemm_using_csr_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

C_CALLER = r'''
#include <stddef.h>
#include "bhsparse_b200.h"

int main(void)
{
    bhb200_ctx *ctx = NULL;
    /* A = [[1, 1, 0], [0, 1, 1]] (2 x 3), pattern only */
    int32_t rowptr[3] = {0, 2, 4}, col[4] = {0, 1, 1, 2};
    int32_t rowptrC[3], colC[16];
    int rc;
    if (bhb200_create(&ctx, 0) != BHB200_SUCCESS) return 0;   /* no device: nothing to run */
    rc = bhb200_init_data_structure(ctx, BHB200_OP_N, BHB200_OP_T, 2, 3, 2, 4, rowptr, col, 4, rowptr, col);   /* A * A^T */
    if (rc == BHB200_SUCCESS) rc = bhb200_spgemm(ctx);
    if (rc == BHB200_SUCCESS) rc = bhb200_get_C_structure(ctx, rowptrC, colC);
    if (rc == BHB200_SUCCESS)   /* device operands without values */
        rc = bhb200_init_data_device(ctx, BHB200_DTYPE_NONE, 0, 0, 0, 0, NULL, rowptr, NULL, 0, NULL, rowptr, NULL);
    bhb200_destroy(ctx);
    return rc == BHB200_SUCCESS ? 0 : 1;
}
'''

CXX_CALLER = r'''
#include "bhsparse.h"

int main()
{
    bool platforms[NUM_PLATFORMS] = {false};
    platforms[BHSPARSE_CUDA] = true;
    bhsparse bh;
    bh.set_verbose(false);
    if (bh.initPlatform(platforms) != BHSPARSE_SUCCESS) return 0;   /* no device: nothing to run */
    index_type rowptr[3] = {0, 2, 4}, col[4] = {0, 1, 1, 2};
    index_type rowptrC[4], colC[16];
    int rc = bh.initDataStructure(2, 3, 2, 4, rowptr, col, 4, rowptr, col, rowptrC, false, true);   /* A * A^T */
    rc |= bh.initDataStructure(3, 2, 3, 4, rowptr, col, 4, rowptr, col, rowptrC, true);            /* A^T * A */
    if (rc == BHSPARSE_SUCCESS) rc = bh.spgemm();
    if (rc == BHSPARSE_SUCCESS) rc = bh.get_C(colC, nullptr);
    return rc == BHSPARSE_SUCCESS ? 0 : 1;
}
'''


def _compile(tmp_path, compiler, std, source, name, extra=()):
    src = tmp_path / name
    src.write_text(source)
    exe = tmp_path / (name.split(".")[0])
    libdir = os.path.dirname(capi.LIB_PATH)
    r = subprocess.run([compiler, f"-std={std}", "-Wall", "-Wextra", "-Werror", *extra, "-I", os.path.join(ROOT, "include"),
                        str(src), "-o", str(exe), "-L", libdir, "-lbhsparse_b200", f"-Wl,-rpath,{libdir}"],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_c99_caller_compiles_and_links(tmp_path):
    cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else shutil.which("gcc")
    if not cc:
        pytest.skip("no C compiler")
    capi.load(build_if_missing=True)
    _compile(tmp_path, cc, "c99", C_CALLER, "caller.c", ["-pedantic"])


@pytest.mark.parametrize("value", ["double", "float"])
def test_cxx_caller_compiles_and_links(tmp_path, value):
    cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else shutil.which("g++")
    if not cxx:
        pytest.skip("no C++ compiler")
    capi.load(build_if_missing=True)
    _compile(tmp_path, cxx, "c++17", CXX_CALLER, "caller.cpp", ["-DBHSPARSE_VALUE_FLOAT"] if value == "float" else [])


def test_dtype_none_in_header_and_binding():
    header = open(os.path.join(ROOT, "include", "bhsparse_b200.h")).read()
    assert "#define BHB200_DTYPE_NONE 2" in header
    assert capi.DTYPE_NONE == 2
    assert "bhb200_init_data_structure" in capi.EXPORTED and "bhb200_get_C_structure" in capi.EXPORTED
