"""CPU check of the masked product in the C++ forwarder: a caller of include/bhsparse.h that uses
setMask / clearMask compiles warning-free and links against the library (no compute call: no GPU
is needed)."""
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
    /* A = [[1, 2], [0, 3]], M = the upper triangle */
    index_type rowptr[3] = {0, 2, 3}, col[3] = {0, 1, 1};
    value_type val[3] = {1, 2, 3};
    index_type rowptrC[3];
    index_type rowptrM[3] = {0, 1, 2}, colM[2] = {1, 1};
    int rc = bh.initData(2, 2, 2, 3, val, rowptr, col, 3, val, rowptr, col, rowptrC);
    rc |= bh.setMask(2, rowptrM, colM);
    rc |= bh.spgemm();
    rc |= bh.clearMask();
    rc |= bh.spgemm();
    return rc == BHSPARSE_SUCCESS ? 0 : 1;
}
'''


@pytest.mark.parametrize("value", ["double", "float"])
def test_setmask_clearmask_compile(tmp_path, value):
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
    assert "#define BHB200_NUM_MASK_BINS 9" in header
