"""Parity on the GPU with the reference itself (bhSPARSE's own CUDA kernels compiled for sm_100a):
this library's C against the reference's outputs stored in tests/golden/ref_outputs.npz, and
against the CPU oracle, same inputs.

Covers the reference driver's own workloads (-spgemm 0..4: the 4x6 known-answer case and the
four stock Poisson sizes, main.cu:30-53,149-246) and the cases of tests/ref_cases.py that walk
the reference's bins up to the global merge path."""
import pytest

import oracle
import ref_cases
from benchmark_spgemm_using_csr_b200 import spgemm
from conftest import assert_csr_equal

pytestmark = pytest.mark.gpu

RTOL = {"f64": 1e-12, "f32": 1e-5}
CASES = dict(ref_cases.SMALL + ref_cases.LARGE)


@pytest.mark.parametrize("dn", ["f64", "f32"])
@pytest.mark.parametrize("name", list(CASES))
def test_library_equals_reference(golden, name, dn):
    A, B = CASES[name](ref_cases.DTYPES[dn])
    ours = spgemm(A, B)
    ref_cases.check(golden("ref_outputs"), name, dn, *ours, RTOL[dn])
    # the reference and the oracle agree within RTOL (tests/test_oracle_pinned.py), so the library
    # and the oracle agree within twice that
    o = oracle.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val)
    assert_csr_equal(ours, o, exact_values=not name.endswith("_real"), rtol=2 * RTOL[dn],
                     what=f"{name}.{dn}: library vs oracle")
