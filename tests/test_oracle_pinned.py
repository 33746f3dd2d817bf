"""The oracle against outputs of THE REFERENCE ITSELF (CPU test, no GPU needed).

tests/golden/ref_outputs.npz was produced on a B200 by oracle/_ref -- the reference's own
kernels and host code (SpGEMM_cuda/bhsparse.h, bhsparse_cuda.h) compiled for sm_100a by
oracle/build_ref.py -- on the inputs of tests/ref_cases.py (tests/golden/make_ref_golden.py is
the generating script).  This pins oracle/spgemm_oracle.c: rowptrC and colC bit-exact, values
bit-exact for the driver's integer-valued inputs, 1e-12 / 1e-5 relative for real-valued ones
(ref_cases.check)."""
import os

import numpy as np
import pytest

import oracle
import ref_cases

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_outputs.npz")
RTOL = {"f64": 1e-12, "f32": 1e-5}


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


def _oracle(A, B):
    return oracle.spgemm(A.rows, A.cols, B.cols, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val)


@pytest.mark.parametrize("dn", ["f64", "f32"])
@pytest.mark.parametrize("name", [n for n, _ in ref_cases.SMALL + ref_cases.LARGE])
def test_oracle_equals_reference_output(gold, name, dn):
    build = dict(ref_cases.SMALL + ref_cases.LARGE)[name]
    A, B = build(ref_cases.DTYPES[dn])
    ref_cases.check(gold, name, dn, *_oracle(A, B), RTOL[dn])


def test_every_case_is_present(gold):
    want = {f"{n}.{d}.nnzC" for n, _ in ref_cases.SMALL + ref_cases.LARGE for d in ("f64", "f32")}
    assert want <= set(gold.files)
