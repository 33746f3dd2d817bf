"""Inputs on which the oracle and the library are pinned by outputs OF THE REFERENCE ITSELF
(oracle/_ref run on a B200 by tests/golden/make_ref_golden.py).  One list, used by the generating
script, by the CPU test that checks the oracle against the committed vectors
(tests/test_oracle_pinned.py) and by the GPU test that checks the library against them
(tests/test_reference_gpu.py).

A case is (name, builder) with builder(dtype) -> (A, B) host CSR.  Values are integers 1..9 as
in the reference driver (main.cu:82,93), so every sum is exact in f32 and f64 and the compare is
bit-for-bit, except the cases named *_real (uniform reals: tolerance path, reference summation
order differs from the oracle's, SURVEY.md App. A.4)."""
import numpy as np

from benchmark_spgemm_using_csr_b200 import generators as gen
from benchmark_spgemm_using_csr_b200.generators import CSR


def _identity(n, dt):
    return CSR(n, n, np.arange(n + 1, dtype=np.int32), np.arange(n, dtype=np.int32), gen.int_values(n, 5, dt))


def _kat(dt):
    # test_small_spgemm, main.cu:153-201
    A = CSR(4, 6, np.array([0, 1, 4, 5, 6], np.int32), np.array([0, 1, 2, 3, 3, 1], np.int32),
            np.array([10, 20, 30, 40, 50, 60], dt))
    B = CSR(6, 4, np.array([0, 1, 3, 5, 5, 5, 7], np.int32), np.array([0, 1, 3, 0, 1, 1, 3], np.int32),
            np.array([1, 2, 3, 4, 5, 6, 7], dt))
    return A, B


# the reference's bins (bhsparse.h:377-406): 0..121 one each, 122-128, 129-256, 257-512, >=513 (EM);
# EM capacities 256/512/1024/2048/2304, then the global merge path (SURVEY.md App. A.3)
REF_EDGES = [0, 1, 2, 3, 16, 31, 32, 33, 63, 64, 65, 96, 97, 121, 122, 123, 128, 129, 255, 256, 257, 511, 512, 513,
             1023, 1024, 1025, 2047, 2048, 2049, 2303, 2304, 2305, 4607, 4608, 4609, 6912, 6913, 9300]


def _edges_identity(dt):
    sizes = np.array(REF_EDGES, dtype=np.int64)
    A = gen.random_csr(sizes.size, 20000, sizes, seed=7, dtype=dt)
    return A, _identity(20000, dt)


def _edges_dups(dt):
    k = 3000
    sizes = np.array([0, 1, 2, 5, 6, 7, 12, 13, 19, 20, 25, 26, 38, 39, 51, 52, 77, 102, 103, 150, 205, 300, 461, 600, 900,
                      1500, 2999], dtype=np.int64)
    A = gen.random_csr(sizes.size, k, sizes, seed=11, dtype=dt)
    B = gen.random_csr(k, 2500, 5, seed=12, value_seed=13, dtype=dt)
    return A, B


def _sq(f, *a, **kw):
    def build(dt):
        A = f(*a, dtype=dt, **kw)
        return A, A
    return build


def _rect(dt):
    A = gen.uniform_rect(1500, 1500, per_row=8, seed=1, dtype=dt)
    B = gen.uniform_rect(1500, 1500, per_row=8, seed=2, value_seed=3, dtype=dt)
    return A, B


# small: full outputs are stored
SMALL = [
    ("kat_small", _kat),
    ("poisson5pt_48x48", _sq(gen.poisson5pt, 48, 48)),
    ("poisson9pt_40x40", _sq(gen.poisson9pt, 40, 40)),
    ("poisson7pt_10", _sq(gen.poisson7pt, 10, 10, 10)),
    ("poisson27pt_10", _sq(gen.poisson27pt, 10, 10, 10)),
    ("rmat9_graph500", _sq(gen.rmat, 9, 16, a=0.57, b=0.19, c=0.19, d=0.05)),
    ("rmat10_mild", _sq(gen.rmat, 10, 8)),
    ("rect_1500x1500", _rect),
    ("edges_identity", _edges_identity),
    ("edges_dups", _edges_dups),
    ("poisson27pt_8_real", _sq(gen.poisson27pt, 8, 8, 8, values="real")),
    ("rmat9_real", _sq(gen.rmat, 9, 16, a=0.57, b=0.19, c=0.19, d=0.05, values="real")),
]
# the reference driver's stock workloads (-spgemm 1..4, main.cu:30-53) + mid-size skewed: digests only
LARGE = [
    ("spgemm1_poisson5pt_256", _sq(gen.poisson5pt, 256, 256)),
    ("spgemm2_poisson9pt_256", _sq(gen.poisson9pt, 256, 256)),
    ("spgemm3_poisson7pt_51", _sq(gen.poisson7pt, 51, 51, 51)),
    ("spgemm4_poisson27pt_51", _sq(gen.poisson27pt, 51, 51, 51)),
    ("rmat14_graph500", _sq(gen.rmat, 14, 16, a=0.57, b=0.19, c=0.19, d=0.05)),
    ("rmat16_mild", _sq(gen.rmat, 16, 16)),
]
DTYPES = {"f64": np.float64, "f32": np.float32}


def digest(a: np.ndarray) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


SAMPLE = 4096          # stored values per real-valued case: their full arrays would not fit the golden file


def row_sums(rp, val) -> np.ndarray:
    rows = np.repeat(np.arange(rp.size - 1), np.diff(np.asarray(rp, dtype=np.int64)))
    return np.bincount(rows, weights=val.astype(np.float64), minlength=rp.size - 1)


def record(name: str, rp, col, val) -> dict:
    """What tests/golden/ref_outputs.npz keeps of the reference's C = (rp, col, val) for one case, keyed
    without the "<name>.<dtype>." prefix: nnzC and the SHA-256 digests of rowptrC (int32), colC and
    valC; for the *_real cases, whose values are compared within a tolerance, also the per-row sums of
    valC and valC at a fixed seeded sample of positions."""
    rec = {"nnzC": np.int64(rp[-1]), "digest": np.array([digest(np.asarray(rp, np.int32)), digest(col), digest(val)])}
    if name.endswith("_real"):
        idx = np.random.default_rng(0).choice(val.size, min(SAMPLE, val.size), replace=False)
        idx = np.sort(idx).astype(np.int32)
        rec.update(sample_idx=idx, sample_val=val[idx], row_sum=row_sums(rp, val))
    return rec


def check(gold, name: str, dn: str, rp, col, val, rtol: float) -> None:
    """Asserts that C = (rp, col, val) is the reference's output stored in `gold` for case `name` in
    dtype `dn`: rowptrC and colC bit-exact; valC bit-exact, or for the *_real cases within rtol
    relative at the sampled positions and in every row sum."""
    key = f"{name}.{dn}"
    assert int(gold[key + ".nnzC"]) == int(rp[-1]), f"{key}: nnzC differs"
    d = gold[key + ".digest"]
    assert d[0] == digest(np.asarray(rp, np.int32)), f"{key}: rowptrC differs"
    assert d[1] == digest(col), f"{key}: colC differs"
    if not name.endswith("_real"):
        assert d[2] == digest(val), f"{key}: valC differs (exact compare)"
        return
    idx, want = gold[key + ".sample_idx"], gold[key + ".sample_val"]
    assert want.dtype == val.dtype
    err = np.abs(val[idx].astype(np.float64) - want.astype(np.float64)) / np.abs(want.astype(np.float64))
    assert err.max() <= rtol, f"{key}: max rel err {err.max()} > {rtol}"
    # every value within rtol of the reference's keeps each row sum within rtol of the row's sum of
    # magnitudes; the factor 2 covers the rounding of the sums themselves
    sum_err = np.abs(row_sums(rp, val) - gold[key + ".row_sum"])
    assert (sum_err <= 2 * rtol * row_sums(rp, np.abs(val))).all(), f"{key}: a row sum differs beyond {rtol}"
