// stage_pattern.cuh -- "diagonal pattern" mode: SpGEMM for operands whose entries sit on few
// distinct diagonals (stencil / banded / structured-grid matrices -- all four stock workloads of
// the reference driver, main.cu:30-53, and BASELINE configs 1 and 2).
//
// If every entry of A has its offset (column - row) in a set DA and every entry of B in DB, with
// |DA|, |DB| <= 64, then every entry of C = A*B has its offset in the sumset D = DA + DB.  When
// |D| <= 256 the position of a product inside its (sorted) output row is a table lookup:
//     out = M[ja][jb]      ja = index of A's offset in DA, jb = index of B's offset in DB,
// D sorted ascending, so ascending `out` is ascending column.  No hashing, no probing, no
// insertion, no compaction, no sort -- the work ESC_bitonic_scan / EM_mergepath do in the
// reference (bhsparse_cuda.h:973-1518, 1707-2157) and the hash kernels do here.  The pipeline is
//   k_offset_set     exact set of offsets of a matrix (device hash set; gives up beyond 64)
//   [host]           DA, DB -> D, M, the full-row masks P, a bank-conflict-free layout of the
//                    accumulator (PatternPlan, cached per context)
//   k_pat_codes      one byte per entry: index of its offset (ta, tb); per row of B the bit mask
//                    of the offsets present
//   k_pat_symbolic   mask of the output offsets of every row of C -> nnz(C_i)  (exact)
//   [scan]           row pointers, allocation of C
//   k_pat_numeric    acc[layout[M[ja][jb]]] += a*b per product, emit the row in place, sorted
// Detection is exact (every entry is looked at), nothing is speculated: a matrix that does not
// fit simply takes the general path.
#pragma once
#include "common.cuh"

namespace bhb {

constexpr int PAT_MAX_OFFS = 64;      // distinct diagonals per operand
constexpr int PAT_MAX_OUT = 256;      // distinct diagonals of C (one byte per lookup)
constexpr int PAT_SET_SLOTS = 512;    // device hash set (power of two, >> PAT_MAX_OFFS + threads racing past it)
constexpr int PAT_EMPTY = (int)0x80808080;   // what cudaMemset(0x80) leaves in a slot

struct PatSet {
    int count;
    int overflow;
    int slot[PAT_SET_SLOTS];
};

// Device tables of a plan (one allocation; offsets in bytes from `base`)
struct PatTables {
    const unsigned char *mphys;   // [nDA][nDB]  accumulator position of product (ja, jb)
    const unsigned char *mlog;    // [nDA][nDB]  output index (sorted) of product (ja, jb)
    const unsigned *pfull;        // [nDA][nw]   output mask of a B row holding every offset of DB
    const int *dcol;              // [nD]        offset of output index o
    const unsigned char *pos;     // [nD]        accumulator position of output index o
    const int *offsA;             // [nDA] sorted
    const int *offsB;             // [nDB] sorted
    int nDA, nDB, nD, nw, acc_len;
    unsigned long long fullB;     // mask with nDB bits set
    const unsigned *fullbits;     // one bit per row of B: the row holds every offset of DB (set by the caller; may be null)
};

// launchers (stage_pattern.cu)
cudaError_t launch_offset_set(const LaunchCtx &lc, int rows, const int *rowptr, const int *col, PatSet *set);
// bad: set to 1 if a column is outside [0, ncols) or (rowmask != nullptr) a row is not strictly ascending
// span = largest - smallest offset + 1 (a small span selects the direct-table kernel)
// miss: set to 1 if an entry's offset is not in `offs` (a cached plan no longer describes the matrix)
// fullbits (with rowmask): one bit per row, "holds every offset" (rowmask == full)
// col_range_out: {max column, INT_MAX - min column} of the matrix by atomicMax (zero-initialised by the caller)
// row_range: such a pair in device memory; only rows inside it are coded and checked (nullptr: all rows)
cudaError_t launch_pat_codes(const LaunchCtx &lc, int rows, int ncols, const int *rowptr, const int *col, const int *offs,
                             int noffs, long long span, unsigned char *code, unsigned long long *rowmask, int *bad, int *miss,
                             unsigned long long full, unsigned *fullbits, int *col_range_out, const int *row_range);
cudaError_t launch_pat_symbolic(const LaunchCtx &lc, int m, Csr A, const unsigned char *ta, const unsigned long long *maskB,
                                PatTables t, unsigned *outmask, int *rc, int *prod, Counters *ctr, int k, double avg_row,
                                const unsigned *fullbits);
// dtype BHB200_DTYPE_NONE: the columns of C from the output masks alone (k_pat_emit); A, B, ta, tb are not read
cudaError_t launch_pat_numeric(const LaunchCtx &lc, int dtype, int m, Csr A, Csr B, const unsigned char *ta,
                               const unsigned char *tb, PatTables t, const unsigned *outmask, const int64_t *rowoff,
                               int *colC, void *valC);

}  // namespace bhb
