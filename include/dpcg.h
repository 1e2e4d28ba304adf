/*
 * dpcg.h — C ABI of libdpcg.so: the B200-native PCG hot path of DeepPreconditioning.
 *
 * The reference (jsappl/DeepPreconditioning) has no FFI: its boundary is a set of duck-typed Python call
 * signatures (SURVEY §8b). Each entry point below names the reference code it replaces (file:line relative
 * to the reference root). The Python shim in deeppreconditioning_b200/ keeps the reference signatures and
 * calls these through ctypes; INTEGRATION.md shows the binding a maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; every pointer is a DEVICE pointer unless named *_host.
 *   - values fp64, indices int32, 16-byte aligned arrays (checked: DP_ERR_ALIGNMENT).
 *   - returns int status, 0 = DP_OK; never throws; no hidden allocation: scratch comes from the caller,
 *     sized by the matching *_workspace_bytes() query; work is enqueued on `stream` (a cudaStream_t passed as
 *     void*) and is asynchronous unless stated.
 *   - one host thread per GPU; re-entrant per stream as long as workspaces are distinct.
 */
#ifndef DPCG_H
#define DPCG_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DP_VERSION 100

enum dp_status {
    DP_OK = 0,
    DP_ERR_INVALID = 1,    /* bad argument (null pointer, negative size, unknown mode) */
    DP_ERR_ALIGNMENT = 2,  /* an array is not 16-byte aligned */
    DP_ERR_WORKSPACE = 3,  /* workspace too small */
    DP_ERR_CUDA = 4,       /* a CUDA runtime call failed; see dp_last_cuda_error() */
    DP_ERR_STRUCTURE = 5,  /* matrix structure violates the contract (reported through a device flag, see below) */
    DP_ERR_TIMEOUT = 6     /* a dependency spin exceeded its budget (device flag) */
};

/* Preconditioner application z = M r inside the loop (reference: `zk = M @ rk`, cg.py:61,81). */
enum dp_precond {
    DP_PRECOND_IDENTITY = 0, /* _construct_vanilla, test.py:70-72 */
    DP_PRECOND_JACOBI = 1,   /* _construct_jacobi, test.py:74-79: z = dinv .* r */
    DP_PRECOND_MULTIPLY = 2, /* _construct_learned, test.py:100-105 in factored form: z = L (L^T r) */
    DP_PRECOND_SOLVE = 3,    /* north_star apply mode for IC(0): z = L^-T (L^-1 r) */
    DP_PRECOND_CSR = 4       /* any explicit CSR M (what test.py:88,105 hand to cg.py): z = M r */
};

enum dp_engine {
    DP_ENGINE_FUSED = 0,   /* one persistent cooperative kernel for the whole solve (device-side loop control) */
    DP_ENGINE_STEPPED = 1  /* one launch per phase; host polls the done counter every `check_every` iterations */
};

enum dp_assemble_mode {
    DP_ASSEMBLE_TRIL = 0,       /* keep row >= col && value != 0  -> L        (test.py:103-105 minus the product) */
    DP_ASSEMBLE_TRIL_T = 1,     /* same entries, transposed          -> L^T as CSR                                  */
    DP_ASSEMBLE_SYMMETRISE = 2  /* T + tril(T,-1)^T                  -> A        (test.py:65-68)                    */
};

int dp_version(void);
const char* dp_status_string(int status);
const char* dp_last_cuda_error(void);
/* sm_count, resident CTAs the fused PCG kernel gets per SM, bytes of L2. Synchronous. */
int dp_device_info(int* sm_count_host, int* pcg_ctas_per_sm_host, int* l2_bytes_host);

/* ---- K1: CSR assembly (bit-exact integer/value output) ------------------------------------------------
 * Replaces the dense round trip of BenchmarkSuite._construct_learned (test.py:100-105) and
 * _reconstruct_system (test.py:61-68). Input is the spconv COO layout of data_set.py:121-125:
 * indices int32[nnz_in,3] = (batch,row,col), unordered; features fp32[nnz_in] (channel 0).
 * Only entries of `batch` with row < n && col < n take part (the `[0, 0, :n, :n]` slice).
 * Output rows sorted by column, values widened fp32 -> fp64 exactly. col/val need capacity for
 * nnz_in entries (2*nnz_in for SYMMETRISE); the stored count is rowptr[n], also written to *nnz_out.
 * *flag_out (device int32) is set to DP_ERR_STRUCTURE when a (row,col) pair occurs twice. */
size_t dp_csr_from_coo_workspace_bytes(int32_t n, int64_t nnz_in);
int dp_csr_from_coo(const int32_t* indices, const float* features, int64_t nnz_in, int32_t batch, int32_t n,
                    int32_t mode, int32_t* rowptr, int32_t* col, double* val, int32_t* nnz_out, int32_t* flag_out,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Explicit transpose CSR -> CSR (the north_star stores L^T explicitly). Same sorting contract. */
size_t dp_csr_transpose_workspace_bytes(int32_t n, int32_t nnz);
int dp_csr_transpose(int32_t n, int32_t nnz, const int32_t* rowptr, const int32_t* col, const double* val,
                     int32_t* rowptr_t, int32_t* col_t, double* val_t, void* workspace, size_t workspace_bytes,
                     void* stream);

/* dinv[i] = 1 / A_ii (test.py:76); rows without a stored diagonal get 0 and raise *flag_out. */
int dp_csr_inv_diagonal(int32_t n, const int32_t* rowptr, const int32_t* col, const double* val, double* dinv,
                        int32_t* flag_out, void* stream);

/* Structural nnz of M = L L^T without forming it: the count behind BenchmarkSuite._compute_sparsity (test.py:107-109:
 * `100 * len(matrix.values()) / n^2` of the explicit product test.py:104-105 stores). rowptr/col = L, rowptr_t/col_t =
 * L^T (dp_csr_transpose / TRIL_T), both with sorted rows. *nnz_out is a DEVICE int64. Exact integer work. */
int dp_csr_aat_nnz(int32_t n, const int32_t* rowptr, const int32_t* col, const int32_t* rowptr_t, const int32_t* col_t,
                   int64_t* nnz_out, void* stream);

/* ---- packed stream copy of a CSR matrix (lossless) -----------------------------------------------------------
 * The operands of this path are fp32 data widened to fp64 (the CNN output and the data set's matrices are fp32,
 * test.py:100-105, data_set.py:121-125) on banded patterns, so the 12 bytes per stored entry of the fp64/int32 CSR
 * are mostly zeros. dp_csr_pack writes the same matrix as 6 bytes per entry: val32[q] = (float)val[q] and
 * col16[q] = col[q] - tile_base[2t], t = the 512-row tile (dp_csr_pack_tile_rows()) that holds entry q; tile_base holds
 * one pair per tile: {smallest column of the tile, number of columns it spans (largest - smallest + 1; 0: empty tile)}. The copy exists only if it is EXACT: *status_out (device int32, OR-ed bits) is 0
 * when every value survives the fp32 round trip bit for bit and every tile spans fewer than 65536 columns; otherwise
 * bit 0 (a value is not an fp32 number) and / or bit 1 (a tile is too wide) is set and the copy must not be used.
 * The kernels that accept a packed copy (dp_spmv_csr_packed_f64, dp_pcg_solve_f64) widen on load and do the same fp64
 * arithmetic in the same order: results are bit-identical to the unpacked path, HBM traffic per entry is halved.
 * col16 / val32 need room for nnz entries rounded up to a multiple of 16 bytes, 16-byte aligned;
 * tile_base int32[2 * ceil(n / 512)], 8-byte aligned. Tiles that span few columns (banded matrices: 2-D stencil factors)
 * let dp_pcg_solve_f64 serve a phase's gathers from a shared-memory window of the vectors instead of L2. */
int32_t dp_csr_pack_tile_rows(void);
int dp_csr_pack(int32_t n, int32_t nnz, const int32_t* rowptr, const int32_t* col, const double* val, uint16_t* col16,
                float* val32, int32_t* tile_base, int32_t* status_out, void* stream);
/* y = A x from the packed copy; same bits as dp_spmv_csr_f64. */
int dp_spmv_csr_packed_f64(int32_t n, int32_t nnz, const int32_t* rowptr, const uint16_t* col16, const float* val32,
                           const int32_t* tile_base, const double* x, double* y, void* stream);

/* ---- K2: CSR SpMV fp64 ---------------------------------------------------------------------------------
 * y = A x. Replaces `A @ p` / `M @ r` (cg.py:60,61,75,81). Row sums are sequential in column order with
 * separately rounded products and sums, i.e. bit-identical to scipy's csr_matvec. */
int dp_spmv_csr_f64(int32_t n, int32_t nnz, const int32_t* rowptr, const int32_t* col, const double* val,
                    const double* x, double* y, void* stream);

/* Batched COO SpMV of utils.py:15-43 (sparse_matvec_mul), fp32: out[b,row] += feat * vec[b,col]
 * (row/col swapped when transpose != 0). out is [nbatch, n] and is zeroed first. */
int dp_coo_spmv_batch_f32(const int32_t* indices, const float* features, int64_t nnz, int32_t nbatch, int32_t n,
                          const float* vec, int32_t transpose, float* out, void* stream);

/* ---- K3: level analysis of a triangular CSR pattern (bit-exact integer output) ---------------------------
 * lower (upper == 0): level[i] = 1 + max(level[j] : j < i stored in row i), 0 if none; the diagonal must be
 * the LAST entry of each row. upper: j > i, diagonal FIRST (L^T as produced by dp_csr_transpose).
 * Outputs: level int32[n]; perm int32[n] = rows stably sorted by level; level_ptr int32[n+1] (first
 * *nlevels_out+1 entries valid); *nlevels_out, *flag_out device int32. No reference counterpart (SURVEY D1). */
size_t dp_sptrsv_analyse_workspace_bytes(int32_t n);
int dp_sptrsv_analyse(int32_t n, const int32_t* rowptr, const int32_t* col, int32_t upper, int32_t* level,
                      int32_t* perm, int32_t* level_ptr, int32_t* nlevels_out, int32_t* flag_out, void* workspace,
                      size_t workspace_bytes, void* stream);

/* Execution plan derived from (perm, level_ptr): rows of a level padded to whole warps (-1 = idle lane).
 * nchunks = sum over levels of ceil(size/32) <= n/32 + nlevels; plan needs 32*nchunks int32.
 * The caller reads level_ptr[0..nlevels] back once per matrix (HOST copy), sizes the plan with
 * dp_sptrsv_plan_chunks, and uploads chunk_ptr[l] = sum_{l'<l} ceil(size(l')/32) (nlevels+1 int32, DEVICE). */
int64_t dp_sptrsv_plan_chunks(int32_t nlevels, const int32_t* level_ptr_host);
/* The same sizes without a host round trip of level_ptr: chunk_ptr (DEVICE int32[n+1], exclusive prefix of the levels'
 * chunk counts, entries past nlevels repeat the total) and summary_out (DEVICE int32[3]) = {nlevels, nchunks, chunks of
 * the widest level}: the caller reads 12 bytes back once per matrix to size the plan. nlevels: the device word written
 * by dp_sptrsv_analyse. */
size_t dp_sptrsv_plan_sizes_workspace_bytes(int32_t n);
int dp_sptrsv_plan_sizes(int32_t n, const int32_t* nlevels, const int32_t* level_ptr, int32_t* chunk_ptr,
                         int32_t* summary_out, void* workspace, size_t workspace_bytes, void* stream);
int dp_sptrsv_plan_build(int32_t n, int32_t nlevels, const int32_t* perm, const int32_t* level_ptr,
                         const int32_t* chunk_ptr, int32_t* plan, int64_t nchunks, void* stream);

/* Level-ordered copy of a triangular factor, the input of the level-stream solve (below): row r of the copy is row
 * perm[r] of T, column indices are renumbered to positions in that order, entries keep T's order inside a row (sums
 * stay bit-identical), the diagonal entry (last of a lower row, first of an upper one) holds 1 / T_ii;
 * level_sorted[r] = level[perm[r]]. rowptr_p int32[n+1], col_p/val_p as large as col/val.
 * stats_out (device int32[3]): most entries in any 512 consecutive rows of the copy, most entries in a row, largest
 * distance in positions between a row and a dependency. The level-stream solve accepts the copy when each is within
 * the matching limit of dp_sptrsv_ls_limits() and no level has more rows than its fourth limit (the caller knows the
 * level sizes from level_ptr). */
size_t dp_sptrsv_permute_workspace_bytes(int32_t n);
int dp_sptrsv_permute(int32_t n, int32_t upper, const int32_t* rowptr, const int32_t* col, const double* val, const int32_t* perm,
                      const int32_t* level, int32_t* rowptr_p, int32_t* col_p, double* val_p, int32_t* level_sorted,
                      int32_t* stats_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- K4: sparse triangular solves ------------------------------------------------------------------------
 * lower: L y = b;  upper: U z = b with U = L^T in CSR. x_i = (b_i - sum_j T_ij x_j) * (1 / T_ii), the sum
 * sequential in column order: bit-identical to plain forward/backward substitution (oracle/kernels.c).
 * Sync-free: one cooperative launch, dependencies resolved by spinning on the solution vector itself.
 * *flag_out receives DP_ERR_TIMEOUT if a dependency never arrives (malformed plan). */
size_t dp_sptrsv_workspace_bytes(void);
int dp_sptrsv_solve_f64(int32_t n, const int32_t* rowptr, const int32_t* col, const double* val, int32_t upper,
                        const int32_t* plan, int64_t nchunks, int32_t max_level_chunks, const double* b, double* x,
                        int32_t* flag_out, void* workspace, size_t workspace_bytes, void* stream);

/* Batch of independent triangular solves in ONE launch (BenchmarkSuite.run's data-parallel axis, test.py:121): the
 * resident warps are dealt to the systems, so the solves advance side by side and the batch's HBM stream hides each
 * system's level-by-level critical path. Same arithmetic (bit-identical) as dp_sptrsv_solve_f64 per system. */
typedef struct dp_trsv_system {
    int32_t n;
    int32_t upper;            /* 0: lower (diagonal last in each row), 1: upper (diagonal first) */
    int32_t max_level_chunks; /* chunks of the widest level (from the analysis) */
    int32_t reserved;
    int64_t nchunks;
    const int32_t* rowptr; const int32_t* col; const double* val;
    const int32_t* plan;
    const double* b;
    double* x;
} dp_trsv_system_t;
size_t dp_sptrsv_batch_workspace_bytes(int32_t nsys);
int dp_sptrsv_solve_batch_f64(const dp_trsv_system_t* systems_host, int32_t nsys, int32_t* flag_out, void* workspace,
                              size_t workspace_bytes, void* stream);

/* Level-stream solve: ONE CTA per system walks the level-ordered copy through the TMA tile pipeline; a row's
 * dependencies are awaited on a shared-memory window of the solution (the pending-NaN protocol of the sync-free solve
 * with a shared-memory round trip in place of the L2 hop), there is no barrier per level. For factors with narrow levels
 * (2-D stencils: 2n-1 levels of <= n rows); a batch keeps one SM busy per system. Bit-identical to dp_sptrsv_solve_f64.
 * perm != NULL: b and x are in the ORIGINAL numbering (gathered / scattered through perm). perm == NULL: the matrix is
 * in this solve's level order already (row r of the copy is row r of T) and b / x are indexed by position: b must be
 * 16-byte aligned and must not alias x. level_sorted is not read. rowptr_p, col_p, val_p must be 16-byte aligned.
 * No cooperative launch, no device flag: the only spins are on shared memory and bounded. */
typedef struct dp_trsv_ls_system {
    int32_t n;
    int32_t nnz;
    int32_t upper;   /* 0: lower (diagonal last in each row), 1: upper (diagonal first) */
    int32_t flags;   /* tile-stream solve only: DP_TRSV_REVERSED */
    const int32_t* rowptr_p; const int32_t* col_p; const double* val_p; /* dp_sptrsv_permute outputs */
    const int32_t* perm;
    const int32_t* level_sorted;
    const double* b;
    double* x;
} dp_trsv_ls_system_t;
void dp_sptrsv_ls_limits(int32_t* limits_host /* [4]: tile entries, row entries, dependency distance, rows per level */);
size_t dp_sptrsv_ls_workspace_bytes(int32_t nsys);
int dp_sptrsv_ls_solve_batch_f64(const dp_trsv_ls_system_t* systems_host, int32_t nsys, void* workspace,
                                 size_t workspace_bytes, void* stream);
/* The same in two steps, for solves that are repeated with the same factors and vector buffers (new right-hand sides
 * are written into the same b): dp_sptrsv_ls_prepare uploads the descriptors once (synchronises the stream),
 * dp_sptrsv_ls_launch only enqueues the kernel (asynchronous, no host work). */
int dp_sptrsv_ls_prepare(const dp_trsv_ls_system_t* systems_host, int32_t nsys, void* workspace, size_t workspace_bytes,
                         void* stream);
int dp_sptrsv_ls_launch(int32_t nsys, void* workspace, size_t workspace_bytes, void* stream);

/* Tile-stream solve: the batch form for factors with WIDE levels (3-D stencils: levels of 10^4..10^5 rows). The
 * 512-row tiles of the level-ordered copies of ALL systems form one sequence that persistent CTAs take round robin;
 * the matrix stream goes through the TMA tile pipeline like an SpMV's, dependencies are awaited on the solution
 * vector in position space. Takes the same descriptors as the level-stream solve (level_sorted may be NULL) and any
 * level-ordered copy (no dp_sptrsv_ls_limits restriction). Bit-identical to dp_sptrsv_solve_f64.
 * perm == NULL: b and x are indexed by POSITION (the caller keeps its vectors in level order, x_pos[r] = x[perm[r]]).
 * perm != NULL: b and x are in the original numbering; the call brackets the solve with a gather and a scatter pass
 * through position-space copies in the workspace (40 B per row of extra traffic). b and x must not alias.
 * flags & DP_TRSV_REVERSED (perm == NULL only): position r is row n-1-r of b and x - the backward solve of a system
 * kept in the level order of its forward solve (the copy is dp_sptrsv_permute of L^T with perm[r] = n-1-r).
 * rowptr_p and b (or perm) must be 16-byte aligned like col_p / val_p: their spans travel by bulk copy too.
 * Cooperative launch; *flag_out receives DP_ERR_TIMEOUT if a dependency never arrives. */
#define DP_TRSV_REVERSED 1
/* flags & DP_TRSV_SHORT_ROWS: no row of the copy has more entries than dp_sptrsv_ts_limits()[1] (5-/7-point stencil
 * factors; stats_out[1] of dp_sptrsv_permute). When every system of the batch says so the solve runs a leaner kernel
 * that finishes rows from registers after handing its pipeline stage back; a violated promise raises DP_ERR_STRUCTURE. */
#define DP_TRSV_SHORT_ROWS 2
void dp_sptrsv_ts_limits(int32_t* limits_host /* [2]: entries per pipeline item, row entries of the register path */);
size_t dp_sptrsv_ts_workspace_bytes(const dp_trsv_ls_system_t* systems_host, int32_t nsys);
int dp_sptrsv_ts_solve_batch_f64(const dp_trsv_ls_system_t* systems_host, int32_t nsys, int32_t* flag_out, void* workspace,
                                 size_t workspace_bytes, void* stream);
/* Two-step form (see dp_sptrsv_ls_prepare): the descriptors are uploaded once; dp_sptrsv_ts_launch enqueues the arming
 * pass, the solve (and the gather / scatter passes of systems in the original numbering) without host work. Its integer
 * arguments describe the prepared batch: most tiles of any system, largest n, 1 if every system carries
 * DP_TRSV_SHORT_ROWS, number of systems with perm != NULL. */
int dp_sptrsv_ts_prepare(const dp_trsv_ls_system_t* systems_host, int32_t nsys, void* workspace, size_t workspace_bytes,
                         void* stream);
int dp_sptrsv_ts_launch(int32_t nsys, int32_t max_tiles, int32_t nmax, int32_t short_rows, int32_t nperm, int32_t* flag_out,
                        void* workspace, void* stream);

/* ---- IC(0) on the pattern of tril(A) (stands in for ilupp.ichol0, test.py:84) -------------------------------
 * Level-scheduled, sync-free numeric factorisation; uses the lower plan of the same pattern.
 * *flag_out: DP_ERR_STRUCTURE on a non-positive pivot. */
int dp_ic0_f64(int32_t n, const int32_t* rowptr, const int32_t* col, const double* a_val, double* l_val,
               const int32_t* plan, int64_t nchunks, int32_t max_level_chunks, int32_t* flag_out, void* workspace,
               size_t workspace_bytes, void* stream);

/* Threshold incomplete Cholesky ICT(p, tau) on the HOST (every pointer is a host pointer): the reference's default
 * comparator `ilupp.icholt(A, add_fill_in=1, threshold=0.1)` (test.py:81-86) is a sequential C++ CPU routine, and so is
 * this stand-in (ilupp is not in the image: values "parity unpinned", scheme and dropping rules in csrc/icholt.cu).
 * Input: CSR of tril(A), rows sorted, diagonal last. Output: CSR of L in the same form; col_out/val_out have `capacity`
 * entries (nnz + n * fill_in is always enough), *nnz_out_host receives the stored count.
 * DP_ERR_STRUCTURE: missing diagonal / entry above the diagonal / non-positive pivot; DP_ERR_WORKSPACE: capacity. */
int dp_icholt_host(int32_t n, const int32_t* rowptr_host, const int32_t* col_host, const double* val_host, int32_t fill_in,
                   double threshold, int32_t* rowptr_out_host, int32_t* col_out_host, double* val_out_host,
                   int64_t capacity, int64_t* nnz_out_host);

/* ---- K5: the whole PCG loop ----------------------------------------------------------------------------------
 * Replaces preconditioned_conjugate_gradient (cg.py:50-90) with its exact semantics: iteration-0 check on
 * <z0,z0>/<b,b> (cg.py:66), later checks on <r,r>/<b,b> < rtol (cg.py:15-17,71,86), at most max_iter bodies,
 * iterations = number of loop bodies executed (cg.py:90). One descriptor per independent system (the
 * data-parallel axis of BenchmarkSuite.run, test.py:121); all systems of a call advance in lock step inside one
 * launch and drop out individually when converged. */
typedef struct dp_pcg_system {
    int32_t n;
    int32_t precond; /* enum dp_precond */
    int32_t a_nnz, m_nnz, mt_nnz;
    int32_t fwd_nchunks, bwd_nchunks;       /* SOLVE: plan sizes */
    int32_t fwd_max_level_chunks, bwd_max_level_chunks;
    int32_t solve_algorithm; /* SOLVE: 0 = level-stream where the copies below are given, else sync-free;
                              * DP_SOLVE_TILE_STREAM (| DP_SOLVE_SHORT_ROWS) = the tile-stream batch solve (see below) */
    const int32_t* a_rowptr; const int32_t* a_col; const double* a_val;     /* A (full symmetric CSR) */
    const int32_t* m_rowptr; const int32_t* m_col; const double* m_val;     /* L (MULTIPLY/SOLVE) or M (CSR) */
    const int32_t* mt_rowptr; const int32_t* mt_col; const double* mt_val;  /* L^T (MULTIPLY/SOLVE) */
    const double* dinv;                                                     /* JACOBI */
    const int32_t* fwd_plan; const int32_t* bwd_plan;                       /* SOLVE */
    /* SOLVE, optional: level-ordered copies of L and L^T (dp_sptrsv_permute). When rowptr / col / val of a direction are
     * set that solve runs as a level-stream solve (one CTA per system) instead of the sync-free one; perm == NULL there
     * says the system is already in that solve's level order (vectors taken by position). */
    const int32_t* fwd_ls_rowptr; const int32_t* fwd_ls_col; const double* fwd_ls_val;
    const int32_t* fwd_ls_perm; const int32_t* fwd_ls_level;
    const int32_t* bwd_ls_rowptr; const int32_t* bwd_ls_col; const double* bwd_ls_val;
    const int32_t* bwd_ls_perm; const int32_t* bwd_ls_level;
    /* solve_algorithm == DP_SOLVE_TILE_STREAM (STEPPED engine, every SOLVE system of the batch): the system is kept in
     * the level order of its forward solve (levels ascend along the rows). fwd_ls_{rowptr,col,val} = dp_sptrsv_permute
     * of L with the identity order, bwd_ls_{rowptr,col,val} = dp_sptrsv_permute of L^T with perm[r] = n-1-r
     * (DP_TRSV_REVERSED); the perm / level pointers are ignored. Both solves of an iteration then run as tile-stream
     * batch solves over all systems, directly on the iteration's vectors. */
    const double* b;   /* right-hand side, n */
    double* x;         /* in: x0, out: x_hat, n */
    double* work;      /* dp_pcg_work_doubles(n) doubles of scratch, contents ignored on entry */
    int32_t* iters_out;   /* 1 */
    double* res_out;      /* 1: last value of the stopping criterion (squared relative residual) */
    double* history;      /* optional, max_iter+1 doubles: criterion before every body (cg.py:67,87) */
    double* coef;         /* optional, 2*(max_iter+1) doubles: coef[2k] = a of body k (cg.py:78), coef[2k+1] = beta that
                           * built p for body k (cg.py:82 of body k-1; 0 for k = 0). The CG coefficients are the Lanczos
                           * tridiagonal of M*A: the host turns them into the condition-number estimate that replaces
                           * the dense torch.linalg.cond of test.py:111-113. */
    /* Optional packed stream copies (dp_csr_pack, status 0) of A, of L / M and of L^T. When EVERY system of a batch
     * without SOLVE-mode systems brings the copies of all the matrices its phases stream, the FUSED engine streams
     * those (6 instead of 12 bytes per entry, same bits); otherwise they are ignored. The unpacked arrays above stay
     * mandatory. */
    const uint16_t* a_col16; const float* a_val32; const int32_t* a_tile_base;
    const uint16_t* m_col16; const float* m_val32; const int32_t* m_tile_base;
    const uint16_t* mt_col16; const float* mt_val32; const int32_t* mt_tile_base;
} dp_pcg_system_t;

#define DP_SOLVE_TILE_STREAM 1
#define DP_SOLVE_SHORT_ROWS 2 /* with DP_SOLVE_TILE_STREAM: L and L^T keep the DP_TRSV_SHORT_ROWS promise */

typedef struct dp_pcg_params {
    double rtol;          /* cg.py:51 default 1e-8, compared with the SQUARED relative residual */
    int32_t max_iter;     /* cg.py:51 default 1024 */
    int32_t engine;       /* enum dp_engine */
    int32_t check_every;  /* STEPPED: iterations between host polls of the done counter (>= 1) */
    int32_t reserved;
} dp_pcg_params_t;

int64_t dp_pcg_work_doubles(int32_t n);
size_t dp_pcg_workspace_bytes(int32_t nsys);
/* systems_host: HOST array of nsys descriptors (device pointers inside). Enqueues the solve on `stream`;
 * FUSED is fully asynchronous, STEPPED synchronises the stream every check_every iterations.
 * *flag_out (device int32): DP_ERR_TIMEOUT / DP_ERR_STRUCTURE raised on the device. */
int dp_pcg_solve_f64(const dp_pcg_system_t* systems_host, int32_t nsys, const dp_pcg_params_t* params_host,
                     int32_t* flag_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- K6: sparse-convolution inference of the factor network (model.PreconditionerNet / PreconditionerTrilNet) --------
 * Replaces the generic PyTorch forward of model.SparseConv2d (key sets, torch.unique, one GEMM and one index_add_ per
 * tap) for inference: stride 1, k = 1 or k = 2 with padding (1,0) / (0,1), at most 64 channels, scalar activations.
 *
 * Site sort: indices int32[nnz,3] = (batch,row,col) of an H x W image, unordered. rowptr int32[batch_size*h + 1] is the
 * "site CSR" over the (batch,row) pairs, col int32[nnz] the columns sorted in each row, perm int32[nnz] the input
 * position of each sorted site. Every site counts, zero-valued ones included. *flag_out (device int32) receives
 * DP_ERR_STRUCTURE for a repeated site or one outside [0,batch_size) x [0,h) x [0,w) (such sites are left out). */
size_t dp_spconv_sort_workspace_bytes(int32_t batch_size, int32_t h);
int dp_spconv_sort_sites(const int32_t* indices, int64_t nnz, int32_t batch_size, int32_t h, int32_t w, int32_t* rowptr,
                         int32_t* col, int32_t* perm, int32_t* flag_out, void* workspace, size_t workspace_bytes,
                         void* stream);
/* Rules of a 2x2 layer with padding (ph,pw) in {(1,0),(0,1)} on a sorted site CSR of an h x w image: output image
 * ho = h + 2ph - 1 by wo = w + 2pw - 1; output site (y,x) is active iff an input site (y + ky - ph, x + kx - pw) is.
 * Two steps, because the caller sizes the outputs: _count writes rowptr_out int32[batch_size*ho + 1] (the total at
 * rowptr_out[batch_size*ho]); _fill writes col_out int32[nout] (sorted per row), rules int32[nout,4] (16-byte aligned):
 * rules[s,2ky+kx] = the input site of tap (ky,kx), -1 where inactive, numbered as the sorted sites, or through perm
 * (perm != NULL) in the numbering of the sorted sites' source. indices_out (optional) int32[nout,3] = (batch,row,col),
 * the order torch.unique gives model.SparseConv2d. */
size_t dp_spconv_rules_workspace_bytes(int32_t batch_size, int32_t h, int32_t ph);
int dp_spconv_rules_count(const int32_t* rowptr_in, const int32_t* col_in, int32_t batch_size, int32_t h, int32_t w,
                          int32_t ph, int32_t pw, int32_t* rowptr_out, void* workspace, size_t workspace_bytes,
                          void* stream);
int dp_spconv_rules_fill(const int32_t* rowptr_in, const int32_t* col_in, const int32_t* perm, int32_t batch_size,
                         int32_t h, int32_t w, int32_t ph, int32_t pw, const int32_t* rowptr_out, int32_t* col_out,
                         int32_t* rules, int32_t* indices_out, void* stream);
/* One layer, fp32 on CUDA cores: out[s,co] = act(((0 + p_0) + p_1 ...) + bias[co]) with p_t = sum over ci ascending of
 * weight[co,t,ci] * in[src[s,t],ci] (one fma chain per tap, inactive taps skipped), act(v) = v > 0 ? v : slope * v.
 * The order is fixed per output value: results do not depend on the batch or the launch geometry.
 * head_weight != NULL: the final 1x1 layer (cout -> 1) follows in the epilogue, y = sum_co head_weight[co] * out[s,co]
 * (+ head_bias), and out is [nout,1]. indices != NULL: the output tail of the factor network on that one channel (the
 * layer's own when cout == 1 without a head): sites with row < col are multiplied by 0, diagonal sites get softplus
 * (threshold 20, log1p(exp(y))). All pointers are device pointers; weights are read at every call. */
typedef struct dp_spconv_layer {
    int64_t nout;              /* output sites */
    int32_t ntaps;             /* 1 (k = 1) or 4 (k = 2, taps in (ky,kx) order) */
    int32_t cin, cout;         /* 1..64 */
    int32_t reserved;
    const int32_t* src;        /* [nout, ntaps] input site per tap (-1: inactive); NULL: site s reads row s (ntaps 1) */
    const float* in;           /* [*, cin] */
    const float* weight;       /* [cout, ntaps, cin]: spconv's [out, k, k, in] */
    const float* bias;         /* [cout] or NULL */
    const float* slope;        /* device scalar (PReLU weight, LeakyReLU slope) or NULL: no activation */
    const float* head_weight;  /* [cout] or NULL */
    const float* head_bias;    /* [1] or NULL */
    const int32_t* indices;    /* [nout,3] (batch,row,col) of the output sites for the tail, or NULL */
    float* out;                /* [nout, cout], [nout, 1] with a head */
} dp_spconv_layer_t;
int dp_spconv_layer_f32(const dp_spconv_layer_t* layer_host, void* stream);

/* Diagnostics: with DPCG_TRACE=1 in the environment the fused engine records (label, clock64) pairs of CTA 0 into the
 * workspace; this copies up to `capacity` pairs to out_host[2*capacity] (label = 8*phase + point). Synchronous. */
int dp_debug_pcg_trace(const void* workspace, int32_t nsys, int64_t* out_host, int32_t capacity);
/* Tuning builds only (-DDPCG_PIPE_TRACE; DP_ERR_INVALID otherwise): per-tile timeline of two warps of CTA 0 through the tile
 * pipeline of the last launch, out_host[2 * capacity] words of (label << 48 | globaltimer ns). Synchronous. */
int dp_debug_pipe_trace(uint64_t* out_host, int32_t capacity, int32_t unit /* 0: PCG kernels, 1: standalone SpMV */);

#ifdef __cplusplus
}
#endif
#endif /* DPCG_H */
