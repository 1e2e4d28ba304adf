// assembly.cu — K1: CSR assembly of L / L^T / A straight from the spconv COO layout, explicit CSR transpose,
// inverse diagonal. Replaces the dense N x N round trips of test.py:61-68 and test.py:100-105.
//
// Pipeline (all integer work exact, values only widened fp32 -> fp64):
//   count  : one thread per COO entry, filter (batch, row < n, col < n, row >= col, value != 0), atomicAdd per row
//   scan   : exclusive prefix sum -> rowptr
//   fill   : entries dropped into their row segment at an atomically claimed slot (order inside a row arbitrary)
//   sort   : every row sorted by column -> the output no longer depends on the atomic order: bit-exact
//            against torch's to_sparse_csr() / scipy; a repeated (row, col) raises DP_ERR_STRUCTURE.
// Symbolic product of two patterns (FSAI power patterns, the density count): count rows, scan, fill first occurrences,
// sort rows - the same integer pipeline with the row union (row_union) as the count and the fill.
#include "common.cuh"
#include "scan.cuh"

namespace dp {

struct CooEntry {
    int r, c;
    float v;
    bool keep;
};

__device__ __forceinline__ CooEntry coo_load(const int* __restrict__ ind, const float* __restrict__ feat, long long e,
                                             int batch, int n) {
    CooEntry t;
    const int b = ind[3 * e];
    t.r = ind[3 * e + 1];
    t.c = ind[3 * e + 2];
    t.v = feat[e];
    // `[batch, 0, :n, :n]` slice, lower triangle (model.py:53-54 zeroes the rest by value), exact zeros dropped
    // like Tensor.to_sparse_csr() (test.py:105). NaN != 0 is kept, -0.0 is dropped, as torch does.
    t.keep = b == batch && (unsigned)t.r < (unsigned)n && (unsigned)t.c < (unsigned)n && t.r >= t.c && t.v != 0.0f;
    return t;
}

__global__ void coo_count_kernel(const int* __restrict__ ind, const float* __restrict__ feat, long long nnz, int batch,
                                 int n, int mode, int* __restrict__ count) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nnz;
         e += (long long)gridDim.x * blockDim.x) {
        const CooEntry t = coo_load(ind, feat, e, batch, n);
        if (!t.keep) continue;
        if (mode == DP_ASSEMBLE_TRIL) {
            atomicAdd(count + t.r, 1);
        } else if (mode == DP_ASSEMBLE_TRIL_T) {
            atomicAdd(count + t.c, 1);
        } else {
            atomicAdd(count + t.r, 1);
            if (t.r > t.c) atomicAdd(count + t.c, 1);
        }
    }
}

__global__ void coo_fill_kernel(const int* __restrict__ ind, const float* __restrict__ feat, long long nnz, int batch,
                                int n, int mode, const int* __restrict__ rowptr, int* __restrict__ cursor,
                                int* __restrict__ col, double* __restrict__ val) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nnz;
         e += (long long)gridDim.x * blockDim.x) {
        const CooEntry t = coo_load(ind, feat, e, batch, n);
        if (!t.keep) continue;
        const double v = (double)t.v;  // exact widening (test.py:68,105: .to(torch.float64))
        if (mode != DP_ASSEMBLE_TRIL_T) {
            const int pos = rowptr[t.r] + atomicAdd(cursor + t.r, 1);
            col[pos] = t.c;
            val[pos] = v;
        }
        if (mode == DP_ASSEMBLE_TRIL_T || (mode == DP_ASSEMBLE_SYMMETRISE && t.r > t.c)) {
            const int pos = rowptr[t.c] + atomicAdd(cursor + t.c, 1);
            col[pos] = t.r;
            val[pos] = v;
        }
    }
}

// One thread per row: insertion sort by column (rows on this path hold 3..~25 entries), then duplicate check.
// val == NULL: a pattern without values; flag == NULL: no duplicate check.
__global__ void csr_sort_rows_kernel(int n, const int* __restrict__ rowptr, int* __restrict__ col,
                                     double* __restrict__ val, int* __restrict__ flag) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int rs = rowptr[i], re = rowptr[i + 1];
        for (int p = rs + 1; p < re; ++p) {
            const int kc = col[p];
            const double kv = val ? val[p] : 0.0;
            int q = p - 1;
            while (q >= rs && col[q] > kc) {
                col[q + 1] = col[q];
                if (val) val[q + 1] = val[q];
                --q;
            }
            col[q + 1] = kc;
            if (val) val[q + 1] = kv;
        }
        if (flag)
            for (int p = rs + 1; p < re; ++p)
                if (col[p] == col[p - 1]) atomicCAS(flag, 0, (int)DP_ERR_STRUCTURE);
    }
}

__global__ void csr_count_cols_kernel(int n, const int* __restrict__ rowptr, const int* __restrict__ col,
                                      int* __restrict__ count) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        for (int p = rowptr[i]; p < rowptr[i + 1]; ++p) atomicAdd(count + col[p], 1);
}

__global__ void csr_transpose_fill_kernel(int n, const int* __restrict__ rowptr, const int* __restrict__ col,
                                          const double* __restrict__ val, const int* __restrict__ rowptr_t,
                                          int* __restrict__ cursor, int* __restrict__ col_t,
                                          double* __restrict__ val_t) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        for (int p = rowptr[i]; p < rowptr[i + 1]; ++p) {
            const int j = col[p];
            const int pos = rowptr_t[j] + atomicAdd(cursor + j, 1);
            col_t[pos] = i;
            val_t[pos] = val[p];
        }
}

__global__ void copy_last_kernel(const int* __restrict__ rowptr, int n, int* __restrict__ nnz_out) {
    if (blockIdx.x == 0 && threadIdx.x == 0) *nnz_out = rowptr[n];
}

__global__ void inv_diagonal_kernel(int n, const int* __restrict__ rowptr, const int* __restrict__ col,
                                    const double* __restrict__ val, double* __restrict__ dinv, int* __restrict__ flag) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        double d = 0.0;
        bool found = false;
        for (int p = rowptr[i]; p < rowptr[i + 1]; ++p)
            if (col[p] == i) {
                d = val[p];
                found = true;
            }
        if (!found) atomicCAS(flag, 0, (int)DP_ERR_STRUCTURE);
        dinv[i] = found ? __ddiv_rn(1.0, d) : 0.0;  // `1 / matrix.diagonal()`, test.py:76
    }
}


// Row i of the structural product C = P Q (values never read, nothing cancels): the union, over the columns c of row i
// of P, of row c of Q. One warp per row; the lanes take the entries of row c of Q 32 at a time, and candidate j is a
// FIRST occurrence iff it lies in none of the rows c' of Q for the columns c' before c in row i of P (binary search:
// every row of Q is sorted). No buffer, so no cap on the length of a row of C. lower: candidates j > i take no part.
// Columns of P or Q outside [0, n) are skipped and raise DP_ERR_STRUCTURE in *flag (when flag != NULL).
// emit(first, j) is called by all 32 lanes together, once per group of 32 candidates and in candidate order (lanes past
// the end of the row of Q pass first = false), so a caller can count by ballot or place first occurrences by prefix.
template <class Emit>
__device__ __forceinline__ void row_union(int i, int n, const int* __restrict__ p_rowptr, const int* __restrict__ p_col,
                                          const int* __restrict__ q_rowptr, const int* __restrict__ q_col, int lower,
                                          int* __restrict__ flag, Emit&& emit) {
    const int lane = threadIdx.x & 31;
    const int rs = p_rowptr[i], re = p_rowptr[i + 1];
    for (int k = rs; k < re; ++k) {
        const int c = p_col[k];
        if ((unsigned)c >= (unsigned)n) {
            if (flag && lane == 0) atomicCAS(flag, 0, (int)DP_ERR_STRUCTURE);
            continue;
        }
        const int ts = q_rowptr[c], te = q_rowptr[c + 1];
        for (int base = ts; base < te; base += 32) {
            const int q = base + lane;
            const int j = q < te ? q_col[q] : -1;
            bool first = false;
            if (q < te && (unsigned)j >= (unsigned)n) {
                if (flag) atomicCAS(flag, 0, (int)DP_ERR_STRUCTURE);
            } else if (q < te && (!lower || j <= i)) {
                first = true;
                for (int k2 = rs; k2 < k && first; ++k2) {
                    const int c2 = p_col[k2];
                    if ((unsigned)c2 >= (unsigned)n) continue;
                    int lo = q_rowptr[c2], hi = q_rowptr[c2 + 1];
                    while (lo < hi) {
                        const int mid = (lo + hi) >> 1;
                        const int v = q_col[mid];
                        if (v == j) { first = false; break; }
                        if (v < j) lo = mid + 1; else hi = mid;
                    }
                }
            }
            emit(first, j);
        }
    }
}

// Entries per row of C = P Q (counts[i], when counts != NULL) and their 64-bit total by atomics. Integer work, exact.
// Also the count behind dp_csr_aat_nnz: nnz(L L^T) without forming the product (test.py:107-109 reports the density of
// the explicit M = L L^T that test.py:104-105 stores) is this count with P = L, Q = L^T.
__global__ void __launch_bounds__(256) pattern_count_kernel(int n, const int* __restrict__ p_rowptr,
                                                            const int* __restrict__ p_col, const int* __restrict__ q_rowptr,
                                                            const int* __restrict__ q_col, int lower,
                                                            int* __restrict__ counts, unsigned long long* __restrict__ total,
                                                            int* __restrict__ flag) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    unsigned long long mine = 0;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
        int row = 0;
        row_union(i, n, p_rowptr, p_col, q_rowptr, q_col, lower, flag,
                  [&](bool first, int) { row += __popc(__ballot_sync(kFull, first)); });
        if (counts && lane == 0) counts[i] = row;
        mine += (unsigned long long)row;
    }
    if (lane == 0 && mine) atomicAdd(total, mine);
}

// Row i of C written at c_rowptr[i] in candidate order (first occurrences only, placed by a warp prefix of the ballot):
// the same entries pattern_count_kernel counted, deterministic, sorted afterwards by csr_sort_rows_kernel.
__global__ void __launch_bounds__(256) pattern_fill_kernel(int n, const int* __restrict__ p_rowptr,
                                                           const int* __restrict__ p_col, const int* __restrict__ q_rowptr,
                                                           const int* __restrict__ q_col, int lower,
                                                           const int* __restrict__ c_rowptr, int* __restrict__ c_col) {
    const int lane = threadIdx.x & 31;
    const int warps = (gridDim.x * blockDim.x) >> 5;
    for (int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += warps) {
        int pos = c_rowptr[i];
        row_union(i, n, p_rowptr, p_col, q_rowptr, q_col, lower, nullptr, [&](bool first, int j) {
            const unsigned mask = __ballot_sync(kFull, first);
            if (first) c_col[pos + __popc(mask & ((1u << lane) - 1u))] = j;
            pos += __popc(mask);
        });
    }
}

static int grid_for(long long items, int threads) {
    long long b = (items + threads - 1) / threads;
    long long cap = (long long)sm_count() * 16;
    if (b > cap) b = cap;
    return b < 1 ? 1 : (int)b;
}

// workspace layout: [cursor/count: (n+1) int][scan scratch]
static size_t assembly_ws_bytes(int n) { return align_up(sizeof(int) * ((size_t)n + 1), 256) + scan_workspace_bytes((long long)n + 1); }

}  // namespace dp

using namespace dp;

extern "C" {

size_t dp_csr_from_coo_workspace_bytes(int32_t n, int64_t nnz_in) {
    (void)nnz_in;
    return assembly_ws_bytes(n < 0 ? 0 : n);
}

int dp_csr_from_coo(const int32_t* indices, const float* features, int64_t nnz_in, int32_t batch, int32_t n,
                    int32_t mode, int32_t* rowptr, int32_t* col, double* val, int32_t* nnz_out, int32_t* flag_out,
                    void* workspace, size_t workspace_bytes, void* stream) {
    if (n < 0 || nnz_in < 0 || mode < 0 || mode > 2 || !rowptr || !flag_out || !workspace) return DP_ERR_INVALID;
    if (nnz_in > 0 && (!indices || !features || !col || !val)) return DP_ERR_INVALID;
    if (!aligned16(col) || !aligned16(val) || !aligned16(workspace)) return DP_ERR_ALIGNMENT;
    if (workspace_bytes < assembly_ws_bytes(n)) return DP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    int* cursor = static_cast<int*>(workspace);
    void* scan_ws = static_cast<char*>(workspace) + align_up(sizeof(int) * ((size_t)n + 1), 256);

    DP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * ((size_t)n + 1), s));
    if (nnz_in > 0) {
        coo_count_kernel<<<grid_for(nnz_in, 256), 256, 0, s>>>(indices, features, nnz_in, batch, n, mode, cursor);
        DP_LAUNCH_CHECK();
    }
    int st = exclusive_scan_i32(cursor, rowptr, (long long)n + 1, scan_ws, s);
    if (st != DP_OK) return st;
    DP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * ((size_t)n + 1), s));
    if (nnz_in > 0) {
        coo_fill_kernel<<<grid_for(nnz_in, 256), 256, 0, s>>>(indices, features, nnz_in, batch, n, mode, rowptr,
                                                              cursor, col, val);
        DP_LAUNCH_CHECK();
        csr_sort_rows_kernel<<<grid_for(n, 128), 128, 0, s>>>(n, rowptr, col, val, flag_out);
        DP_LAUNCH_CHECK();
    }
    if (nnz_out) {
        copy_last_kernel<<<1, 32, 0, s>>>(rowptr, n, nnz_out);
        DP_LAUNCH_CHECK();
    }
    return DP_OK;
}

size_t dp_csr_transpose_workspace_bytes(int32_t n, int32_t nnz) {
    (void)nnz;
    return assembly_ws_bytes(n < 0 ? 0 : n);
}

int dp_csr_transpose(int32_t n, int32_t nnz, const int32_t* rowptr, const int32_t* col, const double* val,
                     int32_t* rowptr_t, int32_t* col_t, double* val_t, void* workspace, size_t workspace_bytes,
                     void* stream) {
    if (n < 0 || nnz < 0 || !rowptr || !rowptr_t || !workspace) return DP_ERR_INVALID;
    if (nnz > 0 && (!col || !val || !col_t || !val_t)) return DP_ERR_INVALID;
    if (!aligned16(col_t) || !aligned16(val_t) || !aligned16(workspace)) return DP_ERR_ALIGNMENT;
    if (workspace_bytes < assembly_ws_bytes(n)) return DP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    int* cursor = static_cast<int*>(workspace);
    void* scan_ws = static_cast<char*>(workspace) + align_up(sizeof(int) * ((size_t)n + 1), 256);

    DP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * ((size_t)n + 1), s));
    if (n > 0 && nnz > 0) {
        csr_count_cols_kernel<<<grid_for(n, 256), 256, 0, s>>>(n, rowptr, col, cursor);
        DP_LAUNCH_CHECK();
    }
    int st = exclusive_scan_i32(cursor, rowptr_t, (long long)n + 1, scan_ws, s);
    if (st != DP_OK) return st;
    DP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * ((size_t)n + 1), s));
    if (n > 0 && nnz > 0) {
        csr_transpose_fill_kernel<<<grid_for(n, 256), 256, 0, s>>>(n, rowptr, col, val, rowptr_t, cursor, col_t, val_t);
        DP_LAUNCH_CHECK();
        // flag: duplicates cannot appear in a transpose of a valid CSR; reuse cursor[n] as a sink
        csr_sort_rows_kernel<<<grid_for(n, 128), 128, 0, s>>>(n, rowptr_t, col_t, val_t, cursor + n);
        DP_LAUNCH_CHECK();
    }
    return DP_OK;
}

int dp_csr_inv_diagonal(int32_t n, const int32_t* rowptr, const int32_t* col, const double* val, double* dinv,
                        int32_t* flag_out, void* stream) {
    if (n < 0 || !rowptr || !dinv || !flag_out) return DP_ERR_INVALID;
    if (n == 0) return DP_OK;
    inv_diagonal_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(n, rowptr, col, val, dinv, flag_out);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

int dp_csr_aat_nnz(int32_t n, const int32_t* rowptr, const int32_t* col, const int32_t* rowptr_t, const int32_t* col_t,
                   int64_t* nnz_out, void* stream) {
    if (n < 0 || !nnz_out || (n > 0 && (!rowptr || !col || !rowptr_t || !col_t))) return DP_ERR_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    DP_CUDA(cudaMemsetAsync(nnz_out, 0, sizeof(int64_t), s));
    if (n == 0) return DP_OK;
    pattern_count_kernel<<<grid_for((long long)n * 32, 256), 256, 0, s>>>(
        n, rowptr, col, rowptr_t, col_t, 0, nullptr, reinterpret_cast<unsigned long long*>(nnz_out), nullptr);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

size_t dp_csr_pattern_product_workspace_bytes(int32_t n) { return scan_workspace_bytes((long long)(n < 0 ? 0 : n) + 1); }

int dp_csr_pattern_product_count(int32_t n, const int32_t* p_rowptr, const int32_t* p_col, const int32_t* q_rowptr,
                                 const int32_t* q_col, int32_t lower, int32_t* c_rowptr, int64_t* nnz_out,
                                 int32_t* flag_out, void* workspace, size_t workspace_bytes, void* stream) {
    if (n < 0 || (lower != 0 && lower != 1)) return DP_ERR_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    if (n == 0) {  // the empty product: rowptr = {0}, total 0 (outputs that are not given are left alone)
        if (c_rowptr) DP_CUDA(cudaMemsetAsync(c_rowptr, 0, sizeof(int32_t), s));
        if (nnz_out) DP_CUDA(cudaMemsetAsync(nnz_out, 0, sizeof(int64_t), s));
        return DP_OK;
    }
    if (!p_rowptr || !p_col || !q_rowptr || !q_col || !c_rowptr || !nnz_out || !flag_out || !workspace)
        return DP_ERR_INVALID;
    if (!aligned16(workspace)) return DP_ERR_ALIGNMENT;
    if (workspace_bytes < dp_csr_pattern_product_workspace_bytes(n)) return DP_ERR_WORKSPACE;
    DP_CUDA(cudaMemsetAsync(nnz_out, 0, sizeof(int64_t), s));
    DP_CUDA(cudaMemsetAsync(c_rowptr + n, 0, sizeof(int32_t), s));
    // row counts land in c_rowptr[0..n) and are scanned in place into the row pointers
    pattern_count_kernel<<<grid_for((long long)n * 32, 256), 256, 0, s>>>(
        n, p_rowptr, p_col, q_rowptr, q_col, lower, c_rowptr, reinterpret_cast<unsigned long long*>(nnz_out), flag_out);
    DP_LAUNCH_CHECK();
    return exclusive_scan_i32(c_rowptr, c_rowptr, (long long)n + 1, workspace, s);
}

int dp_csr_pattern_product_fill(int32_t n, const int32_t* p_rowptr, const int32_t* p_col, const int32_t* q_rowptr,
                                const int32_t* q_col, int32_t lower, const int32_t* c_rowptr, int32_t* c_col,
                                void* stream) {
    if (n < 0 || (lower != 0 && lower != 1)) return DP_ERR_INVALID;
    if (n == 0) return DP_OK;
    if (!p_rowptr || !p_col || !q_rowptr || !q_col || !c_rowptr || !c_col) return DP_ERR_INVALID;
    if (!aligned16(c_col)) return DP_ERR_ALIGNMENT;
    cudaStream_t s = (cudaStream_t)stream;
    pattern_fill_kernel<<<grid_for((long long)n * 32, 256), 256, 0, s>>>(n, p_rowptr, p_col, q_rowptr, q_col, lower,
                                                                         c_rowptr, c_col);
    DP_LAUNCH_CHECK();
    csr_sort_rows_kernel<<<grid_for(n, 128), 128, 0, s>>>(n, c_rowptr, c_col, nullptr, nullptr);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

}  // extern "C"
