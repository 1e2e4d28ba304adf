// losses.cu — the training losses' sparse products in a fixed order (metrics.py, utils.sparse_matvec_mul under
// torch.use_deterministic_algorithms).
//
// dp_coo_spmv_batch_f32 (spmv.cu) adds one product per COO entry into the output with fp32 atomics, so its sums
// depend on the order the atomics land in. Here the sites come sorted (dp_spconv_sort_sites: a per-(batch, row) CSR
// with ascending columns and the permutation back to the input), and every output value is one sequential sum:
//   y[b,p,i] = (((0 + f_0 x_c0) + f_1 x_c1) + ...)      ascending column, __fmul_rn / __fadd_rn (no fma contraction)
// which is the oracle's loop (oracle/kernels.c) on the sorted sites. The transposed product reads the column CSR (the
// sort of the indices with row and column swapped), so it needs no atomics either.
//
// Loss  sum_p || L L^T x_p - b_p ||  per system: t = L^T x, r = L t - b in fp32; sum r^2 in fp64 per fixed chunk of
// kResidualChunk rows (CTA tree of block_sum, a constant shape), the chunk partials and then the probes added in order by
// one thread per system. Neither the grid, the batch nor the site order changes a bit. Its gradient with respect to the
// features of L is a closed form per site (see dp_llt_residual_grad_f32 in dpcg.h): no floating-point accumulation
// across sites, so the backward has no atomics and no reduction at all beyond s = L^T rho, itself a product as above.
#include <math.h>

#include "common.cuh"

namespace dp {

constexpr int kResidualChunk = 8 * kBlock;  // rows per fp64 partial of sum r^2 (8 per thread of a 512-thread CTA)
constexpr int kLossThreads = 256;

__device__ __forceinline__ float row_product(const int* __restrict__ rowptr, const int* __restrict__ col,
                                             const int* __restrict__ perm, const float* __restrict__ feat, int row,
                                             const float* __restrict__ x, int n) {
    float acc = 0.0f;
    const int qe = rowptr[row + 1];
    for (int q = rowptr[row]; q < qe; ++q) {
        const int c = col[q];
        if (c < n) acc = __fadd_rn(acc, __fmul_rn(feat[perm[q]], x[c]));
    }
    return acc;
}

// One thread per output value (b, p, i); rows at or beyond the pattern's `rows` have no sites.
__global__ void sorted_spmv_kernel(const int* __restrict__ rowptr, const int* __restrict__ col,
                                   const int* __restrict__ perm, const float* __restrict__ feat, int nbatch, int rows,
                                   int nvec, int n, const float* __restrict__ x, float* __restrict__ y) {
    const long long total = (long long)nbatch * nvec * n;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e % n);
        const long long bp = e / n;
        const int b = (int)(bp / nvec);
        y[e] = i < rows ? row_product(rowptr, col, perm, feat, b * rows + i, x + bp * n, n) : 0.0f;
    }
}

// (T v + T^T v) - D v, associated as metrics.system_matvec: three products, the diagonal one a single term from 0.
__global__ void system_matvec_kernel(dp_factor_sites_t S, int nvec, int n, const float* __restrict__ v,
                                     float* __restrict__ y) {
    const long long total = (long long)S.nbatch * nvec * n;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const int i = (int)(e % n);
        const long long bp = e / n;
        const int b = (int)(bp / nvec);
        const float* vb = v + bp * n;
        float lower = 0.0f, upper = 0.0f, diag = 0.0f;
        if (i < S.h) {
            const int row = b * S.h + i;
            lower = row_product(S.rowptr, S.col, S.perm, S.features, row, vb, n);
            for (int q = S.rowptr[row]; q < S.rowptr[row + 1]; ++q)
                if (S.col[q] == i) diag = __fadd_rn(0.0f, __fmul_rn(S.features[S.perm[q]], vb[i]));
        }
        if (i < S.w) upper = row_product(S.rowptr_t, S.col_t, S.perm_t, S.features, b * S.w + i, vb, n);
        y[e] = __fsub_rn(__fadd_rn(lower, upper), diag);
    }
}

// One CTA per (system, probe, chunk): r = L t - b over the chunk's rows and the fp64 sum of r^2 in a fixed tree.
__global__ void __launch_bounds__(kBlock) residual_chunk_kernel(dp_factor_sites_t S, int nvec, int n, long long nchunks,
                                                                const float* __restrict__ t, const float* __restrict__ b,
                                                                float* __restrict__ r, double* __restrict__ part) {
    __shared__ double scratch[kWarpsPerBlock];
    const long long items = (long long)S.nbatch * nvec * nchunks;
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        const long long bp = item / nchunks;
        const int chunk = (int)(item % nchunks);
        const int sys = (int)(bp / nvec);
        const float* tb = t + bp * n;
        double acc = 0.0;
#pragma unroll 1
        for (int j = 0; j < kResidualChunk / kBlock; ++j) {
            const int i = chunk * kResidualChunk + j * kBlock + (int)threadIdx.x;
            if (i >= n) break;
            const float u = i < S.h ? row_product(S.rowptr, S.col, S.perm, S.features, sys * S.h + i, tb, n) : 0.0f;
            const float ri = __fsub_rn(u, b[bp * n + i]);
            r[bp * n + i] = ri;
            acc = __dadd_rn(acc, __dmul_rn((double)ri, (double)ri));
        }
        acc = block_sum(acc, scratch);
        if (threadIdx.x == 0) part[item] = acc;
    }
}

// One CTA: per system the chunk partials in chunk order, the probes in probe order, then the terms in system order.
__global__ void residual_finish_kernel(const double* __restrict__ part, int nbatch, int nvec, long long nchunks,
                                       int divisor, int mean, float* __restrict__ terms, float* __restrict__ loss) {
    for (int sys = threadIdx.x; sys < nbatch; sys += blockDim.x) {
        double total = 0.0;
        for (int p = 0; p < nvec; ++p) {
            const double* row = part + ((long long)sys * nvec + p) * nchunks;
            double sq = 0.0;
            for (long long c = 0; c < nchunks; ++c) sq = __dadd_rn(sq, row[c]);
            total = __dadd_rn(total, sq);
        }
        terms[sys] = (float)__dsqrt_rn(__ddiv_rn(total, (double)divisor));
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float sum = 0.0f;
        for (int sys = 0; sys < nbatch; ++sys) sum = __fadd_rn(sum, terms[sys]);
        *loss = mean ? __fdiv_rn(sum, (float)nbatch) : sum;
    }
}

// rho = c_b r with c_b = g' / (divisor terms[b]), 0 for a system whose residual is zero (vector_norm's backward).
__global__ void residual_scale_kernel(int nbatch, int nvec, int n, int divisor, int mean, const float* __restrict__ terms,
                                      const float* __restrict__ grad_loss, const float* __restrict__ r,
                                      float* __restrict__ rho) {
    const long long total = (long long)nbatch * nvec * n;
    const float g = mean ? __fdiv_rn(*grad_loss, (float)nbatch) : *grad_loss;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const float term = terms[e / ((long long)nvec * n)];
        const float c = term > 0.0f ? __fdiv_rn(g, __fmul_rn((float)divisor, term)) : 0.0f;
        rho[e] = __fmul_rn(c, r[e]);
    }
}

// One thread per row (b, i) of L's row CSR: every site (b, i, k) of the row gets sum_p (rho_i t_k + x_i s_k).
__global__ void site_grad_kernel(dp_factor_sites_t S, int nvec, int n, const float* __restrict__ x,
                                 const float* __restrict__ t, const float* __restrict__ rho, const float* __restrict__ s,
                                 float* __restrict__ grad) {
    const long long rows = (long long)S.nbatch * S.h;
    for (long long row = blockIdx.x * (long long)blockDim.x + threadIdx.x; row < rows; row += (long long)gridDim.x * blockDim.x) {
        const int b = (int)(row / S.h), i = (int)(row % S.h);
        const int qe = S.rowptr[row + 1];
        for (int q = S.rowptr[row]; q < qe; ++q) {
            const int k = S.col[q];
            float acc = 0.0f;
            if (i < n && k < n) {
                for (int p = 0; p < nvec; ++p) {
                    const long long base = ((long long)b * nvec + p) * n;
                    const float term = __fadd_rn(__fmul_rn(rho[base + i], t[base + k]), __fmul_rn(x[base + i], s[base + k]));
                    acc = __fadd_rn(acc, term);
                }
            }
            grad[S.perm[q]] = acc;
        }
    }
}

static int grid_for(long long items, int threads) {
    long long b = (items + threads - 1) / threads;
    const long long cap = (long long)sm_count() * 16;
    if (b > cap) b = cap;
    return b < 1 ? 1 : (int)b;
}

static long long residual_chunks(int n) { return ((long long)n + kResidualChunk - 1) / kResidualChunk; }

static size_t llt_ws_bytes(int nbatch, int nvec, int n) {
    const size_t vec = (size_t)nbatch * nvec * n;
    const size_t fwd = sizeof(double) * (size_t)nbatch * nvec * residual_chunks(n);
    const size_t bwd = 2 * align_up(sizeof(float) * vec, 256);
    return align_up(fwd > bwd ? fwd : bwd, 256);
}

static bool sizes_ok(int nvec, int n) { return nvec >= 0 && n >= 0; }

// Shape and pointer checks of a site pattern; `need_rows` / `need_cols`: the CSRs the call reads.
static int sites_ok(const dp_factor_sites_t& S, bool need_rows, bool need_cols) {
    if (S.nnz < 0 || S.nnz > 0x7fffffffLL || S.nbatch < 0 || S.h < 0 || S.w < 0) return DP_ERR_INVALID;
    if ((long long)S.nbatch * S.h >= 0x7fffffffLL || (long long)S.nbatch * S.w >= 0x7fffffffLL) return DP_ERR_INVALID;
    if (S.nnz > 0 && !S.features) return DP_ERR_INVALID;
    if (need_rows && (!S.rowptr || (S.nnz > 0 && (!S.col || !S.perm)))) return DP_ERR_INVALID;
    if (need_cols && (!S.rowptr_t || (S.nnz > 0 && (!S.col_t || !S.perm_t)))) return DP_ERR_INVALID;
    return DP_OK;
}

static bool empty(const dp_factor_sites_t& S, int nvec, int n) { return S.nbatch == 0 || nvec == 0 || n == 0; }

}  // namespace dp

using namespace dp;

extern "C" {

int dp_sorted_spmv_f32(const dp_factor_sites_t* sites_host, int32_t transpose, int32_t nvec, int32_t n, const float* x,
                       float* y, void* stream) {
    if (!sites_host || !sizes_ok(nvec, n) || (transpose != 0 && transpose != 1)) return DP_ERR_INVALID;
    const dp_factor_sites_t& S = *sites_host;
    int st = sites_ok(S, !transpose, transpose != 0);
    if (st != DP_OK) return st;
    if (empty(S, nvec, n)) return DP_OK;
    if (!x || !y) return DP_ERR_INVALID;
    const long long total = (long long)S.nbatch * nvec * n;
    if (transpose)
        sorted_spmv_kernel<<<grid_for(total, kLossThreads), kLossThreads, 0, (cudaStream_t)stream>>>(
            S.rowptr_t, S.col_t, S.perm_t, S.features, S.nbatch, S.w, nvec, n, x, y);
    else
        sorted_spmv_kernel<<<grid_for(total, kLossThreads), kLossThreads, 0, (cudaStream_t)stream>>>(
            S.rowptr, S.col, S.perm, S.features, S.nbatch, S.h, nvec, n, x, y);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

int dp_system_matvec_f32(const dp_factor_sites_t* sites_host, int32_t nvec, int32_t n, const float* v, float* y,
                         void* stream) {
    if (!sites_host || !sizes_ok(nvec, n)) return DP_ERR_INVALID;
    const dp_factor_sites_t& S = *sites_host;
    int st = sites_ok(S, true, true);
    if (st != DP_OK) return st;
    if (empty(S, nvec, n)) return DP_OK;
    if (!v || !y) return DP_ERR_INVALID;
    const long long total = (long long)S.nbatch * nvec * n;
    system_matvec_kernel<<<grid_for(total, kLossThreads), kLossThreads, 0, (cudaStream_t)stream>>>(S, nvec, n, v, y);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

int32_t dp_llt_residual_chunk_rows(void) { return kResidualChunk; }

size_t dp_llt_residual_workspace_bytes(int32_t nbatch, int32_t nvec, int32_t n) {
    return (nbatch >= 0 && sizes_ok(nvec, n)) ? llt_ws_bytes(nbatch, nvec, n) : 0;
}

int dp_llt_residual_f32(const dp_factor_sites_t* sites_host, int32_t nvec, int32_t n, int32_t divisor, int32_t mean,
                        const float* x, const float* b, float* t, float* r, float* terms, float* loss, void* workspace,
                        size_t workspace_bytes, void* stream) {
    if (!sites_host || !sizes_ok(nvec, n) || divisor < 1 || (mean != 0 && mean != 1)) return DP_ERR_INVALID;
    const dp_factor_sites_t& S = *sites_host;
    int st = sites_ok(S, true, true);
    if (st != DP_OK) return st;
    if (empty(S, nvec, n)) return DP_OK;
    if (!x || !b || !t || !r || !terms || !loss || !workspace) return DP_ERR_INVALID;
    if (!aligned16(workspace)) return DP_ERR_ALIGNMENT;
    if (workspace_bytes < llt_ws_bytes(S.nbatch, nvec, n)) return DP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    const long long total = (long long)S.nbatch * nvec * n, nchunks = residual_chunks(n);
    double* part = static_cast<double*>(workspace);
    sorted_spmv_kernel<<<grid_for(total, kLossThreads), kLossThreads, 0, s>>>(S.rowptr_t, S.col_t, S.perm_t, S.features,
                                                                              S.nbatch, S.w, nvec, n, x, t);
    DP_LAUNCH_CHECK();
    const long long items = (long long)S.nbatch * nvec * nchunks;
    const long long cap = (long long)sm_count() * 4;
    residual_chunk_kernel<<<(int)(items < cap ? items : cap), kBlock, 0, s>>>(S, nvec, n, nchunks, t, b, r, part);
    DP_LAUNCH_CHECK();
    residual_finish_kernel<<<1, kLossThreads, 0, s>>>(part, S.nbatch, nvec, nchunks, divisor, mean, terms, loss);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

int dp_llt_residual_grad_f32(const dp_factor_sites_t* sites_host, int32_t nvec, int32_t n, int32_t divisor, int32_t mean,
                             const float* x, const float* t, const float* r, const float* terms, const float* grad_loss,
                             float* grad_features, void* workspace, size_t workspace_bytes, void* stream) {
    if (!sites_host || !sizes_ok(nvec, n) || divisor < 1 || (mean != 0 && mean != 1)) return DP_ERR_INVALID;
    const dp_factor_sites_t& S = *sites_host;
    int st = sites_ok(S, true, true);
    if (st != DP_OK) return st;
    if (S.nnz == 0) return DP_OK;
    if (!grad_features) return DP_ERR_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    if (empty(S, nvec, n)) {  // no vector entry: every site lies beyond the vectors' length
        DP_CUDA(cudaMemsetAsync(grad_features, 0, sizeof(float) * (size_t)S.nnz, s));
        return DP_OK;
    }
    if (!x || !t || !r || !terms || !grad_loss || !workspace) return DP_ERR_INVALID;
    if (!aligned16(workspace)) return DP_ERR_ALIGNMENT;
    if (workspace_bytes < llt_ws_bytes(S.nbatch, nvec, n)) return DP_ERR_WORKSPACE;
    const long long total = (long long)S.nbatch * nvec * n;
    float* rho = static_cast<float*>(workspace);
    float* sv = reinterpret_cast<float*>(static_cast<char*>(workspace) + align_up(sizeof(float) * (size_t)total, 256));
    residual_scale_kernel<<<grid_for(total, kLossThreads), kLossThreads, 0, s>>>(S.nbatch, nvec, n, divisor, mean, terms,
                                                                                 grad_loss, r, rho);
    DP_LAUNCH_CHECK();
    sorted_spmv_kernel<<<grid_for(total, kLossThreads), kLossThreads, 0, s>>>(S.rowptr_t, S.col_t, S.perm_t, S.features,
                                                                              S.nbatch, S.w, nvec, n, rho, sv);
    DP_LAUNCH_CHECK();
    const long long rows = (long long)S.nbatch * S.h;
    if (rows > 0) {
        site_grad_kernel<<<grid_for(rows, kLossThreads), kLossThreads, 0, s>>>(S, nvec, n, x, t, rho, sv, grad_features);
        DP_LAUNCH_CHECK();
    }
    return DP_OK;
}

}  // extern "C"
