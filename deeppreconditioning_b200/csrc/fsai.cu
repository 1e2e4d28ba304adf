// fsai.cu — K8: the FSAI factor (factorized sparse approximate inverse, Kolotilina & Yeremin) on a given pattern.
//
// Convention of the learned factor: L lower triangular, M = L L^T ~ A^-1. The kernel fills U = L^T (CSR, upper): row i
// of U is column i of L, its pattern J = (j_0 = i < j_1 < ... < j_{k-1}). With S = A[J, J] (k x k, SPD for SPD A), the
// row is y / sqrt(y_0) where S y = e_0, which makes (L^T A L)_ii = 1. Rows are independent: one warp per row, lane p owns
// local row p of S, R and the vectors, S / R live in the warp's slice of shared memory (R overwrites S).
//
// Arithmetic order (oracle_fsai in tests/fsai_oracle.c runs the same loops; every product, difference, quotient and square
// root is rounded separately, so the two agree bit for bit):
//   Cholesky S = R R^T by columns q: d = S_qq - R_q0^2 - ... (ascending t), R_qq = sqrt(d);
//                                    R_pq = (S_pq - R_p0 R_q0 - ...) / R_qq (p > q, ascending t)
//   forward   w_0 = 1 / R_00; w_p = (0 - R_p0 w_0 - ...) / R_pp         (ascending t)
//   backward  y_p = (w_p - R_{p+1,p} y_{p+1} - ...) / R_pp                 (ascending t, p from k-1 down to 0)
//   output    g = sqrt(y_0), U[i, j_p] = y_p / g (rounded once to fp32 and widened back when fp32 is set)
// A column step runs its entries on separate lanes, each with its own sequential chain; the forward substitution runs
// column-oriented (lane p subtracts R_pt w_t as soon as w_t is known: still ascending t); the backward substitution's
// first term needs the last result, so it is one chain, run by every lane on broadcast operands.
#include <math.h>

#include "common.cuh"

namespace dp {

constexpr int kFsaiMaxRow = 32;                  // one lane per local row
constexpr int kFsaiStride = kFsaiMaxRow + 1;     // row stride of S / R in doubles
constexpr int kFsaiWarps = 4;                    // warps per CTA: 4 x 8.4 KB of shared memory
constexpr int kFsaiThreads = kFsaiWarps * kWarp;

struct FsaiWarpSmem {
    double r[kFsaiMaxRow * kFsaiStride];  // S, overwritten column by column with R (lower triangle)
    double w[kFsaiMaxRow];                // forward substitution
    double y[kFsaiMaxRow];                // backward substitution
    int j[kFsaiMaxRow];                   // the row's pattern
};

__device__ __forceinline__ void fsai_raise(int* flag, int status) { *(volatile int*)flag = status; }

__global__ void __launch_bounds__(kFsaiThreads) fsai_kernel(int n, const int* __restrict__ a_rowptr,
                                                            const int* __restrict__ a_col, const double* __restrict__ a_val,
                                                            const int* __restrict__ u_rowptr,
                                                            const int* __restrict__ u_col, int fp32,
                                                            double* __restrict__ u_val, int* __restrict__ flag) {
    __shared__ FsaiWarpSmem smem[kFsaiWarps];
    const int lane = threadIdx.x & (kWarp - 1);
    FsaiWarpSmem& sm = smem[threadIdx.x / kWarp];
    double* r = sm.r;
    const int warps = gridDim.x * kFsaiWarps;
    for (int i = blockIdx.x * kFsaiWarps + threadIdx.x / kWarp; i < n; i += warps) {
        __syncwarp();  // the previous row is done with j, S, w and y
        const int rs = u_rowptr[i], k = u_rowptr[i + 1] - rs;
        if (k < 1 || k > kFsaiMaxRow) {
            if (lane == 0) fsai_raise(flag, DP_ERR_STRUCTURE);
            continue;
        }
        // pattern: diagonal first, ascending, inside the matrix
        const int jp = lane < k ? u_col[rs + lane] : 0x7fffffff;
        const int prev = __shfl_up_sync(kFull, jp, 1);
        const bool bad = lane < k && (lane == 0 ? jp != i : (jp <= prev || jp >= n));
        if (__any_sync(kFull, bad)) {
            if (lane == 0) fsai_raise(flag, DP_ERR_STRUCTURE);
            continue;
        }
        if (lane < k) sm.j[lane] = jp;
        __syncwarp();
        // S_pq = A[j_p, j_q] for q <= p: merge row j_p of A with j_0..j_p (not stored: 0)
        bool diag = false;
        if (lane < k) {
            double* row = r + lane * kFsaiStride;
            for (int q = 0; q <= lane; ++q) row[q] = 0.0;
            int a = a_rowptr[jp], q = 0;
            const int ae = a_rowptr[jp + 1];
            while (a < ae && q <= lane) {
                const int c = a_col[a], jq = sm.j[q];
                if (c == jq) {
                    row[q] = a_val[a];
                    diag = q == lane;
                    ++a, ++q;
                } else if (c < jq) {
                    ++a;
                } else {
                    ++q;
                }
            }
        }
        if (__any_sync(kFull, lane < k && !diag)) {
            if (lane == 0) fsai_raise(flag, DP_ERR_STRUCTURE);
            continue;
        }
        __syncwarp();
        // Cholesky, left-looking by columns
        bool spd = true;
        for (int q = 0; q < k; ++q) {
            double s = 0.0;
            if (lane >= q && lane < k) {
                const double* rp = r + lane * kFsaiStride;
                const double* rq = r + q * kFsaiStride;
                s = rp[q];
                for (int t = 0; t < q; ++t) s = __dsub_rn(s, __dmul_rn(rp[t], rq[t]));
            }
            const double d = __shfl_sync(kFull, s, q);
            if (!(d > 0.0)) {
                spd = false;
                break;
            }
            const double rqq = __dsqrt_rn(d);
            if (lane == q) r[q * kFsaiStride + q] = rqq;
            else if (lane > q && lane < k) r[lane * kFsaiStride + q] = __ddiv_rn(s, rqq);
            __syncwarp();
        }
        if (!spd) {
            if (lane == 0) fsai_raise(flag, DP_ERR_NOT_SPD);
            continue;
        }
        // forward substitution R w = e_0, column-oriented
        double acc = lane == 0 ? 1.0 : 0.0;
        for (int t = 0; t < k; ++t) {
            const double wt = __shfl_sync(kFull, lane == t ? __ddiv_rn(acc, r[t * kFsaiStride + t]) : 0.0, t);
            if (lane == t) sm.w[t] = wt;
            if (lane > t && lane < k) acc = __dsub_rn(acc, __dmul_rn(r[lane * kFsaiStride + t], wt));
        }
        __syncwarp();
        // backward substitution R^T y = w: one chain, every lane runs it on broadcast operands
        for (int p = k - 1; p >= 0; --p) {
            double s = sm.w[p];
            for (int t = p + 1; t < k; ++t) s = __dsub_rn(s, __dmul_rn(r[t * kFsaiStride + p], sm.y[t]));
            const double yp = __ddiv_rn(s, r[p * kFsaiStride + p]);
            if (lane == 0) sm.y[p] = yp;
            __syncwarp();
        }
        const double y0 = sm.y[0];
        if (!(y0 > 0.0)) {
            if (lane == 0) fsai_raise(flag, DP_ERR_NOT_SPD);
            continue;
        }
        if (lane < k) {
            double v = __ddiv_rn(sm.y[lane], __dsqrt_rn(y0));
            if (fp32) v = (double)__double2float_rn(v);
            u_val[rs + lane] = v;
        }
    }
}

}  // namespace dp

using namespace dp;

extern "C" {

int32_t dp_fsai_max_row_entries(void) { return kFsaiMaxRow; }

int dp_fsai_f64(int32_t n, const int32_t* a_rowptr, const int32_t* a_col, const double* a_val, const int32_t* u_rowptr,
                const int32_t* u_col, int32_t fp32, double* u_val, int32_t* flag_out, void* stream) {
    if (n < 0 || (fp32 != 0 && fp32 != 1)) return DP_ERR_INVALID;
    if (n == 0) return DP_OK;
    if (!a_rowptr || !a_col || !a_val || !u_rowptr || !u_col || !u_val || !flag_out) return DP_ERR_INVALID;
    if (!aligned16(a_col) || !aligned16(a_val) || !aligned16(u_col) || !aligned16(u_val)) return DP_ERR_ALIGNMENT;
    const int blocks_needed = (n + kFsaiWarps - 1) / kFsaiWarps;
    const int cap = sm_count() * 8;
    const int grid = blocks_needed < cap ? blocks_needed : cap;
    fsai_kernel<<<grid, kFsaiThreads, 0, (cudaStream_t)stream>>>(n, a_rowptr, a_col, a_val, u_rowptr, u_col, fp32, u_val,
                                                                 flag_out);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

}  // extern "C"
