// sparseconv.cu — inference of the sparse CNN that makes the learned factor (model.PreconditionerNet /
// PreconditionerTrilNet) on the device: site sort, rule generation of the 2x2 layers, gather-GEMM per layer.
//
// The network's input is the COO image of tril(A): sites (batch, row, col) of an H x W grid with C channels. A 2x2
// layer with padding (ph, pw) in {(1,0), (0,1)} makes output row y the union of the shifted, clipped column lists of
// input rows y - ph and y + 1 - ph (model.SparseConv2d.forward), so with the sites kept as a per-(batch, row) CSR
// whose rows are sorted, rule generation is a per-row merge of four short sorted lists (count, scan, fill), not a
// hash or a global sort. Its output is sorted by (batch, row, col), the order torch.unique gives the PyTorch layer.
//
// Arithmetic (fp32, CUDA cores, fixed order that depends on neither batch composition nor launch geometry):
//   p_t  = sum_{ci ascending} W_t[co, ci] * x[src_t(s), ci]      one fmaf chain from 0 per tap
//   acc  = ((0 + p_(0,0)) + p_(0,1)) + p_(1,0)) + p_(1,1)        inactive taps add nothing (one index_add_ per tap)
//   y    = act(acc + bias)                                        scalar PReLU / LeakyReLU slope
// The last layer before the final 1x1 (cout -> 1) also applies that 1x1 and the output tail of the reference
// (strict upper triangle multiplied by 0, softplus on the diagonal) in its epilogue.
// The training forward (dp_spconv_layer_train_f32) is the same kernel with kTrain set: it also stores what the backward
// (sparseconv_grad.cu) reads - acc + bias before the activation, and in the fused epilogue the activated rows the head
// reads and the head's value before the tail. Its `out` is bitwise the inference launch's.
#include <math.h>

#include "common.cuh"
#include "scan.cuh"

namespace dp {

constexpr int kConvThreads = 256;
constexpr int kMaxChannels = 64;

// ---- site sort ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool site_in_range(const int* __restrict__ ind, long long e, int nb, int h, int w, int* row,
                                              int* col) {
    const int b = ind[3 * e], r = ind[3 * e + 1], c = ind[3 * e + 2];
    *row = b * h + r;
    *col = c;
    return (unsigned)b < (unsigned)nb && (unsigned)r < (unsigned)h && (unsigned)c < (unsigned)w;
}

__global__ void site_count_kernel(const int* __restrict__ ind, long long nnz, int nb, int h, int w,
                                  int* __restrict__ count, int* __restrict__ flag) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nnz; e += (long long)gridDim.x * blockDim.x) {
        int row, col;
        if (site_in_range(ind, e, nb, h, w, &row, &col)) atomicAdd(count + row, 1);
        else atomicCAS(flag, 0, (int)DP_ERR_STRUCTURE);
    }
}

__global__ void site_fill_kernel(const int* __restrict__ ind, long long nnz, int nb, int h, int w,
                                 const int* __restrict__ rowptr, int* __restrict__ cursor, int* __restrict__ col,
                                 int* __restrict__ perm) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nnz; e += (long long)gridDim.x * blockDim.x) {
        int row, c;
        if (!site_in_range(ind, e, nb, h, w, &row, &c)) continue;
        const int pos = rowptr[row] + atomicAdd(cursor + row, 1);
        col[pos] = c;
        perm[pos] = (int)e;
    }
}

// One thread per row: insertion sort of (col, perm) by column (rows of a stencil image hold a handful of sites), then
// the duplicate check. Columns of a row are distinct afterwards unless the flag is raised, so the result is unique.
__global__ void site_sort_rows_kernel(int rows, const int* __restrict__ rowptr, int* __restrict__ col,
                                      int* __restrict__ perm, int* __restrict__ flag) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rows; i += gridDim.x * blockDim.x) {
        const int rs = rowptr[i], re = rowptr[i + 1];
        for (int p = rs + 1; p < re; ++p) {
            const int kc = col[p], kp = perm[p];
            int q = p - 1;
            while (q >= rs && col[q] > kc) {
                col[q + 1] = col[q];
                perm[q + 1] = perm[q];
                --q;
            }
            col[q + 1] = kc;
            perm[q + 1] = kp;
        }
        for (int p = rs + 1; p < re; ++p)
            if (col[p] == col[p - 1]) atomicCAS(flag, 0, (int)DP_ERR_STRUCTURE);
    }
}

// ---- rules of a 2x2 layer ----------------------------------------------------------------------------------------------
// Tap t = 2 ky + kx reads input row ro + ky - ph at column co + kx - pw, i.e. list t is row (ro + ky - ph) with its
// columns shifted by pw - kx. The merge walks the four lists in ascending output column; columns outside [0, wo) are
// dropped (a shift is at most one column, so at most one leading entry per list is negative).
struct RowMerge {
    int pos[4], end[4], off[4];
    const int* col;
    int wo;
    __device__ __forceinline__ void init(const int* __restrict__ rowptr, const int* __restrict__ col_in, int b, int ro,
                                         int h, int ph, int pw, int wo_) {
        col = col_in;
        wo = wo_;
#pragma unroll
        for (int t = 0; t < 4; ++t) {
            const int r = ro + (t >> 1) - ph;
            off[t] = pw - (t & 1);
            if ((unsigned)r < (unsigned)h) {
                pos[t] = rowptr[b * h + r];
                end[t] = rowptr[b * h + r + 1];
            } else {
                pos[t] = end[t] = 0;
            }
            if (pos[t] < end[t] && col[pos[t]] + off[t] < 0) ++pos[t];
        }
    }
    // Smallest pending output column, or -1 when every list is exhausted or past the last column.
    __device__ __forceinline__ int next() const {
        int m = 0x7fffffff;
#pragma unroll
        for (int t = 0; t < 4; ++t)
            if (pos[t] < end[t]) m = min(m, col[pos[t]] + off[t]);
        return m < wo ? m : -1;
    }
};

__global__ void rules_count_kernel(int rows_out, int ho, const int* __restrict__ rowptr_in, const int* __restrict__ col_in,
                                   int h, int ph, int pw, int wo, int* __restrict__ count) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rows_out; i += gridDim.x * blockDim.x) {
        RowMerge m;
        m.init(rowptr_in, col_in, i / ho, i % ho, h, ph, pw, wo);
        int n = 0;
        for (int c = m.next(); c >= 0; c = m.next()) {
#pragma unroll
            for (int t = 0; t < 4; ++t)
                if (m.pos[t] < m.end[t] && col_in[m.pos[t]] + m.off[t] == c) ++m.pos[t];
            ++n;
        }
        count[i] = n;
    }
}

__global__ void rules_fill_kernel(int rows_out, int ho, const int* __restrict__ rowptr_in, const int* __restrict__ col_in,
                                  const int* __restrict__ perm, int h, int ph, int pw, int wo,
                                  const int* __restrict__ rowptr_out, int* __restrict__ col_out, int* __restrict__ rules,
                                  int* __restrict__ indices_out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < rows_out; i += gridDim.x * blockDim.x) {
        const int b = i / ho, ro = i % ho;
        RowMerge m;
        m.init(rowptr_in, col_in, b, ro, h, ph, pw, wo);
        int s = rowptr_out[i];
        for (int c = m.next(); c >= 0; c = m.next(), ++s) {
            int src[4];
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                src[t] = -1;
                if (m.pos[t] < m.end[t] && col_in[m.pos[t]] + m.off[t] == c) {
                    src[t] = perm ? perm[m.pos[t]] : m.pos[t];
                    ++m.pos[t];
                }
            }
            col_out[s] = c;
            reinterpret_cast<int4*>(rules)[s] = make_int4(src[0], src[1], src[2], src[3]);
            if (indices_out) {
                indices_out[3 * (long long)s] = b;
                indices_out[3 * (long long)s + 1] = ro;
                indices_out[3 * (long long)s + 2] = c;
            }
        }
    }
}

// ---- gather-GEMM ---------------------------------------------------------------------------------------------------------
// A CTA of 256 threads computes tiles of kM output sites x COUTP channels (cout <= COUTP, the rest padded with zero
// weights and never stored). The weights of every tap are staged once per CTA as ws[t][ci][co]; per tap the input rows
// of the tile are gathered into xs[site][ci] (zero rows for inactive taps). Thread (ty, tx) owns sites ty + kNY * i
// (i < kTM) and channels tx * kTN + j (j < kTN). The grid strides over the tiles.
template <int COUTP>
struct ConvShape {
    static constexpr int kTN = COUTP >= 64 ? 8 : COUTP >= 4 ? 4 : COUTP;
    static constexpr int kNX = COUTP / kTN;
    static constexpr int kNY = kConvThreads / kNX;
    static constexpr int kTM = COUTP >= 16 ? 4 : 1;
    static constexpr int kM = kNY * kTM;
};

__host__ __device__ __forceinline__ int xs_pitch(int cin) { return cin + 4; }

template <int COUTP>
static size_t conv_smem_bytes(int ntaps, int cin, bool head) {
    using S = ConvShape<COUTP>;
    const size_t w = (size_t)ntaps * cin * COUTP;
    size_t x = (size_t)S::kM * xs_pitch(cin);
    if (head && x < (size_t)S::kM * (COUTP + 1)) x = (size_t)S::kM * (COUTP + 1);
    return sizeof(float) * (w + x) + sizeof(int) * S::kM;
}

__device__ __forceinline__ float softplus_f32(float x) {  // torch.nn.functional.softplus, beta 1, threshold 20
    return x > 20.0f ? x : log1pf(expf(x));
}

// What a training forward keeps (kTrain): pre [nout, cout] when the layer has an activation; with a head, hidden
// [nout, cout] (the activated rows) and head_pre [nout]; with a tail and no head, head_pre [nout] (the value before it).
struct ConvKeep {
    float* pre;
    float* hidden;
    float* head_pre;
};

template <int COUTP, bool kTrain>
__global__ void __launch_bounds__(kConvThreads, 2) conv_gemm_kernel(dp_spconv_layer_t L, ConvKeep keep) {
    using S = ConvShape<COUTP>;
    constexpr int kTM = S::kTM, kTN = S::kTN, kM = S::kM, kNY = S::kNY;
    extern __shared__ __align__(16) float smem[];
    const int ntaps = L.ntaps, cin = L.cin, cout = L.cout, xp = xs_pitch(cin);
    float* ws = smem;                                     // [ntaps][cin][COUTP]
    float* xs = ws + (size_t)ntaps * cin * COUTP;         // [kM][xp]; in the head epilogue [kM][COUTP + 1]
    const bool head = L.head_weight != nullptr;
    int* srcs = reinterpret_cast<int*>(xs + (size_t)kM * (head && COUTP + 1 > xp ? COUTP + 1 : xp));
    const int tid = threadIdx.x, tx = tid % S::kNX, ty = tid / S::kNX;

    for (int e = tid; e < ntaps * cin * COUTP; e += kConvThreads) {
        const int co = e % COUTP, ci = (e / COUTP) % cin, t = e / (COUTP * cin);
        ws[e] = co < cout ? L.weight[((long long)co * ntaps + t) * cin + ci] : 0.0f;
    }
    const float slope = L.slope ? *L.slope : 0.0f;
    const bool vec = (cin & 3) == 0 && (reinterpret_cast<uintptr_t>(L.in) & 15) == 0;

    const long long ntiles = (L.nout + kM - 1) / kM;
    for (long long tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const long long base = tile * kM;
        float acc[kTM][kTN];
#pragma unroll
        for (int i = 0; i < kTM; ++i)
#pragma unroll
            for (int j = 0; j < kTN; ++j) acc[i][j] = 0.0f;

        for (int t = 0; t < ntaps; ++t) {
            __syncthreads();  // xs / srcs of the previous tap (or tile) are consumed
            for (int s = tid; s < kM; s += kConvThreads) {
                const long long site = base + s;
                int src = -1;
                if (site < L.nout) src = L.src ? L.src[site * ntaps + t] : (int)site;
                srcs[s] = src;
            }
            __syncthreads();
            if (vec) {
                const int c4 = cin >> 2;
                for (int e = tid; e < kM * c4; e += kConvThreads) {
                    const int s = e / c4, q = e % c4;
                    const int src = srcs[s];
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (src >= 0) v = __ldg(reinterpret_cast<const float4*>(L.in + (long long)src * cin) + q);
                    *reinterpret_cast<float4*>(xs + s * xp + 4 * q) = v;
                }
            } else {
                for (int e = tid; e < kM * cin; e += kConvThreads) {
                    const int s = e / cin, ci = e % cin;
                    const int src = srcs[s];
                    xs[s * xp + ci] = src >= 0 ? __ldg(L.in + (long long)src * cin + ci) : 0.0f;
                }
            }
            __syncthreads();

            float p[kTM][kTN];
#pragma unroll
            for (int i = 0; i < kTM; ++i)
#pragma unroll
                for (int j = 0; j < kTN; ++j) p[i][j] = 0.0f;
            const float* wt = ws + (size_t)t * cin * COUTP + tx * kTN;
#pragma unroll 4
            for (int ci = 0; ci < cin; ++ci) {
                float xv[kTM], wv[kTN];
#pragma unroll
                for (int i = 0; i < kTM; ++i) xv[i] = xs[(ty + kNY * i) * xp + ci];
                if constexpr (kTN % 4 == 0) {
#pragma unroll
                    for (int j = 0; j < kTN; j += 4) {
                        const float4 w4 = *reinterpret_cast<const float4*>(wt + ci * COUTP + j);
                        wv[j] = w4.x; wv[j + 1] = w4.y; wv[j + 2] = w4.z; wv[j + 3] = w4.w;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < kTN; ++j) wv[j] = wt[ci * COUTP + j];
                }
#pragma unroll
                for (int i = 0; i < kTM; ++i)
#pragma unroll
                    for (int j = 0; j < kTN; ++j) p[i][j] = __fmaf_rn(wv[j], xv[i], p[i][j]);
            }
#pragma unroll
            for (int i = 0; i < kTM; ++i)
                if (srcs[ty + kNY * i] >= 0)
#pragma unroll
                    for (int j = 0; j < kTN; ++j) acc[i][j] = __fadd_rn(acc[i][j], p[i][j]);
        }

        // epilogue: bias, activation
#pragma unroll
        for (int j = 0; j < kTN; ++j) {
            const int co = tx * kTN + j;
            const float bj = (L.bias && co < cout) ? L.bias[co] : 0.0f;
#pragma unroll
            for (int i = 0; i < kTM; ++i) {
                float v = acc[i][j];
                if (L.bias) v = __fadd_rn(v, bj);
                if constexpr (kTrain) {
                    const long long site = base + ty + kNY * i;
                    if (L.slope && site < L.nout && co < cout) keep.pre[site * cout + co] = v;
                }
                if (L.slope) v = v > 0.0f ? v : __fmul_rn(slope, v);
                acc[i][j] = v;
            }
        }
        if (!head && !L.indices) {
#pragma unroll
            for (int i = 0; i < kTM; ++i) {
                const long long site = base + ty + kNY * i;
                if (site >= L.nout) continue;
                float* o = L.out + site * cout;
#pragma unroll
                for (int j = 0; j < kTN; ++j)
                    if (tx * kTN + j < cout) o[tx * kTN + j] = acc[i][j];
            }
            continue;
        }
        // final 1x1 (cout -> 1) and the output tail, one thread per site
        float* hs = xs;  // [kM][COUTP + 1]
        if (head) {
            __syncthreads();  // every thread is done reading xs
#pragma unroll
            for (int i = 0; i < kTM; ++i)
#pragma unroll
                for (int j = 0; j < kTN; ++j) hs[(ty + kNY * i) * (COUTP + 1) + tx * kTN + j] = acc[i][j];
            if constexpr (kTrain) {
#pragma unroll
                for (int i = 0; i < kTM; ++i) {
                    const long long site = base + ty + kNY * i;
                    if (site >= L.nout) continue;
#pragma unroll
                    for (int j = 0; j < kTN; ++j)
                        if (tx * kTN + j < cout) keep.hidden[site * cout + tx * kTN + j] = acc[i][j];
                }
            }
            __syncthreads();
        }
        for (int s = head ? tid : (tx == 0 ? ty : kM); s < kM; s += head ? kConvThreads : kM) {
            const long long site = base + s;
            if (site >= L.nout) continue;
            float y;
            if (head) {
                y = 0.0f;
                for (int co = 0; co < cout; ++co) y = __fmaf_rn(L.head_weight[co], hs[s * (COUTP + 1) + co], y);
                if (L.head_bias) y = __fadd_rn(y, *L.head_bias);
            } else {
                y = acc[0][0];  // cout == 1 (checked), kTM == 1, thread tx 0 holds the site
            }
            if constexpr (kTrain) {
                if (keep.head_pre) keep.head_pre[site] = y;
            }
            if (L.indices) {
                const int r = L.indices[3 * site + 1], c = L.indices[3 * site + 2];
                if (r < c) y = __fmul_rn(y, 0.0f);  // by value: the site stays active (model.py tail)
                else if (r == c) y = softplus_f32(y);
            }
            L.out[site] = y;
        }
    }
}

static int grid_for_items(long long items, int threads) {
    long long b = (items + threads - 1) / threads;
    const long long cap = (long long)sm_count() * 16;
    if (b > cap) b = cap;
    return b < 1 ? 1 : (int)b;
}

template <int COUTP, bool kTrain>
static int launch_conv(const dp_spconv_layer_t& L, ConvKeep keep, cudaStream_t s) {
    using S = ConvShape<COUTP>;
    const size_t smem = conv_smem_bytes<COUTP>(L.ntaps, L.cin, L.head_weight != nullptr);
    const void* fn = reinterpret_cast<const void*>(conv_gemm_kernel<COUTP, kTrain>);
    int st = allow_dynamic_smem(fn, smem);
    if (st != DP_OK) return st;
    const long long tiles = (L.nout + S::kM - 1) / S::kM;
    const long long cap = coop_grid(fn, kConvThreads, smem);  // resident CTAs (cached per device): the grid strides
    const int grid = (int)(tiles < cap ? tiles : cap);
    conv_gemm_kernel<COUTP, kTrain><<<grid, kConvThreads, smem, s>>>(L, keep);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

static size_t sort_ws_bytes(long long rows) {
    return align_up(sizeof(int) * ((size_t)rows + 1), 256) + scan_workspace_bytes(rows + 1);
}

static bool rows_ok(int nb, int h) { return nb >= 0 && h >= 0 && (long long)nb * h < 0x7fffffffLL; }

static int layer_args(const dp_spconv_layer_t& L) {
    if (L.nout < 0 || L.nout > 0x7fffffffLL || (L.ntaps != 1 && L.ntaps != 4)) return DP_ERR_INVALID;
    if (L.cin < 1 || L.cin > kMaxChannels || L.cout < 1 || L.cout > kMaxChannels) return DP_ERR_INVALID;
    if (L.ntaps == 4 && !L.src) return DP_ERR_INVALID;                // identity sources exist for 1x1 layers only
    if (L.indices && !L.head_weight && L.cout != 1) return DP_ERR_INVALID;  // the tail acts on one channel
    return DP_OK;
}

template <bool kTrain>
static int launch_layer(const dp_spconv_layer_t& L, ConvKeep keep, cudaStream_t s) {
    const int c = L.cout;
    if (c <= 1 && !L.head_weight) return launch_conv<1, kTrain>(L, keep, s);
    if (c <= 4) return launch_conv<4, kTrain>(L, keep, s);
    if (c <= 8) return launch_conv<8, kTrain>(L, keep, s);
    if (c <= 16) return launch_conv<16, kTrain>(L, keep, s);
    if (c <= 32) return launch_conv<32, kTrain>(L, keep, s);
    return launch_conv<64, kTrain>(L, keep, s);
}

}  // namespace dp

using namespace dp;

extern "C" {

size_t dp_spconv_sort_workspace_bytes(int32_t batch_size, int32_t h) {
    return rows_ok(batch_size, h) ? sort_ws_bytes((long long)batch_size * h) : 0;
}

int dp_spconv_sort_sites(const int32_t* indices, int64_t nnz, int32_t batch_size, int32_t h, int32_t w, int32_t* rowptr,
                         int32_t* col, int32_t* perm, int32_t* flag_out, void* workspace, size_t workspace_bytes,
                         void* stream) {
    if (nnz < 0 || nnz > 0x7fffffffLL || w < 0 || !rows_ok(batch_size, h) || !rowptr || !flag_out || !workspace)
        return DP_ERR_INVALID;
    if (nnz > 0 && (!indices || !col || !perm)) return DP_ERR_INVALID;
    if (!aligned16(workspace)) return DP_ERR_ALIGNMENT;
    const long long rows = (long long)batch_size * h;
    if (workspace_bytes < sort_ws_bytes(rows)) return DP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    int* cursor = static_cast<int*>(workspace);
    void* scan_ws = static_cast<char*>(workspace) + align_up(sizeof(int) * ((size_t)rows + 1), 256);
    DP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * ((size_t)rows + 1), s));
    if (nnz > 0) {
        site_count_kernel<<<grid_for_items(nnz, 256), 256, 0, s>>>(indices, nnz, batch_size, h, w, cursor, flag_out);
        DP_LAUNCH_CHECK();
    }
    int st = exclusive_scan_i32(cursor, rowptr, rows + 1, scan_ws, s);
    if (st != DP_OK) return st;
    if (nnz > 0) {
        DP_CUDA(cudaMemsetAsync(cursor, 0, sizeof(int) * ((size_t)rows + 1), s));
        site_fill_kernel<<<grid_for_items(nnz, 256), 256, 0, s>>>(indices, nnz, batch_size, h, w, rowptr, cursor, col, perm);
        DP_LAUNCH_CHECK();
        site_sort_rows_kernel<<<grid_for_items(rows, 128), 128, 0, s>>>((int)rows, rowptr, col, perm, flag_out);
        DP_LAUNCH_CHECK();
    }
    return DP_OK;
}

static bool rules_args_ok(int32_t nb, int32_t h, int32_t w, int32_t ph, int32_t pw) {
    if (!((ph == 1 && pw == 0) || (ph == 0 && pw == 1))) return false;
    if (w < 0 || !rows_ok(nb, h)) return false;
    const long long ho = (long long)h + 2 * ph - 1, wo = (long long)w + 2 * pw - 1;
    return ho >= 0 && wo >= 0 && (long long)nb * ho < 0x7fffffffLL;
}

size_t dp_spconv_rules_workspace_bytes(int32_t batch_size, int32_t h, int32_t ph) {
    const long long ho = (long long)h + 2 * ph - 1;
    return (batch_size >= 0 && ho >= 0) ? scan_workspace_bytes((long long)batch_size * ho + 1) : 0;
}

int dp_spconv_rules_count(const int32_t* rowptr_in, const int32_t* col_in, int32_t batch_size, int32_t h, int32_t w,
                          int32_t ph, int32_t pw, int32_t* rowptr_out, void* workspace, size_t workspace_bytes,
                          void* stream) {
    if (!rules_args_ok(batch_size, h, w, ph, pw) || !rowptr_in || !rowptr_out || !workspace) return DP_ERR_INVALID;
    if (!aligned16(workspace)) return DP_ERR_ALIGNMENT;
    const int ho = h + 2 * ph - 1, wo = w + 2 * pw - 1;
    const long long rows_out = (long long)batch_size * ho;
    if (workspace_bytes < scan_workspace_bytes(rows_out + 1)) return DP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    DP_CUDA(cudaMemsetAsync(rowptr_out + rows_out, 0, sizeof(int), s));
    if (rows_out > 0) {
        rules_count_kernel<<<grid_for_items(rows_out, 128), 128, 0, s>>>((int)rows_out, ho, rowptr_in, col_in, h, ph, pw,
                                                                          wo, rowptr_out);
        DP_LAUNCH_CHECK();
    }
    return exclusive_scan_i32(rowptr_out, rowptr_out, rows_out + 1, workspace, s);
}

int dp_spconv_rules_fill(const int32_t* rowptr_in, const int32_t* col_in, const int32_t* perm, int32_t batch_size,
                         int32_t h, int32_t w, int32_t ph, int32_t pw, const int32_t* rowptr_out, int32_t* col_out,
                         int32_t* rules, int32_t* indices_out, void* stream) {
    if (!rules_args_ok(batch_size, h, w, ph, pw) || !rowptr_in || !rowptr_out) return DP_ERR_INVALID;
    if (!aligned16(rules)) return DP_ERR_ALIGNMENT;
    const int ho = h + 2 * ph - 1, wo = w + 2 * pw - 1;
    const long long rows_out = (long long)batch_size * ho;
    if (rows_out > 0) {
        rules_fill_kernel<<<grid_for_items(rows_out, 128), 128, 0, (cudaStream_t)stream>>>(
            (int)rows_out, ho, rowptr_in, col_in, perm, h, ph, pw, wo, rowptr_out, col_out, rules, indices_out);
        DP_LAUNCH_CHECK();
    }
    return DP_OK;
}

int dp_spconv_layer_f32(const dp_spconv_layer_t* layer_host, void* stream) {
    if (!layer_host) return DP_ERR_INVALID;
    const dp_spconv_layer_t& L = *layer_host;
    int st = layer_args(L);
    if (st != DP_OK) return st;
    if (L.nout == 0) return DP_OK;
    if (!L.in || !L.weight || !L.out) return DP_ERR_INVALID;
    return launch_layer<false>(L, ConvKeep{nullptr, nullptr, nullptr}, (cudaStream_t)stream);
}

int dp_spconv_layer_train_f32(const dp_spconv_layer_t* layer_host, float* pre, float* hidden, float* head_pre,
                              void* stream) {
    if (!layer_host) return DP_ERR_INVALID;
    const dp_spconv_layer_t& L = *layer_host;
    int st = layer_args(L);
    if (st != DP_OK) return st;
    const bool head = L.head_weight != nullptr;
    if (L.nout == 0) return DP_OK;
    if (!L.in || !L.weight || !L.out) return DP_ERR_INVALID;
    if ((L.slope && !pre) || (head && (!hidden || !head_pre)) || (L.indices && !head_pre)) return DP_ERR_INVALID;
    return launch_layer<true>(L, ConvKeep{pre, head ? hidden : nullptr, (head || L.indices) ? head_pre : nullptr},
                              (cudaStream_t)stream);
}

}  // extern "C"
