// sparseconv_grad.cu — backward of the factor network's sparse-convolution layers (training on the device).
//
// For a layer y = act(z), z[s, co] = bias[co] + sum_t sum_ci W[co, t, ci] x[src_t(s), ci] (sparseconv.cu), given the
// upstream gradient g_y and the values the training forward kept (pre = z):
//   g_z[s, co]    = g_y[s, co] * act'(pre[s, co])       act' = 1 (pre > 0), slope (pre <= 0): torch.prelu's backward
//   dW[co, t, ci] = sum_s g_z[s, co] x[src_t(s), ci]     (inactive taps contribute nothing)
//   db[co]        = sum_s g_z[s, co]
//   dslope        = sum_{s, co: pre <= 0} g_y[s, co] pre[s, co]
//   dX            = the same layer run on g_z with W'[ci, t, co] = W[co, t, ci] and the inverted rules (no bias, no
//                   activation): dp_spconv_layer_f32 as it stands, so dX has the forward's fixed order and bound.
// The head (the final 1x1, ntaps 1, cout 1) uses the output tail in place of the activation, with u = head_pre:
//   g_u = g * 0 (row < col), u > 20 ? g : g e / (e + 1) with e = exp(u) (row == col, softplus's backward), g elsewhere.
//
// Determinism without floating-point atomics: the output sites are cut into fixed chunks of kWgradChunk = 1024 sites
// (a constant, not derived from the grid). For a chunk, every dW / db / dslope(co) entry is one fma (add) chain over the
// chunk's sites in ascending order starting from 0, written to the workspace; a second launch adds the chunk partials in
// chunk order in fp64 and rounds once. The results do not depend on the grid or the SM count, and a chunk partial of n
// terms is within n u sum|terms| (u = 2^-24) of exact, so
//   |dW - dW_exact| <= (C + 2) u sum|terms|,  C = kWgradChunk        (same bound for db and dslope)
// (the fp64 sum of at most 2^21 chunk partials adds < 2^-32 sum|terms|, the final rounding u |dW|).
// Workspace: ceil(nout / C) chunk rows of cout (ntaps cin + 2) floats. At 8 systems of 316^2 (bench.py's CNN batch,
// PreconditionerNet, site counts of tools/inference_bench.py::work_counts) the widest layers have 8,772,040 (32 -> 64)
// and 11,962,336 (64 -> 32) output sites: 8,567 chunks of 8,320 floats (285 MB) and 11,682 chunks of 8,256 floats
// (386 MB), about a sixth of the 2.25 GB the 64 -> 32 layer's input features take.
#include "common.cuh"

namespace dp {

constexpr int kWgradChunk = 1024;  // sites per chunk partial
constexpr int kWgradThreads = 256;
constexpr int kWgradSub = 32;      // sites staged in shared memory at a time (16 for the 64 x 256 tile: 48 KB)
constexpr int kWgradNX = 32;       // threads along k = t cin + ci (kWgradThreads / kWgradNX along co)
constexpr int kWgradNY = kWgradThreads / kWgradNX;
constexpr int kMaxGradChannels = 64;

__device__ __forceinline__ float tail_grad(float g, float u, int row, int col) {
    if (row < col) return __fmul_rn(g, 0.0f);
    if (row > col) return g;
    if (u > 20.0f) return g;
    const float e = expf(u);
    return __fdiv_rn(__fmul_rn(g, e), __fadd_rn(e, 1.0f));
}

__host__ __device__ __forceinline__ long long chunk_row(int cout, int k) { return (long long)cout * (k + 2); }

// A CTA takes whole chunks (grid-strided). Per sub-tile of SUB sites: (1) every thread stages the tap sources,
// the upstream gradient and pre into shared memory (the tail's g_u is formed here: it has no chain); (2) threads
// tid < 8 TM form g_z of channel tid from shared memory, carrying the db / dslope chains across the chunk, while the
// others gather the input rows of every tap into xs[site][k = t cin + ci]; (3) thread (ty, tx) adds the sub-tile to its
// register tile dW[co = ty + 8 i][k = tx + 32 j]. Columns beyond cout / K are zero in shared memory, so the inner loop
// has no branches.
template <int TM, int TN>
__global__ void __launch_bounds__(kWgradThreads, 2) wgrad_chunk_kernel(dp_spconv_grad_t G, float* __restrict__ part) {
    constexpr int GP = kWgradNY * TM, KP = kWgradNX * TN, SUB = TM * TN >= 64 ? kWgradSub / 2 : kWgradSub;
    __shared__ __align__(16) float gs[SUB][GP];  // g_y, then g_z
    __shared__ __align__(16) float ps[SUB][GP];  // pre (with an activation)
    __shared__ __align__(16) float xs[SUB][KP];
    __shared__ int srcs[SUB][4];
    const int ntaps = G.ntaps, cin = G.cin, cout = G.cout, K = ntaps * cin;
    const int tid = threadIdx.x, tx = tid % kWgradNX, ty = tid / kWgradNX;
    const float slope = G.slope ? *G.slope : 0.0f;
    const long long nchunks = (G.nout + kWgradChunk - 1) / kWgradChunk;
    const bool vec = (cin & 3) == 0 && (reinterpret_cast<uintptr_t>(G.in) & 15) == 0;

    for (long long chunk = blockIdx.x; chunk < nchunks; chunk += gridDim.x) {
        const long long c0 = chunk * kWgradChunk;
        const long long c1 = min(c0 + kWgradChunk, (long long)G.nout);
        float acc[TM][TN];
#pragma unroll
        for (int i = 0; i < TM; ++i)
#pragma unroll
            for (int j = 0; j < TN; ++j) acc[i][j] = 0.0f;
        float db = 0.0f, dsl = 0.0f;  // threads tid < cout: channel tid

        for (long long b0 = c0; b0 < c1; b0 += SUB) {
            const int ns = (int)min((long long)SUB, c1 - b0);
            __syncthreads();  // the previous sub-tile is consumed
            for (int e = tid; e < SUB * 4; e += kWgradThreads) {
                const int s = e >> 2, t = e & 3;
                int src = -1;
                if (s < ns && t < ntaps) src = G.src ? G.src[(b0 + s) * ntaps + t] : (int)(b0 + s);
                srcs[s][t] = src;
            }
            for (int e = tid; e < SUB * GP; e += kWgradThreads) {
                const int s = e / GP, co = e % GP;
                float g = 0.0f, z = 0.0f;
                if (s < ns && co < cout) {
                    const long long site = b0 + s;
                    g = G.grad_out[site * cout + co];
                    if (G.tail_indices)
                        g = tail_grad(g, G.pre[site], G.tail_indices[3 * site + 1], G.tail_indices[3 * site + 2]);
                    else if (G.slope)
                        z = G.pre[site * cout + co];
                }
                gs[s][co] = g;
                ps[s][co] = z;
            }
            __syncthreads();
            if (tid < GP) {
                const int co = tid;
                for (int s = 0; s < ns; ++s) {
                    const float g = gs[s][co];
                    float gz = g;
                    if (G.slope) {
                        const float z = ps[s][co];
                        if (!(z > 0.0f)) {
                            gz = __fmul_rn(slope, g);
                            dsl = __fmaf_rn(g, z, dsl);
                        }
                    }
                    if (co < cout) {
                        db = __fadd_rn(db, gz);
                        G.grad_pre[(b0 + s) * cout + co] = gz;
                    }
                    gs[s][co] = gz;
                }
            } else if (vec) {
                constexpr int Q = KP / 4;
#pragma unroll 4
                for (int e = tid - GP; e < SUB * Q; e += kWgradThreads - GP) {
                    const int s = e / Q, k = 4 * (e % Q);
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (k < K) {
                        const int t = k / cin;
                        const int src = srcs[s][t];
                        if (src >= 0) v = __ldg(reinterpret_cast<const float4*>(G.in + (long long)src * cin + k - t * cin));
                    }
                    *reinterpret_cast<float4*>(&xs[s][k]) = v;
                }
            } else {
#pragma unroll 4
                for (int e = tid - GP; e < SUB * KP; e += kWgradThreads - GP) {
                    const int s = e / KP, k = e % KP;
                    float v = 0.0f;
                    if (k < K) {
                        const int t = k / cin;
                        const int src = srcs[s][t];
                        if (src >= 0) v = __ldg(G.in + (long long)src * cin + k - t * cin);
                    }
                    xs[s][k] = v;
                }
            }
            __syncthreads();
#pragma unroll 4
            for (int s = 0; s < ns; ++s) {
                float gv[TM], xv[TN];
#pragma unroll
                for (int i = 0; i < TM; ++i) gv[i] = gs[s][ty + kWgradNY * i];
#pragma unroll
                for (int j = 0; j < TN; ++j) xv[j] = xs[s][tx + kWgradNX * j];
#pragma unroll
                for (int i = 0; i < TM; ++i)
#pragma unroll
                    for (int j = 0; j < TN; ++j) acc[i][j] = __fmaf_rn(gv[i], xv[j], acc[i][j]);
            }
        }
        float* row = part + chunk * chunk_row(cout, K);
#pragma unroll
        for (int i = 0; i < TM; ++i) {
            const int co = ty + kWgradNY * i;
#pragma unroll
            for (int j = 0; j < TN; ++j) {
                const int k = tx + kWgradNX * j;
                if (co < cout && k < K) row[(long long)co * K + k] = acc[i][j];
            }
        }
        if (tid < cout) {
            row[(long long)cout * K + tid] = db;
            row[(long long)cout * K + cout + tid] = dsl;
        }
    }
}

// Column sums of the chunk partials in chunk order, fp64, rounded once: dW [cout, ntaps, cin] and db, then (block 0)
// dslope = the per-channel sums added in channel order.
__global__ void wgrad_finish_kernel(const float* __restrict__ part, long long nchunks, int cout, int K,
                                    float* __restrict__ grad_weight, float* __restrict__ grad_bias,
                                    float* __restrict__ grad_slope) {
    const long long width = chunk_row(cout, K), nw = (long long)cout * K;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nw + cout; e += (long long)gridDim.x * blockDim.x) {
        if (e >= nw && !grad_bias) break;
        double sum = 0.0;
#pragma unroll 8
        for (long long c = 0; c < nchunks; ++c) sum += (double)part[c * width + e];
        if (e < nw) grad_weight[e] = (float)sum;
        else grad_bias[e - nw] = (float)sum;
    }
    if (blockIdx.x != 0 || !grad_slope) return;
    __shared__ double per_channel[kMaxGradChannels];
    if (threadIdx.x < cout) {
        double sum = 0.0;
        for (long long c = 0; c < nchunks; ++c) sum += (double)part[c * width + nw + cout + threadIdx.x];
        per_channel[threadIdx.x] = sum;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double sum = 0.0;
        for (int co = 0; co < cout; ++co) sum += per_channel[co];
        *grad_slope = (float)sum;
    }
}

template <int TM, int TN>
static int launch_wgrad(const dp_spconv_grad_t& G, float* part, long long nchunks, cudaStream_t s) {
    const void* fn = reinterpret_cast<const void*>(wgrad_chunk_kernel<TM, TN>);
    const long long cap = coop_grid(fn, kWgradThreads, 0);  // resident CTAs: the grid strides over the chunks
    const int grid = (int)(nchunks < cap ? nchunks : cap);
    wgrad_chunk_kernel<TM, TN><<<grid, kWgradThreads, 0, s>>>(G, part);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

template <int TM>
static int launch_wgrad_k(const dp_spconv_grad_t& G, float* part, long long nchunks, cudaStream_t s) {
    const int K = G.ntaps * G.cin;
    if (K <= kWgradNX) return launch_wgrad<TM, 1>(G, part, nchunks, s);
    if (K <= 2 * kWgradNX) return launch_wgrad<TM, 2>(G, part, nchunks, s);
    if (K <= 4 * kWgradNX) return launch_wgrad<TM, 4>(G, part, nchunks, s);
    return launch_wgrad<TM, 8>(G, part, nchunks, s);
}

static long long wgrad_chunks(long long nout) { return (nout + kWgradChunk - 1) / kWgradChunk; }

static size_t wgrad_ws_bytes(long long nout, int ntaps, int cin, int cout) {
    return align_up(sizeof(float) * (size_t)wgrad_chunks(nout) * (size_t)chunk_row(cout, ntaps * cin), 256);
}

static bool shape_ok(long long nout, int ntaps, int cin, int cout) {
    return nout >= 0 && nout <= 0x7fffffffLL && (ntaps == 1 || ntaps == 4) && cin >= 1 && cin <= kMaxGradChannels &&
           cout >= 1 && cout <= kMaxGradChannels;
}

__global__ void rules_invert_kernel(const int* __restrict__ rules, long long nout, int ntaps, long long nin,
                                    int* __restrict__ inv, int* __restrict__ flag) {
    const long long n = nout * ntaps;
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n; e += (long long)gridDim.x * blockDim.x) {
        const int src = rules[e];
        if (src < 0) continue;
        const int t = (int)(e % ntaps);
        const int s = (int)(e / ntaps);
        if (src >= nin || atomicCAS(inv + (long long)src * ntaps + t, -1, s) != -1) atomicCAS(flag, 0, (int)DP_ERR_STRUCTURE);
    }
}

}  // namespace dp

using namespace dp;

extern "C" {

int32_t dp_spconv_wgrad_chunk_sites(void) { return kWgradChunk; }

size_t dp_spconv_wgrad_workspace_bytes(int64_t nout, int32_t ntaps, int32_t cin, int32_t cout) {
    return shape_ok(nout, ntaps, cin, cout) ? wgrad_ws_bytes(nout, ntaps, cin, cout) : 0;
}

int dp_spconv_rules_invert(const int32_t* rules, int64_t nout, int32_t ntaps, int64_t nin, int32_t* inv,
                           int32_t* flag_out, void* stream) {
    if (nout < 0 || nout > 0x7fffffffLL || nin < 0 || nin > 0x7fffffffLL || (ntaps != 1 && ntaps != 4))
        return DP_ERR_INVALID;
    if ((nout > 0 && (!rules || !flag_out)) || (nin > 0 && !inv)) return DP_ERR_INVALID;
    if (nin == 0 && nout == 0) return DP_OK;
    cudaStream_t s = (cudaStream_t)stream;
    if (nin > 0) DP_CUDA(cudaMemsetAsync(inv, 0xff, sizeof(int32_t) * (size_t)nin * ntaps, s));  // -1 everywhere
    const long long n = nout * ntaps;
    if (n > 0) {
        long long blocks = (n + 255) / 256;
        const long long cap = (long long)sm_count() * 16;
        rules_invert_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, s>>>(rules, nout, ntaps, nin, inv, flag_out);
        DP_LAUNCH_CHECK();
    }
    return DP_OK;
}

int dp_spconv_wgrad_f32(const dp_spconv_grad_t* grad_host, void* workspace, size_t workspace_bytes, void* stream) {
    if (!grad_host) return DP_ERR_INVALID;
    const dp_spconv_grad_t& G = *grad_host;
    if (!shape_ok(G.nout, G.ntaps, G.cin, G.cout)) return DP_ERR_INVALID;
    if (G.ntaps == 4 && !G.src) return DP_ERR_INVALID;  // identity sources exist for 1x1 layers only
    if (G.tail_indices && (G.cout != 1 || G.slope)) return DP_ERR_INVALID;  // the tail acts on one channel, alone
    if ((G.slope || G.tail_indices) && !G.pre) return DP_ERR_INVALID;
    if (G.grad_slope && !G.slope) return DP_ERR_INVALID;
    if (G.nout == 0) return DP_OK;
    if (!G.in || !G.grad_out || !G.grad_pre || !G.grad_weight || !workspace) return DP_ERR_INVALID;
    if (!aligned16(workspace)) return DP_ERR_ALIGNMENT;
    if (workspace_bytes < wgrad_ws_bytes(G.nout, G.ntaps, G.cin, G.cout)) return DP_ERR_WORKSPACE;
    cudaStream_t s = (cudaStream_t)stream;
    float* part = static_cast<float*>(workspace);
    const long long nchunks = wgrad_chunks(G.nout);
    int st;
    if (G.cout <= kWgradNY) st = launch_wgrad_k<1>(G, part, nchunks, s);
    else if (G.cout <= 2 * kWgradNY) st = launch_wgrad_k<2>(G, part, nchunks, s);
    else if (G.cout <= 4 * kWgradNY) st = launch_wgrad_k<4>(G, part, nchunks, s);
    else st = launch_wgrad_k<8>(G, part, nchunks, s);
    if (st != DP_OK) return st;
    const int K = G.ntaps * G.cin;
    const long long cols = (long long)G.cout * K + G.cout;
    const long long blocks = (cols + 255) / 256;
    wgrad_finish_kernel<<<(int)blocks, 256, 0, s>>>(part, nchunks, G.cout, K, G.grad_weight, G.grad_bias, G.grad_slope);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

}  // extern "C"
