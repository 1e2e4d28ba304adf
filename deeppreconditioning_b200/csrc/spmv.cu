// spmv.cu — library plumbing + standalone K2 entry points (dp_spmv_csr_f64, dp_coo_spmv_batch_f32).
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <vector>

#include "tilepipe.cuh"

namespace dp {

static thread_local char g_cuda_error[256] = "";

const char* set_cuda_error(cudaError_t e) {
    snprintf(g_cuda_error, sizeof(g_cuda_error), "%s: %s", cudaGetErrorName(e), cudaGetErrorString(e));
    return g_cuda_error;
}

// Persistent CTAs, one contiguous range of 512-row tiles each, streamed through the tile pipeline (tilepipe.cuh).
constexpr int kSpmvRound = 32;  // tile descriptors per table refill
#ifndef DPCG_SPMV_UNROLL
#define DPCG_SPMV_UNROLL 8
#endif

struct SpmvSmem {
    PipeShared pipe;
    TileDesc tab[kSpmvRound];
};

template <bool kPacked>
__global__ void __launch_bounds__(kBlock, 2)
spmv_csr_kernel(CsrView A, const double* __restrict__ x, double* __restrict__ y) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SpmvSmem& sm = *reinterpret_cast<SpmvSmem*>(smem_raw);
    typename std::conditional<kPacked, PipePacked, Pipe>::type pipe;
    pipe.init(sm.pipe.bytes, &sm.pipe.bar);
    const int ntiles = (A.n + kTileRows - 1) / kTileRows;
    const int quot = ntiles / (int)gridDim.x, rem = ntiles % (int)gridDim.x;  // ranges differ by at most one tile
    const int g0 = (int)blockIdx.x * quot + min((int)blockIdx.x, rem), g1 = g0 + quot + ((int)blockIdx.x < rem ? 1 : 0);
    const GatherReadOnly gx{x};
    for (int ga = g0; ga < g1; ga += kSpmvRound) {
        const int cnt = min(kSpmvRound, g1 - ga);
        __syncthreads();  // the previous round's table is no longer read
        for (int i = threadIdx.x; i < cnt; i += kBlock) {
            TileDesc d;
            tile_desc_fill<kPacked>(d, A, ga + i);
            d.sys = 0;
            sm.tab[i] = d;
        }
        __syncthreads();
        pipe.begin(sm.tab, cnt);
        int rs_n, re_n;
        tile_row_extent(sm.tab[0], rs_n, re_n);
        for (int i = 0; i < cnt; ++i) {
            const TileDesc& d = sm.tab[i];
            const int rs = rs_n, re = re_n;
            if (i + 1 < cnt) tile_row_extent(sm.tab[i + 1], rs_n, re_n);  // one tile ahead
            const double s = pipe.template tile_spmv<DPCG_SPMV_UNROLL>(d, rs, re, gx, true);
            const int row = d.ltile * kTileRows + (int)threadIdx.x;
            if (row < A.n) y[row] = s;
        }
    }
}

// dp_csr_pack: one CTA per 512-row tile. Pass 1 finds the tile's column range, pass 2 writes the 6-byte entries and checks
// that nothing was lost (values bit for bit through fp32, columns within 16 bits of the tile's smallest).
__global__ void __launch_bounds__(kBlock)
csr_pack_kernel(int n, const int* __restrict__ rowptr, const int* __restrict__ col, const double* __restrict__ val,
                unsigned short* __restrict__ col16, float* __restrict__ val32, int* __restrict__ tile_base,
                int* __restrict__ status) {
    __shared__ int s_lo[kWarpsPerBlock], s_hi[kWarpsPerBlock];
    const int tile = blockIdx.x;
    const int cs = __ldg(rowptr + min(tile * kTileRows, n)), ce = __ldg(rowptr + min((tile + 1) * kTileRows, n));
    int lo = 0x7fffffff, hi = -1;
    for (int q = cs + (int)threadIdx.x; q < ce; q += kBlock) {
        const int c = __ldg(col + q);
        lo = min(lo, c), hi = max(hi, c);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(kFull, lo, o));
        hi = max(hi, __shfl_xor_sync(kFull, hi, o));
    }
    if ((threadIdx.x & 31) == 0) s_lo[threadIdx.x >> 5] = lo, s_hi[threadIdx.x >> 5] = hi;
    __syncthreads();
    lo = s_lo[0], hi = s_hi[0];
#pragma unroll
    for (int w = 1; w < kWarpsPerBlock; ++w) lo = min(lo, s_lo[w]), hi = max(hi, s_hi[w]);
    if (ce == cs) lo = 0, hi = 0;
    int bad = (hi - lo > 65535 || lo < 0) ? 2 : 0;
    if (threadIdx.x == 0) tile_base[2 * tile] = lo, tile_base[2 * tile + 1] = ce > cs ? hi - lo + 1 : 0;
    for (int q = cs + (int)threadIdx.x; q < ce; q += kBlock) {
        const double v = val[q];
        const float f = (float)v;
        if (as_bits((double)f) != as_bits(v)) bad |= 1;
        val32[q] = f;
        col16[q] = (unsigned short)(__ldg(col + q) - lo);
    }
    if (bad) atomicOr(status, bad);
}

// utils.py:15-43 — batched COO SpMV in fp32. Accumulation order is unspecified in the reference
// (scatter_reduce("sum")) and here (atomicAdd).
__global__ void coo_spmv_batch_kernel(const int* __restrict__ ind, const float* __restrict__ feat, long long nnz,
                                      int nbatch, int n, const float* __restrict__ vec, int transpose,
                                      float* __restrict__ out) {
    for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < nnz;
         e += (long long)gridDim.x * blockDim.x) {
        const int b = ind[3 * e], r = ind[3 * e + (transpose ? 2 : 1)], c = ind[3 * e + (transpose ? 1 : 2)];
        if ((unsigned)b < (unsigned)nbatch && (unsigned)r < (unsigned)n && (unsigned)c < (unsigned)n)
            atomicAdd(out + (size_t)b * n + r, feat[e] * vec[(size_t)b * n + c]);
    }
}

namespace {
constexpr int kMaxDevices = 64;
struct KernelEntry {
    int device;
    const void* kernel;
    size_t smem;     // dynamic shared memory the kernel has been opted into on that device
    int threads;     // occupancy query the cached grid belongs to (0: none yet)
    size_t occ_smem;
    int grid;
};
std::mutex g_cache_mutex;
std::vector<KernelEntry> g_kernels;
int g_sm_count[kMaxDevices];

int current_device() {
    int dev = 0;
    return cudaGetDevice(&dev) == cudaSuccess ? dev : 0;
}
KernelEntry& kernel_entry(int dev, const void* kernel) {  // caller holds g_cache_mutex
    for (KernelEntry& e : g_kernels)
        if (e.device == dev && e.kernel == kernel) return e;
    g_kernels.push_back(KernelEntry{dev, kernel, 0, 0, 0, 0});
    return g_kernels.back();
}
}  // namespace

int pipe_trace_read_spmv(uint64_t* out_host, int capacity) {
#ifdef DPCG_PIPE_TRACE
    const int cap = capacity < kPipeTraceCap ? capacity : kPipeTraceCap;
    for (int w = 0; w < 2; ++w)
        DP_CUDA(cudaMemcpyFromSymbol(out_host + (size_t)w * capacity, g_pipe_trace, sizeof(unsigned long long) * (size_t)cap,
                                     sizeof(unsigned long long) * (size_t)w * kPipeTraceCap, cudaMemcpyDeviceToHost));
    return DP_OK;
#else
    (void)out_host, (void)capacity;
    return DP_ERR_INVALID;
#endif
}

int sm_count() {
    const int dev = current_device();
    const bool cacheable = dev >= 0 && dev < kMaxDevices;
    if (cacheable && g_sm_count[dev]) return g_sm_count[dev];
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) return 148;
    if (cacheable) g_sm_count[dev] = sms;
    return sms;
}

int allow_dynamic_smem(const void* kernel, size_t bytes) {
    const int dev = current_device();
    std::lock_guard<std::mutex> lock(g_cache_mutex);
    KernelEntry& e = kernel_entry(dev, kernel);
    if (e.smem >= bytes && e.smem > 0) return DP_OK;
    DP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    if (const char* c = getenv("DPCG_CARVEOUT"))  // experiments: shared-memory share of the L1 / shared-memory array, percent
        DP_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, atoi(c)));
    e.smem = bytes;
    e.threads = 0;  // occupancy depends on the attribute
    return DP_OK;
}

int coop_grid(const void* kernel, int threads, size_t smem) {
    const int dev = current_device();
    std::lock_guard<std::mutex> lock(g_cache_mutex);
    KernelEntry& e = kernel_entry(dev, kernel);
    if (e.threads == threads && e.occ_smem == smem && e.grid > 0) return e.grid;
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) sms = 148;
    e.threads = threads, e.occ_smem = smem, e.grid = per_sm * sms;
    return e.grid;
}

}  // namespace dp

using namespace dp;

extern "C" {

int dp_version(void) { return DP_VERSION; }

const char* dp_status_string(int status) {
    switch (status) {
        case DP_OK: return "ok";
        case DP_ERR_INVALID: return "invalid argument";
        case DP_ERR_ALIGNMENT: return "array not 16-byte aligned";
        case DP_ERR_WORKSPACE: return "workspace too small";
        case DP_ERR_CUDA: return "CUDA runtime error";
        case DP_ERR_STRUCTURE: return "matrix structure violates the contract";
        case DP_ERR_TIMEOUT: return "dependency spin timed out";
        case DP_ERR_NOT_SPD: return "matrix is not symmetric positive definite (non-positive pivot)";
        default: return "unknown status";
    }
}

const char* dp_last_cuda_error(void) { return g_cuda_error; }

int dp_spmv_csr_f64(int32_t n, int32_t nnz, const int32_t* rowptr, const int32_t* col, const double* val,
                    const double* x, double* y, void* stream) {
    if (n < 0 || nnz < 0 || !rowptr || !y || (nnz > 0 && (!col || !val || !x))) return DP_ERR_INVALID;
    if (!aligned16(col) || !aligned16(val)) return DP_ERR_ALIGNMENT;
    if (n == 0) return DP_OK;
    if (allow_dynamic_smem((const void*)spmv_csr_kernel<false>, sizeof(SpmvSmem)) != DP_OK) return DP_ERR_CUDA;
    const int tiles = (n + kTileRows - 1) / kTileRows;
    const int resident = 2 * sm_count();
    const int grid = tiles < resident ? tiles : resident;
    CsrView A{rowptr, col, val, n, nnz};
    spmv_csr_kernel<false><<<grid, kBlock, sizeof(SpmvSmem), (cudaStream_t)stream>>>(A, x, y);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

int32_t dp_csr_pack_tile_rows(void) { return kTileRows; }

int dp_csr_pack(int32_t n, int32_t nnz, const int32_t* rowptr, const int32_t* col, const double* val, uint16_t* col16,
                float* val32, int32_t* tile_base, int32_t* status_out, void* stream) {
    if (n < 0 || nnz < 0 || !rowptr || !tile_base || !status_out || (nnz > 0 && (!col || !val || !col16 || !val32)))
        return DP_ERR_INVALID;
    if (!aligned16(col16) || !aligned16(val32)) return DP_ERR_ALIGNMENT;
    if (n == 0) return DP_OK;
    const int tiles = (n + kTileRows - 1) / kTileRows;
    csr_pack_kernel<<<tiles, kBlock, 0, (cudaStream_t)stream>>>(n, rowptr, col, val, col16, val32, tile_base, status_out);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

int dp_spmv_csr_packed_f64(int32_t n, int32_t nnz, const int32_t* rowptr, const uint16_t* col16, const float* val32,
                           const int32_t* tile_base, const double* x, double* y, void* stream) {
    if (n < 0 || nnz < 0 || !rowptr || !y || !tile_base || (nnz > 0 && (!col16 || !val32 || !x))) return DP_ERR_INVALID;
    if (!aligned16(col16) || !aligned16(val32)) return DP_ERR_ALIGNMENT;
    if (n == 0) return DP_OK;
    if (allow_dynamic_smem((const void*)spmv_csr_kernel<true>, sizeof(SpmvSmem)) != DP_OK) return DP_ERR_CUDA;
    const int tiles = (n + kTileRows - 1) / kTileRows;
    const int resident = 2 * sm_count();
    const int grid = tiles < resident ? tiles : resident;
    CsrView A{rowptr, nullptr, nullptr, n, nnz, col16, val32, tile_base};
    spmv_csr_kernel<true><<<grid, kBlock, sizeof(SpmvSmem), (cudaStream_t)stream>>>(A, x, y);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

int dp_coo_spmv_batch_f32(const int32_t* indices, const float* features, int64_t nnz, int32_t nbatch, int32_t n,
                          const float* vec, int32_t transpose, float* out, void* stream) {
    if (nnz < 0 || nbatch < 0 || n < 0 || !out || (nnz > 0 && (!indices || !features || !vec))) return DP_ERR_INVALID;
    cudaStream_t s = (cudaStream_t)stream;
    DP_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)nbatch * (size_t)n, s));
    if (nnz == 0) return DP_OK;
    long long blocks = (nnz + 255) / 256;
    if (blocks > sm_count() * 32) blocks = sm_count() * 32;
    coo_spmv_batch_kernel<<<(int)blocks, 256, 0, s>>>(indices, features, nnz, nbatch, n, vec, transpose, out);
    DP_LAUNCH_CHECK();
    return DP_OK;
}

}  // extern "C"
