// compress_b200/csrc/b2c_api.cu -- C ABI (include/b2c.h) over the sm_100a kernels.
// Plain CUDA runtime: no torch types cross this boundary.  No CPU fallback: without a device
// every call fails with B2C_ERR_NO_DEVICE.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <deque>
#include <chrono>
#include <atomic>
#include "../../include/b2c.h"
#include "b2c_zstd_enc.cuh"
#include "b2c_lz.cuh"
#include "b2c_frame.cuh"
#include "b2c_zstd_dec.cuh"
#include "b2c_zstd_dec_staged.cuh"
#include "b2c_s2_dec.cuh"
#include "b2c_s2_stream.cuh"
#include "b2c_huf0.cuh"

#ifndef TABLES_CTAS_PER_SM
#define TABLES_CTAS_PER_SM 8   // K2: resident CTAs per SM (19 KB static shared memory, 56 registers x 128 threads each)
#endif

using namespace b2c;

struct b2c_ctx {
    int device = 0;
    int sm_count = 0;
    size_t max_chunks = 0;
    uint8_t *d_scratch = nullptr;       // per-CTA parse scratch (two sets: one per pipeline slot)
    size_t scratch_slot = 0;            // bytes of one set
    ChunkWork *d_work[2] = {nullptr, nullptr};   // per-chunk work records, grown on demand
    uint8_t *d_pool[2] = {nullptr, nullptr};     // per-chunk work pool slabs (literals, sequences, codes, state bits)
    size_t work_cap[2] = {0, 0};        // chunks the records hold
    size_t pool_cap[2] = {0, 0};        // bytes
    cudaEvent_t ev_busy = nullptr;      // last launch that used the context's scratch / work buffers
    cudaStream_t busy_stream = nullptr; bool busy_valid = false;
    // host-buffer path staging (slot 0 of the pipeline doubles as the pointer-table path's buffers)
    uint8_t *h_in = nullptr;            // pinned, max_chunks * 64 KiB
    uint8_t *h_out = nullptr;           // pinned, max_chunks * slot
    int64_t *h_sizes = nullptr;         // pinned
    uint8_t *d_in = nullptr;
    uint8_t *d_out = nullptr;           // slots
    uint8_t *d_packed = nullptr;        // packed output
    int64_t *d_sizes = nullptr;
    uint64_t *d_offsets = nullptr;
    uint32_t *d_src_sizes = nullptr;
    uint32_t *h_src_sizes = nullptr;
    cudaStream_t stream = nullptr;
    // second pipeline slot for b2c_zstd_encode_packed (H2D / encode / D2H overlap)
    uint8_t *d_in2 = nullptr, *d_out2 = nullptr, *d_packed2 = nullptr;
    int64_t *d_sizes2 = nullptr, *h_sizes2 = nullptr;
    uint64_t *d_offsets2 = nullptr;
    uint32_t *d_src_sizes2 = nullptr, *h_src_sizes2 = nullptr;
    cudaStream_t stream2 = nullptr;
    cudaStream_t stream3 = nullptr;
    cudaStream_t dec_aux = nullptr;                        // staged decode: the literal kernel runs beside the sequence walk
    uint8_t *d_fr = nullptr; size_t fr_cap = 0;            // frame mode: block / frame tables, block slots (grown on demand)
    uint8_t *d_fr_io = nullptr; size_t fr_io_cap = 0;      // frame mode, host-buffer call: staged input | packed output | results
    uint8_t *d_s2d = nullptr; size_t s2d_cap = 0;          // staged S2 block decode: block heads + element records
    uint8_t *d_s2s = nullptr; size_t s2s_cap = 0;          // S2 stream calls: block slots, sizes, checksums, scan, tables (grown on demand)
    uint8_t *d_s2s_io = nullptr; size_t s2s_io_cap = 0;    //   host-buffer calls: staged input | output
    uint32_t *d_counters = nullptr; uint32_t counter_seq = 0;   // chunk counters of the persistent parse kernels (one per launch, rotating)
    int enc_fused_xxh = 1;                                 // B2C_ENC_XXH=kernel: XXH64 as its own kernel (A/B measurements)
    cudaEvent_t dec_fork = nullptr, dec_join = nullptr;
    uint8_t *h_in2 = nullptr, *h_out2 = nullptr;   // second pinned staging pair: pageable callers of b2c_zstd_encode_packed (lazy)
    cudaEvent_t ev[2] = {nullptr, nullptr};       // compute of the batch in slot s finished
    cudaEvent_t ev_in[2] = {nullptr, nullptr};    // H2D of slot s finished
    cudaEvent_t ev_out[2] = {nullptr, nullptr};   // D2H of slot s finished
    // decoder: per-warp literal scratch, host-path staging (grown on demand)
    uint8_t *d_dec_lit = nullptr; size_t dec_lit_cap = 0;
    uint8_t *d_fd = nullptr; size_t fd_cap = 0;            // staged decoder: records | FSE tables | Huffman tables
    uint32_t *d_fd_const = nullptr;                          //   code maps + predefined tables
    uint8_t *d_fd_seq = nullptr; size_t fd_seq_cap = 0;    //   sequence records
    uint8_t *d_fd_lit = nullptr; size_t fd_lit_cap = 0;    //   decoded literals
    int dec_staged = 1;                                    // B2C_DEC=onewarp: one-warp decoder only (A/B measurements)
    float dec_ms[6] = {0, 0, 0, 0, 0, 0}; cudaEvent_t dec_ev[7] = {}; int dec_prof = 0;
    uint8_t *d_dec_in = nullptr, *d_dec_out = nullptr; size_t dec_in_cap = 0, dec_out_cap = 0;
    uint8_t *d_dec_meta = nullptr; size_t dec_meta_cap = 0;
    uint8_t *h_stg_in = nullptr, *h_stg_out = nullptr; size_t h_stg_in_cap = 0, h_stg_out_cap = 0;   // pinned staging of the pointer-table calls
    // optional per-kernel timing of the encode pipeline (b2c_profile_*): 6 events per encode call
    bool prof = false;
    std::vector<cudaEvent_t> pev;
    size_t pev_used = 0;
    uint64_t launches = 0;
    char err[256] = {0};
};

#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess) {                                                                       \
            if (ctx) snprintf(ctx->err, sizeof(ctx->err), "%s: %s", #call, cudaGetErrorString(e_));    \
            return B2C_ERR_CUDA;                                                                       \
        }                                                                                              \
    } while (0)

// Host-side gather / scatter of many separately addressed pieces (the pointer-table calls): index ranges are spread over a few
// host threads when there is enough to move -- one thread copies about 10 GB/s, which otherwise bounds these calls far
// below the PCIe rate.  fn(i) handles piece i; pieces are independent.
template <class F> static void parallel_pieces(size_t n, size_t total_bytes, F fn) {
    unsigned hw = std::thread::hardware_concurrency();
    unsigned nt = hw ? (hw < 8 ? hw : 8) : 4;
    if (total_bytes < ((size_t)8 << 20) || n < 2 * (size_t)nt || nt < 2) { for (size_t i = 0; i < n; i++) fn(i); return; }
    const size_t per = (n + nt - 1) / nt;
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; t++) {
        const size_t lo = (size_t)t * per, hi = lo + per < n ? lo + per : n;
        if (lo >= n) break;
        th.emplace_back([=]() { for (size_t i = lo; i < hi; i++) fn(i); });
    }
    for (size_t i = 0; i < (per < n ? per : n); i++) fn(i);
    for (auto &x : th) x.join();
}

static const uint32_t kSlot = 65536 + 512;  // >= MaxEncodedSize(65536) = 65536 + 3 + 7 + 4, 16-byte multiple

// ---- small helper kernels -------------------------------------------------------------------
// exclusive scan of the (non-negative) chunk sizes -> packed offsets; single CTA
__global__ void b2c_scan_sizes_kernel(const int64_t *sizes, uint64_t *offsets, uint32_t n) {
    __shared__ uint64_t carry;
    __shared__ uint64_t wsum[32];
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n; base += blockDim.x) {
        uint32_t i = base + threadIdx.x;
        uint64_t v = (i < n && sizes[i] > 0) ? (uint64_t)sizes[i] : 0;
        uint64_t incl = v;
        for (int d = 1; d < 32; d <<= 1) {
            uint64_t t = __shfl_up_sync(0xffffffffu, incl, d);
            if ((threadIdx.x & 31) >= (unsigned)d) incl += t;
        }
        if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            uint64_t x = (threadIdx.x < (blockDim.x >> 5)) ? wsum[threadIdx.x] : 0, xi = x;
            for (int d = 1; d < 32; d <<= 1) {
                uint64_t t = __shfl_up_sync(0xffffffffu, xi, d);
                if (threadIdx.x >= (unsigned)d) xi += t;
            }
            wsum[threadIdx.x] = xi - x;
        }
        __syncthreads();
        uint64_t ex = carry + wsum[threadIdx.x >> 5] + incl - v;
        if (i < n) offsets[i] = ex;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) carry = ex + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) offsets[n] = carry;
}
// copy chunk i's bytes from its slot to packed[offsets[i]]
__global__ void b2c_pack_kernel(const uint8_t *slots, uint64_t slot_stride, const int64_t *sizes,
                                const uint64_t *offsets, uint8_t *packed, uint32_t n) {
    for (uint32_t c = blockIdx.x; c < n; c += gridDim.x) {
        int64_t sz = sizes[c];
        if (sz <= 0) continue;
        const uint8_t *s = slots + (uint64_t)c * slot_stride;
        uint8_t *d = packed + offsets[c];
        uint32_t head = (uint32_t)((16 - (reinterpret_cast<uintptr_t>(d) & 15)) & 15);
        if (head > (uint32_t)sz) head = (uint32_t)sz;
        for (uint32_t i = threadIdx.x; i < head; i += blockDim.x) d[i] = s[i];
        // aligned body: 4-byte stores assembled from (possibly unaligned) source words
        uint32_t body = ((uint32_t)sz - head) & ~3u;
        for (uint32_t i = threadIdx.x * 4; i < body; i += blockDim.x * 4) {
            uint32_t v = ld32u(s, head + i);
            *reinterpret_cast<uint32_t *>(d + head + i) = v;
        }
        for (uint32_t i = head + body + threadIdx.x; i < (uint32_t)sz; i += blockDim.x) d[i] = s[i];
    }
}

// ---- context -----------------------------------------------------------------------------------
extern "C" {

int b2c_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

b2c_ctx *b2c_ctx_create(int device, size_t max_chunks) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0 || device >= n) return nullptr;
    if (cudaSetDevice(device) != cudaSuccess) return nullptr;
    b2c_ctx *ctx = new b2c_ctx();
    ctx->device = device;
    ctx->max_chunks = max_chunks;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { delete ctx; return nullptr; }
    ctx->sm_count = prop.multiProcessorCount;
    bool ok = true;
    {
        size_t a = 0;
        size_t b = (size_t)ctx->sm_count * LzCfg<1>::MIN_CTAS * LzLayout<1>::SCRATCH_BYTES;
        size_t c = (size_t)ctx->sm_count * LzCfg<2>::MIN_CTAS * LzLayout<2>::SCRATCH_BYTES;
        size_t d3 = (size_t)ctx->sm_count * LzCfg<3>::MIN_CTAS * LzLayout<3>::SCRATCH_BYTES;
        size_t d4 = (size_t)ctx->sm_count * LzCfg<4>::MIN_CTAS * LzLayout<4>::SCRATCH_BYTES;
        if (d3 > a) a = d3;
        if (d4 > a) a = d4;
        size_t d5 = (size_t)ctx->sm_count * LzCfg<5>::MIN_CTAS * LzLayout<5>::SCRATCH_BYTES;
        if (d5 > a) a = d5;
        ctx->scratch_slot = ((a > b ? (a > c ? a : c) : (b > c ? b : c)) + 255) & ~(size_t)255;
    }
    ok = ok && cudaMalloc(&ctx->d_scratch, 2 * ctx->scratch_slot) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->ev_busy, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_lz_parse1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)LzLayout<1>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_lz_parse2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)LzLayout<2>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_lz_parse3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)LzLayout<5>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_lz_s2_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LzLayout<3>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_lz_snappy_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LzLayout<3>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_lz_s2_better_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LzLayout<4>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_lz_snappy_better_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LzLayout<4>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_zstd_pack128_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)PackCfg<131072>::SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_zstd_chains_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)CHAIN_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_huf_compress_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)HUF0_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_huf_decompress_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)DEC_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_huf_dec_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)DEC_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_huf_read_table_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)DEC_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_zstd_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)DEC_SMEM_BYTES) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_zstd_dec_lit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(FD_LIT_WARPS * FD_LIT_WARP_BYTES)) == cudaSuccess;
    ok = ok && cudaFuncSetAttribute(b2c_zstd_dec_init_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)DEC_WARP_BYTES) == cudaSuccess;
    ok = ok && cudaMalloc(&ctx->d_fd_const, FD_CONST_ENTRIES * sizeof(uint32_t)) == cudaSuccess;
    if (ok) {
        b2c_zstd_dec_init_kernel<<<1, 32, DEC_WARP_BYTES>>>(ctx->d_fd_const);
        ok = cudaDeviceSynchronize() == cudaSuccess;
    }
    for (int i = 0; i < 7; i++) ok = ok && cudaEventCreate(&ctx->dec_ev[i]) == cudaSuccess;
    ok = ok && cudaStreamCreateWithFlags(&ctx->dec_aux, cudaStreamNonBlocking) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->dec_fork, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&ctx->dec_join, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaMalloc(&ctx->d_counters, 256 * sizeof(uint32_t)) == cudaSuccess;
    {
        const char *es = getenv("B2C_ENC_XXH");
        ctx->enc_fused_xxh = (es && strcmp(es, "kernel") == 0) ? 0 : 1;
    }
    {
        const char *de = getenv("B2C_DEC");
        ctx->dec_staged = (de && strcmp(de, "onewarp") == 0) ? 0 : 1;
    }
    ok = ok && cudaFuncSetAttribute(b2c_zstd_pack_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)PACK_SMEM_BYTES) == cudaSuccess;
    if (ok && max_chunks) {
        ok = ok && cudaMallocHost(&ctx->h_in, max_chunks * (size_t)ENC_MAX_CHUNK) == cudaSuccess;
        ok = ok && cudaMallocHost(&ctx->h_out, max_chunks * (size_t)kSlot) == cudaSuccess;
        ok = ok && cudaMallocHost(&ctx->h_sizes, (max_chunks + 1) * sizeof(int64_t) * 2) == cudaSuccess;
        ok = ok && cudaMallocHost(&ctx->h_src_sizes, max_chunks * sizeof(uint32_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_in, max_chunks * (size_t)ENC_MAX_CHUNK) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_out, max_chunks * (size_t)kSlot) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_packed, max_chunks * (size_t)kSlot) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_sizes, max_chunks * sizeof(int64_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_offsets, (max_chunks + 1) * sizeof(uint64_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_src_sizes, max_chunks * sizeof(uint32_t)) == cudaSuccess;
        ok = ok && cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) == cudaSuccess;
        ok = ok && cudaStreamCreateWithFlags(&ctx->stream3, cudaStreamNonBlocking) == cudaSuccess;
        for (int k = 0; k < 2; k++) {
            ok = ok && cudaEventCreateWithFlags(&ctx->ev[k], cudaEventDisableTiming) == cudaSuccess;
            ok = ok && cudaEventCreateWithFlags(&ctx->ev_in[k], cudaEventDisableTiming) == cudaSuccess;
            ok = ok && cudaEventCreateWithFlags(&ctx->ev_out[k], cudaEventDisableTiming) == cudaSuccess;
        }
        ok = ok && cudaMallocHost(&ctx->h_sizes2, (max_chunks + 1) * sizeof(int64_t) * 2) == cudaSuccess;
        ok = ok && cudaMallocHost(&ctx->h_src_sizes2, max_chunks * sizeof(uint32_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_in2, max_chunks * (size_t)ENC_MAX_CHUNK) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_out2, max_chunks * (size_t)kSlot) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_packed2, max_chunks * (size_t)kSlot) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_sizes2, max_chunks * sizeof(int64_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_offsets2, (max_chunks + 1) * sizeof(uint64_t)) == cudaSuccess;
        ok = ok && cudaMalloc(&ctx->d_src_sizes2, max_chunks * sizeof(uint32_t)) == cudaSuccess;
    }
    if (!ok) { b2c_ctx_destroy(ctx); return nullptr; }
    return ctx;
}

void b2c_ctx_destroy(b2c_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaFreeHost(ctx->h_stg_in); cudaFreeHost(ctx->h_stg_out);
    cudaFree(ctx->d_fd); cudaFree(ctx->d_fd_const); cudaFree(ctx->d_fd_seq); cudaFree(ctx->d_fd_lit);
    cudaFree(ctx->d_dec_lit); cudaFree(ctx->d_dec_in); cudaFree(ctx->d_dec_out); cudaFree(ctx->d_dec_meta);
    cudaFree(ctx->d_fr); cudaFree(ctx->d_fr_io); cudaFree(ctx->d_counters); cudaFree(ctx->d_s2s); cudaFree(ctx->d_s2s_io); cudaFree(ctx->d_s2d);
    cudaFree(ctx->d_scratch); cudaFree(ctx->d_work[0]); cudaFree(ctx->d_work[1]); cudaFree(ctx->d_pool[0]); cudaFree(ctx->d_pool[1]);
    if (ctx->ev_busy) cudaEventDestroy(ctx->ev_busy); cudaFree(ctx->d_in); cudaFree(ctx->d_out); cudaFree(ctx->d_packed);
    cudaFree(ctx->d_sizes); cudaFree(ctx->d_offsets); cudaFree(ctx->d_src_sizes);
    cudaFreeHost(ctx->h_in); cudaFreeHost(ctx->h_out); cudaFreeHost(ctx->h_in2); cudaFreeHost(ctx->h_out2); cudaFreeHost(ctx->h_sizes); cudaFreeHost(ctx->h_src_sizes);
    cudaFree(ctx->d_in2); cudaFree(ctx->d_out2); cudaFree(ctx->d_packed2); cudaFree(ctx->d_sizes2);
    cudaFree(ctx->d_offsets2); cudaFree(ctx->d_src_sizes2); cudaFreeHost(ctx->h_sizes2); cudaFreeHost(ctx->h_src_sizes2);
    for (cudaEvent_t e : ctx->pev) cudaEventDestroy(e);
    for (int k = 0; k < 2; k++) {
        if (ctx->ev[k]) cudaEventDestroy(ctx->ev[k]);
        if (ctx->ev_in[k]) cudaEventDestroy(ctx->ev_in[k]);
        if (ctx->ev_out[k]) cudaEventDestroy(ctx->ev_out[k]);
    }
    if (ctx->dec_aux) cudaStreamDestroy(ctx->dec_aux);
    if (ctx->dec_fork) cudaEventDestroy(ctx->dec_fork);
    if (ctx->dec_join) cudaEventDestroy(ctx->dec_join);
    if (ctx->stream3) cudaStreamDestroy(ctx->stream3);
    if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *b2c_strerror(int code) {
    switch (code) {
    case B2C_OK: return "ok";
    case B2C_ERR_NO_DEVICE: return "no CUDA device (libb200comp has no CPU fallback)";
    case B2C_ERR_CUDA: return "CUDA runtime error";
    case B2C_ERR_ARG: return "invalid argument";
    case B2C_ERR_TOO_BIG: return "chunk too big for this level's block size";
    case B2C_ERR_DST_SMALL: return "destination too small";
    case B2C_ERR_CORRUPT: return "corrupt input";
    case B2C_ERR_MAGIC: return "invalid input: magic number mismatch";
    case B2C_ERR_WINDOW: return "window size exceeded";
    case B2C_ERR_CRC: return "CRC check failed";
    case B2C_ERR_SIZE: return "frame size exceeded / mismatch";
    case B2C_ERR_UNSUPPORTED: return "unsupported";
    default: return "unknown error";
    }
}
const char *b2c_last_cuda_error(b2c_ctx *ctx) { return ctx ? ctx->err : "no context"; }
int b2c_sm_count(b2c_ctx *ctx) { return ctx ? ctx->sm_count : 0; }
uint64_t b2c_launch_count(b2c_ctx *ctx) { return ctx ? ctx->launches : 0; }

int b2c_profile_enable(b2c_ctx *ctx, int on) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    ctx->prof = on != 0;
    ctx->pev_used = 0;
    return B2C_OK;
}
// ms[k] = summed duration of kernel k (0 xxh64, 1 parse, 2 histograms, 3 tables, 4 chains, 5 pack) over the encode launches issued
// since b2c_profile_enable(ctx, 1); *ncalls = number of encode calls.  Synchronises the device.  The histograms are counted
// inside the parse kernel, so slot 2 is an empty interval (about 0 ms); it is kept so that the six slots keep their meaning.
int b2c_profile_read(b2c_ctx *ctx, double *ms, uint32_t *ncalls) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    CK(cudaSetDevice(ctx->device));
    CK(cudaDeviceSynchronize());
    for (int k = 0; k < 6; k++) ms[k] = 0.0;
    for (size_t c = 0; c + 7 <= ctx->pev_used; c += 7)
        for (int k = 0; k < 6; k++) {
            float t = 0.f;
            CK(cudaEventElapsedTime(&t, ctx->pev[c + k], ctx->pev[c + k + 1]));
            ms[k] += (double)t;
        }
    if (ncalls) *ncalls = (uint32_t)(ctx->pev_used / 7);
    ctx->pev_used = 0;
    return B2C_OK;
}

// Decode-side counterpart: ms[0..5] = summed durations of {scan, literals, sequences, execute, xxh64, one-warp decoder} over the
// staged decode launches since b2c_decode_profile_enable(ctx, 1).  Enabled, every decode launch synchronises.
int b2c_decode_profile_enable(b2c_ctx *ctx, int on) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    ctx->dec_prof = on != 0;
    for (int i = 0; i < 6; i++) ctx->dec_ms[i] = 0.f;
    return B2C_OK;
}
// How many of the first nchunks inputs of the most recent decode launch were completed by the staged kernels (the others
// went through the one-warp decoder).  Synchronises the device.  Test / diagnostics hook.
int b2c_decode_staged_count(b2c_ctx *ctx, uint32_t nchunks, uint32_t *staged) {
    if (!ctx || !staged) return B2C_ERR_ARG;
    *staged = 0;
    if (!ctx->d_fd || !ctx->dec_staged || nchunks == 0) return B2C_OK;
    CK(cudaSetDevice(ctx->device));
    CK(cudaDeviceSynchronize());
    if ((size_t)nchunks * sizeof(FdChunk) > ctx->fd_cap) return B2C_ERR_ARG;
    std::vector<uint32_t> st(nchunks);
    CK(cudaMemcpy2D(st.data(), sizeof(uint32_t), ctx->d_fd, sizeof(FdChunk), sizeof(uint32_t), nchunks, cudaMemcpyDeviceToHost));
    uint32_t k = 0;
    for (uint32_t v : st) k += v == 0;
    *staged = k;
    return B2C_OK;
}
// The same for the most recent S2 block decode launch: blocks finished by the staged kernels (tag walk + execution).
int b2c_s2_decode_staged_count(b2c_ctx *ctx, uint32_t nchunks, uint32_t *staged) {
    if (!ctx || !staged) return B2C_ERR_ARG;
    *staged = 0;
    if (!ctx->d_s2d || !ctx->dec_staged || nchunks == 0) return B2C_OK;
    CK(cudaSetDevice(ctx->device));
    CK(cudaDeviceSynchronize());
    if ((size_t)nchunks * sizeof(S2Head) > ctx->s2d_cap) return B2C_ERR_ARG;
    std::vector<uint32_t> st(nchunks);
    CK(cudaMemcpy2D(st.data(), sizeof(uint32_t), ctx->d_s2d, sizeof(S2Head), sizeof(uint32_t), nchunks, cudaMemcpyDeviceToHost));
    uint32_t k = 0;
    for (uint32_t v : st) k += v == 0;
    *staged = k;
    return B2C_OK;
}
int b2c_decode_profile_read(b2c_ctx *ctx, double *ms) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    for (int i = 0; i < 6; i++) { ms[i] = (double)ctx->dec_ms[i]; ctx->dec_ms[i] = 0.f; }
    return B2C_OK;
}

size_t b2c_zstd_bound(size_t size, int level) {
    // Encoder.MaxEncodedSize, zstd/encoder.go:843-873 (crc on)
    size_t blockSize = (level == B2C_LEVEL_FASTEST) ? (1u << 16) : (128u << 10);
    size_t fh = 4 + 2;
    if (size < 256) fh++;
    else if (size < 65536 + 256) fh += 2;
    else if (size < 0x7fffffff) fh += 4;
    else fh += 8;
    fh += 4;
    size_t blocks = (size + blockSize) / blockSize;
    return fh + 3 * blocks + size;
}

// a zeroed chunk counter for one launch of a persistent parse kernel (rotating: launches in flight never share one)
static int next_counter(b2c_ctx *ctx, cudaStream_t st, uint32_t **out) {
    uint32_t *c = ctx->d_counters + (ctx->counter_seq++ & 255u);
    CK(cudaMemsetAsync(c, 0, sizeof(uint32_t), st));
    *out = c;
    return B2C_OK;
}

static uint32_t level_block(int level) { return level == B2C_LEVEL_FASTEST ? (1u << 16) : (128u << 10); }
static bool level_ok(int level) { return level == B2C_LEVEL_FASTEST || level == B2C_LEVEL_DEFAULT || level == B2C_LEVEL_BETTER; }
static size_t level_slot(int level) { return (size_t)level_block(level) + 512; }   // >= MaxEncodedSize(block), 16-byte multiple

// Calls that use the context's scratch / work buffers are ordered among themselves even when they are issued on
// different streams: the next one waits for the event the previous one recorded.
static int ctx_order_begin(b2c_ctx *ctx, cudaStream_t st) {
    if (ctx->busy_valid && ctx->busy_stream != st) CK(cudaStreamWaitEvent(st, ctx->ev_busy, 0));
    return B2C_OK;
}
static int ctx_order_end(b2c_ctx *ctx, cudaStream_t st) {
    CK(cudaEventRecord(ctx->ev_busy, st));
    ctx->busy_stream = st; ctx->busy_valid = true;
    return B2C_OK;
}

// One encode launch = the four encode kernels (parse, tables, chains + XXH64, pack) over at most `sub` chunks at a time
// (the work records and the work pool are sized for `sub` chunks, so a device-resident call of any size needs a bounded
// amount of scratch).
static int launch_encode(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                         const uint32_t *d_sizes, uint32_t size_all, void *d_dst, size_t dst_stride,
                         int64_t *d_out_sizes, uint32_t nchunks, uint32_t *dbg_hdr, uint32_t *dbg_seqs,
                         uint8_t *dbg_lits, uint32_t dbg_cap, cudaStream_t st, unsigned long long *dbg_cycles = nullptr,
                         int slot = 0, const EncBlockDesc *d_desc = nullptr) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!level_ok(level)) return B2C_ERR_UNSUPPORTED;
    if (nchunks == 0) return B2C_OK;
    if (dst_stride > 0xffffffffull) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const uint32_t blockmax = level_block(level);
    const uint64_t pstride = wk_pool_stride(blockmax);
    const uint32_t subMax = blockmax > 65536 ? 4096u : 8192u;   // work pool: 2.8 GB (64 KiB blocks) / 3.4 GB (128 KiB blocks)
    const uint32_t sub = nchunks < subMax ? nchunks : subMax;
    if (ctx->work_cap[slot] < sub || ctx->pool_cap[slot] < (size_t)sub * pstride) {
        // grow the per-chunk work records / pool (kernels of earlier calls on other streams may still use the old ones)
        CK(cudaDeviceSynchronize());
        if (ctx->work_cap[slot] < sub) {
            if (ctx->d_work[slot]) CK(cudaFree(ctx->d_work[slot]));
            ctx->d_work[slot] = nullptr; ctx->work_cap[slot] = 0;
            CK(cudaMalloc(&ctx->d_work[slot], (size_t)sub * sizeof(ChunkWork)));
            ctx->work_cap[slot] = sub;
        }
        if (ctx->pool_cap[slot] < (size_t)sub * pstride) {
            if (ctx->d_pool[slot]) CK(cudaFree(ctx->d_pool[slot]));
            ctx->d_pool[slot] = nullptr; ctx->pool_cap[slot] = 0;
            CK(cudaMalloc(&ctx->d_pool[slot], (size_t)sub * pstride));
            ctx->pool_cap[slot] = (size_t)sub * pstride;
        }
    }
    { int r = ctx_order_begin(ctx, st); if (r) return r; }
    const unsigned sms = (unsigned)ctx->sm_count;
    for (uint32_t c0 = 0; c0 < nchunks; c0 += sub) {
        const uint32_t m = (nchunks - c0 < sub) ? nchunks - c0 : sub;
        ZstdEncParams P;
        memset(&P, 0, sizeof(P));
        P.src_base = d_desc ? (const uint8_t *)d_src : (const uint8_t *)d_src + (size_t)c0 * src_stride; P.src_stride = src_stride;
        P.desc = d_desc ? d_desc + c0 : nullptr;
        P.src_sizes = d_sizes ? d_sizes + c0 : nullptr; P.src_size_all = size_all;
        P.dst_base = (uint8_t *)d_dst + (size_t)c0 * dst_stride; P.dst_stride = dst_stride; P.dst_cap = (uint32_t)dst_stride;
        P.out_sizes = d_out_sizes + c0; P.nchunks = m; P.flags = (uint32_t)flags;
        P.scratch = ctx->d_scratch + (size_t)slot * ctx->scratch_slot;
        P.work = ctx->d_work[slot];
        P.pool = ctx->d_pool[slot]; P.pool_stride = pstride; P.maxseq = wk_maxseq(blockmax); P.blockmax = blockmax;
        P.big = blockmax > 65536 ? 1u : 0u; P.level = (uint32_t)level;
        if (dbg_hdr) {
            P.dbg_hdr = dbg_hdr + (size_t)c0 * 4; P.dbg_seqs = dbg_seqs + (size_t)c0 * dbg_cap * 3;
            P.dbg_lits = dbg_lits + (size_t)c0 * blockmax; P.dbg_seq_cap = dbg_cap;
        }
        P.dbg_cycles = dbg_cycles ? dbg_cycles + (size_t)c0 * 16 * 32 : nullptr;
        cudaEvent_t *pe = nullptr;
        if (ctx->prof) {
            while (ctx->pev.size() < ctx->pev_used + 7) {
                cudaEvent_t e;
                CK(cudaEventCreate(&e));
                ctx->pev.push_back(e);
            }
            pe = ctx->pev.data() + ctx->pev_used;
            ctx->pev_used += 7;
        }
#define PEV(k) do { if (pe) cudaEventRecord(pe[k], st); } while (0)
        PEV(0);
        // XXH64 rides in the chains launch (four more warps per CTA); as its own kernel only for A/B measurements
        const bool wantXxh = (flags & B2C_ZSTD_FRAME) && (flags & B2C_ZSTD_CRC);
        if (wantXxh && !ctx->enc_fused_xxh) {
            b2c_zstd_xxh_kernel<<<(4 * m + 127) / 128, 128, 0, st>>>(P);
            ctx->launches += 1;
        }
        { int r = next_counter(ctx, st, &P.counter); if (r) return r; }
        PEV(1);
        {
            if (level == B2C_LEVEL_FASTEST) {
                const unsigned cap = sms * LzCfg<1>::MIN_CTAS, g1 = cap < m ? cap : m;
                b2c_lz_parse1_kernel<<<g1, LzCfg<1>::NT, LzLayout<1>::SMEM_BYTES, st>>>(P);
            } else if (level == B2C_LEVEL_DEFAULT) {
                const unsigned cap = sms * LzCfg<2>::MIN_CTAS, g1 = cap < m ? cap : m;
                b2c_lz_parse2_kernel<<<g1, LzCfg<2>::NT, LzLayout<2>::SMEM_BYTES, st>>>(P);
            } else {
                const unsigned cap = sms * LzCfg<5>::MIN_CTAS, g1 = cap < m ? cap : m;
                b2c_lz_parse3_kernel<<<g1, LzCfg<5>::NT, LzLayout<5>::SMEM_BYTES, st>>>(P);
            }
            PEV(2);
            ctx->launches += 1;
        }
        PEV(3);     // (the histograms are counted inside the parse kernel: profile slot 2 is an empty interval)
        const unsigned g2 = sms * TABLES_CTAS_PER_SM < m ? sms * TABLES_CTAS_PER_SM : m;
        b2c_zstd_tables_kernel<<<g2, TABLES_NT, 0, st>>>(P);
        PEV(4);
        b2c_zstd_chains_kernel<<<(m + 31) / 32, CHAIN_NT + ((wantXxh && ctx->enc_fused_xxh) ? CHAIN_XXH_NT : 0), CHAIN_SMEM_BYTES, st>>>(P);
        PEV(5);
        if (blockmax > 65536) b2c_zstd_pack128_kernel<<<m, PACK_NT, PackCfg<131072>::SMEM_BYTES, st>>>(P);
        else b2c_zstd_pack_kernel<<<m, PACK_NT, PACK_SMEM_BYTES, st>>>(P);
        PEV(6);
#undef PEV
        ctx->launches += 3;
        CK(cudaGetLastError());
    }
    return ctx_order_end(ctx, st);
}

int b2c_zstd_encode_device(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                           const uint32_t *d_sizes, uint32_t size_all, void *d_dst, size_t dst_stride,
                           int64_t *d_out_sizes, uint32_t nchunks, void *stream) {
    return launch_encode(ctx, level, flags, d_src, src_stride, d_sizes, size_all, d_dst, dst_stride, d_out_sizes,
                         nchunks, nullptr, nullptr, nullptr, 0, (cudaStream_t)stream);
}

int b2c_zstd_encode_device_debug(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                                 const uint32_t *d_sizes, uint32_t size_all, void *d_dst, size_t dst_stride,
                                 int64_t *d_out_sizes, uint32_t nchunks, uint32_t *d_dbg_hdr, uint32_t *d_dbg_seqs,
                                 uint8_t *d_dbg_lits, uint32_t dbg_seq_cap, void *stream) {
    return launch_encode(ctx, level, flags, d_src, src_stride, d_sizes, size_all, d_dst, dst_stride,
                         d_out_sizes, nchunks, d_dbg_hdr, d_dbg_seqs, d_dbg_lits, dbg_seq_cap, (cudaStream_t)stream);
}

int b2c_zstd_encode_device_timed(b2c_ctx *ctx, int flags, const void *d_src, size_t src_stride, uint32_t size_all,
                                 void *d_dst, size_t dst_stride, int64_t *d_out_sizes, uint32_t nchunks,
                                 unsigned long long *d_cycles, void *stream) {
    return launch_encode(ctx, B2C_LEVEL_FASTEST, flags, d_src, src_stride, nullptr, size_all, d_dst, dst_stride,
                         d_out_sizes, nchunks, nullptr, nullptr, nullptr, 0, (cudaStream_t)stream, d_cycles);
}


// ------------------------------------------------------------------------------------------------ frame mode
// zstd.Encoder.EncodeAll of an input larger than one block (zstd/encoder.go:796-830): ONE frame per input -- header with
// the content size, the blocks, the XXH64 of the whole content.  Every block is encoded by the same six-kernel pipeline
// as an independent chunk, with two differences: the match finder sees the `hist` bytes before the block (previous
// blocks of the same frame, already in memory), and the blocks are bare (no frame header / checksum of their own).
// Blocks are entropy-coded independently (no repeat-mode tables between blocks, which would serialise a frame's
// blocks; the reference's seqCoders.setPrev / compModeRepeat, zstd/seqenc.go:19-42, is a size optimisation only).
// XXH64 of every frame's content: one warp per frame (xxh64_warp: the warp streams, four lanes hash)
constexpr int FRAME_XXH_WARPS = 4;
__global__ void __launch_bounds__(FRAME_XXH_WARPS * 32) b2c_zstd_frame_xxh_kernel(const uint8_t *src, const FrameDesc *fr, uint64_t *xxh, uint32_t nframes) {
    __shared__ __align__(16) uint8_t stg[FRAME_XXH_WARPS][2 * XXH_TILE];
    const unsigned w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t f = blockIdx.x * FRAME_XXH_WARPS + w;
    if (f >= nframes || !fr[f].crc) return;
    const uint64_t h = xxh64_warp(src + fr[f].off, fr[f].size, stg[w], lane);
    if (lane == 0) xxh[f] = h;
}
// base[k + 1] = base[k] + bytes of sub-batch k (offsets[m] = total of the scan)
__global__ void b2c_frame_base_kernel(uint64_t *base, uint32_t k, const uint64_t *offsets, uint32_t m) { base[k + 1] = base[k] + offsets[m]; }
__global__ void b2c_frame_place_kernel(const uint8_t *slots, uint64_t slot_stride, const int64_t *sizes, const uint64_t *offsets,
                                       const uint64_t *base, uint32_t k, const EncBlockDesc *desc, const FrameDesc *fr,
                                       uint8_t *packed, uint64_t cap, uint64_t *pos, uint32_t c0, uint32_t m) {
    for (uint32_t c = blockIdx.x; c < m; c += gridDim.x)
        frame_place_block(slots, slot_stride, sizes, offsets, base[k], desc, fr, packed, cap, pos, c0, c, threadIdx.x, blockDim.x);
}
__global__ void b2c_frame_finish_kernel(const FrameDesc *fr, const uint64_t *pos, const int64_t *sizes_all, const uint64_t *xxh,
                                        uint8_t *packed, uint64_t cap, uint64_t *out_offsets, int64_t *out_sizes, uint32_t nframes) {
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f < nframes) frame_finish_one(fr, pos, sizes_all, xxh, packed, cap, out_offsets, out_sizes, f);
}

__global__ void b2c_s2_stream_total_kernel(const uint64_t *base, uint32_t nsub, uint64_t *total) { *total = 10 + base[nsub]; }

size_t b2c_zstd_frame_bound(size_t size, int level) {
    if (!level_ok(level)) return 0;
    const FrameGeom g = frame_geom(level);
    const size_t blocks = size ? (size + g.block - 1) / g.block : 1;
    return 14 + 4 + 3 * blocks + size;        // maxHeaderSize + checksum + one block header per block (raw blocks at worst)
}

// Device-resident frame mode.  Frame f = h_src_sizes[f] bytes at d_src + h_src_offsets[f] (host arrays: the block list is
// planned on the host).  Frames are written back to back into d_dst (capacity dst_cap); d_dst_offsets[f] / d_out_sizes[f]
// (device arrays) receive where frame f starts and its size (negative = error).  Asynchronous on `stream`.
int b2c_zstd_encode_frames_device(b2c_ctx *ctx, int level, int flags, const void *d_src, const uint64_t *h_src_offsets,
                                  const uint64_t *h_src_sizes, uint32_t nframes, void *d_dst, uint64_t dst_cap,
                                  uint64_t *d_dst_offsets, int64_t *d_out_sizes, void *stream) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!level_ok(level)) return B2C_ERR_UNSUPPORTED;
    if (nframes == 0) return B2C_OK;
    if (!h_src_offsets || !h_src_sizes || !d_dst_offsets || !d_out_sizes) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const FrameGeom g = frame_geom(level);
    const bool crc = (flags & B2C_ZSTD_CRC) != 0;
    // ---- plan: block list and frame table
    std::vector<EncBlockDesc> blocks;
    std::vector<FrameDesc> frames;
    if (!frame_plan(level, crc, h_src_offsets, h_src_sizes, nframes, blocks, frames)) return B2C_ERR_ARG;
    const uint32_t nblocks = (uint32_t)blocks.size();
    const uint32_t subMax = level_block(level) > 65536 ? 4096u : 8192u;
    const uint32_t sub = nblocks < subMax ? nblocks : subMax, nsub = (nblocks + sub - 1) / sub;
    const size_t slotB = (size_t)g.block + 512;
    // ---- device memory of the call: descriptors | frame table | per-block sizes, positions | scan offsets | bases | xxh | slots
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 255) & ~(size_t)255; return r; };
    const size_t oDesc = take(sizeof(EncBlockDesc) * nblocks), oFr = take(sizeof(FrameDesc) * nframes),
                 oSizes = take(sizeof(int64_t) * nblocks), oPos = take(sizeof(uint64_t) * nblocks),
                 oScan = take(sizeof(uint64_t) * ((size_t)sub + 1)), oBase = take(sizeof(uint64_t) * ((size_t)nsub + 1)),
                 oXxh = take(sizeof(uint64_t) * nframes), oSlots = take(slotB * sub);
    if (ctx->fr_cap < o) {
        CK(cudaDeviceSynchronize());
        if (ctx->d_fr) CK(cudaFree(ctx->d_fr));
        ctx->d_fr = nullptr; ctx->fr_cap = 0;
        CK(cudaMalloc(&ctx->d_fr, o));
        ctx->fr_cap = o;
    }
    { int r = ctx_order_begin(ctx, st); if (r) return r; }   // (the frame buffers belong to the context like the work pool)
    uint8_t *B = ctx->d_fr;
    EncBlockDesc *d_desc = (EncBlockDesc *)(B + oDesc);
    FrameDesc *d_frames = (FrameDesc *)(B + oFr);
    int64_t *d_sizes = (int64_t *)(B + oSizes);
    uint64_t *d_pos = (uint64_t *)(B + oPos), *d_scan = (uint64_t *)(B + oScan), *d_base = (uint64_t *)(B + oBase),
             *d_xxh = (uint64_t *)(B + oXxh);
    uint8_t *d_slots = B + oSlots;
    // pageable host vectors: the copies complete before cudaMemcpyAsync returns (staged by the runtime)
    CK(cudaMemcpyAsync(d_desc, blocks.data(), sizeof(EncBlockDesc) * nblocks, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(d_frames, frames.data(), sizeof(FrameDesc) * nframes, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(d_base, 0, sizeof(uint64_t), st));
    if (crc) {
        b2c_zstd_frame_xxh_kernel<<<(nframes + FRAME_XXH_WARPS - 1) / FRAME_XXH_WARPS, FRAME_XXH_WARPS * 32, 0, st>>>(
            (const uint8_t *)d_src, d_frames, d_xxh, nframes);
        ctx->launches += 1;
    }
    for (uint32_t k = 0; k < nsub; k++) {
        const uint32_t c0 = k * sub, m = (nblocks - c0 < sub) ? nblocks - c0 : sub;
        int r = launch_encode(ctx, level, 0, d_src, 0, nullptr, 0, d_slots, slotB, d_sizes + c0, m, nullptr, nullptr, nullptr, 0,
                              st, nullptr, 0, d_desc + c0);
        if (r) return r;
        b2c_scan_sizes_kernel<<<1, 1024, 0, st>>>(d_sizes + c0, d_scan, m);
        b2c_frame_base_kernel<<<1, 1, 0, st>>>(d_base, k, d_scan, m);
        b2c_frame_place_kernel<<<(unsigned)ctx->sm_count * 8, 256, 0, st>>>(d_slots, slotB, d_sizes + c0, d_scan, d_base, k, d_desc,
                                                                              d_frames, (uint8_t *)d_dst, dst_cap, d_pos, c0, m);
        ctx->launches += 3;
    }
    b2c_frame_finish_kernel<<<(nframes + 127) / 128, 128, 0, st>>>(d_frames, d_pos, d_sizes, d_xxh, (uint8_t *)d_dst, dst_cap,
                                                                    d_dst_offsets, d_out_sizes, nframes);
    ctx->launches += 1;
    CK(cudaGetLastError());
    return ctx_order_end(ctx, st);
}

// Host-buffer frame mode: what a cgo shim calls for EncodeAll(src) with len(src) > one block (any mix of sizes).
// srcs[i] -> one frame in dsts[i] (capacity dst_caps[i] >= b2c_zstd_frame_bound); sizes_out[i] = frame bytes or a negative error.
int b2c_zstd_encode_frames(b2c_ctx *ctx, int level, int flags, const void *const *srcs, const size_t *src_sizes,
                           void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!level_ok(level)) return B2C_ERR_UNSUPPORTED;
    if (n == 0) return B2C_OK;
    if (n > 0x7fffffffull) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::vector<uint64_t> offs(n), lens(n);
    uint64_t tin = 0, tout = 0;
    for (size_t i = 0; i < n; i++) {
        offs[i] = tin; lens[i] = src_sizes[i];
        tin += (src_sizes[i] + 15) & ~(uint64_t)15;          // frames start 16-byte aligned (bulk-copy staging of their blocks)
        tout += b2c_zstd_frame_bound(src_sizes[i], level);
    }
    const size_t inB = tin + 64, outB = tout + 64, metaB = (sizeof(uint64_t) + sizeof(int64_t)) * n;
    if (ctx->fr_io_cap < inB + outB + metaB + 512) {
        CK(cudaDeviceSynchronize());
        if (ctx->d_fr_io) CK(cudaFree(ctx->d_fr_io));
        ctx->d_fr_io = nullptr; ctx->fr_io_cap = 0;
        CK(cudaMalloc(&ctx->d_fr_io, inB + outB + metaB + 512));
        ctx->fr_io_cap = inB + outB + metaB + 512;
    }
    uint8_t *d_in = ctx->d_fr_io, *d_out = d_in + ((inB + 255) & ~(size_t)255);
    uint64_t *d_off = (uint64_t *)(d_out + ((outB + 255) & ~(size_t)255));
    int64_t *d_sz = (int64_t *)(d_off + n);
    for (size_t i = 0; i < n; i++)
        if (src_sizes[i]) CK(cudaMemcpyAsync(d_in + offs[i], srcs[i], src_sizes[i], cudaMemcpyHostToDevice, st));
    int r = b2c_zstd_encode_frames_device(ctx, level, flags, d_in, offs.data(), lens.data(), (uint32_t)n, d_out, outB, d_off, d_sz, st);
    if (r) { cudaStreamSynchronize(st); return r; }
    std::vector<uint64_t> ho(n);
    std::vector<int64_t> hs(n);
    CK(cudaMemcpyAsync(ho.data(), d_off, sizeof(uint64_t) * n, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(hs.data(), d_sz, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (size_t i = 0; i < n; i++) {
        if (hs[i] > 0 && (size_t)hs[i] > dst_caps[i]) hs[i] = B2C_ERR_DST_SMALL;
        if (hs[i] > 0) CK(cudaMemcpyAsync(dsts[i], d_out + ho[i], (size_t)hs[i], cudaMemcpyDeviceToHost, st));
        sizes_out[i] = hs[i];
    }
    CK(cudaStreamSynchronize(st));
    return B2C_OK;
}

int b2c_zstd_encode_chunks(b2c_ctx *ctx, int level, int flags, const void *const *srcs, const size_t *src_sizes,
                           void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!level_ok(level)) return B2C_ERR_UNSUPPORTED;
    if (!ctx->max_chunks) return B2C_ERR_ARG;
    const size_t blk = level_block(level), slotB = level_slot(level);
    const size_t mcap = ctx->max_chunks * (size_t)ENC_MAX_CHUNK / blk;   // the staging buffers hold max_chunks x 64 KiB
    if (!mcap) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    for (size_t base = 0; base < n; base += mcap) {
        size_t m = n - base;
        if (m > mcap) m = mcap;
        // contiguous equal-sized input needs no host-side staging copy
        bool contiguous = true;
        for (size_t i = 0; i < m; i++) {
            if (src_sizes[base + i] > blk) { contiguous = false; }
            if (i + 1 < m && ((const uint8_t *)srcs[base + i] + src_sizes[base + i] != (const uint8_t *)srcs[base + i + 1] ||
                              src_sizes[base + i] != blk))
                contiguous = false;
            ctx->h_src_sizes[i] = (uint32_t)(src_sizes[base + i] > blk ? blk + 1 : src_sizes[base + i]);
        }
        size_t in_bytes = 0;
        for (size_t i = 0; i < m; i++) in_bytes += src_sizes[base + i];
        if (contiguous) {
            CK(cudaMemcpyAsync(ctx->d_in, srcs[base], in_bytes, cudaMemcpyHostToDevice, st));
        } else {
            {
                uint8_t *hin = ctx->h_in;
                parallel_pieces(m, in_bytes, [=](size_t i) {
                    const size_t sz = src_sizes[base + i] > blk ? 0 : src_sizes[base + i];
                    memcpy(hin + i * (size_t)blk, srcs[base + i], sz);
                });
            }
            CK(cudaMemcpyAsync(ctx->d_in, ctx->h_in, m * (size_t)blk, cudaMemcpyHostToDevice, st));
        }
        CK(cudaMemcpyAsync(ctx->d_src_sizes, ctx->h_src_sizes, m * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        int rc = launch_encode(ctx, level, flags, ctx->d_in, blk, ctx->d_src_sizes, 0, ctx->d_out, slotB,
                               ctx->d_sizes, (uint32_t)m, nullptr, nullptr, nullptr, 0, st);
        if (rc) return rc;
        b2c_scan_sizes_kernel<<<1, 1024, 0, st>>>(ctx->d_sizes, ctx->d_offsets, (uint32_t)m);
        b2c_pack_kernel<<<ctx->sm_count * 4, 256, 0, st>>>(ctx->d_out, slotB, ctx->d_sizes, ctx->d_offsets, ctx->d_packed, (uint32_t)m);
        ctx->launches += 2;
        int64_t *h_sz = ctx->h_sizes;
        uint64_t *h_off = reinterpret_cast<uint64_t *>(ctx->h_sizes + m);
        CK(cudaMemcpyAsync(h_sz, ctx->d_sizes, m * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(h_off, ctx->d_offsets, (m + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        uint64_t total = h_off[m];
        CK(cudaMemcpyAsync(ctx->h_out, ctx->d_packed, total, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        {
            const uint8_t *hout = ctx->h_out;
            parallel_pieces(m, (size_t)total, [=](size_t i) {
                int64_t sz = h_sz[i];
                if (sz > 0 && (size_t)sz > dst_caps[base + i]) sz = B2C_ERR_DST_SMALL;
                if (sz > 0) memcpy(dsts[base + i], hout + h_off[i], (size_t)sz);
                sizes_out[base + i] = sz;
            });
        }
    }
    return B2C_OK;
}



// ---- host-side helpers of the host-buffer calls ---------------------------------------------------------------
// A Go caller's slices are ordinary (pageable) memory: a cudaMemcpyAsync from them is staged by the driver through a
// small pinned window and blocks.  The packed call therefore stages pageable buffers itself: several host threads copy
// into / out of the context's pinned buffers while the copy engines and kernels work on the neighbouring batches.
static bool host_ptr_is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}
static void parallel_memcpy(void *dst, const void *src, size_t bytes) {
    const size_t kMin = 4u << 20;
    unsigned hw = std::thread::hardware_concurrency();
    unsigned nt = hw ? (hw < 8 ? hw : 8) : 4;
    if (bytes < 2 * kMin || nt < 2) { memcpy(dst, src, bytes); return; }
    if ((size_t)nt * kMin > bytes) nt = (unsigned)(bytes / kMin);
    const size_t per = ((bytes / nt) + 4095) & ~(size_t)4095;
    std::vector<std::thread> th;
    for (unsigned t = 1; t < nt; t++) {
        const size_t lo = (size_t)t * per;
        if (lo >= bytes) break;
        const size_t len = (lo + per <= bytes && t + 1 < nt) ? per : bytes - lo;
        th.emplace_back([=]() { memcpy((uint8_t *)dst + lo, (const uint8_t *)src + lo, len); });
    }
    memcpy(dst, src, per < bytes ? per : bytes);
    for (auto &x : th) x.join();
}

// Contiguous host input -> packed host output (concatenated frames).  Three streams (H2D, kernels, D2H) and two
// buffer slots: the H2D copy of batch b+1 and the D2H copy of batch b-1 overlap the kernels of batch b.  This is the
// shape of a large EncodeAll / of a WithConcurrentBlocks job (zstd/enc_jobs.go): the caller gets one valid zstd
// stream plus the per-chunk frame table.  h_src / h_dst should be pinned (cudaHostRegister / torch pin_memory)
// for full PCIe rate; pageable memory works but is staged by the driver.
static int encode_packed_impl(b2c_ctx *ctx, int level, int flags, const void *h_src, size_t src_bytes,
                              uint32_t chunk_size, void *h_dst, size_t dst_cap, int64_t *sizes_out,
                              uint64_t *offsets_out, size_t *total_out) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!level_ok(level)) return B2C_ERR_UNSUPPORTED;
    const size_t blk = level_block(level), slotB = level_slot(level);
    if (!ctx->max_chunks || chunk_size == 0 || chunk_size > blk) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const size_t nchunks = src_bytes == 0 ? 1 : (src_bytes + chunk_size - 1) / chunk_size;
    const size_t B = ctx->max_chunks * (size_t)ENC_MAX_CHUNK / blk;   // the staging buffers hold max_chunks x 64 KiB
    if (!B) return B2C_ERR_ARG;
    // Batch schedule: full batches, then a tail that halves down to about four chunks per SM.  The H2D stream is the
    // bottleneck of the pipeline, so the time after the last H2D copy (kernels + D2H of the last batch) is pure
    // overhead; a small last batch keeps it short.
    std::vector<size_t> bstart, bcount;
    {
        size_t c0 = 0, rem = nchunks;
        // (below about four chunks per SM a batch is bound by the latency of its serial kernels, not by its size)
        const size_t floorB = (size_t)ctx->sm_count * 4 < B ? (size_t)ctx->sm_count * 4 : B;
        while (rem > 0) {
            size_t m;
            if (rem > B) m = B;
            else if (rem > 2 * floorB) m = rem / 2;
            else m = rem;
            bstart.push_back(c0); bcount.push_back(m);
            c0 += m; rem -= m;
        }
    }
    const size_t nb = bcount.size();
    cudaStream_t st_c = ctx->stream, st_in = ctx->stream2, st_out = ctx->stream3;
    // pageable caller memory is staged through the context's pinned buffers (see parallel_memcpy above)
    const bool stage_in = src_bytes > 0 && !host_ptr_is_pinned(h_src);
    const bool stage_out = !host_ptr_is_pinned(h_dst);
    if ((stage_in && !ctx->h_in2) || (stage_out && !ctx->h_out2)) {
        if (!ctx->h_in2) CK(cudaMallocHost(&ctx->h_in2, ctx->max_chunks * (size_t)ENC_MAX_CHUNK));
        if (!ctx->h_out2) CK(cudaMallocHost(&ctx->h_out2, ctx->max_chunks * (size_t)kSlot));
    }
    uint8_t *stg_in[2] = {ctx->h_in, ctx->h_in2}, *stg_out[2] = {ctx->h_out, ctx->h_out2};
    struct Pending { bool live; uint64_t pos, bytes; } pend[2] = {{false, 0, 0}, {false, 0, 0}};
    // a staged D2H copy of slot sl has landed in pinned memory: hand it to the caller's buffer
    auto drain = [&](int sl) -> int {
        if (!pend[sl].live) return B2C_OK;
        if (cudaEventSynchronize(ctx->ev_out[sl]) != cudaSuccess) return B2C_ERR_CUDA;
        parallel_memcpy((uint8_t *)h_dst + pend[sl].pos, stg_out[sl], pend[sl].bytes);
        pend[sl].live = false;
        return B2C_OK;
    };
    struct Slot { uint8_t *d_in, *d_out, *d_packed; int64_t *d_sizes, *h_sizes; uint64_t *d_off;
                  uint32_t *d_ss, *h_ss; } slot[2] = {
        {ctx->d_in, ctx->d_out, ctx->d_packed, ctx->d_sizes, ctx->h_sizes, ctx->d_offsets, ctx->d_src_sizes, ctx->h_src_sizes},
        {ctx->d_in2, ctx->d_out2, ctx->d_packed2, ctx->d_sizes2, ctx->h_sizes2, ctx->d_offsets2, ctx->d_src_sizes2, ctx->h_src_sizes2}};
    uint64_t out_pos = 0;
    int rc = B2C_OK;
    // batch b's kernels are done: place its frames in the output stream and start the D2H copy
    auto finish = [&](size_t b) -> int {
        const int sl = (int)(b & 1);
        Slot &S = slot[sl];
        size_t c0 = bstart[b], m = bcount[b];
        if (cudaEventSynchronize(ctx->ev[sl]) != cudaSuccess) return B2C_ERR_CUDA;
        const int64_t *h_sz = S.h_sizes;
        const uint64_t *h_off = reinterpret_cast<const uint64_t *>(S.h_sizes + m);
        uint64_t total = h_off[m];
        if (out_pos + total > dst_cap) return B2C_ERR_DST_SMALL;
        if (stage_out) {
            { int rd = drain(sl); if (rd) return rd; }            // the slot's pinned buffer still holds batch b-2
            if (cudaMemcpyAsync(stg_out[sl], S.d_packed, total, cudaMemcpyDeviceToHost, st_out) != cudaSuccess) return B2C_ERR_CUDA;
            pend[sl].live = true; pend[sl].pos = out_pos; pend[sl].bytes = total;
        } else if (cudaMemcpyAsync((uint8_t *)h_dst + out_pos, S.d_packed, total, cudaMemcpyDeviceToHost, st_out) != cudaSuccess)
            return B2C_ERR_CUDA;
        if (cudaEventRecord(ctx->ev_out[sl], st_out) != cudaSuccess) return B2C_ERR_CUDA;
        if (stage_out) { int rd = drain(sl ^ 1); if (rd) return rd; }   // batch b-1's bytes have had a whole batch to arrive
        for (size_t i = 0; i < m; i++) {
            sizes_out[c0 + i] = h_sz[i];
            if (offsets_out) offsets_out[c0 + i] = out_pos + h_off[i];
            if (h_sz[i] < 0) rc = (int)h_sz[i];
        }
        out_pos += total;
        return B2C_OK;
    };
    // H2D of batch b into its slot; the slot's input buffer is free once the kernels of batch b-2 have run
    std::vector<const uint32_t *> bss(nb, nullptr);
    auto upload = [&](size_t b) -> int {
        const int sl = (int)(b & 1);
        Slot &S = slot[sl];
        size_t c0 = bstart[b], m = bcount[b];
        size_t off = c0 * (size_t)chunk_size;
        size_t bytes = (off + m * (size_t)chunk_size <= src_bytes) ? m * (size_t)chunk_size : src_bytes - off;
        if (b >= 2) CK(cudaStreamWaitEvent(st_in, ctx->ev[sl], 0));
        const uint8_t *from = (const uint8_t *)h_src + off;
        if (stage_in && bytes) {
            if (b >= 2) CK(cudaEventSynchronize(ctx->ev_in[sl]));      // the H2D copy of batch b-2 has left the pinned buffer
            parallel_memcpy(stg_in[sl], from, bytes);
            from = stg_in[sl];
        }
        if (bytes) CK(cudaMemcpyAsync(S.d_in, from, bytes, cudaMemcpyHostToDevice, st_in));
        if (bytes != m * (size_t)chunk_size) {  // ragged last chunk (or empty input): explicit sizes
            for (size_t i = 0; i < m; i++) {
                size_t o = i * (size_t)chunk_size;
                S.h_ss[i] = (uint32_t)(o >= bytes ? 0 : (bytes - o < chunk_size ? bytes - o : chunk_size));
            }
            CK(cudaMemcpyAsync(S.d_ss, S.h_ss, m * sizeof(uint32_t), cudaMemcpyHostToDevice, st_in));
            bss[b] = S.d_ss;
        }
        CK(cudaEventRecord(ctx->ev_in[sl], st_in));
        return B2C_OK;
    };
    // The copy of batch b+2 is queued before the host waits for batch b-1, so the H2D engine (the bottleneck) always
    // has the next copy in its queue.
    { int r0 = upload(0); if (r0) return r0; }
    if (nb > 1) { int r1 = upload(1); if (r1) return r1; }
    for (size_t b = 0; b < nb; b++) {
        const int sl = (int)(b & 1);
        Slot &S = slot[sl];
        size_t m = bcount[b];
        // kernels: need the input; the packed-output slot is free once batch b-2's D2H copy is done
        CK(cudaStreamWaitEvent(st_c, ctx->ev_in[sl], 0));
        if (b >= 2) CK(cudaStreamWaitEvent(st_c, ctx->ev_out[sl], 0));
        int r = launch_encode(ctx, level, flags, S.d_in, chunk_size, bss[b], chunk_size, S.d_out, slotB, S.d_sizes,
                              (uint32_t)m, nullptr, nullptr, nullptr, 0, st_c, nullptr, sl);
        if (r) return r;
        b2c_scan_sizes_kernel<<<1, 1024, 0, st_c>>>(S.d_sizes, S.d_off, (uint32_t)m);
        b2c_pack_kernel<<<ctx->sm_count * 4, 256, 0, st_c>>>(S.d_out, slotB, S.d_sizes, S.d_off, S.d_packed, (uint32_t)m);
        ctx->launches += 2;
        CK(cudaMemcpyAsync(S.h_sizes, S.d_sizes, m * sizeof(int64_t), cudaMemcpyDeviceToHost, st_c));
        CK(cudaMemcpyAsync(S.h_sizes + m, S.d_off, (m + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, st_c));
        CK(cudaEventRecord(ctx->ev[sl], st_c));
        if (b + 2 < nb) { int r3 = upload(b + 2); if (r3) return r3; }
        if (b >= 1) { int r2 = finish(b - 1); if (r2) return r2; }
    }
    { int r2 = finish(nb - 1); if (r2) return r2; }
    CK(cudaStreamSynchronize(st_in));
    CK(cudaStreamSynchronize(st_c));
    CK(cudaStreamSynchronize(st_out));
    { int rd = drain(0); if (rd) return rd; }
    { int rd = drain(1); if (rd) return rd; }
    if (total_out) *total_out = out_pos;
    return rc;
}

int b2c_zstd_encode_packed(b2c_ctx *ctx, int level, int flags, const void *h_src, size_t src_bytes,
                           uint32_t chunk_size, void *h_dst, size_t dst_cap, int64_t *sizes_out,
                           uint64_t *offsets_out, size_t *total_out) {
    const int rc = encode_packed_impl(ctx, level, flags, h_src, src_bytes, chunk_size, h_dst, dst_cap, sizes_out, offsets_out,
                                      total_out);
    if (rc != B2C_OK && ctx && ctx->stream) {
        // an error return must not leave copies in flight that read h_src / write h_dst, nor the slots mid-pipeline
        cudaStreamSynchronize(ctx->stream2);
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->stream3);
    }
    return rc;
}

// ---- decoder ------------------------------------------------------------------------------------
static int grow(b2c_ctx *ctx, uint8_t **p, size_t *cap, size_t need) {
    if (*cap >= need) return B2C_OK;
    CK(cudaDeviceSynchronize());
    if (*p) CK(cudaFree(*p));
    *p = nullptr; *cap = 0;
    need += need / 4;
    CK(cudaMalloc(p, need));
    *cap = need;
    return B2C_OK;
}

static int grow_host(b2c_ctx *ctx, uint8_t **p, size_t *cap, size_t need) {
    if (*cap >= need) return B2C_OK;
    if (*p) CK(cudaFreeHost(*p));
    *p = nullptr; *cap = 0;
    need += need / 4;
    CK(cudaMallocHost(p, need));
    *cap = need;
    return B2C_OK;
}
// Pointer-table calls: n separately allocated host pieces <-> one packed device range.  Thousands of small
// cudaMemcpyAsync calls cost more than the bytes they move (and block on pageable memory), so the pieces are gathered
// into / scattered from one pinned staging buffer and cross the bus as ONE copy each way.  offs[i] = offset of piece i in
// the device range `d_base[0, total)`.
static const size_t kStageLimit = (size_t)1 << 30;
static int gather_h2d(b2c_ctx *ctx, const void *const *srcs, const size_t *sizes, const uint64_t *offs, size_t n, uint8_t *d_base,
                      size_t total, cudaStream_t st) {
    if (total == 0) return B2C_OK;
    if (total > kStageLimit) {
        for (size_t i = 0; i < n; i++)
            if (sizes[i]) CK(cudaMemcpyAsync(d_base + offs[i], srcs[i], sizes[i], cudaMemcpyHostToDevice, st));
        return B2C_OK;
    }
    int rc = grow_host(ctx, &ctx->h_stg_in, &ctx->h_stg_in_cap, total);
    if (rc) return rc;
    {
        uint8_t *stg = ctx->h_stg_in;
        parallel_pieces(n, total, [=](size_t i) { if (sizes[i]) memcpy(stg + offs[i], srcs[i], sizes[i]); });
    }
    CK(cudaMemcpyAsync(d_base, ctx->h_stg_in, total, cudaMemcpyHostToDevice, st));
    return B2C_OK;
}
// results: piece i = d_base[offs[i], offs[i] + lens[i]) -> dsts[i]; synchronises the stream
static int scatter_d2h(b2c_ctx *ctx, void *const *dsts, const size_t *lens, const uint64_t *offs, size_t n, const uint8_t *d_base,
                       size_t range, cudaStream_t st) {
    size_t useful = 0;
    for (size_t i = 0; i < n; i++) useful += lens[i];
    if (useful == 0) { CK(cudaStreamSynchronize(st)); return B2C_OK; }
    if (range > kStageLimit || useful * 2 < range) {          // sparse or huge: copy the pieces
        for (size_t i = 0; i < n; i++)
            if (lens[i]) CK(cudaMemcpyAsync(dsts[i], d_base + offs[i], lens[i], cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        return B2C_OK;
    }
    int rc = grow_host(ctx, &ctx->h_stg_out, &ctx->h_stg_out_cap, range);
    if (rc) return rc;
    CK(cudaMemcpyAsync(ctx->h_stg_out, d_base, range, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    {
        const uint8_t *stg = ctx->h_stg_out;
        parallel_pieces(n, useful, [=](size_t i) { if (lens[i]) memcpy(dsts[i], stg + offs[i], lens[i]); });
    }
    return B2C_OK;
}

// lit_span: bytes of the output layout (literal areas mirror it: input c's area starts at c * lit_stride, or at
// dst_offsets[c] when lit_stride is 0 -- the caller then guarantees non-overlapping, increasing offsets); 0 = unknown: the
// one-warp decoder takes every input.
static const uint64_t kStagedSpanLimit = 24ull << 30;
static int launch_decode(b2c_ctx *ctx, ZstdDecParams &P, cudaStream_t st, uint64_t lit_span, uint64_t lit_stride) {
    if (P.nchunks == 0) return B2C_OK;
    const unsigned ctasPerSm = (227u * 1024u) / (DEC_SMEM_BYTES + 1024u);
    unsigned grid = (P.nchunks + DEC_WARPS - 1) / DEC_WARPS;
    unsigned maxGrid = (unsigned)ctx->sm_count * (ctasPerSm ? ctasPerSm : 1);
    if (grid > maxGrid) grid = maxGrid;
    int rc = grow(ctx, &ctx->d_dec_lit, &ctx->dec_lit_cap, (size_t)maxGrid * DEC_WARPS * DEC_LIT_SCRATCH);
    if (rc) return rc;
    P.lit_scratch = ctx->d_dec_lit;
    { int r = ctx_order_begin(ctx, st); if (r) return r; }    // the context's scratch is shared by all streams
    const uint32_t n = P.nchunks;
    const bool prof = ctx->dec_prof != 0;
    // Blocks per input the staged kernels take: FD_MAXB with one lane / quad per input (many inputs), up to FD_MAXB_LONG with one
    // lane / quad per (input, block) when the inputs are few -- then long frames are decoded block-parallel.  The tables are
    // [n][maxb], so n * maxb is bounded.
    uint32_t maxb = FD_MAXB;
    if (n <= 4096) { maxb = (uint32_t)(65536 / n); if (maxb > FD_MAXB_LONG) maxb = FD_MAXB_LONG; }      // (>= 16 blocks per input)
    const bool perBlock = maxb > FD_MAXB;
    const bool staged = ctx->dec_staged && lit_span > 0 && lit_span <= kStagedSpanLimit && (uint64_t)n * maxb * FD_TAB_ENTRIES < (1ull << 31);
    if (staged) {
        const size_t recBytes = (((size_t)n * sizeof(FdChunk)) + 255) & ~(size_t)255;
        const size_t blkBytes = (((size_t)n * maxb * sizeof(FdBlock)) + 255) & ~(size_t)255;
        const size_t tabBytes = (size_t)n * maxb * FD_TAB_ENTRIES * sizeof(uint32_t);
        const size_t hufBytes = (size_t)n * maxb * 2048 * sizeof(uint16_t);
        if ((rc = grow(ctx, &ctx->d_fd, &ctx->fd_cap, recBytes + blkBytes + tabBytes + hufBytes))) return rc;
        if ((rc = grow(ctx, &ctx->d_fd_seq, &ctx->fd_seq_cap, 8 * ((size_t)(lit_span / 3) + 2 * (size_t)n + 8)))) return rc;
        if ((rc = grow(ctx, &ctx->d_fd_lit, &ctx->fd_lit_cap, (size_t)lit_span + 64))) return rc;
        P.fd = reinterpret_cast<FdChunk *>(ctx->d_fd);
        P.fd_blk = reinterpret_cast<FdBlock *>(ctx->d_fd + recBytes);
        P.fd_maxb = maxb; P.fd_per_block = perBlock ? 1u : 0u;
        P.fd_tabs = reinterpret_cast<uint32_t *>(ctx->d_fd + recBytes + blkBytes);
        P.fd_huf = reinterpret_cast<uint16_t *>(ctx->d_fd + recBytes + blkBytes + tabBytes);
        P.fd_const = ctx->d_fd_const;
        P.fd_seqs = reinterpret_cast<uint64_t *>(ctx->d_fd_seq);
        P.fd_lits = ctx->d_fd_lit;
        P.fd_lit_stride = lit_stride;
        const uint32_t units = perBlock ? n * maxb : n;            // what the literal and sequence kernels spread over
        const unsigned groups = (units + FD_LIT_GROUP - 1) / FD_LIT_GROUP;
        if (prof) cudaEventRecord(ctx->dec_ev[0], st);
        b2c_zstd_dec_scan_kernel<<<(n + 31) / 32, 32, 0, st>>>(P);
        if (perBlock) {             // index pass above; now the blocks' contents side by side, then the per-input link pass
            b2c_zstd_dec_scan_block_kernel<<<(units + 31) / 32, 32, 0, st>>>(P);
            b2c_zstd_dec_link_kernel<<<(n + 31) / 32, 32, 0, st>>>(P);
            ctx->launches += 2;
        }
        // the literal kernel and the sequence walk both depend on the scan only and both are bound by the latency of their
        // serial walks, not by any unit: they run side by side (one after the other when per-kernel times are wanted)
        if (prof) {
            cudaEventRecord(ctx->dec_ev[1], st);
            b2c_zstd_dec_lit_kernel<<<(groups + FD_LIT_WARPS - 1) / FD_LIT_WARPS, FD_LIT_WARPS * 32, FD_LIT_WARPS * FD_LIT_WARP_BYTES, st>>>(P);
            cudaEventRecord(ctx->dec_ev[2], st);
            b2c_zstd_dec_seq_kernel<<<(units + 31) / 32, 32, 0, st>>>(P);
        } else {
            // (measured both ways round: the literal kernel on the auxiliary stream is 0.6 ms per GiB better than the sequence
            // walk there; neither order overlaps the two fully -- see DESIGN.md section 3.2 on shared-memory carveouts)
            CK(cudaEventRecord(ctx->dec_fork, st));
            CK(cudaStreamWaitEvent(ctx->dec_aux, ctx->dec_fork, 0));
            b2c_zstd_dec_lit_kernel<<<(groups + FD_LIT_WARPS - 1) / FD_LIT_WARPS, FD_LIT_WARPS * 32, FD_LIT_WARPS * FD_LIT_WARP_BYTES, ctx->dec_aux>>>(P);
            CK(cudaEventRecord(ctx->dec_join, ctx->dec_aux));
            b2c_zstd_dec_seq_kernel<<<(units + 31) / 32, 32, 0, st>>>(P);
            CK(cudaStreamWaitEvent(st, ctx->dec_join, 0));
        }
        if (prof) cudaEventRecord(ctx->dec_ev[3], st);
        b2c_zstd_dec_exec_kernel<<<(n + FD_EXEC_WARPS - 1) / FD_EXEC_WARPS, FD_EXEC_WARPS * 32, 0, st>>>(P);
        if (prof) cudaEventRecord(ctx->dec_ev[4], st);
        if (perBlock) b2c_zstd_dec_xxh_warp_kernel<<<(n + 3) / 4, 128, 0, st>>>(P);     // few, long inputs: a warp streams each
        else b2c_zstd_dec_xxh_kernel<<<(unsigned)(((uint64_t)n * 4 + 127) / 128), 128, 0, st>>>(P);
        if (prof) cudaEventRecord(ctx->dec_ev[5], st);
        ctx->launches += 5;
    }
    b2c_zstd_decode_kernel<<<grid, DEC_WARPS * 32, DEC_SMEM_BYTES, st>>>(P);
    ctx->launches += 1;
    if (prof && staged) {
        cudaEventRecord(ctx->dec_ev[6], st);
        cudaEventSynchronize(ctx->dec_ev[6]);
        for (int i = 0; i < 6; i++) { float ms = 0; cudaEventElapsedTime(&ms, ctx->dec_ev[i], ctx->dec_ev[i + 1]); ctx->dec_ms[i] += ms; }
    }
    CK(cudaGetLastError());
    return ctx_order_end(ctx, st);
}

int b2c_zstd_decode_device(b2c_ctx *ctx, const void *d_src, size_t src_stride, const uint64_t *d_src_offsets,
                           const uint32_t *d_src_sizes, void *d_dst, size_t dst_stride, const uint64_t *d_dst_offsets,
                           uint32_t dst_cap, int64_t *d_out_sizes, uint32_t nchunks, void *stream) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!d_src_sizes || !d_out_sizes) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    ZstdDecParams P;
    memset(&P, 0, sizeof(P));
    P.src_base = (const uint8_t *)d_src; P.src_stride = src_stride; P.src_offsets = d_src_offsets; P.src_sizes = d_src_sizes;
    P.dst_base = (uint8_t *)d_dst; P.dst_stride = dst_stride; P.dst_offsets = d_dst_offsets; P.dst_cap = dst_cap;
    P.out_sizes = d_out_sizes; P.nchunks = nchunks;
    // literal areas: one of dst_cap bytes per input
    return launch_decode(ctx, P, (cudaStream_t)stream, (uint64_t)nchunks * dst_cap, dst_cap);
}

// Host pre-scan of a zstd stream (no decompression): the frames it is made of, each with its byte range and -- when the
// header carries one -- its Frame_Content_Size.  Header layout as in frameDec.reset (zstd/framedec.go:65-270) /
// Header.Decode (zstd/decodeheader.go:94-229); frame length = header + block headers' sizes (blockdec.go:128-160) +
// checksum.  Returns false when the stream cannot be walked (truncated, bad magic, reserved block type): the caller then
// hands the whole input to one decoder warp, which reports the error the reference reports.
struct FrameSpan { size_t off, len; uint64_t fcs; bool has_fcs, skippable; };
static bool scan_frames(const uint8_t *p, size_t n, std::vector<FrameSpan> &out) {
    size_t pos = 0;
    while (pos < n) {
        if (n - pos < 4) return false;
        const uint32_t magic = (uint32_t)p[pos] | ((uint32_t)p[pos + 1] << 8) | ((uint32_t)p[pos + 2] << 16) | ((uint32_t)p[pos + 3] << 24);
        if ((magic & 0xfffffff0u) == 0x184D2A50u) {          // skippable frame: magic, 4-byte size, payload
            if (n - pos < 8) return false;
            const uint64_t sz = (uint32_t)p[pos + 4] | ((uint32_t)p[pos + 5] << 8) | ((uint32_t)p[pos + 6] << 16) | ((uint64_t)p[pos + 7] << 24);
            if (n - pos - 8 < sz) return false;
            out.push_back({pos, (size_t)(8 + sz), 0, true, true});
            pos += 8 + sz;
            continue;
        }
        if (magic != 0xFD2FB528u) return false;
        size_t q = pos + 4;
        if (q >= n) return false;
        const uint8_t fhd = p[q++];
        if (fhd & 8) return false;
        const bool single = (fhd & 32) != 0, crc = (fhd & 4) != 0;
        if (!single) { if (q >= n) return false; q++; }
        const unsigned did = fhd & 3, didLen = did == 3 ? 4 : did;
        if (n - q < didLen) return false;
        q += didLen;
        unsigned fcsLen = 0;
        if ((fhd >> 6) == 0) fcsLen = single ? 1 : 0; else fcsLen = 1u << (fhd >> 6);
        if (n - q < fcsLen) return false;
        uint64_t fcs = 0;
        for (unsigned k = 0; k < fcsLen; k++) fcs |= (uint64_t)p[q + k] << (8 * k);
        if (fcsLen == 2) fcs += 256;
        q += fcsLen;
        for (;;) {                                          // blocks
            if (n - q < 3) return false;
            const uint32_t bh = (uint32_t)p[q] | ((uint32_t)p[q + 1] << 8) | ((uint32_t)p[q + 2] << 16);
            q += 3;
            const uint32_t bt = (bh >> 1) & 3, bs = bh >> 3;
            if (bt == 3) return false;
            const size_t body = bt == 1 ? 1 : bs;
            if (n - q < body) return false;
            q += body;
            if (bh & 1) break;
        }
        if (crc) { if (n - q < 4) return false; q += 4; }
        out.push_back({pos, q - pos, fcs, fcsLen != 0, false});
        pos = q;
    }
    return true;
}

// Host-buffer batch decode: inputs are packed back to back, copied H2D, decoded, outputs copied back.  A stream whose
// frames all declare their content size (what every encoder here and the reference's EncodeAll write) is cut into its
// frames: every frame gets its own decoder warp and the device output buffer is sized from the declared sizes instead
// of the caller's cap (DecodeAll of a large EncodeAll output is thousands of independent frames, not one serial stream).
int b2c_zstd_decode_chunks(b2c_ctx *ctx, const void *const *srcs, const size_t *src_sizes, void *const *dsts,
                           const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (n == 0) return B2C_OK;
    if (n > 0xffffffffull) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // work items: one per frame (split inputs) or one per input (everything else)
    struct Item { size_t input; size_t src_off_in_input; uint32_t src_len; uint64_t dst_off_in_input; uint32_t cap; };
    std::vector<Item> items;
    std::vector<size_t> first_item(n + 1, 0);
    std::vector<uint64_t> in_base(n), out_base(n), out_len(n);
    std::vector<char> split(n, 0);
    uint64_t inb = 0, outb = 0;
    std::vector<FrameSpan> fr;
    for (size_t i = 0; i < n; i++) {
        if (src_sizes[i] > 0xffffffffull) return B2C_ERR_ARG;
        first_item[i] = items.size();
        const uint64_t cap = dst_caps[i] > 0xffffffffull ? 0xffffffffull : dst_caps[i];
        fr.clear();
        bool ok = src_sizes[i] > 0 && scan_frames((const uint8_t *)srcs[i], src_sizes[i], fr) && !fr.empty();
        uint64_t total = 0;
        if (ok)
            for (const FrameSpan &f : fr) {
                if (!f.skippable && (!f.has_fcs || f.fcs > 0xffffffffull)) { ok = false; break; }
                total += f.skippable ? 0 : f.fcs;
            }
        if (ok && total > cap) ok = false;               // the serial path reports the reference's "too large" error
        in_base[i] = inb; out_base[i] = outb;
        if (ok) {
            split[i] = 1;
            uint64_t o = 0;
            for (const FrameSpan &f : fr) {
                if (f.skippable) continue;
                items.push_back({i, f.off, (uint32_t)f.len, o, (uint32_t)f.fcs});
                o += f.fcs;
            }
            out_len[i] = total;
        } else {
            items.push_back({i, 0, (uint32_t)src_sizes[i], 0, (uint32_t)cap});
            out_len[i] = cap;
        }
        inb += (src_sizes[i] + 15) & ~(size_t)15;
        outb += (out_len[i] + 15) & ~(uint64_t)15;
    }
    first_item[n] = items.size();
    const size_t m = items.size();
    if (m > 0xffffffffull) return B2C_ERR_ARG;
    // meta: src_off[m] u64 | dst_off[m] u64 | out_sizes[m] i64 | src_sizes[m] u32 | dst_caps[m] u32
    std::vector<uint64_t> meta(3 * m + m);
    uint64_t *so = meta.data(), *dof = so + m;
    uint32_t *ss = reinterpret_cast<uint32_t *>(meta.data() + 3 * m), *dc = ss + m;
    for (size_t k = 0; k < m; k++) {
        so[k] = in_base[items[k].input] + items[k].src_off_in_input;
        dof[k] = out_base[items[k].input] + items[k].dst_off_in_input;
        ss[k] = items[k].src_len; dc[k] = items[k].cap;
    }
    int rc;
    if ((rc = grow(ctx, &ctx->d_dec_in, &ctx->dec_in_cap, inb + 64))) return rc;
    if ((rc = grow(ctx, &ctx->d_dec_out, &ctx->dec_out_cap, outb + 64))) return rc;
    if ((rc = grow(ctx, &ctx->d_dec_meta, &ctx->dec_meta_cap, meta.size() * 8))) return rc;
    if ((rc = gather_h2d(ctx, srcs, src_sizes, in_base.data(), n, ctx->d_dec_in, (size_t)inb, st))) return rc;
    CK(cudaMemcpyAsync(ctx->d_dec_meta, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, st));
    ZstdDecParams P;
    memset(&P, 0, sizeof(P));
    uint64_t *dm = reinterpret_cast<uint64_t *>(ctx->d_dec_meta);
    P.src_base = ctx->d_dec_in; P.src_offsets = dm; P.src_sizes = reinterpret_cast<uint32_t *>(dm + 3 * m);
    P.dst_base = ctx->d_dec_out; P.dst_offsets = dm + m; P.dst_caps = P.src_sizes + m;
    P.out_sizes = reinterpret_cast<int64_t *>(dm + 2 * m); P.nchunks = (uint32_t)m;
    if ((rc = launch_decode(ctx, P, st, outb, 0))) return rc;
    std::vector<int64_t> res(m);
    CK(cudaMemcpyAsync(res.data(), P.out_sizes, m * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (size_t i = 0; i < n; i++) {
        int64_t total = 0;
        for (size_t k = first_item[i]; k < first_item[i + 1]; k++) {
            if (res[k] < 0) {                                                // the first failing frame decides
                // a split frame's capacity is its declared content size: running out of it means the frame is larger
                // than declared, which the reference reports as ErrFrameSizeExceeded (framedec.go:330-412)
                total = (split[i] && res[k] == B2C_ERR_DST_SMALL) ? (int64_t)B2C_ERR_SIZE : res[k];
                break;
            }
            if (split[i] && (uint64_t)res[k] != items[k].cap) { total = B2C_ERR_SIZE; break; }   // declared size not met
            total += res[k];
        }
        sizes_out[i] = total;
        out_len[i] = total > 0 ? (uint64_t)total : 0;
    }
    {
        std::vector<size_t> lens(n);
        for (size_t i = 0; i < n; i++) lens[i] = (size_t)out_len[i];
        if ((rc = scatter_d2h(ctx, dsts, lens.data(), out_base.data(), n, ctx->d_dec_out, (size_t)outb, st))) return rc;
    }
    return B2C_OK;
}


// ---- S2 / Snappy blocks ---------------------------------------------------------------------------
size_t b2c_s2_bound(size_t n) {
    // s2.MaxEncodedLen (s2/encode.go:389-418), 64-bit platform; 0 when the block is too large
    if (n > 0xffffffffull) return 0;
    size_t bits = 0;
    for (size_t v = n; v; v >>= 1) bits++;
    size_t r = n + (bits + 7) / 7;
    if (n) r += n < 60 ? 1 : n < (1u << 8) ? 2 : n < (1u << 16) ? 3 : n < (1u << 24) ? 4 : 5;
    return r > 0xffffffffull ? 0 : r;
}

static int launch_s2_encode(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                            const uint32_t *d_sizes, uint32_t size_all, uint64_t src_total, void *d_dst, size_t dst_stride,
                            int64_t *d_out_sizes, uint32_t nchunks, cudaStream_t st) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (level != B2C_S2_FAST && level != B2C_S2_BETTER) return B2C_ERR_UNSUPPORTED;
    if (nchunks == 0) return B2C_OK;
    if (dst_stride > 0xffffffffull) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    { int r = ctx_order_begin(ctx, st); if (r) return r; }
    ZstdEncParams P;
    memset(&P, 0, sizeof(P));
    P.src_base = (const uint8_t *)d_src; P.src_stride = src_stride; P.src_sizes = d_sizes; P.src_size_all = size_all;
    P.src_total = src_total;
    P.dst_base = (uint8_t *)d_dst; P.dst_stride = dst_stride; P.dst_cap = (uint32_t)dst_stride;
    P.out_sizes = d_out_sizes; P.nchunks = nchunks; P.blockmax = ENC_MAX_CHUNK;
    P.scratch = ctx->d_scratch;
    { int r = next_counter(ctx, st, &P.counter); if (r) return r; }
    const unsigned sms = (unsigned)ctx->sm_count;
    const bool snappy = (flags & B2C_S2_SNAPPY) != 0;
    if (level == B2C_S2_FAST) {
        const unsigned cap = sms * LzCfg<3>::MIN_CTAS, g1 = cap < nchunks ? cap : nchunks;
        if (snappy) b2c_lz_snappy_fast_kernel<<<g1, LzCfg<3>::NT, LzLayout<3>::SMEM_BYTES, st>>>(P);
        else b2c_lz_s2_fast_kernel<<<g1, LzCfg<3>::NT, LzLayout<3>::SMEM_BYTES, st>>>(P);
    } else {
        const unsigned cap = sms * LzCfg<4>::MIN_CTAS, g1 = cap < nchunks ? cap : nchunks;
        if (snappy) b2c_lz_snappy_better_kernel<<<g1, LzCfg<4>::NT, LzLayout<4>::SMEM_BYTES, st>>>(P);
        else b2c_lz_s2_better_kernel<<<g1, LzCfg<4>::NT, LzLayout<4>::SMEM_BYTES, st>>>(P);
    }
    ctx->launches += 1;
    CK(cudaGetLastError());
    return ctx_order_end(ctx, st);
}

int b2c_s2_encode_device(b2c_ctx *ctx, int level, int flags, const void *d_src, size_t src_stride,
                         const uint32_t *d_sizes, uint32_t size_all, void *d_dst, size_t dst_stride,
                         int64_t *d_out_sizes, uint32_t nchunks, void *stream) {
    return launch_s2_encode(ctx, level, flags, d_src, src_stride, d_sizes, size_all, 0, d_dst, dst_stride, d_out_sizes, nchunks,
                            (cudaStream_t)stream);
}

static int launch_s2_decode(b2c_ctx *ctx, S2DecParams &P, uint64_t span, cudaStream_t st);

// ------------------------------------------------------------------------------------------------ S2 / Snappy streams
// s2.Writer.EncodeBuffer / s2.Reader for whole buffers (s2/writer.go:357-470, s2/reader.go:249-420): the framing format
// around the block codecs -- stream identifier, one chunk per block with the masked CRC32-C of its uncompressed bytes.
size_t b2c_s2_stream_bound(size_t n, size_t block) {
    if (block == 0 || block > 65536) return 0;
    const size_t nb = (n + block - 1) / block;
    return 10 + nb * 8 + nb * (b2c_s2_bound(block) - block) + n;
}

// Device-resident: d_src[0, n) -> a complete stream in d_dst; *d_total (device, 8 bytes) = its length; *d_err (device, 4
// bytes) = 0 or a negative error (B2C_ERR_DST_SMALL).  block <= 65536.  Asynchronous on `stream`.
int b2c_s2_encode_stream_device(b2c_ctx *ctx, int level, int flags, const void *d_src, uint64_t n, uint32_t block, void *d_dst,
                                uint64_t dst_cap, uint64_t *d_total, int32_t *d_err, void *stream) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (level != B2C_S2_FAST && level != B2C_S2_BETTER) return B2C_ERR_UNSUPPORTED;
    if (block == 0 || block > 65536 || !d_total || !d_err) return B2C_ERR_ARG;
    if (n / block >= 0x7fffffffull || dst_cap < 10) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const uint32_t nblocks = (uint32_t)((n + block - 1) / block);
    const uint32_t sub = nblocks < 4096 ? (nblocks ? nblocks : 1) : 4096u, nsub = (nblocks + sub - 1) / sub;
    const size_t slotB = (b2c_s2_bound(block) + 15) & ~(size_t)15;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += (bytes + 255) & ~(size_t)255; return r; };
    const size_t oSlots = take(slotB * sub), oEnc = take(sizeof(int64_t) * sub), oPiece = take(sizeof(int64_t) * sub),
                 oCrc = take(sizeof(uint32_t) * sub), oScan = take(sizeof(uint64_t) * ((size_t)sub + 1)),
                 oBase = take(sizeof(uint64_t) * ((size_t)nsub + 1));
    if (ctx->s2s_cap < o) {
        CK(cudaDeviceSynchronize());
        if (ctx->d_s2s) CK(cudaFree(ctx->d_s2s));
        ctx->d_s2s = nullptr; ctx->s2s_cap = 0;
        CK(cudaMalloc(&ctx->d_s2s, o));
        ctx->s2s_cap = o;
    }
    { int r = ctx_order_begin(ctx, st); if (r) return r; }
    uint8_t *B = ctx->d_s2s;
    uint64_t *d_base = (uint64_t *)(B + oBase);
    CK(cudaMemsetAsync(d_base, 0, sizeof(uint64_t), st));
    CK(cudaMemsetAsync(d_err, 0, sizeof(int32_t), st));
    const bool snappy = (flags & B2C_S2_SNAPPY) != 0;
    if (nblocks == 0) {      // an empty input: the identifier alone
        const char *magic = snappy ? "\xff\x06\x00\x00sNaPpY" : "\xff\x06\x00\x00S2sTwO";
        CK(cudaMemcpyAsync(d_dst, magic, 10, cudaMemcpyHostToDevice, st));
    }
    for (uint32_t k = 0; k < nsub && nblocks; k++) {
        const uint32_t c0 = k * sub, m = (nblocks - c0 < sub) ? nblocks - c0 : sub;
        const uint8_t *srck = (const uint8_t *)d_src + (uint64_t)c0 * block;
        int r = launch_s2_encode(ctx, level, flags, srck, block, nullptr, block, n - (uint64_t)c0 * block, B + oSlots, slotB,
                                 (int64_t *)(B + oEnc), m, st);
        if (r) return r;
        S2StreamParams P;
        memset(&P, 0, sizeof(P));
        P.src = (const uint8_t *)d_src; P.total = n; P.block = block;
        P.slots = B + oSlots; P.slot_stride = slotB; P.enc_sizes = (const int64_t *)(B + oEnc);
        P.crc = (uint32_t *)(B + oCrc); P.piece = (int64_t *)(B + oPiece); P.offsets = (const uint64_t *)(B + oScan);
        P.base = d_base; P.k = k; P.dst = (uint8_t *)d_dst; P.cap = dst_cap; P.c0 = c0; P.m = m; P.snappy = snappy ? 1u : 0u;
        P.err = d_err;
        b2c_s2_stream_crc_kernel<<<(unsigned)ctx->sm_count * 4, S2S_WARPS * 32, 0, st>>>(P);
        b2c_scan_sizes_kernel<<<1, 1024, 0, st>>>(P.piece, (uint64_t *)(B + oScan), m);
        b2c_s2_stream_place_kernel<<<(unsigned)ctx->sm_count * 8, 256, 0, st>>>(P);
        b2c_frame_base_kernel<<<1, 1, 0, st>>>(d_base, k, (const uint64_t *)(B + oScan), m);
        ctx->launches += 4;
    }
    // total = identifier + all pieces
    b2c_s2_stream_total_kernel<<<1, 1, 0, st>>>(d_base, nsub * (nblocks ? 1u : 0u), d_total);
    CK(cudaGetLastError());
    return ctx_order_end(ctx, st);
}

// Host buffers: src[0, n) -> stream in dst (capacity cap >= b2c_s2_stream_bound); *out_len = stream bytes.  Synchronous.
int b2c_s2_encode_stream(b2c_ctx *ctx, int level, int flags, const void *src, size_t n, uint32_t block, void *dst, size_t cap,
                         size_t *out_len) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!out_len || block == 0 || block > 65536) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t bound = b2c_s2_stream_bound(n, block);
    const size_t inB = (n + 255) & ~(size_t)255, outB = (bound + 255) & ~(size_t)255;
    if (ctx->s2s_io_cap < inB + outB + 512) {
        CK(cudaDeviceSynchronize());
        if (ctx->d_s2s_io) CK(cudaFree(ctx->d_s2s_io));
        ctx->d_s2s_io = nullptr; ctx->s2s_io_cap = 0;
        CK(cudaMalloc(&ctx->d_s2s_io, inB + outB + 512));
        ctx->s2s_io_cap = inB + outB + 512;
    }
    uint8_t *d_in = ctx->d_s2s_io, *d_out = d_in + inB;
    uint64_t *d_total = (uint64_t *)(d_out + outB);
    int32_t *d_err = (int32_t *)(d_total + 1);
    if (n) CK(cudaMemcpyAsync(d_in, src, n, cudaMemcpyHostToDevice, st));
    int r = b2c_s2_encode_stream_device(ctx, level, flags, d_in, n, block, d_out, bound, d_total, d_err, st);
    if (r) { cudaStreamSynchronize(st); return r; }
    uint64_t total = 0; int32_t err = 0;
    CK(cudaMemcpyAsync(&total, d_total, sizeof(total), cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&err, d_err, sizeof(err), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (err) return err;
    if (total > cap) return B2C_ERR_DST_SMALL;
    CK(cudaMemcpy(dst, d_out, total, cudaMemcpyDeviceToHost));
    *out_len = (size_t)total;
    return B2C_OK;
}

// Host buffers: a complete S2 / Snappy stream -> its content (s2.Reader over a buffer).  The chunk headers are walked on the
// host (4 bytes each, no data is touched there); the device decodes every block, copies uncompressed chunks and verifies
// all checksums.  Errors are the reader's: B2C_ERR_CORRUPT (ErrCorrupt), B2C_ERR_CRC (ErrCRC), B2C_ERR_UNSUPPORTED
// (reserved unskippable chunk), B2C_ERR_DST_SMALL.
int b2c_s2_decode_stream(b2c_ctx *ctx, const void *src, size_t n, void *dst, size_t cap, size_t *out_len) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!out_len) return B2C_ERR_ARG;
    const uint8_t *s = (const uint8_t *)src;
    std::vector<S2StreamBlock> blocks;
    uint64_t o = 0, total = 0;
    bool seen = false, snappyFrame = false;
    const uint32_t maxBlock = 4u << 20;                      // s2/s2.go:87 maxBlockSize
    while (o < n) {
        if (o + 4 > n) return B2C_ERR_CORRUPT;               // io.ErrUnexpectedEOF
        const uint32_t typ = s[o], ln = (uint32_t)s[o + 1] | (uint32_t)s[o + 2] << 8 | (uint32_t)s[o + 3] << 16;
        o += 4;
        if (!seen) { if (typ != 0xff) return B2C_ERR_CORRUPT; seen = true; }
        if (typ == 0x00 || typ == 0x01) {
            if (ln < 4 || o + ln > n) return B2C_ERR_CORRUPT;
            S2StreamBlock b;
            b.type = typ; b.crc = (uint32_t)s[o] | (uint32_t)s[o + 1] << 8 | (uint32_t)s[o + 2] << 16 | (uint32_t)s[o + 3] << 24;
            b.src_off = o + 4; b.src_len = ln - 4; b.dst_off = total;
            if (typ == 0x00) {
                uint64_t v = 0; uint32_t k = 0, shift = 0;             // DecodedLen (s2/decode.go:36-49)
                for (;;) {
                    if (k >= b.src_len || k >= 10) return B2C_ERR_CORRUPT;
                    const uint8_t by = s[b.src_off + k++];
                    v |= (uint64_t)(by & 0x7f) << shift;
                    if (by < 0x80) break;
                    shift += 7;
                }
                if (k > 5 || v > 0xffffffffull) return B2C_ERR_CORRUPT;
                if (v > maxBlock || (snappyFrame && v > 65536)) return B2C_ERR_CORRUPT;
                b.dst_len = (uint32_t)v;
            } else {
                if (b.src_len > maxBlock || (snappyFrame && b.src_len > 65536)) return B2C_ERR_CORRUPT;
                b.dst_len = b.src_len;
            }
            total += b.dst_len;
            blocks.push_back(b);
        } else if (typ == 0xff) {
            if (ln != 6 || o + 6 > n) return B2C_ERR_CORRUPT;
            if (memcmp(s + o, "S2sTwO", 6) == 0) snappyFrame = false;
            else if (memcmp(s + o, "sNaPpY", 6) == 0) snappyFrame = true;
            else return B2C_ERR_CORRUPT;
        } else if (typ <= 0x7f) {
            return B2C_ERR_UNSUPPORTED;                        // reserved unskippable chunk (s2/reader.go:386-391)
        } else if (o + ln > n) {
            return B2C_ERR_CORRUPT;                            // skippable chunk / padding cut short
        }
        o += ln;
    }
    if (total > cap) return B2C_ERR_DST_SMALL;
    *out_len = (size_t)total;
    const uint32_t nb = (uint32_t)blocks.size();
    if (nb == 0) return B2C_OK;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t r = off; off += (bytes + 255) & ~(size_t)255; return r; };
    const size_t oIn = take(n), oOut = take(total + 16), oBlk = take(sizeof(S2StreamBlock) * nb), oSrcOff = take(8 * (size_t)nb),
                 oDstOff = take(8 * (size_t)nb), oSrcSz = take(4 * (size_t)nb), oCaps = take(4 * (size_t)nb),
                 oRes = take(8 * (size_t)nb), oStat = take(4 * (size_t)nb);
    if (ctx->s2s_io_cap < off) {
        CK(cudaDeviceSynchronize());
        if (ctx->d_s2s_io) CK(cudaFree(ctx->d_s2s_io));
        ctx->d_s2s_io = nullptr; ctx->s2s_io_cap = 0;
        CK(cudaMalloc(&ctx->d_s2s_io, off));
        ctx->s2s_io_cap = off;
    }
    uint8_t *B = ctx->d_s2s_io;
    // compressed blocks go to the block decoder; an uncompressed chunk is handed to it as an empty job (size 0 in, cap 0)
    std::vector<uint64_t> so(nb), dof(nb);
    std::vector<uint32_t> ssz(nb), caps(nb);
    for (uint32_t i = 0; i < nb; i++) {
        so[i] = blocks[i].src_off; dof[i] = blocks[i].dst_off;
        ssz[i] = blocks[i].type == 0 ? blocks[i].src_len : 0; caps[i] = blocks[i].type == 0 ? blocks[i].dst_len : 0;
    }
    CK(cudaMemcpyAsync(B + oIn, src, n, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B + oBlk, blocks.data(), sizeof(S2StreamBlock) * nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B + oSrcOff, so.data(), 8 * (size_t)nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B + oDstOff, dof.data(), 8 * (size_t)nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B + oSrcSz, ssz.data(), 4 * (size_t)nb, cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(B + oCaps, caps.data(), 4 * (size_t)nb, cudaMemcpyHostToDevice, st));
    S2DecParams P;
    memset(&P, 0, sizeof(P));
    P.src_base = B + oIn; P.src_offsets = (const uint64_t *)(B + oSrcOff); P.src_sizes = (const uint32_t *)(B + oSrcSz);
    P.dst_base = B + oOut; P.dst_offsets = (const uint64_t *)(B + oDstOff); P.dst_caps = (const uint32_t *)(B + oCaps);
    P.out_sizes = (int64_t *)(B + oRes); P.nchunks = nb;
    { int r = launch_s2_decode(ctx, P, n, st); if (r) return r; }
    unsigned g2 = (nb + S2S_WARPS - 1) / S2S_WARPS;
    if (g2 > (unsigned)ctx->sm_count * 16) g2 = (unsigned)ctx->sm_count * 16;
    b2c_s2_stream_verify_kernel<<<g2, S2S_WARPS * 32, 0, st>>>((const S2StreamBlock *)(B + oBlk), B + oIn, B + oOut,
                                                                (const int64_t *)(B + oRes), (int32_t *)(B + oStat), nb);
    ctx->launches += 1;
    std::vector<int32_t> stat(nb);
    CK(cudaMemcpyAsync(stat.data(), B + oStat, 4 * (size_t)nb, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (uint32_t i = 0; i < nb; i++)
        if (stat[i]) return stat[i] == -4 ? B2C_ERR_CORRUPT : stat[i];      // (a block longer than its declared length is corrupt)
    CK(cudaMemcpy(dst, B + oOut, total, cudaMemcpyDeviceToHost));
    return B2C_OK;
}

// S2 block decode launch.  span = bytes of the input layout (blocks lie inside [0, span) at increasing, non-overlapping offsets) or
// 0 when the host does not know it.  With a span the staged form runs first (tag walk one lane per block, execution one warp per
// block); the one-warp kernel then takes what they left (large or unusual blocks, errors).
static int launch_s2_decode(b2c_ctx *ctx, S2DecParams &P, uint64_t span, cudaStream_t st) {
    const uint32_t n = P.nchunks;
    const bool staged = ctx->dec_staged && span > 0 && span <= ((uint64_t)8 << 30);
    if (staged) {
        const size_t headBytes = (((size_t)n * sizeof(S2Head)) + 255) & ~(size_t)255;
        const size_t recBytes = ((size_t)(span / 3) + n + 16) * sizeof(uint64_t);
        { int r = ctx_order_begin(ctx, st); if (r) return r; }
        int rc = grow(ctx, &ctx->d_s2d, &ctx->s2d_cap, headBytes + recBytes);
        if (rc) return rc;
        P.heads = reinterpret_cast<S2Head *>(ctx->d_s2d);
        P.recs = reinterpret_cast<uint64_t *>(ctx->d_s2d + headBytes);
        b2c_s2_walk_kernel<<<(n + 31) / 32, 32, 0, st>>>(P);
        b2c_s2_exec_kernel<<<(n + S2DEC_WARPS - 1) / S2DEC_WARPS, S2DEC_WARPS * 32, 0, st>>>(P);
        ctx->launches += 2;
    }
    unsigned grid = (n + S2DEC_WARPS - 1) / S2DEC_WARPS, maxGrid = (unsigned)ctx->sm_count * 16;
    if (grid > maxGrid) grid = maxGrid;
    b2c_s2_decode_kernel<<<grid, S2DEC_WARPS * 32, 0, st>>>(P);
    ctx->launches += 1;
    CK(cudaGetLastError());
    if (staged) return ctx_order_end(ctx, st);
    return B2C_OK;
}

int b2c_s2_decode_device(b2c_ctx *ctx, const void *d_src, size_t src_stride, const uint64_t *d_src_offsets,
                         const uint32_t *d_src_sizes, void *d_dst, size_t dst_stride, const uint64_t *d_dst_offsets,
                         uint32_t dst_cap, int64_t *d_out_sizes, uint32_t nchunks, void *stream) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!d_src_sizes || !d_out_sizes) return B2C_ERR_ARG;
    if (nchunks == 0) return B2C_OK;
    CK(cudaSetDevice(ctx->device));
    S2DecParams P;
    memset(&P, 0, sizeof(P));
    P.src_base = (const uint8_t *)d_src; P.src_stride = src_stride; P.src_offsets = d_src_offsets; P.src_sizes = d_src_sizes;
    P.dst_base = (uint8_t *)d_dst; P.dst_stride = dst_stride; P.dst_offsets = d_dst_offsets; P.dst_cap = dst_cap;
    P.out_sizes = d_out_sizes; P.nchunks = nchunks;
    return launch_s2_decode(ctx, P, d_src_offsets ? 0 : (uint64_t)nchunks * src_stride, (cudaStream_t)stream);
}

// Host-buffer batches for the block API (s2.Encode / s2.EncodeSnappy / s2.Decode per element).  Inputs are packed
// back to back on the device, outputs land in per-element slots; one kernel per call.
static int s2_host_batch(b2c_ctx *ctx, bool encode, int level, int flags, const void *const *srcs, const size_t *src_sizes,
                         void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (n == 0) return B2C_OK;
    if (n > 0xffffffffull) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::vector<uint64_t> meta(3 * n + n);
    uint64_t *so = meta.data(), *dof = so + n;
    uint32_t *ss = reinterpret_cast<uint32_t *>(meta.data() + 3 * n), *dc = ss + n;
    uint64_t inb = 0, outb = 0;
    for (size_t i = 0; i < n; i++) {
        if (src_sizes[i] > 0xffffffffull) return B2C_ERR_ARG;
        so[i] = inb; dof[i] = outb;
        ss[i] = (uint32_t)src_sizes[i];
        dc[i] = (uint32_t)(dst_caps[i] > 0xffffffffull ? 0xffffffffull : dst_caps[i]);
        // encode: fixed strides (the kernel addresses chunks by stride)
        inb += encode ? (size_t)ENC_MAX_CHUNK : ((src_sizes[i] + 15) & ~(size_t)15);
        outb += encode ? (size_t)kSlot : (((size_t)dc[i] + 15) & ~(size_t)15);
    }
    int rc;
    if ((rc = grow(ctx, &ctx->d_dec_in, &ctx->dec_in_cap, inb + 256))) return rc;
    if ((rc = grow(ctx, &ctx->d_dec_out, &ctx->dec_out_cap, outb + 256))) return rc;
    if ((rc = grow(ctx, &ctx->d_dec_meta, &ctx->dec_meta_cap, meta.size() * 8))) return rc;
    {
        std::vector<size_t> lens(n);
        for (size_t i = 0; i < n; i++) {
            lens[i] = src_sizes[i];
            if (encode && src_sizes[i] > ENC_MAX_CHUNK) { ss[i] = ENC_MAX_CHUNK + 1; lens[i] = 0; }   // reported as too big
        }
        if ((rc = gather_h2d(ctx, srcs, lens.data(), so, n, ctx->d_dec_in, (size_t)inb, st))) return rc;
    }
    CK(cudaMemcpyAsync(ctx->d_dec_meta, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, st));
    uint64_t *dm = reinterpret_cast<uint64_t *>(ctx->d_dec_meta);
    uint32_t *d_ss = reinterpret_cast<uint32_t *>(dm + 3 * n);
    int64_t *d_res = reinterpret_cast<int64_t *>(dm + 2 * n);
    if (encode)
        rc = b2c_s2_encode_device(ctx, level, flags, ctx->d_dec_in, ENC_MAX_CHUNK, d_ss, 0, ctx->d_dec_out, kSlot, d_res,
                                  (uint32_t)n, st);
    else {
        S2DecParams P;
        memset(&P, 0, sizeof(P));
        P.src_base = ctx->d_dec_in; P.src_offsets = dm; P.src_sizes = d_ss;
        P.dst_base = ctx->d_dec_out; P.dst_offsets = dm + n; P.dst_caps = d_ss + n;
        P.out_sizes = d_res; P.nchunks = (uint32_t)n;
        rc = launch_s2_decode(ctx, P, inb, st);
    }
    if (rc) return rc;
    CK(cudaMemcpyAsync(sizes_out, d_res, n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    {
        std::vector<size_t> lens(n, 0);
        for (size_t i = 0; i < n; i++) {
            if (sizes_out[i] > 0 && (size_t)sizes_out[i] > dst_caps[i]) { sizes_out[i] = B2C_ERR_DST_SMALL; continue; }
            if (sizes_out[i] > 0) lens[i] = (size_t)sizes_out[i];
        }
        if ((rc = scatter_d2h(ctx, dsts, lens.data(), dof, n, ctx->d_dec_out, (size_t)outb, st))) return rc;
    }
    return B2C_OK;
}

int b2c_s2_encode_chunks(b2c_ctx *ctx, int level, int flags, const void *const *srcs, const size_t *src_sizes,
                         void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    if (level != B2C_S2_FAST && level != B2C_S2_BETTER) return ctx ? B2C_ERR_UNSUPPORTED : B2C_ERR_NO_DEVICE;
    return s2_host_batch(ctx, true, level, flags, srcs, src_sizes, dsts, dst_caps, sizes_out, n);
}
int b2c_s2_decode_chunks(b2c_ctx *ctx, const void *const *srcs, const size_t *src_sizes, void *const *dsts,
                         const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    return s2_host_batch(ctx, false, 0, 0, srcs, src_sizes, dsts, dst_caps, sizes_out, n);
}


// ---- standalone huff0 blocks ------------------------------------------------------------------------
int b2c_huf_compress_device(b2c_ctx *ctx, int flags, const void *d_src, size_t src_stride, const uint32_t *d_sizes,
                            uint32_t size_all, void *d_dst, size_t dst_stride, int64_t *d_out_sizes, uint32_t nchunks,
                            void *stream) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (nchunks == 0) return B2C_OK;
    if ((dst_stride & 3) || (reinterpret_cast<uintptr_t>(d_dst) & 3) || dst_stride > 0xffffffffull) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    Huf0Params P;
    memset(&P, 0, sizeof(P));
    P.src_base = (const uint8_t *)d_src; P.src_stride = src_stride; P.src_sizes = d_sizes; P.src_size_all = size_all;
    P.dst_base = (uint8_t *)d_dst; P.dst_stride = dst_stride; P.dst_cap = (uint32_t)dst_stride;
    P.out_sizes = d_out_sizes; P.nchunks = nchunks; P.flags = (flags & B2C_HUF_4X) ? HUF0_FLAG_4X : 0;
    unsigned grid = (unsigned)ctx->sm_count * 2 < nchunks ? (unsigned)ctx->sm_count * 2 : nchunks;
    b2c_huf_compress_kernel<<<grid, HUF0_NT, HUF0_SMEM_BYTES, (cudaStream_t)stream>>>(P);
    ctx->launches += 1;
    CK(cudaGetLastError());
    return B2C_OK;
}

int b2c_huf_decompress_device(b2c_ctx *ctx, int flags, const void *d_src, size_t src_stride, const uint32_t *d_src_sizes,
                              void *d_dst, size_t dst_stride, const uint32_t *d_dst_sizes, int64_t *d_out_sizes,
                              uint32_t nchunks, void *stream) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (!d_src_sizes || !d_dst_sizes || !d_out_sizes) return B2C_ERR_ARG;
    if (nchunks == 0) return B2C_OK;
    CK(cudaSetDevice(ctx->device));
    Huf0Params P;
    memset(&P, 0, sizeof(P));
    P.src_base = (const uint8_t *)d_src; P.src_stride = src_stride; P.src_sizes = d_src_sizes;
    P.dst_base = (uint8_t *)d_dst; P.dst_stride = dst_stride; P.dst_sizes = d_dst_sizes;
    P.out_sizes = d_out_sizes; P.nchunks = nchunks; P.flags = (flags & B2C_HUF_4X) ? HUF0_FLAG_4X : 0;
    const unsigned ctasPerSm = (227u * 1024u) / (DEC_SMEM_BYTES + 1024u);
    unsigned grid = (nchunks + DEC_WARPS - 1) / DEC_WARPS, maxGrid = (unsigned)ctx->sm_count * (ctasPerSm ? ctasPerSm : 1);
    if (grid > maxGrid) grid = maxGrid;
    cudaStream_t st = (cudaStream_t)stream;
    // Staged form (the default): table pass -> the staged zstd decoder's literal-stream kernel -> the one-warp kernel over what
    // is left (errors, unusual blocks).  B2C_DEC=onewarp, very large batches and unaligned slots keep the one-warp kernel alone.
    const bool staged = ctx->dec_staged && nchunks <= (1u << 20) && (dst_stride & 3) == 0;
    if (staged) {
        const size_t recBytes = (((size_t)nchunks * sizeof(FdChunk)) + 255) & ~(size_t)255;
        const size_t blkBytes = (((size_t)nchunks * sizeof(FdBlock)) + 255) & ~(size_t)255;
        const size_t hufBytes = (size_t)nchunks * 2048 * sizeof(uint16_t);
        { int r = ctx_order_begin(ctx, st); if (r) return r; }
        int rc = grow(ctx, &ctx->d_fd, &ctx->fd_cap, recBytes + blkBytes + hufBytes);
        if (rc) return rc;
        P.fd = reinterpret_cast<FdChunk *>(ctx->d_fd);
        P.fd_blk = reinterpret_cast<FdBlock *>(ctx->d_fd + recBytes);
        P.fd_huf = reinterpret_cast<uint16_t *>(ctx->d_fd + recBytes + blkBytes);
        b2c_huf_dec_prep_kernel<<<grid, DEC_WARPS * 32, DEC_SMEM_BYTES, st>>>(P);
        ZstdDecParams Z;
        memset(&Z, 0, sizeof(Z));
        Z.src_base = P.src_base; Z.src_stride = src_stride; Z.src_sizes = d_src_sizes;
        Z.dst_base = P.dst_base; Z.dst_stride = dst_stride; Z.out_sizes = d_out_sizes; Z.nchunks = nchunks;
        Z.fd = P.fd; Z.fd_blk = P.fd_blk; Z.fd_maxb = 1; Z.fd_per_block = 0; Z.fd_huf = P.fd_huf; Z.fd_lits = P.dst_base; Z.fd_lit_stride = dst_stride;
        const unsigned groups = (nchunks + FD_LIT_GROUP - 1) / FD_LIT_GROUP;
        b2c_zstd_dec_lit_kernel<<<(groups + FD_LIT_WARPS - 1) / FD_LIT_WARPS, FD_LIT_WARPS * 32, FD_LIT_WARPS * FD_LIT_WARP_BYTES, st>>>(Z);
        ctx->launches += 2;
    }
    b2c_huf_decompress_kernel<<<grid, DEC_WARPS * 32, DEC_SMEM_BYTES, st>>>(P);
    ctx->launches += 1;
    CK(cudaGetLastError());
    if (staged) return ctx_order_end(ctx, st);
    return B2C_OK;
}

// Host-buffer batches for the standalone huff0 calls (huff0.Compress4X / Compress1X, Decoder.Decompress4X / 1X, ReadTable
// per element): inputs are packed into equal slots on the device, one kernel per call, results copied back.
//   op 0: compress (dst_caps = capacities), op 1: decompress (dst_caps = EXACT decoded sizes), op 2: read table
//   (dsts[i] receives the 260-byte row described in include/b2c.h)
static int huf_host_batch(b2c_ctx *ctx, int op, int flags, const void *const *srcs, const size_t *src_sizes,
                          void *const *dsts, const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    if (!ctx) return B2C_ERR_NO_DEVICE;
    if (n == 0) return B2C_OK;
    if (n > 0xffffffffull) return B2C_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    size_t maxIn = 16, maxOut = 16;
    for (size_t i = 0; i < n; i++) {
        if (src_sizes[i] > 0x7fffffffull) return B2C_ERR_ARG;
        if (src_sizes[i] > maxIn) maxIn = src_sizes[i];
        const size_t want = op == 2 ? 260 : (op == 0 ? (dst_caps[i] < src_sizes[i] ? dst_caps[i] : src_sizes[i]) : dst_caps[i]);
        if (want > maxOut) maxOut = want;
    }
    if (op == 1 && maxOut > 262144) maxOut = 262144;      // larger exact sizes are refused by the kernel (ErrTooBig class)
    const size_t inStride = (maxIn + 15) & ~(size_t)15, outStride = (maxOut + 15) & ~(size_t)15;
    // meta: out_sizes[n] i64 | src_sizes[n] u32 | dst_sizes[n] u32
    std::vector<uint64_t> meta(2 * n);
    uint32_t *ss = reinterpret_cast<uint32_t *>(meta.data() + n), *ds = ss + n;
    for (size_t i = 0; i < n; i++) { ss[i] = (uint32_t)src_sizes[i]; ds[i] = (uint32_t)(dst_caps[i] > 0xffffffffull ? 0xffffffffull : dst_caps[i]); }
    int rc;
    if ((rc = grow(ctx, &ctx->d_dec_in, &ctx->dec_in_cap, n * inStride + 256))) return rc;
    if ((rc = grow(ctx, &ctx->d_dec_out, &ctx->dec_out_cap, n * outStride + 256))) return rc;
    if ((rc = grow(ctx, &ctx->d_dec_meta, &ctx->dec_meta_cap, meta.size() * 8))) return rc;
    for (size_t i = 0; i < n; i++)
        if (src_sizes[i]) CK(cudaMemcpyAsync(ctx->d_dec_in + i * inStride, srcs[i], src_sizes[i], cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_dec_meta, meta.data(), meta.size() * 8, cudaMemcpyHostToDevice, st));
    uint64_t *dm = reinterpret_cast<uint64_t *>(ctx->d_dec_meta);
    int64_t *d_res = reinterpret_cast<int64_t *>(dm);
    uint32_t *d_ss = reinterpret_cast<uint32_t *>(dm + n), *d_ds = d_ss + n;
    if (op == 0)
        rc = b2c_huf_compress_device(ctx, flags, ctx->d_dec_in, inStride, d_ss, 0, ctx->d_dec_out, outStride, d_res, (uint32_t)n, st);
    else if (op == 1)
        rc = b2c_huf_decompress_device(ctx, flags, ctx->d_dec_in, inStride, d_ss, ctx->d_dec_out, outStride, d_ds, d_res, (uint32_t)n, st);
    else {
        Huf0Params P;
        memset(&P, 0, sizeof(P));
        P.src_base = ctx->d_dec_in; P.src_stride = inStride; P.src_sizes = d_ss;
        P.dst_base = ctx->d_dec_out; P.dst_stride = outStride; P.out_sizes = d_res; P.nchunks = (uint32_t)n;
        const unsigned ctasPerSm = (227u * 1024u) / (DEC_SMEM_BYTES + 1024u);
        unsigned grid = ((unsigned)n + DEC_WARPS - 1) / DEC_WARPS, maxGrid = (unsigned)ctx->sm_count * (ctasPerSm ? ctasPerSm : 1);
        if (grid > maxGrid) grid = maxGrid;
        b2c_huf_read_table_kernel<<<grid, DEC_WARPS * 32, DEC_SMEM_BYTES, st>>>(P);
        ctx->launches += 1;
        CK(cudaGetLastError());
        rc = B2C_OK;
    }
    if (rc) return rc;
    CK(cudaMemcpyAsync(sizes_out, d_res, n * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    for (size_t i = 0; i < n; i++) {
        if (sizes_out[i] < 0) continue;
        const size_t bytes = op == 2 ? 260 : (size_t)sizes_out[i];
        if (op == 0 && bytes > dst_caps[i]) { sizes_out[i] = B2C_ERR_DST_SMALL; continue; }
        if (bytes) CK(cudaMemcpyAsync(dsts[i], ctx->d_dec_out + i * outStride, bytes, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return B2C_OK;
}
int b2c_huf_compress_chunks(b2c_ctx *ctx, int flags, const void *const *srcs, const size_t *src_sizes, void *const *dsts,
                            const size_t *dst_caps, int64_t *sizes_out, size_t n) {
    return huf_host_batch(ctx, 0, flags, srcs, src_sizes, dsts, dst_caps, sizes_out, n);
}
int b2c_huf_decompress_chunks(b2c_ctx *ctx, int flags, const void *const *srcs, const size_t *src_sizes, void *const *dsts,
                              const size_t *dst_sizes, int64_t *sizes_out, size_t n) {
    return huf_host_batch(ctx, 1, flags, srcs, src_sizes, dsts, dst_sizes, sizes_out, n);
}
int b2c_huf_read_table(b2c_ctx *ctx, const void *const *srcs, const size_t *src_sizes, void *const *rows, int64_t *sizes_out, size_t n) {
    std::vector<size_t> caps(n, 260);
    return huf_host_batch(ctx, 2, 0, srcs, src_sizes, rows, caps.data(), sizes_out, n);
}

// ---- coalescing queue ---------------------------------------------------------------------------------------------
// The reference's seams are one block per call from many goroutines at once: zstd.Encoder.EncodeAll "can be called
// concurrently" (zstd/encoder.go:717-729), s2.WriterCustomEncoder's hook runs on one goroutine per block
// (s2/writer.go:1052-1064, call sites :455-461), Decoder.DecodeAll likewise.  A GPU wants batches.  b2c_queue is the
// piece of the shim that turns the former into the latter: callers block in b2c_queue_*; one dispatcher thread owns
// the context, collects what is pending (lingering a few microseconds for stragglers), issues ONE *_chunks call per
// kind of request and wakes the callers with their results.  Caller memory is only touched during the call.
struct b2c_req {
    int op, level, flags;                 // op: 0 zstd encode, 1 s2 encode, 2 zstd decode, 3 s2 decode
    const void *src; size_t n; void *dst; size_t cap;
    int64_t result; bool done;
};
struct b2c_queue {
    b2c_ctx *ctx = nullptr;
    size_t max_batch = 0;
    unsigned linger_us = 0;
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    std::deque<b2c_req *> pending;
    bool stop = false;
    std::thread worker;
    std::atomic<uint64_t> calls{0}, batches{0};
};

static void queue_run_batch(b2c_queue *q, std::vector<b2c_req *> &grp) {
    const size_t m = grp.size();
    std::vector<const void *> srcs(m);
    std::vector<void *> dsts(m);
    std::vector<size_t> ssz(m), dcap(m);
    std::vector<int64_t> res(m, 0);
    for (size_t i = 0; i < m; i++) { srcs[i] = grp[i]->src; ssz[i] = grp[i]->n; dsts[i] = grp[i]->dst; dcap[i] = grp[i]->cap; }
    const b2c_req *r0 = grp[0];
    int rc;
    switch (r0->op) {
    case 0: {
        // EncodeAll: inputs of at most one block are single-block frames (encode_chunks); larger ones go through frame mode
        // (one multi-block frame each), both as one device batch
        const size_t blk = level_ok(r0->level) ? level_block(r0->level) : 0;
        std::vector<size_t> big, small;
        for (size_t i = 0; i < m; i++) (ssz[i] > blk ? big : small).push_back(i);
        rc = B2C_OK;
        for (int pass = 0; pass < 2 && rc == B2C_OK; pass++) {
            const std::vector<size_t> &ix = pass ? big : small;
            if (ix.empty()) continue;
            const size_t k = ix.size();
            std::vector<const void *> s2(k); std::vector<void *> d2(k); std::vector<size_t> z2(k), c2(k); std::vector<int64_t> r2(k, 0);
            for (size_t j = 0; j < k; j++) { s2[j] = srcs[ix[j]]; d2[j] = dsts[ix[j]]; z2[j] = ssz[ix[j]]; c2[j] = dcap[ix[j]]; }
            rc = pass ? b2c_zstd_encode_frames(q->ctx, r0->level, r0->flags & B2C_ZSTD_CRC, s2.data(), z2.data(), d2.data(), c2.data(), r2.data(), k)
                      : b2c_zstd_encode_chunks(q->ctx, r0->level, r0->flags, s2.data(), z2.data(), d2.data(), c2.data(), r2.data(), k);
            for (size_t j = 0; j < k; j++) res[ix[j]] = r2[j];
        }
        break;
    }
    case 1: rc = b2c_s2_encode_chunks(q->ctx, r0->level, r0->flags, srcs.data(), ssz.data(), dsts.data(), dcap.data(), res.data(), m); break;
    case 2: rc = b2c_zstd_decode_chunks(q->ctx, srcs.data(), ssz.data(), dsts.data(), dcap.data(), res.data(), m); break;
    default: rc = b2c_s2_decode_chunks(q->ctx, srcs.data(), ssz.data(), dsts.data(), dcap.data(), res.data(), m); break;
    }
    for (size_t i = 0; i < m; i++) grp[i]->result = rc ? (int64_t)rc : res[i];
    q->batches++;
}

static void queue_worker(b2c_queue *q) {
    cudaSetDevice(q->ctx->device);
    std::unique_lock<std::mutex> lk(q->mu);
    for (;;) {
        q->cv_work.wait(lk, [&] { return q->stop || !q->pending.empty(); });
        if (q->pending.empty()) { if (q->stop) return; continue; }
        if (q->linger_us && q->pending.size() < q->max_batch && !q->stop)   // give concurrent callers a moment to arrive
            q->cv_work.wait_for(lk, std::chrono::microseconds(q->linger_us), [&] { return q->stop || q->pending.size() >= q->max_batch; });
        std::vector<b2c_req *> take;
        while (!q->pending.empty() && take.size() < q->max_batch) { take.push_back(q->pending.front()); q->pending.pop_front(); }
        lk.unlock();
        // one device batch per kind of request, in arrival order of the kinds
        std::vector<char> used(take.size(), 0);
        for (size_t i = 0; i < take.size(); i++) {
            if (used[i]) continue;
            std::vector<b2c_req *> grp;
            for (size_t j = i; j < take.size(); j++)
                if (!used[j] && take[j]->op == take[i]->op && take[j]->level == take[i]->level && take[j]->flags == take[i]->flags) {
                    grp.push_back(take[j]); used[j] = 1;
                }
            queue_run_batch(q, grp);
        }
        lk.lock();
        for (b2c_req *r : take) r->done = true;
        q->cv_done.notify_all();
    }
}

static int64_t queue_call(b2c_queue *q, int op, int level, int flags, const void *src, size_t n, void *dst, size_t cap) {
    if (!q) return B2C_ERR_NO_DEVICE;
    b2c_req r{op, level, flags, src, n, dst, cap, 0, false};
    std::unique_lock<std::mutex> lk(q->mu);
    if (q->stop) return B2C_ERR_ARG;
    q->pending.push_back(&r);
    q->calls++;
    q->cv_work.notify_one();
    q->cv_done.wait(lk, [&] { return r.done; });
    return r.result;
}

b2c_queue *b2c_queue_create(int device, size_t max_batch, unsigned linger_us) {
    if (max_batch == 0) max_batch = 1024;
    b2c_ctx *ctx = b2c_ctx_create(device, max_batch);
    if (!ctx) return nullptr;
    b2c_queue *q = new b2c_queue();
    q->ctx = ctx; q->max_batch = max_batch; q->linger_us = linger_us;
    q->worker = std::thread(queue_worker, q);
    return q;
}
void b2c_queue_destroy(b2c_queue *q) {
    if (!q) return;
    { std::lock_guard<std::mutex> lk(q->mu); q->stop = true; }
    q->cv_work.notify_all();
    if (q->worker.joinable()) q->worker.join();
    b2c_ctx_destroy(q->ctx);
    delete q;
}
int64_t b2c_queue_zstd_encode(b2c_queue *q, int level, int flags, const void *src, size_t n, void *dst, size_t cap) {
    return queue_call(q, 0, level, flags, src, n, dst, cap);
}
int64_t b2c_queue_s2_encode(b2c_queue *q, int level, int flags, const void *src, size_t n, void *dst, size_t cap) {
    return queue_call(q, 1, level, flags, src, n, dst, cap);
}
int64_t b2c_queue_zstd_decode(b2c_queue *q, const void *src, size_t n, void *dst, size_t cap) {
    return queue_call(q, 2, 0, 0, src, n, dst, cap);
}
int64_t b2c_queue_s2_decode(b2c_queue *q, const void *src, size_t n, void *dst, size_t cap) {
    return queue_call(q, 3, 0, 0, src, n, dst, cap);
}
int b2c_queue_stats(b2c_queue *q, uint64_t *calls, uint64_t *batches) {
    if (!q) return B2C_ERR_NO_DEVICE;
    if (calls) *calls = q->calls.load();
    if (batches) *batches = q->batches.load();
    return B2C_OK;
}

}  // extern "C"
