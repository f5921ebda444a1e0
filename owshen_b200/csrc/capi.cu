// owshen_b200/csrc/capi.cu -- the extern "C" boundary declared in include/owshen_b200.h.
// Host-pointer entry points stage their buffers in persistent device slots (H2D/D2H on the ctx
// stream, truly asynchronous when the caller's memory is pinned) and return after the result has
// landed; `_dev` entry points only enqueue.  No entry point has a CPU implementation.
#include "common.cuh"
#include "groth16.cuh"
#include "mimc.cuh"
#include "msm.cuh"
#include "ntt.cuh"
#include "withdraw_circuit.hpp"

using namespace og;

void* og_ctx::slot(int id, size_t bytes) {
    if (bytes == 0) bytes = 32;
    if (slot_cap[id] >= bytes) return slot_ptr[id];
    cudaDeviceSynchronize();          // growth is rare; work already enqueued may still be using the old buffer
    if (slot_ptr[id]) cudaFree(slot_ptr[id]);
    slot_ptr[id] = nullptr; slot_cap[id] = 0;
    size_t cap = bytes + bytes / 8;
    cudaError_t e = cudaMalloc(&slot_ptr[id], cap);
    if (e != cudaSuccess) {
        e = cudaMalloc(&slot_ptr[id], bytes);
        cap = bytes;
    }
    if (e != cudaSuccess) {
        snprintf(err, sizeof(err), "slot %d: cudaMalloc(%zu) failed: %s", id, bytes, cudaGetErrorString(e));
        slot_ptr[id] = nullptr;
        return nullptr;
    }
    slot_cap[id] = cap;
    return slot_ptr[id];
}

cudaEvent_t og_ctx::prof_event() {
    if (!ev_pool.empty()) { cudaEvent_t e = ev_pool.back(); ev_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

namespace og {
int32_t clear_flag(og_ctx* ctx) {
    OG_CUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), ctx->stream));
    return OG_OK;
}
int32_t check_flag(og_ctx* ctx) {
    OG_CUDA(ctx, cudaMemcpyAsync(ctx->h_flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    OG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (*ctx->h_flag) { snprintf(ctx->err, sizeof(ctx->err), "non-canonical field element in input"); return OG_E_ENCODING; }
    return OG_OK;
}
}  // namespace og

// every entry point that takes a ctx first makes its device current: several contexts (one per GPU) may live in
// one process (INTEGRATION.md: one Prover per GPU), and launches go to the calling thread's current device
#define OG_ENTER(ctx)                                                                              \
    do {                                                                                           \
        if (!(ctx)) return OG_E_INVALID;                                                           \
        OG_CUDA(ctx, cudaSetDevice((ctx)->device));                                                \
    } while (0)

// a proving key's tables are device memory of the GPU it was loaded on: refuse it on any other context's GPU
#define OG_PK_CHECK(ctx, pk)                                                                           \
    do {                                                                                               \
        if (!pk_on_device_of(pk, ctx)) {                                                               \
            snprintf((ctx)->err, sizeof((ctx)->err), "proving key was loaded on another device");      \
            return OG_E_INVALID;                                                                       \
        }                                                                                              \
    } while (0)

#define H2D(ctx, dst, src, bytes) OG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, (ctx)->stream))
#define D2H(ctx, dst, src, bytes) OG_CUDA(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, (ctx)->stream))

// ---- the G1 / G2 entry points, written once over the coordinate field F (Fq: G1, Fq2: G2) --------------------------
// A point crosses the boundary as 2 * sizeof(F) bytes (x, y canonical), the size of its affine Montgomery form.
template <class F>
static int32_t msm_dev_entry(og_ctx* ctx, const uint8_t* d_points, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out) {
    OG_ENTER(ctx);
    if (!ctx || !d_out || (n && (!d_points || !d_scalars))) return OG_E_INVALID;
    return msm_dev<F>(ctx, d_points, d_scalars, n, d_out);
}
template <class F>
static int32_t msm_host_entry(og_ctx* ctx, const uint8_t* points, const uint8_t* scalars, uint64_t n, uint8_t* out) {
    constexpr uint64_t PB = sizeof(Affine<F>);
    OG_ENTER(ctx);
    if (!ctx || !out || (n && (!points || !scalars))) return OG_E_INVALID;
    OG_SLOT(ctx, dp, uint8_t, S_IO_A, PB * n);
    OG_SLOT(ctx, ds, uint8_t, S_IO_B, 32 * n);
    OG_SLOT(ctx, dout, uint8_t, S_IO_C, PB);
    OG_TRY(clear_flag(ctx));
    if (n) { H2D(ctx, dp, points, PB * n); H2D(ctx, ds, scalars, 32 * n); }
    OG_TRY(msm_dev<F>(ctx, dp, ds, n, dout));
    D2H(ctx, out, dout, PB);
    return check_flag(ctx);
}
template <class F>
static int32_t sum_host_entry(og_ctx* ctx, const uint8_t* points, uint64_t n, uint8_t* out) {
    constexpr uint64_t PB = sizeof(Affine<F>);
    OG_ENTER(ctx);
    if (!ctx || !out || (n && !points)) return OG_E_INVALID;
    OG_SLOT(ctx, dp, uint8_t, S_IO_A, PB * n);
    OG_SLOT(ctx, dout, uint8_t, S_IO_C, PB);
    OG_TRY(clear_flag(ctx));
    if (n) H2D(ctx, dp, points, PB * n);
    OG_TRY(sum_points_dev<F>(ctx, dp, n, dout));
    D2H(ctx, out, dout, PB);
    return check_flag(ctx);
}
template <class F>
static int32_t sum_dev_entry(og_ctx* ctx, const uint8_t* d_points, uint64_t n, uint8_t* d_out) {
    OG_ENTER(ctx);
    if (!d_out || (n && !d_points)) return OG_E_INVALID;
    return sum_points_dev<F>(ctx, d_points, n, d_out);
}
template <class F>
static int32_t generator_mul_dev_entry(og_ctx* ctx, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out_points) {
    OG_ENTER(ctx);
    if (n && (!d_scalars || !d_out_points)) return OG_E_INVALID;
    if (n == 0) return OG_OK;
    OG_SLOT(ctx, dp, Affine<F>, S_IO_B, sizeof(Affine<F>) * n);
    OG_TRY(fixed_base_mul(ctx, d_scalars, n, dp));
    return points_to_bytes(ctx, dp, n, d_out_points);
}
template <class F>
static int32_t generator_mul_host_entry(og_ctx* ctx, const uint8_t* scalars, uint64_t n, uint8_t* out_points) {
    constexpr uint64_t PB = sizeof(Affine<F>);
    OG_ENTER(ctx);
    if (!ctx || (n && (!scalars || !out_points))) return OG_E_INVALID;
    if (n == 0) return OG_OK;
    OG_SLOT(ctx, ds, uint8_t, S_IO_A, 32 * n);
    OG_SLOT(ctx, dp, Affine<F>, S_IO_B, sizeof(Affine<F>) * n);
    OG_SLOT(ctx, dout, uint8_t, S_IO_C, PB * n);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, ds, scalars, 32 * n);
    OG_TRY(fixed_base_mul(ctx, ds, n, dp));
    OG_TRY(points_to_bytes(ctx, dp, n, dout));
    D2H(ctx, out_points, dout, PB * n);
    return check_flag(ctx);
}

extern "C" {

int32_t og_abi_version(void) { return 1; }

const char* og_strerror(int32_t code) {
    switch (code) {
        case OG_OK: return "ok";
        case OG_E_INVALID: return "invalid argument";
        case OG_E_ENCODING: return "malformed or non-canonical encoding";
        case OG_E_NO_DEVICE: return "no usable CUDA device (this library has no CPU path)";
        case OG_E_CUDA: return "CUDA runtime error";
        case OG_E_NOMEM: return "out of device memory";
        case OG_E_VERIFY: return "proof does not verify";
        default: return "unknown error";
    }
}
const char* og_last_error(const og_ctx* ctx) { return ctx ? ctx->err : ""; }

int32_t og_init(int32_t device, og_ctx** out) {
    if (!out) return OG_E_INVALID;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) return OG_E_NO_DEVICE;
    if (cudaSetDevice(device) != cudaSuccess) return OG_E_NO_DEVICE;
    og_ctx* ctx = new og_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
        cudaMalloc(&ctx->d_flag, sizeof(int)) != cudaSuccess || cudaMallocHost(&ctx->h_flag, sizeof(int)) != cudaSuccess) {
        delete ctx;
        return OG_E_CUDA;
    }
    cudaMemset(ctx->d_flag, 0, sizeof(int));
    int32_t rc = mimc_init(ctx);
    if (rc != OG_OK) { og_free(ctx); return rc; }
    *out = ctx;
    return OG_OK;
}

void og_free(og_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (int i = 0; i < N_SLOTS; i++) if (ctx->slot_ptr[i]) cudaFree(ctx->slot_ptr[i]);
    ntt_free_tables(ctx);
    if (ctx->g1_fixed) cudaFree(ctx->g1_fixed);
    if (ctx->g2_fixed) cudaFree(ctx->g2_fixed);
    if (ctx->bjj_fixed) cudaFree(ctx->bjj_fixed);
    if (ctx->d_flag) cudaFree(ctx->d_flag);
    if (ctx->h_flag) cudaFreeHost(ctx->h_flag);
    for (auto& r : ctx->prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

int32_t og_sync(og_ctx* ctx) {
    OG_ENTER(ctx);
    if (!ctx) return OG_E_INVALID;
    OG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return OG_OK;
}
int32_t og_stream(og_ctx* ctx, void** out_cuda_stream) {
    if (!ctx || !out_cuda_stream) return OG_E_INVALID;
    *out_cuda_stream = (void*)ctx->stream;
    return OG_OK;
}
int32_t og_timer_start(og_ctx* ctx) {
    OG_ENTER(ctx);
    if (!ctx) return OG_E_INVALID;
    OG_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    return OG_OK;
}
int32_t og_timer_stop(og_ctx* ctx, float* ms) {
    OG_ENTER(ctx);
    if (!ctx || !ms) return OG_E_INVALID;
    OG_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    OG_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
    OG_CUDA(ctx, cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
    return OG_OK;
}
uint64_t og_launch_count(const og_ctx* ctx) { return ctx ? ctx->launches : 0; }

int32_t og_profile(og_ctx* ctx, int32_t enable) {
    OG_ENTER(ctx);
    if (!ctx) return OG_E_INVALID;
    ctx->prof_on = enable != 0;
    return OG_OK;
}
// "name,launches,total_ms\n" per kernel since the last dump; synchronises the stream
int32_t og_profile_dump(og_ctx* ctx, char* buf, uint64_t cap) {
    OG_ENTER(ctx);
    if (!ctx || !buf || cap == 0) return OG_E_INVALID;
    OG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    struct Agg { const char* name; uint64_t n; double ms; };
    std::vector<Agg> agg;
    for (auto& r : ctx->prof) {
        float ms = 0;
        cudaEventElapsedTime(&ms, r.a, r.b);
        size_t k = 0;
        for (; k < agg.size(); k++) if (strcmp(agg[k].name, r.name) == 0) break;
        if (k == agg.size()) agg.push_back({r.name, 0, 0.0});
        agg[k].n++; agg[k].ms += ms;
        ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b);
    }
    ctx->prof.clear();
    uint64_t off = 0;
    buf[0] = 0;
    for (auto& a : agg) {
        int w = snprintf(buf + off, cap - off, "%s,%llu,%.6f\n", a.name, (unsigned long long)a.n, a.ms);
        if (w < 0 || (uint64_t)w >= cap - off) break;
        off += (uint64_t)w;
    }
    return OG_OK;
}

// ---- field probes --------------------------------------------------------------------------------------
}  // extern "C"

namespace og {
template <class F>
__global__ void __launch_bounds__(128) k_field_op(int op, const uint8_t* __restrict__ a, const uint8_t* __restrict__ b, uint64_t n,
                                                  uint8_t* __restrict__ out, int* flag) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    F x = load_canonical<F>(a + 32 * i, flag), y = load_canonical<F>(b + 32 * i, flag);
    F r = op == 0 ? x * y : (op == 1 ? x + y : x - y);
    store_canonical(out + 32 * i, r);
}

// integer-pipe micro-benchmark.  Every multiply-add takes its own accumulator as a multiplicand, so ptxas
// cannot hoist the product out of the loop (an earlier version with loop-invariant multiplicands was
// strength-reduced to additions and measured the ALU pipe instead).  MODE 0: mad.lo.u32 (IMAD),
// MODE 1: mad.wide.u32 (IMAD.WIDE), MODE 2: mad.lo.cc/madc.hi.cc pairs in 4-pair carry chains, the
// shape of one Montgomery row (IMAD.WIDE.U32.X); a pair counts as ONE 32x32->64 multiply-add.
template <int MODE>
__global__ void __launch_bounds__(256) k_imad(uint32_t* out, uint32_t iters, uint32_t seed) {
    uint32_t x = blockIdx.x * 2654435761u + 12345u + seed, y = x ^ 0x9e3779b9u;
    if (MODE == 0) {
        uint32_t w[8];
#pragma unroll
        for (int k = 0; k < 8; k++) w[k] = threadIdx.x * (2 * k + 3) + seed;
        for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
            for (int r = 0; r < 8; r++)
#pragma unroll
                for (int k = 0; k < 8; k++) asm volatile("mad.lo.u32 %0, %0, %1, %2;" : "+r"(w[k]) : "r"(x), "r"(y));
        }
        uint32_t s = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) s ^= w[k];
        if (s == 0x1234567u) out[0] = s;
    } else if (MODE == 1) {
        unsigned long long w[8];
#pragma unroll
        for (int k = 0; k < 8; k++) w[k] = threadIdx.x * (2 * k + 3) + seed;
        for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
            for (int r = 0; r < 8; r++)
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    uint32_t lo = (uint32_t)w[k];
                    asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(w[k]) : "r"(lo), "r"(x));
                }
        }
        unsigned long long s = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) s ^= w[k];
        if (s == 0x1234567ull) out[0] = (uint32_t)s;
    } else {
        uint32_t e[8], o[8];
#pragma unroll
        for (int k = 0; k < 8; k++) { e[k] = threadIdx.x * (2 * k + 3) + seed; o[k] = e[k] ^ y; }
        CC cc;
        for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
            for (int r = 0; r < 4; r++) {
                uint32_t m0 = e[7] | 1u, m1 = o[7] | 1u;      // multiplicand depends on the previous chain
                e[0] = mad_lo_cc(m0, x, e[0], cc); e[1] = madc_hi_cc(m0, x, e[1], cc);
                e[2] = madc_lo_cc(m0, y, e[2], cc); e[3] = madc_hi_cc(m0, y, e[3], cc);
                e[4] = madc_lo_cc(m0, x, e[4], cc); e[5] = madc_hi_cc(m0, x, e[5], cc);
                e[6] = madc_lo_cc(m0, y, e[6], cc); e[7] = madc_hi(m0, y, e[7], cc);
                o[0] = mad_lo_cc(m1, x, o[0], cc); o[1] = madc_hi_cc(m1, x, o[1], cc);
                o[2] = madc_lo_cc(m1, y, o[2], cc); o[3] = madc_hi_cc(m1, y, o[3], cc);
                o[4] = madc_lo_cc(m1, x, o[4], cc); o[5] = madc_hi_cc(m1, x, o[5], cc);
                o[6] = madc_lo_cc(m1, y, o[6], cc); o[7] = madc_hi(m1, y, o[7], cc);
            }
        }
        uint32_t s = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) s ^= e[k] ^ o[k];
        if (s == 0x1234567u) out[0] = s;
    }
}
// latency probe: cycles per DEPENDENT Montgomery multiplication for one warp alone on its scheduler
// (the MiMC chains are exactly this), and with two independent chains interleaved
template <int CHAINS>
__global__ void __launch_bounds__(32) k_mul_latency(Fr* io, uint32_t iters, long long* cycles) {
    Fr x = io[threadIdx.x], y = io[32 + threadIdx.x], k = io[64 + threadIdx.x];
    long long t0 = clock64();
    for (uint32_t i = 0; i < iters; i++) {
        x = x * x + k;
        if (CHAINS == 2) y = y * y + k;
    }
    long long t1 = clock64();
    io[threadIdx.x] = x + y;
    if (threadIdx.x == 0 && blockIdx.x == 0) cycles[0] = (t1 - t0);
}

// FP64 pipe probe (round-2 planning: DFMA-based 52-bit-limb products would run beside the integer pipe)
__global__ void __launch_bounds__(256) k_dfma(double* out, uint32_t iters, double seed) {
    double w[8], x = 1.0000001 + seed * 1e-9, y = 0.9999999;
#pragma unroll
    for (int k = 0; k < 8; k++) w[k] = threadIdx.x * 0.001 + k + seed;
    for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 8; r++)
#pragma unroll
            for (int k = 0; k < 8; k++) w[k] = __fma_rz(w[k], x, y);
    }
    double s = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) s += w[k];
    if (s == 1.2345) out[0] = s;
}

// Hybrid-multiplier probe (round-2 planning).  A 52x52-bit product on the FP64 pipe costs two DFMA, one DADD and
// two 64-bit integer adds (Emmart et al.: hi = fma_rz(a, b, 2^104), lo = fma_rz(a, b, 2^104 + 2^52 - hi), the bit
// patterns accumulate as integers).  MODE 0: those products alone; MODE 1: the carry-chain IMAD.WIDE rows alone;
// MODE 2: both interleaved in every warp -- does the chip run the two multipliers at the same time?
template <int MODE>
__global__ void __launch_bounds__(256) k_hybrid(unsigned long long* out, uint32_t iters, uint32_t seed) {
    const double C1 = 20282409603651670423947251286016.0;                  // 2^104
    const double C2 = 20282409603651670423947251286016.0 + 4503599627370496.0;   // 2^104 + 2^52
    double a[4], b[4];
    long long acc_hi[4] = {0, 0, 0, 0}, acc_lo[4] = {0, 0, 0, 0};
    uint32_t e[8], o[8];
    uint32_t x = blockIdx.x * 2654435761u + 12345u + seed, y = x ^ 0x9e3779b9u;
#pragma unroll
    for (int k = 0; k < 4; k++) { a[k] = (double)((threadIdx.x * 977u + k * 131u + seed) & 0xFFFFF) + 4503599627370.0; b[k] = a[k] * 0.5 + 7.0; }
#pragma unroll
    for (int k = 0; k < 8; k++) { e[k] = threadIdx.x * (2 * k + 3) + seed; o[k] = e[k] ^ y; }
    CC cc;
    for (uint32_t i = 0; i < iters; i++) {
#pragma unroll
        for (int r = 0; r < 4; r++) {
            if (MODE == 0 || MODE == 2) {
#pragma unroll
                for (int k = 0; k < 4; k++) {                                 // 4 products of 52 x 52 bits
                    double hi = __fma_rz(a[k], b[(k + r) & 3], C1);
                    double sub = C2 - hi;
                    double lo = __fma_rz(a[k], b[(k + r) & 3], sub);
                    acc_hi[k] += __double_as_longlong(hi);
                    acc_lo[k] += __double_as_longlong(lo);
                }
                a[r] = a[r] + 1.0;                                            // keep the products loop-variant
            }
            if (MODE == 1 || MODE == 2) {                                     // 8 products of 32 x 32 -> 64 bits (lo and hi halves fuse)
                uint32_t m0 = e[7] | 1u, m1 = o[7] | 1u;
                e[0] = mad_lo_cc(m0, x, e[0], cc); e[1] = madc_hi_cc(m0, x, e[1], cc);
                e[2] = madc_lo_cc(m0, y, e[2], cc); e[3] = madc_hi_cc(m0, y, e[3], cc);
                e[4] = madc_lo_cc(m0, x, e[4], cc); e[5] = madc_hi_cc(m0, x, e[5], cc);
                e[6] = madc_lo_cc(m0, y, e[6], cc); e[7] = madc_hi(m0, y, e[7], cc);
                o[0] = mad_lo_cc(m1, x, o[0], cc); o[1] = madc_hi_cc(m1, x, o[1], cc);
                o[2] = madc_lo_cc(m1, y, o[2], cc); o[3] = madc_hi_cc(m1, y, o[3], cc);
                o[4] = madc_lo_cc(m1, x, o[4], cc); o[5] = madc_hi_cc(m1, x, o[5], cc);
                o[6] = madc_lo_cc(m1, y, o[6], cc); o[7] = madc_hi(m1, y, o[7], cc);
            }
        }
    }
    unsigned long long s = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) s ^= (unsigned long long)acc_hi[k] ^ (unsigned long long)acc_lo[k];
#pragma unroll
    for (int k = 0; k < 8; k++) s ^= e[k] ^ o[k];
    if (s == 0x1234567ull) out[0] = s;
}

}  // namespace og

extern "C" {

// rates[0] = 52x52 FP64-pipe products/s alone, rates[1] = 32x32->64 carry-chain IMAD.WIDE/s alone,
// rates[2], rates[3] = the same two rates when both run interleaved in every warp
int32_t og_hybrid_probe(og_ctx* ctx, double* rates4) {
    OG_ENTER(ctx);
    if (!rates4) return OG_E_INVALID;
    OG_SLOT(ctx, d_out, unsigned long long, S_IO_A, 64);
    const uint32_t iters = 1024, ctas = ctx->sm_count * 8, threads = 256;
    const double lanes = (double)ctas * threads * iters * 4.0;        // 4 rounds per iteration
    float ms[3] = {0, 0, 0};
    for (int mode = 0; mode < 3; mode++) {
        float best = 1e30f, t = 0;
        for (int rep = 0; rep < 4; rep++) {
            OG_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
            if (mode == 0) OG_LAUNCH(ctx, k_hybrid<0>, ctas, threads, 0, d_out, iters, (uint32_t)rep);
            else if (mode == 1) OG_LAUNCH(ctx, k_hybrid<1>, ctas, threads, 0, d_out, iters, (uint32_t)rep);
            else OG_LAUNCH(ctx, k_hybrid<2>, ctas, threads, 0, d_out, iters, (uint32_t)rep);
            OG_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
            OG_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
            OG_CUDA(ctx, cudaEventElapsedTime(&t, ctx->ev0, ctx->ev1));
            if (rep > 0 && t < best) best = t;
        }
        ms[mode] = best;
    }
    rates4[0] = lanes * 4.0 / (ms[0] * 1e-3);
    rates4[1] = lanes * 8.0 / (ms[1] * 1e-3);      // lo+hi of one product fuse into one IMAD.WIDE
    rates4[2] = lanes * 4.0 / (ms[2] * 1e-3);
    rates4[3] = lanes * 8.0 / (ms[2] * 1e-3);
    return OG_OK;
}

int32_t og_mul_latency(og_ctx* ctx, double* cycles_dependent, double* cycles_two_chains) {
    OG_ENTER(ctx);
    if (!ctx || !cycles_dependent || !cycles_two_chains) return OG_E_INVALID;
    OG_SLOT(ctx, io, Fr, S_IO_A, sizeof(Fr) * 96 + 64);
    long long* d_cyc = reinterpret_cast<long long*>(io + 96);
    OG_CUDA(ctx, cudaMemsetAsync(io, 1, sizeof(Fr) * 96, ctx->stream));
    const uint32_t iters = 20000;
    long long h = 0;
    OG_LAUNCH(ctx, k_mul_latency<1>, 1, 32, 0, io, iters, d_cyc);
    OG_CUDA(ctx, cudaMemcpyAsync(&h, d_cyc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    OG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *cycles_dependent = (double)h / iters;
    OG_LAUNCH(ctx, k_mul_latency<2>, 1, 32, 0, io, iters, d_cyc);
    OG_CUDA(ctx, cudaMemcpyAsync(&h, d_cyc, 8, cudaMemcpyDeviceToHost, ctx->stream));
    OG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *cycles_two_chains = (double)h / iters;
    return OG_OK;
}

int32_t og_fp64_peak(og_ctx* ctx, double* dfma_per_s) {
    OG_ENTER(ctx);
    if (!ctx || !dfma_per_s) return OG_E_INVALID;
    OG_SLOT(ctx, d_out, double, S_IO_A, 64);
    const uint32_t iters = 2048, ctas = ctx->sm_count * 8, threads = 256;
    float ms = 0;
    double best = 0;
    for (int rep = 0; rep < 4; rep++) {
        OG_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        OG_LAUNCH(ctx, k_dfma, ctas, threads, 0, d_out, iters, (double)rep);
        OG_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        OG_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
        OG_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
        double rate = (double)ctas * threads * iters * 64.0 / (ms * 1e-3);
        if (rep > 0 && rate > best) best = rate;
    }
    *dfma_per_s = best;
    return OG_OK;
}

int32_t og_imad_peak(og_ctx* ctx, double* mad_per_s, double* wide_mad_per_s) {
    OG_ENTER(ctx);
    if (!ctx || !mad_per_s || !wide_mad_per_s) return OG_E_INVALID;
    double chain = 0;
    return og_int_pipe_peaks(ctx, mad_per_s, wide_mad_per_s, &chain);
}

int32_t og_int_pipe_peaks(og_ctx* ctx, double* mad_per_s, double* wide_mad_per_s, double* carry_chain_wide_per_s) {
    OG_ENTER(ctx);
    if (!ctx || !mad_per_s || !wide_mad_per_s || !carry_chain_wide_per_s) return OG_E_INVALID;
    OG_SLOT(ctx, d_out, uint32_t, S_IO_A, 64);
    const uint32_t iters = 2048, ctas = ctx->sm_count * 8, threads = 256;
    float ms = 0;
    double* outs[3] = {mad_per_s, wide_mad_per_s, carry_chain_wide_per_s};
    const double per_iter[3] = {64.0, 64.0, 32.0};
    for (int mode = 0; mode < 3; mode++) {
        double best = 0;
        for (int rep = 0; rep < 4; rep++) {
            OG_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
            if (mode == 0) OG_LAUNCH(ctx, k_imad<0>, ctas, threads, 0, d_out, iters, (uint32_t)rep);
            else if (mode == 1) OG_LAUNCH(ctx, k_imad<1>, ctas, threads, 0, d_out, iters, (uint32_t)rep);
            else OG_LAUNCH(ctx, k_imad<2>, ctas, threads, 0, d_out, iters, (uint32_t)rep);
            OG_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
            OG_CUDA(ctx, cudaEventSynchronize(ctx->ev1));
            OG_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
            double rate = (double)ctas * threads * iters * per_iter[mode] / (ms * 1e-3);
            if (rep > 0 && rate > best) best = rate;
        }
        *outs[mode] = best;
    }
    return OG_OK;
}

int32_t og_field_op(og_ctx* ctx, int32_t field, int32_t op, const uint8_t* a, const uint8_t* b, uint64_t n, uint8_t* out) {
    OG_ENTER(ctx);
    if (!ctx || !a || !b || !out || field < 0 || field > 1 || op < 0 || op > 2) return OG_E_INVALID;
    if (n == 0) return OG_OK;
    OG_SLOT(ctx, da, uint8_t, S_IO_A, 32 * n);
    OG_SLOT(ctx, db, uint8_t, S_IO_B, 32 * n);
    OG_SLOT(ctx, dout, uint8_t, S_IO_C, 32 * n);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, da, a, 32 * n); H2D(ctx, db, b, 32 * n);
    unsigned grid = (unsigned)((n + 127) / 128);
    if (field == 0) OG_LAUNCH(ctx, k_field_op<Fq>, grid, 128, 0, op, da, db, n, dout, ctx->d_flag);
    else OG_LAUNCH(ctx, k_field_op<Fr>, grid, 128, 0, op, da, db, n, dout, ctx->d_flag);
    D2H(ctx, out, dout, 32 * n);
    return check_flag(ctx);
}

// ---- MiMC7 ----------------------------------------------------------------------------------------------
int32_t og_mimc7_constants(uint8_t* out, uint32_t* n_rounds) {
    if (!out || !n_rounds) return OG_E_INVALID;
    Fr c[MIMC_ROUNDS];
    mimc_constants_host(c);
    for (int i = 0; i < MIMC_ROUNDS; i++) host_store(out + 32 * i, c[i]);
    *n_rounds = MIMC_ROUNDS;
    return OG_OK;
}

int32_t og_mimc7_hash2(og_ctx* ctx, const uint8_t* left, const uint8_t* right, uint64_t n, uint8_t* out) {
    OG_ENTER(ctx);
    if (!ctx || !left || !right || !out) return OG_E_INVALID;
    if (n == 0) return OG_OK;
    OG_SLOT(ctx, da, uint8_t, S_IO_A, 32 * n);
    OG_SLOT(ctx, db, uint8_t, S_IO_B, 32 * n);
    OG_SLOT(ctx, dout, uint8_t, S_IO_C, 32 * n);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, da, left, 32 * n); H2D(ctx, db, right, 32 * n);
    OG_TRY(mimc_hash2_dev(ctx, da, db, n, dout));
    D2H(ctx, out, dout, 32 * n);
    return check_flag(ctx);
}

int32_t og_mimc7_merkle_paths_dev(og_ctx* ctx, const uint8_t* d_leaves, const uint8_t* d_siblings, const uint32_t* d_path_bits,
                                  uint32_t n_paths, uint32_t depth, uint8_t* d_out_nodes) {
    OG_ENTER(ctx);
    if (!ctx || !d_leaves || !d_siblings || !d_path_bits || !d_out_nodes || depth > 32) return OG_E_INVALID;
    return mimc_merkle_paths_dev(ctx, d_leaves, d_siblings, d_path_bits, n_paths, depth, d_out_nodes);
}

int32_t og_mimc7_merkle_paths(og_ctx* ctx, const uint8_t* leaves, const uint8_t* siblings, const uint32_t* path_bits,
                              uint32_t n_paths, uint32_t depth, uint8_t* out_nodes) {
    OG_ENTER(ctx);
    if (!ctx || !leaves || !siblings || !path_bits || !out_nodes || depth > 32) return OG_E_INVALID;
    if (n_paths == 0) return OG_OK;
    size_t nl = 32ull * n_paths, ns = 32ull * n_paths * depth, no = 32ull * n_paths * (depth + 1);
    OG_SLOT(ctx, dl, uint8_t, S_IO_A, nl);
    OG_SLOT(ctx, ds, uint8_t, S_IO_B, ns);
    OG_SLOT(ctx, dbits, uint32_t, S_IO_C, 4ull * n_paths);
    OG_SLOT(ctx, dout, uint8_t, S_IO_D, no);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dl, leaves, nl);
    if (ns) H2D(ctx, ds, siblings, ns);
    H2D(ctx, dbits, path_bits, 4ull * n_paths);
    OG_TRY(mimc_merkle_paths_dev(ctx, dl, ds, dbits, n_paths, depth, dout));
    D2H(ctx, out_nodes, dout, no);
    return check_flag(ctx);
}

int32_t og_mimc7_merkle_build(og_ctx* ctx, const uint8_t* leaves, uint64_t n, uint8_t* out_levels) {
    OG_ENTER(ctx);
    if (!ctx || !leaves || !out_levels || n == 0 || (n & (n - 1)) || n > (1ull << 28)) return OG_E_INVALID;
    uint64_t total = 2 * n - 1;
    OG_SLOT(ctx, din, uint8_t, S_IO_A, 32 * n);
    OG_SLOT(ctx, lv, Fr, S_IO_B, sizeof(Fr) * total);
    OG_SLOT(ctx, dout, uint8_t, S_IO_C, 32 * total);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, din, leaves, 32 * n);
    OG_TRY(mimc_to_mont_dev(ctx, din, n, lv));
    OG_TRY(mimc_tree_build_dev(ctx, lv, n));
    OG_TRY(mimc_from_mont_dev(ctx, lv, total, dout));
    D2H(ctx, out_levels, dout, 32 * total);
    return check_flag(ctx);
}

// nodes of levels 1..depth touched by appending n leaves at index `start` to a depth-`depth` sparse tree: one call, no
// host round trip per level.  Level l contributes ((start+n-1)>>l) - (start>>l) + 1 nodes, lowest index first.
int32_t og_mimc7_merkle_append(og_ctx* ctx, uint32_t depth, uint64_t start, const uint8_t* leaves, uint64_t n, const uint8_t* left_boundary,
                               const uint8_t* zeros, uint8_t* out_nodes) {
    OG_ENTER(ctx);
    if (!ctx || !leaves || !left_boundary || !zeros || !out_nodes || depth == 0 || depth > 32 || n == 0 || n > (1ull << 28)) return OG_E_INVALID;
    if (start + n > (1ull << depth)) return OG_E_INVALID;
    uint64_t total = 0;
    for (uint32_t l = 1; l <= depth; l++) total += ((start + n - 1) >> l) - (start >> l) + 1;
    Fr aux[64];
    for (uint32_t l = 0; l < depth; l++)
        if (!host_load(aux[l], left_boundary + 32 * l) || !host_load(aux[depth + l], zeros + 32 * l)) return OG_E_ENCODING;
    OG_SLOT(ctx, din, uint8_t, S_IO_A, 32 * n);
    OG_SLOT(ctx, nodes, Fr, S_IO_B, sizeof(Fr) * (n + total));
    OG_SLOT(ctx, dout, uint8_t, S_IO_C, 32 * total);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, din, leaves, 32 * n);
    OG_TRY(mimc_to_mont_dev(ctx, din, n, nodes));
    OG_TRY(mimc_tree_append_dev(ctx, depth, start, n, aux, nodes));
    OG_TRY(mimc_from_mont_dev(ctx, nodes + n, total, dout));
    D2H(ctx, out_nodes, dout, 32 * total);
    return check_flag(ctx);
}

// ---- BabyJubJub (the reference's own signature scheme, babyjubjub/mod.rs) -----------------------------------
int32_t og_bjj_verify_batch(og_ctx* ctx, const uint8_t* pk_x, const uint8_t* pk_is_odd, const uint8_t* messages, const uint8_t* signatures,
                            uint32_t n, int32_t hash_kind, uint8_t* out_status) {
    OG_ENTER(ctx);
    if (!ctx || !pk_x || !pk_is_odd || !messages || !signatures || !out_status || hash_kind < 0 || hash_kind > 1) return OG_E_INVALID;
    if (n == 0) return OG_OK;
    OG_SLOT(ctx, dx, uint8_t, S_IO_A, 32ull * n);
    OG_SLOT(ctx, dodd, uint8_t, S_IO_B, n);
    OG_SLOT(ctx, dm, uint8_t, S_IO_C, 32ull * n);
    OG_SLOT(ctx, dsg, uint8_t, S_IO_D, 96ull * n);
    OG_SLOT(ctx, dout, uint8_t, S_IO_E, n);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dx, pk_x, 32ull * n); H2D(ctx, dodd, pk_is_odd, n); H2D(ctx, dm, messages, 32ull * n); H2D(ctx, dsg, signatures, 96ull * n);
    OG_TRY(bjj_verify_dev(ctx, dx, dodd, dm, dsg, n, hash_kind, dout));
    D2H(ctx, out_status, dout, n);
    return check_flag(ctx);
}

int32_t og_bjj_verify_batch_dev(og_ctx* ctx, const uint8_t* d_pk_x, const uint8_t* d_pk_is_odd, const uint8_t* d_messages,
                                const uint8_t* d_signatures, uint32_t n, int32_t hash_kind, uint8_t* d_out_status) {
    OG_ENTER(ctx);
    if (!ctx || hash_kind < 0 || hash_kind > 1 || (n && (!d_pk_x || !d_pk_is_odd || !d_messages || !d_signatures || !d_out_status))) return OG_E_INVALID;
    return bjj_verify_dev(ctx, d_pk_x, d_pk_is_odd, d_messages, d_signatures, n, hash_kind, d_out_status);
}
int32_t og_bjj_sign_batch_dev(og_ctx* ctx, const uint8_t* d_secret_keys, const uint8_t* d_randomness, const uint8_t* d_messages, uint32_t n,
                              int32_t hash_kind, uint8_t* d_out_pk_x, uint8_t* d_out_pk_is_odd, uint8_t* d_out_signatures, uint8_t* d_out_status) {
    OG_ENTER(ctx);
    if (!ctx || hash_kind < 0 || hash_kind > 1 ||
        (n && (!d_secret_keys || !d_randomness || !d_messages || !d_out_pk_x || !d_out_pk_is_odd || !d_out_signatures || !d_out_status))) return OG_E_INVALID;
    return bjj_sign_dev(ctx, d_secret_keys, d_randomness, d_messages, n, hash_kind, d_out_pk_x, d_out_pk_is_odd, d_out_signatures, d_out_status);
}
int32_t og_bjj_sign_batch(og_ctx* ctx, const uint8_t* secret_keys, const uint8_t* randomness, const uint8_t* messages, uint32_t n,
                          int32_t hash_kind, uint8_t* out_pk_x, uint8_t* out_pk_is_odd, uint8_t* out_signatures, uint8_t* out_status) {
    OG_ENTER(ctx);
    if (!ctx || !secret_keys || !randomness || !messages || !out_pk_x || !out_pk_is_odd || !out_signatures || !out_status || hash_kind < 0 || hash_kind > 1)
        return OG_E_INVALID;
    if (n == 0) return OG_OK;
    OG_SLOT(ctx, dsk, uint8_t, S_IO_A, 32ull * n);
    OG_SLOT(ctx, drn, uint8_t, S_IO_B, 32ull * n);
    OG_SLOT(ctx, dm, uint8_t, S_IO_C, 32ull * n);
    OG_SLOT(ctx, dpx, uint8_t, S_IO_D, 32ull * n);
    OG_SLOT(ctx, dodd, uint8_t, S_IO_E, n);
    OG_SLOT(ctx, dsg, uint8_t, S_IO_F, 96ull * n);
    OG_SLOT(ctx, dst, uint8_t, S_IO_G, n);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dsk, secret_keys, 32ull * n); H2D(ctx, drn, randomness, 32ull * n); H2D(ctx, dm, messages, 32ull * n);
    OG_TRY(bjj_sign_dev(ctx, dsk, drn, dm, n, hash_kind, dpx, dodd, dsg, dst));
    D2H(ctx, out_pk_x, dpx, 32ull * n); D2H(ctx, out_pk_is_odd, dodd, n); D2H(ctx, out_signatures, dsg, 96ull * n); D2H(ctx, out_status, dst, n);
    return check_flag(ctx);
}

// ---- MSM --------------------------------------------------------------------------------------------------
int32_t og_msm_g1_dev(og_ctx* ctx, const uint8_t* d_points, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out64) {
    return msm_dev_entry<Fq>(ctx, d_points, d_scalars, n, d_out64);
}
int32_t og_msm_g2_dev(og_ctx* ctx, const uint8_t* d_points, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out128) {
    return msm_dev_entry<Fq2>(ctx, d_points, d_scalars, n, d_out128);
}
int32_t og_msm_g1(og_ctx* ctx, const uint8_t* points, const uint8_t* scalars, uint64_t n, uint8_t* out64) {
    return msm_host_entry<Fq>(ctx, points, scalars, n, out64);
}
int32_t og_msm_g2(og_ctx* ctx, const uint8_t* points, const uint8_t* scalars, uint64_t n, uint8_t* out128) {
    return msm_host_entry<Fq2>(ctx, points, scalars, n, out128);
}
int32_t og_g1_sum(og_ctx* ctx, const uint8_t* points, uint64_t n, uint8_t* out64) { return sum_host_entry<Fq>(ctx, points, n, out64); }
int32_t og_g2_sum(og_ctx* ctx, const uint8_t* points, uint64_t n, uint8_t* out128) { return sum_host_entry<Fq2>(ctx, points, n, out128); }

int32_t og_g1_sum_dev(og_ctx* ctx, const uint8_t* d_points, uint64_t n, uint8_t* d_out64) { return sum_dev_entry<Fq>(ctx, d_points, n, d_out64); }
int32_t og_g2_sum_dev(og_ctx* ctx, const uint8_t* d_points, uint64_t n, uint8_t* d_out128) { return sum_dev_entry<Fq2>(ctx, d_points, n, d_out128); }
int32_t og_g1_generator_mul_dev(og_ctx* ctx, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out_points) {
    return generator_mul_dev_entry<Fq>(ctx, d_scalars, n, d_out_points);
}
int32_t og_g2_generator_mul_dev(og_ctx* ctx, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out_points) {
    return generator_mul_dev_entry<Fq2>(ctx, d_scalars, n, d_out_points);
}

// out[i] = scalars[i] * G (fixed-base, generator of G1 / G2): used by the setup and to synthesise MSM inputs
int32_t og_g1_generator_mul(og_ctx* ctx, const uint8_t* scalars, uint64_t n, uint8_t* out_points) {
    return generator_mul_host_entry<Fq>(ctx, scalars, n, out_points);
}
int32_t og_g2_generator_mul(og_ctx* ctx, const uint8_t* scalars, uint64_t n, uint8_t* out_points) {
    return generator_mul_host_entry<Fq2>(ctx, scalars, n, out_points);
}

// ---- NTT ----------------------------------------------------------------------------------------------------
int32_t og_ntt_dev(og_ctx* ctx, uint8_t* d_data, uint32_t log_n, uint32_t batch, int32_t inverse, int32_t coset) {
    OG_ENTER(ctx);
    if (!ctx || !d_data || log_n > 27 || !aligned32(d_data)) return OG_E_INVALID;
    uint64_t tot = (uint64_t)batch << log_n;
    if (tot == 0) return OG_OK;
    OG_SLOT(ctx, work, Fr, S_NTT_DATA, sizeof(Fr) * tot * 2);
    OG_TRY(mimc_to_mont_dev(ctx, d_data, tot, work));
    OG_TRY(ntt_mont_dev(ctx, work, work + tot, log_n, batch, inverse, coset));
    return mimc_from_mont_dev(ctx, work, tot, d_data);
}
int32_t og_ntt(og_ctx* ctx, uint8_t* data, uint32_t log_n, uint32_t batch, int32_t inverse, int32_t coset) {
    OG_ENTER(ctx);
    if (!ctx || !data || log_n > 27) return OG_E_INVALID;
    uint64_t tot = (uint64_t)batch << log_n;
    if (tot == 0) return OG_OK;
    OG_SLOT(ctx, dd, uint8_t, S_IO_A, 32 * tot);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dd, data, 32 * tot);
    OG_TRY(og_ntt_dev(ctx, dd, log_n, batch, inverse, coset));
    D2H(ctx, data, dd, 32 * tot);
    return check_flag(ctx);
}

// ---- withdraw statement ----------------------------------------------------------------------------------------
int32_t og_withdraw_r1cs_info(uint32_t depth, uint32_t* n_constraints, uint32_t* n_vars, uint32_t* n_pub, uint32_t* log_m) {
    if (depth == 0 || depth > 32) return OG_E_INVALID;
    WithdrawLayout L = WithdrawLayout::make(depth);
    if (n_constraints) *n_constraints = L.n_constraints;
    if (n_vars) *n_vars = L.n_vars;
    if (n_pub) *n_pub = WITHDRAW_N_PUB;
    if (log_m) *log_m = groth16_domain_log(L.n_constraints, WITHDRAW_N_PUB);
    return OG_OK;
}
int32_t og_withdraw_r1cs_export(uint32_t depth, int32_t which, uint32_t* row_ptr, uint32_t* col_idx, uint8_t* coeffs, uint64_t* nnz) {
    if (depth == 0 || depth > 32 || which < 0 || which > 2 || !nnz) return OG_E_INVALID;
    R1cs cs = WithdrawBuilder::build(depth);
    const Csr& M = which == 0 ? cs.A : (which == 1 ? cs.B : cs.C);
    *nnz = M.col.size();
    if (!row_ptr || !col_idx || !coeffs) return OG_OK;
    memcpy(row_ptr, M.row_ptr.data(), 4 * M.row_ptr.size());
    memcpy(col_idx, M.col.data(), 4 * M.col.size());
    for (size_t i = 0; i < M.val.size(); i++) host_store(coeffs + 32 * i, M.val[i]);
    return OG_OK;
}
int32_t og_withdraw_witness(og_ctx* ctx, uint32_t depth, const uint8_t* nullifiers, const uint8_t* secrets, const uint8_t* recipients,
                            const uint8_t* siblings, const uint32_t* path_bits, uint32_t batch, uint8_t* witnesses) {
    OG_ENTER(ctx);
    if (!ctx || depth == 0 || depth > 32 || !nullifiers || !secrets || !recipients || !siblings || !path_bits || !witnesses) return OG_E_INVALID;
    if (batch == 0) return OG_OK;
    WithdrawLayout L = WithdrawLayout::make(depth);
    OG_SLOT(ctx, dn, uint8_t, S_IO_A, 32ull * batch);
    OG_SLOT(ctx, dsx, uint8_t, S_IO_B, 32ull * batch);
    OG_SLOT(ctx, dr, uint8_t, S_IO_C, 32ull * batch);
    OG_SLOT(ctx, dsib, uint8_t, S_IO_D, 32ull * batch * depth);
    OG_SLOT(ctx, dbits, uint32_t, S_IO_E, 4ull * batch);
    OG_SLOT(ctx, dout, uint8_t, S_IO_F, 32ull * batch * L.n_vars);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dn, nullifiers, 32ull * batch); H2D(ctx, dsx, secrets, 32ull * batch); H2D(ctx, dr, recipients, 32ull * batch);
    H2D(ctx, dsib, siblings, 32ull * batch * depth); H2D(ctx, dbits, path_bits, 4ull * batch);
    OG_TRY(withdraw_witness_bytes_dev(ctx, depth, dn, dsx, dr, dsib, dbits, batch, dout));
    D2H(ctx, witnesses, dout, 32ull * batch * L.n_vars);
    return check_flag(ctx);
}

// ---- Groth16 -------------------------------------------------------------------------------------------------------
int32_t og_groth16_setup_withdraw(og_ctx* ctx, uint32_t depth, const uint8_t* toxic160, uint8_t* pk_out, uint64_t* pk_len,
                                  uint8_t* vk_out, uint64_t* vk_len) {
    OG_ENTER(ctx);
    if (!ctx || !pk_len || !vk_len || ((pk_out || vk_out) && !toxic160)) return OG_E_INVALID;
    return setup_withdraw(ctx, depth, toxic160, pk_out, pk_len, vk_out, vk_len);
}
int32_t og_load_pk(og_ctx* ctx, const uint8_t* pk_bytes, uint64_t len, og_pk** out) {
    OG_ENTER(ctx);
    if (!ctx || !pk_bytes || !out) return OG_E_INVALID;
    return pk_load(ctx, pk_bytes, len, out);
}
void og_free_pk(og_pk* pk) { pk_free(pk); }
int32_t og_pk_info(const og_pk* pk, uint32_t* n_vars, uint32_t* n_pub, uint32_t* log_m, uint32_t* depth) {
    if (!pk) return OG_E_INVALID;
    pk_info(pk, n_vars, n_pub, log_m, depth);
    return OG_OK;
}

int32_t og_groth16_prove(og_ctx* ctx, const og_pk* pk, const uint8_t* witnesses, uint32_t batch, const uint8_t* rs, uint8_t* proofs) {
    OG_ENTER(ctx);
    if (!ctx || !pk || !witnesses || !rs || !proofs) return OG_E_INVALID;
    OG_PK_CHECK(ctx, pk);
    if (batch == 0) return OG_OK;
    uint32_t nv; pk_info(pk, &nv, nullptr, nullptr, nullptr);
    OG_SLOT(ctx, dw, uint8_t, S_IO_A, 32ull * batch * nv);
    OG_SLOT(ctx, drs, uint8_t, S_IO_B, 64ull * batch);
    OG_SLOT(ctx, dpr, uint8_t, S_IO_C, 256ull * batch);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dw, witnesses, 32ull * batch * nv); H2D(ctx, drs, rs, 64ull * batch);
    OG_TRY(prove_witness_dev(ctx, pk, dw, batch, drs, dpr));
    D2H(ctx, proofs, dpr, 256ull * batch);
    return check_flag(ctx);
}

int32_t og_groth16_prove_withdraw_dev(og_ctx* ctx, const og_pk* pk, const uint8_t* d_nullifiers, const uint8_t* d_secrets,
                                      const uint8_t* d_recipients, const uint8_t* d_siblings, const uint32_t* d_path_bits, uint32_t batch,
                                      const uint8_t* d_rs, uint8_t* d_proofs, uint8_t* d_public_out) {
    OG_ENTER(ctx);
    if (!ctx || !pk || !d_nullifiers || !d_secrets || !d_recipients || !d_siblings || !d_path_bits || !d_rs || !d_proofs) return OG_E_INVALID;
    OG_PK_CHECK(ctx, pk);
    return prove_withdraw_dev(ctx, pk, d_nullifiers, d_secrets, d_recipients, d_siblings, d_path_bits, batch, d_rs, d_proofs, d_public_out);
}

int32_t og_groth16_prove_withdraw(og_ctx* ctx, const og_pk* pk, const uint8_t* nullifiers, const uint8_t* secrets, const uint8_t* recipients,
                                  const uint8_t* siblings, const uint32_t* path_bits, uint32_t batch, const uint8_t* rs, uint8_t* proofs,
                                  uint8_t* public_out) {
    OG_ENTER(ctx);
    if (!ctx || !pk || !nullifiers || !secrets || !recipients || !siblings || !path_bits || !rs || !proofs) return OG_E_INVALID;
    OG_PK_CHECK(ctx, pk);
    if (batch == 0) return OG_OK;
    uint32_t depth, n_pub; pk_info(pk, nullptr, &n_pub, nullptr, &depth);
    if (depth == 0) return OG_E_INVALID;
    OG_SLOT(ctx, dn, uint8_t, S_IO_A, 32ull * batch);
    OG_SLOT(ctx, dsx, uint8_t, S_IO_B, 32ull * batch);
    OG_SLOT(ctx, dr, uint8_t, S_IO_C, 32ull * batch);
    OG_SLOT(ctx, dsib, uint8_t, S_IO_D, 32ull * batch * depth);
    OG_SLOT(ctx, dbits, uint32_t, S_IO_E, 4ull * batch);
    OG_SLOT(ctx, drs, uint8_t, S_IO_F, 64ull * batch);
    OG_SLOT(ctx, dpr, uint8_t, S_IO_G, 256ull * batch);
    OG_SLOT(ctx, dpub, uint8_t, S_IO_H, 32ull * batch * n_pub);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dn, nullifiers, 32ull * batch); H2D(ctx, dsx, secrets, 32ull * batch); H2D(ctx, dr, recipients, 32ull * batch);
    H2D(ctx, dsib, siblings, 32ull * batch * depth); H2D(ctx, dbits, path_bits, 4ull * batch); H2D(ctx, drs, rs, 64ull * batch);
    OG_TRY(prove_withdraw_dev(ctx, pk, dn, dsx, dr, dsib, dbits, batch, drs, dpr, public_out ? dpub : nullptr));
    D2H(ctx, proofs, dpr, 256ull * batch);
    if (public_out) D2H(ctx, public_out, dpub, 32ull * batch * n_pub);
    return check_flag(ctx);
}

int32_t og_groth16_h_evals(og_ctx* ctx, const og_pk* pk, const uint8_t* witness, uint8_t* out) {
    OG_ENTER(ctx);
    if (!ctx || !pk || !witness || !out) return OG_E_INVALID;
    OG_PK_CHECK(ctx, pk);
    uint32_t nv, log_m; pk_info(pk, &nv, nullptr, &log_m, nullptr);
    OG_SLOT(ctx, dw, uint8_t, S_IO_A, 32ull * nv);
    OG_SLOT(ctx, dout, uint8_t, S_IO_B, 32ull << log_m);
    OG_TRY(clear_flag(ctx));
    H2D(ctx, dw, witness, 32ull * nv);
    OG_TRY(h_evals_dev(ctx, pk, dw, dout));
    D2H(ctx, out, dout, 32ull << log_m);
    return check_flag(ctx);
}

int32_t og_groth16_verify(const uint8_t* vk, uint64_t vk_len, const uint8_t* public_inputs, uint32_t n_pub, const uint8_t* proof256) {
    if (!vk || !proof256 || (n_pub && !public_inputs)) return OG_E_INVALID;
    return groth16_verify_host(vk, vk_len, public_inputs, n_pub, proof256);
}

}  // extern "C"
