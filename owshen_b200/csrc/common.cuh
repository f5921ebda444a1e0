// owshen_b200/csrc/common.cuh -- context, error plumbing, launch accounting and the byte<->Montgomery
// boundary kernels shared by every translation unit of libowshen_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <vector>
#include "../../include/owshen_b200.h"
#include "fp.cuh"
#include "ec.cuh"

namespace og {

constexpr int N_SLOTS = 64;

struct NttTables;   // ntt.cu

}  // namespace og

struct og_ctx {
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;        // every launch and copy of the library (og_stream returns it)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    uint64_t launches = 0;
    char err[512] = {0};
    // persistent scratch slots: grown on demand, never shrunk, so steady-state calls do not allocate
    void* slot_ptr[og::N_SLOTS] = {nullptr};
    size_t slot_cap[og::N_SLOTS] = {0};
    int* d_flag = nullptr;           // device error flag (encoding errors found inside kernels)
    int* h_flag = nullptr;           // pinned mirror
    og::NttTables* ntt[32] = {nullptr};
    void* g1_fixed = nullptr;        // fixed-base tables of the generators (setup only)
    void* g2_fixed = nullptr;
    void* bjj_fixed = nullptr;       // window multiples of the BabyJubJub BASE (bjj_impl.cuh)
    bool digits_smem_opt_in = false; // cudaFuncSetAttribute(k_digits_count_tiled) done for this device

    // optional per-kernel timing: CUDA events around every launch of this library (og_profile)
    bool prof_on = false;
    struct ProfRec { const char* name; cudaEvent_t a, b; };
    std::vector<ProfRec> prof;
    std::vector<cudaEvent_t> ev_pool;
    cudaEvent_t prof_event();

    void* slot(int id, size_t bytes);   // nullptr on allocation failure (err is set)
};

namespace og {

#define OG_CUDA(ctx, call)                                                                        \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            snprintf((ctx)->err, sizeof((ctx)->err), "%s:%d: %s: %s", __FILE__, __LINE__, #call,  \
                     cudaGetErrorString(e_));                                                     \
            return OG_E_CUDA;                                                                     \
        }                                                                                         \
    } while (0)

#define OG_TRY(expr)                  \
    do {                              \
        int32_t rc_ = (expr);         \
        if (rc_ != OG_OK) return rc_; \
    } while (0)

// every kernel launch of the library goes through this so og_launch_count is exact
#define OG_LAUNCHN(ctx, name, kernel, grid, block, smem, ...)                                     \
    do {                                                                                          \
        cudaEvent_t pa_ = nullptr, pb_ = nullptr;                                                 \
        if ((ctx)->prof_on) { pa_ = (ctx)->prof_event(); pb_ = (ctx)->prof_event();               \
                              cudaEventRecord(pa_, (ctx)->stream); }                              \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                          \
        if (pa_) { cudaEventRecord(pb_, (ctx)->stream); (ctx)->prof.push_back({(name), pa_, pb_}); } \
        (ctx)->launches++;                                                                        \
        OG_CUDA(ctx, cudaGetLastError());                                                         \
    } while (0)
#define OG_LAUNCH(ctx, kernel, grid, block, smem, ...) OG_LAUNCHN(ctx, #kernel, kernel, grid, block, smem, __VA_ARGS__)

#define OG_SLOT(ctx, var, type, id, bytes)                       \
    type* var = (type*)(ctx)->slot((id), (bytes));               \
    if (!var) return OG_E_NOMEM

// scratch slot ids (one owner each; a slot is only reused by the call that owns it)
enum Slot {
    S_IO_A = 0, S_IO_B, S_IO_C, S_IO_D, S_IO_E, S_IO_F, S_IO_G, S_IO_H,   // staged host buffers
    S_MSM_POINTS, S_MSM_SCALARS, S_MSM_COUNTS, S_MSM_OFFSETS, S_MSM_CURSOR, S_MSM_SORTED, S_MSM_BUCKETS,
    S_MSM_SEG, S_MSM_OUT, S_MSM_HEAVY, S_MSM_MISC,
    S_NTT_DATA,
    S_PR_WIT, S_PR_ABC, S_PR_SCALARS, S_PR_SORTED, S_PR_COUNTS, S_PR_OFFSETS, S_PR_CURSOR, S_PR_BUCKETS,
    S_PR_SEG, S_PR_SUMS, S_PR_OUT, S_PR_PUB, S_PR_MISC, S_PR_HEAVY,
    S_SETUP_A, S_SETUP_B, S_SETUP_C,
    S_COUNT
};
static_assert(S_COUNT <= N_SLOTS, "grow N_SLOTS");

static inline bool aligned32(const void* p) { return (((uintptr_t)p) & 31) == 0; }

int32_t check_flag(og_ctx* ctx);          // sync + read device error flag -> OG_E_ENCODING
int32_t clear_flag(og_ctx* ctx);

// canonical little-endian bytes -> Montgomery limbs (device side of the boundary)
template <class F>
__device__ __forceinline__ F load_canonical(const uint8_t* p, int* flag) {
    const uint32_t* q = reinterpret_cast<const uint32_t*>(p);
    uint32_t c[8];
#pragma unroll
    for (int i = 0; i < 8; i++) c[i] = q[i];
    if (!F::canonical_lt_mod(c)) { atomicOr(flag, 1); for (int i = 0; i < 8; i++) c[i] = 0; }
    return F::from_canonical(c);
}
template <class F>
__device__ __forceinline__ void store_canonical(uint8_t* p, const F& v) {
    uint32_t c[8];
    v.to_canonical(c);
    uint32_t* q = reinterpret_cast<uint32_t*>(p);
#pragma unroll
    for (int i = 0; i < 8; i++) q[i] = c[i];
}

// host-side helpers for canonical bytes (setup / verify / tests of the host code)
template <class F>
static inline bool host_load(F& out, const uint8_t* p) {
    uint32_t c[8];
    memcpy(c, p, 32);
    if (!F::canonical_lt_mod(c)) return false;
    out = F::from_canonical(c);
    return true;
}
template <class F>
static inline void host_store(uint8_t* p, const F& v) {
    uint32_t c[8];
    v.to_canonical(c);
    memcpy(p, c, 32);
}

// ---- module entry points (implemented in the .cu files, called from capi.cu) ----------------------
int32_t mimc_init(og_ctx* ctx);
void mimc_constants_host(Fr* out91);   // Montgomery form

}  // namespace og
