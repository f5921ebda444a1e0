// owshen_b200/csrc/msm_sort.cu -- the curve-independent half of the MSM engine (msm.cuh): signed c-bit digits of the
// scalars, counted, scanned and scattered into per-bucket lists of (point index, sign) entries.  Stages 1-3 of the
// pipeline in msm.cu; the same lists feed the G1 and the G2 bucket kernels.
#include "msm.cuh"

namespace og {

// ---- 1/3: digits -> histogram / scatter ---------------------------------------------------------------
// Signed c-bit digits of one scalar: v = bits + carry; v > 2^(c-1) -> digit v - 2^c, carry 1.  n_windows*c >= 255
// guarantees that the top window absorbs the last carry for every scalar < r < 2^254.
struct DigitIter {
    uint32_t s[9];
    __device__ __forceinline__ bool load(const DigitPlan& P, uint32_t prob, uint64_t i, int* flag) {
        const uint32_t* sp = P.scalars + ((uint64_t)prob * P.scalar_stride + i) * 8;
        if (P.montgomery) {
            Fr v;
#pragma unroll
            for (int j = 0; j < 8; j++) v.l[j] = sp[j];
            v.to_canonical(s);
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) s[j] = sp[j];
            if (!Fr::canonical_lt_mod(s)) { atomicOr(flag, 1); return false; }
        }
        s[8] = 0;
        return (s[0] | s[1] | s[2] | s[3] | s[4] | s[5] | s[6] | s[7]) != 0;
    }
    // calls f(window, magnitude - 1, negative) for every non-zero signed digit
    template <class Fn>
    __device__ __forceinline__ void for_each(const DigitPlan& P, Fn f) const {
        const uint32_t c = P.c, half = 1u << (c - 1), mask = (1u << c) - 1;
        uint32_t carry = 0;
        for (uint32_t w = 0; w < P.n_windows; w++) {
            uint32_t bit = w * c, word = bit >> 5, sh = bit & 31;
            uint64_t two = ((uint64_t)s[word + 1] << 32) | s[word];
            uint32_t v = ((uint32_t)(two >> sh) & mask) + carry;
            uint32_t neg = v > half;
            uint32_t mag = neg ? (1u << c) - v : v;
            carry = neg;
            if (mag) f(w, mag - 1, neg);
        }
    }
};

// one thread per scalar, global atomics (one-shot MSMs: up to 2^15 buckets x 16 windows of keys).  The scatter is pure
// atomic round-trip latency (ncu, profiles/r2_ncu_digits.md: 93 % of the warp samples on the long scoreboard, issue slots 17 %
// busy); cutting eight windows first and issuing their eight atomics back to back was measured SLOWER (21.3 vs 20.1 ms per 1024
// proofs, profiles/r2_small_ab.md): the L2 atomic units, not the per-thread dependency, are what the kernel waits for.
template <bool SCATTER>
__global__ void __launch_bounds__(256) k_digits(DigitPlan P, uint32_t* __restrict__ counts, const uint32_t* __restrict__ offsets,
                                                uint32_t* __restrict__ cursor, uint32_t* __restrict__ sorted, int* flag) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t prob = blockIdx.y;
    if (i >= P.n) return;
    DigitIter it;
    if (!it.load(P, prob, i, flag)) return;
    it.for_each(P, [&](uint32_t w, uint32_t b, uint32_t neg) {
        uint32_t key = (prob * P.key_stride_problem + w * P.key_stride_window) * P.nb + b;
        if (!SCATTER) {
            atomicAdd(&counts[key], 1u);
        } else {
            uint32_t pos = atomicAdd(&cursor[key], 1u);          // cursor starts at the bucket's offset (k_scan_apply)
            sorted[pos] = (((uint32_t)i + w * P.tidx_window_stride) << 1) | neg;
        }
    });
}

// Tiled histogram for the batched prover (one group per proof, nb <= 32768): a CTA owns a tile of one problem's
// scalars, counts its digits in shared memory and touches global memory once per bucket instead of once per
// digit (5x faster than global atomics: 5 vs 24 ms per 1024 proofs).  The scatter stays the plain k_digits<true>:
// a tiled scatter with run reservation and a one-CTA-per-proof shared-memory sort were both measured slower
// (39 vs 33 ms and 56.6 vs 29 ms per 1024 proofs, profiles/r1_*; their code was removed in round 2).
constexpr uint32_t DIG_TILE = 4096, DIG_THREADS = 256, DIG_MAX_NB_COUNT = 32768;

__global__ void __launch_bounds__(DIG_THREADS) k_digits_count_tiled(DigitPlan P, uint32_t* __restrict__ counts, int* flag) {
    extern __shared__ uint32_t hist[];                    // nb counters (dynamic: up to 128 KB)
    const uint32_t prob = blockIdx.y, nb = P.nb;
    const uint64_t lo = (uint64_t)blockIdx.x * DIG_TILE;
    const uint64_t hi = lo + DIG_TILE < P.n ? lo + DIG_TILE : P.n;
    const uint32_t key0 = prob * P.key_stride_problem * nb;          // key_stride_window == 0 in this mode
    for (uint32_t b = threadIdx.x; b < nb; b += DIG_THREADS) hist[b] = 0;
    __syncthreads();
    for (uint64_t i = lo + threadIdx.x; i < hi; i += DIG_THREADS) {
        DigitIter it;
        if (it.load(P, prob, i, flag)) it.for_each(P, [&](uint32_t, uint32_t b, uint32_t) { atomicAdd(&hist[b], 1u); });
    }
    __syncthreads();
    for (uint32_t b = threadIdx.x; b < nb; b += DIG_THREADS) if (hist[b]) atomicAdd(&counts[key0 + b], hist[b]);
}

// ---- 2: exclusive scan: tile sums -> scan of the tile sums (one CTA) -> tile rescan with offsets ----------
constexpr uint32_t SCAN_THREADS = 256, SCAN_PER_THREAD = 8, SCAN_TILE = SCAN_THREADS * SCAN_PER_THREAD;

__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total) {   // 256 threads
    __shared__ uint32_t warp_sums[SCAN_THREADS / 32];
    __shared__ uint32_t block_total;
    uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, inc, d); if (lane >= (uint32_t)d) inc += t; }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t w = lane < SCAN_THREADS / 32 ? warp_sums[lane] : 0, winc = w;
#pragma unroll
        for (int d = 1; d < 8; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, winc, d); if (lane >= (uint32_t)d) winc += t; }
        if (lane < SCAN_THREADS / 32) warp_sums[lane] = winc - w;
        if (lane == SCAN_THREADS / 32 - 1) block_total = winc;
    }
    __syncthreads();
    uint32_t r = inc - v + warp_sums[wid];
    *total = block_total;
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tiles(const uint32_t* __restrict__ counts, uint32_t n, uint32_t* __restrict__ tile_sums) {
    uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_PER_THREAD, s = 0;
#pragma unroll
    for (uint32_t k = 0; k < SCAN_PER_THREAD; k++) if (base + k < n) s += counts[base + k];
    uint32_t total;
    block_exclusive_scan(s, &total);
    if (threadIdx.x == 0) tile_sums[blockIdx.x] = total;
}
// in-place exclusive scan of up to SCAN_TILE * 64 tile sums by one CTA
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_tile_sums(uint32_t* __restrict__ tile_sums, uint32_t n_tiles, uint32_t* __restrict__ grand_total) {
    uint32_t run = 0;
    for (uint32_t base = 0; base < n_tiles; base += SCAN_THREADS) {
        uint32_t i = base + threadIdx.x;
        uint32_t v = i < n_tiles ? tile_sums[i] : 0, total;
        uint32_t ex = block_exclusive_scan(v, &total);
        if (i < n_tiles) tile_sums[i] = run + ex;
        run += total;
    }
    if (threadIdx.x == 0) *grand_total = run;
}
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_apply(const uint32_t* __restrict__ counts, uint32_t n, const uint32_t* __restrict__ tile_sums,
                                                            uint32_t* __restrict__ offsets, uint32_t* __restrict__ cursor) {
    uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * SCAN_PER_THREAD;
    uint32_t c[SCAN_PER_THREAD], s = 0;
#pragma unroll
    for (uint32_t k = 0; k < SCAN_PER_THREAD; k++) { c[k] = base + k < n ? counts[base + k] : 0; s += c[k]; }
    uint32_t total;
    uint32_t run = tile_sums[blockIdx.x] + block_exclusive_scan(s, &total);
#pragma unroll
    for (uint32_t k = 0; k < SCAN_PER_THREAD; k++) {      // the scatter's cursors start at the offsets: one random access per entry fewer
        if (base + k < n) { offsets[base + k] = run; cursor[base + k] = run; }
        run += c[k];
    }
}

int32_t msm_sort_digits(og_ctx* ctx, const DigitPlan& plan, uint32_t n_keys, uint32_t* d_counts, uint32_t* d_offsets,
                        uint32_t* d_cursor, uint32_t* d_sorted) {
    OG_CUDA(ctx, cudaMemsetAsync(d_counts, 0, sizeof(uint32_t) * (size_t)n_keys, ctx->stream));
    if (plan.n == 0 || plan.n_problems == 0) {
        OG_CUDA(ctx, cudaMemsetAsync(d_offsets, 0, sizeof(uint32_t) * ((size_t)n_keys + 1), ctx->stream));
        return OG_OK;
    }
    const bool tiled = plan.key_stride_window == 0 && plan.nb <= DIG_MAX_NB_COUNT;
    if (tiled && !ctx->digits_smem_opt_in) {      // per device, hence per context
        OG_CUDA(ctx, cudaFuncSetAttribute(k_digits_count_tiled, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(4 * DIG_MAX_NB_COUNT)));
        ctx->digits_smem_opt_in = true;
    }
    dim3 grid((unsigned)((plan.n + 255) / 256), plan.n_problems);
    dim3 tgrid((unsigned)((plan.n + DIG_TILE - 1) / DIG_TILE), plan.n_problems);
    if (tiled) OG_LAUNCH(ctx, k_digits_count_tiled, tgrid, DIG_THREADS, 4 * (size_t)plan.nb, plan, d_counts, ctx->d_flag);
    else OG_LAUNCHN(ctx, "k_digits_count", k_digits<false>, grid, 256, 0, plan, d_counts, nullptr, nullptr, nullptr, ctx->d_flag);
    {   // offsets[n_keys] receives the grand total; cursor[k] = offsets[k] for the scatter
        uint32_t n_tiles = (n_keys + SCAN_TILE - 1) / SCAN_TILE;
        OG_SLOT(ctx, tile_sums, uint32_t, S_MSM_MISC, 4 * (size_t)n_tiles);
        OG_LAUNCH(ctx, k_scan_tiles, n_tiles, SCAN_THREADS, 0, d_counts, n_keys, tile_sums);
        OG_LAUNCH(ctx, k_scan_tile_sums, 1, SCAN_THREADS, 0, tile_sums, n_tiles, d_offsets + n_keys);
        OG_LAUNCH(ctx, k_scan_apply, n_tiles, SCAN_THREADS, 0, d_counts, n_keys, tile_sums, d_offsets, d_cursor);
    }
    OG_LAUNCHN(ctx, "k_digits_scatter", k_digits<true>, grid, 256, 0, plan, d_counts, d_offsets, d_cursor, d_sorted, ctx->d_flag);
    return OG_OK;
}

}  // namespace og
