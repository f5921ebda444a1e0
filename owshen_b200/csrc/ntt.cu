// owshen_b200/csrc/ntt.cu -- batched radix-2 NTT over BN254 Fr for sm_100a.
//
// No counterpart in the reference (SURVEY.md section 0); convention follows its field generator 7
// (/root/reference/src/blockchain/tx/owshen_airdrop/babyjubjub/mod.rs:9): omega_n = 7^((r-1)/n),
// forward out[k] = sum_j in[j] omega^(jk), natural order in and out; "coset" evaluates on g*omega^k
// with g = omega_{2n}.
//
// Decimation-in-time with the stages grouped into passes; a pass stages a tile of <= 1024
// coefficients (32 KB) in shared memory and runs up to 10 butterfly levels there, so a 2^15
// transform (the Groth16 domain of the withdraw circuit) is two global passes.  Pass 1 gathers its
// tile in bit-reversed order (32 B elements = one DRAM sector each, so the gather wastes no
// bandwidth) and fuses the coset scaling; the last pass fuses 1/n and the inverse coset shift.
// Later passes own 2^K strided rows x 8 consecutive columns so that global accesses are 256 B runs.
// One table per size serves everything: T2[j] = omega_{2n}^j (j < n): coset factors are T2[j],
// stage twiddles are omega_n^e = T2[2e], inverses are -T2[n - j].
#include "ntt.cuh"

namespace og {

struct NttTables {
    uint32_t log_n;
    Fr* d_t2;      // omega_{2n}^j, j < n, Montgomery form
    Fr* d_t2n;     // omega_{2n}^j / n: coset factors that also carry the 1/n of a preceding inverse transform (ntt_mont_dev: fold)
    Fr n_inv;      // 1/n, Montgomery form
};

__global__ void __launch_bounds__(256) k_ntt_table(Fr g, uint64_t n, Fr* __restrict__ t2) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    Fr acc = Fr::one(), base = g;
    for (uint64_t e = j; e; e >>= 1) {
        if (e & 1) acc = acc * base;
        base = base.sqr();
    }
    t2[j] = acc;
}

__global__ void __launch_bounds__(256) k_ntt_table_scaled(const Fr* __restrict__ t2, Fr n_inv, uint64_t n, Fr* __restrict__ t2n) {
    uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < n) t2n[j] = t2[j] * n_inv;
}

// omega_{2n}^(+-j), 0 <= j < n
__device__ __forceinline__ Fr tw2(const Fr* __restrict__ t2, uint32_t n, uint32_t j, bool inverse) {
    if (!inverse || j == 0) return t2[j];
    return t2[n - j].neg();
}

struct PassPlan {
    uint32_t log_n;
    uint32_t s0;        // first (1-based) DIT stage of this pass
    uint32_t K;         // stages in this pass
    uint32_t L;         // log2 of consecutive columns per tile (0 in the first pass)
    uint32_t first, last, inverse, coset;
    uint32_t fold;      // 1: inverse transform whose 1/n is left to the next transform; 2: forward coset transform that applies it
                        // (its coset factors come from t2n = t2 / n): one product per element fewer for the pair (groth16.cu)
};

__device__ __forceinline__ uint32_t bitrev(uint32_t x, uint32_t bits) { return __brev(x) >> (32 - bits); }

// ---- the pass kernel ------------------------------------------------------------------------------------
// Three things taken from the ncu capture of the first version (one level per barrier, plain array-of-structures
// tile; profiles/r1_*; its code was removed in round 2): (1) two butterfly levels per
// barrier with the four operands in registers (half the shared-memory round trips and barriers); (2) the 32-byte
// elements are stored as two 16-byte chunks whose position is XOR-swizzled with bit 2 of the element index, which
// removes the 2-way bank conflict of the plain array-of-structures layout (58 % of the wavefronts were replays);
// (3) the first level of the first pass has twiddle 1 everywhere and skips its products.
__device__ __forceinline__ uint32_t sw_chunk(uint32_t e, uint32_t h) { return ((e << 1) | h) ^ ((e >> 2) & 1); }
__device__ __forceinline__ Fr sm_get(const uint4* sm, uint32_t e) {
    uint4 a = sm[sw_chunk(e, 0)], b = sm[sw_chunk(e, 1)];
    Fr r;
    r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w; r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
    return r;
}
__device__ __forceinline__ void sm_put(uint4* sm, uint32_t e, const Fr& v) {
    sm[sw_chunk(e, 0)] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
    sm[sw_chunk(e, 1)] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
}

// 3 resident CTAs of 256 threads per SM (80 registers): measured 35.7 -> 31.9 ms per 1024 proofs against 2 CTAs,
// 4 CTAs (64 registers) was equal
__global__ void __launch_bounds__(256, 3) k_ntt_pass2(PassPlan P, const Fr* __restrict__ in, Fr* __restrict__ out,
                                                   const Fr* __restrict__ t2, const Fr* __restrict__ t2n, Fr n_inv) {
    extern __shared__ __align__(32) unsigned char smem_raw[];
    uint4* sm = reinterpret_cast<uint4*>(smem_raw);
    const uint32_t n = 1u << P.log_n;
    const uint32_t B0 = P.s0 - 1;
    const uint32_t tile = 1u << (P.K + P.L);
    const uint32_t t = blockIdx.x;
    const uint32_t mid = t & ((1u << (B0 - P.L)) - 1), top = t >> (B0 - P.L);
    const uint32_t base = (top << (B0 + P.K)) | (mid << P.L);
    const Fr* src = in + (size_t)blockIdx.y * n;
    Fr* dst = out + (size_t)blockIdx.y * n;
    const uint32_t lmask = (1u << P.L) - 1;

    for (uint32_t e = threadIdx.x; e < tile; e += blockDim.x) {
        uint32_t lo = e & lmask, k = e >> P.L;
        uint32_t i = base | (k << B0) | lo;
        Fr v;
        if (P.first) {
            uint32_t j = bitrev(i, P.log_n);
            v = src[j];
            if (P.coset && !P.inverse) v = v * (P.fold == 2 ? t2n[j] : t2[j]);
        } else {
            v = src[i];
        }
        sm_put(sm, e, v);
    }
    __syncthreads();

    uint32_t q = 1;
    for (; q + 1 <= P.K; q += 2) {                      // two levels per barrier
        const uint32_t s = P.s0 + q - 1;
        const bool unit = P.first && q == 1;            // all twiddles of level 1 (and w2a of level 2) are omega^0
        for (uint32_t g = threadIdx.x; g < (tile >> 2); g += blockDim.x) {
            uint32_t lo = g & lmask, kb = g >> P.L;
            uint32_t klow = kb & ((1u << (q - 1)) - 1), khigh = kb >> (q - 1);
            uint32_t k00 = (khigh << (q + 1)) | klow;
            uint32_t e00 = (k00 << P.L) | lo, d1 = (1u << (q - 1)) << P.L, d2 = (1u << q) << P.L;
            uint32_t j1 = (klow << B0) | (mid << P.L) | lo;                       // < 2^(s-1)
            uint32_t j2b = j1 + (1u << (q - 1 + B0));                             // < 2^s
            Fr x00 = sm_get(sm, e00), x01 = sm_get(sm, e00 + d1), x10 = sm_get(sm, e00 + d2), x11 = sm_get(sm, e00 + d1 + d2);
            Fr a0, a1, b0, b1;
            if (unit) {
                a0 = x00 + x01; a1 = x00 - x01; b0 = x10 + x11; b1 = x10 - x11;
            } else {
                Fr w1 = tw2(t2, n, j1 << (P.log_n + 1 - s), P.inverse);
                Fr u = x01 * w1, v = x11 * w1;
                a0 = x00 + u; a1 = x00 - u; b0 = x10 + v; b1 = x10 - v;
            }
            Fr w2b = tw2(t2, n, j2b << (P.log_n - s), P.inverse);
            Fr p0 = unit ? b0 : b0 * tw2(t2, n, j1 << (P.log_n - s), P.inverse);
            Fr p1 = b1 * w2b;
            sm_put(sm, e00, a0 + p0);
            sm_put(sm, e00 + d2, a0 - p0);
            sm_put(sm, e00 + d1, a1 + p1);
            sm_put(sm, e00 + d1 + d2, a1 - p1);
        }
        __syncthreads();
    }
    if (q <= P.K) {                                      // odd number of levels: one plain level
        const uint32_t s = P.s0 + q - 1;
        for (uint32_t b = threadIdx.x; b < (tile >> 1); b += blockDim.x) {
            uint32_t lo = b & lmask, kb = b >> P.L;
            uint32_t klow = kb & ((1u << (q - 1)) - 1);
            uint32_t k0 = ((kb >> (q - 1)) << q) | klow;
            uint32_t e0 = (k0 << P.L) | lo, e1 = e0 + ((1u << (q - 1)) << P.L);
            uint32_t j = (klow << B0) | (mid << P.L) | lo;
            Fr u = sm_get(sm, e0);
            Fr v = (P.first && q == 1) ? sm_get(sm, e1) : sm_get(sm, e1) * tw2(t2, n, j << (P.log_n + 1 - s), P.inverse);
            sm_put(sm, e0, u + v);
            sm_put(sm, e1, u - v);
        }
        __syncthreads();
    }

    for (uint32_t e = threadIdx.x; e < tile; e += blockDim.x) {
        uint32_t lo = e & lmask, k = e >> P.L;
        uint32_t i = base | (k << B0) | lo;
        Fr v = sm_get(sm, e);
        if (P.last && P.inverse) {
            if (P.fold != 1) v = v * n_inv;
            if (P.coset) v = v * tw2(t2, n, i, true);
        }
        dst[i] = v;
    }
}

static int32_t get_tables(og_ctx* ctx, uint32_t log_n, NttTables** out) {
    if (log_n > 27) return OG_E_INVALID;
    if (!ctx->ntt[log_n]) {
        NttTables* T = new NttTables();
        T->log_n = log_n;
        uint64_t n = 1ull << log_n;
        OG_CUDA(ctx, cudaMalloc(&T->d_t2, sizeof(Fr) * n));
        // g = 7^((r-1) >> (log_n+1)) on the host
        uint32_t e[8];
        for (int i = 0; i < 8; i++) e[i] = FrParams::mod(i);
        e[0] -= 1;
        for (uint32_t k = 0; k < log_n + 1; k++) {
            for (int i = 0; i < 7; i++) e[i] = (e[i] >> 1) | (e[i + 1] << 31);
            e[7] >>= 1;
        }
        Fr g = Fr::from_u32(7).pow(e);
        OG_LAUNCH(ctx, k_ntt_table, (unsigned)((n + 255) / 256), 256, 0, g, n, T->d_t2);
        uint32_t nn[8] = {0};
        nn[log_n >> 5] = 1u << (log_n & 31);
        T->n_inv = Fr::from_canonical(nn).inv();
        OG_CUDA(ctx, cudaMalloc(&T->d_t2n, sizeof(Fr) * n));
        OG_LAUNCH(ctx, k_ntt_table_scaled, (unsigned)((n + 255) / 256), 256, 0, T->d_t2, T->n_inv, n, T->d_t2n);
        ctx->ntt[log_n] = T;
    }
    *out = ctx->ntt[log_n];
    return OG_OK;
}

void ntt_free_tables(og_ctx* ctx) {
    for (int i = 0; i < 32; i++)
        if (ctx->ntt[i]) { cudaFree(ctx->ntt[i]->d_t2); cudaFree(ctx->ntt[i]->d_t2n); delete ctx->ntt[i]; ctx->ntt[i] = nullptr; }
}

// In-place on `data` (Montgomery form); `tmp` must hold batch * n elements when log_n > 10.
// fold = 1 (inverse, no coset): the 1/n is NOT applied; fold = 2 (forward coset): the coset scaling also applies that 1/n.
int32_t ntt_mont_dev(og_ctx* ctx, Fr* data, Fr* tmp, uint32_t log_n, uint32_t batch, int inverse, int coset, int fold) {
    if (batch == 0) return OG_OK;
    if ((fold == 1 && !(inverse && !coset)) || (fold == 2 && !(!inverse && coset)) || fold < 0 || fold > 2) return OG_E_INVALID;
    NttTables* T;
    OG_TRY(get_tables(ctx, log_n, &T));
    if (log_n == 0) {
        return OG_OK;   // size-1 transform: identity (coset factor g^0 = 1, 1/n = 1)
    }
    // plan the passes
    PassPlan plans[8];
    int np = 0;
    uint32_t done = 0;
    while (done < log_n) {
        PassPlan p;
        p.log_n = log_n; p.s0 = done + 1; p.inverse = inverse; p.coset = coset; p.first = (done == 0); p.last = 0; p.fold = (uint32_t)fold;
        if (done == 0) { p.K = log_n < 10 ? log_n : 10; p.L = 0; }
        else {
            p.L = done < 3 ? done : 3;
            uint32_t rest = log_n - done, maxk = 10 - p.L;
            // balance the remaining stages over the passes still needed
            uint32_t passes = (rest + maxk - 1) / maxk;
            p.K = (rest + passes - 1) / passes;
        }
        done += p.K;
        plans[np++] = p;
    }
    plans[np - 1].last = 1;
    for (int i = 0; i < np; i++) {
        const PassPlan& p = plans[i];
        const Fr* src = (i == 0) ? data : tmp;
        Fr* dst = (i == np - 1) ? data : tmp;
        if (np == 1) { src = data; dst = data; }
        uint32_t tile = 1u << (p.K + p.L);
        dim3 grid((1u << log_n) / tile, batch);
        uint32_t threads = tile / 4 < 32 ? 32 : (tile / 4 > 256 ? 256 : tile / 4);
        // the swizzle permutes chunks inside groups of 8 elements: pad tiny tiles up to one group
        size_t smem = (tile < 8 ? 8 : tile) * sizeof(Fr);
        OG_LAUNCHN(ctx, "k_ntt_pass", k_ntt_pass2, grid, threads, smem, p, src, dst, T->d_t2, T->d_t2n, T->n_inv);
    }
    return OG_OK;
}

}  // namespace og
