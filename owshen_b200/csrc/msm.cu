// owshen_b200/csrc/msm.cu -- bucket-method (Pippenger) multi-scalar multiplication on BN254 G1/G2
// for sm_100a.  BASELINE configs 3 and 5 and the inner engine of the batched Groth16 prover.
//
// No counterpart in the reference (SURVEY.md section 0).  Pipeline (DESIGN.md section 5.3):
//   1-3. msm_sort.cu     signed c-bit digits -> histogram -> exclusive scan -> counting-sort scatter of
//                        (point index, sign) entries: one coalesced list per bucket
//   3b. k_bucket_order   bucket ids of every group ordered by decreasing load
//   4. k_bucket_acc      one thread per bucket: XYZZ += affine point (8M+2S), accumulator in shared memory
//      k_bucket_heavy    buckets above a cap are cut into segments of one CTA each (witness-like scalars: 0/1 pile-ups)
//   5. k_reduce_level    sum_b (b+1) B_b by 8-way running sums, log_8(nb) levels; one-shot MSMs take the levels
//                        above 0 as tree sums (k_tail_sums / k_tail_finish)
//   6. k_group_total (prover) / k_horner over the windows (one-shot MSM)
// All arithmetic is 8x32-bit Montgomery limbs (fp.cuh); the kernels are bound by the integer multiply-add pipe,
// not HBM: a G1 mixed add moves 64 B + 4 B and costs ~3.5k instructions.
//
// Everything here is a template over the coordinate field F (Fq for G1, Fq2 for G2).  The file is compiled once per
// field (-DOG_MSM_G1 / -DOG_MSM_G2, see the end of the file), so that the two heavy units build in parallel and the G2
// unit can keep its Fq2 products out of line (-DOG_FP_MUL_CALL).
#include "msm.cuh"
#include "glv.cuh"

namespace og {

// ---- boundary conversions ---------------------------------------------------------------------------
template <class F> struct FieldIO;
template <> struct FieldIO<Fq> {
    static constexpr int BYTES = 32;
    static __device__ __forceinline__ Fq load(const uint8_t* p, int* flag) { return load_canonical<Fq>(p, flag); }
    static __device__ __forceinline__ void store(uint8_t* p, const Fq& v) { store_canonical(p, v); }
};
template <> struct FieldIO<Fq2> {
    static constexpr int BYTES = 64;
    static __device__ __forceinline__ Fq2 load(const uint8_t* p, int* flag) {
        return Fq2{load_canonical<Fq>(p, flag), load_canonical<Fq>(p + 32, flag)};
    }
    static __device__ __forceinline__ void store(uint8_t* p, const Fq2& v) { store_canonical(p, v.c0); store_canonical(p + 32, v.c1); }
};

template <class F>
__global__ void __launch_bounds__(128) k_points_to_mont(const uint8_t* __restrict__ in, uint64_t n, Affine<F>* __restrict__ out, int* flag) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    constexpr int B = FieldIO<F>::BYTES;
    const uint8_t* p = in + 2 * B * i;
    out[i] = Affine<F>{FieldIO<F>::load(p, flag), FieldIO<F>::load(p + B, flag)};   // all-zero stays (0,0) = infinity
}
template <class F>
__global__ void __launch_bounds__(128) k_points_from_mont(const Affine<F>* __restrict__ in, uint64_t n, uint8_t* __restrict__ out) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    constexpr int B = FieldIO<F>::BYTES;
    Affine<F> p = in[i];
    FieldIO<F>::store(out + 2 * B * i, p.x);
    FieldIO<F>::store(out + 2 * B * i + B, p.y);
}

template <class F>
int32_t points_to_mont(og_ctx* ctx, const uint8_t* d_in, uint64_t n, Affine<F>* d_out) {
    if (n) OG_LAUNCH(ctx, k_points_to_mont<F>, (unsigned)((n + 127) / 128), 128, 0, d_in, n, d_out, ctx->d_flag);
    return OG_OK;
}
template <class F>
int32_t points_to_bytes(og_ctx* ctx, const Affine<F>* d_in, uint64_t n, uint8_t* d_out) {
    if (n) OG_LAUNCH(ctx, k_points_from_mont<F>, (unsigned)((n + 127) / 128), 128, 0, d_in, n, d_out);
    return OG_OK;
}

// ---- 3b: order the buckets of every group by decreasing load ------------------------------------------------
// Bucket loads are Poisson-distributed, so a warp of 32 neighbouring buckets waits for its longest list
// (ncu: 26.5-28.4 of 32 lanes active on G1, 24.8 on G2).  A counting sort of the bucket ids by their count
// puts equal loads in the same warp and schedules the longest lists first.
constexpr uint32_t ORDER_BINS = 2048;
template <class F>   // (template only so that each translation unit gets its own copy)
__global__ void __launch_bounds__(1024) k_bucket_order(const uint32_t* __restrict__ counts, uint32_t nb, uint32_t* __restrict__ perm) {
    __shared__ uint32_t hist[ORDER_BINS];
    const uint32_t g = blockIdx.x, t = threadIdx.x;
    const uint32_t* c = counts + (size_t)g * nb;
    for (uint32_t i = t; i < ORDER_BINS; i += 1024) hist[i] = 0;
    __syncthreads();
    for (uint32_t b = t; b < nb; b += 1024) atomicAdd(&hist[ORDER_BINS - 1 - min(c[b], ORDER_BINS - 1)], 1u);
    __syncthreads();
    // exclusive scan of 2048 bins by 1024 threads (two bins each) + Hillis-Steele over the pair sums
    __shared__ uint32_t pair[1024];
    uint32_t a0 = hist[2 * t], a1 = hist[2 * t + 1];
    pair[t] = a0 + a1;
    __syncthreads();
    for (uint32_t d = 1; d < 1024; d <<= 1) {
        uint32_t v = t >= d ? pair[t - d] : 0;
        __syncthreads();
        pair[t] += v;
        __syncthreads();
    }
    uint32_t base = t ? pair[t - 1] : 0;
    hist[2 * t] = base;
    hist[2 * t + 1] = base + a0;
    __syncthreads();
    for (uint32_t b = t; b < nb; b += 1024) {
        uint32_t pos = atomicAdd(&hist[ORDER_BINS - 1 - min(c[b], ORDER_BINS - 1)], 1u);
        perm[(size_t)g * nb + pos] = g * nb + b;
    }
}

// ---- 4: bucket accumulation ----------------------------------------------------------------------------
template <class F>
__device__ __forceinline__ Affine<F> fetch_point(const Affine<F>* __restrict__ table, uint32_t e) {
    Affine<F> p = table[e >> 1];
    if (e & 1) p.y = p.y.neg();
    return p;
}

// The accumulator lives in shared memory, 16-byte chunks interleaved over the CTA's 128 threads so that every access is
// conflict-free (the layout of RedSm below): registers hold only the temporaries of one mixed addition, which buys resident
// warps in a kernel whose top stall is the fixed-latency wait of the carry chains (profiles/r1_bucket_acc_smem_sweep.md).
template <class F> struct SmAcc {
    static constexpr int CH = sizeof(F) / 16;
    uint4* base;    // [4 coordinates][CH chunks][128 threads]
    // the Fq halves of a coordinate: the coordinate itself in G1, c0 and c1 in G2.  Limbs are copied one by one with constant
    // indices: a reinterpret_cast of the coordinate, or a limb pointer, costs the G1 kernel 16 bytes of stack and 16 instructions.
    static __device__ __forceinline__ Fq& half(Fq& v, int) { return v; }
    static __device__ __forceinline__ const Fq& half(const Fq& v, int) { return v; }
    static __device__ __forceinline__ Fq& half(Fq2& v, int h) { return h ? v.c1 : v.c0; }
    static __device__ __forceinline__ const Fq& half(const Fq2& v, int h) { return h ? v.c1 : v.c0; }
    __device__ __forceinline__ F ld(int coord) const {
        uint4 q[CH];
#pragma unroll
        for (int c = 0; c < CH; c++) q[c] = base[(coord * CH + c) * 128];
        F v;
#pragma unroll
        for (int c = 0; c < CH; c++) {
            uint32_t* l = half(v, c >> 1).l + 4 * (c & 1);
            l[0] = q[c].x; l[1] = q[c].y; l[2] = q[c].z; l[3] = q[c].w;
        }
        return v;
    }
    __device__ __forceinline__ void st(int coord, const F& v) const {
#pragma unroll
        for (int h = 0; h < CH / 2; h++) {
            const Fq& x = half(v, h);
            base[(coord * CH + 2 * h) * 128] = make_uint4(x.l[0], x.l[1], x.l[2], x.l[3]);
            base[(coord * CH + 2 * h + 1) * 128] = make_uint4(x.l[4], x.l[5], x.l[6], x.l[7]);
        }
    }
};

// What the bucket kernel does differently per field.
template <class F> struct BucketAcc;
// G1: 8 CTAs of 128 threads per SM (64 registers); only the next 4-byte ENTRY is read ahead, the 64-byte gather is covered by
// the other warps (measured against 6/7 CTAs and against a prefetched point: profiles/r1_bucket_acc_smem_sweep.md).
// The two squarings of a mixed addition go through ONE out-of-line copy of the wide squarer (8 registers in, 8 out): with the
// squarer inlined twice next to eight inlined products the kernel outgrew the instruction cache (ncu: 12.7 % of the warp samples
// waiting for instructions after the wide squarer replaced the interleaved one, profiles/r2_small_ab.md).
static __device__ __noinline__ Fq fq_sqr_call(Fq a) { return a.sqr(); }
template <> struct BucketAcc<Fq> {
    static constexpr int MIN_CTAS = 8;
    static __device__ __forceinline__ Fq sqr(const Fq& a) { return fq_sqr_call(a); }
    // y3 = r (q1 - x3) - y ppp in the statement order each kernel was measured with: one order for both fields changes the
    // other field's code (G1 with G2's order: 4160 -> 4152 SASS instructions; G2 with G1's: 3112 -> 3080), and neither
    // alternative has been timed.
    static __device__ __forceinline__ Fq y3(const SmAcc<Fq>& A, const Fq& r, const Fq& q1, const Fq& x3, const Fq& ppp) {
        return r * (q1 - x3) - A.ld(1) * ppp;
    }
};
// G2: 6 CTAs (4, 5 and 6 resident CTAs were measured in round 1, profiles/r1_bucket_acc_smem_sweep.md); Fq2 products and
// squarings are out of line in this translation unit already (-DOG_FP_MUL_CALL, fp.cuh).
template <> struct BucketAcc<Fq2> {
    static constexpr int MIN_CTAS = 6;
    static __device__ __forceinline__ Fq2 sqr(const Fq2& a) { return a.sqr(); }
    static __device__ __forceinline__ Fq2 y3(const SmAcc<Fq2>& A, const Fq2& r, const Fq2& q1, const Fq2& x3, const Fq2& ppp) {
        Fq2 t = A.ld(1) * ppp;
        return r * (q1 - x3) - t;
    }
};

template <class F>
__global__ void __launch_bounds__(128, BucketAcc<F>::MIN_CTAS) k_bucket_acc(const Affine<F>* __restrict__ table, const uint32_t* __restrict__ sorted,
                                                                           const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ counts,
                                                                           uint32_t n_keys, uint32_t cap, XYZZ<F>* __restrict__ buckets,
                                                                           uint32_t* __restrict__ heavy, const uint32_t* __restrict__ perm) {
    __shared__ uint4 sm_acc[4 * SmAcc<F>::CH * 128];
    uint32_t slot_ = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot_ >= n_keys) return;
    uint32_t key = perm[slot_];
    uint32_t cnt = counts[key], off = offsets[key];
    if (cnt > cap) {                               // left to k_bucket_heavy
        uint32_t slot = atomicAdd(heavy, 1u);
        heavy[1 + slot] = key;
        buckets[key] = XYZZ<F>::inf();
        return;
    }
    SmAcc<F> A{sm_acc + threadIdx.x};
    bool inf = true;
    uint32_t e = cnt ? sorted[off] : 0;
    for (uint32_t k = 0; k < cnt; k++) {
        uint32_t en = k + 1 < cnt ? sorted[off + k + 1] : 0;
        Affine<F> q = fetch_point(table, e);
        e = en;
        if (q.is_inf()) continue;
        if (inf) { A.st(0, q.x); A.st(1, q.y); A.st(2, F::one()); A.st(3, F::one()); inf = false; continue; }
        F p = q.x * A.ld(2) - A.ld(0);
        F r = q.y * A.ld(3) - A.ld(1);
        if (p.is_zero()) {
            if (r.is_zero()) { XYZZ<F> d = XYZZ<F>::dbl_affine(q); A.st(0, d.x); A.st(1, d.y); A.st(2, d.zz); A.st(3, d.zzz); }
            else inf = true;
            continue;
        }
        // ordered so that few temporaries are live at a time (in G2, across the out-of-line multiplier calls, each Fq2 one
        // is 16 registers that would otherwise be spilled around every call): zz and zzz are updated as soon as pp / ppp exist
        F pp = BucketAcc<F>::sqr(p);
        A.st(2, A.ld(2) * pp);
        F ppp = p * pp;
        A.st(3, A.ld(3) * ppp);
        F q1 = A.ld(0) * pp;
        F x3 = BucketAcc<F>::sqr(r) - ppp - q1.dbl();
        A.st(0, x3);
        A.st(1, BucketAcc<F>::y3(A, r, q1, x3, ppp));
    }
    buckets[key] = inf ? XYZZ<F>::inf() : XYZZ<F>{A.ld(0), A.ld(1), A.ld(2), A.ld(3)};
}

// Heavy buckets (lists above the cap: witness-like scalars put 30 % of all points into bucket "1" of window 0) are cut
// into segments of `seg` entries; every segment gets a CTA, a second kernel adds the partial sums of each bucket.
// Round 1 gave a whole list to ONE CTA: 3*10^5 entries on 256 threads were 5.5 of the 13.9 ms of a witness-like 2^20 MSM.
// heavy[0] = number of heavy buckets, heavy[1 ..] = their keys, heavy[1 + n_keys ..] = first segment of each (+ total).
template <class F>   // (template only so that each translation unit gets its own copy)
__global__ void __launch_bounds__(256) k_heavy_plan(uint32_t* __restrict__ heavy, const uint32_t* __restrict__ counts, uint32_t n_keys, uint32_t seg) {
    __shared__ uint32_t part[256];
    __shared__ uint32_t carry;
    const uint32_t n_heavy = heavy[0];
    uint32_t* seg_base = heavy + 1 + n_keys;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (uint32_t base = 0; base < n_heavy; base += 256) {
        uint32_t h = base + threadIdx.x;
        uint32_t v = h < n_heavy ? (counts[heavy[1 + h]] + seg - 1) / seg : 0;
        part[threadIdx.x] = v;
        __syncthreads();
        for (uint32_t d = 1; d < 256; d <<= 1) {
            uint32_t t = threadIdx.x >= d ? part[threadIdx.x - d] : 0;
            __syncthreads();
            part[threadIdx.x] += t;
            __syncthreads();
        }
        if (h < n_heavy) seg_base[h] = carry + part[threadIdx.x] - v;
        __syncthreads();
        if (threadIdx.x == 255) carry += part[255];
        __syncthreads();
    }
    if (threadIdx.x == 0) seg_base[n_heavy] = carry;
}

template <class F, int THREADS>
__global__ void __launch_bounds__(THREADS) k_bucket_heavy(const Affine<F>* __restrict__ table, const uint32_t* __restrict__ sorted,
                                                          const uint32_t* __restrict__ offsets, const uint32_t* __restrict__ counts,
                                                          uint32_t n_keys, uint32_t seg, XYZZ<F>* __restrict__ partials,
                                                          const uint32_t* __restrict__ heavy) {
    extern __shared__ __align__(32) unsigned char smem_raw[];
    XYZZ<F>* sh = reinterpret_cast<XYZZ<F>*>(smem_raw);
    const uint32_t n_heavy = heavy[0];
    const uint32_t* seg_base = heavy + 1 + n_keys;
    const uint32_t n_seg = n_heavy ? seg_base[n_heavy] : 0;
    for (uint32_t g = blockIdx.x; g < n_seg; g += gridDim.x) {
        uint32_t lo = 0, hi = n_heavy;                          // largest h with seg_base[h] <= g
        while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (seg_base[mid] <= g) lo = mid; else hi = mid; }
        const uint32_t key = heavy[1 + lo];
        const uint32_t cnt = counts[key], off = offsets[key];
        const uint32_t k0 = (g - seg_base[lo]) * seg, k1 = k0 + seg < cnt ? k0 + seg : cnt;
        XYZZ<F> acc = XYZZ<F>::inf();
        for (uint32_t k = k0 + threadIdx.x; k < k1; k += THREADS) { Affine<F> q = fetch_point(table, sorted[off + k]); xyzz_madd_ni(&acc, &q); }
        sh[threadIdx.x] = acc;
        __syncthreads();
        for (int s = THREADS / 2; s > 0; s >>= 1) {
            if ((int)threadIdx.x < s) xyzz_add_ni(&sh[threadIdx.x], &sh[threadIdx.x + s]);
            __syncthreads();
        }
        if (threadIdx.x == 0) partials[g] = sh[0];
        __syncthreads();
    }
}

// buckets[key] = sum of the bucket's segment sums (one warp per heavy bucket)
template <class F>
__global__ void __launch_bounds__(32) k_heavy_combine(const XYZZ<F>* __restrict__ partials, uint32_t n_keys, XYZZ<F>* __restrict__ buckets,
                                                      const uint32_t* __restrict__ heavy) {
    __shared__ XYZZ<F> sh[32];
    const uint32_t n_heavy = heavy[0];
    const uint32_t* seg_base = heavy + 1 + n_keys;
    for (uint32_t h = blockIdx.x; h < n_heavy; h += gridDim.x) {
        const uint32_t s0 = seg_base[h], s1 = seg_base[h + 1];
        XYZZ<F> acc = XYZZ<F>::inf();
        for (uint32_t s = s0 + threadIdx.x; s < s1; s += 32) xyzz_add_ni(&acc, &partials[s]);
        sh[threadIdx.x] = acc;
        __syncwarp();
        for (int w = 16; w > 0; w >>= 1) {
            if ((int)threadIdx.x < w) xyzz_add_ni(&sh[threadIdx.x], &sh[threadIdx.x + w]);
            __syncwarp();
        }
        if (threadIdx.x == 0) buckets[heavy[1 + h]] = sh[0];
        __syncwarp();
    }
}

constexpr uint32_t RED_FAN_LOG2 = 3, RED_FAN = 1u << RED_FAN_LOG2;   // 8 children per parent: more threads, shorter chains
// ---- 5: weighted reduction, RED_FAN children per parent -------------------------------------------------------
// Element e of a level carries S_e (plain sum of the buckets under e) and U_e (their 0-based weighted sum
// relative to e's first bucket).  Merging children c_0..c_k, each covering 2^w_log2 buckets:
//   S_p = sum S_c;   U_p = sum U_c + 2^w_log2 * sum_c idx(c) * S_c   (running-sum trick for the last term).
// HAS_U = false is level 0 (children are raw buckets, no weighted part yet): most of the work, and one 4-coordinate
// accumulator fewer to keep in registers.  (A variant with R and T in shared memory -- 128 instead of 226 registers,
// twice the resident warps -- was measured slower, 32.7 vs 30.7 ms per step for G1: the R -> T chain, not occupancy,
// is what this kernel waits on.)
// Group operations of the reduction.  G1: ONE out-of-line copy of add and dbl with operands and result in registers (by
// value): the fully inlined kernel (three adds and a doubling, ~13k instructions) spent 15 % of its warp samples waiting for
// instructions (ncu, profiles/r2_ncu_reduce.md) at 8 resident warps per SM.  G2 keeps the inlined group law over the
// out-of-line Fq2 multiplier (128 registers of arguments would not travel in registers).
template <class F> struct RedOps {
    static __device__ __forceinline__ void add(XYZZ<F>& a, const XYZZ<F>& b) { a.add(b); }
    static __device__ __forceinline__ void dbl(XYZZ<F>& a) { a = a.dbl(); }
};
static __device__ __noinline__ XYZZ<Fq> g1_add_rv(XYZZ<Fq> a, XYZZ<Fq> b) { a.add(b); return a; }
static __device__ __noinline__ XYZZ<Fq> g1_dbl_rv(XYZZ<Fq> a) { return a.dbl(); }
template <> struct RedOps<Fq> {
    static __device__ __forceinline__ void add(XYZZ<Fq>& a, const XYZZ<Fq>& b) { a = g1_add_rv(a, b); }
    static __device__ __forceinline__ void dbl(XYZZ<Fq>& a) { a = g1_dbl_rv(a); }
};

// measured (profiles/r2_small_ab.md): G1 25.5 (registers, out-of-line ops) vs 29.6 ms (shared memory); G2 25.3 (registers, spilling) vs 24.1 ms
template <class F> constexpr bool RED_SM_DEFAULT = sizeof(F) != 32;

// (64 threads, 206 registers for G1: 4 resident CTAs per SM; asking ptxas for 6 or 8 costs spills: 26.4 / 27.6 vs 25.2 ms)
template <class F, bool HAS_U>
__global__ void __launch_bounds__(64) k_reduce_level(const XYZZ<F>* __restrict__ S_in, const XYZZ<F>* __restrict__ U_in,
                                                     uint32_t n_in, uint32_t n_out, uint32_t n_groups, uint32_t w_log2,
                                                     uint32_t fan_log2, XYZZ<F>* __restrict__ S_out, XYZZ<F>* __restrict__ U_out) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_groups * n_out) return;
    uint32_t g = t / n_out, p = t % n_out;
    const XYZZ<F>* S = S_in + (size_t)g * n_in;
    uint32_t lo = p << fan_log2, hi = min(n_in, lo + (1u << fan_log2));
    XYZZ<F> R = XYZZ<F>::inf(), T = XYZZ<F>::inf();
    for (uint32_t i = hi - 1; i > lo; i--) {
        RedOps<F>::add(R, S[i]);
        RedOps<F>::add(T, R);
    }
    RedOps<F>::add(R, S[lo]);
    for (uint32_t k = 0; k < w_log2; k++) RedOps<F>::dbl(T);
    if (HAS_U) {
        const XYZZ<F>* U = U_in + (size_t)g * n_in;
        for (uint32_t i = lo; i < hi; i++) RedOps<F>::add(T, U[i]);
    }
    S_out[(size_t)g * n_out + p] = R;
    U_out[(size_t)g * n_out + p] = T;
}

// ---- the same level with the running sums R and T in shared memory -----------------------------------------------------
// G2: R, T and one addend are 192 registers before a single temporary, so the register version spills 2.4-3 KB per thread
// (706 LDL / 586 STL in its SASS).  Here R and T live in shared memory (16-byte chunks interleaved over the CTA's 64 threads:
// conflict-free), addend coordinates are fetched where the formula uses them, and only the temporaries of ONE addition are
// in registers.  Infinity is tracked in a flag per running sum instead of zz == 0.
template <class F> struct RedSm {
    static constexpr int CH = sizeof(F) / 16, THREADS = 64;
    uint4* base;                                        // [2 sums][4 coordinates][CH chunks][64 threads]
    __device__ __forceinline__ F ld(int acc, int coord) const {
        F v; uint32_t* w = reinterpret_cast<uint32_t*>(&v);
#pragma unroll
        for (int c = 0; c < CH; c++) { uint4 q = base[((acc * 4 + coord) * CH + c) * THREADS]; w[4 * c] = q.x; w[4 * c + 1] = q.y; w[4 * c + 2] = q.z; w[4 * c + 3] = q.w; }
        return v;
    }
    __device__ __forceinline__ void st(int acc, int coord, const F& v) const {
        const uint32_t* w = reinterpret_cast<const uint32_t*>(&v);
#pragma unroll
        for (int c = 0; c < CH; c++) base[((acc * 4 + coord) * CH + c) * THREADS] = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
    }
};
template <class F> struct RedGlobalOp {                 // addend in global memory
    const XYZZ<F>* p;
    __device__ __forceinline__ bool inf() const { return p->zz.is_zero(); }
    __device__ __forceinline__ F coord(int c) const { return c == 0 ? p->x : (c == 1 ? p->y : (c == 2 ? p->zz : p->zzz)); }
};
template <class F> struct RedSmOp {                     // addend = the other running sum
    RedSm<F> M; int acc; bool is_inf;
    __device__ __forceinline__ bool inf() const { return is_inf; }
    __device__ __forceinline__ F coord(int c) const { return M.ld(acc, c); }
};

template <class F, class Op>
__device__ __forceinline__ void red_sm_add(const RedSm<F>& M, int a, bool& a_inf, const Op& o) {
    if (o.inf()) return;
    if (a_inf) {
#pragma unroll
        for (int c = 0; c < 4; c++) M.st(a, c, o.coord(c));
        a_inf = false;
        return;
    }
    F u1 = M.ld(a, 0) * o.coord(2);
    F p = o.coord(0) * M.ld(a, 2) - u1;
    F s1 = M.ld(a, 1) * o.coord(3);
    F r = o.coord(1) * M.ld(a, 3) - s1;
    if (p.is_zero()) {
        if (r.is_zero()) {                              // equal points: double through registers (rare)
            XYZZ<F> t{M.ld(a, 0), M.ld(a, 1), M.ld(a, 2), M.ld(a, 3)};
            t = t.dbl();
            M.st(a, 0, t.x); M.st(a, 1, t.y); M.st(a, 2, t.zz); M.st(a, 3, t.zzz);
        } else {
            a_inf = true;
        }
        return;
    }
    F pp = p.sqr();
    F ppp = p * pp;
    F q1 = u1 * pp;
    F x3 = r.sqr() - ppp - q1.dbl();
    M.st(a, 0, x3);
    M.st(a, 1, r * (q1 - x3) - s1 * ppp);
    M.st(a, 2, M.ld(a, 2) * o.coord(2) * pp);
    M.st(a, 3, M.ld(a, 3) * o.coord(3) * ppp);
}

template <class F, bool HAS_U>
__global__ void __launch_bounds__(64) k_reduce_level_sm(const XYZZ<F>* __restrict__ S_in, const XYZZ<F>* __restrict__ U_in,
                                                        uint32_t n_in, uint32_t n_out, uint32_t n_groups, uint32_t w_log2,
                                                        uint32_t fan_log2, XYZZ<F>* __restrict__ S_out, XYZZ<F>* __restrict__ U_out) {
    __shared__ uint4 red_sm[2 * 4 * RedSm<F>::CH * 64];
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_groups * n_out) return;
    uint32_t g = t / n_out, p = t % n_out;
    const XYZZ<F>* S = S_in + (size_t)g * n_in;
    uint32_t lo = p << fan_log2, hi = min(n_in, lo + (1u << fan_log2));
    RedSm<F> M{red_sm + threadIdx.x};
    bool r_inf = true, t_inf = true;
    for (uint32_t i = hi - 1; i > lo; i--) {
        red_sm_add(M, 0, r_inf, RedGlobalOp<F>{S + i});
        red_sm_add(M, 1, t_inf, RedSmOp<F>{M, 0, r_inf});
    }
    red_sm_add(M, 0, r_inf, RedGlobalOp<F>{S + lo});
    if (w_log2 && !t_inf) {
        XYZZ<F> tt{M.ld(1, 0), M.ld(1, 1), M.ld(1, 2), M.ld(1, 3)};
        for (uint32_t k = 0; k < w_log2; k++) tt = tt.dbl();
        M.st(1, 0, tt.x); M.st(1, 1, tt.y); M.st(1, 2, tt.zz); M.st(1, 3, tt.zzz);
    }
    if (HAS_U) {
        const XYZZ<F>* U = U_in + (size_t)g * n_in;
        for (uint32_t i = lo; i < hi; i++) red_sm_add(M, 1, t_inf, RedGlobalOp<F>{U + i});
    }
    S_out[(size_t)g * n_out + p] = r_inf ? XYZZ<F>::inf() : XYZZ<F>{M.ld(0, 0), M.ld(0, 1), M.ld(0, 2), M.ld(0, 3)};
    U_out[(size_t)g * n_out + p] = t_inf ? XYZZ<F>::inf() : XYZZ<F>{M.ld(1, 0), M.ld(1, 1), M.ld(1, 2), M.ld(1, 3)};
}

// total_g = U_g + S_g   (weights are b+1)
template <class F>
__global__ void __launch_bounds__(64) k_group_total(const XYZZ<F>* __restrict__ S, const XYZZ<F>* __restrict__ U, uint32_t n_groups,
                                                    XYZZ<F>* __restrict__ out) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups) return;
    XYZZ<F> a = U[g];
    xyzz_add_ni(&a, &S[g]);
    out[g] = a;
}

// ---- 5b: the reduction above level 0 when there are FEW groups (one-shot MSMs: groups = windows) -------------------------
// Levels 1.. of k_reduce_level then run a few thousand threads that each walk ~23 additions and up to 12 doublings in sequence:
// four such levels were 0.7 of the 5.3 ms of a 2^20-point G1 MSM and 2 of the 6 ms of a 2^18-point G2 one.  With R_p, T_p the
// level-0 sums of chunk p (2^f buckets each) a group's total is  sum_p (T_p + R_p) + 2^f sum_p p R_p,  and the weighted part
// is taken bit by bit:  sum_p p R_p = sum_k 2^k Q_k,  Q_k = sum of the R_p whose index has bit k set.  The two plain sums and the
// log2(n1) sums Q_k are independent tree reductions (one CTA each: a few strided additions per thread, then log2(threads) levels
// in shared memory); one thread per group finishes with a Horner over the bits.  Depth ~16 + 28 group operations instead of ~120.
constexpr uint32_t TAIL_THREADS = 128, TAIL_SLICE = 512;
template <class F>
__global__ void __launch_bounds__(TAIL_THREADS, 1) k_tail_sums(const XYZZ<F>* __restrict__ R, const XYZZ<F>* __restrict__ T, uint32_t n1,
                                                            uint32_t n_sums, uint32_t n_slices, XYZZ<F>* __restrict__ out) {
    __shared__ XYZZ<F> a[TAIL_THREADS];
    const uint32_t q = blockIdx.x, g = blockIdx.y, sl = blockIdx.z, tid = threadIdx.x;    // q = 0: sum T, 1: sum R, 2 + k: Q_k
    const XYZZ<F>* src = (q == 0 ? T : R) + (size_t)g * n1;
    XYZZ<F> acc = XYZZ<F>::inf();
    if (q < 2) {
        const uint32_t lo = sl * TAIL_SLICE, hi = min(n1, lo + TAIL_SLICE);
        for (uint32_t p = lo + tid; p < hi; p += TAIL_THREADS) xyzz_add_ni(&acc, &src[p]);
    } else {                                              // the n1 / 2 indices with bit k set, enumerated densely: no idle lanes
        const uint32_t k = q - 2, half = n1 >> 1, lo = sl * (TAIL_SLICE / 2), hi = min(half, lo + TAIL_SLICE / 2);
        for (uint32_t j = lo + tid; j < hi; j += TAIL_THREADS) {
            uint32_t p = ((j >> k) << (k + 1)) | (1u << k) | (j & ((1u << k) - 1));
            xyzz_add_ni(&acc, &src[p]);
        }
    }
    a[tid] = acc;
    __syncthreads();
    for (uint32_t s = TAIL_THREADS / 2; s > 0; s >>= 1) {
        if (tid < s) xyzz_add_ni(&a[tid], &a[tid + s]);
        __syncthreads();
    }
    if (tid == 0) out[((size_t)g * n_sums + q) * n_slices + sl] = a[0];
}

// total_g = sum T + sum R + 2^f * sum_k 2^k Q_k: the slices of every sum are added by a small tree, then one lane walks the
// Horner over the bits (one CTA per group so that the groups sit on different SMs)
template <class F>
__global__ void __launch_bounds__(TAIL_THREADS) k_tail_finish(const XYZZ<F>* __restrict__ partials, uint32_t n_sums, uint32_t n_slices, uint32_t f,
                                                              XYZZ<F>* __restrict__ totals) {
    __shared__ XYZZ<F> a[TAIL_THREADS];
    const uint32_t tid = threadIdx.x, n = n_sums * n_slices;      // <= 128: n_sums <= 16 sums of <= 8 slices
    if (tid < n) a[tid] = partials[(size_t)blockIdx.x * n + tid];
    __syncthreads();
    for (uint32_t s = n_slices / 2; s > 0; s >>= 1) {             // n_slices is a power of two; slice 0 of every sum collects
        if (tid < n && (tid % n_slices) < s) xyzz_add_ni(&a[tid], &a[tid + s]);
        __syncthreads();
    }
    if (tid) return;
    XYZZ<F> v = XYZZ<F>::inf();
    for (int k = (int)n_sums - 3; k >= 0; k--) {
        xyzz_dbl_ni(&v);
        xyzz_add_ni(&v, &a[(2 + k) * n_slices]);
    }
    for (uint32_t i = 0; i < f; i++) xyzz_dbl_ni(&v);
    xyzz_add_ni(&v, &a[0]);
    xyzz_add_ni(&v, &a[n_slices]);
    totals[blockIdx.x] = v;
}

template <class F>
int32_t msm_buckets(og_ctx* ctx, const Affine<F>* d_table, const uint32_t* d_sorted, const uint32_t* d_offsets,
                           const uint32_t* d_counts, uint32_t n_groups, uint32_t nb, uint64_t n_entries_max, XYZZ<F>* d_buckets,
                           XYZZ<F>* d_lvl, uint32_t* d_heavy, uint32_t* d_perm, XYZZ<F>* d_totals, bool few_groups) {
    uint32_t n_keys = n_groups * nb;
    constexpr int HT = sizeof(F) == 32 ? 256 : 128;
    OG_CUDA(ctx, cudaMemsetAsync(d_heavy, 0, sizeof(uint32_t), ctx->stream));
    OG_LAUNCHN(ctx, "k_bucket_order", k_bucket_order<F>, n_groups, 1024, 0, d_counts, nb, d_perm);
    // cap: a bucket that would keep one thread busy far longer than the average goes to a whole CTA
    // (skewed scalars: witness 0/1 values, short scalars whose top window has few distinct digits)
    uint64_t avg = n_entries_max / (n_keys ? n_keys : 1);
    uint32_t cap = (uint32_t)(4 * avg < 128 ? 128 : 4 * avg);
    OG_LAUNCHN(ctx, sizeof(F) == 32 ? "k_bucket_acc_g1" : "k_bucket_acc_g2", k_bucket_acc<F>, (n_keys + 127) / 128, 128, 0, d_table, d_sorted,
               d_offsets, d_counts, n_keys, cap, d_buckets, d_heavy, d_perm);
    {
        // segment length: long enough that the segment sums of ALL heavy buckets fit in the (still unused) reduction scratch
        // (at most n_keys / 4 heavy buckets, since each holds more than 4 x the average load)
        uint32_t seg = (uint32_t)(4 * avg < 2048 ? 2048 : 4 * avg);
        auto k_heavy = k_bucket_heavy<F, HT>;
        OG_LAUNCHN(ctx, "k_heavy_plan", k_heavy_plan<F>, 1, 256, 0, d_heavy, d_counts, n_keys, seg);
        OG_LAUNCHN(ctx, sizeof(F) == 32 ? "k_bucket_heavy_g1" : "k_bucket_heavy_g2", k_heavy, 4 * ctx->sm_count, HT, HT * sizeof(XYZZ<F>), d_table, d_sorted,
                   d_offsets, d_counts, n_keys, seg, d_lvl, d_heavy);
        OG_LAUNCH(ctx, k_heavy_combine<F>, ctx->sm_count, 32, 0, d_lvl, n_keys, d_buckets, d_heavy);
    }
    // reduction levels
    size_t lvl_stride = (size_t)n_groups * ((nb + RED_FAN - 1) / RED_FAN) + 16;
    XYZZ<F>* bufS[2] = {d_lvl, d_lvl + lvl_stride};
    XYZZ<F>* bufU[2] = {d_lvl + 2 * lvl_stride, d_lvl + 3 * lvl_stride};
    const XYZZ<F>* S_in = d_buckets;
    const XYZZ<F>* U_in = nullptr;
    uint32_t n_in = nb, w_log2 = 0;
    int pp = 0;
    do {
        uint32_t n_out = (n_in + RED_FAN - 1) >> RED_FAN_LOG2;
        uint32_t threads = n_groups * n_out;
        const char* rn = sizeof(F) == 32 ? "k_reduce_level_g1" : "k_reduce_level_g2";
        // G1: running sums in registers, group operations out of line; G2: running sums in shared memory (profiles/r2_small_ab.md;
        // the losing combination of each was removed from the library after the measurement)
        if constexpr (RED_SM_DEFAULT<F>) {
            if (U_in) { auto k = k_reduce_level_sm<F, true>; OG_LAUNCHN(ctx, rn, k, (threads + 63) / 64, 64, 0, S_in, U_in, n_in, n_out, n_groups, w_log2, RED_FAN_LOG2, bufS[pp], bufU[pp]); }
            else { auto k = k_reduce_level_sm<F, false>; OG_LAUNCHN(ctx, rn, k, (threads + 63) / 64, 64, 0, S_in, U_in, n_in, n_out, n_groups, w_log2, RED_FAN_LOG2, bufS[pp], bufU[pp]); }
        } else {
            if (U_in) { auto k = k_reduce_level<F, true>; OG_LAUNCHN(ctx, rn, k, (threads + 63) / 64, 64, 0, S_in, U_in, n_in, n_out, n_groups, w_log2, RED_FAN_LOG2, bufS[pp], bufU[pp]); }
            else { auto k = k_reduce_level<F, false>; OG_LAUNCHN(ctx, rn, k, (threads + 63) / 64, 64, 0, S_in, U_in, n_in, n_out, n_groups, w_log2, RED_FAN_LOG2, bufS[pp], bufU[pp]); }
        }
        S_in = bufS[pp]; U_in = bufU[pp];
        pp ^= 1;
        n_in = n_out;
        w_log2 += RED_FAN_LOG2;
        if (few_groups && w_log2 == RED_FAN_LOG2 && n_in >= 64 && (n_in & (n_in - 1)) == 0) {
            // one-shot MSM: everything above level 0 as independent tree sums + one Horner per group (5b above)
            uint32_t n_bits = 0;
            while ((1u << n_bits) < n_in) n_bits++;
            const uint32_t n_sums = n_bits + 2, n_slices = (n_in + TAIL_SLICE - 1) / TAIL_SLICE;
            if (n_sums * n_slices <= TAIL_THREADS) {
                XYZZ<F>* partials = bufS[pp];                           // the other ping-pong buffer: n_groups * n_in / 8 + 16 >= n_groups * n_sums * n_slices
                OG_LAUNCHN(ctx, sizeof(F) == 32 ? "k_tail_sums_g1" : "k_tail_sums_g2", k_tail_sums<F>, dim3(n_sums, n_groups, n_slices), TAIL_THREADS, 0,
                           S_in, U_in, n_in, n_sums, n_slices, partials);
                OG_LAUNCHN(ctx, sizeof(F) == 32 ? "k_tail_finish_g1" : "k_tail_finish_g2", k_tail_finish<F>, n_groups, TAIL_THREADS, 0, partials, n_sums, n_slices,
                           w_log2, d_totals);
                return OG_OK;
            }
        }
    } while (n_in > 1);
    OG_LAUNCH(ctx, k_group_total<F>, (n_groups + 63) / 64, 64, 0, S_in, U_in, n_groups, d_totals);
    return OG_OK;
}



// ---- 6: one-shot MSM = Horner over the window totals ------------------------------------------------------
// sum_w 2^(c w) T_w needs c (W - 1) ~ 240 SEQUENTIAL doublings whatever the order, and one thread's multiplier issues a
// product every ~630 cycles, so round 1's single-thread Horner cost 0.7 ms (G1) / 2.2 ms (G2) of every one-shot MSM.
// The nine products of an XYZZ doubling form three dependency levels of (2, 4, 3) independent products; four warps -- which
// sit on the SM's four schedulers -- take one product each per level and meet at barriers:
//   level 1: v = (2y)^2, xx = x^2     level 2: w = 2y v, s = x v, mm = (3xx)^2, zz' = v zz
//   level 3: m (s - x3), w y, zzz' = w zzz   with x3 = mm - 2s, y3 = m (s - x3) - w y
template <class F>
__global__ void __launch_bounds__(128) k_horner(const XYZZ<F>* __restrict__ totals, uint32_t n_windows, uint32_t c, uint8_t* __restrict__ out) {
    // acc.y is PENDING after a doubling: y = yt - ywy; the warps that need it form it themselves, so a doubling is three
    // barriers (one per dependency level) and no serial epilogue.  Who touches what: x is read in levels 1-2 and rewritten in
    // level 3; zz only by warp 3 (level 2), zzz only by warp 2 (level 3); y is published by warp 0 in level 1.
    __shared__ XYZZ<F> acc;
    __shared__ F l1v, l1xx, l2w, l2s, l2mm, yt, ywy;
    __shared__ int acc_inf;
    const int warp = threadIdx.x >> 5;
    const bool lead = (threadIdx.x & 31) == 0;
    if (threadIdx.x == 0) { acc = XYZZ<F>::inf(); acc_inf = 1; }
    __syncthreads();
    for (int w = (int)n_windows - 1; w >= 0; w--) {
        const int inf_now = acc_inf;                      // every thread reads the flag BEFORE thread 0 may rewrite it below
        __syncthreads();                                  // (racecheck found the missing barrier on the skip path)
        bool ypend = false;
        if (!inf_now) {
            for (uint32_t k = 0; k < c; k++) {
                if (lead) {                               // level 1: v = (2y)^2, xx = x^2
                    if (warp == 0) { F y = ypend ? yt - ywy : acc.y; acc.y = y; F u = y.dbl(); l1v = u.sqr(); }
                    else if (warp == 1) l1xx = acc.x.sqr();
                }
                __syncthreads();
                if (lead) {                               // level 2: w = 2y v, s = x v, mm = (3 xx)^2, zz' = v zz
                    F v = l1v;
                    if (warp == 0) { F u = acc.y.dbl(); l2w = u * v; }
                    else if (warp == 1) l2s = acc.x * v;
                    else if (warp == 2) { F xx = l1xx; F m = xx.dbl() + xx; l2mm = m.sqr(); }
                    else acc.zz = v * acc.zz;
                }
                __syncthreads();
                if (lead) {                               // level 3: m (s - x3), w y, zzz' = w zzz, x3
                    if (warp == 0) { F s = l2s; F x3 = l2mm - s.dbl(); F xx = l1xx; F m = xx.dbl() + xx; yt = m * (s - x3); }
                    else if (warp == 1) ywy = l2w * acc.y;
                    else if (warp == 2) acc.zzz = l2w * acc.zzz;
                    else { F s = l2s; acc.x = l2mm - s.dbl(); }
                }
                __syncthreads();
                ypend = true;
            }
        }
        if (threadIdx.x == 0) {
            XYZZ<F> a = acc;
            if (ypend) a.y = yt - ywy;
            xyzz_add_ni(&a, &totals[w]);
            acc = a;
            acc_inf = a.is_inf() ? 1 : 0;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        XYZZ<F> a = acc;
        Affine<F> r;
        xyzz_to_affine_ni(&r, &a);
        constexpr int B = FieldIO<F>::BYTES;
        FieldIO<F>::store(out, r.x);
        FieldIO<F>::store(out + B, r.y);
    }
}

// GLV front end of the one-shot MSM (glv.cuh): only G1 has the endomorphism, so for any other field it does nothing.
// G1: (P_i, k_i) -> (+-P_i, |k1_i|) at index i and (+-phi(P_i), |k2_i|) at index n + i; the signs go into the points and
// d_scalars is pointed at the new scalars.  phi(P_i) is MATERIALISED: applying beta at fetch time instead (entries >= n standing
// for phi of point index - n, signs in the scalars) keeps the table at 64 MB but costs a product per phi entry in the accumulation
// kernel and measured 3.61 vs 3.27 ms of accumulation at 2^20 points (profiles/r2_msm_oneshot_breakdown.md)
template <class F>
static int32_t glv_expand(og_ctx*, const uint8_t*&, uint64_t, Affine<F>*) { return OG_OK; }

#ifdef OG_MSM_G1
__global__ void __launch_bounds__(128) k_glv_expand(const uint8_t* __restrict__ scalars, uint64_t n, Fq beta, Affine<Fq>* __restrict__ pts,
                                                    uint32_t* __restrict__ sc2, int* flag) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* sp = reinterpret_cast<const uint32_t*>(scalars + 32 * i);
    uint32_t k[8], m1[8], m2[8];
#pragma unroll
    for (int j = 0; j < 8; j++) k[j] = sp[j];
    if (!Fr::canonical_lt_mod(k)) {
        atomicOr(flag, 1);
#pragma unroll
        for (int j = 0; j < 8; j++) k[j] = 0;
    }
    bool n1, n2;
    glv_decompose(k, m1, n1, m2, n2);
    Affine<Fq> p = pts[i];
    const Fq yn = p.y.neg();
    Affine<Fq> q{p.x * beta, n2 ? yn : p.y};          // (0, 0) stays (0, 0)
    if (n1) p.y = yn;
    pts[i] = p;
    pts[n + i] = q;
    uint32_t* o1 = sc2 + 8 * i;
    uint32_t* o2 = sc2 + 8 * (n + i);
#pragma unroll
    for (int j = 0; j < 8; j++) { o1[j] = m1[j]; o2[j] = m2[j]; }
}
template <>
int32_t glv_expand<Fq>(og_ctx* ctx, const uint8_t*& d_scalars, uint64_t n, Affine<Fq>* pts) {
    OG_SLOT(ctx, sc2, uint32_t, S_MSM_SCALARS, 32 * 2 * (size_t)n);
    uint32_t bl[8];
    for (int i = 0; i < 8; i++) bl[i] = Glv::beta(i);
    const Fq beta = Fq::from_canonical(bl);
    OG_LAUNCH(ctx, k_glv_expand, (unsigned)((n + 127) / 128), 128, 0, d_scalars, n, beta, pts, sc2, ctx->d_flag);
    d_scalars = reinterpret_cast<const uint8_t*>(sc2);
    return OG_OK;
}
#endif  // OG_MSM_G1

static uint32_t pick_window(uint64_t n) {
    uint32_t lg = 0;
    while ((1ull << (lg + 1)) <= n) lg++;
    int c = (int)lg - 3;
    if (c < 2) c = 2;
    if (c > 16) c = 16;
    return (uint32_t)c;
}

template <class F>
int32_t msm_dev(og_ctx* ctx, const uint8_t* d_points, const uint8_t* d_scalars, uint64_t n, uint8_t* d_out) {
    constexpr int PB = 2 * FieldIO<F>::BYTES;
    if (n >= (1ull << 28)) return OG_E_INVALID;
    if (!aligned32(d_points) || !aligned32(d_scalars)) return OG_E_INVALID;
    if (n == 0) { OG_CUDA(ctx, cudaMemsetAsync(d_out, 0, PB, ctx->stream)); return OG_OK; }
    // G1: GLV halves the scalar length (2n points, 127-bit scalars): same bucket additions, half the windows to reduce and half
    // the sequential doublings of the Horner
    const bool glv = sizeof(F) == 32 && n >= 1024;
    const uint64_t n_in = n;
    if (glv) n = 2 * n;
    uint32_t c = pick_window(n), W = glv ? (128 + c - 1) / c : msm_windows(c), nb = 1u << (c - 1);
    uint32_t n_keys = W * nb;
    OG_SLOT(ctx, pts, Affine<F>, S_MSM_POINTS, sizeof(Affine<F>) * n);
    OG_SLOT(ctx, counts, uint32_t, S_MSM_COUNTS, 4 * (size_t)n_keys);
    OG_SLOT(ctx, offsets, uint32_t, S_MSM_OFFSETS, 4 * ((size_t)n_keys + 1));
    OG_SLOT(ctx, cursor, uint32_t, S_MSM_CURSOR, 4 * (size_t)n_keys);
    OG_SLOT(ctx, sorted, uint32_t, S_MSM_SORTED, 4 * (size_t)n * W);
    OG_SLOT(ctx, buckets, XYZZ<F>, S_MSM_BUCKETS, sizeof(XYZZ<F>) * (size_t)n_keys);
    OG_SLOT(ctx, lvl, XYZZ<F>, S_MSM_SEG, sizeof(XYZZ<F>) * msm_lvl_elems(W, nb));
    OG_SLOT(ctx, heavy, uint32_t, S_MSM_HEAVY, 4 * (2 * (size_t)n_keys + 4));
    OG_SLOT(ctx, totals, XYZZ<F>, S_MSM_OUT, sizeof(XYZZ<F>) * W);
    OG_TRY(points_to_mont(ctx, d_points, n_in, pts));
    if (glv) OG_TRY(glv_expand(ctx, d_scalars, n_in, pts));
    DigitPlan plan;
    plan.scalars = reinterpret_cast<const uint32_t*>(d_scalars);
    plan.n = n; plan.scalar_stride = 0; plan.n_problems = 1;
    plan.c = c; plan.n_windows = W; plan.nb = nb;
    plan.key_stride_problem = 0; plan.key_stride_window = 1; plan.tidx_window_stride = 0;
    plan.montgomery = 0;
    OG_TRY(msm_sort_digits(ctx, plan, n_keys, counts, offsets, cursor, sorted));
    OG_TRY((msm_buckets<F>(ctx, pts, sorted, offsets, counts, W, nb, n * W, buckets, lvl, heavy, cursor, totals, true)));
    OG_LAUNCH(ctx, k_horner<F>, 1, 128, 0, totals, W, c, d_out);
    return OG_OK;
}

// ---- plain sum of affine points (post all-gather combine in the sharded MSM) ------------------------------------
template <class F, int THREADS>
__global__ void __launch_bounds__(THREADS) k_sum_points(const uint8_t* __restrict__ pts, uint64_t n, uint8_t* __restrict__ out, int* flag) {
    extern __shared__ __align__(32) unsigned char smem_raw[];
    XYZZ<F>* sh = reinterpret_cast<XYZZ<F>*>(smem_raw);
    constexpr int B = FieldIO<F>::BYTES;
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint64_t i = threadIdx.x; i < n; i += THREADS) {
        const uint8_t* p = pts + 2 * B * i;
        Affine<F> q{FieldIO<F>::load(p, flag), FieldIO<F>::load(p + B, flag)};
        xyzz_madd_ni(&acc, &q);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) xyzz_add_ni(&sh[threadIdx.x], &sh[threadIdx.x + s]);
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        Affine<F> a;
        xyzz_to_affine_ni(&a, &sh[0]);
        FieldIO<F>::store(out, a.x);
        FieldIO<F>::store(out + B, a.y);
    }
}
template <class F>
int32_t sum_points_dev(og_ctx* ctx, const uint8_t* d_points, uint64_t n, uint8_t* d_out) {
    auto k = k_sum_points<F, 128>;
    OG_LAUNCH(ctx, k, 1, 128, 128 * sizeof(XYZZ<F>), d_points, n, d_out, ctx->d_flag);
    return OG_OK;
}

// ---- fixed-base window tables ------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(64) k_build_table(Affine<F>* __restrict__ table, uint32_t n, uint32_t c, uint32_t n_windows) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Affine<F> p = table[i];
    for (uint32_t w = 1; w < n_windows; w++) {
        XYZZ<F> x = XYZZ<F>::from_affine(p);
        for (uint32_t k = 0; k < c; k++) xyzz_dbl_ni(&x);
        xyzz_to_affine_ni(&p, &x);
        table[(size_t)w * n + i] = p;
    }
}
template <class F>
int32_t build_table(og_ctx* ctx, Affine<F>* d_table, uint32_t n, uint32_t c, uint32_t n_windows) {
    if (n) OG_LAUNCH(ctx, k_build_table<F>, (n + 63) / 64, 64, 0, d_table, n, c, n_windows);
    return OG_OK;
}

// ---- fixed-base multiplication by the generators (development setup only) ------------------------------------------
// gen_table[w * 255 + d - 1] = d * 2^(8w) * G,  w < 32, d in 1..255
template <class F>
__global__ void __launch_bounds__(32) k_gen_table(Affine<F> gen, Affine<F>* __restrict__ tab) {
    uint32_t w = threadIdx.x;
    if (w >= 32) return;
    XYZZ<F> x = XYZZ<F>::from_affine(gen);
    for (uint32_t k = 0; k < 8 * w; k++) xyzz_dbl_ni(&x);
    Affine<F> base, t;
    xyzz_to_affine_ni(&base, &x);
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t d = 1; d < 256; d++) {
        xyzz_madd_ni(&acc, &base);
        xyzz_to_affine_ni(&t, &acc);
        tab[w * 255 + d - 1] = t;
    }
}
template <class F>
__global__ void __launch_bounds__(128) k_fixed_mul(const Affine<F>* __restrict__ tab, const uint8_t* __restrict__ scalars, uint64_t n,
                                                   Affine<F>* __restrict__ out, int* flag) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t* sp = reinterpret_cast<const uint32_t*>(scalars + 32 * i);
    uint32_t s[8];
#pragma unroll
    for (int j = 0; j < 8; j++) s[j] = sp[j];
    if (!Fr::canonical_lt_mod(s)) { atomicOr(flag, 1); out[i] = Affine<F>::inf(); return; }
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t w = 0; w < 32; w++) {
        uint32_t d = (s[w >> 2] >> ((w & 3) * 8)) & 255;
        if (d) xyzz_madd_ni(&acc, &tab[w * 255 + d - 1]);
    }
    Affine<F> r;
    xyzz_to_affine_ni(&r, &acc);
    out[i] = r;
}

template <class F> struct Generator;
template <> struct Generator<Fq> {
    static G1Affine get() { return G1Affine{Fq::from_u32(1), Fq::from_u32(2)}; }
};
template <> struct Generator<Fq2> {
    static G2Affine get() {
        static const uint32_t X0[8] = {0xd992f6edu, 0x46debd5cu, 0xf75edaddu, 0x674322d4u, 0x5e5c4479u, 0x426a0066u, 0x121f1e76u, 0x1800deefu};
        static const uint32_t X1[8] = {0xaef312c2u, 0x97e485b7u, 0x35a9e712u, 0xf1aa4933u, 0x31fb5d25u, 0x7260bfb7u, 0x920d483au, 0x198e9393u};
        static const uint32_t Y0[8] = {0x66fa7daau, 0x4ce6cc01u, 0x0c43d37bu, 0xe3d1e769u, 0x8dcb408fu, 0x4aab7180u, 0xdb8c6debu, 0x12c85ea5u};
        static const uint32_t Y1[8] = {0xd122975bu, 0x55acdadcu, 0x70b38ef3u, 0xbc4b3133u, 0x690c3395u, 0xec9e99adu, 0x585ff075u, 0x090689d0u};
        return G2Affine{Fq2{Fq::from_canonical(X0), Fq::from_canonical(X1)}, Fq2{Fq::from_canonical(Y0), Fq::from_canonical(Y1)}};
    }
};

template <class F>
int32_t fixed_base_mul(og_ctx* ctx, const uint8_t* d_scalars, uint64_t n, Affine<F>* d_out) {
    void*& fixed = sizeof(F) == 32 ? ctx->g1_fixed : ctx->g2_fixed;    // built on first use, freed with the context
    if (!fixed) {
        Affine<F>* tab;
        OG_CUDA(ctx, cudaMalloc(&tab, sizeof(Affine<F>) * 32 * 255));
        OG_LAUNCH(ctx, k_gen_table<F>, 1, 32, 0, Generator<F>::get(), tab);
        fixed = tab;
    }
    if (n) OG_LAUNCH(ctx, k_fixed_mul<F>, (unsigned)((n + 127) / 128), 128, 0, (const Affine<F>*)fixed, d_scalars, n, d_out, ctx->d_flag);
    return OG_OK;
}

// ---- the field of this translation unit ---------------------------------------------------------------------------
#if defined(OG_MSM_G1)
using MsmField = Fq;
#elif defined(OG_MSM_G2)
using MsmField = Fq2;
#else
#error "compile msm.cu with -DOG_MSM_G1 or -DOG_MSM_G2"
#endif
template int32_t points_to_mont<MsmField>(og_ctx*, const uint8_t*, uint64_t, Affine<MsmField>*);
template int32_t points_to_bytes<MsmField>(og_ctx*, const Affine<MsmField>*, uint64_t, uint8_t*);
template int32_t msm_buckets<MsmField>(og_ctx*, const Affine<MsmField>*, const uint32_t*, const uint32_t*, const uint32_t*, uint32_t, uint32_t,
                                       uint64_t, XYZZ<MsmField>*, XYZZ<MsmField>*, uint32_t*, uint32_t*, XYZZ<MsmField>*, bool);
template int32_t msm_dev<MsmField>(og_ctx*, const uint8_t*, const uint8_t*, uint64_t, uint8_t*);
template int32_t sum_points_dev<MsmField>(og_ctx*, const uint8_t*, uint64_t, uint8_t*);
template int32_t build_table<MsmField>(og_ctx*, Affine<MsmField>*, uint32_t, uint32_t, uint32_t);
template int32_t fixed_base_mul<MsmField>(og_ctx*, const uint8_t*, uint64_t, Affine<MsmField>*);

}  // namespace og
