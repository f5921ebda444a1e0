// owshen_b200/csrc/groth16.cu -- batched Groth16 prover for sm_100a (BASELINE config 4) plus the
// development setup.  The reference has no prover (SURVEY.md section 0); conventions are frozen in
// DESIGN.md section 4 and checked bit-for-bit against oracle/groth16.py and oracle/cpu.
//
// Once per batch:  witness  k_withdraw_witness (mimc.cu): MiMC7 Merkle path + every round value -> W[batch][n_vars+2]
// Per chunk of B proofs (default 1024; everything stays in HBM, nothing returns to the host until the proofs):
//   a, b, c      k_abc: sparse A.w, B.w over the CSR kept in L2, c = a*b
//   h            3 iNTT + 3 coset NTT (ntt.cu), k_pointwise: d = a'b' - c' written straight into
//                the scalar vector of the C multi-scalar multiplication
//   MSMs         three fixed-base MSMs per proof on precomputed window tables 2^(c*w) * P_i, so all
//                windows of a proof share one bucket set (no doublings, one reduction):
//                  A  = <[A_query; alpha1; delta1],           [w; 1; r]>                 (G1)
//                  B  = <[B2_query|supp; beta2; delta2],      [w|supp; 1; s]>            (G2)
//                  C' = <[L_query; B1_query|supp; H_query; beta1], [w_priv; r*w|supp; d; r]>  (G1)
// Once per batch:  assemble  C = C' + s*A  (the only variable-base scalar multiplication), affine, bytes.
// Identity used: s*A + r*B1 - r*s*delta1 = s*A + r*beta1 + sum (r*w_i) B1_i.
#include "groth16.cuh"
#include "mimc.cuh"
#include "msm.cuh"
#include "ntt.cuh"
#include "withdraw_circuit.hpp"
#include <stdlib.h>

namespace og {

// ---- kernels ------------------------------------------------------------------------------------------
// W[p][n_vars] = 1, W[p][n_vars+1] = r ; rs_m[p] = (r, s) in Montgomery form
__global__ void __launch_bounds__(128) k_extras(const uint8_t* __restrict__ rs, uint32_t batch, uint32_t n_vars, uint32_t w_stride,
                                                Fr* __restrict__ W, Fr* __restrict__ rs_m, int* flag) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= batch) return;
    Fr r = load_canonical<Fr>(rs + 64ull * p, flag);
    Fr s = load_canonical<Fr>(rs + 64ull * p + 32, flag);
    Fr* w = W + (size_t)p * w_stride;
    w[n_vars] = Fr::one();
    w[n_vars + 1] = r;
    rs_m[2 * p] = r;
    rs_m[2 * p + 1] = s;
}

// canonical witness bytes -> Montgomery rows (og_groth16_prove from full witnesses)
__global__ void __launch_bounds__(128) k_witness_in(const uint8_t* __restrict__ in, uint32_t batch, uint32_t n_vars, uint32_t w_stride,
                                                    Fr* __restrict__ W, int* flag) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint64_t)batch * n_vars) return;
    uint32_t p = (uint32_t)(t / n_vars), i = (uint32_t)(t % n_vars);
    W[(size_t)p * w_stride + i] = load_canonical<Fr>(in + 32 * t, flag);
}
__global__ void __launch_bounds__(128) k_witness_out(const Fr* __restrict__ W, uint32_t batch, uint32_t n_vars, uint32_t w_stride,
                                                     uint8_t* __restrict__ out) {
    uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (uint64_t)batch * n_vars) return;
    uint32_t p = (uint32_t)(t / n_vars), i = (uint32_t)(t % n_vars);
    store_canonical(out + 32 * t, W[(size_t)p * w_stride + i]);
}

struct CsrDev { const uint32_t* row_ptr; const uint32_t* col; const Fr* val; };

// abc[p][0..2][m]: a_j = <A_j, w>, b_j = <B_j, w>, c_j = a_j * b_j; rows n_constraints+i (i <= n_pub) carry x_i in A
__global__ void __launch_bounds__(128) k_abc(CsrDev A, CsrDev B, uint32_t n_constraints, uint32_t n_pub, uint32_t log_m,
                                             const Fr* __restrict__ W, uint32_t w_stride, uint32_t batch, Fr* __restrict__ abc) {
    uint32_t m = 1u << log_m;
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t p = blockIdx.y;
    if (j >= m) return;
    const Fr* w = W + (size_t)p * w_stride;
    Fr a = Fr::zero(), b = Fr::zero();
    if (j < n_constraints) {
        for (uint32_t k = A.row_ptr[j]; k < A.row_ptr[j + 1]; k++) a = a + A.val[k] * w[A.col[k]];
        for (uint32_t k = B.row_ptr[j]; k < B.row_ptr[j + 1]; k++) b = b + B.val[k] * w[B.col[k]];
    } else if (j <= n_constraints + n_pub) {
        a = w[j - n_constraints];
    }
    Fr* o = abc + (size_t)p * 3 * m;
    o[j] = a;
    o[m + j] = b;
    o[2 * m + j] = a * b;
}

// d_j = a'_j b'_j - c'_j  ->  C-scalars[p][off + j]
__global__ void __launch_bounds__(128) k_pointwise(const Fr* __restrict__ abc, uint32_t log_m, uint32_t batch, Fr* __restrict__ csc,
                                                   uint32_t csc_stride, uint32_t off) {
    uint32_t m = 1u << log_m;
    uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t p = blockIdx.y;
    if (j >= m) return;
    const Fr* o = abc + (size_t)p * 3 * m;
    csc[(size_t)p * csc_stride + off + j] = o[j] * o[m + j] - o[2 * m + j];
}

// B2-scalars[p] = [w|supp; 1; s]     C-scalars[p] = [w_priv; r*w|supp; (d filled by k_pointwise); r]
__global__ void __launch_bounds__(128) k_compose(const Fr* __restrict__ W, uint32_t w_stride, const Fr* __restrict__ rs_m,
                                                 const uint32_t* __restrict__ supp, uint32_t n_supp, uint32_t n_vars, uint32_t n_pub,
                                                 uint32_t m, Fr* __restrict__ bsc, uint32_t bsc_stride, Fr* __restrict__ csc,
                                                 uint32_t csc_stride) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t p = blockIdx.y;
    const Fr* w = W + (size_t)p * w_stride;
    Fr* bs = bsc + (size_t)p * bsc_stride;
    Fr* cs = csc + (size_t)p * csc_stride;
    uint32_t n_priv = n_vars - n_pub - 1;
    Fr r = rs_m[2 * p], s = rs_m[2 * p + 1];
    if (t < n_priv) cs[t] = w[n_pub + 1 + t];
    if (t < n_supp) {
        Fr v = w[supp[t]];
        bs[t] = v;
        cs[n_priv + t] = r * v;
    }
    if (t == 0) {
        bs[n_supp] = Fr::one();
        bs[n_supp + 1] = s;
        cs[n_priv + n_supp + m] = r;
    }
}

// proofs[p] = A || B || C  with C = C' + s*A
__global__ void __launch_bounds__(32) k_assemble_g1(const G1XYZZ* __restrict__ totA, const G1XYZZ* __restrict__ totC,
                                                    const Fr* __restrict__ rs_m, uint32_t batch, uint8_t* __restrict__ proofs) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= batch) return;
    G1XYZZ a = totA[p];
    G1Affine A;
    xyzz_to_affine_ni(&A, &a);
    uint32_t s[8];
    rs_m[2 * p + 1].to_canonical(s);
    G1XYZZ acc = G1XYZZ::inf();
    for (int i = 255; i >= 0; i--) {
        xyzz_dbl_ni(&acc);
        if ((s[i >> 5] >> (i & 31)) & 1) xyzz_madd_ni(&acc, &A);
    }
    G1XYZZ c = totC[p];
    xyzz_add_ni(&c, &acc);
    G1Affine C;
    xyzz_to_affine_ni(&C, &c);
    uint8_t* o = proofs + 256ull * p;
    store_canonical(o, A.x); store_canonical(o + 32, A.y);
    store_canonical(o + 192, C.x); store_canonical(o + 224, C.y);
}
__global__ void __launch_bounds__(32) k_assemble_g2(const G2XYZZ* __restrict__ totB, uint32_t batch, uint8_t* __restrict__ proofs) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= batch) return;
    G2XYZZ b = totB[p];
    G2Affine B;
    xyzz_to_affine_ni(&B, &b);
    uint8_t* o = proofs + 256ull * p + 64;
    store_canonical(o, B.x.c0); store_canonical(o + 32, B.x.c1);
    store_canonical(o + 64, B.y.c0); store_canonical(o + 96, B.y.c1);
}

__global__ void __launch_bounds__(128) k_public_out(const Fr* __restrict__ W, uint32_t w_stride, uint32_t batch, uint32_t n_pub,
                                                    uint8_t* __restrict__ out) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= batch * n_pub) return;
    uint32_t p = t / n_pub, i = t % n_pub;
    store_canonical(out + 32ull * t, W[(size_t)p * w_stride + 1 + i]);
}

}  // namespace og

// ---- proving key ----------------------------------------------------------------------------------------
using namespace og;

struct og_pk {
    int device = -1;                     // the GPU the tables live on (a key is bound to the device it was loaded on)
    uint32_t depth = 0, n_constraints = 0, n_vars = 0, n_pub = 0, log_m = 0;
    uint32_t n_supp = 0;                 // |{i : B_query[i] != infinity}|
    // window size per MSM: index 0 = A (G1), 1 = B (G2), 2 = C' (G1); nb = 2^(c-1) buckets per proof
    uint32_t c[3] = {0, 0, 0}, n_windows[3] = {0, 0, 0}, nb[3] = {0, 0, 0};
    uint32_t max_nb = 0, max_windows = 0;
    uint32_t nA = 0, nB = 0, nC = 0;     // points per MSM (incl. the folded fixed terms)
    // device
    uint32_t *a_ptr = nullptr, *a_col = nullptr, *b_ptr = nullptr, *b_col = nullptr, *supp = nullptr;
    Fr *a_val = nullptr, *b_val = nullptr;
    G1Affine *tabA = nullptr, *tabC = nullptr;
    G2Affine* tabB = nullptr;
};

namespace og {

struct Reader {
    const uint8_t* p; uint64_t left; bool ok = true;
    const uint8_t* take(uint64_t n) { if (n > left) { ok = false; return nullptr; } const uint8_t* r = p; p += n; left -= n; return r; }
    uint32_t u32() { const uint8_t* q = take(4); uint32_t v = 0; if (q) memcpy(&v, q, 4); return v; }
};

static bool all_zero(const uint8_t* p, size_t n) { for (size_t i = 0; i < n; i++) if (p[i]) return false; return true; }

static uint32_t env_u32(const char* name, uint32_t dflt) {
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    long x = strtol(v, nullptr, 10);
    return x > 0 ? (uint32_t)x : dflt;
}

template <class T>
static int32_t upload(og_ctx* ctx, T** dst, const void* src, size_t bytes) {
    OG_CUDA(ctx, cudaMalloc(dst, bytes ? bytes : 1));
    if (bytes) OG_CUDA(ctx, cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return OG_OK;
}

static int32_t upload_csr(og_ctx* ctx, Reader& rd, uint32_t n_rows, uint32_t n_vars, uint32_t** d_ptr, uint32_t** d_col, Fr** d_val) {
    uint32_t nnz = rd.u32();
    const uint8_t* ptr = rd.take(4ull * (n_rows + 1));
    const uint8_t* col = rd.take(4ull * nnz);
    const uint8_t* val = rd.take(32ull * nnz);
    if (!rd.ok) return OG_E_ENCODING;
    std::vector<uint32_t> hp(n_rows + 1), hc(nnz);
    memcpy(hp.data(), ptr, 4ull * (n_rows + 1));
    memcpy(hc.data(), col, 4ull * nnz);
    if (hp[0] != 0 || hp[n_rows] != nnz) return OG_E_ENCODING;
    for (uint32_t i = 0; i < n_rows; i++) if (hp[i] > hp[i + 1]) return OG_E_ENCODING;
    for (uint32_t i = 0; i < nnz; i++) if (hc[i] >= n_vars) return OG_E_ENCODING;
    std::vector<Fr> hv(nnz);
    for (uint32_t i = 0; i < nnz; i++) if (!host_load(hv[i], val + 32ull * i)) return OG_E_ENCODING;
    OG_TRY(upload(ctx, d_ptr, hp.data(), 4ull * (n_rows + 1)));
    OG_TRY(upload(ctx, d_col, hc.data(), 4ull * nnz));
    OG_TRY(upload(ctx, d_val, hv.data(), sizeof(Fr) * (size_t)nnz));
    OG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // host vectors die at return
    return OG_OK;
}

void pk_free(og_pk* pk) {
    if (!pk) return;
    if (pk->device >= 0) cudaSetDevice(pk->device);    // the key may outlive the context that loaded it
    cudaFree(pk->a_ptr); cudaFree(pk->a_col); cudaFree(pk->b_ptr); cudaFree(pk->b_col); cudaFree(pk->supp);
    cudaFree(pk->a_val); cudaFree(pk->b_val); cudaFree(pk->tabA); cudaFree(pk->tabC); cudaFree(pk->tabB);
    delete pk;
}

// stage a base-point list (boundary bytes), convert it to Montgomery form and extend it to the window table of MSM `which`
template <class F>
static int32_t load_table(og_ctx* ctx, const og_pk* pk, int which, const std::vector<uint8_t>& pts, uint32_t n, Affine<F>** table) {
    uint8_t* stage;
    OG_TRY(upload(ctx, &stage, pts.data(), pts.size()));
    if (cudaMalloc(table, sizeof(Affine<F>) * (size_t)n * pk->n_windows[which]) != cudaSuccess) { cudaFree(stage); return OG_E_NOMEM; }
    int32_t rc = points_to_mont(ctx, stage, n, *table);
    if (rc == OG_OK) rc = build_table(ctx, *table, n, pk->c[which], pk->n_windows[which]);
    cudaStreamSynchronize(ctx->stream); cudaFree(stage);
    return rc;
}

int32_t pk_load(og_ctx* ctx, const uint8_t* bytes, uint64_t len, og_pk** out) {
    Reader rd{bytes, len};
    const uint8_t* magic = rd.take(4);
    if (!magic || memcmp(magic, "OGPK", 4) != 0) return OG_E_ENCODING;
    if (rd.u32() != 1) return OG_E_ENCODING;
    og_pk* pk = new og_pk();
    pk->device = ctx->device;
    pk->depth = rd.u32(); pk->n_constraints = rd.u32(); pk->n_vars = rd.u32(); pk->n_pub = rd.u32(); pk->log_m = rd.u32();
    if (!rd.ok || pk->log_m > 24 || pk->n_vars == 0 || pk->n_pub > (1u << 16) || pk->n_pub + 1 > pk->n_vars ||
        (uint64_t)pk->n_constraints + pk->n_pub + 1 > (1ull << pk->log_m)) { delete pk; return OG_E_ENCODING; }
    const uint32_t nv = pk->n_vars, n_priv = nv - pk->n_pub - 1, m = 1u << pk->log_m;
    const uint8_t* alpha1 = rd.take(64); const uint8_t* beta1 = rd.take(64); const uint8_t* beta2 = rd.take(128);
    const uint8_t* delta1 = rd.take(64); const uint8_t* delta2 = rd.take(128);
    const uint8_t* qa = rd.take(64ull * nv); const uint8_t* qb1 = rd.take(64ull * nv); const uint8_t* qb2 = rd.take(128ull * nv);
    const uint8_t* ql = rd.take(64ull * n_priv); const uint8_t* qh = rd.take(64ull * m);
    if (!rd.ok) { delete pk; return OG_E_ENCODING; }

    // support of the B queries (v_i(tau) != 0)
    std::vector<uint32_t> supp;
    for (uint32_t i = 0; i < nv; i++)
        if (!all_zero(qb1 + 64ull * i, 64) || !all_zero(qb2 + 128ull * i, 128)) supp.push_back(i);
    pk->n_supp = (uint32_t)supp.size();
    // measured on B200 (profiles/r1_window_sweep.md): 15 bits for A and B, 16 for C' (3x the points); OG_WINDOW_BITS overrides all three, OG_C_A / OG_C_B / OG_C_C one each
    const uint32_t dflt[3] = {15, 15, 16};
    const char* names[3] = {"OG_C_A", "OG_C_B", "OG_C_C"};
    for (int k = 0; k < 3; k++) {
        uint32_t c = env_u32(names[k], env_u32("OG_WINDOW_BITS", dflt[k]));
        if (c < 2 || c > 16) c = dflt[k];
        pk->c[k] = c; pk->n_windows[k] = msm_windows(c); pk->nb[k] = 1u << (c - 1);
        if (pk->nb[k] > pk->max_nb) pk->max_nb = pk->nb[k];
        if (pk->n_windows[k] > pk->max_windows) pk->max_windows = pk->n_windows[k];
    }
    pk->nA = nv + 2; pk->nB = pk->n_supp + 2; pk->nC = n_priv + pk->n_supp + m + 1;

    // assemble the base-point lists in boundary bytes, then convert + extend on the GPU
    std::vector<uint8_t> hA(64ull * pk->nA), hB(128ull * pk->nB), hC(64ull * pk->nC);
    memcpy(hA.data(), qa, 64ull * nv); memcpy(hA.data() + 64ull * nv, alpha1, 64); memcpy(hA.data() + 64ull * (nv + 1), delta1, 64);
    for (uint32_t k = 0; k < pk->n_supp; k++) {
        memcpy(hB.data() + 128ull * k, qb2 + 128ull * supp[k], 128);
        memcpy(hC.data() + 64ull * (n_priv + k), qb1 + 64ull * supp[k], 64);
    }
    memcpy(hB.data() + 128ull * pk->n_supp, beta2, 128); memcpy(hB.data() + 128ull * (pk->n_supp + 1), delta2, 128);
    memcpy(hC.data(), ql, 64ull * n_priv);
    memcpy(hC.data() + 64ull * (n_priv + pk->n_supp), qh, 64ull * m);
    memcpy(hC.data() + 64ull * (n_priv + pk->n_supp + m), beta1, 64);

    int32_t rc = OG_OK;
    auto fail = [&](int32_t code) { pk_free(pk); return code; };
    if ((rc = clear_flag(ctx)) != OG_OK) return fail(rc);
    if ((rc = load_table(ctx, pk, 0, hA, pk->nA, &pk->tabA)) != OG_OK) return fail(rc);
    if ((rc = load_table(ctx, pk, 2, hC, pk->nC, &pk->tabC)) != OG_OK) return fail(rc);
    if ((rc = load_table(ctx, pk, 1, hB, pk->nB, &pk->tabB)) != OG_OK) return fail(rc);
    if ((rc = upload(ctx, &pk->supp, supp.data(), 4ull * supp.size())) != OG_OK) return fail(rc);
    cudaStreamSynchronize(ctx->stream);
    if ((rc = upload_csr(ctx, rd, pk->n_constraints, nv, &pk->a_ptr, &pk->a_col, &pk->a_val)) != OG_OK) return fail(rc);
    if ((rc = upload_csr(ctx, rd, pk->n_constraints, nv, &pk->b_ptr, &pk->b_col, &pk->b_val)) != OG_OK) return fail(rc);
    if ((rc = check_flag(ctx)) != OG_OK) return fail(rc);
    *out = pk;
    return OG_OK;
}

bool pk_on_device_of(const og_pk* pk, const og_ctx* ctx) { return pk && ctx && pk->device == ctx->device; }

void pk_info(const og_pk* pk, uint32_t* n_vars, uint32_t* n_pub, uint32_t* log_m, uint32_t* depth) {
    if (n_vars) *n_vars = pk->n_vars;
    if (n_pub) *n_pub = pk->n_pub;
    if (log_m) *log_m = pk->log_m;
    if (depth) *depth = pk->depth;
}

// ---- the prover ---------------------------------------------------------------------------------------------
// A batch is cut into chunks of CB proofs that run one after another on the context's stream and share one set of
// chunk scratch.
struct ChunkBufs {
    Fr *W, *rs_m, *abc, *ntt_tmp, *bsc, *csc;
    uint32_t *counts, *offsets, *cursor, *sorted, *heavy;
    void *buckets, *lvl;                 // bucket and reduction scratch of one MSM (sized for G2; the MSMs run one after another)
    G1XYZZ *totA, *totC;
    G2XYZZ* totB;
    uint32_t w_stride, bsc_stride, csc_stride;
};

// W, rs_m and the per-proof totals cover the whole batch; everything else is per chunk of B proofs
static int32_t alloc_chunk(og_ctx* ctx, const og_pk* pk, uint32_t batch, uint32_t B, ChunkBufs& b) {
    const uint32_t m = 1u << pk->log_m;
    b.w_stride = pk->n_vars + 2;
    b.bsc_stride = pk->nB;
    b.csc_stride = pk->nC;
    size_t max_pts = pk->nC > pk->nA ? pk->nC : pk->nA;
    size_t n_keys = (size_t)B * pk->max_nb;
    b.W = (Fr*)ctx->slot(S_PR_WIT, sizeof(Fr) * (size_t)batch * b.w_stride);
    b.rs_m = (Fr*)ctx->slot(S_PR_MISC, sizeof(Fr) * 2 * (size_t)batch);
    b.abc = (Fr*)ctx->slot(S_PR_ABC, sizeof(Fr) * (size_t)B * 3 * m * 2);
    b.bsc = (Fr*)ctx->slot(S_PR_SCALARS, sizeof(Fr) * (size_t)B * (b.bsc_stride + b.csc_stride));
    b.sorted = (uint32_t*)ctx->slot(S_PR_SORTED, 4 * (size_t)B * max_pts * pk->max_windows);
    b.counts = (uint32_t*)ctx->slot(S_PR_COUNTS, 4 * n_keys);
    b.offsets = (uint32_t*)ctx->slot(S_PR_OFFSETS, 4 * (n_keys + 1));
    b.cursor = (uint32_t*)ctx->slot(S_PR_CURSOR, 4 * n_keys);
    b.heavy = (uint32_t*)ctx->slot(S_PR_HEAVY, 4 * (2 * n_keys + 4));
    b.buckets = ctx->slot(S_PR_BUCKETS, sizeof(G2XYZZ) * n_keys);
    b.lvl = ctx->slot(S_PR_SEG, sizeof(G2XYZZ) * msm_lvl_elems(B, pk->max_nb));
    b.totA = (G1XYZZ*)ctx->slot(S_PR_SUMS, (sizeof(G1XYZZ) * 2 + sizeof(G2XYZZ)) * (size_t)batch);
    if (!b.W || !b.rs_m || !b.abc || !b.bsc || !b.sorted || !b.counts || !b.offsets || !b.cursor || !b.heavy || !b.buckets || !b.lvl || !b.totA)
        return OG_E_NOMEM;
    b.ntt_tmp = b.abc + (size_t)B * 3 * m;
    b.csc = b.bsc + (size_t)B * b.bsc_stride;
    b.totC = b.totA + batch;
    b.totB = reinterpret_cast<G2XYZZ*>(b.totC + batch);
    return OG_OK;
}

template <class F>
static int32_t run_msm(og_ctx* ctx, const og_pk* pk, int which, ChunkBufs& b, uint32_t B, const Affine<F>* table, uint32_t n_pts,
                       const Fr* scalars, uint32_t stride, XYZZ<F>* totals) {
    DigitPlan plan;
    plan.scalars = reinterpret_cast<const uint32_t*>(scalars);
    plan.n = n_pts; plan.scalar_stride = stride; plan.n_problems = B;
    plan.c = pk->c[which]; plan.n_windows = pk->n_windows[which]; plan.nb = pk->nb[which];
    plan.key_stride_problem = 1; plan.key_stride_window = 0; plan.tidx_window_stride = n_pts;
    plan.montgomery = 1;
    uint32_t n_keys = B * pk->nb[which];
    OG_TRY(msm_sort_digits(ctx, plan, n_keys, b.counts, b.offsets, b.cursor, b.sorted));
    return msm_buckets(ctx, table, b.sorted, b.offsets, b.counts, B, pk->nb[which], (uint64_t)B * n_pts * pk->n_windows[which],
                       static_cast<XYZZ<F>*>(b.buckets), static_cast<XYZZ<F>*>(b.lvl), b.heavy, b.cursor, totals);
}

// where a chunk's witness rows come from
struct WitnessSource {
    const uint8_t *d_null = nullptr, *d_sec = nullptr, *d_rec = nullptr, *d_sib = nullptr;   // secret inputs (prove_withdraw)
    const uint32_t* d_bits = nullptr;
    const uint8_t* d_wit = nullptr;                                                         // or full witnesses (prove)
    uint8_t* d_public = nullptr;
};

// proofs [off, off+B) on the current stream: witness rows -> per-proof MSM totals -> proof bytes
static int32_t prove_chunk(og_ctx* ctx, const og_pk* pk, ChunkBufs& b, const WitnessSource& src, uint32_t off, uint32_t B,
                           const uint8_t* d_rs, uint8_t* d_proofs) {
    const uint32_t m = 1u << pk->log_m, n_priv = pk->n_vars - pk->n_pub - 1;
    Fr* W = b.W + (size_t)off * b.w_stride;
    Fr* rs_m = b.rs_m + 2 * (size_t)off;
    if (src.d_wit) {
        uint64_t tot = (uint64_t)B * pk->n_vars;
        OG_LAUNCH(ctx, k_witness_in, (unsigned)((tot + 127) / 128), 128, 0, src.d_wit + 32ull * off * pk->n_vars, B, pk->n_vars, b.w_stride, W, ctx->d_flag);
    } else {
        WithdrawLayout L = WithdrawLayout::make(pk->depth);
        OG_TRY(withdraw_witness_strided_dev(ctx, L, b.w_stride, src.d_null + 32ull * off, src.d_sec + 32ull * off, src.d_rec + 32ull * off,
                                            src.d_sib + 32ull * off * pk->depth, src.d_bits + off, B, W));
        if (src.d_public) OG_LAUNCH(ctx, k_public_out, (B * pk->n_pub + 127) / 128, 128, 0, W, b.w_stride, B, pk->n_pub, src.d_public + 32ull * off * pk->n_pub);
    }
    OG_LAUNCH(ctx, k_extras, (B + 127) / 128, 128, 0, d_rs + 64ull * off, B, pk->n_vars, b.w_stride, W, rs_m, ctx->d_flag);
    CsrDev A{pk->a_ptr, pk->a_col, pk->a_val}, Bm{pk->b_ptr, pk->b_col, pk->b_val};
    OG_LAUNCH(ctx, k_abc, dim3((m + 127) / 128, B), 128, 0, A, Bm, pk->n_constraints, pk->n_pub, pk->log_m, W, b.w_stride, B, b.abc);
    OG_TRY(ntt_mont_dev(ctx, b.abc, b.ntt_tmp, pk->log_m, 3 * B, 1, 0, 1));      // 1/n folded into ...
    OG_TRY(ntt_mont_dev(ctx, b.abc, b.ntt_tmp, pk->log_m, 3 * B, 0, 1, 2));      // ... the coset factors of the forward transform
    uint32_t mx = n_priv > pk->n_supp ? n_priv : pk->n_supp;
    OG_LAUNCH(ctx, k_compose, dim3((mx + 127) / 128, B), 128, 0, W, b.w_stride, rs_m, pk->supp, pk->n_supp, pk->n_vars, pk->n_pub, m,
              b.bsc, b.bsc_stride, b.csc, b.csc_stride);
    OG_LAUNCH(ctx, k_pointwise, dim3((m + 127) / 128, B), 128, 0, b.abc, pk->log_m, B, b.csc, b.csc_stride, n_priv + pk->n_supp);
    OG_TRY(run_msm(ctx, pk, 0, b, B, pk->tabA, pk->nA, W, b.w_stride, b.totA + off));
    OG_TRY(run_msm(ctx, pk, 2, b, B, pk->tabC, pk->nC, b.csc, b.csc_stride, b.totC + off));
    OG_TRY(run_msm(ctx, pk, 1, b, B, pk->tabB, pk->nB, b.bsc, b.bsc_stride, b.totB + off));
    OG_LAUNCH(ctx, k_assemble_g1, (B + 31) / 32, 32, 0, b.totA + off, b.totC + off, rs_m, B, d_proofs + 256ull * off);
    OG_LAUNCH(ctx, k_assemble_g2, (B + 31) / 32, 32, 0, b.totB + off, B, d_proofs + 256ull * off);
    return OG_OK;
}

// offsets into the sorted digit lists and bucket keys are 32-bit: bound the chunk so they cannot overflow
static uint32_t chunk_limit(const og_pk* pk) {
    uint64_t max_pts = pk->nC > pk->nA ? pk->nC : pk->nA;
    uint64_t by_entries = 0xF0000000ull / (max_pts * pk->max_windows);
    uint64_t by_keys = 0x7FFFFFFFull / pk->max_nb;
    uint64_t lim = by_entries < by_keys ? by_entries : by_keys;
    return (uint32_t)(lim < 1 ? 1 : lim);
}

// OG_CHUNK proofs per chunk (default 1024 = the whole BASELINE batch, ~28 GB of scratch; profiles/r2_lanes_sweep.md)
static uint32_t chunk_size(const og_pk* pk, uint32_t batch) {
    uint32_t c = env_u32("OG_CHUNK", 1024);
    if (c > chunk_limit(pk)) c = chunk_limit(pk);
    return c < batch ? c : batch;
}

static int32_t prove_batch(og_ctx* ctx, const og_pk* pk, const WitnessSource& src, uint32_t batch, const uint8_t* d_rs, uint8_t* d_proofs) {
    const uint32_t CB = chunk_size(pk, batch);
    ChunkBufs b;
    OG_TRY(alloc_chunk(ctx, pk, batch, CB, b));
    for (uint32_t off = 0; off < batch; off += CB) OG_TRY(prove_chunk(ctx, pk, b, src, off, batch - off < CB ? batch - off : CB, d_rs, d_proofs));
    return OG_OK;
}

int32_t prove_withdraw_dev(og_ctx* ctx, const og_pk* pk, const uint8_t* d_null, const uint8_t* d_sec, const uint8_t* d_rec,
                           const uint8_t* d_sib, const uint32_t* d_bits, uint32_t batch, const uint8_t* d_rs, uint8_t* d_proofs,
                           uint8_t* d_public) {
    if (pk->depth == 0) return OG_E_INVALID;
    if (batch == 0) return OG_OK;
    WithdrawLayout L = WithdrawLayout::make(pk->depth);
    if (L.n_vars != pk->n_vars) return OG_E_INVALID;
    WitnessSource src;
    src.d_null = d_null; src.d_sec = d_sec; src.d_rec = d_rec; src.d_sib = d_sib; src.d_bits = d_bits; src.d_public = d_public;
    return prove_batch(ctx, pk, src, batch, d_rs, d_proofs);
}

int32_t prove_witness_dev(og_ctx* ctx, const og_pk* pk, const uint8_t* d_wit, uint32_t batch, const uint8_t* d_rs, uint8_t* d_proofs) {
    if (batch == 0) return OG_OK;
    WitnessSource src;
    src.d_wit = d_wit;
    return prove_batch(ctx, pk, src, batch, d_rs, d_proofs);
}

// debug / parity probe: d_j for one witness (canonical bytes on device in and out)
int32_t h_evals_dev(og_ctx* ctx, const og_pk* pk, const uint8_t* d_wit, uint8_t* d_out) {
    ChunkBufs b;
    OG_TRY(alloc_chunk(ctx, pk, 1, 1, b));
    const uint32_t m = 1u << pk->log_m, n_priv = pk->n_vars - pk->n_pub - 1;
    OG_LAUNCH(ctx, k_witness_in, (pk->n_vars + 127) / 128, 128, 0, d_wit, 1, pk->n_vars, b.w_stride, b.W, ctx->d_flag);
    CsrDev A{pk->a_ptr, pk->a_col, pk->a_val}, Bm{pk->b_ptr, pk->b_col, pk->b_val};
    OG_LAUNCH(ctx, k_abc, dim3((m + 127) / 128, 1), 128, 0, A, Bm, pk->n_constraints, pk->n_pub, pk->log_m, b.W, b.w_stride, 1, b.abc);
    OG_TRY(ntt_mont_dev(ctx, b.abc, b.ntt_tmp, pk->log_m, 3, 1, 0, 1));
    OG_TRY(ntt_mont_dev(ctx, b.abc, b.ntt_tmp, pk->log_m, 3, 0, 1, 2));
    OG_LAUNCH(ctx, k_pointwise, dim3((m + 127) / 128, 1), 128, 0, b.abc, pk->log_m, 1, b.csc, b.csc_stride, n_priv + pk->n_supp);
    return mimc_from_mont_dev(ctx, b.csc + n_priv + pk->n_supp, m, d_out);
}

int32_t withdraw_witness_bytes_dev(og_ctx* ctx, uint32_t depth, const uint8_t* d_null, const uint8_t* d_sec, const uint8_t* d_rec,
                                   const uint8_t* d_sib, const uint32_t* d_bits, uint32_t batch, uint8_t* d_out) {
    WithdrawLayout L = WithdrawLayout::make(depth);
    Fr* W = (Fr*)ctx->slot(S_PR_WIT, sizeof(Fr) * (size_t)batch * L.n_vars);
    if (!W) return OG_E_NOMEM;
    OG_TRY(withdraw_witness_strided_dev(ctx, L, L.n_vars, d_null, d_sec, d_rec, d_sib, d_bits, batch, W));
    uint64_t tot = (uint64_t)batch * L.n_vars;
    OG_LAUNCH(ctx, k_witness_out, (unsigned)((tot + 127) / 128), 128, 0, W, batch, L.n_vars, L.n_vars, d_out);
    return OG_OK;
}

}  // namespace og
