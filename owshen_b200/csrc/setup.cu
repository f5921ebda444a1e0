// owshen_b200/csrc/setup.cu -- development Groth16 setup for the withdraw statement ("toxic waste in
// the clear": tau, alpha, beta, gamma, delta are inputs, so that every pk/vk byte is reproducible and
// can be compared with oracle/groth16.py).  A production deployment would load a ceremony's key with
// og_load_pk instead.  QAP evaluation at tau is ~10^5 host field operations; the ~1.6*10^5
// fixed-base scalar multiplications run on the GPU (msm.cu: fixed_base_mul).
// Conventions: DESIGN.md section 4 (domain, input-consistency rows, coset-Lagrange H query).
#include "groth16.cuh"
#include "msm.cuh"
#include "withdraw_circuit.hpp"

namespace og {

static Fr host_root_of_unity(uint32_t log_n) {
    uint32_t e[8];
    for (int i = 0; i < 8; i++) e[i] = FrParams::mod(i);
    e[0] -= 1;
    for (uint32_t k = 0; k < log_n; k++) {
        for (int i = 0; i < 7; i++) e[i] = (e[i] >> 1) | (e[i + 1] << 31);
        e[7] >>= 1;
    }
    return Fr::from_u32(7).pow(e);
}

static Fr host_pow_u64(Fr base, uint64_t e) {
    Fr acc = Fr::one();
    for (; e; e >>= 1) { if (e & 1) acc = acc * base; base = base.sqr(); }
    return acc;
}

// [L_j(x)] for the size-2^log_m domain, L_j(x) = (x^m - 1)/m * w^j / (x - w^j); false if x is in the domain
static bool lagrange_at(const Fr& x, uint32_t log_m, std::vector<Fr>& out) {
    const uint32_t m = 1u << log_m;
    Fr omega = host_root_of_unity(log_m);
    Fr xm = host_pow_u64(x, m);
    Fr z = xm - Fr::one();
    if (z.is_zero()) return false;
    Fr zm = z * Fr::from_u32(m).inv();
    std::vector<Fr> wj(m), den(m), pre(m);
    Fr w = Fr::one();
    for (uint32_t j = 0; j < m; j++) { wj[j] = w; den[j] = x - w; w = w * omega; }
    // batch inversion
    Fr acc = Fr::one();
    for (uint32_t j = 0; j < m; j++) { pre[j] = acc; acc = acc * den[j]; }
    Fr inv = acc.inv();
    out.resize(m);
    for (uint32_t j = m; j-- > 0;) {
        Fr dinv = inv * pre[j];
        inv = inv * den[j];
        out[j] = zm * wj[j] * dinv;
    }
    return true;
}

static void put_u32(std::vector<uint8_t>& v, uint32_t x) { for (int i = 0; i < 4; i++) v.push_back((uint8_t)(x >> (8 * i))); }
static void put_bytes(std::vector<uint8_t>& v, const uint8_t* p, size_t n) { v.insert(v.end(), p, p + n); }
static void put_csr(std::vector<uint8_t>& v, const Csr& M) {
    put_u32(v, (uint32_t)M.col.size());
    put_bytes(v, reinterpret_cast<const uint8_t*>(M.row_ptr.data()), 4 * M.row_ptr.size());
    put_bytes(v, reinterpret_cast<const uint8_t*>(M.col.data()), 4 * M.col.size());
    for (const Fr& c : M.val) { uint8_t b[32]; host_store(b, c); put_bytes(v, b, 32); }
}

// out = boundary bytes of scalars[i] * generator (G1 or G2) for the n canonical scalars in s, through the setup's scratch slots
template <class F>
static int32_t generator_mul(og_ctx* ctx, const std::vector<uint8_t>& s, uint64_t n, uint8_t* d_s, uint8_t* d_pts, uint8_t* d_bytes,
                             std::vector<uint8_t>& out) {
    out.resize(sizeof(Affine<F>) * n);
    OG_CUDA(ctx, cudaMemcpyAsync(d_s, s.data(), 32 * n, cudaMemcpyHostToDevice, ctx->stream));
    OG_TRY(fixed_base_mul<F>(ctx, d_s, n, reinterpret_cast<Affine<F>*>(d_pts)));
    OG_TRY(points_to_bytes(ctx, reinterpret_cast<Affine<F>*>(d_pts), n, d_bytes));
    OG_CUDA(ctx, cudaMemcpyAsync(out.data(), d_bytes, out.size(), cudaMemcpyDeviceToHost, ctx->stream));
    OG_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return OG_OK;
}

int32_t setup_withdraw(og_ctx* ctx, uint32_t depth, const uint8_t* toxic160, uint8_t* pk_out, uint64_t* pk_len,
                       uint8_t* vk_out, uint64_t* vk_len) {
    if (depth == 0 || depth > 32 || !pk_len || !vk_len) return OG_E_INVALID;
    WithdrawLayout L = WithdrawLayout::make(depth);
    const uint32_t nv = L.n_vars, n_pub = WITHDRAW_N_PUB, n_priv = nv - n_pub - 1;
    const uint32_t log_m = groth16_domain_log(L.n_constraints, n_pub), m = 1u << log_m;
    // sizes first, so callers can allocate
    uint64_t csr_bound = 0;   // filled after the build; the size query needs the build as well (cheap)
    R1cs cs = WithdrawBuilder::build(depth);
    if (cs.n_constraints() != L.n_constraints) return OG_E_INVALID;
    csr_bound = 4 + 4ull * (cs.n_constraints() + 1) + 36ull * cs.A.col.size() + 4 + 4ull * (cs.n_constraints() + 1) + 36ull * cs.B.col.size();
    const uint64_t need_pk = 8 + 20 + 64 + 64 + 128 + 64 + 128 + 64ull * nv * 2 + 128ull * nv + 64ull * n_priv + 64ull * m + csr_bound;
    const uint64_t need_vk = 8 + 4 + 64 + 128 + 128 + 128 + 64ull * (n_pub + 1);
    if (!pk_out || !vk_out) { *pk_len = need_pk; *vk_len = need_vk; return OG_OK; }
    if (*pk_len < need_pk || *vk_len < need_vk) return OG_E_INVALID;

    Fr tau, alpha, beta, gamma, delta;
    if (!host_load(tau, toxic160) || !host_load(alpha, toxic160 + 32) || !host_load(beta, toxic160 + 64) ||
        !host_load(gamma, toxic160 + 96) || !host_load(delta, toxic160 + 128)) return OG_E_ENCODING;
    if (gamma.is_zero() || delta.is_zero()) return OG_E_INVALID;

    std::vector<Fr> Lg, Lc;
    if (!lagrange_at(tau, log_m, Lg)) return OG_E_INVALID;
    Fr g = host_root_of_unity(log_m + 1);
    if (!lagrange_at(tau * g.inv(), log_m, Lc)) return OG_E_INVALID;

    std::vector<Fr> u(nv, Fr::zero()), v(nv, Fr::zero()), w(nv, Fr::zero());
    for (uint32_t j = 0; j < cs.n_constraints(); j++) {
        for (uint32_t k = cs.A.row_ptr[j]; k < cs.A.row_ptr[j + 1]; k++) u[cs.A.col[k]] = u[cs.A.col[k]] + cs.A.val[k] * Lg[j];
        for (uint32_t k = cs.B.row_ptr[j]; k < cs.B.row_ptr[j + 1]; k++) v[cs.B.col[k]] = v[cs.B.col[k]] + cs.B.val[k] * Lg[j];
        for (uint32_t k = cs.C.row_ptr[j]; k < cs.C.row_ptr[j + 1]; k++) w[cs.C.col[k]] = w[cs.C.col[k]] + cs.C.val[k] * Lg[j];
    }
    for (uint32_t i = 0; i <= n_pub; i++) u[i] = u[i] + Lg[cs.n_constraints() + i];
    Fr dinv = delta.inv(), ginv = gamma.inv();
    Fr zt = host_pow_u64(tau, m) - Fr::one();
    Fr hfac = zt * (Fr::from_u32(2).neg() * delta).inv();

    // scalar lists -> canonical bytes
    // G1: [alpha, beta, delta, a (nv), b (nv), l (n_priv), ic (n_pub+1), h (m)]   G2: [beta, delta, gamma, b (nv)]
    const uint64_t n1 = 3 + 2ull * nv + n_priv + (n_pub + 1) + m, n2 = 3 + (uint64_t)nv;
    std::vector<uint8_t> s1(32 * n1), s2(32 * n2);
    uint64_t o = 0;
    auto put1 = [&](const Fr& x) { host_store(s1.data() + 32 * o, x); o++; };
    put1(alpha); put1(beta); put1(delta);
    for (uint32_t i = 0; i < nv; i++) put1(u[i]);
    for (uint32_t i = 0; i < nv; i++) put1(v[i]);
    for (uint32_t i = n_pub + 1; i < nv; i++) put1((beta * u[i] + alpha * v[i] + w[i]) * dinv);
    for (uint32_t i = 0; i <= n_pub; i++) put1((beta * u[i] + alpha * v[i] + w[i]) * ginv);
    for (uint32_t j = 0; j < m; j++) put1(Lc[j] * hfac);
    host_store(s2.data(), beta); host_store(s2.data() + 32, delta); host_store(s2.data() + 64, gamma);
    for (uint32_t i = 0; i < nv; i++) host_store(s2.data() + 32 * (3 + (uint64_t)i), v[i]);

    OG_TRY(clear_flag(ctx));
    OG_SLOT(ctx, d_s, uint8_t, S_SETUP_A, 32 * (n1 > n2 ? n1 : n2));
    OG_SLOT(ctx, d_pts, uint8_t, S_SETUP_B, sizeof(G2Affine) * (n1 > n2 ? n1 : n2));
    OG_SLOT(ctx, d_bytes, uint8_t, S_SETUP_C, 128 * (n1 > n2 ? n1 : n2));
    std::vector<uint8_t> p1, p2;
    OG_TRY(generator_mul<Fq>(ctx, s1, n1, d_s, d_pts, d_bytes, p1));
    OG_TRY(generator_mul<Fq2>(ctx, s2, n2, d_s, d_pts, d_bytes, p2));
    OG_TRY(check_flag(ctx));

    const uint8_t* alpha1 = p1.data(); const uint8_t* beta1 = p1.data() + 64; const uint8_t* delta1 = p1.data() + 128;
    const uint8_t* qa = p1.data() + 64 * 3; const uint8_t* qb1 = qa + 64ull * nv; const uint8_t* ql = qb1 + 64ull * nv;
    const uint8_t* ic = ql + 64ull * n_priv; const uint8_t* qh = ic + 64ull * (n_pub + 1);
    const uint8_t* beta2 = p2.data(); const uint8_t* delta2 = p2.data() + 128; const uint8_t* gamma2 = p2.data() + 256;
    const uint8_t* qb2 = p2.data() + 384;

    std::vector<uint8_t> pk;
    pk.reserve(need_pk);
    put_bytes(pk, reinterpret_cast<const uint8_t*>("OGPK"), 4); put_u32(pk, 1);
    put_u32(pk, depth); put_u32(pk, cs.n_constraints()); put_u32(pk, nv); put_u32(pk, n_pub); put_u32(pk, log_m);
    put_bytes(pk, alpha1, 64); put_bytes(pk, beta1, 64); put_bytes(pk, beta2, 128); put_bytes(pk, delta1, 64); put_bytes(pk, delta2, 128);
    put_bytes(pk, qa, 64ull * nv); put_bytes(pk, qb1, 64ull * nv); put_bytes(pk, qb2, 128ull * nv);
    put_bytes(pk, ql, 64ull * n_priv); put_bytes(pk, qh, 64ull * m);
    put_csr(pk, cs.A); put_csr(pk, cs.B);
    std::vector<uint8_t> vk;
    put_bytes(vk, reinterpret_cast<const uint8_t*>("OGVK"), 4); put_u32(vk, 1); put_u32(vk, n_pub);
    put_bytes(vk, alpha1, 64); put_bytes(vk, beta2, 128); put_bytes(vk, gamma2, 128); put_bytes(vk, delta2, 128);
    put_bytes(vk, ic, 64ull * (n_pub + 1));
    if (pk.size() > *pk_len || vk.size() > *vk_len) return OG_E_INVALID;
    memcpy(pk_out, pk.data(), pk.size()); *pk_len = pk.size();
    memcpy(vk_out, vk.data(), vk.size()); *vk_len = vk.size();
    return OG_OK;
}

}  // namespace og
