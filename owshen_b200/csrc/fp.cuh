// owshen_b200/csrc/fp.cuh -- 256-bit prime-field arithmetic for sm_100a, 8 x 32-bit limbs in registers.
//
// Montgomery form with R = 2^256.  The multiplier is the even/odd split CIOS: the running sum is
// kept in two staggered 8-limb arrays so every 32x32->64 partial product lands in a (lo, hi) pair
// of ONE array and each row is a single carry chain of mad.lo.cc / madc.hi.cc pairs, which ptxas
// fuses into IMAD.WIDE.U32(.X).  No tensor cores: this is modular big-integer work (DESIGN.md 5.1).
//
// Field definition: Fr follows /root/reference/src/blockchain/tx/owshen_airdrop/babyjubjub/mod.rs:7-11
// (modulus, little-endian canonical bytes); Fq is the public alt_bn128 base field.
//
// The same source compiles for the host (carry flag emulated in `CC`) so that tests/ can run the
// exact limb algorithm without a GPU; the product never executes the host path for proving.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define OG_HD __host__ __device__ __forceinline__
#else
#define OG_HD inline
#endif

namespace og {

struct CC { uint32_t c = 0; };  // host-side carry/borrow flag; the device uses the PTX CC register

#if defined(__CUDA_ARCH__)
#define OG_ASM asm volatile
OG_HD uint32_t add_cc(uint32_t a, uint32_t b, CC&) { uint32_t r; OG_ASM("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
OG_HD uint32_t addc_cc(uint32_t a, uint32_t b, CC&) { uint32_t r; OG_ASM("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
OG_HD uint32_t addc(uint32_t a, uint32_t b, CC&) { uint32_t r; OG_ASM("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
OG_HD uint32_t sub_cc(uint32_t a, uint32_t b, CC&) { uint32_t r; OG_ASM("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
OG_HD uint32_t subc_cc(uint32_t a, uint32_t b, CC&) { uint32_t r; OG_ASM("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
OG_HD uint32_t subc(uint32_t a, uint32_t b, CC&) { uint32_t r; OG_ASM("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
OG_HD uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c, CC&) { uint32_t r; OG_ASM("mad.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
OG_HD uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c, CC&) { uint32_t r; OG_ASM("madc.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
OG_HD uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c, CC&) { uint32_t r; OG_ASM("madc.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
OG_HD uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c, CC&) { uint32_t r; OG_ASM("madc.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
OG_HD uint32_t mul_lo(uint32_t a, uint32_t b) { return a * b; }
OG_HD uint32_t mul_hi(uint32_t a, uint32_t b) { return __umulhi(a, b); }
#else
OG_HD uint32_t add_cc(uint32_t a, uint32_t b, CC& cc) { uint64_t t = (uint64_t)a + b; cc.c = (uint32_t)(t >> 32); return (uint32_t)t; }
OG_HD uint32_t addc_cc(uint32_t a, uint32_t b, CC& cc) { uint64_t t = (uint64_t)a + b + cc.c; cc.c = (uint32_t)(t >> 32); return (uint32_t)t; }
OG_HD uint32_t addc(uint32_t a, uint32_t b, CC& cc) { return a + b + cc.c; }
OG_HD uint32_t sub_cc(uint32_t a, uint32_t b, CC& cc) { uint64_t t = (uint64_t)a - b; cc.c = (uint32_t)(t >> 63); return (uint32_t)t; }
OG_HD uint32_t subc_cc(uint32_t a, uint32_t b, CC& cc) { uint64_t t = (uint64_t)a - b - cc.c; cc.c = (uint32_t)(t >> 63); return (uint32_t)t; }
OG_HD uint32_t subc(uint32_t a, uint32_t b, CC& cc) { return a - b - cc.c; }
OG_HD uint32_t mul_lo(uint32_t a, uint32_t b) { return a * b; }
OG_HD uint32_t mul_hi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
OG_HD uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c, CC& cc) { uint64_t t = (uint64_t)mul_lo(a, b) + c; cc.c = (uint32_t)(t >> 32); return (uint32_t)t; }
OG_HD uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c, CC& cc) { uint64_t t = (uint64_t)mul_lo(a, b) + c + cc.c; cc.c = (uint32_t)(t >> 32); return (uint32_t)t; }
OG_HD uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c, CC& cc) { uint64_t t = (uint64_t)mul_hi(a, b) + c + cc.c; cc.c = (uint32_t)(t >> 32); return (uint32_t)t; }
OG_HD uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c, CC& cc) { return mul_hi(a, b) + c + cc.c; }
#endif

// ---- field parameters ---------------------------------------------------------------------------
// mod(i)/r2(i)/one(i) are constexpr functions so that fully unrolled loops fold them to immediates.
struct FqParams {  // alt_bn128 base field p
    static constexpr uint32_t INV = 0xe4866389u;  // -p^-1 mod 2^32
    OG_HD static constexpr uint32_t mod(int i) {
        constexpr uint32_t m[8] = {0xd87cfd47u, 0x3c208c16u, 0x6871ca8du, 0x97816a91u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
        return m[i];
    }
    OG_HD static constexpr uint32_t r2(int i) {   // 2^512 mod p
        constexpr uint32_t m[8] = {0x538afa89u, 0xf32cfc5bu, 0xd44501fbu, 0xb5e71911u, 0x0a417ff6u, 0x47ab1effu, 0xcab8351fu, 0x06d89f71u};
        return m[i];
    }
    OG_HD static constexpr uint32_t one(int i) {  // 2^256 mod p
        constexpr uint32_t m[8] = {0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u, 0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
        return m[i];
    }
};
struct FrParams {  // BN254 scalar field r  (reference: babyjubjub/mod.rs:8)
    static constexpr uint32_t INV = 0xefffffffu;
    OG_HD static constexpr uint32_t mod(int i) {
        constexpr uint32_t m[8] = {0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u};
        return m[i];
    }
    OG_HD static constexpr uint32_t r2(int i) {
        constexpr uint32_t m[8] = {0xae216da7u, 0x1bb8e645u, 0xe35c59e3u, 0x53fe3ab1u, 0x53bb8085u, 0x8c49833du, 0x7f4e44a5u, 0x0216d0b1u};
        return m[i];
    }
    OG_HD static constexpr uint32_t one(int i) {
        constexpr uint32_t m[8] = {0x4ffffffbu, 0xac96341cu, 0x9f60cd29u, 0x36fc7695u, 0x7879462eu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u};
        return m[i];
    }
};

// ---- raw limb routines ----------------------------------------------------------------------------
// r = (r >= p) ? r - p : r     (r < 2p)
template <class P>
OG_HD void final_sub(uint32_t* r) {
    uint32_t t[8];
    CC cc;
    t[0] = sub_cc(r[0], P::mod(0), cc);
#pragma unroll
    for (int j = 1; j < 8; j++) t[j] = subc_cc(r[j], P::mod(j), cc);
    uint32_t borrow = subc(0u, 0u, cc);  // 0xffffffff when r < p
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = borrow ? r[j] : t[j];
}

// One interleaved Montgomery row.  E is the array aligned at limb 0, O the one aligned at limb 1;
// on entry (when !first) O is the previous row's E: its limb 0 is dead (zero by construction), O[1] sits
// at limb 0 (the "orphan") and O[2..7] at limbs 1..6.
//  * every a*b chain starts with mad.lo.cc so that ptxas fuses the (lo, hi) pairs into IMAD.WIDE.U32(.X);
//  * the orphan is folded while forming s = E[0] + orphan: its carry enters the q*p chain on O (limb 1),
//    and because s + lo(q*p0) == 0 (mod 2^32) the low product is never computed: its carry is (s != 0),
//    injected with add.cc(s, 0xffffffff) into the q*p chain on E, which starts at limb 1.
// No limb ripples through a whole array, so successive rows overlap and the dependency chain per product
// is short (this kernel family is latency-bound at 4 warps/scheduler; see profiles/).
template <class P>
OG_HD void mont_row(uint32_t* E, uint32_t* O, const uint32_t* a, uint32_t bi, bool first) {
    CC cc;
    uint32_t orphan = 0;
    if (first) {
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
            E[j] = mul_lo(a[j], bi);
            E[j + 1] = mul_hi(a[j], bi);
            O[j] = mul_lo(a[j + 1], bi);
            O[j + 1] = mul_hi(a[j + 1], bi);
        }
    } else {
        orphan = O[1];
        // O' = (O >> 2 limbs) + a_odd * bi
        O[0] = mad_lo_cc(a[1], bi, O[2], cc);
        O[1] = madc_hi_cc(a[1], bi, O[3], cc);
#pragma unroll
        for (int j = 2; j < 6; j += 2) {
            O[j] = madc_lo_cc(a[j + 1], bi, O[j + 2], cc);
            O[j + 1] = madc_hi_cc(a[j + 1], bi, O[j + 3], cc);
        }
        O[6] = madc_lo_cc(a[7], bi, 0u, cc);
        O[7] = madc_hi(a[7], bi, 0u, cc);
        // E += a_even * bi ; carry lands on limb 8 = O[7]
        E[0] = mad_lo_cc(a[0], bi, E[0], cc);
        E[1] = madc_hi_cc(a[0], bi, E[1], cc);
#pragma unroll
        for (int j = 2; j < 8; j += 2) {
            E[j] = madc_lo_cc(a[j], bi, E[j], cc);
            E[j + 1] = madc_hi_cc(a[j], bi, E[j + 1], cc);
        }
        O[7] = addc(O[7], 0u, cc);
    }
    uint32_t s = add_cc(E[0], orphan, cc);            // carry -> limb 1
    uint32_t q = mul_lo(s, P::INV);
    O[0] = madc_lo_cc(P::mod(1), q, O[0], cc);
    O[1] = madc_hi_cc(P::mod(1), q, O[1], cc);
#pragma unroll
    for (int j = 2; j < 6; j += 2) {
        O[j] = madc_lo_cc(P::mod(j + 1), q, O[j], cc);
        O[j + 1] = madc_hi_cc(P::mod(j + 1), q, O[j + 1], cc);
    }
    O[6] = madc_lo_cc(P::mod(7), q, O[6], cc);
    O[7] = madc_hi(P::mod(7), q, O[7], cc);           // T < 2^288: no carry out of limb 8
    (void)add_cc(s, 0xffffffffu, cc);                 // carry = (s != 0) = carry of s + lo(q*p0)
    E[1] = madc_hi_cc(P::mod(0), q, E[1], cc);
#pragma unroll
    for (int j = 2; j < 8; j += 2) {
        E[j] = madc_lo_cc(P::mod(j), q, E[j], cc);
        E[j + 1] = madc_hi_cc(P::mod(j), q, E[j + 1], cc);
    }
    O[7] = addc(O[7], 0u, cc);
    E[0] = 0;                                         // dead from here on
}

// 2p as limbs (p < 2^254, so 2p < 2^255)
template <class P>
OG_HD constexpr uint32_t mod2(int i) { return (P::mod(i) << 1) | (i ? P::mod(i - 1) >> 31 : 0u); }

// r = (r >= 2p) ? r - 2p : r     (r < 4p): the one conditional subtraction per round that keeps a chain of lazy products
// (operands and results in [0, 2p), see mont_mul_lazy) from growing
template <class P>
OG_HD void cond_sub_2p(uint32_t* r) {
    uint32_t t[8];
    CC cc;
    t[0] = sub_cc(r[0], mod2<P>(0), cc);
#pragma unroll
    for (int j = 1; j < 8; j++) t[j] = subc_cc(r[j], mod2<P>(j), cc);
    uint32_t borrow = subc(0u, 0u, cc);
#pragma unroll
    for (int j = 0; j < 8; j++) r[j] = borrow ? r[j] : t[j];
}

// r = (a * b + m * p) / 2^256 with m < 2^256, i.e. r == a * b * 2^-256 (mod p) and r < a * b / 2^256 + p.  For a, b < 2p
// that is r < (4p / 2^256 + 1) p < 1.76 p (p < 0.19 * 2^256): products of values in [0, 2p) stay in [0, 2p) without any final
// subtraction, and no running sum leaves 2^288 (a + p < 2^256).  r may alias a or b.
template <class P>
OG_HD void mont_mul_lazy(uint32_t* r, const uint32_t* a, const uint32_t* b) {
    uint32_t E[8], O[8];
    mont_row<P>(E, O, a, b[0], true);
    mont_row<P>(O, E, a, b[1], false);
    mont_row<P>(E, O, a, b[2], false);
    mont_row<P>(O, E, a, b[3], false);
    mont_row<P>(E, O, a, b[4], false);
    mont_row<P>(O, E, a, b[5], false);
    mont_row<P>(E, O, a, b[6], false);
    mont_row<P>(O, E, a, b[7], false);
    CC cc;
    r[0] = add_cc(E[0], O[1], cc);
#pragma unroll
    for (int j = 1; j < 7; j++) r[j] = addc_cc(E[j], O[j + 1], cc);
    r[7] = addc(E[7], 0u, cc);
}

// r = a * b * 2^-256 mod p, fully reduced   (a, b < p; r may alias a or b)
template <class P>
OG_HD void mont_mul(uint32_t* r, const uint32_t* a, const uint32_t* b) {
    mont_mul_lazy<P>(r, a, b);
    final_sub<P>(r);
}

// ---- wide (512-bit) products and their Montgomery reduction ----------------------------------------------
// Used where the interleaved multiplier wastes work: squarings (36 instead of 64 partial products) and
// Fq2 products with lazy reduction (3 wide products, 2 reductions instead of 3 full multiplications).
// T = sum T[k] 2^(32k), 16 limbs.  All multiply chains start with mad.lo.cc / mul so ptxas fuses them.

// T = a * b  (16 chains of 4 wide multiply-adds; even- and odd-aligned pairs kept in separate arrays)
OG_HD void mul_wide(uint32_t* T, const uint32_t* a, const uint32_t* b) {
    uint32_t E[16], O[16];          // E[k] at limb k (pairs start at even limbs); O[k] at limb k+1 (pairs start at odd limbs)
#pragma unroll
    for (int k = 0; k < 16; k++) { E[k] = 0; O[k] = 0; }
    CC cc;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        // products a_j * b_i land at limb i + j: same parity as i for even j, opposite for odd j
        uint32_t* X = (i & 1) ? O : E;      // pairs starting at limb i      (j even)
        uint32_t* Y = (i & 1) ? E : O;      // pairs starting at limb i + 1  (j odd)
        const int x0 = (i & 1) ? i - 1 : i; // index in X of limb i
        const int y0 = (i & 1) ? i + 1 : i; // index in Y of limb i + 1
        X[x0] = mad_lo_cc(a[0], b[i], X[x0], cc);
        X[x0 + 1] = madc_hi_cc(a[0], b[i], X[x0 + 1], cc);
#pragma unroll
        for (int j = 2; j < 8; j += 2) {
            X[x0 + j] = madc_lo_cc(a[j], b[i], X[x0 + j], cc);
            X[x0 + j + 1] = madc_hi_cc(a[j], b[i], X[x0 + j + 1], cc);
        }
        if (x0 + 8 < 16) X[x0 + 8] = addc(X[x0 + 8], 0u, cc);
        Y[y0] = mad_lo_cc(a[1], b[i], Y[y0], cc);
        Y[y0 + 1] = madc_hi_cc(a[1], b[i], Y[y0 + 1], cc);
#pragma unroll
        for (int j = 2; j < 8; j += 2) {
            Y[y0 + j] = madc_lo_cc(a[j + 1], b[i], Y[y0 + j], cc);
            Y[y0 + j + 1] = madc_hi_cc(a[j + 1], b[i], Y[y0 + j + 1], cc);
        }
        if (y0 + 8 < 16) Y[y0 + 8] = addc(Y[y0 + 8], 0u, cc);
    }
    T[0] = E[0];
    T[1] = add_cc(E[1], O[0], cc);
#pragma unroll
    for (int k = 2; k < 15; k++) T[k] = addc_cc(E[k], O[k - 1], cc);
    T[15] = addc(E[15], O[14], cc);
}

// T = a^2: the 28 products a_i a_j (i < j) once, doubled, plus the 8 squares on the diagonal
OG_HD void sqr_wide(uint32_t* T, const uint32_t* a) {
    uint32_t E[16], O[16];
#pragma unroll
    for (int k = 0; k < 16; k++) { E[k] = 0; O[k] = 0; }
    CC cc;
#pragma unroll
    for (int i = 0; i < 7; i++) {
        // j = i+1, i+3, ... -> limb i+j odd-offset from 2i ; j = i+2, i+4, ... -> even offset
        // limb(i, j) = i + j.  Pairs starting at limb 2i+1 (j = i+1, step 2) and at limb 2i+2 (j = i+2, step 2).
        {   // j = i + 1, i + 3, ...   first limb L = 2i + 1 (odd)  -> array O, index L - 1
            const int L = 2 * i + 1;
            bool head = true;
#pragma unroll
            for (int j = i + 1; j < 8; j += 2) {
                const int k = L - 1 + (j - i - 1);
                if (head) { O[k] = mad_lo_cc(a[i], a[j], O[k], cc); head = false; }
                else O[k] = madc_lo_cc(a[i], a[j], O[k], cc);
                O[k + 1] = madc_hi_cc(a[i], a[j], O[k + 1], cc);
            }
            const int kend = L - 1 + 2 * ((8 - i) / 2);      // first index after the chain
            if (kend < 16) O[kend] = addc(O[kend], 0u, cc);
        }
        if (i + 2 < 8) {   // j = i + 2, i + 4, ...   first limb L = 2i + 2 (even) -> array E, index L
            const int L = 2 * i + 2;
            bool head = true;
#pragma unroll
            for (int j = i + 2; j < 8; j += 2) {
                const int k = L + (j - i - 2);
                if (head) { E[k] = mad_lo_cc(a[i], a[j], E[k], cc); head = false; }
                else E[k] = madc_lo_cc(a[i], a[j], E[k], cc);
                E[k + 1] = madc_hi_cc(a[i], a[j], E[k + 1], cc);
            }
            const int kend = L + 2 * ((7 - i) / 2);
            if (kend < 16) E[kend] = addc(E[kend], 0u, cc);
        }
    }
    // S = E + (O << 32); T = 2 S
    uint32_t S[16];
    S[0] = E[0];
    S[1] = add_cc(E[1], O[0], cc);
#pragma unroll
    for (int k = 2; k < 15; k++) S[k] = addc_cc(E[k], O[k - 1], cc);
    S[15] = addc(E[15], O[14], cc);
    T[0] = S[0] << 1;
#pragma unroll
    for (int k = 1; k < 16; k++) T[k] = (S[k] << 1) | (S[k - 1] >> 31);
    // diagonal: a_i^2 at limbs (2i, 2i+1): one chain over all 16 limbs
    T[0] = mad_lo_cc(a[0], a[0], T[0], cc);
    T[1] = madc_hi_cc(a[0], a[0], T[1], cc);
#pragma unroll
    for (int i = 1; i < 8; i++) {
        T[2 * i] = madc_lo_cc(a[i], a[i], T[2 * i], cc);
        T[2 * i + 1] = madc_hi_cc(a[i], a[i], T[2 * i + 1], cc);
    }
}

// One reduction-only row of the even/odd scheme (mont_row without the a*b part): E is the window base, O the
// array one limb up; on entry (when !first) O is the previous base (O[0] dead, O[1] the orphan, O[2..7] at
// window limbs 1..6).  t_in, the limb of T that enters the window this row, lands on window limb 8 = O[7];
// carries out of limb 8 wait in `ctop` for the next row.
template <class P>
OG_HD void mont_redc_row(uint32_t* E, uint32_t* O, bool first, uint32_t t_in, uint32_t& ctop) {
    CC cc;
    uint32_t orphan = 0;
    if (!first) {
        orphan = O[1];
#pragma unroll
        for (int j = 0; j < 6; j++) O[j] = O[j + 2];
        O[6] = 0;
    }
    O[7] = add_cc(t_in, ctop, cc);
    ctop = addc(0u, 0u, cc);
    uint32_t s = add_cc(E[0], orphan, cc);
    uint32_t q = mul_lo(s, P::INV);
    O[0] = madc_lo_cc(P::mod(1), q, O[0], cc);
    O[1] = madc_hi_cc(P::mod(1), q, O[1], cc);
#pragma unroll
    for (int j = 2; j < 8; j += 2) {
        O[j] = madc_lo_cc(P::mod(j + 1), q, O[j], cc);
        O[j + 1] = madc_hi_cc(P::mod(j + 1), q, O[j + 1], cc);
    }
    ctop = addc(ctop, 0u, cc);
    (void)add_cc(s, 0xffffffffu, cc);
    E[1] = madc_hi_cc(P::mod(0), q, E[1], cc);
#pragma unroll
    for (int j = 2; j < 8; j += 2) {
        E[j] = madc_lo_cc(P::mod(j), q, E[j], cc);
        E[j + 1] = madc_hi_cc(P::mod(j), q, E[j + 1], cc);
    }
    O[7] = addc_cc(O[7], 0u, cc);
    ctop = addc(ctop, 0u, cc);
    E[0] = 0;
}

// r = (T + m p) / 2^256 for T < 2^256 * p (any product of operands < 2p qualifies): r == T * 2^-256 (mod p), r < T / 2^256 + p
template <class P>
OG_HD void mont_reduce_wide_lazy(uint32_t* r, const uint32_t* T) {
    uint32_t E[8], O[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { E[k] = T[k]; O[k] = 0; }
    uint32_t ctop = 0;
    mont_redc_row<P>(E, O, true, T[8], ctop);
    mont_redc_row<P>(O, E, false, T[9], ctop);
    mont_redc_row<P>(E, O, false, T[10], ctop);
    mont_redc_row<P>(O, E, false, T[11], ctop);
    mont_redc_row<P>(E, O, false, T[12], ctop);
    mont_redc_row<P>(O, E, false, T[13], ctop);
    mont_redc_row<P>(E, O, false, T[14], ctop);
    mont_redc_row<P>(O, E, false, T[15], ctop);
    // E is aligned at limb 0 of the result, O[1..7] at limbs 0..6 (O[0] dead); ctop is zero for T < 2^256 p
    CC cc;
    r[0] = add_cc(E[0], O[1], cc);
#pragma unroll
    for (int j = 1; j < 7; j++) r[j] = addc_cc(E[j], O[j + 1], cc);
    r[7] = addc(E[7], 0u, cc);
}

// r = T * 2^-256 mod p, fully reduced
template <class P>
OG_HD void mont_reduce_wide(uint32_t* r, const uint32_t* T) {
    mont_reduce_wide_lazy<P>(r, T);
    final_sub<P>(r);
}

// ---- the field element type -----------------------------------------------------------------------
template <class P>
struct alignas(32) Fp {
    uint32_t l[8];

    OG_HD static Fp zero() { Fp r; for (int i = 0; i < 8; i++) r.l[i] = 0; return r; }
    OG_HD static Fp one() { Fp r;
#pragma unroll
        for (int i = 0; i < 8; i++) r.l[i] = P::one(i);
        return r; }
    OG_HD bool is_zero() const { uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) o |= l[i];
        return o == 0; }
    OG_HD bool operator==(const Fp& b) const { uint32_t o = 0;
#pragma unroll
        for (int i = 0; i < 8; i++) o |= l[i] ^ b.l[i];
        return o == 0; }
    OG_HD bool operator!=(const Fp& b) const { return !(*this == b); }

    OG_HD friend Fp operator*(const Fp& a, const Fp& b) { Fp r; mont_mul<P>(r.l, a.l, b.l); return r; }
    // the wide squarer: with the bucket accumulators in shared memory it beats squaring through the interleaved multiplier by
    // 0.8 % (231.5 vs 233.3 ms per 1024 proofs, profiles/r2_small_ab.md)
    OG_HD Fp sqr() const { Fp r; uint32_t T[16]; sqr_wide(T, l); mont_reduce_wide<P>(r.l, T); return r; }   // 36 + 64 products

    // lazy forms for long dependent chains (MiMC): values in [0, 2p), no final subtraction (bounds at mont_mul_lazy)
    OG_HD static Fp mul_lazy(const Fp& a, const Fp& b) { Fp r; mont_mul_lazy<P>(r.l, a.l, b.l); return r; }
    OG_HD Fp sqr_lazy() const { Fp r; uint32_t T[16]; sqr_wide(T, l); mont_reduce_wide_lazy<P>(r.l, T); return r; }
    // a + b as integers (the caller knows the sum is below 2^256)
    OG_HD static Fp add_raw(const Fp& a, const Fp& b) {
        Fp r; CC cc;
        r.l[0] = add_cc(a.l[0], b.l[0], cc);
#pragma unroll
        for (int j = 1; j < 7; j++) r.l[j] = addc_cc(a.l[j], b.l[j], cc);
        r.l[7] = addc(a.l[7], b.l[7], cc);
        return r;
    }
    // value < 4p -> [0, 2p)  /  value < 2p -> [0, p)
    OG_HD Fp reduce_4p_to_2p() const { Fp r = *this; cond_sub_2p<P>(r.l); return r; }
    OG_HD Fp reduce_2p_to_p() const { Fp r = *this; final_sub<P>(r.l); return r; }

    OG_HD friend Fp operator+(const Fp& a, const Fp& b) {
        Fp r; CC cc;
        r.l[0] = add_cc(a.l[0], b.l[0], cc);
#pragma unroll
        for (int j = 1; j < 7; j++) r.l[j] = addc_cc(a.l[j], b.l[j], cc);
        r.l[7] = addc(a.l[7], b.l[7], cc);   // p < 2^254: no carry out
        final_sub<P>(r.l);
        return r;
    }
    OG_HD friend Fp operator-(const Fp& a, const Fp& b) {
        Fp r; CC cc;
        r.l[0] = sub_cc(a.l[0], b.l[0], cc);
#pragma unroll
        for (int j = 1; j < 8; j++) r.l[j] = subc_cc(a.l[j], b.l[j], cc);
        uint32_t borrow = subc(0u, 0u, cc);
        r.l[0] = add_cc(r.l[0], P::mod(0) & borrow, cc);
#pragma unroll
        for (int j = 1; j < 7; j++) r.l[j] = addc_cc(r.l[j], P::mod(j) & borrow, cc);
        r.l[7] = addc(r.l[7], P::mod(7) & borrow, cc);
        return r;
    }
    OG_HD Fp neg() const { return zero() - *this; }
    OG_HD Fp dbl() const { return *this + *this; }

    // canonical integer (little-endian limbs) <-> Montgomery form
    OG_HD static Fp from_canonical(const uint32_t* c) {
        Fp t, r2;
#pragma unroll
        for (int i = 0; i < 8; i++) { t.l[i] = c[i]; r2.l[i] = P::r2(i); }
        return t * r2;
    }
    OG_HD void to_canonical(uint32_t* c) const {
        Fp o = zero(); o.l[0] = 1;
        Fp t = *this * o;
#pragma unroll
        for (int i = 0; i < 8; i++) c[i] = t.l[i];
    }
    OG_HD static bool canonical_lt_mod(const uint32_t* c) {
        for (int i = 7; i >= 0; i--) {
            if (c[i] < P::mod(i)) return true;
            if (c[i] > P::mod(i)) return false;
        }
        return false;
    }
    OG_HD static Fp from_u32(uint32_t v) { uint32_t c[8] = {v, 0, 0, 0, 0, 0, 0, 0}; return from_canonical(c); }

    // x^e, e given as canonical 8-limb integer (not constant time; used for inversion / roots only)
    OG_HD Fp pow(const uint32_t* e) const {
        Fp acc = one();
        for (int i = 255; i >= 0; i--) {
            acc = acc.sqr();
            if ((e[i >> 5] >> (i & 31)) & 1) acc = acc * *this;
        }
        return acc;
    }
    OG_HD Fp inv() const {  // Fermat: x^(p-2); inv(0) = 0
        uint32_t e[8];
#pragma unroll
        for (int i = 0; i < 8; i++) e[i] = P::mod(i);
        e[0] -= 2;          // p is odd and p mod 2^32 >= 2 for both fields
        return pow(e);
    }
};

typedef Fp<FqParams> Fq;
typedef Fp<FrParams> Fr;

// ---- Fq2 = Fq[i]/(i^2+1) ----------------------------------------------------------------------------
struct Fq2 {
    Fq c0, c1;
    OG_HD static Fq2 zero() { return Fq2{Fq::zero(), Fq::zero()}; }
    OG_HD static Fq2 one() { return Fq2{Fq::one(), Fq::zero()}; }
    OG_HD bool is_zero() const { return c0.is_zero() && c1.is_zero(); }
    OG_HD bool operator==(const Fq2& b) const { return c0 == b.c0 && c1 == b.c1; }
    OG_HD bool operator!=(const Fq2& b) const { return !(*this == b); }
    OG_HD friend Fq2 operator+(const Fq2& a, const Fq2& b) { return Fq2{a.c0 + b.c0, a.c1 + b.c1}; }
    OG_HD friend Fq2 operator-(const Fq2& a, const Fq2& b) { return Fq2{a.c0 - b.c0, a.c1 - b.c1}; }
    // Karatsuba with lazy reduction: 3 wide (512-bit) products and 2 Montgomery reductions instead of 3 full
    // multiplications (320 instead of 384 32x32->64 products).  c1 = (a0+a1)(b0+b1) - a0b0 - a1b1 >= 0 exactly;
    // c0 = a0b0 - a1b1 is made non-negative by adding p * 2^256 (= 0 mod p) before the reduction.
    OG_HD static Fq2 mul_inl(const Fq2& a, const Fq2& b) {
        uint32_t T0[16], T1[16], T2[16], sa[8], sb[8];
        CC cc;
        mul_wide(T0, a.c0.l, b.c0.l);
        mul_wide(T1, a.c1.l, b.c1.l);
        sa[0] = add_cc(a.c0.l[0], a.c1.l[0], cc);
        for (int j = 1; j < 7; j++) sa[j] = addc_cc(a.c0.l[j], a.c1.l[j], cc);
        sa[7] = addc(a.c0.l[7], a.c1.l[7], cc);                    // < 2p < 2^255: no carry out
        sb[0] = add_cc(b.c0.l[0], b.c1.l[0], cc);
        for (int j = 1; j < 7; j++) sb[j] = addc_cc(b.c0.l[j], b.c1.l[j], cc);
        sb[7] = addc(b.c0.l[7], b.c1.l[7], cc);
        mul_wide(T2, sa, sb);
        // T2 -= T0 ; T2 -= T1
        T2[0] = sub_cc(T2[0], T0[0], cc);
        for (int j = 1; j < 15; j++) T2[j] = subc_cc(T2[j], T0[j], cc);
        T2[15] = subc(T2[15], T0[15], cc);
        T2[0] = sub_cc(T2[0], T1[0], cc);
        for (int j = 1; j < 15; j++) T2[j] = subc_cc(T2[j], T1[j], cc);
        T2[15] = subc(T2[15], T1[15], cc);
        // T0 = T0 - T1 + p * 2^256   (mod 2^512 arithmetic; the true value lies in (0, p^2 + p 2^256))
        T0[0] = sub_cc(T0[0], T1[0], cc);
        for (int j = 1; j < 15; j++) T0[j] = subc_cc(T0[j], T1[j], cc);
        T0[15] = subc(T0[15], T1[15], cc);
        T0[8] = add_cc(T0[8], FqParams::mod(0), cc);
        for (int j = 1; j < 7; j++) T0[8 + j] = addc_cc(T0[8 + j], FqParams::mod(j), cc);
        T0[15] = addc(T0[15], FqParams::mod(7), cc);
        Fq2 r;
        mont_reduce_wide<FqParams>(r.c0.l, T0);                   // < 2.25 p before its final_sub
        final_sub<FqParams>(r.c0.l);
        mont_reduce_wide<FqParams>(r.c1.l, T2);
        return r;
    }
    OG_HD static Fq2 sqr_inl(const Fq2& a) {                    // 2 Fq muls
        Fq m = a.c0 * a.c1;
        return Fq2{(a.c0 + a.c1) * (a.c0 - a.c1), m + m};
    }
    OG_HD friend Fq2 operator*(const Fq2& a, const Fq2& b);
    OG_HD Fq2 sqr() const;
    OG_HD Fq2 neg() const { return Fq2{c0.neg(), c1.neg()}; }
    OG_HD Fq2 dbl() const { return Fq2{c0.dbl(), c1.dbl()}; }
    OG_HD Fq2 inv() const {
        Fq n = (c0.sqr() + c1.sqr()).inv();
        return Fq2{c0 * n, (c1 * n).neg()};
    }
    OG_HD Fq2 conj() const { return Fq2{c0, c1.neg()}; }
    OG_HD Fq2 mul_fq(const Fq& s) const { return Fq2{c0 * s, c1 * s}; }
};

// Fq2 products are inlined.  Kernels keep ptxas time sane by calling the out-of-line group operations of
// ec.cuh (xyzz_*_ni) everywhere except in the bucket-accumulation inner loop (a G2 group operation is
// ~10k instructions; inlining several of them into one kernel once cost 30 minutes of ptxas).
#if defined(__CUDA_ARCH__) && defined(OG_FP_MUL_CALL)
// Translation units whose kernels would inline dozens of Fq2 products per group operation keep ONE copy of
// the Fq2 multiplier / squarer (arguments and result travel in registers): the fully inlined G2 bucket kernel
// overflowed the instruction cache (ncu: 30 % of warp samples in "no_instructions", profiles/).
static __device__ __noinline__ Fq2 fq2_mul_call(Fq2 a, Fq2 b) { return Fq2::mul_inl(a, b); }
static __device__ __noinline__ Fq2 fq2_sqr_call(Fq2 a) { return Fq2::sqr_inl(a); }
OG_HD Fq2 operator*(const Fq2& a, const Fq2& b) { return fq2_mul_call(a, b); }
OG_HD Fq2 Fq2::sqr() const { return fq2_sqr_call(*this); }
#else
OG_HD Fq2 operator*(const Fq2& a, const Fq2& b) { return Fq2::mul_inl(a, b); }
OG_HD Fq2 Fq2::sqr() const { return Fq2::sqr_inl(*this); }
#endif

}  // namespace og
