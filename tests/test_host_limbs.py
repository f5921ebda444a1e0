"""The product's limb algorithms (fp.cuh even/odd Montgomery rows, ec.cuh XYZZ formulas) compiled for
the host with the PTX carry chain emulated, against the oracle.  This checks the algorithm the GPU
runs, without a GPU; the -m gpu tests check the real PTX path."""
import ctypes as C
import os
import random
import subprocess

import pytest

from oracle import bn254 as bn
from oracle import cport

R, P = bn.R, bn.P
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def h(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("harness") / "libhost_harness.so")
    src = os.path.join(ROOT, "tests", "harness", "host_harness.cpp")
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I" + os.path.join(ROOT, "owshen_b200", "csrc"),
                    "-o", so, src], check=True)
    return C.CDLL(so)


def _binop(h, name, a, b):
    out = C.create_string_buffer(len(a))
    getattr(h, name)(a, b, out, C.c_uint64(len(a) // 32))
    return out.raw


def test_field_limbs(h):
    rng = random.Random(1)
    for F, mod, pack in (("fq", P, cport.fqs), ("fr", R, cport.frs)):
        xs = [rng.randrange(mod) for _ in range(3000)] + [0, 1, mod - 1, mod - 1, 2**253, mod - 2, 2**32 - 1]
        ys = [rng.randrange(mod) for _ in range(3000)] + [mod - 1, mod - 1, mod - 1, 1, 2**253, mod - 2, 2**224]
        assert cport.unfr(_binop(h, f"ht_{F}_mul", pack(xs), pack(ys))) == [a * b % mod for a, b in zip(xs, ys)]
        assert cport.unfr(_binop(h, f"ht_{F}_add", pack(xs), pack(ys))) == [(a + b) % mod for a, b in zip(xs, ys)]
        assert cport.unfr(_binop(h, f"ht_{F}_sub", pack(xs), pack(ys))) == [(a - b) % mod for a, b in zip(xs, ys)]
        out = C.create_string_buffer(32 * 5)
        getattr(h, f"ht_{F}_inv")(pack(xs[:5]), out, C.c_uint64(5))
        assert cport.unfr(out.raw) == [pow(a, -1, mod) for a in xs[:5]]


def test_fq2(h):
    rng = random.Random(2)
    a = (rng.randrange(P), rng.randrange(P)); b = (rng.randrange(P), rng.randrange(P))
    o = C.create_string_buffer(64)
    h.ht_fq2_mul(cport.fqs(a), cport.fqs(b), o); assert tuple(cport.unfr(o.raw)) == bn.f2_mul(a, b)
    h.ht_fq2_sqr(cport.fqs(a), o); assert tuple(cport.unfr(o.raw)) == bn.f2_sqr(a)
    h.ht_fq2_inv(cport.fqs(a), o); assert tuple(cport.unfr(o.raw)) == bn.f2_inv(a)


def test_group_formulas_with_exceptional_cases(h):
    rng = random.Random(3)
    for k in [0, 1, 2, 3, R - 1, rng.randrange(R)]:
        o = C.create_string_buffer(64); h.ht_g1_mul(bn.g1_to_bytes(bn.G1_GEN), bn.fr_to_bytes(k), o)
        assert o.raw == bn.g1_to_bytes(bn.g1_mul(bn.G1_GEN, k))
        o = C.create_string_buffer(128); h.ht_g2_mul(bn.g2_to_bytes(bn.G2_GEN), bn.fr_to_bytes(k), o)
        assert o.raw == bn.g2_to_bytes(bn.g2_mul(bn.G2_GEN, k))
    pts = [bn.g1_mul(bn.G1_GEN, rng.randrange(R)) for _ in range(6)]
    pts = pts + [pts[0], None, bn.g1_neg(pts[1]), pts[2], pts[2]]       # P+P, infinity, P+(-P)
    exp = None
    for p in pts:
        exp = bn.g1_add(exp, p)
    for mode in (0, 1):
        o = C.create_string_buffer(64)
        h.ht_g1_sum(b"".join(map(bn.g1_to_bytes, pts)), C.c_uint64(len(pts)), mode, o)
        assert o.raw == bn.g1_to_bytes(exp)
    seq = [pts[0], pts[0], bn.g1_neg(bn.g1_mul(pts[0], 2))]
    o = C.create_string_buffer(64); h.ht_g1_sum(b"".join(map(bn.g1_to_bytes, seq)), C.c_uint64(3), 0, o)
    assert o.raw == bytes(64)
    pts2 = [bn.g2_mul(bn.G2_GEN, rng.randrange(R)) for _ in range(3)]
    pts2 = pts2 + [pts2[0], None, bn.g2_neg(pts2[1])]
    exp = None
    for p in pts2:
        exp = bn.g2_add(exp, p)
    for mode in (0, 1):
        o = C.create_string_buffer(128)
        h.ht_g2_sum(b"".join(map(bn.g2_to_bytes, pts2)), C.c_uint64(len(pts2)), mode, o)
        assert o.raw == bn.g2_to_bytes(exp)


def test_babyjubjub_verification_core_on_host(h):
    """bjj_core.cuh (the code the GPU kernel runs) against the oracle's restatement of the reference."""
    from oracle import babyjubjub as bjj
    from tests.test_babyjubjub import _cases, _pack
    rng = random.Random(5)
    pks, msgs, sigs, expect = _cases(rng, 16, 0)
    pkx, odd, m, s = _pack(pks + [(3, 0)], msgs + [1], sigs + [sigs[0]])
    out = C.create_string_buffer(len(odd))
    h.ht_bjj_verify(pkx, odd, m, s, len(odd), bn.fr_to_bytes(bjj.BASE[0]) + bn.fr_to_bytes(bjj.BASE[1]), out)
    assert list(out.raw) == [1 if e else 0 for e in expect] + [2]


def test_babyjubjub_signing_core_on_host(h):
    """bjj_sign_one (key derivation + signing, mod.rs:206-237) compiled for the host against the oracle's restatement,
    and its integer step s = (r + h a) mod ORDER on crafted operands -- including results in [r, ORDER), the case the
    reference answers with Err("Invalid repr") and which random signatures reach with probability ~3 * 10^-39."""
    from oracle import babyjubjub as bjj
    rng = random.Random(17)
    n = 6
    sks = [rng.randrange(R) for _ in range(n - 2)] + [0, 1]
    rnds = [rng.randrange(R) for _ in range(n)]
    msgs = [rng.randrange(R) for _ in range(n - 1)] + [0]
    fb = bn.fr_to_bytes
    pkx, odd = C.create_string_buffer(32 * n), C.create_string_buffer(n)
    sigs, st = C.create_string_buffer(96 * n), C.create_string_buffer(n)
    h.ht_bjj_sign(b"".join(map(fb, sks)), b"".join(map(fb, rnds)), b"".join(map(fb, msgs)), n, fb(bjj.BASE[0]) + fb(bjj.BASE[1]), pkx, odd, sigs, st)
    for i in range(n):
        pk = bjj.to_pub(sks[i])
        (rx, ry), s_ = bjj.sign(sks[i], rnds[i], msgs[i])
        assert st.raw[i] == 1
        assert pkx.raw[32 * i:32 * i + 32] == fb(pk[0]) and odd.raw[i] == pk[1]
        assert sigs.raw[96 * i:96 * i + 96] == fb(rx) + fb(ry) + fb(s_)
        assert bjj.verify(pk, msgs[i], ((rx, ry), s_))
    ks = [rng.randrange(R) for _ in range(20)] + [0, 1, 15, 16, R - 1, 1 << 252]
    assert h.ht_bjj_table_mul_matches(b"".join(map(fb, ks)), len(ks), fb(bjj.BASE[0]) + fb(bjj.BASE[1])) == 1     # window-table k * BASE
    O = bjj.ORDER
    cases = [(rng.randrange(R), rng.randrange(R), rng.randrange(R)) for _ in range(200)]
    cases += [(0, 0, 0), (R - 1, R - 1, R - 1), (O - 1 - 5 * 7 % O, 5, 7), (R, 0, 0) if False else (R - 1, 1, 1)]
    # force results into [R, ORDER): s = target  <=  r = target - h*a mod ORDER (must itself be < R to be a field element)
    forced = 0
    while forced < 20:
        hh, aa = rng.randrange(R), rng.randrange(R)
        target = rng.randrange(R, O)
        rr = (target - hh * aa) % O
        if rr < R:
            cases.append((rr, hh, aa)); forced += 1
    le = lambda v: v.to_bytes(32, "little")
    out = C.create_string_buffer(32 * len(cases))
    h.ht_bjj_s_mod_order(b"".join(le(c[0]) for c in cases), b"".join(le(c[1]) for c in cases), b"".join(le(c[2]) for c in cases), out, len(cases))
    got = [int.from_bytes(out.raw[32 * i:32 * i + 32], "little") for i in range(len(cases))]
    assert got == [(r_ + h_ * a_) % O for r_, h_, a_ in cases]
    assert sum(g >= R for g in got) >= 20


def test_wide_products_and_separate_reduction(h):
    """mul_wide / sqr_wide / mont_reduce_wide (squarings and the lazy Fq2 product are built on them)."""
    rng = random.Random(6)
    xs = [rng.randrange(P) for _ in range(3000)] + [0, 1, P - 1, P - 1, 2**253, P - 2, 2**32 - 1]
    ys = [rng.randrange(P) for _ in range(3000)] + [P - 1, P - 1, P - 1, 1, 2**253, P - 2, 2**224]
    n = len(xs)
    m = C.create_string_buffer(32 * n); s = C.create_string_buffer(32 * n)
    h.ht_wide(cport.fqs(xs), cport.fqs(ys), m, s, C.c_uint64(n))
    assert cport.unfr(m.raw) == [a * b % P for a, b in zip(xs, ys)]
    assert cport.unfr(s.raw) == [a * a % P for a in xs]


def test_lazy_fq2_product_extremes(h):
    rng = random.Random(7)
    cases = [((rng.randrange(P), rng.randrange(P)), (rng.randrange(P), rng.randrange(P))) for _ in range(500)]
    cases += [((0, P - 1), (0, P - 1)), ((P - 1, 0), (P - 1, 0)), ((P - 1, P - 1), (P - 1, P - 1)), ((P - 1, 1), (P - 1, 1)),
              ((1, P - 1), (1, P - 1)), ((P - 2, P - 1), (P - 1, P - 2)), ((0, 0), (5, 7)), ((0, P - 1), (P - 1, 0))]
    o = C.create_string_buffer(64)
    for a, b in cases:
        h.ht_fq2_mul(cport.fqs(a), cport.fqs(b), o)
        assert tuple(cport.unfr(o.raw)) == bn.f2_mul(a, b), (a, b)


def test_field_limbs_hypothesis(h):
    """Property test with boundary-biased operands: limb carries are where Montgomery code breaks."""
    from hypothesis import given, settings, strategies as st

    def elems(mod):
        edges = [0, 1, 2, mod - 1, mod - 2, (mod - 1) // 2, 2**32 - 1, 2**32, 2**64 - 1, 2**128, 2**224 - 1, 2**253, 2**253 + 2**32 - 1]
        limbs = st.lists(st.sampled_from([0, 1, 0xFFFFFFFF, 0xFFFFFFFE, 0x80000000, 0x7FFFFFFF]) | st.integers(0, 2**32 - 1), min_size=8, max_size=8)
        from_limbs = limbs.map(lambda l: sum(v << (32 * i) for i, v in enumerate(l)) % mod)
        return st.sampled_from([e % mod for e in edges]) | from_limbs | st.integers(0, mod - 1)

    for F, mod, pack in (("fq", P, cport.fqs), ("fr", R, cport.frs)):
        @settings(max_examples=300, deadline=None)
        @given(st.lists(st.tuples(elems(mod), elems(mod)), min_size=1, max_size=20))
        def check(pairs):
            xs = [a for a, _ in pairs]; ys = [b for _, b in pairs]
            assert cport.unfr(_binop(h, f"ht_{F}_mul", pack(xs), pack(ys))) == [a * b % mod for a, b in pairs]
            assert cport.unfr(_binop(h, f"ht_{F}_add", pack(xs), pack(ys))) == [(a + b) % mod for a, b in pairs]
            assert cport.unfr(_binop(h, f"ht_{F}_sub", pack(xs), pack(ys))) == [(a - b) % mod for a, b in pairs]
            if F == "fq":
                n = len(xs)
                m = C.create_string_buffer(32 * n); s = C.create_string_buffer(32 * n)
                h.ht_wide(pack(xs), pack(ys), m, s, C.c_uint64(n))
                assert cport.unfr(m.raw) == [a * b % mod for a, b in pairs] and cport.unfr(s.raw) == [a * a % mod for a in xs]
        check()


def test_lazy_chain_ops_stay_below_2p(h):
    """mul_lazy / sqr_lazy on operands anywhere in [0, 2p): congruent to a*b/2^256 and again below 2p (fp.cuh: mont_mul_lazy);
    add_raw + reduce_4p_to_2p on operands whose sum is below 4p."""
    rng = random.Random(11)
    Rm = pow(2, -256, R)
    edges = [0, 1, R - 1, R, R + 1, 2 * R - 1, 2 * R - 2, 2**254, 2**254 - 1, 2**255 - 1 if 2**255 - 1 < 2 * R else 2 * R - 1, (2 * R - 1) & ~0xFFFFFFFF]
    xs = [rng.randrange(2 * R) for _ in range(2000)] + edges + edges
    ys = [rng.randrange(2 * R) for _ in range(2000)] + edges + edges[::-1]
    raw = lambda vs: b"".join(v.to_bytes(32, "little") for v in vs)
    n = len(xs)
    for op in (0, 1, 2):
        out = C.create_string_buffer(32 * n)
        h.ht_fr_lazy_raw(op, raw(xs), raw(ys), out, C.c_uint64(n))
        got = [int.from_bytes(out.raw[32 * i:32 * i + 32], "little") for i in range(n)]
        for a, b, g in zip(xs, ys, got):
            if op == 0:
                assert g < 2 * R and g % R == a * b * Rm % R, (a, b)
            elif op == 1:
                assert g < 2 * R and g % R == a * a * Rm % R, a
            else:
                assert g < 2 * R and g % R == (a + b) % R, (a, b)


def test_mimc7_lazy_chain_matches_spec(h):
    """mimc_core.cuh (one conditional subtraction per round, values in [0, 2p)) against the circomlib-style spec."""
    from oracle import mimc7
    rng = random.Random(12)
    ls = [rng.randrange(R) for _ in range(40)] + [0, 0, R - 1, R - 1, 1, 2**253]
    rs = [rng.randrange(R) for _ in range(40)] + [0, R - 1, 0, R - 1, 2, R - 2]
    out = C.create_string_buffer(32 * len(ls))
    h.ht_mimc7_hash2_lazy(cport.frs(ls), cport.frs(rs), out, C.c_uint64(len(ls)))
    assert cport.unfr(out.raw) == [mimc7.hash2(a, b) for a, b in zip(ls, rs)]


def test_glv_decomposition(h):
    """glv.cuh: k = k1 + k2 * lambda (mod r), |k1|, |k2| < 2^127, and (beta x, y) = lambda (x, y) on G1 -- against big integers
    and the oracle's group law."""
    LAM = 0xb3c4d79d41a917585bfc41088d8daaa78b17ea66b99c90dd
    o = C.create_string_buffer(32); h.ht_glv_beta(o)
    beta = int.from_bytes(o.raw, "little")
    assert pow(beta, 3, P) == 1 and beta != 1 and pow(LAM, 3, R) == 1 and LAM != 1
    rng = random.Random(21)
    for k in (1, 2, 12345, rng.randrange(R)):
        g = bn.g1_mul(bn.G1_GEN, k)
        assert bn.g1_mul(g, LAM) == (beta * g[0] % P, g[1])
    ks = [0, 1, 2, R - 1, R - 2, R // 2, R // 2 + 1, LAM, R - LAM, LAM - 1, 2**253, 2**128, 2**127, 2**127 - 1, 2**64] + [rng.randrange(R) for _ in range(20000)]
    ks += [rng.randrange(2**b) for b in (1, 8, 33, 64, 65, 127, 128, 129, 200, 250) for _ in range(50)]
    out = C.create_string_buffer(65 * len(ks))
    h.ht_glv_decompose(b"".join(k.to_bytes(32, "little") for k in ks), out, C.c_uint64(len(ks)))
    worst = 0
    for i, k in enumerate(ks):
        rec = out.raw[65 * i:65 * i + 65]
        m1, m2, sg = int.from_bytes(rec[:32], "little"), int.from_bytes(rec[32:64], "little"), rec[64]
        k1 = -m1 if sg & 1 else m1
        k2 = -m2 if sg & 2 else m2
        assert (k1 + k2 * LAM - k) % R == 0, k
        assert m1 < 2**127 and m2 < 2**127, k
        worst = max(worst, m1, m2)
    assert worst < int(0.56 * 2**127)
