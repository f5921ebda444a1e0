"""Parity tests proper: the CUDA path, called through the C ABI, against the oracle on the same seeded
inputs (bit-exact: this is integer / byte work), plus size-independent properties at BASELINE sizes."""
import hashlib
import json
import os
import random

import pytest

import owshen_b200 as ob
from owshen_b200 import api
from oracle import bn254 as bn
from oracle import cport, mimc7
from oracle import withdraw_circuit as wc
from tests.helpers import pk_blob, rand_fr_bytes, rand_g1, rand_g2, rand_inputs, vk_blob

pytestmark = pytest.mark.gpu
R, P = bn.R, bn.P
GOLD = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "vectors.json")))


def test_library_is_the_cuda_one(ctx):
    n0 = ctx.launch_count
    ctx.field_op("fr", "mul", bn.fr_to_bytes(3), bn.fr_to_bytes(5))
    assert ctx.launch_count == n0 + 1
    a, b = ctx.imad_peak()
    assert a > 1e12 and b > 1e12


def test_field_ops_ptx_path(ctx):
    rng = random.Random(1)
    for F, mod, pack in (("fq", P, cport.fqs), ("fr", R, cport.frs)):
        xs = [rng.randrange(mod) for _ in range(20000)] + [0, 1, mod - 1, mod - 1, 2**253, mod - 2, 2**32 - 1]
        ys = [rng.randrange(mod) for _ in range(20000)] + [mod - 1, mod - 1, mod - 1, 1, 2**253, mod - 2, 2**224]
        assert cport.unfr(ctx.field_op(F, "mul", pack(xs), pack(ys))) == [a * b % mod for a, b in zip(xs, ys)]
        assert cport.unfr(ctx.field_op(F, "add", pack(xs), pack(ys))) == [(a + b) % mod for a, b in zip(xs, ys)]
        assert cport.unfr(ctx.field_op(F, "sub", pack(xs), pack(ys))) == [(a - b) % mod for a, b in zip(xs, ys)]
    for v in GOLD["field"]:
        pack = cport.fqs if v["field"] == "fq" else cport.frs
        a, b = pack([int(x) for x in v["a"]]), pack([int(x) for x in v["b"]])
        for op in ("mul", "add", "sub"):
            assert cport.unfr(ctx.field_op(v["field"], op, a, b)) == [int(x) for x in v[op]]
    with pytest.raises(ob.OwshenB200Error) as e:
        ctx.field_op("fr", "mul", R.to_bytes(32, "little"), bytes(32))
    assert e.value.code == -2


def test_mimc7_hash_and_merkle_paths(ctx):
    rng = random.Random(2)
    xs = [rng.randrange(R) for _ in range(100)] + [0, 1, R - 1]
    ys = [rng.randrange(R) for _ in range(100)] + [0, 2, R - 1]
    assert cport.unfr(ctx.mimc7_hash2(cport.frs(xs), cport.frs(ys))) == [cport.mimc7_multi_hash([a, b]) for a, b in zip(xs, ys)]
    assert mimc7.hash2(xs[0], ys[0]) == cport.mimc7_multi_hash([xs[0], ys[0]])
    g = GOLD["mimc7"]
    assert cport.unfr(ctx.mimc7_hash2(cport.frs([1]), cport.frs([2])))[0] == int(g["multi_hash_1_2"])
    pth = g["path"]
    got = cport.unfr(ctx.merkle_paths(cport.frs([int(pth["leaf"])]), cport.frs([int(x) for x in pth["siblings"]]), [pth["bits"]], 3))
    assert got == [int(x) for x in pth["nodes"]]
    for n, depth in ((1, 1), (5, 7), (300, 32)):
        leaves, sib = rand_fr_bytes(rng, n), rand_fr_bytes(rng, n * depth)
        bits = [rng.randrange(1 << depth) for _ in range(n)]
        assert ctx.merkle_paths(leaves, sib, bits, depth) == cport.merkle_paths(leaves, sib, bits, depth)
    assert ctx.merkle_paths(b"", b"", [], 5) == b""


def test_merkle_paths_config2_full_size(ctx):
    """BASELINE config 2: 4096 leaves x depth 32, bit-exact vs the oracle."""
    rng = random.Random(3)
    n, depth = 4096, 32
    leaves, sib = rand_fr_bytes(rng, n), rand_fr_bytes(rng, n * depth)
    bits = [rng.randrange(1 << 32) for _ in range(n)]
    assert ctx.merkle_paths(leaves, sib, bits, depth) == cport.merkle_paths(leaves, sib, bits, depth)


def test_merkle_tree_api(ctx):
    rng = random.Random(4)
    leaves = [rng.randrange(R) for _ in range(4)]
    t = ob.MerkleTree(ctx, 2)
    t.insert_batch(leaves)
    ref = mimc7.MerkleTree(2)
    for l in leaves:
        ref.insert(l)
    assert int.from_bytes(t.root(), "little") == ref.root()
    gl = [int(x) for x in GOLD["mimc7"]["tree4_leaves"]]
    tg = ob.MerkleTree(ctx, 2); tg.insert_batch(gl)
    assert int.from_bytes(tg.root(), "little") == int(GOLD["mimc7"]["tree4_root"])
    # deeper sparse tree: incremental inserts, paths re-derive the root on the GPU
    t = ob.MerkleTree(ctx, 20); ref = mimc7.MerkleTree(20)
    vals = [rng.randrange(R) for _ in range(9)]
    t.insert_batch(vals[:5]); t.insert(vals[5]); t.insert_batch(vals[6:])
    for v in vals:
        ref.insert(v)
    assert int.from_bytes(t.root(), "little") == ref.root()
    sibs, bits = t.path(6)
    nodes = ctx.merkle_paths(bn.fr_to_bytes(vals[6]), sibs, [bits], 20)
    assert nodes[-32:] == t.root()
    # persistence behind the KvStore-shaped interface: reopen the same store
    reopened = ob.MerkleTree(ctx, 20, store=t.store)
    assert reopened.n_leaves == 9 and reopened.root() == t.root() and reopened.path(6) == (sibs, bits)
    reopened.insert(123)
    ref.insert(123)
    assert int.from_bytes(reopened.root(), "little") == ref.root()
    with pytest.raises(ValueError):
        ob.MerkleTree(ctx, 19, store=t.store)
    lv = ctx.merkle_build(cport.frs(vals[:8]))
    r8 = mimc7.MerkleTree(3)
    for v in vals[:8]:
        r8.insert(v)
    assert int.from_bytes(lv[-32:], "little") == r8.root()


def test_ntt_matches_oracle_all_modes(ctx):
    rng = random.Random(5)
    for log_n in (0, 1, 2, 3, 7, 10, 11, 12, 13, 14, 15, 16, 17):     # every parity of levels per pass
        n = 1 << log_n
        batch = 3 if log_n <= 12 else (2 if log_n <= 16 else 1)
        data = rand_fr_bytes(rng, n * batch)
        for inv in (False, True):
            for co in (False, True):
                got = ctx.ntt(data, log_n, batch, inv, co)
                exp = b"".join(cport.ntt(data[32 * n * b:32 * n * (b + 1)], inv, co) for b in range(batch))
                assert got == exp, (log_n, inv, co)
    for v in GOLD["ntt"]:
        r2 = random.Random(v["seed"])
        data = cport.frs([r2.randrange(R) for _ in range(1 << v["log_n"])])
        got = ctx.ntt(data, v["log_n"], 1, v["inverse"], v["coset"])
        assert hashlib.sha256(got).hexdigest() == v["sha256"]


def test_ntt_properties_2_20(ctx):
    """Size-independent properties at n = 2^20: round trip and linearity (oracle-free)."""
    rng = random.Random(6)
    log_n, n = 20, 1 << 20
    a, b = rand_fr_bytes(rng, n), rand_fr_bytes(rng, n)
    fa = ctx.ntt(a, log_n, 1, False, True)
    assert ctx.ntt(fa, log_n, 1, True, True) == a
    fb = ctx.ntt(b, log_n)
    fa0 = ctx.ntt(a, log_n)
    ab = ctx.field_op("fr", "add", a, b)
    assert ctx.ntt(ab, log_n) == ctx.field_op("fr", "add", fa0, fb)
    assert fa0 == cport.ntt(a)            # and the oracle agrees at full size


def test_msm_g1_glv_edge_scalars(ctx):
    """One-shot G1 MSMs of >= 1024 points run the GLV front end (glv.cuh): k = k1 + k2 lambda with the signs folded into the
    points.  Scalars around the lattice constants, the 2^127 boundary and r, points at infinity, P / -P pairs that cancel."""
    rng = random.Random(77)
    LAM = 0xb3c4d79d41a917585bfc41088d8daaa78b17ea66b99c90dd
    A1, A2 = 9931322734385697763, 147946756881789319010696353538189108491
    special = [0, 1, 2, R - 1, R - 2, LAM, R - LAM, LAM - 1, LAM + 1, LAM * LAM % R, 2**127, 2**127 - 1, 2**127 + 1, 2**128, 2**126,
               A1, A2, R - A1, R - A2, (A1 * LAM) % R, (A2 * LAM) % R, R // 2, R // 2 + 1, 2**253, 2**64, 2**64 - 1, 2**32]
    n = 3000
    sc = [special[i % len(special)] if i % 3 else rng.randrange(R) for i in range(n)]
    pts = bytearray(rand_g1(rng, n))
    for i in range(0, 200, 2):                           # P, -P with the same scalar: the pair cancels
        x, y = pts[64 * i:64 * i + 32], int.from_bytes(pts[64 * i + 32:64 * i + 64], "little")
        pts[64 * (i + 1):64 * (i + 2)] = x + ((bn.P - y) % bn.P).to_bytes(32, "little")
        sc[i + 1] = sc[i]
    for i in (5, 1023, 1024, 2999):
        pts[64 * i:64 * (i + 1)] = bytes(64)             # infinity
    pts = bytes(pts)
    assert ctx.msm_g1(pts, cport.frs(sc)) == cport.g1_msm(pts, cport.frs(sc))
    for k in special:                                    # every special scalar on every point at once: sum = k * (sum of points)
        m = 1024
        assert ctx.msm_g1(pts[:64 * m], cport.frs([k] * m)) == cport.g1_msm(pts[:64 * m], cport.frs([k] * m)), hex(k)


def test_msm_edge_cases(ctx):
    rng = random.Random(7)
    for n in (0, 1, 2, 3, 33, 255, 1024, 5000):
        pts = rand_g1(rng, n)
        sc = [rng.randrange(R) for _ in range(n)]
        if n >= 3:
            sc[0] = 0; sc[1] = 1; sc[2] = R - 1
        if n >= 33:
            pts = pts[:64 * 5] + pts[64 * 4:64 * 5] + pts[64 * 6:]      # duplicate point
            pts = pts[:64 * 7] + bytes(64) + pts[64 * 8:]                 # point at infinity
        assert ctx.msm_g1(pts, cport.frs(sc)) == cport.g1_msm(pts, cport.frs(sc)), n
    for n in (0, 1, 2, 77, 600):
        pts = rand_g2(rng, n)
        sc = cport.frs([rng.randrange(R) for _ in range(n)])
        assert ctx.msm_g2(pts, sc) == cport.g2_msm(pts, sc), n
    for v in GOLD["msm"]:
        f = ctx.msm_g1 if v["curve"] == "g1" else ctx.msm_g2
        assert f(bytes.fromhex(v["points"]), bytes.fromhex(v["scalars"])).hex() == v["out"]
    n = 20000                                                            # all-equal points and scalars: P+P in every bucket
    pts = rand_g1(rng, 1) * n
    sc = cport.frs([7] * n)
    assert ctx.msm_g1(pts, sc) == cport.g1_msm(pts, sc)
    pts = rand_g1(rng, n)                                                # witness-like scalars: heavy buckets
    sc = cport.frs([rng.choice([0, 1, 1, rng.randrange(1 << 64), rng.randrange(R)]) for _ in range(n)])
    assert ctx.msm_g1(pts, sc) == cport.g1_msm(pts, sc)
    with pytest.raises(ob.OwshenB200Error):
        ctx.msm_g1(pts[:64], R.to_bytes(32, "little"))
    s9 = rand_g1(rng, 9)
    exp = bytes(64)
    for i in range(9):
        exp = cport.g1_add(exp, s9[64 * i:64 * i + 64])
    assert ctx.g1_sum(s9) == exp
    s5 = rand_g2(rng, 5)
    exp = bytes(128)
    for i in range(5):
        exp = cport.g2_add(exp, s5[128 * i:128 * i + 128])
    assert ctx.g2_sum(s5) == exp


def test_generator_mul_and_probes(ctx):
    rng = random.Random(21)
    ks = cport.frs([0, 1, R - 1] + [rng.randrange(R) for _ in range(30)])
    assert ctx.g1_generator_mul(ks) == cport.g1_fixed_mul_batch(bn.g1_to_bytes(bn.G1_GEN), ks)
    assert ctx.g2_generator_mul(ks) == cport.g2_fixed_mul_batch(bn.g2_to_bytes(bn.G2_GEN), ks)
    p = ctx.int_pipe_peaks()
    assert p["imad_per_s"] > p["imad_wide_carry_chain_per_s"] > 1e12
    assert ctx.fp64_peak() > 1e12


def test_msm_config3_2_20(ctx):
    """BASELINE config 3: 2^20-point G1 MSM, uniform and witness-like scalars, bit-exact vs the CPU MSM;
    plus linearity msm(P, a) + msm(P, b) == msm(P, a + b)."""
    rng = random.Random(8)
    n = 1 << 20
    pts = rand_g1(rng, n)
    a = rand_fr_bytes(rng, n)
    ra = ctx.msm_g1(pts, a)
    assert ra == cport.g1_msm(pts, a)
    wl = bytearray(rand_fr_bytes(rng, n))
    for i in range(n):                     # 60 % in {0,1}, 30 % < 2^64, 10 % uniform
        u = rng.random()
        if u < 0.6:
            wl[32 * i:32 * i + 32] = (rng.randrange(2)).to_bytes(32, "little")
        elif u < 0.9:
            wl[32 * i + 8:32 * i + 32] = bytes(24)
    wl = bytes(wl)
    rb = ctx.msm_g1(pts, wl)
    assert rb == cport.g1_msm(pts, wl)
    ab = ctx.field_op("fr", "add", a, wl)
    assert ctx.msm_g1(pts, ab) == cport.g1_add(ra, rb)


def test_withdraw_witness(ctx):
    rng = random.Random(9)
    for depth, batch in ((1, 2), (2, 3), (32, 5)):
        nul, sec, rec, sib, bits = rand_inputs(rng, batch, depth)
        assert ctx.withdraw_witness(depth, nul, sec, rec, sib, bits) == cport.withdraw_witness(nul, sec, rec, sib, bits, depth)


@pytest.fixture(scope="module")
def keys32(ctx):
    rng = random.Random(10)
    tw = [rng.randrange(1, R) for _ in range(5)]
    pk, vk = ob.setup_withdraw(ctx, 32, *tw)
    cs = wc.build_r1cs(32)
    pkb, vkb = cport.setup_bytes(cs, *tw)
    return pk, vk, cs, pkb, vkb


def test_setup_matches_oracle(ctx, keys32):
    pk, vk, cs, pkb, vkb = keys32
    assert vk == vk_blob(vkb)
    assert pk == pk_blob(cs, pkb, 32)
    rng = random.Random(11)
    tw = [rng.randrange(1, R) for _ in range(5)]
    pk2, vk2 = ob.setup_withdraw(ctx, 2, *tw)
    cs2 = wc.build_r1cs(2)
    pkb2, vkb2 = cport.setup_bytes(cs2, *tw)
    assert pk2 == pk_blob(cs2, pkb2, 2) and vk2 == vk_blob(vkb2)
    with pytest.raises(ob.OwshenB200Error):
        ob.setup_withdraw(ctx, 2, 1, 2, 3, 4, 5)         # tau = 1 lies in the evaluation domain


def test_groth16_golden_proof(ctx):
    g = GOLD["groth16"]
    depth = g["depth"]
    pk, vk = ob.setup_withdraw(ctx, depth, *[int(x) for x in g["toxic"]])
    v = g["vk"]
    assert vk[12:].hex() == v["alpha1"] + v["beta2"] + v["gamma2"] + v["delta2"] + v["ic"]
    PK = ob.ProvingKey(ctx, pk)
    f = lambda k: bn.fr_to_bytes(int(g[k]))
    proofs, pub = ob.prove(PK, f("nullifier"), f("secret"), f("recipient"), f("sibling"), [g["bits"]], f("r") + f("s"))
    assert proofs.hex() == g["proof"]
    assert cport.unfr(pub) == [int(x) for x in g["public"]]
    assert ob.verify(vk, pub, proofs)
    wit = ctx.withdraw_witness(depth, f("nullifier"), f("secret"), f("recipient"), f("sibling"), [g["bits"]])
    assert hashlib.sha256(wit).hexdigest() == g["witness_sha256"]
    PK.close()


def test_groth16_prove_bit_exact_vs_oracle(ctx, keys32, monkeypatch):
    monkeypatch.setenv("OG_CHUNK", "64")         # the 70-proof batch below then spans two chunks of the prover
    pk, vk, cs, pkb, vkb = keys32
    rng = random.Random(12)
    PK = ob.ProvingKey(ctx, pk)
    assert (PK.n_vars, PK.n_pub, PK.log_m, PK.depth) == (cs.n_vars, 3, 15, 32)
    batch = 70
    nul, sec, rec, sib, bits = rand_inputs(rng, batch, 32)
    rs = cport.frs([rng.randrange(R) for _ in range(2 * batch)])
    wit = cport.withdraw_witness(nul, sec, rec, sib, bits, 32)
    opr = cport.Prover(cs, pkb)
    assert PK.h_evals(wit[:32 * cs.n_vars]) == opr.h_evals(wit[:32 * cs.n_vars])
    proofs, pub = ob.prove(PK, nul, sec, rec, sib, bits, rs)
    nck = 12
    idx = [0, 1, 2, 3, 4, 5, 62, 63, 64, 65, 68, 69]
    w_sel = b"".join(wit[32 * cs.n_vars * i:32 * cs.n_vars * (i + 1)] for i in idx)
    rs_sel = b"".join(rs[64 * i:64 * i + 64] for i in idx)
    exp = opr.prove_batch(w_sel, rs_sel)
    for k, i in enumerate(idx):
        assert proofs[256 * i:256 * i + 256] == exp[256 * k:256 * k + 256], i
    for i in (0, 63, 64, 69):
        p, x = proofs[256 * i:256 * i + 256], pub[96 * i:96 * i + 96]
        assert x == wit[32 * cs.n_vars * i + 32:32 * cs.n_vars * i + 128]
        assert ob.verify(vk, x, p)
        bad = bytearray(x); bad[40] ^= 1
        assert not ob.verify(vk, bytes(bad), p)
    assert PK.prove_witnesses(wit[:32 * cs.n_vars * 3], rs[:192]) == proofs[:768]
    # r = s = 0 and identical inputs in one batch
    z = ob.prove(PK, nul[:32] * 2, sec[:32] * 2, rec[:32] * 2, sib[:32 * 32] * 2, bits[:1] * 2, bytes(128))[0]
    assert z[:256] == z[256:] == opr.prove(wit[:32 * cs.n_vars], 0, 0)
    with pytest.raises(ob.OwshenB200Error):
        ob.prove(PK, R.to_bytes(32, "little"), sec[:32], rec[:32], sib[:32 * 32], bits[:1], rs[:64])
    PK.close()


def test_groth16_batch_1024_default_chunk(ctx, keys32):
    """BASELINE config 4 at its full size and with the default chunking (what bench.py times): 1024 proofs in one call;
    the first, the last and two seeded-random proofs are compared byte for byte with the oracle's C prover, 16 proofs
    spread over the batch must verify against their own public inputs, and all proofs are pairwise distinct."""
    pk, vk, cs, pkb, vkb = keys32
    rng = random.Random(1024)
    PK = ob.ProvingKey(ctx, pk)
    batch = 1024
    nul, sec, rec, sib, bits = rand_inputs(rng, batch, 32)
    rs = cport.frs([rng.randrange(R) for _ in range(2 * batch)])
    proofs, pub = ob.prove(PK, nul, sec, rec, sib, bits, rs)
    PK.close()
    assert len(proofs) == 256 * batch and len(pub) == 96 * batch
    idx = [0, batch - 1] + sorted(rng.sample(range(1, batch - 1), 2))
    sel = lambda b, w: b"".join(b[w * i:w * i + w] for i in idx)
    wit = cport.withdraw_witness(sel(nul, 32), sel(sec, 32), sel(rec, 32), sel(sib, 32 * 32), [bits[i] for i in idx], 32)
    exp = cport.Prover(cs, pkb).prove_batch(wit, sel(rs, 64))
    for k, i in enumerate(idx):
        assert proofs[256 * i:256 * i + 256] == exp[256 * k:256 * k + 256], i
        assert pub[96 * i:96 * i + 96] == wit[32 * cs.n_vars * k + 32:32 * cs.n_vars * k + 128], i
    for i in range(0, batch, 64):
        assert ob.verify(vk, pub[96 * i:96 * i + 96], proofs[256 * i:256 * i + 256]), i
    assert len({proofs[256 * i:256 * i + 256] for i in range(batch)}) == batch


def test_groth16_chunks_match_single_chunk(ctx, keys32, monkeypatch):
    """A batch cut into chunks (the last one partial) must produce the bytes of one chunk covering the whole batch."""
    pk = keys32[0]
    rng = random.Random(77)
    PK = ob.ProvingKey(ctx, pk)
    batch = 45
    nul, sec, rec, sib, bits = rand_inputs(rng, batch, 32)
    rs = cport.frs([rng.randrange(R) for _ in range(2 * batch)])
    monkeypatch.setenv("OG_CHUNK", "1024")
    ref = ob.prove(PK, nul, sec, rec, sib, bits, rs)
    for chunk in (16, 7):
        monkeypatch.setenv("OG_CHUNK", str(chunk))
        assert ob.prove(PK, nul, sec, rec, sib, bits, rs) == ref, chunk
    PK.close()


def test_merkle_append_and_rollback(ctx):
    """og_mimc7_merkle_append against the spec tree (odd start indices, batches crossing subtree boundaries), then the
    undo path: pop_batch / rollback restore earlier roots bit for bit; a full tree refuses more leaves."""
    rng = random.Random(41)
    depth = 9
    t = ob.MerkleTree(ctx, depth); ref = mimc7.MerkleTree(depth)
    roots, sizes, vals = [t.root()], [0], []
    for n in (1, 2, 5, 1, 64, 3, 100):
        batch = [rng.randrange(R) for _ in range(n)]
        t.insert_batch(batch); vals += batch
        for v in batch:
            ref.insert(v)
        assert int.from_bytes(t.root(), "little") == ref.root(), n
        roots.append(t.root()); sizes.append(t.n_leaves)
    for i in (0, 7, 8, 72, 175):
        sib, bits = t.path(i)
        assert sib == b"".join(bn.fr_to_bytes(x) for x in ref.path(i)[0])
        assert ctx.merkle_paths(bn.fr_to_bytes(vals[i]), sib, [bits], depth)[-32:] == t.root()
    assert t.pop_batch() == 100 and t.root() == roots[-2]
    t.rollback(sizes[3])
    assert t.root() == roots[3] and t.n_leaves == sizes[3]
    t.rollback(5)                                            # inside the third batch
    r5 = mimc7.MerkleTree(depth)
    for v in vals[:5]:
        r5.insert(v)
    assert int.from_bytes(t.root(), "little") == r5.root()
    t.rollback(0)
    assert t.root() == roots[0]
    small = ob.MerkleTree(ctx, 2)
    small.insert_batch([1, 2, 3])
    with pytest.raises(OverflowError):
        small.insert_batch([4, 5])
    small.insert(4)
    with pytest.raises(OverflowError):
        small.insert(5)
    with pytest.raises(ValueError):
        ctx.merkle_append(2, 3, bytes(64), bytes(64), bytes(64))      # 2 leaves at index 3 of a 4-leaf tree


def test_msm_adversarial_bucket_lists(ctx):
    """Bucket lists that hit every exceptional branch of the accumulation and the segmented heavy-bucket path: infinity
    points, one point repeated with the same scalar (P + P, then 2P + P ... in one bucket of every window), P and -P with
    the same scalar (P - P), scalars r - 1 / 0 / 1, and an MSM whose every list is the whole input (all buckets heavy:
    k_heavy_plan / k_bucket_heavy segments / k_heavy_combine)."""
    rng = random.Random(303)
    n = 3000
    pts = bytearray(rand_g1(rng, n))
    sc = [rng.randrange(R) for _ in range(n)]
    for i in range(0, 300, 3):
        pts[64 * i:64 * i + 64] = bytes(64)                                   # infinity points
    for i in range(300, 900):
        pts[64 * i:64 * i + 64] = pts[64 * 300:64 * 300 + 64]                 # one point 600 times ...
    for i in range(300, 600):
        sc[i] = sc[300]                                                       # ... 300 of them with the same scalar
    neg = bn.g1_to_bytes(bn.g1_neg(bn.g1_from_bytes(bytes(pts[64 * 1000:64 * 1000 + 64]))))
    pts[64 * 1001:64 * 1001 + 64] = neg; sc[1001] = sc[1000]                  # P and -P with the same scalar: P - P
    sc[1500], sc[1501], sc[1502] = R - 1, 0, 1
    for i in range(2000, 2064):                                               # 64 equal entries in one bucket of every window
        pts[64 * i:64 * i + 64] = pts[64 * 2000:64 * 2000 + 64]; sc[i] = sc[2000]
    pts, scb = bytes(pts), cport.frs(sc)
    assert ctx.msm_g1(pts, scb) == cport.g1_msm(pts, scb)
    same = cport.frs([sc[7]] * n)                                             # every bucket list = the whole input
    assert ctx.msm_g1(pts, same) == cport.g1_msm(pts, same)
    n2 = 700
    p2 = bytearray(rand_g2(rng, n2)); s2 = [rng.randrange(R) for _ in range(n2)]
    for i in range(100, 400):
        p2[128 * i:128 * i + 128] = p2[128 * 100:128 * 100 + 128]; s2[i] = s2[100]      # 300 equal entries: heavy in G2
    p2[128 * 5:128 * 5 + 128] = bytes(128)
    p2, s2b = bytes(p2), cport.frs(s2)
    assert ctx.msm_g2(p2, s2b) == cport.g2_msm(p2, s2b)
    big = rand_g1(rng, 1 << 16)
    wl = bytearray(rand_fr_bytes(rng, 1 << 16))
    for i in range(0, 1 << 16, 2):
        wl[32 * i:32 * i + 32] = (1).to_bytes(32, "little")                  # half the scalars are 1: one bucket of 32768 entries
    assert ctx.msm_g1(big, bytes(wl)) == cport.g1_msm(big, bytes(wl))


def test_external_known_answers(ctx):
    """The CUDA library against published vectors it did not produce (tests/golden/external_vectors.json): EIP-196 point
    addition / scalar multiplication through og_g1_sum / og_msm_g1 / the fixed-base generator path."""
    ext = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "external_vectors.json")))["eip196"]
    pt = lambda xy: bn.g1_to_bytes((int(xy[0], 16), int(xy[1], 16)))
    add = ext["add_chfast1"]
    assert ctx.g1_sum(pt(add["a"]) + pt(add["b"])) == pt(add["sum"])
    mul = ext["mul_chfast1"]
    assert ctx.msm_g1(pt(mul["p"]), cport.frs([int(mul["k"], 16)])) == pt(mul["product"])
    two = pt([ext["g1_generator_doubled"]["x"], ext["g1_generator_doubled"]["y"]])
    assert ctx.g1_generator_mul(cport.frs([2])) == two
    assert ctx.g1_sum(bn.g1_to_bytes(bn.G1_GEN) * 2) == two
    assert ctx.msm_g1(pt(add["a"]) + pt(add["b"]), cport.frs([1, 1])) == pt(add["sum"])


def _nccl_world1():
    import socket
    import torch.distributed as dist
    if not dist.is_initialized():
        s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
        dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1)
    return dist


def test_msm_sharded_world1_vs_oracle_and_single_gpu(ctx):
    """BASELINE config 5 through the product function owshen_b200.sharded.msm_sharded (NCCL process group of this box's
    one visible rank): 2^16 G1 / 2^13 G2 against the oracle's CPU MSM, 2^20 G1 against the single-GPU entry point, and
    the device-tensor variant against the host-buffer one."""
    import torch
    from owshen_b200.sharded import msm_sharded, msm_sharded_dev
    dist = _nccl_world1()
    try:
        rng = random.Random(55)
        n = 1 << 16
        pts, sc = rand_g1(rng, n), rand_fr_bytes(rng, n)
        got = msm_sharded(ctx, pts, sc, "g1")
        assert got == cport.g1_msm(pts, sc)
        n2 = 1 << 13
        pts2, sc2 = rand_g2(rng, n2), rand_fr_bytes(rng, n2)
        assert msm_sharded(ctx, pts2, sc2, "g2") == cport.g2_msm(pts2, sc2)
        dev = torch.device("cuda", ctx.device)
        d_p = torch.frombuffer(bytearray(pts), dtype=torch.uint8).to(dev)
        d_s = torch.frombuffer(bytearray(sc), dtype=torch.uint8).to(dev)
        torch.cuda.synchronize()
        res = msm_sharded_dev(ctx, d_p, d_s, "g1")
        ctx.sync()
        assert bytes(res.cpu().numpy().tobytes()) == got
        n = 1 << 20
        ks = rand_fr_bytes(rng, n)
        big = ctx.g1_generator_mul(ks)
        sc = rand_fr_bytes(rng, n)
        assert msm_sharded(ctx, big, sc, "g1") == ctx.msm_g1(big, sc)
        assert msm_sharded(ctx, b"", b"", "g1") == bytes(64)
        with pytest.raises(ValueError):
            msm_sharded(ctx, pts[:64], sc[:64], "g1")
    finally:
        dist.destroy_process_group()


def _sharded_worker(rank, world, port, pts, sc, pts2, sc2, q):
    import torch
    import torch.distributed as dist
    from owshen_b200.sharded import msm_sharded
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    c = ob.Context(rank)
    try:
        q.put((rank, msm_sharded(c, pts, sc, "g1"), msm_sharded(c, pts2, sc2, "g2")))
        dist.barrier()
    finally:
        c.close()
        dist.destroy_process_group()


def test_msm_sharded_two_gpus(ctx):
    """The same function over a real NCCL all-gather: two ranks, two GPUs, results equal the single-GPU MSM and the oracle."""
    import socket
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    rng = random.Random(56)
    n, n2 = 50001, 3001
    pts, sc = rand_g1(rng, n), rand_fr_bytes(rng, n)
    pts2, sc2 = rand_g2(rng, n2), rand_fr_bytes(rng, n2)
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    procs = [mpc.Process(target=_sharded_worker, args=(r, 2, port, pts, sc, pts2, sc2, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in range(2)]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    e1, e2 = cport.g1_msm(pts, sc), cport.g2_msm(pts2, sc2)
    assert e1 == ctx.msm_g1(pts, sc) and e2 == ctx.msm_g2(pts2, sc2)
    for _, g1, g2 in got:
        assert g1 == e1 and g2 == e2


def test_pk_blob_rejects_garbage(ctx, keys32):
    pk = keys32[0]
    with pytest.raises(ob.OwshenB200Error):
        ob.ProvingKey(ctx, b"NOPE" + pk[4:])
    with pytest.raises(ob.OwshenB200Error):
        ob.ProvingKey(ctx, pk[:len(pk) // 2])


def test_two_contexts_in_one_process(ctx):
    """One context per GPU inside one process (INTEGRATION.md: one Prover per GPU): interleaved calls must each
    run on their own device.  Needs two GPUs; skipped on a single-GPU box."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    rng = random.Random(31)
    c1 = ob.Context(1)
    try:
        pts = rand_g1(rng, 500)
        sc = cport.frs([rng.randrange(R) for _ in range(500)])
        exp = cport.g1_msm(pts, sc)
        for _ in range(3):
            assert ctx.msm_g1(pts, sc) == exp
            assert c1.msm_g1(pts, sc) == exp
        x, y = cport.frs([3, 5]), cport.frs([7, 11])
        assert c1.mimc7_hash2(x, y) == ctx.mimc7_hash2(x, y)
        # a proving key is bound to the GPU that loaded it: another context's GPU must refuse it, not fault
        pk_bytes, _ = ob.setup_withdraw(ctx, 2, 11, 12, 13, 14, 15)
        PK = ob.ProvingKey(ctx, pk_bytes)
        PK.ctx = c1
        with pytest.raises(ob.OwshenB200Error) as e:
            PK.prove_withdraw(cport.frs([1]), cport.frs([2]), cport.frs([3]), cport.frs([1, 2]), [0], cport.frs([1, 2]))
        assert e.value.code == api.OG_E_INVALID and "another device" in str(e.value)
        PK.ctx = ctx
        PK.close()
    finally:
        c1.close()
