"""Small end-to-end workload for compute-sanitizer (memcheck / racecheck / initcheck).
  compute-sanitizer --tool memcheck python scripts/sanitize_small.py
Touches every kernel family at sizes that finish in seconds under the sanitizer; checks nothing against the oracle
(tests/ do that) -- the point is address / race / uninitialised-read errors."""
import os, random, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import owshen_b200 as ob

R = ob.FR_MODULUS
rng = random.Random(1)
fr = lambda n: b"".join(rng.randrange(R).to_bytes(32, "little") for _ in range(n))
ctx = ob.Context(0)
ctx.field_op("fr", "mul", fr(100), fr(100))
n, depth = 8, 4
ctx.merkle_paths(fr(n), fr(n * depth), [rng.randrange(16) for _ in range(n)], depth)
ctx.merkle_build(fr(8))
for log_n in (3, 11):
    ctx.ntt(fr(2 << log_n), log_n, 2, False, True)
    ctx.ntt(fr(2 << log_n), log_n, 2, True, True)
pts = ctx.g1_generator_mul(fr(300)); ctx.msm_g1(pts, fr(300)); ctx.g1_sum(pts[:64 * 9])
pts = ctx.g2_generator_mul(fr(50)); ctx.msm_g2(pts, fr(50)); ctx.g2_sum(pts[:128 * 5])
ctx.msm_g1(ctx.g1_generator_mul(fr(1)) * 400, (7).to_bytes(32, "little") * 400)      # heavy-bucket path
pk, vk = ob.setup_withdraw(ctx, 1, *[rng.randrange(1, R) for _ in range(5)])
PK = ob.ProvingKey(ctx, pk)
b = 3
proofs, pub = ob.prove(PK, fr(b), fr(b), fr(b), fr(b), [rng.randrange(2) for _ in range(b)], fr(2 * b))
assert all(ob.verify(vk, pub[96 * i:96 * i + 96], proofs[256 * i:256 * i + 256]) for i in range(b))
ctx.bjj_verify_batch(fr(4), bytes(4), fr(4), fr(12))
msgs = fr(4)
pkx, odd, sigs, st = ctx.bjj_sign_batch(fr(4), fr(4), msgs)                            # window-table fixed-base path
assert list(ctx.bjj_verify_batch(pkx, odd, msgs, sigs)) == [1] * 4
# round 2 kernels: tree append, a batch in several chunks, G2 heavy buckets, shared-memory G2 reduction, cooperative Horner
t = ob.MerkleTree(ctx, 5)
t.insert_batch([1, 2, 3]); t.insert(4); t.insert_batch(list(range(5, 16))); t.rollback(6); t.pop_batch()
os.environ["OG_CHUNK"] = "2"
b = 5
proofs, pub = ob.prove(PK, fr(b), fr(b), fr(b), fr(b), [rng.randrange(2) for _ in range(b)], fr(2 * b))
assert all(ob.verify(vk, pub[96 * i:96 * i + 96], proofs[256 * i:256 * i + 256]) for i in range(b))
p2 = ctx.g2_generator_mul(fr(1)) * 300
ctx.msm_g2(p2, (5).to_bytes(32, "little") * 300)
# later in round 2: reduction tail of one-shot MSMs (k_tail_sums / k_tail_finish need >= 512 buckets per window, i.e. >= 2^13 points),
# three-barrier Horner, lazy MiMC chain (covered by merkle_paths above)
os.environ.pop("OG_CHUNK")
pts = ctx.g1_generator_mul(fr(8192)); ctx.msm_g1(pts, fr(8192))
pts = ctx.g2_generator_mul(fr(8192)); ctx.msm_g2(pts, fr(8192))
PK.close(); ctx.close()
print("sanitize workload done")
