"""The one-shot MSM (og_msm_g1 / og_msm_g2) at every window size it can pick, and at the 2^24-point size of BASELINE config 5.

`msm_dev` (owshen_b200/csrc/msm.cu) derives its whole shape from n: the window c, the window count, whether the levels
above reduction level 0 run through k_reduce_level or the tail sums (and in how many slices), and the cap and segment
length of the heavy-bucket path.  Every test here feeds the same input recipe -- special scalars, digit-boundary scalars
for that c, points at infinity, P / -P pairs that cancel and a run of identical entries long enough to go down the
heavy path -- at one size per (curve, c) and at the sizes around the window changes, and requires the bytes of a
reference:
  * up to CPORT_MAX points the oracle's C MSM (cport.g1_msm / g2_msm);
  * above it a linear-combination oracle: with P_i = k_i G for known k_i, sum s_i P_i = (sum k_i s_i mod r) G, one
    fixed-base multiplication of an integer dot product.  Infinity is k = 0, -P is r - k and a repeated point repeats k,
    so the recipe carries over unchanged.  test_linear_oracle_agrees_with_cport anchors this oracle against the first.
"""
import random

import numpy as np
import pytest

from owshen_b200 import api
from oracle import bn254 as bn
from oracle import cport

R = bn.R
GEN = {"g1": bn.g1_to_bytes(bn.G1_GEN), "g2": bn.g2_to_bytes(bn.G2_GEN)}
PB = {"g1": 64, "g2": 128}
FIXED_MUL = {"g1": cport.g1_fixed_mul_batch, "g2": cport.g2_fixed_mul_batch}
CPU_MSM = {"g1": cport.g1_msm, "g2": cport.g2_msm}
CPORT_MAX = 150_000                     # above this the CPU MSM (and making its points) costs seconds per call
LAM = 0xb3c4d79d41a917585bfc41088d8daaa78b17ea66b99c90dd                  # GLV eigenvalue and lattice constants (glv.cuh)
A1, A2 = 9931322734385697763, 147946756881789319010696353538189108491


def window(curve: str, n: int):
    """(c, glv) of an n-point one-shot MSM, as `msm_dev` / `pick_window` in owshen_b200/csrc/msm.cu choose them: G1 from 1024
    points runs the GLV front end, which doubles the point count before the window is picked; c = floor(log2 m) - 3 for
    m points, clamped to 2..16."""
    glv = curve == "g1" and n >= 1024
    m = 2 * n if glv else n
    return max(2, min(16, m.bit_length() - 4)), glv


def heavy_shape(curve: str, n: int):
    """(cap, seg) of msm_buckets: a bucket holding more than `cap` entries goes to the heavy path, which cuts it into
    segments of `seg` entries.  Both follow from the average bucket load."""
    c, glv = window(curve, n)
    avg = (2 * n if glv else n) // (1 << (c - 1))
    return max(128, 4 * avg), max(2048, 4 * avg)


def reachable():
    """Every (curve, c, glv) the rule gives for 1 <= n < 2^28 (c is monotone in n: both ends of each octave suffice)."""
    return {(cv,) + window(cv, n) for cv in ("g1", "g2") for lg in range(28) for n in (1 << lg, (2 << lg) - 1)}


# one awkward size per (curve, c), plus 2^k - 1 / 2^k around window changes that also change the reduction path:
# G1 1023 / 1024 (GLV on), 8191 / 8192 and G2 8191 / 8192 (c = 10 vs 11 / 9 vs 10: level-by-level reduction vs tail
# sums), G1 2^17 - 1 / 2^17 and G2 2^18 - 1 / 2^18 (two vs four tail slices), G1 2^18 - 1 / 2^18 and G2 2^19 - 1 / 2^19
# (four vs eight tail slices)
SIZES = [("g1", n) for n in (45, 63, 64, 101, 127, 128, 200, 389, 511, 512, 777, 1023, 1024, 1500, 3001, 6007, 8191, 8192,
                             12289, 20011, 45013, 99991, 131071, 131072, 143417, 262143, 262144, 300007)] + \
        [("g2", n) for n in (50, 99, 201, 333, 700, 1500, 3000, 6001, 8191, 8192, 12007, 30001, 50021, 100003, 140001,
                             262143, 262144, 270001, 524287, 524288, 600001)]


def _truncate(v: int) -> int:
    """v cut to 254 bits and, if still >= r, to 253: a canonical scalar that keeps most of the pattern."""
    v &= (1 << 254) - 1
    return v - (1 << 253) if v >= R else v


def digit_scalars(rng: random.Random, c: int):
    """Scalars whose every c-bit chunk is 2^(c-1) (the largest positive signed digit), 2^(c-1) + 1 (the smallest negative
    one: a carry into the next window) or 2^c - 1 (digit -1 and a carry), whole and cut to 126 bits (for G1, a scalar
    below ~2^126 is its own GLV half k1, so the pattern reaches the 128-bit windows intact)."""
    ds = (1 << (c - 1), (1 << (c - 1)) + 1, (1 << c) - 1)
    chunks = -(-256 // c)
    pats = [sum(d << (c * j) for j in range(chunks)) for d in ds]
    pats += [sum(rng.choice(ds) << (c * j) for j in range(chunks)) for _ in range(3)]
    return [_truncate(v) for v in pats] + [v & ((1 << 126) - 1) for v in pats]


def special_scalars(rng: random.Random):
    return ([0, 1, 2, R - 1, R - 2, (R - 1) // 2, (R + 1) // 2, 2**253, 2**127 - 1, 2**127, 2**127 + 1, 2**128, 2**64 - 1,
             2**64, LAM, R - LAM, A1, A2, R - A2] + [rng.randrange(1 << 64) for _ in range(6)] + [rng.randrange(1 << 16) for _ in range(2)])


def recipe(rng: random.Random, n: int, c: int, run: int):
    """Overrides [(index, k, s)] of a uniform (k_i, s_i) input: every special and digit-boundary scalar once, three points at
    infinity (k = 0), three P / -P pairs with equal scalars, and `run` copies of one (point, scalar) entry, which land in one
    bucket of every window.  Features are cut short on small inputs so that a quarter of the entries stay uniform."""
    feats = [(rng.randrange(1, R), s) for s in special_scalars(rng) + digit_scalars(rng, c)]
    feats += [(0, rng.randrange(R)) for _ in range(3)]
    for _ in range(3):
        k, s = rng.randrange(1, R), rng.randrange(R)
        feats += [(k, s), (R - k, s)]
    budget = n - n // 4
    feats = feats[:budget]
    k, s = rng.randrange(1, R), rng.randrange(R)
    feats += [(k, s)] * max(0, min(run, n // 4, budget - len(feats)))
    pos = rng.sample(range(n), len(feats))
    return [(i, k, s) for i, (k, s) in zip(pos, feats)]


def heavy_run(curve: str, n: int) -> int:
    """A run longer than the cap and than two segments: heavy path, one bucket cut into three segments."""
    cap, seg = heavy_shape(curve, n)
    return 2 * max(cap, seg) + 1


def make_case(seed: int, curve: str, n: int):
    rng = random.Random(seed)
    c, _ = window(curve, n)
    ks = [rng.randrange(1, R) for _ in range(n)]
    ss = [rng.randrange(R) for _ in range(n)]
    for i, k, s in recipe(rng, n, c, heavy_run(curve, n)):
        ks[i], ss[i] = k, s
    return ks, ss


def linear_expected(curve: str, ks, ss) -> bytes:
    return FIXED_MUL[curve](GEN[curve], cport.frs([sum(k * s for k, s in zip(ks, ss)) % R]))


def dot_mod_r(k: np.ndarray, s: np.ndarray) -> int:
    """sum_i k_i s_i mod r of two (n, 32) uint8 arrays of little-endian scalars, exactly: 16-bit limbs in float64, one
    16 x 16 matrix product per block of 2^20 rows.  Every entry (and every partial sum) of a block's product is an
    integer below 2^20 (2^16 - 1)^2 < 2^52, so float64 holds it exactly whatever order the BLAS adds in."""
    total, blk = 0, 1 << 20
    for lo in range(0, len(k), blk):
        a = np.ascontiguousarray(k[lo:lo + blk]).view("<u2").astype(np.float64)
        b = np.ascontiguousarray(s[lo:lo + blk]).view("<u2").astype(np.float64)
        m = a.T @ b
        total += sum(int(m[i, j]) << (16 * (i + j)) for i in range(16) for j in range(16))
    return total % R


# ---- the rule and the oracles themselves (no GPU) ------------------------------------------------------------------

def test_sizes_cover_every_window():
    """The size list reaches every (curve, c, glv) the rule can produce, so a change of the rule cannot drop a window size
    from this file unnoticed."""
    got = {(cv,) + window(cv, n) for cv, n in SIZES}
    assert reachable() <= got, sorted(reachable() - got)
    assert {c for cv, c, _ in got if cv == "g1"} == {2, 3, 4, 5, 6} | set(range(8, 17))
    assert {c for cv, c, _ in got if cv == "g2"} == set(range(2, 17))
    assert window("g1", 1023) == (6, False) and window("g1", 1024) == (8, True)
    assert window("g1", 1 << 17) == (15, True) and window("g2", 1 << 19) == (16, False)
    # the window counts that use up all 255 (or 128 GLV) bits exactly are among them
    assert {c for cv, c, glv in got if not glv and 255 % c == 0} == {3, 5, 15}
    assert {c for cv, c, glv in got if glv and 128 % c == 0} == {8, 16}


def test_dot_mod_r_matches_python_integers():
    rng = np.random.default_rng(3)
    n = (1 << 20) + 4097                                   # two blocks, the second partial
    k = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    s = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    k[:, 31] &= 0x1F
    s[:5] = 0xFF; s[:5, 31] = 0x1F                        # top of the 253-bit range
    k[5:9] = 0
    ki = [int.from_bytes(k[i].tobytes(), "little") for i in range(n)]
    si = [int.from_bytes(s[i].tobytes(), "little") for i in range(n)]
    assert dot_mod_r(k, s) == sum(a * b for a, b in zip(ki, si)) % R


@pytest.mark.parametrize("curve,n", [("g1", 3000), ("g2", 1 << 14)])
def test_linear_oracle_agrees_with_cport(curve, n):
    """On identical inputs (the full recipe: infinity, P / -P, the heavy run) the linear-combination oracle and the C MSM
    give the same bytes."""
    ks, ss = make_case(11, curve, n)
    pts = FIXED_MUL[curve](GEN[curve], cport.frs(ks))
    assert CPU_MSM[curve](pts, cport.frs(ss)) == linear_expected(curve, ks, ss)


# ---- the CUDA MSM ----------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("curve,n", SIZES, ids=[f"{cv}-n{n}-c{window(cv, n)[0]}" for cv, n in SIZES])
def test_msm_every_window(ctx, curve, n):
    ks, ss = make_case(1000 + n, curve, n)
    msm = ctx.msm_g1 if curve == "g1" else ctx.msm_g2
    sc = cport.frs(ss)
    if n <= CPORT_MAX:
        pts = FIXED_MUL[curve](GEN[curve], cport.frs(ks))
        assert msm(pts, sc) == CPU_MSM[curve](pts, sc)
        return
    gen = ctx.g1_generator_mul if curve == "g1" else ctx.g2_generator_mul
    pts = gen(cport.frs(ks))
    pb = PB[curve]
    rng = random.Random(n)
    sample = rng.sample(range(n), 48) + [i for i in range(n) if ks[i] == 0][:3]
    assert b"".join(pts[pb * i:pb * i + pb] for i in sample) == FIXED_MUL[curve](GEN[curve], cport.frs([ks[i] for i in sample]))
    assert msm(pts, sc) == linear_expected(curve, ks, ss)
    if curve == "g2":
        # one scalar everywhere: one non-empty bucket per window, the tail sums mostly infinity
        s = ss[rng.randrange(n)]
        assert msm(pts, cport.frs([s]) * n) == FIXED_MUL[curve](GEN[curve], cport.frs([sum(ks) * s % R]))


@pytest.mark.gpu
def test_msm_2_24_g1_g2_on_device(ctx):
    """BASELINE config 5 on one GPU: a 2^24-point G1 and G2 MSM over shared scalars, inputs made and kept on the device
    (og_g*_generator_mul_dev, og_msm_g*_dev), against the linear-combination oracle.  Both curves run at c = 16."""
    import torch
    n = 1 << 24
    assert window("g1", n) == (16, True) and window("g2", n) == (16, False)
    g = np.random.default_rng(24)
    k = g.integers(0, 256, (n, 32), dtype=np.uint8)
    s = g.integers(0, 256, (n, 32), dtype=np.uint8)
    k[:, 31] &= 0x1F                                       # < 2^253 < r
    s[:, 31] &= 0x1F
    rng = random.Random(24)
    over = recipe(rng, n, 16, max(heavy_run("g1", n), heavy_run("g2", n)))
    for i, ki, si in over:
        k[i] = np.frombuffer(bn.fr_to_bytes(ki), dtype=np.uint8)
        s[i] = np.frombuffer(bn.fr_to_bytes(si), dtype=np.uint8)
    exp_d = dot_mod_r(k, s)

    L = api.lib()
    dev = torch.device("cuda", ctx.device)
    kd = torch.from_numpy(k.reshape(-1)).to(dev)
    sd = torch.from_numpy(s.reshape(-1)).to(dev)
    p1 = torch.empty(64 * n, dtype=torch.uint8, device=dev)
    p2 = torch.empty(128 * n, dtype=torch.uint8, device=dev)
    o1 = torch.empty(64, dtype=torch.uint8, device=dev)
    o2 = torch.empty(128, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    api._check(L.og_g1_generator_mul_dev(ctx._h, kd.data_ptr(), n, p1.data_ptr()), ctx)
    api._check(L.og_g2_generator_mul_dev(ctx._h, kd.data_ptr(), n, p2.data_ptr()), ctx)
    api._check(L.og_msm_g1_dev(ctx._h, p1.data_ptr(), sd.data_ptr(), n, o1.data_ptr()), ctx)
    api._check(L.og_msm_g2_dev(ctx._h, p2.data_ptr(), sd.data_ptr(), n, o2.data_ptr()), ctx)
    ctx.sync()
    got1, got2 = o1.cpu().numpy().tobytes(), o2.cpu().numpy().tobytes()
    sample = sorted(rng.sample(range(n), 48) + [i for i, ki, _ in over if ki == 0] + [i for i, _, _ in over[:8]])
    idx = torch.tensor(sample, dtype=torch.long, device=dev)
    sp1 = p1.view(n, 64).index_select(0, idx).cpu().numpy().tobytes()
    sp2 = p2.view(n, 128).index_select(0, idx).cpu().numpy().tobytes()
    del kd, sd, p1, p2, idx
    torch.cuda.empty_cache()
    ks = b"".join(k[i].tobytes() for i in sample)
    assert sp1 == cport.g1_fixed_mul_batch(GEN["g1"], ks)
    assert sp2 == cport.g2_fixed_mul_batch(GEN["g2"], ks)
    assert got1 == cport.g1_fixed_mul_batch(GEN["g1"], cport.frs([exp_d]))
    assert got2 == cport.g2_fixed_mul_batch(GEN["g2"], cport.frs([exp_d]))
