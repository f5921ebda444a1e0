"""The batched Groth16 prover at every MSM window setting a key can load with, and at every domain size of the withdraw
circuit, bit for bit against the oracle's C prover.

Window bits: `pk_load` (owshen_b200/csrc/groth16.cu) reads OG_WINDOW_BITS (all three MSMs) and OG_C_A / OG_C_B / OG_C_C
(one each), accepts 2..16 and otherwise keeps the defaults 15 / 15 / 16.  The window decides the reduction-level count,
the `max_nb` / `max_windows` scratch sizes and the tiled histogram of every prover MSM, so each setting is a different
set of shapes; a depth-1 key (the golden proof's) keeps each load cheap.
Domain sizes: depths 2, 5 and 12 give log_m = 12, 13 and 14 (the suite also proves at 11 and 15), which is where the
quotient's NTTs -- with the inverse transform's 1/n folded into the coset factors -- change size.
"""
import json
import os
import random

import pytest

import owshen_b200 as ob
from oracle import bn254 as bn
from oracle import cport
from oracle import withdraw_circuit as wc
from tests.helpers import pk_blob, rand_inputs, vk_blob

pytestmark = pytest.mark.gpu
R = bn.R
WINDOW_VARS = ("OG_WINDOW_BITS", "OG_C_A", "OG_C_B", "OG_C_C")


@pytest.fixture(autouse=True)
def _no_window_settings(monkeypatch):
    """Whatever the caller's environment holds, every key here loads with the settings the test sets itself."""
    for v in WINDOW_VARS:
        monkeypatch.delenv(v, raising=False)


def _cat(b: bytes, w: int, idx):
    return b"".join(b[w * i:w * i + w] for i in idx)


@pytest.fixture(scope="module")
def depth1(ctx):
    """Depth-1 key from the golden toxic values, a batch of five (three random inputs, then two copies of the first with
    the same r, s) and the oracle's proofs of it."""
    gold = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "vectors.json")))["groth16"]
    assert gold["depth"] == 1
    tw = [int(x) for x in gold["toxic"]]
    pk, vk = ob.setup_withdraw(ctx, 1, *tw)
    cs = wc.build_r1cs(1)
    pkb, _ = cport.setup_bytes(cs, *tw)
    rng = random.Random(151)
    nul, sec, rec, sib, bits = rand_inputs(rng, 3, 1)
    rs = cport.frs([rng.randrange(R) for _ in range(6)])
    idx = [0, 1, 2, 0, 0]
    inputs = (_cat(nul, 32, idx), _cat(sec, 32, idx), _cat(rec, 32, idx), _cat(sib, 32, idx), [bits[i] for i in idx], _cat(rs, 64, idx))
    wit = cport.withdraw_witness(*inputs[:5], 1)
    expected = cport.Prover(cs, pkb).prove_batch(wit, inputs[5])
    return pk, vk, inputs, expected


def _prove_fresh_key(ctx, pk: bytes, inputs) -> bytes:
    PK = ob.ProvingKey(ctx, pk)
    try:
        return ob.prove(PK, *inputs)[0]
    finally:
        PK.close()


def test_default_windows_match_oracle(ctx, depth1):
    pk, vk, inputs, expected = depth1
    PK = ob.ProvingKey(ctx, pk)
    proofs, pub = ob.prove(PK, *inputs)
    PK.close()
    assert proofs == expected
    assert proofs[:256] == proofs[768:1024] == proofs[1024:1280]
    assert len({proofs[256 * i:256 * i + 256] for i in range(3)}) == 3
    for i in range(5):
        assert ob.verify(vk, pub[96 * i:96 * i + 96], proofs[256 * i:256 * i + 256]), i


@pytest.mark.parametrize("c", range(2, 17))
def test_window_bits_every_c(ctx, depth1, monkeypatch, c):
    pk, _, inputs, expected = depth1
    monkeypatch.setenv("OG_WINDOW_BITS", str(c))
    assert _prove_fresh_key(ctx, pk, inputs) == expected


@pytest.mark.parametrize("a,b,c", [(2, 16, 9), (16, 3, 2)])
def test_window_bits_mixed(ctx, depth1, monkeypatch, a, b, c):
    """Different windows per MSM: the shared scratch is sized by the largest bucket count of one MSM and the largest window
    count of another."""
    pk, _, inputs, expected = depth1
    monkeypatch.setenv("OG_C_A", str(a))
    monkeypatch.setenv("OG_C_B", str(b))
    monkeypatch.setenv("OG_C_C", str(c))
    assert _prove_fresh_key(ctx, pk, inputs) == expected


@pytest.mark.parametrize("var", ["OG_WINDOW_BITS", "OG_C_C"])
@pytest.mark.parametrize("value", ["0", "1", "17", "x"])
def test_window_bits_invalid_fall_back(ctx, depth1, monkeypatch, var, value):
    pk, _, inputs, expected = depth1
    monkeypatch.setenv(var, value)
    assert _prove_fresh_key(ctx, pk, inputs) == expected


@pytest.mark.parametrize("depth,log_m", [(2, 12), (5, 13), (12, 14)])
def test_prover_every_domain_size(ctx, monkeypatch, depth, log_m):
    """Setup, the quotient evaluations and a batch proved in two chunks, at one depth per domain size."""
    rng = random.Random(7000 + depth)
    tw = [rng.randrange(1, R) for _ in range(5)]
    pk, vk = ob.setup_withdraw(ctx, depth, *tw)
    cs = wc.build_r1cs(depth)
    pkb, vkb = cport.setup_bytes(cs, *tw)
    assert vk == vk_blob(vkb)
    assert pk == pk_blob(cs, pkb, depth)
    PK = ob.ProvingKey(ctx, pk)
    try:
        assert (PK.depth, PK.log_m, PK.n_vars) == (depth, log_m, cs.n_vars)
        batch, nv = 3, cs.n_vars
        nul, sec, rec, sib, bits = rand_inputs(rng, batch, depth)
        rs = cport.frs([rng.randrange(R) for _ in range(2 * batch)])
        wit = cport.withdraw_witness(nul, sec, rec, sib, bits, depth)
        opr = cport.Prover(cs, pkb)
        assert PK.h_evals(wit[:32 * nv]) == opr.h_evals(wit[:32 * nv])
        monkeypatch.setenv("OG_CHUNK", "2")               # a chunk of two proofs, then one of one
        proofs, pub = ob.prove(PK, nul, sec, rec, sib, bits, rs)
    finally:
        PK.close()
    assert proofs == opr.prove_batch(wit, rs)
    for i in range(batch):
        x, p = pub[96 * i:96 * i + 96], proofs[256 * i:256 * i + 256]
        assert x == wit[32 * nv * i + 32:32 * nv * i + 128]
        assert ob.verify(vk, x, p), i
        bad = bytearray(x)
        bad[33] ^= 1
        assert not ob.verify(vk, bytes(bad), p), i
