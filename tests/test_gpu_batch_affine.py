"""GPU: the batched-affine rounds in front of the bucket accumulation (msm_pair.cuh) against the CPU oracle, bit-exact.
Registered 2^16-point sets use the precomputed window tables (about 34 entries per bucket, 1.1 M entries): the rounds
are the default for BN254 G2 there, and every group is also run with the rounds forced (sb_set_tuning(4, 2)) and off
(4, 1).  Inputs cover bases at infinity, equal points with equal scalars (P + P in several rounds), P and -P in one
bucket and witness-like scalars (one giant bucket)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import oracle as O  # noqa: E402  (checker only)

BN, BLS = O.BN254, O.BLS12_381
N = 1 << 16


@pytest.fixture(scope="module")
def curves():
    import snarkjs_b200
    cs = {BN: snarkjs_b200.getCurveFromName("bn128"), BLS: snarkjs_b200.getCurveFromName("bls12381")}
    yield cs
    for c in cs.values():
        c.terminate()


def _special_bases(cid, grp, seed, n):
    """Oracle points with bases at infinity and one P / -P pair (indices 600, 601)."""
    ci = O.CURVES[cid]
    fb = len(ci.fq_to_mont(1)) * (1 if grp == 1 else 2)            # bytes of one coordinate
    b = O.gen_points(cid, grp, seed, n).reshape(n, 2 * fb).copy()
    b[3] = 0; b[4] = 0; b[9000] = 0
    b[601] = b[600]
    if grp == 1:
        b[601, fb:] = np.frombuffer(ci.fq_to_mont((ci.q - ci.fq_from_mont(b[600, fb:].tobytes())) % ci.q), np.uint8)
    else:
        h = fb // 2
        for k in range(2):
            y = b[600, fb + k * h:fb + (k + 1) * h].tobytes()
            b[601, fb + k * h:fb + (k + 1) * h] = np.frombuffer(ci.fq_to_mont((ci.q - ci.fq_from_mont(y)) % ci.q), np.uint8)
    b[500:540] = b[500]                                             # equal points ...
    return b


def _scalars(cid, seed, n, witness_like):
    sc = O.random_scalars(seed, n, O.CURVES[cid].r).reshape(n, 32).copy()
    sc[500:540] = sc[500]                                           # ... with equal scalars: doublings in every round
    sc[601] = sc[600]                                               # P and -P in the same buckets
    if witness_like:                                                # 50 % zeros, 25 % ones, rest uniform: one giant bucket
        kind = np.random.default_rng(seed).integers(0, 4, n)
        sc[kind < 2] = 0
        sc[kind == 2] = 0
        sc[kind == 2, 0] = 1
    return sc.reshape(-1)


@pytest.mark.parametrize("witness_like", [False, True])
@pytest.mark.parametrize("grp", [1, 2])
@pytest.mark.parametrize("cid", [BN, BLS])
def test_registered_msm_matches_oracle(curves, cid, grp, witness_like):
    c = curves[cid]
    G = c.G1 if grp == 1 else c.G2
    bases = _special_bases(cid, grp, 40 + grp, N).reshape(-1)
    sc = _scalars(cid, 50 + grp, N, witness_like)
    want = O.g_to_affine(cid, grp, O.multiexp_affine(cid, grp, bases, sc))
    h = G.registerBases(bases)
    got = {}
    try:
        for mode in (0, 1, 2):                                      # default, plain XYZZ, rounds forced
            c.lib.sb_set_tuning(4, mode)
            got[mode] = G.toAffine(G.multiExpRegistered(h, sc)).tobytes()
        c.lib.sb_set_tuning(4, 2); c.lib.sb_set_tuning(5, 1)         # one round, the rest through the XYZZ pipeline
        got[3] = G.toAffine(G.multiExpRegistered(h, sc)).tobytes()
    finally:
        c.lib.sb_set_tuning(4, 0); c.lib.sb_set_tuning(5, 0)
    for mode, v in got.items():
        assert v == want, f"mode {mode}"


def test_groth16_padded_c_bases_rounds_forced(curves):
    """Groth16 on a 2^15 chain circuit with every MSM through the rounds, including C, whose bases carry the nPublic+1
    points at infinity of the key layout: the proof bytes are the oracle's."""
    from snarkjs_b200 import groth16, synth
    bn = curves[BN]
    L = 15
    zkey = synth.synth_groth16_zkey(bn, L, seed=12)
    w = synth.chain_witness(bn.r, L)
    wt = synth.wtns_container(bn.r, w)
    ci = O.CURVES[BN]
    r, s = ci.fr_to_mont(5), ci.fr_to_mont(6)
    oproof, opub = O.groth16_prove(zkey, wt, r, s)
    pk = groth16.ProvingKey(zkey, curve=bn)
    bn.lib.sb_set_tuning(4, 2)
    try:
        proof, pub = groth16.prove(pk, wt, r, s)
    finally:
        bn.lib.sb_set_tuning(4, 0)
        pk.release()
    assert proof == oproof and pub == [str(x) for x in opub]
