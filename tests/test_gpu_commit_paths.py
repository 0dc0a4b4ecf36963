"""Both ways a Params commits -- the fixed-base window tables (k <= 19) and the bucket MSM over the raw bases (k >= 20, or
Params built with BZ_FORCE_GENERAL_MSM=1) -- through every entry point that commits over a Params basis: Params.commit,
keygen_vk's commitments, the round-by-round IPA and the verifier (its instance commitments and the fixed-base part of its
final check).  Points are compared with the oracle bit for bit, verdicts with the oracle verifier."""
import random
import numpy as np
import pytest
from tests.util_msm import modulus, oracle_msms, urs_points
from tests.util_prover import Job, VK_REPR, tiny_circuit

pytestmark = pytest.mark.gpu

PATHS = ["tables", "bucket"]


def _params(ctx, path, k, g, gl, w, u, curve=0):
    """Params on the requested path; the switch is read by bz_params_create only."""
    from battlezips_halo2_b200.plonk import prover as PR
    with pytest.MonkeyPatch.context() as mp:
        if path == "bucket":
            mp.setenv("BZ_FORCE_GENERAL_MSM", "1")
        return PR.Params(ctx, k, g, gl, w, u, curve=curve, window_bits=8)


@pytest.fixture(scope="module")
def tiny():
    """The tiny circuit's job and the oracle's trace of one proof (the IPA rounds' L_j, R_j and c)."""
    job = Job(*tiny_circuit(5))
    tr = {}
    job.oracle_proof(index=5, trace=tr)
    return job, tr


@pytest.fixture(params=PATHS)
def keys(request, ctx, tiny):
    from battlezips_halo2_b200.plonk import prover as PR
    job, _ = tiny
    op = job.oparams
    params = _params(ctx, request.param, job.k, op.g, op.g_lagrange, op.w, op.u)
    pk = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR)
    yield job, params, pk
    pk.close(); params.close()


@pytest.mark.parametrize("curve", [0, 1])
@pytest.mark.parametrize("path", PATHS)
def test_params_commit(path, curve, ctx, oracle_c):
    """Params.commit over g || w and g_lagrange || w, k = 5: random, zero, single-term and all r - 1 polynomials with blinds
    0, 1, r - 1 and random."""
    co = oracle_c
    k, n = 5, 32
    urs = urs_points(ctx, co, curve, 2 * n + 2)
    g, w, u, gl = urs[:n], urs[n], urs[n + 1], urs[n + 2:]
    sf = co.CURVES[curve][1]
    r = modulus(sf)
    rng = random.Random(7 + curve)
    polys = [[rng.randrange(r) for _ in range(n)], [0] * n, [0] * 5 + [rng.randrange(r)] + [0] * (n - 6), [r - 1] * n]
    blinds = [rng.randrange(r), 0, 1, r - 1, 0]
    cases = [(polys[i % len(polys)], blinds[i]) for i in range(len(blinds))]
    params = _params(ctx, path, k, g, gl, w, u, curve=curve)
    try:
        for lagrange in (False, True):
            bases = np.concatenate([gl if lagrange else g, w[None]])
            exp = oracle_msms(co, curve, [(co.to_mont(sf, p + [b]), bases) for p, b in cases])
            for (p, b), e in zip(cases, exp):
                got = params.commit(co.to_mont(sf, p), co.to_mont(sf, [b])[0], lagrange=lagrange)
                assert np.array_equal(got, e), (path, curve, lagrange, b)
    finally:
        params.close()


def test_vk_commitments(keys, oracle_c):
    job, params, pk = keys
    fc, pc = pk.vk_commitments()
    assert np.array_equal(fc, oracle_c.points_to_mont(0, job.opk.fixed_commitments))
    assert np.array_equal(pc, oracle_c.points_to_mont(0, job.opk.perm_commitments))


@pytest.mark.parametrize("path", PATHS)
def test_ipa_rounds(path, ctx, tiny, oracle_c):
    job, tr = tiny
    V, ipa, op = job.V, tr["ipa"], job.oparams
    rounds = [(V.m(r["l_rand"]), V.m(r["r_rand"]), (lambda L, R, u=r["u"]: (V.m(u), V.m(pow(u, -1, V.p))))) for r in ipa["rounds"]]
    params = _params(ctx, path, job.k, op.g, op.g_lagrange, op.w, op.u)
    try:
        got, c = params.ipa_open(ipa["p_prime"], V.m(ipa["x3"]), V.m(ipa["z"]), rounds)
    finally:
        params.close()
    for (L, R), r in zip(got, ipa["rounds"]):
        assert oracle_c.points_from_mont(0, np.stack([L, R])) == [r["L"], r["R"]]
    assert V.int1(c) == ipa["c"]


def _flip(proof, byte, bit=0):
    b = bytearray(proof)
    b[byte] ^= 1 << bit
    return bytes(b)


def test_verify_proofs(keys):
    """One batch of six proofs: three good ones, one with the IPA scalar c and one with the blind f changed by one bit (both
    still canonical, so only the final check can reject them), and a good one with a wrong instance; then a truncated proof."""
    from battlezips_halo2_b200.plonk import prover as PR
    job, params, pk = keys
    good = PR.create_proofs(pk, [job.instances] * 3, np.stack([job.advice] * 3), np.stack([job.wide(i) for i in range(3)]))
    assert good == [job.oracle_proof(index=i) for i in range(3)]
    plen = len(good[0])
    proofs = good + [_flip(good[0], plen - 64), _flip(good[1], plen - 32), good[2]]
    instances = [job.instances] * 5 + [[[12]]]
    got = PR.verify_proofs(pk, instances, proofs)
    assert got == [job.verify(p, instances=i) for p, i in zip(proofs, instances)]
    assert got == [True, True, True, False, False, False]
    assert PR.verify_proofs(pk, [job.instances], [good[0][:-32]]) == [False]
