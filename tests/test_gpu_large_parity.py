"""GPU parity at the sizes bench.py and DESIGN.md quote (VERDICT r1 item 1a): the general MSM at 2^18 / 2^20 / 2^22 on
Vesta and Pallas with uniform and witness-like scalars, the NTT and the coset extension at 2^22 / 2^24, and the scaled
Board circuit at k = 15 / 16 -- every one compared with the oracle's output on the same inputs, bit for bit.

Bases of the large MSMs are the URS points g[i] = hash_to_curve("Halo2-Parameters")(0 || i_le32) computed on the device
(bz_hash_to_curve; a sample of them is re-derived by the oracle's own hash-to-curve first), so 2^22 distinct points do
not cost minutes of Python curve arithmetic."""
import ctypes
import random
import numpy as np
import pytest
from battlezips_halo2_b200 import arithmetic as ar
from tests.util_msm import urs_points as _urs_points

pytestmark = pytest.mark.gpu


def _scalars(co, curve, n, kind, seed):
    sf = co.CURVES[curve][1]
    rng = np.random.default_rng(seed)
    s = co.from_u512(sf, rng.integers(0, 2**63, size=(n, 8), dtype=np.uint64) * 2 + rng.integers(0, 2, size=(n, 8), dtype=np.uint64))
    if kind == "witness":                       # SURVEY 8d "W": 70 % zero, 20 % one, 5 % below 2^10, 5 % uniform
        u = rng.random(n)
        one = co.to_mont(sf, [1])[0]
        small = co.to_mont(sf, [int(v) for v in rng.integers(2, 1 << 10, size=n)])
        s[u < 0.95] = small[u < 0.95]
        s[u < 0.90] = one
        s[u < 0.70] = 0
    return s


_BASES = {}


@pytest.mark.parametrize("curve,log_n,kind", [(0, 18, "uniform"), (0, 18, "witness"), (1, 18, "uniform"), (1, 18, "witness"),
                                              (0, 20, "uniform"), (1, 20, "witness"), (1, 20, "uniform"), (0, 20, "witness"),
                                              (1, 22, "uniform"), (0, 22, "witness")])
def test_best_multiexp_large_vs_oracle(curve, log_n, kind, ctx, oracle_c):
    co = oracle_c
    n = 1 << log_n
    if curve not in _BASES or len(_BASES[curve]) < n:
        _BASES[curve] = _urs_points(ctx, co, curve, max(n, 1 << 20))
    bases = _BASES[curve][:n]
    sc = _scalars(co, curve, n, kind, seed=log_n * 4 + curve * 2 + (kind == "witness"))
    got = co.to_affine(curve, ar.best_multiexp(ctx, curve, sc, bases))
    exp = co.to_affine(curve, co.best_multiexp(curve, sc, bases))
    assert np.array_equal(got, exp)
    if log_n == 22:
        _BASES.pop(curve, None)


@pytest.mark.parametrize("field,log_n", [(0, 22), (1, 22), (0, 24)])
def test_best_fft_large_vs_oracle(field, log_n, ctx, oracle_c):
    co = oracle_c
    F = co.FIELDS[field]
    n = 1 << log_n
    rng = np.random.default_rng(log_n + field)
    a = co.from_u512(field, rng.integers(0, 2**63, size=(n, 8), dtype=np.uint64))
    om = pow(F.root_of_unity, 1 << (32 - log_n), F.p)
    for w in (om, pow(om, -1, F.p)) if log_n == 22 else (om,):
        wm = co.to_mont(field, [w])
        assert np.array_equal(ar.best_fft(ctx, field, a, wm, log_n), co.best_fft(field, a, wm, log_n))


@pytest.mark.parametrize("k", [19, 21])
def test_coset_extension_large_vs_oracle(k, ctx, oracle_c):
    """coeff_to_extended n -> 8n and extended_to_coeff at 2^22 / 2^24 extended points (degree 9 as Board / Shot)."""
    from oracle.domain import EvaluationDomain
    co = oracle_c
    dom = EvaluationDomain(0, 9, k)
    assert dom.extended_k == k + 3
    rng = np.random.default_rng(k)
    a = co.from_u512(0, rng.integers(0, 2**63, size=(dom.n, 8), dtype=np.uint64))
    ext = ar.coeff_to_extended(ctx, 0, a, k, dom.extended_k)
    assert np.array_equal(ext, dom.coeff_to_extended(a))
    back = ar.extended_to_coeff(ctx, 0, ext, dom.extended_k)
    assert np.array_equal(back[: dom.n], a) and not back[dom.n:].any()
    if k == 19:
        big = co.from_u512(0, rng.integers(0, 2**63, size=(1 << dom.extended_k, 8), dtype=np.uint64))
        got = ar.extended_to_coeff(ctx, 0, big, dom.extended_k)[: dom.n * dom.quotient_poly_degree]
        assert np.array_equal(got, dom.extended_to_coeff(big))


@pytest.mark.parametrize("k,batch", [(15, 1), (16, 1), (16, 2)], ids=["15", "16", "16-batch2"])
def test_scaled_board_proof_bytes_match_oracle(k, batch, ctx):
    """BASELINE config 5 on the way up: the Board circuit tiled down 2^15 / 2^16 rows, proof bytes against the oracle
    prover and accepted by the restated verifier and by verify_proof on the device.  The batch of two (RNG indices 2 and 3
    in one create_proofs call) runs every per-proof launch site of the large-domain paths with B = 2: the two-level
    grand-product scan, the split Horner evaluation and Kate division, the lookup permutation per proof and the split
    IPA inner products."""
    from battlezips_halo2_b200.circuits import board_circuit_scaled
    from battlezips_halo2_b200.plonk import prover as PR
    from tests.util_prover import Job, first_diff
    cs, cfg, asg = board_circuit_scaled(k)
    job = Job(cs, asg, params_from_device=ctx)
    params, pk = job.device_keys(ctx)
    indices = range(2, 2 + batch)
    proofs = PR.create_proofs(pk, [job.instances] * batch, np.stack([job.advice] * batch), np.stack([job.wide(i) for i in indices]))
    for i, proof in zip(indices, proofs):
        exp = job.oracle_proof(index=i)
        assert first_diff(proof, exp) is None, (i, first_diff(proof, exp))
        assert job.verify(proof)
    assert PR.verify_proofs(pk, [job.instances] * batch, proofs) == [True] * batch
    pk.close(); params.close()
