"""CPU: the restated halo2 prover/verifier (oracle/halo2.py) round-trips and rejects tampering -- the shape of the
reference's own `production` tests (/root/reference/src/circuits/shot.rs:880-941, board.rs:879-933)."""
import pytest
from tests.util_prover import Job, tiny_circuit


@pytest.fixture(scope="module")
def tiny():
    return Job(*tiny_circuit(5))


def test_roundtrip_tiny(tiny):
    proof = tiny.oracle_proof()
    assert tiny.verify(proof)
    assert tiny.oracle_proof() == proof                       # deterministic under the seeded RNG
    assert tiny.oracle_proof(index=1) != proof


def test_tamper_rejected(tiny):
    proof = bytearray(tiny.oracle_proof())
    for pos in (5, 40, len(proof) // 2, len(proof) - 1):
        bad = bytearray(proof); bad[pos] ^= 1
        assert not tiny.verify(bytes(bad))
    assert not tiny.verify(bytes(proof), instances=[[12]])
    assert not tiny.verify(bytes(proof[:-32]))


def test_unsatisfied_witness_does_not_verify(tiny):
    adv = tiny.advice.copy()
    adv[2, 0] = tiny.V.m(13)                                   # 3 * 4 != 13 and breaks the copy to the constant 12
    assert not tiny.verify(tiny.oracle_proof(advice=adv))


def test_lookup_failure_is_an_error(tiny):
    adv = tiny.advice.copy()
    adv[0, 0] = tiny.V.m(1000)                                 # not in the 16-row table
    with pytest.raises(ValueError):
        tiny.oracle_proof(advice=adv)


def test_shot_circuit_shape_and_roundtrip():
    """Shot mirror: 24 gates, 13 permutation columns, degree 9, bf 5, 4238 RNG draws (SURVEY App. A / C)."""
    from battlezips_halo2_b200.circuits import shot_circuit
    cs, cfg, asg = shot_circuit(0)
    assert len(cs.gates) == 24 and cs.degree() == 9 and cs.blinding_factors() == 5
    assert len(cs.permutation) == 13 and cs.num_advice == 11 and len(cs.lookups) == 1
    assert asg.check_satisfied() is None
    job = Job(cs, asg)
    assert job.num_random() == 4238
    proof = job.oracle_proof()
    assert len(proof) == 4000
    assert job.verify(proof)
    bad = bytearray(proof); bad[100] ^= 0x10
    assert not job.verify(bytes(bad))


def test_board_circuit_shape():
    from battlezips_halo2_b200.circuits import board_circuit
    cs, cfg, asg = board_circuit(0)
    assert len(cs.gates) == 57 and cs.degree() == 9 and len(cs.permutation) == 13 and cs.num_advice == 11
    assert cs.blinding_factors() == 7
    assert asg.check_satisfied() is None


def test_oracle_reproduces_committed_golden_proofs(tiny):
    """tests/golden/proofs.npz (made by tests/golden/make_proofs.py) freezes the oracle's proof bytes: any drift in the
    restated protocol order, RNG draw order or transcript shows up here, on the CPU, before a GPU run is spent."""
    import os
    import numpy as np
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proofs.npz"))
    assert tiny.oracle_proof(index=0) == bytes(gold["tiny_k5_idx0"])
    assert tiny.oracle_proof(index=3) == bytes(gold["tiny_k5_idx3"])
    from battlezips_halo2_b200.circuits import shot_circuit
    cs, _, asg = shot_circuit(0)
    job = Job(cs, asg)
    proof = job.oracle_proof(index=0)
    assert proof == bytes(gold["shot_w0_idx0"]) and job.verify(proof)


def test_oracle_batch_invert_assigned_is_division():
    """The restated poly::batch_invert_assigned equals numerator / denominator (0 for a zero denominator) in big integers."""
    import random
    from oracle import c_oracle as co, halo2 as H
    from oracle.vec import Vec
    for f in (0, 1):
        F = co.FIELDS[f]
        p, rnd = F.p, random.Random(f)
        num = [rnd.randrange(p) for _ in range(200)]
        den = [rnd.choice([0, 1, 2, p - 1, rnd.randrange(p)]) for _ in range(200)]
        got = H.batch_invert_assigned(Vec(f), co.to_mont(f, num), co.to_mont(f, den))
        assert co.from_mont(f, got) == [x * F.inv(d) % p for x, d in zip(num, den)]


def _check_permuted_pair(V, usable, cin, ctab, a, s):
    """halo2's invariants of permute_expression_pair on the usable rows, in canonical integers."""
    ai, si = V.ints(a), V.ints(s)
    assert len(ai) == len(si) == usable
    assert ai == sorted(V.ints(cin[:usable]))                        # A' is the input sorted by canonical value
    assert sorted(si) == sorted(V.ints(ctab[:usable]))              # S' is a permutation of the table's usable rows
    for i in range(usable):
        if i == 0 or ai[i] != ai[i - 1]:
            assert ai[i] == si[i], i                                 # A'[i] == S'[i] at the start of every run


def test_oracle_permute_expression_pair_invariants():
    """The restated lookup permute_expression_pair, used as the reference of the device kernels, holds halo2's invariants
    on hand-made and random columns (repeated inputs, duplicate-heavy tables, 0 and p - 1, usable < n), and an input
    value found only in the table's unusable rows raises."""
    import random
    from oracle import halo2 as H
    from oracle.vec import Vec
    V = Vec(0)
    p = V.p
    cases = [
        (8, 8, [3, 3, 3, 3, 3, 3, 3, 3], [3, 1, 2, 0, 7, 5, 4, 6]),
        (8, 6, [0, p - 1, 0, p - 1, 5, 5, 9, 9], [p - 1, 5, 0, 5, 5, 0, 9, 9]),
        (8, 7, [4, 2, 4, 2, 4, 2, 4, 1], [2, 2, 2, 4, 4, 1, 1, 8]),
        (4, 4, [1, 2, 3, 0], [0, 3, 2, 1]),
        (4, 0, [1, 2, 3, 0], [7, 7, 7, 7]),
    ]
    rnd = random.Random(7)
    for n in (16, 64, 256):
        for _ in range(6):
            usable = rnd.choice([n, n - 1, n - 10, rnd.randrange(1, n)])
            distinct = [rnd.choice([0, p - 1, rnd.randrange(p)]) for _ in range(rnd.choice([1, 3, n // 4]))]
            table = [rnd.choice(distinct) for _ in range(n)]
            inputs = [rnd.choice(table[:usable]) for _ in range(n)]
            cases.append((n, usable, inputs, table))
    for n, usable, inputs, table in cases:
        cin, ctab = V.arr(inputs), V.arr(table)
        a, s = H.permute_expression_pair(V, usable, cin, ctab)
        _check_permuted_pair(V, usable, cin, ctab, a, s)
    cin, ctab = V.arr([5, 1, 2, 2]), V.arr([1, 2, 3, 5])
    with pytest.raises(ValueError, match="ConstraintSystemFailure"):
        H.permute_expression_pair(V, 3, cin, ctab)                    # 5 is only in table row 3 >= usable
    H.permute_expression_pair(V, 3, V.arr([1, 2, 2, 9]), ctab)        # 9 only in input row 3 >= usable: fine


def test_oracle_grand_products_match_integer_formula():
    """The restated permutation and lookup grand products against the formula in Python integers, on both fields, with a
    zero numerator and zero denominators: halo2's batch_invert leaves a zero denominator's inverse at zero, so z is
    non-zero up to that row and zero after it."""
    import random
    from oracle import halo2 as H
    from oracle.vec import Vec
    for f in (0, 1):
        V = Vec(f)
        p, delta, rnd = V.p, V.F.delta, random.Random(f)
        n, omega = 16, pow(V.F.root_of_unity, 1 << 28, V.p)
        beta, gamma, d0, z0 = (rnd.randrange(p) for _ in range(4))
        for kind, row in (("num", 3), ("den", 0), ("den", 9), ("den", n - 1)):
            vals = [[rnd.randrange(p) for _ in range(n)] for _ in range(2)]
            sig = [[rnd.randrange(p) for _ in range(n)] for _ in range(2)]
            if kind == "num":
                vals[0][row] = -(beta * d0 * pow(omega, row, p) + gamma) % p
            else:
                vals[1][row] = -(beta * sig[1][row] + gamma) % p
            z = V.ints(H.permutation_product(V, omega, [V.arr(c) for c in vals], [V.arr(c) for c in sig], beta, gamma, d0, z0))
            exp = [z0]
            for i in range(n - 1):
                num = den = 1
                for j in range(2):
                    num = num * (vals[j][i] + beta * d0 * pow(delta, j, p) * pow(omega, i, p) + gamma) % p
                    den = den * (vals[j][i] + beta * sig[j][i] + gamma) % p
                exp.append(exp[-1] * num * (pow(den, -1, p) if den else 0) % p)
            assert z == exp and all(z[:row + 1]) and not any(z[row + 1:]), (kind, row)
        cols = [[rnd.randrange(p) for _ in range(n)] for _ in range(4)]
        cols[3][5] = -gamma % p                                                   # denominator zero at row 5
        z = V.ints(H.lookup_product(V, *[V.arr(c) for c in cols], beta, gamma))
        exp = [1]
        for i in range(n - 1):
            den = (cols[2][i] + beta) * (cols[3][i] + gamma) % p
            exp.append(exp[-1] * (cols[0][i] + beta) * (cols[1][i] + gamma) * (pow(den, -1, p) if den else 0) % p)
        assert z == exp and all(z[:6]) and not any(z[6:])
