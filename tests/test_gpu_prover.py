"""GPU parity for create_proof through the C ABI: proof bytes identical to the oracle's under the same RNG words, and
every GPU proof accepted by the restated reference verifier (BASELINE.json north_star)."""
import numpy as np
import pytest
from tests.util_prover import Job, tiny_circuit, first_diff

pytestmark = pytest.mark.gpu


def _prove(job, pk, indices):
    from battlezips_halo2_b200.plonk import prover as PR
    B = len(indices)
    advice = np.stack([job.advice] * B)
    wide = np.stack([job.wide(i) for i in indices])
    return PR.create_proofs(pk, [job.instances] * B, advice, wide)


def test_params_commit_parity(ctx, oracle_c):
    co = oracle_c
    job = Job(*tiny_circuit(5))
    params, pk = job.device_keys(ctx)
    rng = np.random.default_rng(0)
    poly = co.from_u512(0, rng.integers(0, 2**63, size=(32, 8), dtype=np.uint64))
    blind = co.from_u512(0, rng.integers(0, 2**63, size=(1, 8), dtype=np.uint64))[0]
    V = job.V
    for lag in (False, True):
        got = params.commit(poly, blind, lagrange=lag)
        exp = (job.oparams.commit_lagrange if lag else job.oparams.commit)(poly, V.int1(blind))
        assert np.array_equal(got, co.to_affine(0, exp)[0])
    pk.close(); params.close()


@pytest.mark.parametrize("window_bits", [4, 9])
def test_tiny_proof_bytes_match_oracle(ctx, window_bits):
    job = Job(*tiny_circuit(5))
    params, pk = job.device_keys(ctx, window_bits=window_bits)
    proofs = _prove(job, pk, [0, 1, 2])
    for i, proof in enumerate(proofs):
        exp = job.oracle_proof(index=i)
        assert first_diff(proof, exp) is None, first_diff(proof, exp)
        assert job.verify(proof)
    pk.close(); params.close()


def test_lookup_failure_maps_to_synthesis_error(ctx):
    import battlezips_halo2_b200 as bz
    from battlezips_halo2_b200.plonk import prover as PR
    job = Job(*tiny_circuit(5))
    params, pk = job.device_keys(ctx, window_bits=4)
    adv = job.advice.copy()
    adv[0, 0] = job.V.m(1000)
    with pytest.raises(bz.BzError) as e:
        PR.create_proofs(pk, [job.instances], adv[None], job.wide(0)[None])
    assert e.value.code == -4
    pk.close(); params.close()


def test_shot_proof_bytes_match_oracle(ctx):
    """BASELINE config 1/3 shape: Shot k=11, batch of 2 proofs with different RNG streams."""
    from battlezips_halo2_b200.circuits import shot_circuit
    cs, cfg, asg = shot_circuit(0)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx)
    assert pk.proof_size == 4000 and pk.num_random == 4238
    proofs = _prove(job, pk, [0, 7])
    for idx, proof in zip([0, 7], proofs):
        exp = job.oracle_proof(index=idx)
        assert first_diff(proof, exp) is None, first_diff(proof, exp)
        assert job.verify(proof)
    pk.close(); params.close()


def test_board_proof_bytes_match_oracle(ctx):
    """BASELINE config 2: Board k=12 single proof, bit-exact bytes, accepted by the restated verifier."""
    from battlezips_halo2_b200.circuits import board_circuit
    cs, cfg, asg = board_circuit(0)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx)
    proof = _prove(job, pk, [0])[0]
    exp = job.oracle_proof(index=0)
    assert first_diff(proof, exp) is None, first_diff(proof, exp)
    assert job.verify(proof)
    pk.close(); params.close()


@pytest.mark.parametrize("force_general", [False, True])
def test_scaled_board_k13_both_commit_paths(ctx, force_general, monkeypatch):
    """BASELINE config 5 in small: the Board circuit tiled down a 2^13-row table (3 boards per proof), proved once with
    the fixed-base window tables and once with the large-n path (bucket MSM over the raw bases, what k >= 15 uses)."""
    from battlezips_halo2_b200.circuits import board_circuit_scaled
    if force_general:
        monkeypatch.setenv("BZ_FORCE_GENERAL_MSM", "1")
    cs, cfg, asg = board_circuit_scaled(13)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx)
    proof = _prove(job, pk, [3])[0]
    exp = job.oracle_proof(index=3)
    assert first_diff(proof, exp) is None, first_diff(proof, exp)
    assert job.verify(proof)
    pk.close(); params.close()


@pytest.mark.parametrize("force_general", [False, True])
@pytest.mark.parametrize("mat_log", [3, 6, 10])
def test_ipa_with_materialised_generators_gives_the_same_proof(ctx, force_general, mat_log, monkeypatch):
    """Large single proofs (k >= 16) materialise the folded generators G' once they are down to 2^10 points and run the late IPA
    rounds on them (prover.cu step 21, msm_multi_run: MSMs with shared scalars).  Forced here on the k = 13 scaled Board at three
    lengths of G', on both commitment paths: the proof bytes must not change."""
    from battlezips_halo2_b200.circuits import board_circuit_scaled
    if force_general:
        monkeypatch.setenv("BZ_FORCE_GENERAL_MSM", "1")
    monkeypatch.setenv("BZ_IPA_MATERIALIZE_LOG", str(mat_log))
    cs, cfg, asg = board_circuit_scaled(13)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx)
    proof = _prove(job, pk, [3])[0]
    exp = job.oracle_proof(index=3)
    assert first_diff(proof, exp) is None, first_diff(proof, exp)
    assert job.verify(proof)
    pk.close(); params.close()


@pytest.mark.parametrize("which", ["tiny", "shot"])
def test_keygen_on_device_matches_oracle(ctx, oracle_c, which):
    """keygen_vk / keygen_pk on the device (SURVEY §8f rank 2; reference call sites /root/reference/benches/shot.rs:60-61):
    fixed and permutation commitments equal the oracle keygen's, and the sigma columns assembled on the device from the
    copy-constraint cycles give the same proof bytes as host-computed sigma values."""
    from battlezips_halo2_b200.plonk import prover as PR
    from tests.util_prover import VK_REPR
    if which == "tiny":
        job = Job(*tiny_circuit(5))
    else:
        from battlezips_halo2_b200.circuits import shot_circuit
        cs, cfg, asg = shot_circuit(1)
        job = Job(cs, asg)
    params, pk = job.device_keys(ctx, window_bits=8)
    fc, pc = pk.vk_commitments()
    assert np.array_equal(fc, oracle_c.points_to_mont(0, job.opk.fixed_commitments))
    assert np.array_equal(pc, oracle_c.points_to_mont(0, job.opk.perm_commitments))
    pk2 = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR, host_sigma=True)
    fc2, pc2 = pk2.vk_commitments()
    assert np.array_equal(fc, fc2) and np.array_equal(pc, pc2)
    a = _prove(job, pk, [2])[0]
    b = _prove(job, pk2, [2])[0]
    assert a == b == job.oracle_proof(index=2)
    pk2.close(); pk.close(); params.close()


def test_lookup_permutation_paths_agree(ctx):
    """permute_expression_pair: the one-CTA kernel (n <= 4096) and the device-wide radix-sort path (n = 8192) give the
    oracle's proof bytes; a lookup input missing from the table is Error::ConstraintSystemFailure."""
    import battlezips_halo2_b200 as bz
    from battlezips_halo2_b200.plonk import prover as PR
    from battlezips_halo2_b200.circuits import board_circuit_scaled
    job = Job(*tiny_circuit(5))
    params, pk = job.device_keys(ctx, window_bits=6)
    assert _prove(job, pk, [4])[0] == job.oracle_proof(index=4)
    pk.close(); params.close()
    cs, cfg, asg = board_circuit_scaled(13)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx)
    dev = _prove(job, pk, [1])[0]
    assert first_diff(dev, job.oracle_proof(index=1)) is None, first_diff(dev, job.oracle_proof(index=1))
    # break the range-check lookup: input = q_lookup * (...advice...), so poison the advice column it reads on the rows
    # where the lookup selector is on (a value far outside the 10-bit table)
    adv = job.advice.copy()
    lk_in = job.ir["lookups"][0]["input"][0]
    assert lk_in[0] == "product" and lk_in[1][0] == "fixed"
    sel_col = lk_in[1][1]

    def first_advice(e):
        if e[0] == "advice":
            return e[1]
        for sub in e[1:]:
            if isinstance(sub, list):
                r = first_advice(sub)
                if r is not None:
                    return r
        return None
    col = first_advice(lk_in)
    rows = [r for r, v in enumerate(job.asg.fixed[sel_col]) if v][:4]
    assert rows
    for r in rows:
        adv[col, r] = job.V.m(123456789)
    with pytest.raises(bz.BzError) as e:
        PR.create_proofs(pk, [job.instances], adv[None], job.wide(0)[None])
    assert e.value.code == -4
    pk.close(); params.close()


def test_sanity_checks_flag_catches_broken_copy_constraint(ctx, monkeypatch):
    """halo2_proofs' optional `sanity-checks` feature, here BZ_SANITY_CHECKS: a witness that violates a copy constraint makes
    the permutation grand product miss 1 on the first unusable row -> Error::ConstraintSystemFailure instead of an
    (invalid) proof; a good witness is unaffected."""
    import battlezips_halo2_b200 as bz
    from battlezips_halo2_b200.plonk import prover as PR
    job = Job(*tiny_circuit(5))
    params, pk = job.device_keys(ctx, window_bits=6)
    monkeypatch.setenv("BZ_SANITY_CHECKS", "1")
    assert _prove(job, pk, [0])[0] == job.oracle_proof(index=0)
    adv = job.advice.copy()
    adv[1, 3] = job.V.m(5)                   # b[3] is copy-constrained to b[0] = 4
    with pytest.raises(bz.BzError) as e:
        PR.create_proofs(pk, [job.instances], adv[None], job.wide(0)[None])
    assert e.value.code == -4
    monkeypatch.delenv("BZ_SANITY_CHECKS")
    bad = PR.create_proofs(pk, [job.instances], adv[None], job.wide(0)[None])[0]     # without the flag: a proof that does not verify
    assert PR.verify_proofs(pk, [job.instances], [bad]) == [False]
    pk.close(); params.close()


def test_grand_products_batched_and_sequential_agree(ctx, monkeypatch):
    """All grand products of a batch in lockstep (one scan / finish launch, one shared inversion) and the one-product-at-a-
    time path (what large domains use) write the same proof; both equal the oracle's."""
    from battlezips_halo2_b200.circuits import shot_circuit
    cs, cfg, asg = shot_circuit(3)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx, window_bits=10)
    a = _prove(job, pk, [1, 4])
    monkeypatch.setenv("BZ_GP_SEQUENTIAL", "1")
    b = _prove(job, pk, [1, 4])
    monkeypatch.delenv("BZ_GP_SEQUENTIAL")
    assert a == b
    assert first_diff(a[1], job.oracle_proof(index=4)) is None
    pk.close(); params.close()


@pytest.mark.parametrize("which", ["shot", "board"])
def test_quotient_dag_and_tree_programs_agree(ctx, which, monkeypatch):
    """h(X) compiled as one DAG per tier (shared sub-expressions, hoisted factors: csrc/evalprog.h) and as the
    reference-shaped one-tree-per-polynomial program give the same proof bytes; the DAG costs fewer multiplications."""
    from battlezips_halo2_b200.circuits import shot_circuit, board_circuit
    cs, cfg, asg = (shot_circuit if which == "shot" else board_circuit)(1)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx)
    monkeypatch.setenv("BZ_QUOTIENT_CSE", "0")
    from battlezips_halo2_b200.plonk import prover as PR
    from tests.util_prover import VK_REPR
    pk_tree = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR)       # programs are compiled at pk creation
    monkeypatch.delenv("BZ_QUOTIENT_CSE")
    a, b = _prove(job, pk, [2])[0], _prove(job, pk_tree, [2])[0]
    assert first_diff(a, b) is None, first_diff(a, b)
    assert job.verify(a)
    cost = lambda k: sum(m * p for m, p in k.quotient_muls)
    assert cost(pk) < cost(pk_tree), (pk.quotient_muls, pk_tree.quotient_muls)
    print(which, "multiplications per proof in h(X): DAG", cost(pk), "tree", cost(pk_tree), pk.quotient_muls, pk_tree.quotient_muls)
    pk_tree.close(); pk.close(); params.close()


@pytest.mark.parametrize("which", ["shot", "board"])
def test_generated_quotient_matches_interpreter(ctx, which, monkeypatch):
    """h(X) as generated straight-line code (csrc/gen_quotient.cu) and through the interpreter: same proof bytes; the Shot and
    Board keys do pick the generated kernels, other circuits (the tiny one) run the interpreter."""
    from battlezips_halo2_b200.circuits import shot_circuit, board_circuit
    from battlezips_halo2_b200.plonk import prover as PR
    from tests.util_prover import VK_REPR
    cs, cfg, asg = (shot_circuit if which == "shot" else board_circuit)(3)
    job = Job(cs, asg)
    params, pk = job.device_keys(ctx)
    lib = ctx.lib
    assert [lib.bz_pk_quotient_generated(pk.h, t) for t in range(3)] == [1, 1, 1]
    monkeypatch.setenv("BZ_QUOTIENT_GENERATED", "0")
    pk_int = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR)
    monkeypatch.delenv("BZ_QUOTIENT_GENERATED")
    assert [lib.bz_pk_quotient_generated(pk_int.h, t) for t in range(3)] == [0, 0, 0]
    a, b = _prove(job, pk, [6])[0], _prove(job, pk_int, [6])[0]
    assert first_diff(a, b) is None, first_diff(a, b)
    assert a == job.oracle_proof(index=6)
    pk_int.close(); pk.close(); params.close()
    tiny = Job(*tiny_circuit(5))
    p2, k2 = tiny.device_keys(ctx, window_bits=6)
    assert lib.bz_pk_quotient_generated(k2.h, 0) == 0
    k2.close(); p2.close()


def test_table_msm_degenerate_bases_parity(ctx, oracle_c):
    """The table MSM (fixedmsm.cu): same commitments as the oracle's best_multiexp on a URS with repeated, opposite and
    identity bases, and the Shot golden proof bytes."""
    import os
    from battlezips_halo2_b200.plonk import prover as PR
    from battlezips_halo2_b200.circuits import shot_circuit
    from tests.util_prover import VK_REPR
    from oracle import halo2 as H
    co = oracle_c
    C = co.CURVES[0][0]
    h = C.hash_to_curve("bz-pairs")
    k, n = 6, 64
    pts = [h(bytes([i])) for i in range(n + 2)]
    pts[1] = pts[0]; pts[2] = C.neg(pts[0]); pts[3] = None; pts[40] = pts[8]; pts[41] = pts[8]
    g = co.points_to_mont(0, pts[:n])
    w, u = co.points_to_mont(0, [pts[n]])[0], co.points_to_mont(0, [pts[n + 1]])[0]
    params = PR.Params(ctx, k, g, g, w, u, window_bits=5)
    rng = np.random.default_rng(5)
    for trial in range(4):
        poly = co.from_u512(0, rng.integers(0, 2**63, size=(n, 8), dtype=np.uint64))
        if trial == 1:
            poly[:] = poly[0]                                   # equal scalars: equal digits on the repeated bases
        if trial == 2:
            poly[4:] = 0
        blind = co.from_u512(0, rng.integers(0, 2**63, size=(1, 8), dtype=np.uint64))
        exp = co.to_affine(0, co.best_multiexp(0, np.concatenate([poly, blind]), np.concatenate([g, w[None]])))
        assert np.array_equal(params.commit(poly, blind[0], lagrange=False), exp[0]), trial
    params.close()
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proofs.npz"))
    cs, _, asg = shot_circuit(0)
    fx = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"params_vesta_k{asg.k}.npz"))
    params = PR.Params(ctx, asg.k, fx["g"], fx["g_lagrange"], fx["w"], fx["u"], window_bits=12)
    pk = PR.ProvingKey(ctx, params, cs.to_ir(), asg.fixed, asg.permutation_mapping(), VK_REPR)
    advice = np.stack([PR.mont(col) for col in asg.advice])
    wide = H.splitmix64_wide(0xB200B200B200B200, pk.num_random)
    proof = PR.create_proofs(pk, [asg.instance], advice[None], wide[None])[0]
    assert proof == bytes(gold["shot_w0_idx0"])
    pk.close(); params.close()


def test_device_proofs_equal_committed_goldens(ctx):
    """The committed oracle goldens (tests/golden/proofs.npz): tiny k = 5, Shot k = 11 and Board k = 12 proofs from the
    device are byte-identical -- no oracle run needed on the GPU box for this comparison (the witness / keys still come
    from the circuit mirrors)."""
    import os
    from battlezips_halo2_b200.plonk import prover as PR
    from battlezips_halo2_b200.circuits import shot_circuit, board_circuit
    from tests.util_prover import VK_REPR
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proofs.npz"))
    job = Job(*tiny_circuit(5))
    params, pk = job.device_keys(ctx, window_bits=7)
    got = _prove(job, pk, [0, 3])
    assert got[0] == bytes(gold["tiny_k5_idx0"]) and got[1] == bytes(gold["tiny_k5_idx3"])
    pk.close(); params.close()
    for make, name in ((shot_circuit, "shot_w0_idx0"), (board_circuit, "board_w0_idx0")):
        cs, _, asg = make(0)
        k = asg.k
        fx = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", f"params_vesta_k{k}.npz"))
        params = PR.Params(ctx, k, fx["g"], fx["g_lagrange"], fx["w"], fx["u"])
        pk = PR.ProvingKey(ctx, params, cs.to_ir(), asg.fixed, asg.permutation_mapping(), VK_REPR)
        advice = np.stack([PR.mont(col) for col in asg.advice])
        from oracle import halo2 as H
        wide = H.splitmix64_wide(0xB200B200B200B200, pk.num_random)
        proof = PR.create_proofs(pk, [asg.instance], advice[None], wide[None])[0]
        assert proof == bytes(gold[name]), name
        assert PR.verify_proofs(pk, [asg.instance], [proof]) == [True]
        pk.close(); params.close()
