"""GPU: verify_proof from a verifying key alone (bz_vk_create / bz_verify_proofs_vk).  A vk holds what halo2's VerifyingKey
holds -- the constraint system, keygen_vk's fixed and permutation commitments and the vk.hash_into scalar -- and no fixed
values or sigma columns.  Its verdicts equal the restated reference verifier's and those of the proving-key path, it works
after the proving key is closed, a wrong vk rejects valid proofs, bad commitments are refused at creation, and creating one
takes no device memory."""
import copy
import ctypes
import numpy as np
import pytest
from oracle import c_oracle as co, halo2 as H
from tests.util_prover import Job, tiny_circuit, VK_REPR

pytestmark = pytest.mark.gpu

Q = 0x40000000000000000000000000000000224698fc0994a8dd8c46eb2100000001     # Vesta base field: the commitments' coordinates


def _prove(job, pk, indices):
    from battlezips_halo2_b200.plonk import prover as PR
    B = len(indices)
    return PR.create_proofs(pk, [job.instances] * B, np.stack([job.advice] * B), np.stack([job.wide(i) for i in indices]))


def _flip(proof, byte, bit=0):
    b = bytearray(proof)
    b[byte] ^= 1 << bit
    return bytes(b)


def _params(ctx, job, window_bits=0):
    from battlezips_halo2_b200.plonk import prover as PR
    op = job.oparams
    return PR.Params(ctx, job.k, op.g, op.g_lagrange, op.w, op.u, window_bits=window_bits)


def _oracle_commitments(opk):
    return (np.ascontiguousarray(co.points_to_mont(0, opk.fixed_commitments)),
            np.ascontiguousarray(co.points_to_mont(0, opk.perm_commitments)))


def _oracle_vk(ctx, job, params, fc=None, pc=None, vk_repr=VK_REPR):
    """A vk from the oracle keygen's commitments: no device proving key is involved."""
    from battlezips_halo2_b200.plonk import prover as PR
    ofc, opc = _oracle_commitments(job.opk)
    return PR.VerifyingKey(ctx, params, job.ir, ofc if fc is None else fc, opc if pc is None else pc, vk_repr)


def test_tiny_vk_from_oracle_keygen_verifies_like_the_oracle_and_the_pk(ctx):
    from battlezips_halo2_b200.plonk import prover as PR
    job = Job(*tiny_circuit(5))
    params = _params(ctx, job, window_bits=6)
    vk = _oracle_vk(ctx, job, params)
    # no proving key exists yet: oracle proofs
    assert PR.verify_proofs(vk, [job.instances] * 2, [job.oracle_proof(index=5), job.oracle_proof(index=6)]) == [True, True]
    pk = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR)
    assert vk.proof_size == pk.proof_size
    fc, pc = pk.vk_commitments()
    ofc, opc = _oracle_commitments(job.opk)
    assert np.array_equal(fc, ofc) and np.array_equal(pc, opc)
    good = _prove(job, pk, [0, 1, 2])
    assert PR.verify_proofs(vk, [job.instances] * 3, good) == [True, True, True]
    # one flipped bit in every 32-byte item of the proof (points, evaluations, u-evaluations, L/R, c, f)
    proof = good[0]
    items = len(proof) // 32
    bad = [_flip(proof, 32 * i + (7 * i) % 31, i % 8) for i in range(items)]
    got = PR.verify_proofs(vk, [job.instances] * items, bad)
    assert got == [job.verify(p) for p in bad]
    assert got == PR.verify_proofs(pk, [job.instances] * items, bad)
    assert not any(got)
    # a mixed batch keeps per-proof verdicts
    assert PR.verify_proofs(vk, [job.instances] * 4, [good[1], bad[3], good[2], bad[-1]]) == [True, False, True, False]
    # wrong public input
    assert PR.verify_proofs(vk, [[[12]]], [proof]) == [False] == PR.verify_proofs(pk, [[[12]]], [proof])
    assert not job.verify(proof, instances=[[12]])
    # wrong lengths
    assert PR.verify_proofs(vk, [job.instances], [proof[:-32]]) == [False]
    assert PR.verify_proofs(vk, [job.instances], [proof + bytes(32)]) == [False]
    vk.close(); pk.close(); params.close()


def test_tiny_vk_rejects_malformed_encodings(ctx):
    from battlezips_halo2_b200.plonk import prover as PR
    job = Job(*tiny_circuit(5))
    params = _params(ctx, job, window_bits=6)
    vk = _oracle_vk(ctx, job, params)
    proof = job.oracle_proof(index=0)
    p = 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001
    bad = [bytes(32) + proof[32:],                                       # identity where a commitment is expected
           b"\xff" * 31 + b"\x7f" + proof[32:]]                          # x >= q
    x_not_on_curve = next(x for x in range(1, 50) if pow((x ** 3 + 5) % Q, (Q - 1) // 2, Q) != 1)
    bad.append(x_not_on_curve.to_bytes(32, "little") + proof[32:])
    ev_off = len(proof) - 64                                             # the scalar c: p itself is not canonical
    bad.append(proof[:ev_off] + p.to_bytes(32, "little") + proof[ev_off + 32:])
    got = PR.verify_proofs(vk, [job.instances] * len(bad), bad)
    assert got == [False] * len(bad)
    assert [job.verify(b) for b in bad] == got
    pk = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR)
    assert PR.verify_proofs(pk, [job.instances] * len(bad), bad) == got
    vk.close(); pk.close(); params.close()


def test_wrong_vk_rejects_valid_proofs_like_the_oracle(ctx):
    from battlezips_halo2_b200.plonk import prover as PR
    job = Job(*tiny_circuit(5))
    params = _params(ctx, job, window_bits=6)
    proof = job.oracle_proof(index=3)
    fc, pc = _oracle_commitments(job.opk)
    assert len(fc) >= 2 and len(pc) >= 2
    # one fixed commitment replaced by another valid point, two sigma commitments swapped, another vk repr
    fc_wrong = fc.copy(); fc_wrong[0] = fc[1]
    pc_swapped = pc.copy(); pc_swapped[[0, 1]] = pc[[1, 0]]
    o_fix, o_sig, o_rep = copy.copy(job.opk), copy.copy(job.opk), copy.copy(job.opk)
    o_fix.fixed_commitments = [job.opk.fixed_commitments[1]] + list(job.opk.fixed_commitments[1:])
    o_sig.perm_commitments = [job.opk.perm_commitments[1], job.opk.perm_commitments[0]] + list(job.opk.perm_commitments[2:])
    o_rep.vk_repr = VK_REPR + 1
    right = _oracle_vk(ctx, job, params)
    assert PR.verify_proofs(right, [job.instances], [proof]) == [True]
    for vk_args, opk in (({"fc": fc_wrong}, o_fix), ({"pc": pc_swapped}, o_sig), ({"vk_repr": VK_REPR + 1}, o_rep)):
        vk = _oracle_vk(ctx, job, params, **vk_args)
        assert PR.verify_proofs(vk, [job.instances], [proof]) == [False]
        assert not H.verify_proof(job.oparams, opk, job.instances, proof)
        vk.close()
    right.close(); params.close()


def test_shot_and_board_vk_from_pk_outlives_the_pk(ctx):
    """Shot: 8 proofs, a tampered one; Board: one proof and a flipped bit.  The vk comes from ProvingKey.verifying_key() and the
    pk is closed before the vk verifies; verdicts equal the pk path's on the same batch.  Board's vk given a Shot proof (the
    wrong length) rejects it."""
    from battlezips_halo2_b200.circuits import shot_circuit, board_circuit
    from battlezips_halo2_b200.plonk import prover as PR
    cs, cfg, asg = shot_circuit(0)
    shot = Job(cs, asg)
    s_params = _params(ctx, shot)
    s_pk = PR.ProvingKey(ctx, s_params, shot.ir, shot.asg.fixed, shot.mapping, VK_REPR)
    proofs = _prove(shot, s_pk, list(range(8)))
    batch = proofs + [_flip(proofs[3], 1000, 2)]
    by_pk = PR.verify_proofs(s_pk, [shot.instances] * len(batch), batch)
    s_vk = s_pk.verifying_key()
    assert s_vk.proof_size == s_pk.proof_size
    s_pk.close()
    by_vk = PR.verify_proofs(s_vk, [shot.instances] * len(batch), batch)
    assert by_vk == by_pk == [True] * 8 + [False]
    s_vk.close(); s_params.close()

    cs, cfg, asg = board_circuit(0)
    board = Job(cs, asg)
    b_params = _params(ctx, board)
    b_pk = PR.ProvingKey(ctx, b_params, board.ir, board.asg.fixed, board.mapping, VK_REPR)
    proof = _prove(board, b_pk, [0])[0]
    batch = [proof, _flip(proof, 2048)]
    by_pk = PR.verify_proofs(b_pk, [board.instances] * 2, batch)
    b_vk = b_pk.verifying_key()
    assert b_vk.proof_size == b_pk.proof_size
    b_pk.close()
    assert PR.verify_proofs(b_vk, [board.instances] * 2, batch) == by_pk == [True, False]
    # a Shot proof under Board's vk: wrong length, rejected (the Board instance shape is what the vk expects)
    assert len(proofs[0]) != b_vk.proof_size
    assert PR.verify_proofs(b_vk, [board.instances], [proofs[0]]) == [False]
    b_vk.close(); b_params.close()


def test_scaled_board_k15_vk_on_device_only(ctx):
    from battlezips_halo2_b200 import arithmetic as ar
    from battlezips_halo2_b200.circuits import board_circuit_scaled
    from battlezips_halo2_b200.plonk import prover as PR
    k = 15
    cs, cfg, asg = board_circuit_scaled(k)
    ir = cs.to_ir()
    urs = ar.params_new(ctx, k, curve=0)
    params = PR.Params(ctx, k, urs["g"], urs["g_lagrange"], urs["w"], urs["u"])
    pk = PR.ProvingKey(ctx, params, ir, asg.fixed, asg.permutation_mapping(), VK_REPR)
    advice = np.stack([PR.mont(col) for col in asg.advice])
    wide = H.splitmix64_wide(0xB200 + k, pk.num_random)
    proof = PR.create_proofs(pk, [asg.instance], advice[None], wide[None])[0]
    vk = pk.verifying_key()
    pk.close()
    assert PR.verify_proofs(vk, [asg.instance] * 2, [proof, _flip(proof, len(proof) // 2)]) == [True, False]
    vk.close(); params.close()


def test_vk_creation_errors(ctx):
    """Each bad input gives BZ_ERR_INVALID with a message, without a crash, and the context keeps working afterwards."""
    from battlezips_halo2_b200 import arithmetic as ar, BzError
    from battlezips_halo2_b200.plonk import prover as PR
    job = Job(*tiny_circuit(5))
    params = _params(ctx, job, window_bits=6)
    fc, pc = _oracle_commitments(job.opk)

    def refused(fc2=fc, pc2=pc, p=params, what=""):
        with pytest.raises(BzError) as e:
            PR.VerifyingKey(ctx, p, job.ir, fc2, pc2, VK_REPR)
        assert e.value.code == -1 and what in str(e.value), str(e.value)

    off = fc.copy(); off[2, 4:] = off[2, :4]                                 # y := x, both canonical: not on the curve
    refused(fc2=off, what="not on y^2 = x^3 + 5")
    q_limbs = np.frombuffer(Q.to_bytes(32, "little"), dtype=np.uint64)
    nc = pc.copy(); nc[1, :4] = q_limbs                                     # x = q
    refused(pc2=nc, what="not canonical")
    ident = fc.copy(); ident[0] = 0
    refused(fc2=ident, what="identity")
    ident = pc.copy(); ident[-1] = 0
    refused(pc2=ident, what="identity")
    urs = ar.params_new(ctx, 5, curve=1)                                  # Pallas params
    pallas = PR.Params(ctx, 5, urs["g"], urs["g_lagrange"], urs["w"], urs["u"], curve=1, window_bits=6)
    refused(p=pallas, what="Vesta")
    pallas.close()
    # through the C ABI: k mismatch and null pointers
    lib = ctx.lib
    h = ctypes.c_void_p()
    fcp, pcp = fc.ctypes.data_as(ctypes.c_void_p), pc.ctypes.data_as(ctypes.c_void_p)
    circ6, keep6 = PR.flatten_circuit(job.ir, 6, VK_REPR)
    assert lib.bz_vk_create(ctx.h, params.h, ctypes.byref(circ6), fcp, pcp, ctypes.byref(h)) == -1 and not h.value
    assert b"k" in lib.bz_last_error(ctx.h)
    circ, keep = PR.flatten_circuit(job.ir, 5, VK_REPR)
    for args in ((None, params.h, ctypes.byref(circ), fcp, pcp, ctypes.byref(h)),
                 (ctx.h, None, ctypes.byref(circ), fcp, pcp, ctypes.byref(h)),
                 (ctx.h, params.h, None, fcp, pcp, ctypes.byref(h)),
                 (ctx.h, params.h, ctypes.byref(circ), None, pcp, ctypes.byref(h)),
                 (ctx.h, params.h, ctypes.byref(circ), fcp, None, ctypes.byref(h)),
                 (ctx.h, params.h, ctypes.byref(circ), fcp, pcp, None)):
        assert lib.bz_vk_create(*args) == -1 and not h.value
    assert lib.bz_vk_proof_size(None) == 0
    lib.bz_vk_destroy(None)
    res = np.zeros(1, np.uint8)
    assert lib.bz_verify_proofs_vk(ctx.h, None, 1, None, None, 1, res.ctypes.data_as(ctypes.c_void_p), 32, res.ctypes.data_as(ctypes.c_void_p)) == -1
    # the context still works
    vk = PR.VerifyingKey(ctx, params, job.ir, fc, pc, VK_REPR)
    assert PR.verify_proofs(vk, [job.instances], [job.oracle_proof(index=1)]) == [True]
    vk.close(); params.close()
    ctx.sync()


def test_board_vk_creation_allocates_no_device_memory(ctx):
    """A Board pk holds ~150 MB of device images; its vk holds host data only (the staging grows on the first verify)."""
    import torch
    from battlezips_halo2_b200.circuits import board_circuit
    from battlezips_halo2_b200.plonk import prover as PR
    cs, cfg, asg = board_circuit(0)
    job = Job(cs, asg)
    params = _params(ctx, job)
    fc, pc = _oracle_commitments(job.opk)
    torch.cuda.mem_get_info(0)
    # another process on the GPU can only make a difference look larger: keep the smallest of three
    used = []
    for _ in range(3):
        ctx.sync()
        free0 = torch.cuda.mem_get_info(0)[0]
        vk = PR.VerifyingKey(ctx, params, job.ir, fc, pc, VK_REPR)
        ctx.sync()
        used.append(free0 - torch.cuda.mem_get_info(0)[0])
        vk.close()
    assert min(used) < 2 << 20, used
    ctx.sync()
    free0 = torch.cuda.mem_get_info(0)[0]
    pk = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR)
    ctx.sync()
    assert free0 - torch.cuda.mem_get_info(0)[0] > 50 << 20
    pk.close(); params.close()
