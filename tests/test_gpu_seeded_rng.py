"""GPU: create_proof's blinding randomness expanded on the device from one ChaCha20 seed per proof.

bz_chacha20_blocks against the oracle keystream (oracle/chacha.py, itself checked against the `cryptography` package on the
CPU) bit for bit, into host and device buffers; bz_create_proofs_seeded against bz_create_proofs fed that keystream as
rand_wide and against the oracle's create_proof fed it through halo2.Draws, on both commitment paths (fixed-base tables and
the bucket MSM, selected as tests/test_gpu_commit_paths.py selects them); every seeded proof verified through a VerifyingKey;
the error cases of the seeded entry point."""
import numpy as np
import pytest
from oracle import chacha, halo2 as H
from tests.util_prover import Job, VK_REPR, first_diff, tiny_circuit

pytestmark = pytest.mark.gpu

R_SHOT = 4238                   # bz_pk_num_random of the Shot circuit (k = 11)
BIG = (1 << 20) + 3


def _seeds(count, salt):
    rng = np.random.default_rng(salt)
    s = rng.integers(0, 256, size=(count, 32), dtype=np.uint8)
    assert len({bytes(r) for r in s}) == count
    return s


def _keystreams(seeds, blocks):
    return np.stack([chacha.keystream_wide(bytes(s), blocks) for s in seeds])


# ---- the keystream on its own ----------------------------------------------------------------------------------------------
CASES = [(B, blocks, where) for B in (1, 3, 64) for blocks in (1, 2, 17, R_SHOT, BIG) for where in ("host", "device")
         if not (B == 64 and blocks == BIG and where == "host")]      # 4.3 GB of host memory; the device case covers the size


@pytest.mark.parametrize("B,blocks,where", CASES)
def test_chacha20_blocks_match_oracle(B, blocks, where, ctx):
    from battlezips_halo2_b200 import arithmetic as ar
    seeds = _seeds(B, B * 7919 + blocks)
    # B = 64 at 2^20 + 3 blocks: rows 0, 31 and 63 in full, and the first and last block of every row
    full = [0, 31, 63] if B * blocks > 1 << 24 else list(range(B))
    if where == "host":
        got = ar.chacha20_blocks(ctx, seeds, blocks)
    else:
        import torch
        buf = torch.full((B, blocks, 8), -1, dtype=torch.int64, device="cuda:0")
        torch.cuda.synchronize()            # the fill runs on torch's stream, the context has a stream of its own
        ar.chacha20_blocks(ctx, seeds, blocks, out=buf.data_ptr())
        got = None
    for b in range(B):
        row = got[b] if got is not None else buf[b].cpu().numpy().view(np.uint64)
        if b in full:
            exp = chacha.keystream_wide(bytes(seeds[b]), blocks)
            assert np.array_equal(row, exp), (b, int(np.argmin((row == exp).all(axis=1))))
        else:
            for j in (0, blocks - 1):
                assert row[j].astype("<u8").tobytes() == chacha.block(bytes(seeds[b]), j), (b, j)


def test_chacha20_blocks_unaligned_device_output(ctx):
    """A device buffer that is not 16-byte aligned is written through the staging copy, with the same bytes."""
    import torch
    from battlezips_halo2_b200 import arithmetic as ar
    seeds = _seeds(2, 5)
    raw = torch.zeros(2 * 17 * 64 + 16, dtype=torch.uint8, device="cuda:0")
    torch.cuda.synchronize()
    ar.chacha20_blocks(ctx, seeds, 17, out=raw.data_ptr() + 4)
    got = raw[4:4 + 2 * 17 * 64].cpu().numpy().view(np.uint64).reshape(2, 17, 8)
    assert np.array_equal(got, _keystreams(seeds, 17))
    assert not raw[:4].any() and not raw[4 + 2 * 17 * 64:].any()


# ---- seeded proofs ---------------------------------------------------------------------------------------------------------
def _oracle_seeded(job, seed):
    T = H.Blake2bTranscript(0)
    draws = H.Draws(chacha.keystream_wide(bytes(seed), job.num_random()))
    H.create_proof(job.oparams, job.opk, job.instances, [job.advice[i] for i in range(len(job.advice))], draws, T)
    assert draws.pos == job.num_random()
    return T.finalize()


def _keys(ctx, job, path):
    from battlezips_halo2_b200.plonk import prover as PR
    op = job.oparams
    with pytest.MonkeyPatch.context() as mp:
        if path == "bucket":
            mp.setenv("BZ_FORCE_GENERAL_MSM", "1")
        params = PR.Params(ctx, job.k, op.g, op.g_lagrange, op.w, op.u, window_bits=8)
    pk = PR.ProvingKey(ctx, params, job.ir, job.asg.fixed, job.mapping, VK_REPR)
    assert pk.num_random == job.num_random()
    return params, pk


_JOBS = {}


def _job(which):
    if which not in _JOBS:
        if which == "tiny":
            _JOBS[which] = Job(*tiny_circuit(5))
        else:
            from battlezips_halo2_b200.circuits import shot_circuit, board_circuit
            cs, _, asg = (shot_circuit if which == "shot" else board_circuit)(0)
            _JOBS[which] = Job(cs, asg)
    return _JOBS[which]


def _check_seeded(ctx, job, params, pk, seeds, oracle_rows):
    """seeded == create_proofs(keystream) for every proof; == the oracle for `oracle_rows`; every proof verifies through a
    VerifyingKey and the seeded proofs of distinct seeds are distinct."""
    from battlezips_halo2_b200.plonk import prover as PR
    B = len(seeds)
    advice = np.stack([job.advice] * B)
    seeded = PR.create_proofs_seeded(pk, [job.instances] * B, advice, seeds)
    plain = PR.create_proofs(pk, [job.instances] * B, advice, _keystreams(seeds, pk.num_random))
    for b in range(B):
        assert seeded[b] == plain[b], (b, first_diff(seeded[b], plain[b]))
    for b in oracle_rows:
        exp = _oracle_seeded(job, seeds[b])
        assert seeded[b] == exp, (b, first_diff(seeded[b], exp))
    assert len(set(seeded)) == B
    vk = pk.verifying_key()
    try:
        assert PR.verify_proofs(vk, [job.instances] * B, seeded) == [True] * B
    finally:
        vk.close()
    return seeded


PROOF_CASES = [("tiny", 1), ("tiny", 3), ("shot", 1), ("shot", 3), ("shot", 64), ("board", 1), ("board", 3)]


@pytest.mark.parametrize("path", ["tables", "bucket"])
@pytest.mark.parametrize("which,batch", PROOF_CASES, ids=[f"{w}-b{b}" for w, b in PROOF_CASES])
def test_seeded_proofs_match_keystream_and_oracle(which, batch, path, ctx):
    job = _job(which)
    params, pk = _keys(ctx, job, path)
    try:
        oracle_rows = list(range(batch)) if which == "tiny" else [0, batch - 1] if batch > 1 else [0]
        _check_seeded(ctx, job, params, pk, _seeds(batch, 1000 * PROOF_CASES.index((which, batch)) + (path == "bucket")), sorted(set(oracle_rows)))
    finally:
        pk.close(); params.close()


def test_seeded_scaled_board_k16(ctx):
    """The Board circuit tiled down 2^16 rows, one proof: the large-domain path mirrors only the short stream ranges the host
    reads (blinds) back from the device."""
    from battlezips_halo2_b200.circuits import board_circuit_scaled
    cs, _, asg = board_circuit_scaled(16)
    job = Job(cs, asg, params_from_device=ctx)
    params, pk = job.device_keys(ctx)
    try:
        _check_seeded(ctx, job, params, pk, _seeds(1, 16), [0])
    finally:
        pk.close(); params.close()


def test_same_seed_same_proof_and_errors(ctx):
    """Two calls with the same seed and witness give identical bytes; a null pointer, batch = 0 and a repeated seed in one call
    are BZ_ERR_INVALID with nothing written, and the context proves correctly afterwards."""
    import battlezips_halo2_b200 as bz
    from battlezips_halo2_b200.plonk import prover as PR
    from battlezips_halo2_b200.binding import _np_ptr
    job = _job("tiny")
    params, pk = job.device_keys(ctx, window_bits=8)
    try:
        seeds = _seeds(2, 99)
        one = PR.create_proofs_seeded(pk, [job.instances], job.advice[None], seeds[:1])
        again = PR.create_proofs_seeded(pk, [job.instances] * 2, np.stack([job.advice] * 2), [bytes(seeds[1]), bytes(seeds[0])])
        assert again[1] == one[0] and again[0] != one[0]

        lib = ctx.lib
        inst, lens, stride = PR._pack_instances(pk, [job.instances] * 2, 2)
        adv = np.ascontiguousarray(np.stack([job.advice] * 2), dtype=np.uint64)
        out = np.zeros((2, pk.proof_size), dtype=np.uint8)
        dup = np.ascontiguousarray(np.stack([seeds[0], seeds[0]]))
        args = lambda B, s, o: (ctx.h, pk.h, B, _np_ptr(inst), _np_ptr(lens), stride, _np_ptr(adv), s, o)
        assert lib.bz_create_proofs_seeded(*args(2, None, _np_ptr(out))) == -1
        assert lib.bz_create_proofs_seeded(*args(2, _np_ptr(seeds), None)) == -1
        assert lib.bz_create_proofs_seeded(ctx.h, None, 1, _np_ptr(inst), _np_ptr(lens), stride, _np_ptr(adv), _np_ptr(seeds), _np_ptr(out)) == -1
        assert lib.bz_create_proofs_seeded(*args(0, _np_ptr(seeds), _np_ptr(out))) == -1
        assert lib.bz_create_proofs_seeded(*args(2, _np_ptr(dup), _np_ptr(out))) == -1
        assert b"repeats" in lib.bz_last_error(ctx.h)
        assert not out.any()
        assert lib.bz_chacha20_blocks(ctx.h, None, 1, 1, _np_ptr(out)) == -1
        assert lib.bz_chacha20_blocks(ctx.h, _np_ptr(seeds), 1, 1, None) == -1
        with pytest.raises(bz.BzError):
            PR.create_proofs_seeded(pk, [job.instances] * 2, adv, dup)

        after = PR.create_proofs_seeded(pk, [job.instances] * 2, adv, seeds)
        assert after == [one[0], again[0]]
        assert after[0] == _oracle_seeded(job, seeds[0])
        assert PR.create_proofs(pk, [job.instances], job.advice[None], job.wide(0)[None])[0] == job.oracle_proof(index=0)
    finally:
        pk.close(); params.close()
