"""CPU: oracle/chacha.py, the ChaCha20 keystream that bz_create_proofs_seeded expands on the device, against an independent
implementation (the `cryptography` package's ChaCha20, OpenSSL underneath) and the RFC 8439 §2.3.2 block vector.

cryptography takes a 16-byte nonce that is loaded verbatim into state words 12-15 (its documentation: the counter followed by
the nonce).  All zero, it gives the stream of ChaCha20Rng::from_seed: counter 0, stream id 0."""
import os
import struct
import numpy as np
import pytest
from oracle import chacha

cryptography = pytest.importorskip("cryptography")
from cryptography.hazmat.primitives.ciphers import Cipher, algorithms  # noqa: E402


def _reference_stream(key, nonce16, nbytes):
    enc = Cipher(algorithms.ChaCha20(key, nonce16), mode=None).encryptor()
    return enc.update(b"\0" * nbytes)


@pytest.mark.parametrize("blocks", [1, 2, 17, 4238])
def test_keystream_matches_cryptography(blocks):
    rng = np.random.default_rng(blocks)
    for _ in range(3):
        seed = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
        exp = _reference_stream(seed, b"\0" * 16, 64 * blocks)
        got = chacha.keystream_wide(seed, blocks)
        assert got.shape == (blocks, 8) and got.dtype == np.uint64
        assert got.astype("<u8").tobytes() == exp
        for j in sorted({0, blocks - 1, blocks // 2}):
            assert chacha.block(seed, j) == exp[64 * j:64 * j + 64]


def test_keystream_offset_and_counter_high_word():
    """A window starting past block 0, and blocks around the 2^32 carry into word 13 (the 64-bit counter): the scalar
    block function against the vectorised one, and cryptography (whose counter word 13 is the first nonce word) below it."""
    seed = bytes(range(32))
    assert chacha.keystream_wide(seed, 5, start=100).astype("<u8").tobytes() == b"".join(chacha.block(seed, j) for j in range(100, 105))
    lo = (1 << 32) - 2
    wide = chacha.keystream_wide(seed, 4, start=lo).astype("<u8").tobytes()
    assert wide == b"".join(chacha.block(seed, j) for j in range(lo, lo + 4))
    for j in range(lo, lo + 4):
        nonce16 = struct.pack("<II", j & 0xFFFFFFFF, j >> 32) + b"\0" * 8
        assert chacha.block(seed, j) == _reference_stream(seed, nonce16, 64)


def test_rfc8439_block_vector():
    """RFC 8439 §2.3.2: key 00..1f, counter 1, nonce 00:00:00:09:00:00:00:4a:00:00:00:00."""
    key = bytes(range(32))
    nonce = bytes.fromhex("000000090000004a00000000")
    exp = bytes.fromhex(
        "10f1e7e4d13b5915500fdd1fa32071c4c7d1f4c733c068030422aa9ac3d46c4e"
        "d2826446079faa0914c2d705d98b02a2b5129cd1de164eb9cbd083e8a2503c4e")
    assert _reference_stream(key, struct.pack("<I", 1) + nonce, 64) == exp
    words = chacha.block_words(struct.unpack("<8I", key), (1,) + struct.unpack("<3I", nonce))
    assert struct.pack("<16I", *words) == exp


def test_keystream_feeds_draws():
    """keystream_wide rows are what halo2.Draws consumes, like splitmix64_wide's."""
    from oracle import halo2 as H
    seed = os.urandom(32)
    d = H.Draws(chacha.keystream_wide(seed, 6))
    assert d.take(0, 6).shape == (6, 4) and d.pos == 6
