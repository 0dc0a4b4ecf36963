"""ChaCha20 keystream (test infrastructure): the stream `rand_chacha::ChaCha20Rng::from_seed(seed)` feeds to
`Scalar::random`, restated from the cipher's definition (D. J. Bernstein, "ChaCha, a variant of Salsa20"; RFC 8439 §2.1-2.3).

State: the constants "expand 32-byte k", the 8 little-endian key words = seed, a 64-bit block counter in words 12-13 and
stream id 0 in words 14-15 (the original layout rand_chacha uses; for counters below 2^32 it is RFC 8439 with an all-zero
nonce).  20 rounds (10 double rounds), then the input is added back.  One 64-byte block is one Scalar::random draw
(8 x next_u64, low word first), so `keystream_wide(seed, R)` is a rand_wide row that `halo2.Draws` consumes."""
import struct
import numpy as np

SIGMA = (0x61707865, 0x3320646E, 0x79622D32, 0x6B206574)
M32 = 0xFFFFFFFF


def _rotl(x, r):
    return ((x << r) | (x >> (32 - r))) & M32


def _quarter(s, a, b, c, d):
    s[a] = (s[a] + s[b]) & M32; s[d] = _rotl(s[d] ^ s[a], 16)
    s[c] = (s[c] + s[d]) & M32; s[b] = _rotl(s[b] ^ s[c], 12)
    s[a] = (s[a] + s[b]) & M32; s[d] = _rotl(s[d] ^ s[a], 8)
    s[c] = (s[c] + s[d]) & M32; s[b] = _rotl(s[b] ^ s[c], 7)


def block_words(key_words, counter_nonce_words):
    """The block function over a 16-word input: 4 constants, 8 key words, 4 counter / nonce words -> 16 output words."""
    init = list(SIGMA) + list(key_words) + list(counter_nonce_words)
    assert len(init) == 16
    s = list(init)
    for _ in range(10):
        _quarter(s, 0, 4, 8, 12); _quarter(s, 1, 5, 9, 13); _quarter(s, 2, 6, 10, 14); _quarter(s, 3, 7, 11, 15)
        _quarter(s, 0, 5, 10, 15); _quarter(s, 1, 6, 11, 12); _quarter(s, 2, 7, 8, 13); _quarter(s, 3, 4, 9, 14)
    return [(x + y) & M32 for x, y in zip(s, init)]


def block(seed, counter):
    """64-byte block `counter` of the keystream of a 32-byte seed (64-bit counter in words 12-13, stream id 0)."""
    assert len(seed) == 32 and 0 <= counter < 1 << 64
    out = block_words(struct.unpack("<8I", seed), (counter & M32, counter >> 32, 0, 0))
    return struct.pack("<16I", *out)


def _rotl_np(x, r):
    return (x << np.uint32(r)) | (x >> np.uint32(32 - r))


def keystream_wide(seed, n, start=0):
    """Blocks start .. start+n-1 of seed's keystream as (n, 8) uint64 -- the shape of halo2.splitmix64_wide, one row per
    Scalar::random draw.  The same block function as `block`, evaluated for all counters at once over numpy uint32 columns."""
    assert len(seed) == 32
    ctr = np.arange(start, start + n, dtype=np.uint64)
    init = [np.full(n, w, dtype=np.uint32) for w in SIGMA + struct.unpack("<8I", seed)]
    init += [(ctr & np.uint64(M32)).astype(np.uint32), (ctr >> np.uint64(32)).astype(np.uint32),
             np.zeros(n, np.uint32), np.zeros(n, np.uint32)]
    s = [w.copy() for w in init]

    def q(a, b, c, d):
        s[a] += s[b]; s[d] = _rotl_np(s[d] ^ s[a], 16)
        s[c] += s[d]; s[b] = _rotl_np(s[b] ^ s[c], 12)
        s[a] += s[b]; s[d] = _rotl_np(s[d] ^ s[a], 8)
        s[c] += s[d]; s[b] = _rotl_np(s[b] ^ s[c], 7)

    for _ in range(10):
        q(0, 4, 8, 12); q(1, 5, 9, 13); q(2, 6, 10, 14); q(3, 7, 11, 15)
        q(0, 5, 10, 15); q(1, 6, 11, 12); q(2, 7, 8, 13); q(3, 4, 9, 14)
    words = np.stack([x + y for x, y in zip(s, init)], axis=1)          # (n, 16) uint32, little-endian word order
    return np.ascontiguousarray(words.astype("<u4")).view("<u8").astype(np.uint64).reshape(n, 8)
