"""Scalars for the MSM tests: the signed-digit recoding both MSM engines use, stated in Python, and labelled scalar
families that reach its boundary cases at a given window width c.

Both engines (the bucket MSM, msm.cu `msm_for_each_digit`; the table MSM, fixedmsm.cu `fb_decode_kernel`) cut the
canonical scalar into W = ceil(256 / c) windows of c bits and recode window w as

    v = raw_w + carry;  neg = v > 2^(c-1);  d = neg ? 2^c - v : v;  carry = neg

so the digit is -d when neg is set, else d.  The cases where a small mistake is easy:
    half  v = 2^(c-1) exactly: stays positive, in the largest bucket
    neg   v > 2^(c-1): negative digit, carries into the next window
    full  v = 2^c (all-ones window plus a carry): zero digit that still carries
    top   a carry into, or a non-zero digit in, the top window W - 1

Both scalar fields have a modulus r = 2^254 + eps with eps < 2^126: uniform scalars almost never set bit 254, but every
small negative r - x does."""
import random
import numpy as np
from battlezips_halo2_b200.binding import _np_ptr

CASES = ("half", "neg", "full", "top")
FAMILIES = ("edges", "half", "half_after_carry", "carry_chain", "negatives", "uniform", "witness")


def modulus(field):
    from oracle import pasta
    return (pasta.FP, pasta.FQ)[field].p


def recode(s, c):
    """The kernels' recoding of the canonical scalar s at width c -> (digits, cases, carry_out): W signed digits with
    s == sum(d_w * 2^(c w)), the subset of CASES the scalar hits, and the carry left after window W - 1."""
    W = (256 + c - 1) // c
    half, full = 1 << (c - 1), 1 << c
    digits, cases, carry = [], set(), 0
    for w in range(W):
        raw = (s >> (w * c)) & (full - 1)
        v = raw + carry
        neg = v > half
        d = full - v if neg else v
        carry = 1 if neg else 0
        digits.append(-d if neg else d)
        if v == half:
            cases.add("half")
        if neg:
            cases.add("neg")
        if v == full:
            cases.add("full")
        if w == W - 1 and v:
            cases.add("top")
    return digits, cases, carry


def top_reachable(c):
    """Whether a canonical scalar can put anything into the top window at width c.  For c in {3, 5, 15} the top window
    starts at bit (W - 1) c = 255 and could only receive a carry out of window W - 2, which ends at bit 254.  Bits
    126 .. 253 of a canonical s >= 2^254 are zero (eps < 2^126), so a window inside them has raw = 0 and passes on no
    carry, and window W - 2 then holds at most raw = 2^(c-1) (bit 254 alone): v = half, no carry.  A scalar below 2^254
    gives window W - 2 at most 2^(c-1) - 1 plus a carry, again no more than half."""
    W = (256 + c - 1) // c
    return (W - 1) * c < 255


def _structured(r, c):
    W = (256 + c - 1) // c
    half = 1 << (c - 1)
    full_windows = [w for w in range(W) if (w + 1) * c <= 254]           # every full window below bit 254
    m = 254 // c
    return {
        "edges": [0, 1, 2, r - 1, r - 2, r - (1 << 32), 1 << 254, (1 << 254) - 1, (r - 1) // 2, (r + 1) // 2,
                  half, (1 << c) - 1, 1 << c],
        "half": [sum(half << (w * c) for w in full_windows)],
        # raw = half + 1 (negative, carries) then raw = half - 1 (plus the carry: exactly half), alternating
        "half_after_carry": [sum((half + 1 if i % 2 == 0 else half - 1) << (w * c) for i, w in enumerate(full_windows))],
        # first digit -1, every later window v = 2^c (zero digit, carry), the carry ends in window m
        "carry_chain": [(1 << (c * m)) - 1],
    }


def family_ints(field, c, count, seed):
    """{label: count canonical ints}.  Lists shorter than count are cycled (edges starting at an offset from seed, so
    different seeds of count 1 see different edges)."""
    r = modulus(field)
    rnd = random.Random(seed * 1000003 + field * 17 + c)
    out = {}
    for label, vals in _structured(r, c).items():
        k = seed % len(vals)
        out[label] = [vals[(k + i) % len(vals)] for i in range(count)]
    negs = [r - x for x in [1, 2, 3, 1 << 10] + [rnd.randrange(1, 1 << 64) for _ in range(4)]]
    out["negatives"] = [negs[(seed + i) % len(negs)] for i in range(count)]
    out["uniform"] = [rnd.randrange(r) for _ in range(count)]
    wit = []
    for _ in range(count):                      # SURVEY 8d "W": 70 % zero, 20 % one, 5 % below 2^10, 5 % uniform
        u = rnd.random()
        wit.append(0 if u < 0.7 else 1 if u < 0.9 else rnd.randrange(2, 1 << 10) if u < 0.95 else rnd.randrange(r))
    out["witness"] = wit
    assert list(out) == list(FAMILIES)
    assert all(0 <= s < r for vals in out.values() for s in vals)
    return out


def families(field, c, count, seed):
    """{label: (count, 4) uint64 Montgomery limbs}: family_ints encoded by the oracle."""
    from oracle import c_oracle as co
    return {label: co.to_mont(field, vals) for label, vals in family_ints(field, c, count, seed).items()}


def pick_window(n):
    """msm.cu `pick_window`: the bucket MSM's window for n points when the caller passes window_bits = 0."""
    def top_bits(c):
        return 255 - ((256 + c - 1) // c - 1) * c
    best, best_cost = 4, 1e300
    for c in range(4, 17):
        tb = top_bits(c)
        if c > 4 and 0 < tb < c // 2:
            continue
        cost = ((256 + c - 1) // c) * (n + 2.8 * (1 << (c - 1)))
        if cost < best_cost:
            best, best_cost = c, cost
    return best


# n of the window_bits = 0 bucket-MSM tests, and the window each one is meant to exercise (the last n of the c = 10 band,
# the first of the c = 13 and c = 16 bands)
AUTO_WINDOW_SIZES = {100: 5, 5000: 10, 32017: 10, 32018: 13, 320000: 15, 321127: 16}


def oracle_msms(co, curve, jobs):
    """Affine (len(jobs), 8) results of the oracle's best_multiexp over [(scalars, bases)], many small MSMs at once: one
    oracle thread per MSM, the MSMs spread over the CPU cores (ctypes releases the GIL during the call)."""
    from concurrent.futures import ThreadPoolExecutor
    jobs = [(np.ascontiguousarray(s, dtype=np.uint64), np.ascontiguousarray(b, dtype=np.uint64)) for s, b in jobs]
    threads = co.get_threads()
    co.set_threads(1)                       # the oracle's pool is process-wide: a one-thread oracle runs inline
    try:
        with ThreadPoolExecutor(max_workers=max(1, threads)) as ex:
            jac = list(ex.map(lambda j: co.best_multiexp(curve, j[0], j[1]), jobs))
    finally:
        co.set_threads(threads)
    return co.to_affine(curve, np.stack(jac)) if jac else np.zeros((0, 8), dtype=np.uint64)


def urs_points(ctx, co, curve, n):
    """g[i] = hash_to_curve("Halo2-Parameters")(0 || i_le32) for i < n, computed on the device (bz_hash_to_curve); a
    sample is re-derived by the oracle's own hash-to-curve first.  (n, 8) uint64 Montgomery affine."""
    msgs = np.zeros((n, 5), dtype=np.uint8)
    msgs[:, 1:] = np.arange(n, dtype="<u4").view(np.uint8).reshape(n, 4)
    out = np.zeros((n, 8), dtype=np.uint64)
    ctx._check(ctx.lib.bz_hash_to_curve(ctx.h, curve, b"Halo2-Parameters", _np_ptr(msgs), 5, n, _np_ptr(out)))
    C = co.CURVES[curve][0]
    h = C.hash_to_curve("Halo2-Parameters")
    for i in sorted({i for i in (0, 1, n // 2 + 3, n - 1) if i < n}):
        assert co.points_from_mont(curve, out[i][None, :])[0] == h(b"\x00" + int(i).to_bytes(4, "little")), i
    return out
