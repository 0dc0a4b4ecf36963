"""Mirror of `halo2_proofs::arithmetic` and `halo2_proofs::poly::EvaluationDomain` entry points over the C ABI
(U: halo2_proofs 0.2.0 src/arithmetic.rs, src/poly/domain.rs; SURVEY §8 a2/a4/a5).

Arrays are numpy uint64 of shape (n, 4) [field elements], (n, 8) [affine points], (12,) [Jacobian], holding
pasta's in-memory Montgomery limbs -- exactly the bytes the Rust side owns."""
import ctypes
import numpy as np
from .binding import _np_ptr, _seed_array


def best_multiexp(ctx, curve, coeffs, bases):
    """arithmetic::best_multiexp(coeffs, bases) -> C::Curve (Jacobian, 12 limbs)."""
    coeffs = np.ascontiguousarray(coeffs, dtype=np.uint64).reshape(-1, 4)
    bases = np.ascontiguousarray(bases, dtype=np.uint64).reshape(-1, 8)
    assert len(coeffs) == len(bases), "assert_eq!(coeffs.len(), bases.len())"
    out = np.zeros(12, dtype=np.uint64)
    ctx._check(ctx.lib.bz_best_multiexp(ctx.h, curve, _np_ptr(coeffs), _np_ptr(bases), len(coeffs), _np_ptr(out)))
    return out


def best_fft(ctx, field, a, omega, log_n):
    """arithmetic::best_fft(&mut a, omega, log_n): in place on a copy, returned."""
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4).copy()
    assert len(a) == 1 << log_n, "assert_eq!(n, 1 << log_n)"
    omega = np.ascontiguousarray(omega, dtype=np.uint64).reshape(4)
    ctx._check(ctx.lib.bz_best_fft(ctx.h, field, _np_ptr(a), _np_ptr(omega), log_n))
    return a


def lagrange_to_coeff(ctx, field, a, k):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4).copy()
    assert len(a) == 1 << k
    ctx._check(ctx.lib.bz_lagrange_to_coeff(ctx.h, field, _np_ptr(a), k))
    return a


def coeff_to_extended(ctx, field, a, k, extended_k):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
    assert len(a) == 1 << k
    out = np.empty((1 << extended_k, 4), dtype=np.uint64)
    ctx._check(ctx.lib.bz_coeff_to_extended(ctx.h, field, _np_ptr(a), _np_ptr(out), k, extended_k))
    return out


def extended_to_coeff(ctx, field, a, extended_k):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4).copy()
    assert len(a) == 1 << extended_k
    ctx._check(ctx.lib.bz_extended_to_coeff(ctx.h, field, _np_ptr(a), extended_k))
    return a


def batch_invert_assigned(ctx, field, numerators, denominators):
    """poly::batch_invert_assigned on one column (or any flat slice): Assigned<F> = numerator / denominator -> F, with
    ff::BatchInvert semantics (denominator 0 -> 0).  U: halo2_proofs 0.2.0 src/poly.rs."""
    num = np.ascontiguousarray(numerators, dtype=np.uint64).reshape(-1, 4)
    den = np.ascontiguousarray(denominators, dtype=np.uint64).reshape(-1, 4)
    assert len(num) == len(den)
    out = np.empty_like(num)
    ctx._check(ctx.lib.bz_batch_invert_assigned(ctx.h, field, _np_ptr(num), _np_ptr(den), _np_ptr(out), len(num)))
    return out


_FIELD_OPS = {"mul": 0, "add": 1, "sub": 2, "inv": 3, "from_u512": 4, "from_mont": 5, "to_mont": 6, "neg": 7, "sqr": 8, "inv_gcd": 9}


def field_op(ctx, field, op, a, b=None):
    """Element-wise ff::Field operation on slices (see bz_field_op)."""
    code = _FIELD_OPS[op]
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 8 if code == 4 else 4)
    n = len(a)
    if b is None:
        b = np.zeros((n, 4), dtype=np.uint64)
    b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 4)
    out = np.empty((n, 4), dtype=np.uint64)
    ctx._check(ctx.lib.bz_field_op(ctx.h, field, code, _np_ptr(a), _np_ptr(b), _np_ptr(out), n))
    return out


_CURVE_OPS = {"add": 0, "double": 1, "sub": 2, "double_add": 3, "mul_u32": 4}


def curve_op(ctx, curve, op, a, b):
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 8)
    b = np.ascontiguousarray(b, dtype=np.uint64).reshape(-1, 8)
    out = np.empty_like(a)
    ctx._check(ctx.lib.bz_curve_op(ctx.h, curve, _CURVE_OPS[op], _np_ptr(a), _np_ptr(b), _np_ptr(out), len(a)))
    return out


def hash_to_curve(ctx, curve, domain_prefix, messages):
    """pasta `C::hash_to_curve(domain_prefix)` over equal-length byte messages -> (count, 8) uint64 Montgomery affine."""
    msgs = [bytes(m) for m in messages]
    L = len(msgs[0]) if msgs else 0
    assert all(len(m) == L for m in msgs)
    buf = np.frombuffer(b"".join(msgs) or b"\0", dtype=np.uint8).copy()
    out = np.zeros((len(msgs), 8), dtype=np.uint64)
    ctx._check(ctx.lib.bz_hash_to_curve(ctx.h, curve, domain_prefix.encode(), _np_ptr(buf), L, len(msgs), _np_ptr(out)))
    return out


def chacha20_blocks(ctx, seeds, blocks, out=None):
    """ChaCha20 keystream blocks 0 .. blocks-1 of every 32-byte seed (bz_chacha20_blocks): seeds = (B, 32) uint8 or a list of
    32-byte strings.  Returns (B, blocks, 8) uint64 -- rand_wide's layout, the words create_proof's Scalar::random draws read.
    out: optional device address (int) of B x blocks x 64 bytes to write instead; then nothing is returned."""
    seeds = _seed_array(seeds)
    if out is not None:
        ctx._check(ctx.lib.bz_chacha20_blocks(ctx.h, _np_ptr(seeds), len(seeds), blocks, ctypes.c_void_p(int(out))))
        return None
    res = np.empty((len(seeds), blocks, 8), dtype=np.uint64)
    ctx._check(ctx.lib.bz_chacha20_blocks(ctx.h, _np_ptr(seeds), len(seeds), blocks, _np_ptr(res)))
    return res


def params_new(ctx, k, curve=0):
    """`Params::new(k)` on the device -> dict(g, g_lagrange: (n, 8); w, u: (8,)) of Montgomery affine points."""
    n = 1 << k
    g, gl = np.zeros((n, 8), dtype=np.uint64), np.zeros((n, 8), dtype=np.uint64)
    w, u = np.zeros(8, dtype=np.uint64), np.zeros(8, dtype=np.uint64)
    ctx._check(ctx.lib.bz_params_new(ctx.h, k, curve, _np_ptr(g), _np_ptr(gl), _np_ptr(w), _np_ptr(u)))
    return {"g": g, "g_lagrange": gl, "w": w, "u": u}


def points_compress(ctx, curve, affine):
    """(n, 8) uint64 Montgomery affine -> n x 32 bytes (pasta `to_bytes`)."""
    affine = np.ascontiguousarray(affine, dtype=np.uint64).reshape(-1, 8)
    out = np.zeros((len(affine), 32), dtype=np.uint8)
    ctx._check(ctx.lib.bz_points_compress(ctx.h, curve, _np_ptr(affine), len(affine), _np_ptr(out)))
    return out


def points_decompress(ctx, curve, data):
    """n x 32 bytes -> ((n, 8) uint64 Montgomery affine, status (n,) uint8: 0 ok, 1 identity, 2 invalid)."""
    buf = np.frombuffer(bytes(data), dtype=np.uint8).reshape(-1, 32).copy()
    out = np.zeros((len(buf), 8), dtype=np.uint64)
    st = np.zeros(len(buf), dtype=np.uint8)
    ctx._check(ctx.lib.bz_points_decompress(ctx.h, curve, _np_ptr(buf), len(buf), _np_ptr(out), _np_ptr(st)))
    return out, st


def params_write(ctx, urs, k, curve=0):
    """`Params::write`: k as u32 LE, then g, g_lagrange (2^k points each), w, u in pasta's compressed encoding."""
    pts = np.concatenate([urs["g"], urs["g_lagrange"], urs["w"][None, :], urs["u"][None, :]])
    return int(k).to_bytes(4, "little") + points_compress(ctx, curve, pts).tobytes()


def params_read(ctx, data, curve=0):
    """`Params::read`: inverse of params_write; raises ValueError on a malformed stream (io::Error upstream)."""
    if len(data) < 4:
        raise ValueError("Params::read: truncated")
    k = int.from_bytes(data[:4], "little")
    if k > 24 or len(data) != 4 + 32 * (2 * (1 << k) + 2):
        raise ValueError("Params::read: wrong length for k")
    n = 1 << k
    pts, st = points_decompress(ctx, curve, data[4:])
    if (st == 2).any():
        raise ValueError("Params::read: invalid point encoding")
    return k, {"g": pts[:n].copy(), "g_lagrange": pts[n:2 * n].copy(), "w": pts[2 * n].copy(), "u": pts[2 * n + 1].copy()}


# ---- fine-grained prover arithmetic (include/bzhalo2.h "Fine-grained prover arithmetic"; SURVEY 8b) -------------------
def _ptr_array(arrs):
    arrs = [np.ascontiguousarray(a, dtype=np.uint64) for a in arrs]
    ptrs = (ctypes.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
    return arrs, ptrs


def _scalar(x):
    return np.ascontiguousarray(x, dtype=np.uint64).reshape(4)


def eval_polynomials(ctx, field, polys, points):
    """arithmetic::eval_polynomial for many (poly, point) pairs: polys = list of (n,4) arrays, points = (count,4)."""
    keep, ptrs = _ptr_array(polys)
    points = np.ascontiguousarray(points, dtype=np.uint64).reshape(-1, 4)
    assert len(points) == len(keep)
    out = np.zeros((len(keep), 4), dtype=np.uint64)
    ctx._check(ctx.lib.bz_eval_many(ctx.h, field, len(keep[0]) if keep else 0, len(keep), ptrs, _np_ptr(points), _np_ptr(out)))
    return out


def kate_division(ctx, field, a, point):
    """arithmetic::kate_division(a, b) -> n - 1 coefficients."""
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4)
    out = np.zeros((len(a) - 1, 4), dtype=np.uint64)
    ctx._check(ctx.lib.bz_kate_div(ctx.h, field, len(a), _np_ptr(a), _np_ptr(_scalar(point)), _np_ptr(out)))
    return out


def axpy(ctx, field, acc, x, poly):
    """acc * x + poly (returned; multiopen's accumulation step)."""
    acc = np.ascontiguousarray(acc, dtype=np.uint64).reshape(-1, 4).copy()
    poly = np.ascontiguousarray(poly, dtype=np.uint64).reshape(-1, 4)
    assert len(acc) == len(poly)
    ctx._check(ctx.lib.bz_axpy(ctx.h, field, len(acc), _np_ptr(acc), _np_ptr(_scalar(x)), _np_ptr(poly)))
    return acc


def divide_by_vanishing_poly(ctx, field, a, k, extended_k):
    """EvaluationDomain::divide_by_vanishing_poly on 2^extended_k extended-Lagrange values (returned)."""
    a = np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4).copy()
    assert len(a) == 1 << extended_k
    ctx._check(ctx.lib.bz_divide_by_vanishing(ctx.h, field, k, extended_k, _np_ptr(a)))
    return a


def permutation_product(ctx, field, k, values, sigmas, beta, gamma, delta_omega0, z0):
    """permutation::Argument::commit for one column set -> z (n,4) before blinding."""
    vk, vp = _ptr_array(values)
    sk, sp = _ptr_array(sigmas)
    out = np.zeros((1 << k, 4), dtype=np.uint64)
    ctx._check(ctx.lib.bz_perm_product(ctx.h, field, k, len(vk), vp, sp, _np_ptr(_scalar(beta)), _np_ptr(_scalar(gamma)),
                                       _np_ptr(_scalar(delta_omega0)), _np_ptr(_scalar(z0)), _np_ptr(out)))
    return out


def lookup_permute(ctx, field, k, usable_rows, compressed_input, compressed_table):
    """lookup::permute_expression_pair -> (permuted_input, permuted_table), rows >= usable_rows zero."""
    ci = np.ascontiguousarray(compressed_input, dtype=np.uint64).reshape(-1, 4)
    ct = np.ascontiguousarray(compressed_table, dtype=np.uint64).reshape(-1, 4)
    assert len(ci) == len(ct) == 1 << k
    a, s = np.zeros_like(ci), np.zeros_like(ci)
    ctx._check(ctx.lib.bz_lookup_permute(ctx.h, field, k, usable_rows, _np_ptr(ci), _np_ptr(ct), _np_ptr(a), _np_ptr(s)))
    return a, s


def lookup_product(ctx, field, k, compressed_input, compressed_table, permuted_input, permuted_table, beta, gamma):
    """lookup::Permuted::commit_product -> z (n,4) before blinding."""
    arrs = [np.ascontiguousarray(a, dtype=np.uint64).reshape(-1, 4) for a in (compressed_input, compressed_table, permuted_input, permuted_table)]
    assert all(len(a) == 1 << k for a in arrs)
    out = np.zeros((1 << k, 4), dtype=np.uint64)
    ctx._check(ctx.lib.bz_lookup_product(ctx.h, field, k, *[_np_ptr(a) for a in arrs], _np_ptr(_scalar(beta)), _np_ptr(_scalar(gamma)), _np_ptr(out)))
    return out
