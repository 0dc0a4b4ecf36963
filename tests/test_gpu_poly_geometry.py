"""The polynomial layer's kernels against the oracle at every launch geometry they pick, on both fields, through the
fine-grained C ABI (arithmetic.py).  The kernels choose their geometry from the input length: the grand-product scan goes
two-level above 8 tiles (n > 16 384) and reaches ntiles == SCAN_TILE at n = 2^22; Horner evaluation and Kate division split
into n / 16 384 slices from n = 32 768 on, with uneven slices and per-thread chunks at lengths that are not powers of two;
the lookup permutation leaves shared memory for CUB above n = 4 096.  Proofs only ever reach power-of-two lengths, Fp and
honest circuit data, so every case here is also one a proof does not run: Fq, odd lengths, zero numerators and
denominators in the grand products, duplicate-heavy lookup tables.  Every device result is compared bit for bit with
the oracle's restatement of the same halo2 loop (oracle/halo2.py, oracle/vec.py) or, for the vanishing division, with
halo2's formula in Python integers."""
import random
import numpy as np
import pytest
from battlezips_halo2_b200 import arithmetic as ar
from battlezips_halo2_b200.binding import BzError, _np_ptr
from oracle import c_oracle as co, halo2 as H
from oracle.domain import EvaluationDomain
from oracle.vec import Vec

pytestmark = pytest.mark.gpu

FIELD_NAME = {0: "Fp", 1: "Fq"}
ERR_INVALID, ERR_UNSUPPORTED, ERR_SYNTHESIS = -1, -3, -4


def _rand(f, n, seed):
    """n random field elements (Montgomery limbs) from a seed: any 254-bit value is below p and a valid representation."""
    a = np.random.default_rng(seed).integers(0, 2**64, size=(n, 4), dtype=np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a


def _omega(f, k):
    """The 2^k-th root of unity halo2 uses for a domain of 2^k rows."""
    F = co.FIELDS[f]
    return pow(F.root_of_unity, 1 << (32 - k), F.p)


def _mismatch(got, exp):
    bad = np.flatnonzero((got != exp).any(axis=1))
    return f"{len(bad)} of {len(exp)} rows differ, first at {bad[:4].tolist()}"


def _zero_from(z, row):
    """z is non-zero on rows 0..row and zero after: the shape a zero factor at `row` gives the grand product."""
    nz = z.any(axis=1)
    return nz[:row + 1].all() and not nz[row + 1:].any()


def _row(case, n):
    return {"first": 0, "mid": (5 * n) // 8, "last": n - 1}[case.rsplit("_", 1)[1]]


# ---- permutation grand product ---------------------------------------------------------------------------------------
# k = 14 / 15 is the single-CTA / two-level scan edge, k = 22 has exactly SCAN_TILE tiles
_PERM_NCOLS = {1: 2, 2: 8, 3: 5, 11: 4, 14: 3, 15: 2, 17: 3, 22: 2}
_GP_ZERO_CASES = ("num_zero_mid", "den_zero_first", "den_zero_mid", "den_zero_last")


def _perm_params():
    out = []
    for f in (0, 1):
        out += [pytest.param(f, 3, c, "random", id=f"{FIELD_NAME[f]}-n8-c{c}-random") for c in range(1, 9)]
        for k, c in _PERM_NCOLS.items():
            for case in (("den_zero_last", "num_zero_mid") if k == 22 else _GP_ZERO_CASES):
                out.append(pytest.param(f, k, c, case, id=f"{FIELD_NAME[f]}-n{1 << k}-c{c}-{case}"))
    return out


@pytest.mark.parametrize("f,k,ncols,case", _perm_params())
def test_permutation_product(f, k, ncols, case, ctx):
    """bz_perm_product against the restated permutation::Argument::commit, with delta_omega0 and z0 != 1.  A zero
    numerator v = -(beta delta^j delta_omega0 omega^i + gamma) or a zero denominator v = -(beta sigma + gamma) at row i
    leaves z non-zero up to row i and zero after it (halo2's batch_invert maps 1/0 to 0); at the last row it changes
    nothing, so that case checks the whole scan on a z that is non-zero everywhere."""
    V, n = Vec(f), 1 << k
    p = V.p
    seed = (f * 32 + k) * 16 + ncols
    beta, gamma, d0, z0 = (V.int1(x) for x in _rand(f, 4, seed))
    values = [_rand(f, n, seed * 32 + j) for j in range(ncols)]
    sigmas = [_rand(f, n, seed * 32 + 16 + j) for j in range(ncols)]
    omega = _omega(f, k)
    if case != "random":
        row, j = _row(case, n), ncols - 1
        if case.startswith("num"):
            v = -(beta * d0 * pow(V.F.delta, j, p) * pow(omega, row, p) + gamma)
        else:
            v = -(beta * V.int1(sigmas[j][row]) + gamma)
        values[j][row] = V.m(v)
    exp = H.permutation_product(V, omega, values, sigmas, beta, gamma, d0, z0)
    if case != "random":
        assert _zero_from(exp, n - 1 if case == "den_zero_last" else _row(case, n))
    got = ar.permutation_product(ctx, f, k, values, sigmas, V.m(beta), V.m(gamma), V.m(d0), V.m(z0))
    assert np.array_equal(got, exp), _mismatch(got, exp)


# ---- lookup grand product --------------------------------------------------------------------------------------------
def _lookup_params():
    out = []
    for f in (0, 1):
        for k in _PERM_NCOLS:
            for case in (("den_zero_last", "num_zero_mid") if k == 22 else _GP_ZERO_CASES):
                out.append(pytest.param(f, k, case, id=f"{FIELD_NAME[f]}-n{1 << k}-{case}"))
    return out


@pytest.mark.parametrize("f,k,case", _lookup_params())
def test_lookup_product(f, k, case, ctx):
    """bz_lookup_product against the restated lookup::Permuted::commit_product, with a zero factor on the numerator side
    (compressed table = -gamma) or on the denominator side (permuted input = -beta, permuted table = -gamma)."""
    V, n = Vec(f), 1 << k
    seed = 7000 + f * 32 + k
    beta, gamma = (V.int1(x) for x in _rand(f, 2, seed))
    cols = [_rand(f, n, seed * 8 + j) for j in range(4)]          # compressed input, compressed table, A', S'
    row = _row(case, n)
    if case.startswith("num"):
        cols[1][row] = V.m(-gamma)
    elif case == "den_zero_mid":
        cols[3][row] = V.m(-gamma)
    else:
        cols[2][row] = V.m(-beta)
    exp = H.lookup_product(V, *cols, beta, gamma)
    assert _zero_from(exp, n - 1 if case == "den_zero_last" else row)
    got = ar.lookup_product(ctx, f, k, *cols, V.m(beta), V.m(gamma))
    assert np.array_equal(got, exp), _mismatch(got, exp)


# ---- Horner evaluation -----------------------------------------------------------------------------------------------
# 16 384 / 32 768 is the single-CTA / split edge; 32 769, 49 151 and 2^20 + 1 leave the last slice short
_EVAL_N = [1, 2, 127, 128, 129, 16383, 32767, 32768, 32769, 49151, 49152, (1 << 20) + 1, 1 << 22]


def _points(f, n):
    """0, 1, p - 1, the root of unity of the smallest power-of-two domain holding n, and a random point."""
    p = co.FIELDS[f].p
    return [0, 1, p - 1, _omega(f, max(1, (n - 1).bit_length())), Vec(f).int1(_rand(f, 1, 11 * n + f)[0])]


@pytest.mark.parametrize("n", _EVAL_N, ids=lambda n: f"n{n}")
@pytest.mark.parametrize("f", [0, 1], ids=FIELD_NAME.get)
def test_eval_polynomials(f, n, ctx):
    """bz_eval_many against arithmetic::eval_polynomial for a random, a zero and an all-(p - 1) polynomial at every
    point of _points, in one call.  The random polynomial is passed under two host pointers (one a copy) and each
    pointer several times, in an order that does not follow the upload slots."""
    V = Vec(f)
    rnd = _rand(f, n, 3 * n + f)
    polys = [rnd, V.zeros(n), V.const(V.p - 1, n), rnd.copy()]
    queries = [(i, pt) for j, pt in enumerate(_points(f, n)) for i in ((j + t) % 4 for t in range(4))]
    got = ar.eval_polynomials(ctx, f, [polys[i] for i, _ in queries], np.stack([V.m(pt) for _, pt in queries]))
    ref = {}
    for i, pt in queries:
        if (i % 3, pt) not in ref:                                   # polys[3] is a copy of polys[0]
            ref[(i % 3, pt)] = V.eval_polynomial(polys[i], pt)
    exp = np.stack([V.m(ref[(i % 3, pt)]) for i, pt in queries])
    assert np.array_equal(got, exp), _mismatch(got, exp)


@pytest.mark.parametrize("n", [129, 32769], ids=lambda n: f"n{n}")
@pytest.mark.parametrize("f", [0, 1], ids=FIELD_NAME.get)
def test_eval_polynomials_many_queries(f, n, ctx):
    """300 (polynomial, point) queries over 7 polynomials in one bz_eval_many call, single-CTA and split."""
    V = Vec(f)
    polys = [_rand(f, n, 100 * n + 10 * f + s) for s in range(7)]
    which = np.random.default_rng(n + f).integers(0, 7, size=300)
    pts = _rand(f, 300, 5 * n + f)
    got = ar.eval_polynomials(ctx, f, [polys[i] for i in which], pts)
    exp = np.stack([V.m(V.eval_polynomial(polys[i], V.int1(pt))) for i, pt in zip(which, pts)])
    assert np.array_equal(got, exp), _mismatch(got, exp)


# ---- Kate division ---------------------------------------------------------------------------------------------------
# 2, 255, 256, 257: threads with empty and with short chunks of the 256-thread CTA
@pytest.mark.parametrize("n", sorted(set(_EVAL_N) | {2, 255, 256, 257}), ids=lambda n: f"n{n}")
@pytest.mark.parametrize("f", [0, 1], ids=FIELD_NAME.get)
def test_kate_division(f, n, ctx):
    """bz_kate_div against arithmetic::kate_division at the points 0, 1, p - 1 and a random one."""
    V = Vec(f)
    a = _rand(f, n, 13 * n + f)
    for pt in _points(f, n)[:3] + _points(f, n)[4:]:
        got = ar.kate_division(ctx, f, a, V.m(pt))
        exp = V.kate_division(a, pt)
        assert np.array_equal(got, exp), (pt, _mismatch(got, exp))


# ---- multiopen accumulation ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 127, 129, (1 << 20) + 3], ids=lambda n: f"n{n}")
@pytest.mark.parametrize("f", [0, 1], ids=FIELD_NAME.get)
def test_axpy(f, n, ctx):
    """bz_axpy: acc * x + poly for x = 0, 1, p - 1."""
    V = Vec(f)
    acc, poly = _rand(f, n, 17 * n + f), _rand(f, n, 19 * n + f)
    for x in (0, 1, V.p - 1):
        got = ar.axpy(ctx, f, acc, V.m(x), poly)
        exp = V.add(V.scale(acc, x), poly)
        assert np.array_equal(got, exp), (x, _mismatch(got, exp))


# ---- division by the vanishing polynomial ----------------------------------------------------------------------------
@pytest.mark.parametrize("k,d", [(2, 1), (2, 2), (2, 3), (2, 4), (2, 8), (2, 16), (20, 3)], ids=lambda v: str(v))
@pytest.mark.parametrize("f", [0, 1], ids=FIELD_NAME.get)
def test_divide_by_vanishing_poly(f, k, d, ctx):
    """bz_divide_by_vanishing at extended_k = k + d against halo2's formula in integers,
    a[i] * (zeta^n * omega_ext^(n i) - 1)^-1 with i taken mod 2^d, cross-checked with EvaluationDomain of degree 2^d + 1
    (the constraint-system degree that gives this extended_k)."""
    F = co.FIELDS[f]
    p, ek = F.p, k + d
    a = _rand(f, 1 << ek, 23 * ek + f)
    cur, step = pow(F.zeta, 1 << k, p), pow(_omega(f, ek), 1 << k, p)
    t = []
    for _ in range(1 << d):
        t.append(pow((cur - 1) % p, -1, p))
        cur = cur * step % p
    exp = co.field_mul(f, a, np.ascontiguousarray(co.to_mont(f, t)[np.arange(1 << ek) % (1 << d)]))
    if k < 20:
        dom = EvaluationDomain(f, (1 << d) + 1, k)
        assert dom.extended_k == ek and np.array_equal(dom.divide_by_vanishing_poly(a), exp)
    got = ar.divide_by_vanishing_poly(ctx, f, a, k, ek)
    assert np.array_equal(got, exp), _mismatch(got, exp)


# ---- lookup permutation ----------------------------------------------------------------------------------------------
# k = 12 is the largest domain of the shared-memory kernel, k = 13 the first of the CUB path
_LKP_K = [1, 5, 12, 13, 17]
_LKP_CASES = ["dups", "input_const", "table_const", "perm", "zero_pm1", "missing"]


def _usables(n):
    return sorted({0, 1, n - 1, n} | ({n - 10} if n > 10 else set()))


def _lookup_columns(case, n, usable, rng, p):
    """Compressed input / table (canonical ints) for one case.  Input rows >= usable always hold values that are in
    no table row: halo2 ignores them.  `missing` puts an input value only in table rows >= usable."""
    fresh = lambda: rng.randrange(2**64, p)                        # never one of the small values below
    if case == "table_const":
        c = fresh()
        table = [c] * n
    elif case == "perm":
        table = [fresh() for _ in range(n)]                        # all distinct (with overwhelming probability)
    elif case == "zero_pm1":
        table = [rng.choice([0, p - 1, 1, 2]) for _ in range(n)]
    else:                                                          # heavy duplicates, 0 and p - 1 among them
        distinct = [0, p - 1] + [fresh() for _ in range(max(1, n // 16))]
        table = [rng.choice(distinct) for _ in range(n)]
    pool = table[:usable]
    if case == "perm":
        inputs = rng.sample(pool, usable)
    elif case == "input_const":
        inputs = [table[0]] * usable
    else:
        inputs = [rng.choice(pool) for _ in range(usable)]
    if case == "missing":
        x = fresh()
        table[usable] = x
        inputs[rng.randrange(usable)] = x
    return inputs + [fresh() for _ in range(n - usable)], table


@pytest.mark.parametrize("case", _LKP_CASES)
@pytest.mark.parametrize("k", _LKP_K, ids=lambda k: f"Fp-n{1 << k}")
def test_lookup_permute(k, case, ctx):
    """bz_lookup_permute against the restated permute_expression_pair for usable = 0, 1, n - 10, n - 1, n: A' and S' on the
    usable rows, zero on the others; an input value found only in table rows >= usable is BZ_ERR_SYNTHESIS."""
    V, n = Vec(0), 1 << k
    rng = random.Random(k * 100 + _LKP_CASES.index(case))
    for usable in _usables(n):
        if case in ("input_const", "table_const") and usable == 0 or case == "missing" and not 0 < usable < n:
            continue
        inputs, table = _lookup_columns(case, n, usable, rng, V.p)
        cin, ctab = V.arr(inputs), V.arr(table)
        if case == "missing":
            with pytest.raises(ValueError, match="ConstraintSystemFailure"):
                H.permute_expression_pair(V, usable, cin, ctab)
            with pytest.raises(BzError) as e:
                ar.lookup_permute(ctx, 0, k, usable, cin, ctab)
            assert e.value.code == ERR_SYNTHESIS, usable
            continue
        ea, es = H.permute_expression_pair(V, usable, cin, ctab)
        a, s = ar.lookup_permute(ctx, 0, k, usable, cin, ctab)
        assert np.array_equal(a[:usable], ea) and not a[usable:].any(), (usable, _mismatch(a[:usable], ea))
        assert np.array_equal(s[:usable], es) and not s[usable:].any(), (usable, _mismatch(s[:usable], es))


# ---- rejections ------------------------------------------------------------------------------------------------------
def _code(fn):
    with pytest.raises(BzError) as e:
        fn()
    return e.value.code, str(e.value)


def test_rejections_are_clean_errors(ctx):
    """Out-of-range arguments come back as error codes, and the context keeps working after each."""
    V = Vec(0)
    one, col = V.m(1), V.zeros(8)
    _, ptrs = ar._ptr_array([col])
    out = V.zeros(8)
    assert ctx.lib.bz_perm_product(ctx.h, 0, 3, 0, ptrs, ptrs, _np_ptr(one), _np_ptr(one), _np_ptr(one), _np_ptr(one), _np_ptr(out)) == ERR_UNSUPPORTED
    assert _code(lambda: ar.permutation_product(ctx, 0, 3, [col] * 9, [col] * 9, one, one, one, one))[0] == ERR_UNSUPPORTED
    big = V.zeros(1 << 23)
    code, msg = _code(lambda: ar.permutation_product(ctx, 0, 23, [big], [big], one, one, one, one))
    assert code == ERR_INVALID and "two-level scan" in msg, msg
    del big
    assert _code(lambda: ar.lookup_permute(ctx, 1, 3, 8, col, col))[0] == ERR_UNSUPPORTED
    assert _code(lambda: ar.lookup_permute(ctx, 0, 3, 9, col, col))[0] == ERR_INVALID
    assert _code(lambda: ar.divide_by_vanishing_poly(ctx, 0, col, 3, 3))[0] == ERR_INVALID
    assert _code(lambda: ar.divide_by_vanishing_poly(ctx, 0, col[:4], 3, 2))[0] == ERR_INVALID
    assert ctx.lib.bz_eval_many(ctx.h, 0, 0, 1, ptrs, _np_ptr(one), _np_ptr(out)) == ERR_INVALID
    assert ctx.lib.bz_kate_div(ctx.h, 0, 0, _np_ptr(col), _np_ptr(one), _np_ptr(out)) == ERR_INVALID
    a = _rand(0, 8, 1)
    assert np.array_equal(ar.kate_division(ctx, 0, a, V.m(5)), V.kate_division(a, 5))
