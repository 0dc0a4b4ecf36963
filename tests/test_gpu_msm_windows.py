"""Both MSM engines against the oracle at every window width, on scalars at the digit boundaries of the signed recoding
(tests/util_msm.py) and in every launch shape:

  - the table MSM (fixedmsm.cu) through Params.commit at c = 4 .. 16, and through Params.commit_batch_dev across its
    chunk loop, both fold widths, the two-level fold and empty MSMs in the flat entry space;
  - the bucket MSM (msm.cu) through bz_msm_dev at window_bits = 2 .. 16 and at its own choice, on skewed scalars, and as
    the batched commit of Params built with BZ_FORCE_GENERAL_MSM=1;
  - bz_batch_normalize_dev (Jacobian -> affine).

Every point is compared bit for bit with the oracle's best_multiexp over the same bases, after to_affine.  A failure
names the family, the width and the shape."""
import os
import subprocess
import sys
import numpy as np
import pytest
import battlezips_halo2_b200 as bz
from tests.util_msm import AUTO_WINDOW_SIZES, FAMILIES, families, modulus, oracle_msms, urs_points

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

K5 = 5
N5 = 1 << K5


_URS = {}


def _urs(ctx, co, curve, n):
    """The first n URS points of a curve, computed once per module (grown when a test needs more)."""
    if curve not in _URS or len(_URS[curve]) < n:
        _URS[curve] = urs_points(ctx, co, curve, max(n, 4096))
    return _URS[curve][:n]


def _k5_bases(ctx, co, curve, degenerate):
    """g (32 points), w, u and a g_lagrange of 32 other points; with `degenerate`, g and g_lagrange hold a repeated, an
    opposite and an identity base and a base that appears three times."""
    urs = _urs(ctx, co, curve, 2 * N5 + 2)
    g, w, u, gl = urs[:N5].copy(), urs[N5], urs[N5 + 1], urs[N5 + 2:2 * N5 + 2].copy()
    if degenerate:
        C = co.CURVES[curve][0]
        for t in (g, gl):
            p0 = co.points_from_mont(curve, t[0][None])[0]
            t[1] = t[0]
            t[2] = co.points_to_mont(curve, [C.neg(p0)])[0]
            t[3] = 0
            t[9] = t[8]; t[10] = t[8]
    return g, w, u, gl


def _free(*bufs):
    for b in bufs:
        b.free()


# ---- 1. table MSM at every width ------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", range(4, 17))
@pytest.mark.parametrize("curve", [0, 1])
def test_table_msm_every_width(curve, c, ctx, oracle_c):
    """Params(k = 5, window_bits = c).commit(poly, blind) for every scalar family and both bases (lagrange).  Odd widths
    on Vesta and even widths on Pallas run over degenerate bases."""
    from battlezips_halo2_b200.plonk import prover as PR
    co = oracle_c
    sf = co.CURVES[curve][1]
    g, w, u, gl = _k5_bases(ctx, co, curve, degenerate=(c % 2 != curve))
    fams = families(sf, c, N5 + 1, seed=2 * c + curve)
    jobs, keys = [], []
    for lagrange in (False, True):
        bases = np.concatenate([gl if lagrange else g, w[None]])
        for label in FAMILIES:
            jobs.append((fams[label], bases))
            keys.append((label, lagrange))
    exp = oracle_msms(co, curve, jobs)
    bad = []
    params = PR.Params(ctx, K5, g, gl, w, u, curve=curve, window_bits=c)
    try:
        for (label, lagrange), e in zip(keys, exp):
            got = params.commit(fams[label][:N5], fams[label][N5], lagrange=lagrange)
            if not np.array_equal(got, e):
                bad.append((label, f"c={c}", f"lagrange={lagrange}"))
    finally:
        params.close()
    assert not bad, bad


# ---- 2. table MSM launch shapes ---------------------------------------------------------------------------------------
def _batch_inputs(co, curve, c, count, seed):
    """count polynomials of N5 scalars and count blinds: every fifth polynomial zero from the fifth on (empty MSMs between
    full ones), one with a single non-zero scalar, one of all r - 1, the rest from the families; every third blind zero."""
    sf = co.CURVES[curve][1]
    pool = families(sf, c, count * (N5 + 1), seed)
    polys = np.zeros((count, N5, 4), dtype=np.uint64)
    blinds = np.zeros((count, 4), dtype=np.uint64)
    labels = []
    for j in range(count):
        label = FAMILIES[j % len(FAMILIES)]
        chunk = pool[label][j * (N5 + 1):(j + 1) * (N5 + 1)]
        polys[j], blinds[j] = chunk[:N5], chunk[N5]
        if j % 5 == 4:
            polys[j] = 0; label = "zero"
        elif j == 1:
            polys[j] = 0; polys[j, 17] = pool["uniform"][0]; label = "single"
        elif j == 2:
            polys[j] = co.to_mont(sf, [modulus(sf) - 1])[0]; label = "minus_one"
        if j % 3 == 0:
            blinds[j] = 0
        labels.append(label)
    return polys, blinds, labels


def _commit_batch(cx, params, polys, blinds, count, lagrange, launches=None):
    """commit_batch_dev of the first count polynomials -> (count, 8) affine.  With `launches`, also asserts how many kernels
    the call launched: 3 per chunk of the table MSM (decode, accumulate, single-level fold), 4 with the two-level fold."""
    d_p, d_b, d_o = cx.to_device(polys[:count]), cx.to_device(blinds[:count]), cx.alloc(count * 64)
    try:
        before = cx.kernel_launches()
        params.commit_batch_dev(d_p.ptr, d_b.ptr, count, d_o.ptr, lagrange=lagrange)
        if launches is not None:
            assert cx.kernel_launches() - before == launches, (f"count={count}", "kernel launches", cx.kernel_launches() - before, launches)
        return d_o.download((count, 8))
    finally:
        _free(d_p, d_b, d_o)


def _check_batch(got, exp, labels, what):
    bad = [(j, labels[j]) for j in range(len(got)) if not np.array_equal(got[j], exp[j])]
    assert not bad, (what, len(bad), bad[:8])


@pytest.mark.parametrize("c", [4, 16])
def test_table_msm_launch_shapes(c, ctx, oracle_c):
    """commit_batch_dev at count 1, 2, 47, 48, 64, 65, 4 096 and 4 097 (the second pass of the chunk loop) with empty
    MSMs interleaved.  Vesta at c = 4, Pallas at c = 16.

    Which fold runs depends on how many threads the accumulation wave has.  On a B200 (4 resident CTAs per SM) every count up to 65 leaves each MSM enough thread partials for the two-level fold; 4 096 MSMs always fold in a
    single level, by the narrow fold (asserted through the launch count).  The single-level folds of fewer MSMs, the wide
    one among them, are tested by test_table_msm_single_level_fold_widths."""
    from battlezips_halo2_b200.plonk import prover as PR
    co = oracle_c
    curve = 0 if c == 4 else 1
    g, w, u, gl = _k5_bases(ctx, co, curve, degenerate=False)
    counts = [1, 2, 47, 48, 64, 65, 4096, 4097]
    polys, blinds, labels = _batch_inputs(co, curve, c, max(counts), seed=c)
    exp = {}
    for lagrange in (False, True):
        bases = np.concatenate([gl if lagrange else g, w[None]])
        exp[lagrange] = oracle_msms(co, curve, [(np.concatenate([polys[j], blinds[j][None]]), bases) for j in range(len(polys))])
    params = PR.Params(ctx, K5, g, gl, w, u, curve=curve, window_bits=c)
    try:
        for count in counts:
            for lagrange in (False, True):
                launches = 3 if count == 4096 else None
                got = _commit_batch(ctx, params, polys, blinds, count, lagrange, launches)
                _check_batch(got, exp[lagrange][:count], labels, (f"c={c}", f"count={count}", f"lagrange={lagrange}"))
    finally:
        params.close()


def _single_level_fold_child():
    """Body of test_table_msm_single_level_fold_widths, run in a process started with BZ_FB_CTAS_PER_SM=1."""
    from oracle import c_oracle as co
    from battlezips_halo2_b200.plonk import prover as PR
    ctx = bz.Context(0)
    for curve, c in ((0, 8), (1, 13)):
        g, w, u, gl = _k5_bases(ctx, co, curve, degenerate=(curve == 0))
        polys, blinds, labels = _batch_inputs(co, curve, c, 48, seed=48 + c)
        params = PR.Params(ctx, K5, g, gl, w, u, curve=curve, window_bits=c)
        for lagrange in (False, True):
            bases = np.concatenate([gl if lagrange else g, w[None]])
            exp = oracle_msms(co, curve, [(np.concatenate([polys[j], blinds[j][None]]), bases) for j in range(48)])
            for count in (20, 47, 48):
                got = _commit_batch(ctx, params, polys, blinds, count, lagrange, launches=3)
                _check_batch(got, exp[:count], labels, (f"c={c}", "1 CTA per SM", f"count={count}", f"lagrange={lagrange}"))
        params.close()
    ctx.close()
    print("single-level fold ok")


def test_table_msm_single_level_fold_widths():
    """The single-level folds of a batch of fewer than 4 096 MSMs: with one resident CTA per SM in the accumulation wave
    (BZ_FB_CTAS_PER_SM=1), 20 and 47 MSMs fold in one level with the wide fold (512 threads per MSM, fewer than 48 MSMs)
    and 48 MSMs with the narrow one.  The launch count shows that no two-level fold ran.  BZ_FB_CTAS_PER_SM is read once
    per process, so this runs in a child process."""
    env = dict(os.environ, BZ_FB_CTAS_PER_SM="1")
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + \
          ["-c", "from tests.test_gpu_msm_windows import _single_level_fold_child as f; f()"]
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "single-level fold ok" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]


# ---- 3. two-level fold ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve,c", [(1, 4), (0, 8)])
def test_table_msm_two_level_fold(curve, c, ctx, oracle_c):
    """k = 16: millions of table entries per call, so every thread of the accumulation wave holds more than the minimum
    share and the G slices of the two-level fold (fb_prefold_kernel) all fold real partials.  count 1, 3 and 16 (with an
    empty MSM) through commit_batch_dev -- the launch count shows the two-level fold ran -- and one commit."""
    from battlezips_halo2_b200.plonk import prover as PR
    co = oracle_c
    k, n = 16, 1 << 16
    sf = co.CURVES[curve][1]
    urs = _urs(ctx, co, curve, 2 * n + 2)
    g, w, u, gl = urs[:n], urs[n], urs[n + 1], urs[n + 2:2 * n + 2]
    fams = families(sf, c, n + 1, seed=k + c)
    order = ["uniform", "negatives", "witness", "edges", "half", "half_after_carry", "carry_chain"]
    polys = np.zeros((16, n, 4), dtype=np.uint64)
    blinds = np.zeros((16, 4), dtype=np.uint64)
    labels = []
    for j in range(16):
        label = order[j % len(order)]
        v = np.roll(fams[label], 977 * j, axis=0)              # repeated families still give distinct polynomials
        polys[j], blinds[j] = v[:n], v[n]
        if j == 11:
            polys[j] = 0; blinds[j] = 0; label = "zero"
        labels.append(label)
    bases = np.concatenate([g, w[None]])
    exp = np.stack([co.to_affine(curve, co.best_multiexp(curve, np.concatenate([polys[j], blinds[j][None]]), bases))[0]
                    for j in range(16)])
    params = PR.Params(ctx, k, g, gl, w, u, curve=curve, window_bits=c)
    try:
        for count in (1, 3, 16):
            got = _commit_batch(ctx, params, polys, blinds, count, lagrange=False, launches=4)
            _check_batch(got, exp[:count], labels, (f"c={c}", f"k={k}", f"count={count}"))
        got = params.commit(polys[1], blinds[1], lagrange=True)
        e = co.to_affine(curve, co.best_multiexp(curve, np.concatenate([polys[1], blinds[1][None]]), np.concatenate([gl, w[None]])))[0]
        assert np.array_equal(got, e), (labels[1], f"c={c}", f"k={k}", "commit lagrange")
    finally:
        params.close()


# ---- 4. / 5. bucket MSM -------------------------------------------------------------------------------------------------
def _msm_dev(ctx, co, curve, scalars, bases, window_bits):
    d_s, d_b, d_o = ctx.to_device(scalars), ctx.to_device(bases), ctx.alloc(96)
    try:
        ctx._check(ctx.lib.bz_msm_dev(ctx.h, curve, d_s.ptr, d_b.ptr, len(scalars), d_o.ptr, window_bits))
        return co.to_affine(curve, d_o.download(12))[0]
    finally:
        _free(d_s, d_b, d_o)


@pytest.mark.parametrize("c", range(2, 17))
@pytest.mark.parametrize("curve", [0, 1])
def test_bucket_msm_every_width(curve, c, ctx, oracle_c):
    """bz_msm_dev(window_bits = c) at n = 1, 33, 2 055 (and 2^14 at c = 2, 10, 15, 16) for every family; then 4 096 equal
    scalars (one bucket of 4 096 entries per window: the CTA-wide fold of oversized buckets) and 2 048 equal + 2 048
    uniform."""
    co = oracle_c
    sf = co.CURVES[curve][1]
    sizes = [1, 33, 2055] + ([1 << 14] if c in (2, 10, 15, 16) else [])
    cases = []
    for n in sizes:
        fams = families(sf, c, n, seed=n + c)
        cases += [(label, n, fams[label]) for label in FAMILIES]
    uni = families(sf, c, 4096, seed=c)["uniform"]
    cases.append(("equal", 4096, np.repeat(uni[:1], 4096, axis=0)))
    cases.append(("half_equal", 4096, np.concatenate([np.repeat(uni[:1], 2048, axis=0), uni[2048:]])))
    urs = _urs(ctx, co, curve, max(n for _, n, _ in cases))
    exp = oracle_msms(co, curve, [(s, urs[:n]) for _, n, s in cases])
    bad = [(label, f"c={c}", f"n={n}") for (label, n, s), e in zip(cases, exp)
           if not np.array_equal(_msm_dev(ctx, co, curve, s, urs[:n], c), e)]
    assert not bad, bad


def test_bucket_msm_window_bits_out_of_range(ctx, oracle_c):
    """window_bits outside 0 and 2 .. 16 is refused by the host-side argument check (nothing runs on the device)."""
    co = oracle_c
    urs = _urs(ctx, co, 0, 33)
    s = families(0, 4, 33, seed=1)["uniform"]
    for wb in (1, 17):
        with pytest.raises(bz.BzError):
            _msm_dev(ctx, co, 0, s, urs, wb)
    assert np.array_equal(_msm_dev(ctx, co, 0, s, urs, 2), oracle_msms(co, 0, [(s, urs)])[0])


@pytest.mark.parametrize("n", sorted(AUTO_WINDOW_SIZES))
@pytest.mark.parametrize("curve", [0, 1])
def test_bucket_msm_own_window(curve, n, ctx, oracle_c):
    """bz_msm_dev(window_bits = 0) at the edges of its window bands (tests/test_msm_digits.py pins n to c), uniform and
    negative scalars."""
    co = oracle_c
    c = AUTO_WINDOW_SIZES[n]
    fams = families(co.CURVES[curve][1], c, n, seed=n)
    urs = _urs(ctx, co, curve, n)
    for label in ("uniform", "negatives"):
        exp = co.to_affine(curve, co.best_multiexp(curve, fams[label], urs))[0]
        assert np.array_equal(_msm_dev(ctx, co, curve, fams[label], urs, 0), exp), (label, f"c={c}", f"n={n}")


# ---- 6. bucket path of the batched commit ------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [0, 1])
def test_general_msm_batched_commit(curve, ctx, oracle_c, monkeypatch):
    """Params built with BZ_FORCE_GENERAL_MSM=1 commit through msm_run_batch, 16 MSMs per chunk: count 1, 16, 17, 33."""
    from battlezips_halo2_b200.plonk import prover as PR
    co = oracle_c
    g, w, u, gl = _k5_bases(ctx, co, curve, degenerate=(curve == 1))
    polys, blinds, labels = _batch_inputs(co, curve, 4, 33, seed=50 + curve)
    monkeypatch.setenv("BZ_FORCE_GENERAL_MSM", "1")
    params = PR.Params(ctx, K5, g, gl, w, u, curve=curve)
    monkeypatch.delenv("BZ_FORCE_GENERAL_MSM")
    try:
        for lagrange in (False, True):
            bases = np.concatenate([gl if lagrange else g, w[None]])
            exp = oracle_msms(co, curve, [(np.concatenate([polys[j], blinds[j][None]]), bases) for j in range(33)])
            for count in (1, 16, 17, 33):
                got = _commit_batch(ctx, params, polys, blinds, count, lagrange)
                _check_batch(got, exp[:count], labels, ("general", f"count={count}", f"lagrange={lagrange}"))
    finally:
        params.close()


# ---- 7. bz_batch_normalize_dev ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 7, 1000])
@pytest.mark.parametrize("curve", [0, 1])
def test_batch_normalize_dev(curve, n, ctx, oracle_c):
    """Jacobian (x z^2, y z^3, z) of URS points with random z -- z = 1, z = p - 1, and some z = 0 (the identity, whatever
    x and y hold) -- back to affine, against the oracle's to_affine and the original points."""
    import random
    co = oracle_c
    bf = co.CURVES[curve][2]
    p = modulus(bf)
    aff = co.points_from_mont(curve, _urs(ctx, co, curve, n))
    rnd = random.Random(n * 2 + curve)
    zs = [rnd.randrange(1, p) for _ in range(n)]
    if n > 1:
        zs[1] = 0
    if n >= 7:
        zs[2], zs[3], zs[5] = 1, p - 1, 0
    flat = []
    for (x, y), z in zip(aff, zs):
        flat += [x * z * z % p, y * z * z * z % p, z] if z else [x, y, 0]
    jac = co.to_mont(bf, flat).reshape(n, 12)
    d_j, d_a = ctx.to_device(jac), ctx.alloc(n * 64)
    try:
        ctx._check(ctx.lib.bz_batch_normalize_dev(ctx.h, curve, d_j.ptr, d_a.ptr, n))
        got = d_a.download((n, 8))
    finally:
        _free(d_j, d_a)
    exp = co.to_affine(curve, jac)
    assert np.array_equal(got, exp)
    assert co.points_from_mont(curve, got) == [pt if z else None for pt, z in zip(aff, zs)]
