"""The gather pipeline of the table MSM's accumulation (fixedmsm.cu `fb_accumulate_kernel`) at its stage boundaries.

Each thread of the accumulation wave stages the table points of its next FB_STAGES entries in shared memory (cp.async,
one commit group per entry; a piece starts with FB_STAGES copies in flight and ends with none).  The entries of all
MSMs of a launch form one flat index space cut into ranges of 32 q entries, one per warp; q is the minimum share, 16,
whenever the launch holds at most 16 entries per resident thread (every launch here: fewer than 50 000 entries against
at least 16 x 128 x the SM count).  Inside a warp's range every MSM is one piece, and lane l of a piece of L entries
adds ceil((L - l) / 32) of them.  So the entry count of each MSM decides exactly which per-lane piece lengths a launch
runs, and the scalars below are built to hit given entry counts:

  - pieces whose lanes add 0, 1, ..., 9 entries, each piece starting at a warp's first entry: the lengths around every
    stage boundary (0 .. S + 2) of a pipeline up to S = 7 deep (the kernel ships S = 1);
  - after each of them, in the same warp's range, a piece of the next MSM that fills the range (two MSMs per warp);
  - MSMs without entries between them;
  - launches with fewer entries than the wave has threads, and one without any entry.

Every commitment is compared bit for bit with the oracle's best_multiexp over g || w."""
import random
import numpy as np
import pytest
from tests.util_msm import modulus, oracle_msms, recode, urs_points

K = 5
N = 1 << K
MAX_LANE_LEN = 9
Q = 16                         # FB_MIN_SHARE: entries per lane of a full warp range
RANGE = 32 * Q


def _scalar_with_digits(rnd, c, t, exact):
    """A canonical scalar with t non-zero windows among the windows below bit 252.  exact: raw digits 1 .. 2^(c-1)
    (positive, no carries: exactly t signed digits); otherwise raw digits 1 .. 2^c - 1 (negative digits and carries
    too: the digit count is whatever recode gives)."""
    W = (256 + c - 1) // c
    usable = [w for w in range(W) if (w + 1) * c <= 252]
    hi = (1 << (c - 1)) if exact else (1 << c) - 1
    return sum(rnd.randint(1, hi) << (w * c) for w in rnd.sample(usable, t))


def _msm_with_entries(rnd, c, entries):
    """N + 1 canonical scalars (polynomial || blind) whose signed recoding at width c has exactly `entries` non-zero
    digits, spread over random positions, with negative digits among them."""
    W = (256 + c - 1) // c
    tmax = len([w for w in range(W) if (w + 1) * c <= 252])
    scalars, left = [], entries
    while left > tmax:
        s = _scalar_with_digits(rnd, c, rnd.randint(tmax // 2, tmax), exact=False)
        d = sum(1 for v in recode(s, c)[0] if v)
        if d <= left:
            scalars.append(s)
            left -= d
    if left:
        scalars.append(_scalar_with_digits(rnd, c, left, exact=True))
    assert len(scalars) <= N + 1
    out = [0] * (N + 1)
    for pos, s in zip(rnd.sample(range(N + 1), len(scalars)), scalars):
        out[pos] = s
    assert sum(1 for s in out for v in recode(s, c)[0] if v) == entries
    return out


def lane_lengths(entry_counts):
    """{per-lane entry count of a piece} over all pieces of a launch of MSMs with these entry counts (q = Q)."""
    seen, off = set(), 0
    for e in entry_counts:
        lo, hi = off, off + e
        while lo < hi:
            end = min(hi, (lo // RANGE + 1) * RANGE)
            seen.update(-(-(end - lo - l) // 32) if end - lo > l else 0 for l in range(32))
            lo = end
        off = hi
    return seen


def _layouts():
    """{name: entry counts of the MSMs of one launch}"""
    aligned = []
    for j in range(MAX_LANE_LEN):              # lanes of the piece add j or j + 1 entries
        for r in (0, 1, 17, 31):
            L = 32 * j + r
            aligned += [L, 0, RANGE - L] if L else [0, RANGE]
    return {
        # every piece starts at a warp's first entry; its per-lane counts cover 0 .. MAX_LANE_LEN
        "stage_boundaries": aligned,
        # MSMs that start and end anywhere inside warp ranges, and span several
        "unaligned": [3, 70, 0, 0, 129, 1, 511, 513, 0, 95, 1100, 33, 0, 64, 7],
        # fewer entries than threads in the wave: one warp works, most of its lanes stage nothing
        "tiny": [1, 0, 2, 5, 0],
        "one_entry": [1],
        "empty": [0, 0, 0],
    }


def test_layouts_reach_the_stage_boundaries():
    """The per-lane piece lengths the launches below run (CPU check of the construction)."""
    got = lane_lengths(_layouts()["stage_boundaries"])
    assert set(range(MAX_LANE_LEN + 1)) <= got, sorted(got)
    assert {0, 1} <= lane_lengths(_layouts()["tiny"])


@pytest.mark.gpu
@pytest.mark.parametrize("curve,c", [(0, 4), (1, 5)])
def test_fb_pipeline_stage_boundaries(curve, c, ctx, oracle_c):
    from battlezips_halo2_b200.plonk import prover as PR
    co = oracle_c
    sf = co.CURVES[curve][1]
    urs = urs_points(ctx, co, curve, 2 * N + 2)
    g, w, u, gl = urs[:N], urs[N], urs[N + 1], urs[N + 2:]
    bases = np.concatenate([g, w[None]])
    rnd = random.Random(97 + 13 * curve + c)
    params = PR.Params(ctx, K, g, gl, w, u, curve=curve, window_bits=c)
    bad = []
    try:
        for name, counts in _layouts().items():
            msms = [_msm_with_entries(rnd, c, e) for e in counts]
            assert all(0 <= s < modulus(sf) for m in msms for s in m)
            enc = np.stack([co.to_mont(sf, m) for m in msms])
            exp = oracle_msms(co, curve, [(e, bases) for e in enc])
            d_p = ctx.to_device(np.ascontiguousarray(enc[:, :N]))
            d_b = ctx.to_device(np.ascontiguousarray(enc[:, N]))
            d_o = ctx.alloc(len(msms) * 64)
            try:
                params.commit_batch_dev(d_p.ptr, d_b.ptr, len(msms), d_o.ptr)
                got = d_o.download((len(msms), 8))
            finally:
                d_p.free(); d_b.free(); d_o.free()
            bad += [(name, j, counts[j]) for j in range(len(msms)) if not np.array_equal(got[j], exp[j])]
    finally:
        params.close()
    assert not bad, (f"c={c}", len(bad), bad[:8])
