"""The scalar families of tests/util_msm.py against the recoding rule, on the CPU: they reconstruct, stay in range and
really reach the boundary cases at every window width, so a green GPU run of tests/test_gpu_msm_windows.py covers them.
Also pins the GPU test sizes to the window bands of the bucket MSM's cost model."""
import os, re, subprocess
import pytest
from tests.util_msm import (AUTO_WINDOW_SIZES, CASES, FAMILIES, family_ints, families, modulus, pick_window, recode,
                            top_reachable)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("field", [0, 1])
def test_modulus_is_just_above_2_254(field):
    """The premise of the edge families and of top_reachable: r = 2^254 + eps with eps < 2^126."""
    eps = modulus(field) - (1 << 254)
    assert 0 < eps < 1 << 126


@pytest.mark.parametrize("field", [0, 1])
@pytest.mark.parametrize("c", range(2, 17))
def test_families_reach_every_digit_case(field, c):
    W = (256 + c - 1) // c
    half = 1 << (c - 1)
    hit = {}
    for label, vals in family_ints(field, c, 64, seed=c).items():
        for s in vals:
            digits, cases, carry = recode(s, c)
            assert len(digits) == W
            assert sum(d << (w * c) for w, d in enumerate(digits)) == s, (label, c, hex(s))
            assert all(-half <= d <= half for d in digits), (label, c, hex(s))
            assert carry == 0, (label, c, hex(s))
            for case in cases:
                hit.setdefault(case, set()).add(label)
    assert {"half", "neg", "full"} <= set(hit), (c, sorted(hit))
    if top_reachable(c):
        assert "top" in hit, c
    else:
        assert (W - 1) * c == 255 and c in (3, 5, 15)
        assert "top" not in hit, c
    # the structured families hit what they are named for
    assert {"half", "half_after_carry"} <= hit["half"]
    assert {"half_after_carry", "negatives"} <= hit["neg"]
    assert "carry_chain" in hit["full"]
    if top_reachable(c):
        assert {"carry_chain", "negatives"} <= hit["top"]


@pytest.mark.parametrize("c", range(2, 17))
def test_recode_cases_by_hand(c):
    """Each boundary case on a scalar built for it."""
    half, full = 1 << (c - 1), 1 << c
    assert recode(half, c)[0][:2] == [half, 0] and "half" in recode(half, c)[1]
    d, cases, _ = recode(half + 1, c)
    assert d[:2] == [-(half - 1), 1] and "neg" in cases
    d, cases, _ = recode(full - 1 + (full - 1) * full, c)            # two all-ones windows: -1, then v = 2^c
    assert d[:3] == [-1, 0, 1] and "full" in cases
    W = (256 + c - 1) // c
    if top_reachable(c):
        assert "top" in recode(1 << ((W - 1) * c), c)[1]


@pytest.mark.parametrize("field", [0, 1])
def test_families_encode_through_the_oracle(field):
    from oracle import c_oracle as co
    ints = family_ints(field, 9, 5, seed=3)
    enc = families(field, 9, 5, seed=3)
    assert list(enc) == list(FAMILIES)
    for label in FAMILIES:
        assert enc[label].shape == (5, 4)
        assert co.from_mont(field, enc[label]) == ints[label], label


_BAND_EDGES = [(1, 4), (74, 4), (75, 5), (169, 5), (170, 6), (462, 6), (463, 7), (967, 7), (968, 8), (4300, 8),
               (4301, 10), (32017, 10), (32018, 13), (298188, 13), (298189, 15), (321126, 15), (321127, 16), (1 << 22, 16)]


def test_pick_window_bands():
    """The bucket MSM's window bands: 4 below 75 points, then 5, 6, 7, 8, 10, 13, 15 and from 321 127 points on 16."""
    assert [(n, pick_window(n)) for n, _ in _BAND_EDGES] == _BAND_EDGES


def test_pick_window_restates_msm_cu(tmp_path):
    """The restatement against msm.cu's own pick_window, compiled for the host from the source text, at every band edge
    and on a sweep of n."""
    src = open(os.path.join(ROOT, "battlezips-halo2_b200", "csrc", "msm.cu")).read()
    m = re.search(r"static uint32_t pick_window\(uint32_t n\) \{.*?\n\}\n", src, re.S)
    assert m, "pick_window not found in msm.cu"
    cc, exe = tmp_path / "pick_window.cc", str(tmp_path / "pick_window")
    cc.write_text("#include <cstdint>\n#include <cstdio>\n" + m.group(0) +
                  "int main() { unsigned n; while (scanf(\"%u\", &n) == 1) printf(\"%u\\n\", pick_window(n)); }\n")
    subprocess.run(["g++", "-O1", "-std=c++17", "-w", "-o", exe, str(cc)], check=True)
    ns = sorted({n for n, _ in _BAND_EDGES} | set(AUTO_WINDOW_SIZES) | set(range(1, 5000, 7)) | set(range(5000, 1 << 21, 997)))
    out = subprocess.run([exe], input="".join(f"{n}\n" for n in ns), capture_output=True, text=True, check=True).stdout.split()
    assert [int(c) for c in out] == [pick_window(n) for n in ns]


def test_auto_window_test_sizes_hit_their_bands():
    """The n values of the window_bits = 0 GPU tests land where they claim; a change to the cost model flags them here
    instead of quietly moving the tests to other widths."""
    assert {n: pick_window(n) for n in AUTO_WINDOW_SIZES} == AUTO_WINDOW_SIZES
    assert {5, 10, 13, 15, 16} <= set(AUTO_WINDOW_SIZES.values())
