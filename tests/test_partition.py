"""Host logic of the row-sweep backward: the CTA work partition (csrc/sl_partition.cuh), run on the CPU through
tests/partition_harness.cu.  Invariants: the ranges tile the (plane, own row) space in order; in cut mode two cuts of one
plane are at least rr + NT rows apart (rows_grow_fix_kernel relies on it); the modelled cost of the most expensive CTA is
within a few percent of the mean (min-max partition) and never worse than an equal-rows split."""
import json
import os
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W0 = 4      # kRowW0 (sl_partition.cuh)

# interp H W planes own0 ownN arr0 arrN cfl cut grid consumers
SHAPES = [
    (1, 721, 1440, 64, 0, 721, 0, 721, 6.0, 0, 148, 6),        # C3, full mesh (warm-up scheme)
    (1, 721, 1440, 64, 0, 721, 0, 721, 6.0, 1, 148, 6),        # C3, cut mode forced
    (2, 721, 1440, 64, 0, 721, 0, 721, 6.0, 1, 148, 8),        # bicubic
    (1, 721, 1440, 64, 0, 47, 0, 56, 6.0, 1, 148, 6),          # southern polar band of the 8-way split
    (1, 721, 1440, 64, 149, 105, 140, 123, 6.0, 1, 148, 6),    # a mid-latitude band of it
    (1, 721, 1440, 64, 361, 360, 352, 369, 6.0, 1, 148, 6),    # northern half (2-way split)
    (1, 181, 360, 3, 0, 181, 0, 181, 8.0, 1, 45, 6),           # few planes: short ranges
    (1, 96, 192, 6, 0, 96, 0, 96, 8.0, 1, 48, 6),
    (2, 33, 64, 4, 0, 33, 0, 33, 3.0, 1, 11, 2),
    (1, 64, 128, 2, 0, 12, 0, 21, 6.0, 1, 4, 4),               # ranges shorter than the guard depth
]


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("partition") / "harness")
    cmd = [nvcc, "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
           os.path.join(ROOT, "tests", "partition_harness.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    return exe


def run(exe, shapes):
    text = "\n".join(" ".join(str(v) for v in s) for s in shapes) + "\n"
    res = subprocess.run([exe], input=text, capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr[-2000:]
    out = [json.loads(line) for line in res.stdout.splitlines() if line.startswith("{")]
    assert len(out) == len(shapes)
    return out


def row_cost(hx, W, wc):
    n = min(W, wc + 2 * min(hx, W))
    k = (n + 31) >> 5
    if k & 3 == 0:
        k += 1
    return W0 + k


def range_cost(shape, res, g0, g1, prefix):
    interp, H, W, planes, own0, ownN, arr0, arrN, cfl, _, grid, _ = shape
    nt, omin = (2, 0) if interp == 1 else (4, -1)
    rr, ring, cut, GR = int(-(-cfl // 1)), res["ring"], res["cut"], res["GR"]
    cost, g = 0.0, g0
    while g < g1:
        pl, r = divmod(g, ownN)
        n = min(ownN - r, g1 - g)
        ra, rb = own0 + r, own0 + r + n
        cut_lo, cut_hi = bool(cut) and r > 0, bool(cut) and r + n < ownN
        y0 = ra if cut_lo else ra - (ring - 1) + rr - omin
        y1 = rb - 1 if cut_hi else rb - 1 + rr - omin
        y0, y1 = max(y0, arr0), min(y1, arr0 + arrN - 1)
        if y1 >= y0:
            cost += prefix[y1 + 1] - prefix[y0]
        cost += W0 * GR * (int(cut_lo) + int(cut_hi))
        g += n
    return cost


def test_partition_invariants(harness):
    results = run(harness, SHAPES)
    for shape, res in zip(SHAPES, results):
        interp, H, W, planes, own0, ownN, arr0, arrN, cfl, want_cut, grid, _ = shape
        b = res["bound"]
        assert len(b) == grid + 1 and b[0] == 0 and b[-1] == planes * ownN, shape
        assert all(b[c] <= b[c + 1] for c in range(grid)), shape
        assert res["cut"] in (0, want_cut)
        if res["cut"]:
            cuts = sorted({g for g in b[1:-1] if g % ownN != 0})
            for a, c in zip(cuts, cuts[1:]):
                assert a // ownN != c // ownN or c - a >= res["GR"], (shape, a, c)
        prefix = [0.0]
        for y in range(H):
            prefix.append(prefix[-1] + row_cost(res["hx"][y], W, res["wc"]))
        costs = [range_cost(shape, res, b[c], b[c + 1], prefix) for c in range(grid) if b[c + 1] > b[c]]
        total = planes * ownN
        equal = [range_cost(shape, res, total * c // grid, total * (c + 1) // grid, prefix) for c in range(grid)]
        if not (res["cut"] and total < 3 * res["GR"] * grid):      # (there the minimum cut spacing decides, not the cost)
            assert max(costs) <= max(equal) * 1.001, (shape, max(costs), max(equal))
        if total >= 40 * grid:          # long ranges: the partition is level to a few rows' worth of cost
            assert max(costs) <= 1.03 * sum(costs) / len(costs), (shape, max(costs), sum(costs) / len(costs))


def test_partition_is_deterministic_and_cached(harness):
    twice = run(harness, [SHAPES[1], SHAPES[3], SHAPES[1]])
    assert twice[0]["bound"] == twice[2]["bound"]          # second time from the per-shape cache
    assert twice[0]["bound"] != twice[1]["bound"]
