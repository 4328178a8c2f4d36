"""Checks of the lifter's hand-restated helper semantics against the exported functions of the reference binary
(rt_GetLookupIndex @0xf470, rt_Lookup @0xf530, rt_Lookup2D_Normal @0xf590; their results on these probes are recorded in
tests/golden/refbin_kat.npz by tests/golden/make_golden_refbin.py), including exact ties, and of the branch-free breakpoint
count the generated code uses."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'tools', 'lift'))
KAT = os.path.join(ROOT, 'tests', 'golden', 'refbin_kat.npz')       # loaded by the tests: make_golden_refbin imports axes / probes


def axes(rng):
    for n in (2, 3, 4, 6, 9, 11, 17, 22):
        for lo in (-0.3, 0.0, 0.2):
            yield np.sort(lo + np.cumsum(rng.uniform(0.01, 0.3, n)))
        yield np.linspace(-1.0, 1.0, n)          # has an exact 0.0 breakpoint for odd n


def probes(x, rng):
    u = list(rng.uniform(x[0] - 0.5, x[-1] + 0.5, 40)) + list(x) + [0.0, -0.0, x[0] - 1, x[-1] + 1]
    u += list((x[:-1] + x[1:]) / 2)
    return u


def count_rule(x, u):
    """the generated code's index: number of interior breakpoints below u, `<=` for negative breakpoints (codegen.index_of)."""
    return sum((xj <= u) if xj < 0 else (xj < u) for xj in x[1:-1])


def test_lookup_index_restatements_equal_the_binary():
    import symtrace as S
    rng = np.random.RandomState(0)
    want = np.load(KAT)['lookup_index'].tolist()
    n = 0
    for x in axes(rng):
        for u in probes(x, rng):
            ref = want[n]
            n += 1
            assert S.Tracer.lookup_index(list(x), float(u)) == ref, (list(x), u)
            assert count_rule(x, u) == ref, (list(x), u)
    assert n == len(want)


def test_lookup_formulas_equal_the_binary():
    import symtrace as S
    rng = np.random.RandomState(1)
    li = S.Tracer.lookup_index
    kat = np.load(KAT)
    want2, want1 = iter(kat['lookup2d'].tolist()), iter(kat['lookup1d'].tolist())
    for _ in range(30):
        nx, ny = rng.randint(2, 12), rng.randint(2, 12)
        xs = np.sort(rng.uniform(-1, 1, nx)); ys = np.sort(rng.uniform(-1, 1, ny)); zs = rng.normal(0, 1, nx * ny)
        for _ in range(20):
            x, y = rng.uniform(-1.3, 1.3), rng.uniform(-1.3, 1.3)
            ix, iy = li(list(xs), x), li(list(ys), y)
            dx, ux = xs[ix + 1] - xs[ix], x - xs[ix]
            a = (zs[ix + 1 + nx * iy] - zs[ix + nx * iy]) / dx * ux + zs[ix + nx * iy]
            b = (zs[ix + 1 + nx * (iy + 1)] - zs[ix + nx * (iy + 1)]) / dx * ux + zs[ix + nx * (iy + 1)]
            mine = (b - a) / (ys[iy + 1] - ys[iy]) * (y - ys[iy]) + a
            assert mine == next(want2)           # bit-exact
            i = li(list(xs), x)
            zz = zs[:nx]
            mine1 = (zz[i + 1] - zz[i]) / (xs[i + 1] - xs[i]) * (x - xs[i]) + zz[i]
            assert mine1 == next(want1)
