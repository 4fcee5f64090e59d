"""CPU tests of the two pieces of the encircled-energy radius solve that csrc/ee_geometry.h shares with ee_kernel,
compiled for the host by nvcc through tools/ee_solve_check.cu:

* ``row_window``: the rows a disc can reach, for centres inside, on and far outside the image (up to 1e300) and
  radii from 0 to +inf, against a numpy restatement of the rule and against exact rational arithmetic; a build
  with the undefined-behaviour sanitizer shows that no int conversion or product overflows.
* ``fraction_bracket``: the starting bracket of r_q from the tabulated (r_k, EE_k), always ordered with
  EE(lo) < target <= EE(hi), independent of the order of the radii (duplicates included), and on an image with
  negative pixels (where EE falls) the bracket below the first tabulated crossing."""
import itertools
import os
import shutil
import subprocess
import tempfile
from fractions import Fraction

import numpy as np
import pytest

import ee_oracle as eo

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, 'tools', 'ee_solve_check.cu')
UBSAN = ['-Xcompiler', '-fsanitize=undefined', '-Xcompiler', '-fsanitize=float-cast-overflow',
         '-Xcompiler', '-fno-sanitize-recover=all', '-Xlinker', '-lubsan']


def _nvcc():
    nvcc = next((c for c in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc')
                 if c and os.path.exists(c)), None)
    if nvcc is None:
        pytest.skip('nvcc not found')
    return nvcc


def _compile(tmp, name, flags=()):
    exe = os.path.join(tmp, name)
    subprocess.run([_nvcc(), '-O2', *flags, '-I', os.path.join(ROOT, 'muse_psfr_b200', 'csrc'), SRC, '-o', exe],
                   check=True, cwd=tmp, capture_output=True)
    return exe


@pytest.fixture(scope='module')
def driver():
    """Run the host build of the helpers on a list of input lines; returns the output lines."""
    with tempfile.TemporaryDirectory() as tmp:
        exe = _compile(tmp, 'ee_solve_check')

        def run(lines, exe=exe):
            res = subprocess.run([exe], input='\n'.join(lines) + '\n', capture_output=True, text=True, timeout=120)
            assert res.returncode == 0, res.stderr
            out = res.stdout.splitlines()
            assert len(out) == len(lines)
            return out
        yield run


def num(v):
    return repr(float(v))       # shortest round-trip form; scanf reads 'inf' and '-inf'


# ---------------------------------------------------------------- row window
NY = (3, 7, 40, 1706)           # 1706 x 3 is the tallest image the kernel's shared memory takes


def window_cases():
    out = []
    for ny in NY:
        centres = [0.0, 1.3, ny / 2, ny - 1.0, -0.5, 0.5, ny - 0.5, 10.5, -3.0, -1000.0, ny + 5.0, ny + 1000.0,
                   1e8, -1e8, 3e9, -3e9, 1e300, -1e300, np.nextafter(0.5, 1.0) + 1e-15]
        for y0 in centres:
            for r in (0.0, 1e-300, 0.3, 0.5, 1.0, 2.5, 17.0, 1e8, 3e9, 1e300, np.inf):
                out.append((y0, r, ny))
    return out


def window_rule(y0, r, ny):
    """numpy restatement: one row of margin beyond [y0 - r - 1/2, y0 + r + 1/2], clamped to [0, ny] before the
    conversion to an integer."""
    p0 = np.minimum(np.maximum(0.0, np.floor(y0 - r - 0.5)), float(ny))
    p1 = np.maximum(0.0, np.minimum(float(ny), np.ceil(y0 + r + 0.5) + 1.0))
    return int(p0), int(p1)


def reachable_rows(y0, r, ny):
    """Rows p whose span [p - 1/2, p + 1/2] meets [y0 - r, y0 + r], in exact rational arithmetic."""
    if np.isinf(r):
        return range(ny)
    y, rr, h = Fraction(y0), Fraction(r), Fraction(1, 2)
    return [p for p in range(ny) if p + h >= y - rr and p - h <= y + rr]


def test_row_window(driver):
    cases = window_cases()
    got = [tuple(map(int, line.split())) for line in driver(['w %s %s %d' % (num(y), num(r), ny)
                                                              for y, r, ny in cases])]
    empty = 0
    for (y0, r, ny), (p0, p1) in zip(cases, got):
        assert (p0, p1) == window_rule(y0, r, ny), (y0, r, ny)
        assert 0 <= p0 <= ny and 0 <= p1 <= ny, (y0, r, ny)
        rows = reachable_rows(y0, r, ny)
        assert all(p0 <= p < p1 for p in rows), (y0, r, ny, p0, p1)
        if not rows:
            # no row in reach: the window is empty when the disc ends more than a row of margin from the image
            if y0 + r < -2 or y0 - r > ny + 1:
                assert p0 >= p1, (y0, r, ny, p0, p1)
                empty += 1
        elif abs(y0) + r < 1e6:
            # away from huge values the window is tight: at most one row beyond the reachable ones on each side
            assert p0 >= rows[0] - 1 and p1 <= rows[-1] + 2, (y0, r, ny, p0, p1)
    assert empty > 100


def test_row_window_far_centres(driver):
    """The centres of the far-outside example: the window is empty, not a wrapped int product."""
    lines = ['w 1e8 1 40', 'w -1e8 1 40', 'w 3e9 1 40', 'w -3e9 1 40', 'w 1e300 1e8 40', 'w -1e300 1 1706',
             'w 1e8 1e300 40', 'w -1e8 inf 40', 'w 20 0 40', 'w 20 1e-300 40']
    got = [tuple(map(int, line.split())) for line in driver(lines)]
    assert got[:6] == [(40, 40), (0, 0), (40, 40), (0, 0), (40, 40), (0, 0)]
    assert got[6:8] == [(0, 40), (0, 40)]
    assert got[8:] == [(19, 22), (19, 22)]


def test_row_window_has_no_undefined_behaviour():
    """The same cases through a build with -fsanitize=undefined,float-cast-overflow that aborts on the first
    finding: an int product or a double-to-int conversion out of range would stop it."""
    with tempfile.TemporaryDirectory() as tmp:
        try:
            exe = _compile(tmp, 'ee_solve_check_ubsan', UBSAN)
        except subprocess.CalledProcessError as exc:
            pytest.skip('the host compiler cannot build with the undefined-behaviour sanitizer: %s' % exc.stderr[-200:])
        cases = window_cases()
        res = subprocess.run([exe], input='\n'.join('w %s %s %d' % (num(y), num(r), ny) for y, r, ny in cases),
                             capture_output=True, text=True, timeout=120)
        assert res.returncode == 0 and 'runtime error' not in res.stderr, res.stderr[-2000:]
        assert [tuple(map(int, line.split())) for line in res.stdout.splitlines()] == \
            [window_rule(*c) for c in cases]


# ---------------------------------------------------------------- fraction bracket
def bracket(driver, cases):
    """cases: (target, rmax, total, radii, ee) -> [(lo, elo, hi, ehi)]"""
    lines = []
    for target, rmax, total, r, e in cases:
        lines.append('b %s %s %s %d %s' % (num(target), num(rmax), num(total), len(r),
                                           ' '.join('%s %s' % (num(a), num(b)) for a, b in zip(r, e))))
    return [tuple(float(t) for t in line.split()) for line in driver(lines)]


def worked_example():
    """1.0 at (20, 20), -0.8 spread over the ring 4.5 < d < 5.5 and +0.8 over 9.5 < d < 10.5: TOTAL = 1, EE rises
    to 1 by r = sqrt(1/2), falls to 0.2 across the first ring and rises back to 1 across the second."""
    img = np.zeros((40, 40))
    img[20, 20] = 1.0
    p, q = np.mgrid[:40, :40]
    d = np.hypot(p - 20, q - 20)
    inner, outer = (d > 4.5) & (d < 5.5), (d > 9.5) & (d < 10.5)
    img[inner] = -0.8 / inner.sum()
    img[outer] = 0.8 / outer.sum()
    return img


def test_bracket_worked_example(driver):
    """EE(2) = 1.0 and EE(7) = 0.2 about the target 0.5: the bracket is [0, 2], where EE crosses 0.5 once (at
    0.3989), not the inverted [7, 2] of a rule that takes the largest radius with EE below the target."""
    img = worked_example()
    total = float(np.sum(np.asarray(img, dtype=eo.LD)))
    e2, e7 = float(eo.ee(img, 2.0)), float(eo.ee(img, 7.0))
    assert abs(total - 1.0) < 1e-15 and abs(e2 - 1.0) < 1e-15 and abs(e7 - 0.2) < 1e-12
    rmax = np.hypot(20.5, 20.5)
    got = bracket(driver, [(0.5 * total, rmax, total, [2.0, 7.0], [e2, e7]),
                           (0.5 * total, rmax, total, [7.0, 2.0], [e7, e2])])
    assert got[0] == got[1] == (0.0, 0.0, 2.0, e2)


def bracket_rule(target, rmax, total, r, e):
    hi, ehi = min([(a, b) for a, b in zip(r, e) if b >= target and a < rmax] + [(rmax, total)])
    lo, elo = max([(a, b) for a, b in zip(r, e) if b < target and a < hi] + [(0.0, 0.0)])
    return lo, elo, hi, ehi


def random_tables(seed, n_tables):
    """Tables of an EE that rises and falls (sums of a few random bumps, 0 at r = 0 and TOTAL from rmax on), at
    radii drawn with duplicates, zeros, rmax itself and radii beyond it; targets from 1e-12 to 1 - 1e-12 of
    TOTAL, and exactly equal to a tabulated EE."""
    rng = np.random.default_rng(seed)
    out = []
    for t in range(n_tables):
        rmax = rng.uniform(3, 30)
        total = rng.uniform(0.1, 10)
        amp, mu, sig = rng.normal(0, 2, 4), rng.uniform(0, rmax, 4), rng.uniform(0.3, 4, 4)

        def ee(x):
            if x >= rmax:
                return total
            s = np.sin(np.pi / 2 * x / rmax)
            return total * s * s + float(np.sum(amp * np.sin(np.pi * x / rmax) * np.exp(-(x - mu) ** 2 / sig ** 2)))
        n = int(rng.integers(0, 12))
        r = list(rng.uniform(0, 1.2 * rmax, n))
        r += list(rng.choice(r, int(rng.integers(0, 4)))) if r else []
        if t % 5 == 0:
            r += [0.0, rmax]
        e = [0.0 if x == 0 else ee(x) for x in r]
        for q in (1e-12, 0.1, 0.5, 0.9, 1 - 1e-12):
            out.append((q * total, rmax, total, r, e))
        out += [(b, rmax, total, r, e) for b in e[:2] if 0 < b < total]
    return out


def test_bracket_is_ordered_and_valid(driver):
    cases = random_tables(11, 300)
    falls = 0
    for (target, rmax, total, r, e), (lo, elo, hi, ehi) in zip(cases, bracket(driver, cases)):
        assert (lo, elo, hi, ehi) == bracket_rule(target, rmax, total, r, e)
        assert 0.0 <= lo < hi <= rmax and elo < target <= ehi, (target, r, e, lo, hi)
        assert (lo, elo) in list(zip(r, e)) + [(0.0, 0.0)] and (hi, ehi) in list(zip(r, e)) + [(rmax, total)]
        # no tabulated radius inside (lo, hi) has EE >= target, or lies below hi with EE < target above lo
        assert not any(lo < a < hi for a in r)
        old_lo = max([a for a, b in zip(r, e) if b < target] + [0.0])
        falls += old_lo > hi
    assert falls > 20          # tables on which the bracket of the largest radius below the target was inverted


def test_bracket_ignores_the_order_of_the_radii(driver):
    rng = np.random.default_rng(5)
    cases, groups = [], []
    for target, rmax, total, r, e in random_tables(12, 60):
        if len(r) < 2:
            continue
        perms = [np.arange(len(r))[::-1]] + [rng.permutation(len(r)) for _ in range(4)]
        if len(r) <= 5:
            perms = [np.array(p) for p in itertools.permutations(range(len(r)))]
        groups.append(len(perms) + 1)
        cases.append((target, rmax, total, r, e))
        cases += [(target, rmax, total, [r[k] for k in p], [e[k] for k in p]) for p in perms]
    got = bracket(driver, cases)
    k = 0
    for g in groups:
        assert len(set(got[k:k + g])) == 1, cases[k]
        k += g
    assert k == len(cases) > 500


def test_bracket_of_a_rising_table_is_unchanged(driver):
    """Where EE never falls (no negative pixel), the bracket is the largest radius with EE < target and the
    smallest with EE >= target: the one the solve started from before, so r_q of such images keeps its bits."""
    rng = np.random.default_rng(6)
    cases = []
    for _ in range(200):
        rmax, total = 29.0, rng.uniform(0.5, 2)
        r = rng.uniform(0, 35, int(rng.integers(0, 20)))
        e = np.where(r >= rmax, total, total * np.sqrt(np.minimum(r / rmax, 1.0)))
        cases.append((total * rng.uniform(0.01, 0.99), rmax, total, list(r), list(e)))
    for (target, rmax, total, r, e), got in zip(cases, bracket(driver, cases)):
        below = [(a, b) for a, b in zip(r, e) if b < target]
        above = [(a, b) for a, b in zip(r, e) if b >= target and a < rmax]
        assert got == max(below + [(0.0, 0.0)]) + min(above + [(rmax, total)])
