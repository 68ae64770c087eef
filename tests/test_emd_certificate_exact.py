"""The EMD certificate (psd_emd_dual_bound, psd_emd_certified) against exact arithmetic.

The certificate promises bounds that are rigorous for the fp32 inputs: every term rounded towards its bound in fp64, the
sums in a fixed order.  A round-to-nearest reference cannot check that promise, because the difference is a few ulps.
Here the reference is exact: every fp32 value is an integer multiple of 2^-149, so a squared distance S is an exact integer
in units of 2^-298 and sqrt(S) is bracketed by math.isqrt at P = 160 bits below the unit of the coordinates (an interval
that is a single point when S is a perfect square).  Prices are exact too.  L and U are then intervals of integers in
units of 2^-(149 + P), and the GPU doubles are compared with them as exact fractions:

* soundness, no tolerance: bounds[b, 0] n <= L and bounds[b, 1] n >= U;
* tightness: the distance to the exact value is at most (n + 8) 2^-52 times the sum of the magnitudes of the terms
  (derivation at `tight_tol`), far below what an fp32 evaluation could reach.

The input families target the rounding steps that random [0, 1] data cannot expose: one-pair clouds (a single square
root), odd n (the final division), coincident clouds with prices of widely different exponents (the two price sums,
whose exact difference is 0), coordinates from 1e-30 to FLT_MAX, extreme prices, the kernels' tile and grid edges."""
import ctypes
import functools
import math

import numpy as np
import pytest

from conftest import make_clouds
from test_emd_certified import case, dual_bound

P = 160                   # bits of the square roots below the unit of the coordinates
SCALE = 149               # an fp32 value is an integer multiple of 2^-149
UNIT = SCALE + P          # exact values of L and U are integers in units of 2^-UNIT
ULP = 2.0 ** -52          # one rounding step of a directed fp64 operation, relative
FLT_MAX = float(np.finfo(np.float32).max)


# ---------------------------------------------------------------------------------------------------------------------
# exact reference
# ---------------------------------------------------------------------------------------------------------------------
def f32_ints(a):
    """Exact integer images v * 2^149 of the fp32 values of a, as a flat list of Python ints."""
    out = []
    for v in np.asarray(a, np.float32).ravel().tolist():
        num, den = v.as_integer_ratio()
        out.append(num * ((1 << SCALE) // den))
    return out


def sqrt_interval(s):
    """(floor, ceil) of sqrt(s) 2^P for an integer s >= 0: sqrt of a squared distance in units of 2^-2*SCALE, in units of
    2^-UNIT.  The two are equal when s 2^2P is a perfect square."""
    m = s << (2 * P)
    r = math.isqrt(m)
    return r, r + (r * r != m)


# The filter.  numpy evaluates v_jk = d_jk + p_k in fp64 from the fp32 inputs: the three differences (each rounded,
# relative error u = 2^-53), their squares and two additions of non-negative terms (S within (1 + 5u) of the exact sum),
# the square root (d within 3.5u relative, to first order) and the addition of p (u |d + p|).  So |v_computed - v| <=
# 3.5u d + u (d + |p|) <= 2^-50 (d + |p|).  FILTER_REL = 2^-48 is four times that.  Object k can be a row's exact minimiser
# only if v_k - err_k <= min_k' (v_k' + err_k') in computed values; the exact evaluation runs over those k alone.  The
# same set also holds every k whose GPU value (error <= 4 ulps of d + |p|, see tight_tol) can be the GPU's minimum.
FILTER_REL = 2.0 ** -48


def _candidates(x1, x2, p, all_pairs):
    """Per row of one cloud: the candidate objects and s_j = max over them of (d_jk + |p_k|), rounded up generously."""
    n = x1.shape[0]
    x1d, x2d, pd = x1.astype(np.float64), x2.astype(np.float64), p.astype(np.float64)
    cand, srow = [], np.empty(n)
    step = max(1, (1 << 22) // n)
    for j0 in range(0, n, step):
        d = np.sqrt(((x1d[j0:j0 + step, None, :] - x2d[None, :, :]) ** 2).sum(-1))
        v = d + pd[None, :]
        err = FILTER_REL * (d + np.abs(pd)[None, :])
        keep = np.ones(v.shape, bool) if all_pairs else (v - err) <= (v + err).min(1)[:, None]
        mag = d + np.abs(pd)[None, :]
        for r in range(d.shape[0]):
            ks = np.flatnonzero(keep[r])
            cand.append(ks.tolist())
            srow[j0 + r] = mag[r, ks].max() * (1 + 2.0 ** -40)
    return cand, srow


class Exact:
    """Exact certificate of one cloud: L in [l_lo, l_hi] and U in [u_lo, u_hi] (None if the assignment is not a
    permutation), integers in units of 2^-UNIT; scale_l, scale_u: the magnitudes the tightness tolerance is taken of."""

    def __init__(self, n, l_lo, l_hi, u_lo, u_hi, scale_l, scale_u):
        self.n, self.l_lo, self.l_hi, self.u_lo, self.u_hi = n, l_lo, l_hi, u_lo, u_hi
        self.scale_l, self.scale_u = scale_l, scale_u

    def mid(self):
        """(L / n, U / n) to double precision (the midpoints of the intervals)."""
        f = lambda a, b: float((a + b) / 2 / (1 << UNIT) / self.n) if a is not None else float("nan")
        return f(self.l_lo, self.l_hi), f(self.u_lo, self.u_hi)


def exact_certificate(x, y, assignment, price=None, all_pairs=False):
    """The certificate of every cloud in exact arithmetic: a list of Exact.  all_pairs=False evaluates exactly only the
    filter's candidates (see FILTER_REL)."""
    x, y = np.asarray(x, np.float32), np.asarray(y, np.float32)
    b, n, _ = x.shape
    p = np.zeros((b, n), np.float32) if price is None else np.asarray(price, np.float32)
    a = np.asarray(assignment)
    out = []
    for c in range(b):
        cand, srow = _candidates(x[c], y[c], p[c], all_pairs)
        X1, X2, Pi = f32_ints(x[c]), f32_ints(y[c]), f32_ints(p[c])
        l_lo = l_hi = 0
        for j in range(n):
            ax, ay, az = X1[3 * j], X1[3 * j + 1], X1[3 * j + 2]
            best_lo = best_hi = None
            for k in cand[j]:
                dx, dy, dz = ax - X2[3 * k], ay - X2[3 * k + 1], az - X2[3 * k + 2]
                lo, hi = sqrt_interval(dx * dx + dy * dy + dz * dz)
                pk = Pi[k] << P
                if best_lo is None or lo + pk < best_lo:
                    best_lo = lo + pk
                if best_hi is None or hi + pk < best_hi:
                    best_hi = hi + pk
            l_lo += best_lo
            l_hi += best_hi
        sp = sum(Pi) << P
        l_lo -= sp
        l_hi -= sp
        ac = a[c]
        perm = bool(((ac >= 0) & (ac < n)).all()) and np.unique(ac).size == n
        u_lo = u_hi = None
        scale_u = 0.0
        if perm:
            u_lo = u_hi = 0
            for j in range(n):
                k = int(ac[j])
                dx, dy, dz = X1[3 * j] - X2[3 * k], X1[3 * j + 1] - X2[3 * k + 1], X1[3 * j + 2] - X2[3 * k + 2]
                lo, hi = sqrt_interval(dx * dx + dy * dy + dz * dz)
                u_lo += lo
                u_hi += hi
            scale_u = float(np.sqrt(((x[c].astype(np.float64) - y[c][ac].astype(np.float64)) ** 2).sum(-1)).sum()) * (1 + 2.0 ** -40)
        scale_l = float(srow.sum() + np.abs(p[c].astype(np.float64)).sum()) * (1 + 2.0 ** -40)
        out.append(Exact(n, l_lo, l_hi, u_lo, u_hi, scale_l, scale_u))
    return out


def tight_tol(n, scale):
    """How far a directed-rounded bound (times n) may lie from the exact value, in units of 2^-UNIT.

    A term d + p of L: the absolute difference (1 rounding), its square and two fused multiply-adds (3), the square root
    (1) and the addition of p (1), all towards -inf, each at most one ulp = 2^-52 relative: within 4 ulps of d + |p|
    (first order; the square root halves the error of S).  The minimum over k of such terms is within that of the exact
    row minimum, taken at one of the filter's candidates, so within 4 ulps of s_j.  The row sum (n additions) and sum_k p_k
    (a tree of at most n additions) each lose at most n ulps of the sum of the magnitudes; the final subtraction and
    the division by n one each.  Altogether (n + 6) ulps of scale = sum_j s_j + sum_k |p_k| for L; U has no prices and
    the same count.  (n + 8) leaves room for second-order terms."""
    return math.ceil((n + 8) * ULP * scale * (1 << UNIT))


def _frac(v):
    return v.as_integer_ratio()


def check_bounds(bounds, status, ref, tight=True):
    """Soundness (exact, no tolerance) and tightness of every cloud's GPU bounds against the exact reference; returns the
    list of violations (empty when all hold)."""
    bad = []
    for c, r in enumerate(ref):
        lo, hi, st = float(bounds[c, 0]), float(bounds[c, 1]), int(status[c])
        want_st = 1 if r.u_lo is not None else 0
        if st != want_st:
            bad.append(f"cloud {c}: status {st}, want {want_st}")
            continue
        if not math.isfinite(lo):
            bad.append(f"cloud {c}: lower bound {lo}")
            continue
        num, den = _frac(lo)
        got = num * r.n * (1 << UNIT)           # lo n, in units of 2^-UNIT / den
        if got > r.l_lo * den:
            bad.append(f"cloud {c}: lower bound {lo!r} above the exact L / n = {r.mid()[0]!r}")
        elif tight and r.l_hi * den - got > tight_tol(r.n, r.scale_l) * den:
            bad.append(f"cloud {c}: lower bound {lo!r} looser than the tolerance below L / n = {r.mid()[0]!r}")
        if want_st:
            if not math.isfinite(hi):
                bad.append(f"cloud {c}: upper bound {hi}")
                continue
            num, den = _frac(hi)
            got = num * r.n * (1 << UNIT)
            if got < r.u_hi * den:
                bad.append(f"cloud {c}: upper bound {hi!r} below the exact U / n = {r.mid()[1]!r}")
            elif tight and got - r.u_lo * den > tight_tol(r.n, r.scale_u) * den:
                bad.append(f"cloud {c}: upper bound {hi!r} looser than the tolerance above U / n = {r.mid()[1]!r}")
        elif not math.isnan(hi):
            bad.append(f"cloud {c}: upper bound {hi} without a permutation")
    return bad


def assert_exact(bounds, status, ref, tight=True):
    bad = check_bounds(bounds, status, ref, tight)
    assert not bad, f"{len(bad)} of {len(ref)} clouds wrong: " + "; ".join(bad[:6])


# ---------------------------------------------------------------------------------------------------------------------
# input families: each returns dict(x, y, a, p) with x, y [B, n, 3] float32, a [B, n] int32, p [B, n] float32 or None
# ---------------------------------------------------------------------------------------------------------------------
def _perms(rng, b, n, identity_every=2):
    a = np.stack([np.arange(n) if i % identity_every == 0 else rng.permutation(n) for i in range(b)])
    return a.astype(np.int32)


def fam_tiny(n, prices, b=2048, seed=0):
    """Many tiny clouds: a one-pair cloud tests a single square root, odd n the final division.  Half the clouds have
    the identity assignment, half a random permutation."""
    rng = np.random.default_rng(seed * 100 + n)
    x = rng.random((b, n, 3), dtype=np.float32)
    y = rng.random((b, n, 3), dtype=np.float32)
    p = None if prices is None else (rng.random((b, n), dtype=np.float32) * 2 - 1) * np.float32(prices)
    return dict(x=x, y=y, a=_perms(rng, b, n), p=p)


def _wide_prices(rng, shape, top=-21):
    """0, -0.0, +-2^-k for k in (-top ... 120), the same with random mantissas, and fp32 subnormals: sums of these are
    inexact in fp64 in every order."""
    kind = rng.integers(0, 5, size=shape)
    sign = np.where(rng.random(shape) < 0.5, -1.0, 1.0)
    k = rng.integers(-top, 121, size=shape).astype(np.float64)
    mant = 1.0 + rng.integers(0, 1 << 23, size=shape) / float(1 << 23)
    sub = rng.integers(1, 1 << 23, size=shape) * 2.0 ** -149
    v = np.select([kind == 0, kind == 1, kind == 2, kind == 3], [0.0, -0.0, sign * 2.0 ** -k, sign * mant * 2.0 ** -k],
                  sign * sub)
    v = v.astype(np.float32)
    v[kind == 1] = np.float32(-0.0)
    return v


def fam_coincident(n, b, seed=0):
    """y = x[perm] with wide-exponent prices below half the smallest distance between distinct points, so each point's
    own copy is its row minimum: L = 0 exactly, and U = 0 for a = the inverse permutation.  The row sum (row order,
    rounded down) and sum_k p_k (a strided tree, rounded up) only keep L <= 0 in the right directions."""
    rng = np.random.default_rng(1000 + seed * 7 + n)
    x = rng.random((b, n, 3), dtype=np.float32)
    perm = np.stack([rng.permutation(n) for _ in range(b)])
    y = np.take_along_axis(x, perm[..., None], 1)
    a = np.argsort(perm, axis=1).astype(np.int32)
    p = _wide_prices(rng, (b, n))
    if n > 1:
        xd = x.astype(np.float64)
        dmin = min(np.sqrt(((xd[c][:, None] - xd[c][None]) ** 2).sum(-1) + np.eye(n)).min() for c in range(b))
        assert np.abs(p.astype(np.float64)).max() < dmin / 2
    return dict(x=x, y=np.ascontiguousarray(y), a=a, p=p)


def _wide_coords(rng, shape):
    """A mixture of +-10^[-30, 30], fp32 subnormals, +-FLT_MAX, +-0 and [0, 1)."""
    kind = rng.integers(0, 6, size=shape)
    sign = np.where(rng.random(shape) < 0.5, -1.0, 1.0)
    wide = sign * 10.0 ** rng.uniform(-30, 30, size=shape)
    sub = sign * rng.integers(1, 1 << 23, size=shape) * 2.0 ** -149
    v = np.select([kind == 0, kind == 1, kind == 2, kind == 3, kind == 4], [wide, wide, sub, sign * FLT_MAX, sign * 0.0],
                  rng.random(shape))
    return v.astype(np.float32)


def fam_wide(n, b=256, seed=0):
    """Wide-range coordinates, where the difference of two floats is not exact in fp64 and an fp32 evaluation overflows.
    Half of y's points are x's points with one coordinate moved by one fp32 ulp."""
    rng = np.random.default_rng(2000 + seed * 7 + n)
    x = _wide_coords(rng, (b, n, 3))
    y = _wide_coords(rng, (b, n, 3))
    near = rng.random((b, n)) < 0.5
    src = np.take_along_axis(x, np.stack([rng.permutation(n) for _ in range(b)])[..., None], 1)
    ax = rng.integers(0, 3, size=(b, n))
    moved = src.copy()
    bi, ni = np.nonzero(near)
    c = ax[bi, ni]
    s = src[bi, ni, c]
    toward = np.where(rng.random(bi.size) < 0.5, np.inf, -np.inf)
    toward = np.where(np.abs(s) == FLT_MAX, np.where(s > 0, -np.inf, np.inf), toward).astype(np.float32)   # stay finite
    moved[bi, ni, c] = np.nextafter(s, toward)
    y = np.where(near[..., None], moved, y).astype(np.float32)
    assert np.isfinite(y).all()
    p = (rng.random((b, n), dtype=np.float32) - np.float32(0.5)) * np.float32(1e-3)
    return dict(x=x, y=y, a=_perms(rng, b, n), p=p)


def fam_wide_exact(n, b=1024, seed=0):
    """Pairs that differ along one axis only: x = m 2^k (m odd, at most 12 bits) and y = +-m' 2^(k - 60 - r), a value below
    half an fp64 ulp of x.  The exact |x - y| is then not a double, while its neighbour |x| has an exact square: the
    difference must be rounded down for L (same signs) and up for U (opposite signs), or the bound crosses the exact value.
    The points of a cloud sit 8 apart along another axis."""
    rng = np.random.default_rng(6000 + n + seed)
    x = np.zeros((b, n, 3), np.float64)
    for c in range(b):
        for j in range(n):
            k = int(rng.integers(-40, 41))
            x[c, j, 0] = (2 * int(rng.integers(0, 2048)) + 1) * 2.0 ** k * rng.choice([-1.0, 1.0])
            x[c, j, 1] = 8.0 * j + rng.random()
            x[c, j, 2] = rng.random()
    y = x.copy()
    tiny_exp = np.log2(np.abs(x[..., 0])).astype(int) - 60 - rng.integers(0, 20, size=(b, n))
    y[..., 0] = np.sign(x[..., 0]) * rng.choice([-1.0, 1.0], size=(b, n)) * rng.integers(1, 1 << 12, size=(b, n)) * 2.0 ** tiny_exp
    ax = rng.permutation(3)                              # the axis that carries the difference
    x, y = x[..., ax].astype(np.float32), y[..., ax].astype(np.float32)
    assert (y[..., ax.tolist().index(0)] != 0).all()
    return dict(x=x, y=y, a=np.tile(np.arange(n, dtype=np.int32), (b, 1)), p=None)


def fam_prices(kind, n=33, b=64, seed=0):
    """Uniform clouds with extreme prices: negative, of magnitude 1e30, subnormal, NULL, all zero."""
    rng = np.random.default_rng(3000 + seed)
    x = rng.random((b, n, 3), dtype=np.float32)
    y = rng.random((b, n, 3), dtype=np.float32)
    shape = (b, n)
    if kind == "negative":
        p = -rng.random(shape, dtype=np.float32) * np.float32(4.0)
    elif kind == "huge":
        p = ((rng.random(shape) * 2 - 1) * 1e30).astype(np.float32)
    elif kind == "subnormal":
        p = (np.where(rng.random(shape) < 0.5, -1.0, 1.0) * rng.integers(1, 1 << 23, size=shape) * 2.0 ** -149).astype(np.float32)
    elif kind == "zero":
        p = np.zeros(shape, np.float32)
    elif kind == "null":
        p = None
    else:
        raise ValueError(kind)
    return dict(x=x, y=y, a=_perms(rng, b, n), p=p)


def fam_sizes(n, b=2, seed=0):
    """The row-CTA (64 bidders) and object-tile (2048) edges: uniform clouds, random permutations and prices."""
    x, y = make_clouds("uniform", b, n, n, seed=4000 + n + seed)
    rng = np.random.default_rng(4100 + n)
    return dict(x=x, y=y, a=_perms(rng, b, n, identity_every=b + 1), p=rng.random((b, n), dtype=np.float32) * np.float32(0.1))


def fam_pythagorean(n, b=512, seed=0):
    """Every point j of y is x_j moved by an integer vector of integer length (3-4-5, 1-2-2, 2-3-6, ... scaled by a power
    of two), the points far apart: every distance and both bounds are exact, so L / n and U / n are single rationals
    and the final division rounds in its direction (n odd: inexact)."""
    vecs = [(3, 4, 0), (1, 2, 2), (2, 3, 6), (1, 4, 8), (4, 4, 7), (2, 6, 9), (0, 5, 12), (6, 6, 7), (0, 0, 1)]
    rng = np.random.default_rng(5000 + n + seed)
    x = np.zeros((b, n, 3), np.float32)
    y = np.zeros((b, n, 3), np.float32)
    for c in range(b):
        for j in range(n):
            v = np.array(vecs[rng.integers(len(vecs))], np.float64)
            v = v[rng.permutation(3)] * np.where(rng.random(3) < 0.5, -1, 1) * 2.0 ** int(rng.integers(-12, -4))
            base = np.array([j * 4.0, rng.integers(0, 4), 0.0]) + 0.5   # 4 apart: nothing else is nearer than 1
            x[c, j], y[c, j] = base, base + v
    a = np.tile(np.arange(n, dtype=np.int32), (b, 1))
    return dict(x=x, y=y, a=a, p=None)


FAMILIES = {}
for _n in (1, 2, 3, 5, 7):
    FAMILIES[f"tiny_n{_n}_prices"] = functools.partial(fam_tiny, _n, 1.0)
    FAMILIES[f"tiny_n{_n}_noprice"] = functools.partial(fam_tiny, _n, None)
for _n, _b in ((1, 512), (2, 512), (3, 512), (64, 96), (65, 96), (300, 16)):
    FAMILIES[f"coincident_n{_n}"] = functools.partial(fam_coincident, _n, _b)
for _n in (1, 3, 16, 33):
    FAMILIES[f"wide_n{_n}"] = functools.partial(fam_wide, _n)
for _n in (1, 3):
    FAMILIES[f"wide_exact_n{_n}"] = functools.partial(fam_wide_exact, _n)
for _k in ("negative", "huge", "subnormal", "zero", "null"):
    FAMILIES[f"prices_{_k}"] = functools.partial(fam_prices, _k)
for _n in (63, 64, 65, 2047, 2048, 2049, 4099):
    FAMILIES[f"size_n{_n}"] = functools.partial(fam_sizes, _n)
for _n in (1, 3, 5, 7):
    FAMILIES[f"pythagorean_n{_n}"] = functools.partial(fam_pythagorean, _n)

_DATA, _REF = {}, {}


def family(name):
    if name not in _DATA:
        _DATA[name] = FAMILIES[name]()
    return _DATA[name]


def reference(name):
    if name not in _REF:
        d = family(name)
        _REF[name] = exact_certificate(d["x"], d["y"], d["a"], d["p"])
    return _REF[name]


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference itself
# ---------------------------------------------------------------------------------------------------------------------
def test_sqrt_interval():
    for s in (0, 1, 4, 9, 2, 3, (1 << 300) + 1, 25 << 298):
        lo, hi = sqrt_interval(s)
        assert lo * lo <= s << (2 * P) <= hi * hi and hi - lo == (math.isqrt(s) ** 2 != s)


def test_f32_ints_are_exact():
    v = np.array([0.0, -0.0, 1.0, -2.5, 2.0 ** -149, 2.0 ** -126, FLT_MAX, 1e-30, 0.1], np.float32)
    for f, i in zip(v.tolist(), f32_ints(v)):
        num, den = f.as_integer_ratio()
        assert i * den == num << SCALE
    assert f32_ints(np.float32(2.0 ** -149)) == [1] and f32_ints(np.float32(-3.0)) == [-3 << SCALE]


@pytest.mark.parametrize("name", ["tiny_n3_prices", "tiny_n7_noprice", "coincident_n3", "wide_n16", "wide_exact_n3", "prices_huge",
                                  "prices_negative", "size_n63"])
def test_filter_matches_all_pairs(name):
    d = family(name)
    b = min(d["x"].shape[0], 24)
    p = None if d["p"] is None else d["p"][:b]
    full = exact_certificate(d["x"][:b], d["y"][:b], d["a"][:b], p, all_pairs=True)
    filt = exact_certificate(d["x"][:b], d["y"][:b], d["a"][:b], p)
    for f, g in zip(full, filt):
        assert (f.l_lo, f.l_hi, f.u_lo, f.u_hi) == (g.l_lo, g.l_hi, g.u_lo, g.u_hi)
        assert g.scale_l <= f.scale_l


@pytest.mark.parametrize("name", ["tiny_n5_prices", "size_n65", "prices_negative", "coincident_n64"])
def test_midpoint_matches_numpy_certificate(name):
    d = family(name)
    b = min(d["x"].shape[0], 64)
    want, wstatus = dual_bound(d["x"][:b], d["y"][:b], d["a"][:b], None if d["p"] is None else d["p"][:b])
    ref = reference(name)[:b]
    got = np.array([r.mid() for r in ref])
    assert np.array_equal(wstatus, [1 if r.u_lo is not None else 0 for r in ref])
    scale = np.array([[r.scale_l, r.scale_u] for r in ref]) / d["x"].shape[1]
    assert (np.abs(got - want) <= 1e-12 * np.maximum(np.abs(want), scale)).all(), (got, want)


def test_pythagorean_pairs_give_points():
    x = np.zeros((4, 1, 3), np.float32)
    y = np.array([[[3, 4, 0]], [[1, 2, 2]], [[-3 * 2.0 ** -20, 0, 4 * 2.0 ** -20]], [[2.0 ** 40, 2 * 2.0 ** 40, -2 * 2.0 ** 40]]],
                 np.float32)
    ref = exact_certificate(x, y, np.zeros((4, 1), np.int32))
    for r, want in zip(ref, (5.0, 3.0, 5 * 2.0 ** -20, 3 * 2.0 ** 40)):
        assert r.l_lo == r.l_hi == r.u_lo == r.u_hi
        assert r.l_lo == int(want * 2 ** 60) << (UNIT - 60)
    for r in reference("pythagorean_n3"):
        assert r.l_lo == r.l_hi == r.u_lo == r.u_hi


@pytest.mark.parametrize("name", ["tiny_n2_prices", "wide_n33", "wide_exact_n3", "size_n64"])
def test_interval_widths(name):
    for r in reference(name):
        assert r.l_hi - r.l_lo <= (r.scale_l * 2.0 ** -100) * (1 << UNIT) + 1
        assert r.u_hi - r.u_lo <= (r.scale_u * 2.0 ** -100) * (1 << UNIT) + 1


def test_tolerance_rejects_fp32_evaluation():
    """An fp32 evaluation of d (directed, so still sound) is ~1e-7 relative away: far outside the tolerance."""
    name = "tiny_n1_noprice"
    d, ref = family(name), reference(name)
    x1, x2 = d["x"].astype(np.float64), d["y"].astype(np.float64)
    s = ((x1 - x2) ** 2).sum(-1)[:, 0]
    lo32 = np.nextafter(np.sqrt(s).astype(np.float32), np.float32(-np.inf)).astype(np.float64)   # a sound fp32 value
    bounds = np.stack([lo32, np.full_like(lo32, np.inf)], 1)
    bad = check_bounds(bounds, np.ones(len(ref), np.int32), ref)
    assert sum("lower" in m and "looser" in m for m in bad) > len(ref) // 2


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def vp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def gpu_dual_bound(pkg, dev, x, y, a, p, stream=None):
    """psd_emd_dual_bound on host arrays; returns (bounds, status) as numpy."""
    import torch
    b, n, _ = x.shape
    tx, ty = torch.from_numpy(np.ascontiguousarray(x)).to(dev), torch.from_numpy(np.ascontiguousarray(y)).to(dev)
    ta = torch.from_numpy(np.ascontiguousarray(a, np.int32)).to(dev)
    tp = None if p is None else torch.from_numpy(np.ascontiguousarray(p, np.float32)).to(dev)
    bounds = torch.full((b, 2), -7.0, device=dev, dtype=torch.float64)
    status = torch.full((b,), 7, device=dev, dtype=torch.int32)
    if stream is not None:
        stream.wait_stream(torch.cuda.current_stream())
    s = pkg._lib.stream_of(tx) if stream is None else ctypes.c_void_p(stream.cuda_stream)
    rc = pkg._lib.lib.psd_emd_dual_bound(vp(tx), vp(ty), b, n, vp(ta), vp(tp), vp(bounds), vp(status), s)
    assert rc == 1, pkg._lib.last_error()
    torch.cuda.synchronize()
    return bounds.cpu().numpy(), status.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(FAMILIES))
def test_gpu_bounds_exact(pkg, cuda, name):
    d = family(name)
    bounds, status = gpu_dual_bound(pkg, cuda, d["x"], d["y"], d["a"], d["p"])
    assert_exact(bounds, status, reference(name))
    if name.startswith("coincident"):
        assert (bounds[:, 1] == 0).all()          # the matching's own cost, exactly


@pytest.mark.gpu
def test_gpu_null_and_zero_prices_bit_identical(pkg, cuda):
    z, nul = family("prices_zero"), family("prices_null")
    assert np.array_equal(z["x"], nul["x"]) and np.array_equal(z["a"], nul["a"])
    bz, sz = gpu_dual_bound(pkg, cuda, z["x"], z["y"], z["a"], z["p"])
    bn, sn = gpu_dual_bound(pkg, cuda, nul["x"], nul["y"], nul["a"], None)
    assert np.array_equal(bz.view(np.int64), bn.view(np.int64)) and np.array_equal(sz, sn)


def _certified(pkg, dev, x, y, eps_end, max_iters=20000):
    import torch
    b, n, _ = x.shape
    tx, ty = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    dist, ass, price = torch.empty(b, n, device=dev), torch.empty(b, n, device=dev, dtype=torch.int32), torch.empty(b, n, device=dev)
    bounds, status = torch.empty(b, 2, device=dev, dtype=torch.float64), torch.empty(b, device=dev, dtype=torch.int32)
    rc = pkg._lib.lib.psd_emd_certified(vp(tx), vp(ty), b, n, 0.05, eps_end, 4.0, max_iters, vp(dist), vp(ass), vp(price),
                                        vp(bounds), vp(status), pkg._lib.stream_of(tx))
    assert rc == 1, pkg._lib.last_error()
    torch.cuda.synchronize()
    return [t.cpu().numpy() for t in (dist, ass, price, bounds, status)]


@pytest.mark.gpu
@pytest.mark.parametrize("kind,n", [("uniform", 1024), ("clustered", 1024), ("uniform", 2048), ("clustered", 2048)])
def test_gpu_certified_outputs_exact(pkg, cuda, kind, n):
    """psd_emd_certified's own (assignment, prices) and bounds, against the exact certificate."""
    x, y = make_clouds(kind, 2, n, n, seed=600 + n)
    _, ass, price, bounds, status = _certified(pkg, cuda, x, y, 1e-4)
    assert (status == 1).all()
    assert_exact(bounds, status, exact_certificate(x, y, ass, price))


@pytest.mark.gpu
def test_gpu_training_setting_exact(pkg, cuda):
    """The (assignment, price) that the 14-tensor psd_emd_forward leaves at the training setting."""
    import torch
    b, n = 2, 1024
    x, y = make_clouds("uniform", b, n, n, seed=27)
    tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
    z = lambda dt=torch.float32: torch.zeros(b, n, device=cuda, dtype=dt)
    dist, ass, price, inv = z(), z(torch.int32) - 1, z(), z(torch.int32) - 1
    assert pkg._lib.lib.psd_emd_forward(vp(tx), vp(ty), b, n, n, vp(dist), vp(ass), vp(price), vp(inv), vp(z(torch.int32)),
                                        vp(z()), vp(z()), None, None, None, None, None, 0.05, 3000, None) == 1
    a, p = ass.cpu().numpy(), price.cpu().numpy()
    bounds, status = gpu_dual_bound(pkg, cuda, x, y, a, p)
    assert_exact(bounds, status, exact_certificate(x, y, a, p))


@pytest.mark.gpu
def test_gpu_batch_limit(pkg, cuda):
    """b = 65535 one-point clouds (the grid's y limit), exact; b = 65536 is refused before any device work."""
    import torch
    b = 65535
    rng = np.random.default_rng(31)
    x, y = rng.random((b, 1, 3), dtype=np.float32), rng.random((b, 1, 3), dtype=np.float32)
    p = rng.random((b, 1), dtype=np.float32) - np.float32(0.5)
    a = np.zeros((b, 1), np.int32)
    bounds, status = gpu_dual_bound(pkg, cuda, x, y, a, p)
    assert_exact(bounds, status, exact_certificate(x, y, a, p))
    t = torch.zeros(8 * (b + 1), device=cuda, dtype=torch.float64)
    assert pkg._lib.lib.psd_emd_dual_bound(vp(t), vp(t), b + 1, 1, vp(t), vp(t), vp(t), vp(t), None) == -1
    torch.cuda.synchronize()
    assert float(t.abs().sum()) == 0.0


@pytest.mark.gpu
def test_gpu_largest_cloud(pkg, cuda):
    """n = 2^20 (a 128 KB permutation bitmap): y = x[perm], a = its inverse, prices 0 (cloud 0) and 2^-3 (cloud 1).  Every
    term is exact, so both bounds are exactly 0."""
    n = 1 << 20
    rng = np.random.default_rng(32)
    x = rng.random((2, n, 3), dtype=np.float32)
    perm = np.stack([rng.permutation(n) for _ in range(2)])
    y = np.ascontiguousarray(np.take_along_axis(x, perm[..., None], 1))
    a = np.argsort(perm, axis=1).astype(np.int32)
    p = np.zeros((2, n), np.float32)
    p[1] = 0.125
    bounds, status = gpu_dual_bound(pkg, cuda, x, y, a, p)
    assert (status == 1).all() and (bounds == 0).all(), bounds


@pytest.mark.gpu
def test_gpu_non_permutations_at_bitmap_word_edges(pkg, cuda):
    """Objects 31 / 32 taken twice, n - 1 taken twice, -1 and n: status 0 and a NaN upper bound; the lower bound does not
    depend on the assignment and is the same in every cloud, bit for bit."""
    n = 100
    rng = np.random.default_rng(33)
    x1, y1 = rng.random((1, n, 3), dtype=np.float32), rng.random((1, n, 3), dtype=np.float32)
    base = rng.permutation(n).astype(np.int32)
    rows = [base.copy()]
    for edit in ((31, 31), (32, 32), (31, 32), (n - 1, n - 1), (-1,), (n,)):
        a = base.copy()
        if len(edit) == 2 and edit[0] == edit[1]:
            a[np.flatnonzero(a != edit[0])[0]] = edit[0]            # the object twice (and one object free)
        elif len(edit) == 2:
            i31, i32 = np.flatnonzero(a == 31)[0], np.flatnonzero(a == 32)[0]
            a[i31] = 32                                             # 32 twice, 31 free
        else:
            a[7] = edit[0]
        rows.append(a)
    b = len(rows)
    x, y = np.repeat(x1, b, 0), np.repeat(y1, b, 0)
    a = np.stack(rows)
    p = np.repeat(rng.random((1, n), dtype=np.float32), b, 0)
    bounds, status = gpu_dual_bound(pkg, cuda, x, y, a, p)
    assert status.tolist() == [1] + [0] * (b - 1)
    assert np.isnan(bounds[1:, 1]).all()
    assert len(set(bounds[:, 0].view(np.int64).tolist())) == 1
    assert_exact(bounds, status, exact_certificate(x, y, a, p))


@pytest.mark.gpu
def test_gpu_reproducible_across_streams_and_graphs(pkg, cuda):
    """The same call gives the same bits on the default stream, on a side stream, after unrelated kernels, and replayed
    from a captured CUDA graph."""
    import torch
    d = family("size_n2049")
    x, y, a, p = d["x"], d["y"], d["a"].copy(), d["p"]
    a[1, 3] = a[1, 4]      # one cloud without a permutation
    want, wstatus = gpu_dual_bound(pkg, cuda, x, y, a, p)
    assert wstatus.tolist() == [1, 0]
    runs = [gpu_dual_bound(pkg, cuda, x, y, a, p, stream=torch.cuda.Stream())]
    junk = torch.randn(4096, 4096, device=cuda)
    for _ in range(3):
        junk = junk @ junk.T / 64
    pkg.emdModule()(torch.rand(4, 1024, 3, device=cuda), torch.rand(4, 1024, 3, device=cuda), 0.005, 50)
    gpu_dual_bound(pkg, cuda, y, x, a[::-1].copy(), None)
    runs.append(gpu_dual_bound(pkg, cuda, x, y, a, p))
    b, n, _ = x.shape
    tx, ty = torch.from_numpy(x).to(cuda), torch.from_numpy(y).to(cuda)
    ta, tp = torch.from_numpy(a).to(cuda), torch.from_numpy(p).to(cuda)
    bounds, status = torch.empty(b, 2, device=cuda, dtype=torch.float64), torch.empty(b, device=cuda, dtype=torch.int32)
    call = lambda: pkg._lib.lib.psd_emd_dual_bound(vp(tx), vp(ty), b, n, vp(ta), vp(tp), vp(bounds), vp(status),
                                                   pkg._lib.stream_of(tx))
    assert call() == 1
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        assert call() == 1, pkg._lib.last_error()
    bounds.fill_(float("inf"))
    status.fill_(7)
    g.replay()
    torch.cuda.synchronize()
    runs.append((bounds.cpu().numpy(), status.cpu().numpy()))
    for got, st in runs:
        assert np.array_equal(got.view(np.int64), want.view(np.int64)) and np.array_equal(st, wstatus)


# ---------------------------------------------------------------------------------------------------------------------
# non-finite input: a cloud with a NaN or infinite coordinate has no certificate
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_dual_bound_non_finite(pkg, cuda):
    """NaN / +-inf coordinates in xyz1 or xyz2: both bounds NaN, status 0.  A NaN price: the lower bound NaN, the upper
    bound and status as with finite prices.  The other clouds of the batch are the same bits as on their own."""
    n = 65
    rng = np.random.default_rng(34)
    b = 7
    x, y = rng.random((b, n, 3), dtype=np.float32), rng.random((b, n, 3), dtype=np.float32)
    a = np.stack([rng.permutation(n) for _ in range(b)]).astype(np.int32)
    p = rng.random((b, n), dtype=np.float32)
    x[1, 5, 0] = np.nan
    y[2, 64, 2] = np.inf
    x[3, 0, 1] = -np.inf
    y[4, 10, 1] = np.nan
    p[5, 3] = np.nan
    bounds, status = gpu_dual_bound(pkg, cuda, x, y, a, p)
    assert status.tolist() == [1, 0, 0, 0, 0, 1, 1], status
    assert np.isnan(bounds[1:5]).all(), bounds
    assert np.isnan(bounds[5, 0]) and np.isfinite(bounds[5, 1])
    clean = [0, 5, 6]
    pc = p[clean].copy()
    pc[1, 3] = 0.0
    alone, st = gpu_dual_bound(pkg, cuda, x[clean], y[clean], a[clean], pc)
    assert np.array_equal(st, [1, 1, 1])
    assert np.array_equal(bounds[[0, 6]].view(np.int64), alone[[0, 2]].view(np.int64))
    assert bounds[5, 1].view(np.int64) == alone[1, 1].view(np.int64)
    # NULL prices: the same verdicts for the coordinates
    bn, sn = gpu_dual_bound(pkg, cuda, x, y, a, None)
    assert sn.tolist() == [1, 0, 0, 0, 0, 1, 1] and np.isnan(bn[1:5]).all() and np.isfinite(bn[[0, 5, 6]]).all()


@pytest.mark.gpu
def test_gpu_certified_non_finite(pkg, cuda):
    """psd_emd_certified on a batch with a NaN coordinate in xyz1 (cloud 0) and an infinite one in xyz2 (cloud 1): no
    certificate for them, and the clean cloud 2 is the same bits as on its own."""
    n = 1024
    x, y = make_clouds("uniform", 3, n, n, seed=35)
    x[0, 100, 1] = np.nan
    y[1, 1000, 0] = np.inf
    dist, ass, price, bounds, status = _certified(pkg, cuda, x, y, 1e-3)
    assert status.tolist() == [0, 0, 1], status
    assert np.isnan(bounds[:2]).all(), bounds
    alone = _certified(pkg, cuda, x[2:], y[2:], 1e-3)
    for got, want in zip((dist, ass, price, bounds, status), alone):
        assert np.array_equal(got[2:].view(np.uint8), want.view(np.uint8))


# ---------------------------------------------------------------------------------------------------------------------
# a result that is not a matching: gradients and the metric
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_gradient_of_shared_objects(pkg, oracle, cuda, monkeypatch):
    """A budget-exhausted run ends with objects that several points share: xyz2's gradient sums their terms (fp64
    np.add.at reference), and certified_emd_distance reports a NaN gap."""
    import torch
    c = case(oracle, "uniform", 2, 1024, 1e-4, max_iters_per_phase=3)
    x, y = c["x"], c["y"]
    tx = torch.from_numpy(x).to(cuda).requires_grad_(True)
    ty = torch.from_numpy(y).to(cuda).requires_grad_(True)
    dist, ass, bounds, status = pkg.emd_certified(tx, ty, eps_end=1e-4, max_iters_per_phase=3)
    a = ass.cpu().numpy()
    assert (status.cpu().numpy() == 0).all() and np.isnan(bounds.cpu().numpy()[:, 1]).all()
    assert max(np.bincount(r[r >= 0], minlength=1024).max() for r in a) > 1      # shared objects
    w = np.random.default_rng(36).random((2, 1024), dtype=np.float32)
    (dist * torch.from_numpy(w).to(cuda)).sum().backward()
    g1 = oracle.emd_backward(x, y, w, a)
    assert np.array_equal(tx.grad.cpu().numpy(), g1)
    want = np.zeros(y.shape, np.float64)
    for k in range(2):
        ok = a[k] >= 0
        np.add.at(want[k], a[k][ok], -g1[k][ok].astype(np.float64))
    got = ty.grad.cpu().numpy().astype(np.float64)
    mult = np.stack([np.bincount(r[r >= 0], minlength=1024) for r in a])[..., None]     # terms per object
    mag = np.zeros(y.shape, np.float64)
    for k in range(2):
        ok = a[k] >= 0
        np.add.at(mag[k], a[k][ok], np.abs(g1[k][ok]).astype(np.float64))
    assert (np.abs(got - want) <= mult * 2.0 ** -23 * mag).all()
    real = pkg.emd_module.emd_certified
    monkeypatch.setattr(pkg.metrics.emd_func, "emd_certified",
                        lambda p1, p2, eps_end: real(p1, p2, eps_end=eps_end, max_iters_per_phase=3))
    value, gap = pkg.certified_emd_distance(tx.detach(), ty.detach(), eps_end=1e-4)
    assert math.isfinite(value) and math.isnan(gap)
