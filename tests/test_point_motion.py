"""Frame-to-frame motion (``silent_estimate_motion``, ``_ops.estimate_motion``, ``LineEndPipeline.run_frames_motion`` /
``run_host_motion``).

Per pair of consecutive frames, a seeded RANSAC over the correspondences the matcher leaves (splitmix64 draws, a float64
three-point affine fit, float32 scoring) and one least-squares refit in a fixed summation order; see ``PointMotion``.
``motion_reference`` restates that definition in numpy; the CPU tests check it against a scalar restatement and
hand-built cases, and check the binding, every status code and the Python validation. The GPU tests check the device
results bit for bit against the reference, the pipeline on every route the matches serve, and the motion recovered
from a panned and from an affinely warped scene.
"""
import ctypes
import math
import os

import numpy as np
import pytest

from test_point_matches import PAN, PIPELINE_CASES, _assert_matches, _check_records, panned_frames
from test_point_records import CASES, SENTINEL, SQRT2, _lib_status, _np, _pipe
from pysilent_b200 import _lib

M64 = (1 << 64) - 1
THREADS, WARPS = 256, 8   # the refit's fixed summation order


# ---- the reference ---------------------------------------------------------------------------------------------------------

def splitmix64(z):
    """Vigna's splitmix64 step on uint64 arrays (64-bit wrapping)."""
    with np.errstate(over="ignore"):
        z = np.asarray(z, np.uint64) + np.uint64(0x9e3779b97f4a7c15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xbf58476d1ce4e5b9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94d049bb133111eb)
        return z ^ (z >> np.uint64(31))


def draws(seed, f, hypotheses, m):
    """[H, 3] correspondence indices: mulhi64(splitmix64(seed ^ splitmix64((f << 32) | (h << 2) | d)), M)."""
    assert 0 < m < 2 ** 32
    h = np.arange(hypotheses, dtype=np.uint64)[:, None]
    d = np.arange(3, dtype=np.uint64)[None]
    key = (np.uint64(f) << np.uint64(32)) | (h << np.uint64(2)) | d
    u = splitmix64(np.uint64(seed) ^ splitmix64(key))
    hi, lo = u >> np.uint64(32), u & np.uint64(0xffffffff)
    mm = np.uint64(m)
    return ((hi * mm + ((lo * mm) >> np.uint64(32))) >> np.uint64(32)).astype(np.int64)


def fit3(c, k):
    """Hypotheses of the draws k [H, 3] over c [M, 4] float32: (t [H, 6] float64, live [H])."""
    k = np.asarray(k)
    p0, p1, p2 = (c[k[:, j]].astype(np.float64) for j in range(3))
    live = (k[:, 0] != k[:, 1]) & (k[:, 0] != k[:, 2]) & (k[:, 1] != k[:, 2])
    y0, x0 = p0[:, 0], p0[:, 1]
    dy1, dx1, dy2, dx2 = p1[:, 0] - y0, p1[:, 1] - x0, p2[:, 0] - y0, p2[:, 1] - x0
    det = dy1 * dx2 - dx1 * dy2
    live &= np.abs(det) >= 1.0
    t = np.zeros((len(k), 6))
    with np.errstate(divide="ignore", invalid="ignore"):
        for r in range(2):
            du1, du2 = p1[:, 2 + r] - p0[:, 2 + r], p2[:, 2 + r] - p0[:, 2 + r]
            a = (du1 * dx2 - dx1 * du2) / det
            b = (dy1 * du2 - du1 * dy2) / det
            t[:, 3 * r], t[:, 3 * r + 1], t[:, 3 * r + 2] = a, b, p0[:, 2 + r] - (a * y0 + b * x0)
    return t, live


def inliers(t, c, threshold):
    """[H, M] inlier masks of the models t [H, 6] (float32 once, every operation rounded)."""
    with np.errstate(over="ignore", invalid="ignore"):
        m = np.atleast_2d(t).astype(np.float32)
        thr2 = np.float32(threshold) * np.float32(threshold)
        y0, x0, y1, x1 = (c[None, :, j] for j in range(4))
        ey = y1 - ((m[:, 0:1] * y0 + m[:, 1:2] * x0) + m[:, 2:3])
        ex = x1 - ((m[:, 3:4] * y0 + m[:, 4:5] * x0) + m[:, 5:6])
        return (ey * ey + ex * ex) <= thr2


def fixed_sum(terms):
    """Sum of terms [M, Q] in the refit's order: thread t over k = t, t + 256, ...; xor butterfly within each warp;
    the warps' lane-0 sums in warp order."""
    m, q = terms.shape
    pad = np.concatenate([terms, np.zeros(((-m) % THREADS, q))]).reshape(-1, THREADS, q)
    s = np.zeros((THREADS, q))
    for row in pad:
        s = s + row
    s = s.reshape(WARPS, 32, q)
    lanes = np.arange(32)
    for b in (16, 8, 4, 2, 1):
        s = s + s[:, lanes ^ b]
    total = s[0, 0]
    for w in range(1, WARPS):
        total = total + s[w, 0]
    return total


def refit(c, mask, first):
    """One least-squares step on the correspondences c[mask], relative to c[first]: t [6] float64."""
    p = c[first].astype(np.float64)
    py, px, qy, qx = (float(v) for v in p)
    v = c.astype(np.float64)
    Y, X, U, V = v[:, 0] - py, v[:, 1] - px, v[:, 2] - qy, v[:, 3] - qx
    terms = np.stack([Y, X, Y * Y, Y * X, X * X, U, Y * U, X * U, V, Y * V, X * V], axis=1)
    S = [float(s) for s in fixed_sum(np.where(mask[:, None], terms, 0.0))]
    n = float(mask.sum())
    Sy, Sx, Syy, Syx, Sxx = S[:5]
    c00, c01, c02 = Sxx * n - Sx * Sx, Sx * Sy - Syx * n, Syx * Sx - Sxx * Sy
    c11, c12, c22 = Syy * n - Sy * Sy, Syx * Sy - Syy * Sx, Syy * Sxx - Syx * Syx
    det = (Syy * c00 + Syx * c01) + Sy * c02
    t = np.zeros(6)
    with np.errstate(divide="ignore", invalid="ignore"):
        for o, (r0, r1, r2, q) in enumerate(((S[6], S[7], S[5], qy), (S[9], S[10], S[8], qx))):
            num = np.array([(c00 * r0 + c01 * r1) + c02 * r2, (c01 * r0 + c11 * r1) + c12 * r2,
                            (c02 * r0 + c12 * r1) + c22 * r2])
            a, b, cc = num / np.float64(det)
            t[3 * o: 3 * o + 3] = a, b, (q + cc) - (a * py + b * px)
    return t


def correspondences(frame_offsets, frame_yx, nxt, count, f):
    """(rows, c [M, 4] float32) of pair f."""
    cap = len(nxt)
    rows = int(min(max(int(count), 0), cap))
    lo = min(max(int(frame_offsets[f]), 0), rows)
    hi = min(max(int(frame_offsets[f + 1]), lo), rows)
    i = np.arange(lo, hi)
    j = nxt[lo:hi]
    ok = (j >= 0) & (j < rows)
    i, j = i[ok], j[ok]
    c = np.concatenate([frame_yx[i], frame_yx[j]], axis=1).astype(np.float32).reshape(-1, 4)
    fin = np.isfinite(c).all(axis=1)
    return i[fin], c[fin]


def motion_reference(frame_offsets, frame_yx, nxt, count, hypotheses, threshold, seed):
    """``(transform, inlier_count, matched, inlier)`` as ``PointMotion`` defines them, and the winning h per pair (-1
    without one)."""
    frame_offsets, frame_yx, nxt = np.asarray(frame_offsets), np.asarray(frame_yx, np.float32), np.asarray(nxt)
    pairs = len(frame_offsets) - 2
    T = np.full((pairs, 2, 3), np.nan)
    n_in = np.zeros(pairs, np.int64)
    matched = np.zeros(pairs, np.int64)
    flags = np.zeros(len(nxt), np.uint8)
    best_h = np.full(pairs, -1)
    for f in range(pairs):
        rows, c = correspondences(frame_offsets, frame_yx, nxt, count, f)
        m = len(rows)
        matched[f] = m
        if m < 3:
            continue
        k = draws(seed, f, hypotheses, m)
        t, live = fit3(c, k)
        if not live.any():
            continue
        counts = np.zeros(hypotheses, np.int64)
        for s in range(0, hypotheses, 64):
            counts[s:s + 64] = np.where(live[s:s + 64], inliers(t[s:s + 64], c, threshold).sum(axis=1), -1)
        h = int(np.argmax(counts))   # the first of the largest
        best_h[f] = h
        mask = inliers(t[h], c, threshold)[0]
        t2 = refit(c, mask, k[h, 0])
        mask2 = inliers(t2, c, threshold)[0]
        keep = np.isfinite(t2).all() and mask2.sum() >= mask.sum()
        final, fmask = (t2, mask2) if keep else (t[h], mask)
        T[f] = final.reshape(2, 3)
        n_in[f] = fmask.sum()
        flags[rows[fmask]] = 1
    return (T, n_in, matched, flags), best_h


def scalar_motion(frame_offsets, frame_yx, nxt, count, hypotheses, threshold, seed):
    """The definition again, one scalar at a time: Python integers for the hash, Python floats (float64) for the fits
    and the sums, numpy float32 scalars for the scores."""
    f32 = np.float32

    def sm(z):
        z = (z + 0x9e3779b97f4a7c15) & M64
        z = ((z ^ (z >> 30)) * 0xbf58476d1ce4e5b9) & M64
        z = ((z ^ (z >> 27)) * 0x94d049bb133111eb) & M64
        return z ^ (z >> 31)

    def score(t, c):
        m = [f32(v) for v in t]
        t2 = f32(f32(threshold) * f32(threshold))
        out = []
        for y0, x0, y1, x1 in c:
            ey = f32(y1 - f32(f32(f32(m[0] * y0) + f32(m[1] * x0)) + m[2]))
            ex = f32(x1 - f32(f32(f32(m[3] * y0) + f32(m[4] * x0)) + m[5]))
            out.append(bool(f32(f32(ey * ey) + f32(ex * ex)) <= t2))
        return out

    pairs = len(frame_offsets) - 2
    T = np.full((pairs, 2, 3), np.nan)
    n_in, matched, flags = np.zeros(pairs, np.int64), np.zeros(pairs, np.int64), np.zeros(len(nxt), np.uint8)
    rows_used = int(min(max(int(count), 0), len(nxt)))
    with np.errstate(over="ignore", invalid="ignore"):
        for f in range(pairs):
            lo = min(max(int(frame_offsets[f]), 0), rows_used)
            hi = min(max(int(frame_offsets[f + 1]), lo), rows_used)
            rows, c = [], []
            for i in range(lo, hi):
                j = int(nxt[i])
                if 0 <= j < rows_used:
                    v = [f32(frame_yx[i][0]), f32(frame_yx[i][1]), f32(frame_yx[j][0]), f32(frame_yx[j][1])]
                    if all(math.isfinite(x) for x in v):
                        rows.append(i)
                        c.append(v)
            m = len(c)
            matched[f] = m
            if m < 3:
                continue
            best = None
            for h in range(hypotheses):
                k = [(sm(seed ^ sm((f << 32) | (h << 2) | d)) * m) >> 64 for d in range(3)]
                if len(set(k)) < 3:
                    continue
                (y0, x0, a0, b0), p1, p2 = (c[k[0]], c[k[1]], c[k[2]])
                y0, x0 = float(y0), float(x0)
                dy1, dx1, dy2, dx2 = float(p1[0]) - y0, float(p1[1]) - x0, float(p2[0]) - y0, float(p2[1]) - x0
                D = dy1 * dx2 - dx1 * dy2
                if not abs(D) >= 1:
                    continue
                t = []
                for r in range(2):
                    u0 = float(c[k[0]][2 + r])
                    du1, du2 = float(p1[2 + r]) - u0, float(p2[2 + r]) - u0
                    a = (du1 * dx2 - dx1 * du2) / D
                    b = (dy1 * du2 - du1 * dy2) / D
                    t += [a, b, u0 - (a * y0 + b * x0)]
                n = sum(score(t, c))
                if best is None or n > best[0]:
                    best = (n, h, t, k[0])
            if best is None:
                continue
            n, h, t, k0 = best
            mask = score(t, c)
            py, px, qy, qx = (float(v) for v in c[k0])
            part = [[0.0] * 11 for _ in range(THREADS)]
            for kk in range(m):
                if mask[kk]:
                    Y, X = float(c[kk][0]) - py, float(c[kk][1]) - px
                    U, V = float(c[kk][2]) - qy, float(c[kk][3]) - qx
                    for q, term in enumerate((Y, X, Y * Y, Y * X, X * X, U, Y * U, X * U, V, Y * V, X * V)):
                        part[kk % THREADS][q] += term
            S = []
            for q in range(11):
                s = [part[tt][q] for tt in range(THREADS)]
                for b in (16, 8, 4, 2, 1):
                    s = [s[tt] + s[tt ^ b] for tt in range(THREADS)]
                tot = s[0]
                for w in range(1, WARPS):
                    tot = tot + s[32 * w]
                S.append(tot)
            nn = float(sum(mask))
            Sy, Sx, Syy, Syx, Sxx = S[:5]
            c00, c01, c02 = Sxx * nn - Sx * Sx, Sx * Sy - Syx * nn, Syx * Sx - Sxx * Sy
            c11, c12, c22 = Syy * nn - Sy * Sy, Syx * Sy - Syy * Sx, Syy * Sxx - Syx * Syx
            det = (Syy * c00 + Syx * c01) + Sy * c02
            t2 = []
            for r0, r1, r2, q in ((S[6], S[7], S[5], qy), (S[9], S[10], S[8], qx)):
                nums = ((c00 * r0 + c01 * r1) + c02 * r2, (c01 * r0 + c11 * r1) + c12 * r2,
                        (c02 * r0 + c12 * r1) + c22 * r2)
                a, b, cc = (float(np.float64(v) / np.float64(det)) for v in nums)
                t2 += [a, b, (q + cc) - (a * py + b * px)]
            mask2 = score(t2, c) if all(math.isfinite(v) for v in t2) else [False] * m
            keep = all(math.isfinite(v) for v in t2) and sum(mask2) >= sum(mask)
            final, fmask = (t2, mask2) if keep else (t, mask)
            T[f] = np.array(final).reshape(2, 3)
            n_in[f] = sum(fmask)
            for kk in range(m):
                flags[rows[kk]] = int(fmask[kk])
    return T, n_in, matched, flags


def motion_rows(seed, per_frame, models=None, outliers=0.3, unmatched=0.2, nan=0.0, noise=0.3, size=(1080, 1920),
                junk=0):
    """Records and links of ``len(per_frame)`` frames: frame_offsets, frame_yx [K, 2] float32 and next [K]. Row i of
    frame f links to a row of frame f + 1 (or -1, share ``unmatched``) whose coordinates are ``models[f]`` applied to
    row i's plus Gaussian noise, or random coordinates (share ``outliers``); a share ``nan`` of rows has a NaN axis.
    ``junk`` rows past K link anywhere; they lie outside the call."""
    rs = np.random.RandomState(seed)
    per_frame = list(per_frame)
    B = len(per_frame)
    offs = np.concatenate([[0], np.cumsum(per_frame)]).astype(np.int64)
    K = int(offs[-1])
    H, W = size
    yx = np.stack([rs.uniform(0, H - 1, K), rs.uniform(0, W - 1, K)], axis=1)
    nxt = np.full(K + junk, -1, np.int64)
    for f in range(B - 1):
        T = np.asarray(models[f] if models is not None else
                       [[1 + rs.normal(0, .02), rs.normal(0, .02), rs.normal(0, 5)],
                        [rs.normal(0, .02), 1 + rs.normal(0, .02), rs.normal(0, 5)]])
        src = np.arange(offs[f], offs[f + 1])
        dst = rs.permutation(np.arange(offs[f + 1], offs[f + 2]))
        n = min(len(src), len(dst))
        src = rs.permutation(src)[:n]
        dst = dst[:n]
        keep = rs.rand(n) >= unmatched
        src, dst = src[keep], dst[keep]
        moved = yx[src] @ T[:, :2].T + T[:, 2] + rs.normal(0, noise, (len(src), 2))
        bad = rs.rand(len(src)) < outliers
        moved[bad] = np.stack([rs.uniform(0, H, bad.sum()), rs.uniform(0, W, bad.sum())], axis=1)
        yx[dst] = moved
        nxt[src] = dst
    yx = yx.astype(np.float32)
    if nan:
        idx = np.nonzero(rs.rand(K) < nan)[0]
        yx[idx, rs.randint(0, 2, len(idx))] = np.nan
    allyx = np.concatenate([yx, rs.uniform(0, 100, (junk, 2)).astype(np.float32)])
    if junk:
        nxt[K:] = rs.randint(0, K + junk, junk)
    return offs, allyx, nxt, K


EXACT_T = np.array([[1.25, -0.5, 3.0], [0.25, 0.75, -7.5]])


def exact_rows(m, B=2):
    """m correspondences per pair on integer points, moved by EXACT_T: every value exact in float32."""
    rs = np.random.RandomState(m)
    src = rs.randint(0, 200, (m, 2)).astype(np.float64)
    frames = [src]
    for _ in range(B - 1):
        frames.append(frames[-1] @ EXACT_T[:, :2].T + EXACT_T[:, 2])
    yx = np.concatenate(frames).astype(np.float32)
    assert np.array_equal(yx.astype(np.float64), np.concatenate(frames))
    nxt = np.full(B * m, -1, np.int64)
    nxt[:(B - 1) * m] = np.arange(m, B * m)
    return np.arange(0, (B + 1) * m, m, dtype=np.int64), yx, nxt, B * m


def _case(name):
    """Small hand-built cases: (frame_offsets, frame_yx, next, count, hypotheses, threshold, seed)."""
    if name == "exact":
        o, yx, n, k = exact_rows(40, 3)
        return o, yx, n, k, 64, 0.5, 7
    if name == "outliers":
        o, yx, n, k = motion_rows(1, [60, 70, 50], outliers=0.35)
        return o, yx, n, k, 100, 2.0, 1
    if name == "collinear":   # every source on one line: every hypothesis is degenerate
        o, yx, n, k = exact_rows(30)
        yx[:30, 1] = 2 * yx[:30, 0] + 1
        return o, yx, n, k, 50, 2.0, 0
    if name == "repeated":   # M = 3: most draws repeat an index
        o, yx, n, k = exact_rows(3)
        return o, yx, n, k, 40, 1.0, 3
    if name.startswith("m"):
        o, yx, n, k = motion_rows(5, [int(name[1:]), 8, int(name[1:])], unmatched=0, outliers=0)
        return o, yx, n, k, 30, 2.0, 0
    if name == "nan":
        o, yx, n, k = motion_rows(2, [80, 80, 80], nan=0.2)
        return o, yx, n, k, 64, 3.0, 11
    if name == "ties":   # two motions of equal support: every hypothesis of either scores the same count
        o, yx, n, k = exact_rows(40)
        yx[60:80] = yx[20:40] + np.float32(100)
        return o, yx, n, k, 200, 0.5, 5
    if name == "one_frame":
        o, yx, n, k = motion_rows(3, [25])
        return o, yx, n, k, 10, 2.0, 0
    if name in ("count_below", "count_above", "count_negative"):
        o, yx, n, k = motion_rows(4, [50, 40, 60, 30], junk=9)
        count = dict(count_below=k - 45, count_above=len(n) + 20, count_negative=-3)[name]
        return o, yx, n, count, 64, 2.0, 2 ** 64 - 1
    raise KeyError(name)


SMALL_CASES = ("exact", "outliers", "collinear", "repeated", "m0", "m1", "m2", "m3", "nan", "ties", "one_frame",
               "count_below", "count_above", "count_negative")


def _same_f64(got, want, what):
    got, want = np.asarray(got), np.asarray(want)
    assert got.dtype == want.dtype == np.float64 and got.shape == want.shape, (what, got.dtype, got.shape, want.shape)
    nan_g, nan_w = np.isnan(got), np.isnan(want)
    assert np.array_equal(nan_g, nan_w), "%s: NaN masks differ" % what
    differ = (got.view(np.uint64) != want.view(np.uint64)) & ~nan_g
    assert not differ.any(), "%s: %d of %d values differ: %s vs %s" % (what, differ.sum(), got.size, got[differ][:4],
                                                                       want[differ][:4])


def _assert_motion(got, want, what):
    g = [_np(t) for t in got]
    _same_f64(g[0], want[0], what + " transform")
    for i, name in ((1, "inlier_count"), (2, "matched"), (3, "inlier")):
        assert g[i].dtype == want[i].dtype, (what, name, g[i].dtype)
        assert np.array_equal(g[i], want[i]), "%s %s: %d of %d differ" % (what, name, (g[i] != want[i]).sum(),
                                                                          len(want[i]))


# ---- CPU: the reference --------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", SMALL_CASES)
def test_reference_equals_the_scalar_restatement(name):
    args = _case(name)
    want = scalar_motion(*args)
    got, _ = motion_reference(*args)
    _assert_motion(got, want, name)


def test_splitmix64_and_mulhi():
    """splitmix64 from seed 0 gives Vigna's published first outputs; mulhi64 equals the 128-bit product's top half."""
    outs = [int(splitmix64(np.uint64((i * 0x9e3779b97f4a7c15) & M64))) for i in range(3)]
    assert outs == [0xe220a8397b1dcdaf, 0x6e789e6aa1b965f4, 0x06c45d188009454f]
    rs = np.random.RandomState(0)
    for m in (1, 2, 3, 1000, 2 ** 32 - 1):
        k = draws(int(rs.randint(0, 2 ** 62)), 5, 64, m)
        assert k.min() >= 0 and k.max() < m
    f, h, d, seed, m = 3, 17, 2, 12345, 999
    sm = lambda z: int(splitmix64(np.uint64(z)))  # noqa: E731
    u = sm(seed ^ sm((f << 32) | (h << 2) | d))
    assert draws(seed, f, 18, m)[h, d] == (u * m) >> 64


def test_exact_affine_is_recovered():
    args = _case("exact")
    (T, n, m, flags), _ = motion_reference(*args)
    assert list(m) == [40, 40] and list(n) == [40, 40] and flags[:80].all() and not flags[80:].any()
    np.testing.assert_allclose(T, np.stack([EXACT_T, EXACT_T]), rtol=0, atol=1e-9)


def test_reference_cases_say_what_they_are_for():
    (T, n, m, flags), best = motion_reference(*_case("outliers"))
    for f in range(2):   # the injected outliers are mostly rejected, the model is near the planted one
        assert 0.45 * m[f] < n[f] < m[f]
    (T, n, m, flags), best = motion_reference(*_case("collinear"))
    assert m[0] == 30 and np.isnan(T).all() and n[0] == 0 and not flags.any() and best[0] == -1
    (T, n, m, flags), best = motion_reference(*_case("repeated"))
    k = draws(3, 0, 40, 3)
    live = np.nonzero((k[:, 0] != k[:, 1]) & (k[:, 0] != k[:, 2]) & (k[:, 1] != k[:, 2]))[0]
    assert 0 < len(live) < 40 and best[0] == live[0] and n[0] == 3
    np.testing.assert_allclose(T[0], EXACT_T, atol=1e-9)
    for mm in (0, 1, 2):
        (T, n, m, flags), best = motion_reference(*_case("m%d" % mm))
        assert m[0] == mm and np.isnan(T[0]).all() and n[0] == 0 and best[0] == -1
    (T, n, m, flags), best = motion_reference(*_case("m3"))
    assert m[0] == 3
    (T, n, m, flags), _ = motion_reference(*_case("nan"))
    o, yx, nxt, k = _case("nan")[:4]
    assert (flags[np.isnan(yx).any(axis=1)] == 0).all() and m[0] < (nxt[:80] >= 0).sum()
    (T, n, m, flags), best = motion_reference(*_case("ties"))
    o, yx, nxt, k, H, thr, seed = _case("ties")
    t, live = fit3(correspondences(o, yx, nxt, k, 0)[1], draws(seed, 0, H, 40))
    counts = np.where(live, inliers(t, correspondences(o, yx, nxt, k, 0)[1], thr).sum(axis=1), -1)
    assert (counts == counts.max()).sum() > 1 and best[0] == np.nonzero(counts == counts.max())[0][0]
    out, _ = motion_reference(*_case("one_frame"))
    assert out[0].shape == (0, 2, 3) and out[1].shape == out[2].shape == (0,) and not out[3].any()
    for name in ("count_below", "count_above", "count_negative"):
        o, yx, nxt, count, H, thr, seed = _case(name)
        (T, n, m, flags), _ = motion_reference(o, yx, nxt, count, H, thr, seed)
        rows = int(min(max(count, 0), len(nxt)))
        assert not flags[rows:].any() and m.sum() <= rows, name
    assert (motion_reference(*_case("count_negative"))[0][2] == 0).all()


def test_threshold_at_an_exact_residual():
    """A residual of exactly the threshold is an inlier; one float32 ulp more, or a threshold one ulp less, is not."""
    t = np.array([1.0, 0.0, 5.0, 0.0, 1.0, -2.0])
    c = np.array([[10, 20, 15, 18], [10, 20, 18, 18], [10, 20, 15, 21], [10, 20, 18, 21],
                  [10, 20, np.nextafter(np.float32(18), np.float32(19)), 18]], np.float32)
    assert list(inliers(t, c, 3.0)[0]) == [True, True, True, False, False]
    assert list(inliers(t, c, np.nextafter(np.float32(3), np.float32(2)))[0]) == [True, False, False, False, False]


# ---- CPU: binding, status codes, validation ------------------------------------------------------------------------------

def test_symbols_exported_and_bound(built_lib):
    for name in ("silent_motion_workspace_bytes", "silent_estimate_motion"):
        assert name in _lib.SYMBOLS and hasattr(built_lib, name)
    args = built_lib.silent_estimate_motion.argtypes
    assert len(args) == 16 and args[7] is ctypes.c_float and args[8] is ctypes.c_uint64
    assert built_lib.silent_motion_workspace_bytes(1000) == 24000
    assert built_lib.silent_motion_workspace_bytes(0) == built_lib.silent_motion_workspace_bytes(-5) == 0
    header = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include",
                               "silent_b200.h")).read()
    assert "int silent_estimate_motion(" in header and "#define SILENT_MOTION_HYPOTHESES_MAX 4096" in header
    assert _lib.MOTION_HYPOTHESES_MAX == 4096


def test_status_codes_before_any_cuda_call(built_lib):
    """Every check fails on the host. A call that passes them all reaches CUDA, so it is made only without a device
    (the pointers here are fake)."""
    L = built_lib
    fake = ctypes.c_void_p(256)
    good = dict(offsets=fake, yx=fake, next=fake, count=fake, capacity=8, batch=3, hyp=256, thr=2.0, seed=0, ws=fake,
                ws_bytes=8 * 24, transform=fake, inlier_count=fake, matched=fake, inlier=fake)

    def call(**kw):
        a = dict(good, **kw)
        return L.silent_estimate_motion(a["offsets"], a["yx"], a["next"], a["count"], a["capacity"], a["batch"],
                                        a["hyp"], a["thr"], a["seed"], a["ws"], a["ws_bytes"], a["transform"],
                                        a["inlier_count"], a["matched"], a["inlier"], None)
    for kw in (dict(capacity=-1), dict(batch=0), dict(batch=-2), dict(offsets=None), dict(yx=None), dict(next=None),
               dict(count=None), dict(ws=None), dict(inlier=None), dict(transform=None), dict(inlier_count=None),
               dict(matched=None), dict(thr=float("nan")), dict(thr=float("inf")), dict(thr=0.0), dict(thr=-1.0),
               dict(ws=ctypes.c_void_p(264)), dict(capacity=0, thr=0.0), dict(batch=1, thr=float("nan"))):
        assert call(**kw) == _lib_status("INVAL"), kw
        assert b"silent_estimate_motion" in L.silent_last_error()
    for kw in (dict(hyp=0), dict(hyp=-1), dict(hyp=4097), dict(hyp=2 ** 31 - 1)):
        assert call(**kw) == _lib_status("SHAPE"), kw
    assert call(ws_bytes=8 * 24 - 1) == _lib_status("CAPACITY")
    # capacity 0 or batch 1 launches nothing; capacity 0 needs no buffers, batch 1 no pair outputs
    assert call(capacity=0, offsets=None, yx=None, next=None, count=None, ws=None, ws_bytes=0, transform=None,
                inlier_count=None, matched=None, inlier=None) == 0
    assert call(batch=1, transform=None, inlier_count=None, matched=None) == 0
    assert call(hyp=1, seed=2 ** 64 - 1, batch=1) == 0
    if L.silent_device_count() <= 0:
        assert call() == _lib_status("CUDA")
        assert call(hyp=4096, thr=1e-30, batch=2) == _lib_status("CUDA")


BAD_THRESHOLDS = (0, 0.0, -1.0, float("nan"), float("inf"), 1e-60, 1e39, True, "2", None)
BAD_HYPOTHESES = (0, -1, 4097, 2.0, True, "256", None, np.float32(8))
BAD_SEEDS = (-1, 2 ** 64, 1.5, True, "0", None)


def test_python_validation_raises_before_the_gpu():
    import torch
    from pysilent_b200 import LineEndPipeline, _ops
    assert _ops.motion_args(2, 256, 0) == (2.0, 256, 0)
    assert _ops.motion_args(np.float32(0.5), np.int64(4096), 2 ** 64 - 1) == (0.5, 4096, 2 ** 64 - 1)
    frames = torch.zeros((2, 48, 64, 3), dtype=torch.uint8)
    pipe = LineEndPipeline(output_size=(34, 18), zoom_ratio=SQRT2)
    for field, bads in (("threshold", BAD_THRESHOLDS), ("hypotheses", BAD_HYPOTHESES), ("seed", BAD_SEEDS)):
        for bad in bads:
            kw = {field: bad}
            with pytest.raises(ValueError, match=field):
                _ops.motion_args(**dict(dict(threshold=2.0, hypotheses=256, seed=0), **kw))
            with pytest.raises(ValueError, match=field):
                pipe.run_frames_motion(frames, 2, 8, **kw)
            with pytest.raises(ValueError, match=field):
                pipe.run_host_motion(frames.numpy(), 2, 8, **kw)
    with pytest.raises(ValueError, match="search radius"):
        pipe.run_frames_motion(frames, 2, -1)
    with pytest.raises(ValueError, match="max_ratio"):
        pipe.run_host_motion(frames.numpy(), 2, 8, max_ratio=0)
    with pytest.raises(ValueError, match="patch radius"):
        pipe.run_frames_motion(frames, 32, 8)

    cap = 6
    offs, yx, nxt, cnt = (torch.tensor([0, 3, 6]), torch.zeros((cap, 2)), torch.zeros(cap, dtype=torch.int64),
                          torch.zeros(1, dtype=torch.int64))
    for kw in (dict(frame_offsets=offs.int()), dict(frame_offsets=torch.zeros(1, dtype=torch.int64)),
               dict(frame_offsets=offs[None]), dict(frame_yx=yx.double()), dict(frame_yx=torch.zeros((cap, 3))),
               dict(next=nxt.int()), dict(next=torch.zeros(cap + 1, dtype=torch.int64)), dict(count=cnt.float()),
               dict(count=torch.zeros(0, dtype=torch.int64)), dict(frame_yx=None), dict(hypotheses=0),
               dict(threshold=float("nan")), dict(seed=-1), dict(transform=torch.zeros((1, 2, 3))),
               dict(transform=torch.zeros((2, 2, 3), dtype=torch.float64)),
               dict(inlier_count=torch.zeros(1, dtype=torch.int32)), dict(matched=torch.zeros(2, dtype=torch.int64)),
               dict(inlier=torch.zeros(cap, dtype=torch.bool)), dict(workspace=torch.zeros(cap * 24 - 1, dtype=torch.uint8)),
               dict(workspace=torch.zeros(cap * 24, dtype=torch.int8)), {}):   # {}: CPU tensors
        a = dict(frame_offsets=offs, frame_yx=yx, next=nxt, count=cnt, hypotheses=8, threshold=2.0)
        a.update(kw)
        with pytest.raises(ValueError):
            _ops.estimate_motion(**a)


# ---- GPU -----------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cuda(built_lib):
    torch = pytest.importorskip("torch")
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _run_op(torch, offs, yx, nxt, count, H, thr, seed, sentinel=True):
    from pysilent_b200 import _ops
    cap, pairs = len(nxt), len(offs) - 2
    dev = dict(device="cuda")
    outs = dict(transform=torch.full((pairs, 2, 3), -777.25, dtype=torch.float64, **dev),
                inlier_count=torch.full((pairs,), SENTINEL, dtype=torch.int64, **dev),
                matched=torch.full((pairs,), SENTINEL, dtype=torch.int64, **dev),
                inlier=torch.full((cap,), 0xA5, dtype=torch.uint8, **dev)) if sentinel else {}
    got = _ops.estimate_motion(torch.from_numpy(np.asarray(offs, np.int64)).cuda(),
                               torch.from_numpy(np.ascontiguousarray(yx, np.float32)).cuda(),
                               torch.from_numpy(np.asarray(nxt, np.int64)).cuda(),
                               torch.full((1,), int(count), dtype=torch.int64, **dev), H, thr, seed, **outs)
    if sentinel:
        assert all(g is o for g, o in zip(got, outs.values()))
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL_CASES)
def test_op_small_cases_equal_the_reference(name, cuda):
    args = _case(name)
    _assert_motion(_run_op(cuda, *args), motion_reference(*args)[0], name)


# frames of very different sizes in one call: pairs of thousands of correspondences, hundreds, a handful, none
MIXED = [3000, 2800, 5, 4, 0, 400, 380, 3, 3, 2500, 2400, 2, 1]


@pytest.mark.gpu
@pytest.mark.parametrize("hypotheses", [1, 7, 128, 129, 1000, 4096])
@pytest.mark.parametrize("seed", [0, 12345, 2 ** 64 - 1])
def test_op_equals_the_reference(hypotheses, seed, cuda):
    offs, yx, nxt, k = motion_rows(hypotheses + seed % 1000, MIXED, outliers=0.3, nan=0.01, junk=31)
    for count, thr in ((k, 2.0), (k - 700, 4.5)):
        want, _ = motion_reference(offs, yx, nxt, count, hypotheses, thr, seed)
        if count == k and hypotheses >= 128:
            assert (want[1] > 0).sum() >= 3, "few fitted pairs: the case tests little"
        got = _run_op(cuda, offs, yx, nxt, count, hypotheses, thr, seed)
        _assert_motion(got, want, "H=%d seed=%d count=%d" % (hypotheses, seed, count))
        again = _run_op(cuda, offs, yx, nxt, count, hypotheses, thr, seed, sentinel=False)
        _assert_motion(again, tuple(_np(t) for t in got), "second call")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(PIPELINE_CASES))
def test_pipeline_motion_equals_the_reference(name, cuda):
    torch = cuda
    case, r, R, ratio, extra = PIPELINE_CASES[name]
    make, size, zoom, kw, _ = CASES[case]
    pipe = _pipe(torch, size, zoom, dict(kw, **extra))
    frames = torch.from_numpy(make()).cuda()
    rec, m, mo = pipe.run_frames_motion(frames, r, R, ratio, threshold=3.0, hypotheses=300, seed=9)
    want_rec, want_m = pipe.run_frames_matches(frames, r, R, ratio)
    _check_records(rec, want_rec, name)
    _assert_matches(m, tuple(_np(t) for t in want_m), name)
    assert mo.transform.is_cuda and mo.transform.dtype == torch.float64 and mo.inlier.dtype == torch.uint8
    B = len(_np(rec.frame_offsets)) - 1
    assert tuple(mo.transform.shape) == (B - 1, 2, 3) and tuple(mo.inlier.shape) == (len(rec.points),)
    want, _ = motion_reference(_np(rec.frame_offsets), _np(rec.frame_yx), _np(m.next), len(rec.points), 300, 3.0, 9)
    _assert_motion(mo, want, name)


def _pan_truth(pan):
    """Frame f + 1 shows frame f's content shifted by -pan: [y1, x1] = [y0, x0] - pan."""
    return np.array([[1.0, 0.0, -pan[0]], [0.0, 1.0, -pan[1]]])


# measured on the panned scene of test_point_matches (peaks 0.5, r = 2, R = 8, max_ratio 0.64, 4 frames of 240 x 320,
# output 96 x 64 at zoom 1.5, threshold 2, 256 hypotheses; NVIDIA B200 at a 1000 W power limit): 184-192 matches per
# pair, max |A - I| 0.0048, max |t + pan| 0.21 px, smallest inlier share 0.947. The bounds leave a margin for the seed
PAN_MAX_LINEAR = 0.015    # |T[:, :2] - I|
PAN_MAX_SHIFT = 0.75      # |T[:, 2] + pan|, frame pixels
PAN_MIN_INLIERS = 0.85    # inlier_count / matched


@pytest.mark.gpu
def test_panned_scene_motion_is_the_pan(cuda):
    torch = cuda
    frames = panned_frames(90, 4, 240, 320, PAN)
    pipe = _pipe(torch, (96, 64), 1.5, dict(peaks=0.5))
    rec, m, mo = pipe.run_frames_motion(torch.from_numpy(frames).cuda(), 2, 8, 0.64)
    T, n, M = _np(mo.transform), _np(mo.inlier_count), _np(mo.matched)
    truth = _pan_truth(PAN)
    lin = np.abs(T[:, :, :2] - truth[:, :2]).max()
    shift = np.abs(T[:, :, 2] - truth[:, 2]).max()
    share = (n / M).min()
    print("panned scene: matched %s inliers %s max |A - I| %.5f max |t + pan| %.4f min share %.4f"
          % (list(M), list(n), lin, shift, share))
    assert lin <= PAN_MAX_LINEAR and shift <= PAN_MAX_SHIFT and share >= PAN_MIN_INLIERS, (lin, shift, share)
    assert np.array_equal(_np(mo.inlier).astype(bool).sum(), n.sum())


def warped_frames(seed, batch, h, w, angle_deg, scale, shift):
    """``batch`` frames of one seeded texture, frame f + 1 = frame f moved by the affine map A (rotation by
    ``angle_deg`` about the frame centre, ``scale``, then ``shift``) in (y, x) frame pixels: returns the frames and
    A as a [2, 3] (y, x) map from frame f to frame f + 1."""
    from scipy.ndimage import affine_transform, gaussian_filter
    H, W = h + 160, w + 160
    tex = np.random.RandomState(seed).rand(H, W, 3)
    tex = gaussian_filter(tex, (1.5, 1.5, 0))
    tex = (tex - tex.mean()) / tex.std() * 60 + 128
    a = np.deg2rad(angle_deg)
    lin = scale * np.array([[np.cos(a), -np.sin(a)], [np.sin(a), np.cos(a)]])
    ctr = np.array([(h - 1) / 2.0, (w - 1) / 2.0])
    A = np.concatenate([lin, (ctr - lin @ ctr + np.asarray(shift, float))[:, None]], axis=1)
    out = []
    # frame f: output pixel p shows texture point M_f^-1 p + 80, with M_f = A^f
    Mf = np.eye(3)
    A3 = np.vstack([A, [0, 0, 1]])
    for _ in range(batch):
        inv = np.linalg.inv(Mf)
        chans = [affine_transform(tex[..., c], inv[:2, :2], offset=inv[:2, 2] + 80, output_shape=(h, w), order=1)
                 for c in range(3)]
        out.append(np.clip(np.stack(chans, axis=-1), 0, 255).astype(np.uint8))
        Mf = A3 @ Mf
    return np.stack(out), A


WARP = dict(angle_deg=1.5, scale=1.02, shift=(2.0, -3.0))
# measured (peaks 0.5, r = 2, R = 8, max_ratio 0.64, 4 frames of 240 x 320, output 96 x 64 at zoom 1.5, threshold 2,
# 256 hypotheses; NVIDIA B200 at a 1000 W power limit): 184-216 matches per pair, max |dA| 0.0033, max |dt| 0.66 px,
# smallest inlier share 0.959. The bounds leave a margin for the seed
WARP_MAX_LINEAR = 0.015
WARP_MAX_SHIFT = 2.0
WARP_MIN_INLIERS = 0.85


@pytest.mark.gpu
def test_warped_scene_motion_is_the_warp(cuda):
    torch = cuda
    frames, A = warped_frames(91, 4, 240, 320, **WARP)
    pipe = _pipe(torch, (96, 64), 1.5, dict(peaks=0.5))
    rec, m, mo = pipe.run_frames_motion(torch.from_numpy(frames).cuda(), 2, 8, 0.64)
    T, n, M = _np(mo.transform), _np(mo.inlier_count), _np(mo.matched)
    lin = np.abs(T[:, :, :2] - A[:, :2]).max()
    shift = np.abs(T[:, :, 2] - A[:, 2]).max()
    share = (n / M).min()
    print("warped scene: matched %s inliers %s max |dA| %.5f max |dt| %.4f min share %.4f"
          % (list(M), list(n), lin, shift, share))
    assert lin <= WARP_MAX_LINEAR and shift <= WARP_MAX_SHIFT and share >= WARP_MIN_INLIERS, (lin, shift, share)


@pytest.mark.gpu
def test_estimate_motion_with_outputs_takes_no_host_synchronisation(cuda):
    torch = cuda
    from pysilent_b200 import _ops
    offs, yx, nxt, k = motion_rows(8, MIXED)
    dev = dict(device="cuda")
    ins = (torch.from_numpy(offs).cuda(), torch.from_numpy(yx).cuda(), torch.from_numpy(nxt).cuda(),
           torch.full((1,), k, dtype=torch.int64, **dev))
    pairs = len(offs) - 2
    outs = dict(transform=torch.empty((pairs, 2, 3), dtype=torch.float64, **dev),
                inlier_count=torch.empty(pairs, dtype=torch.int64, **dev),
                matched=torch.empty(pairs, dtype=torch.int64, **dev),
                inlier=torch.empty(len(nxt), dtype=torch.uint8, **dev),
                workspace=torch.empty(_ops.motion_workspace_bytes(len(nxt)), dtype=torch.uint8, **dev))
    _ops.estimate_motion(*ins, 500, 2.0, 4, **outs)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        got = _ops.estimate_motion(*ins, 500, 2.0, 4, **outs)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    _assert_motion(got, motion_reference(offs, yx, nxt, k, 500, 2.0, 4)[0], "no sync")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["bgr", "nv12_peaks", "bank8_f16"])
def test_host_motion_equals_device_motion(fmt, cuda):
    torch = cuda
    from test_point_records import _bgr, random_nv12
    if fmt == "nv12_peaks":
        frames, kw = random_nv12(63, 240, 320, 3), dict(frame_format="nv12", peaks=0.5)
    elif fmt == "bank8_f16":
        frames, kw = _bgr([("noise", 64, i) for i in range(3)], 96, 128), dict(orientations=8, out_dtype="f16")
    else:
        frames, kw = panned_frames(65, 3, 240, 320, PAN), dict(peaks=0.3)
    size = (48, 32) if fmt == "bank8_f16" else (96, 64)
    pipe = _pipe(torch, size, 1.5, kw)
    r, R, ratio = 3, 8, 0.8
    drec, dm, dmo = pipe.run_frames_motion(torch.from_numpy(frames).cuda(), r, R, ratio, seed=3)
    hrec, hm, hmo = pipe.run_host_motion(frames, r, R, ratio, seed=3, points_capacity=8)   # also redoes the call
    hrec2, hm2 = pipe.run_host_matches(frames, r, R, ratio)
    for tup in (hrec, hm, hmo):
        for field in tup._fields:
            assert isinstance(getattr(tup, field), np.ndarray), field
    _assert_motion(hmo, tuple(_np(t) for t in dmo), fmt)
    _assert_matches(hm, tuple(_np(t) for t in dm), fmt)
    assert np.array_equal(hrec.points, _np(drec.points)) and np.array_equal(hrec.points, hrec2.points)
    for field in ("frame_yx", "gray", "orient", "line_end"):
        assert np.array_equal(getattr(hrec, field).view(np.uint32), getattr(hrec2, field).view(np.uint32)), field


@pytest.mark.gpu
def test_one_frame_and_no_points(cuda):
    """B = 1 gives empty pair outputs and no flag; capacity 0 gives NaN models and zero counts."""
    torch = cuda
    o, yx, n, k = motion_rows(3, [25])
    got = _run_op(torch, o, yx, n, k, 10, 2.0, 0)
    assert tuple(got[0].shape) == (0, 2, 3) and not _np(got[3]).any()
    got = _run_op(torch, np.zeros(4, np.int64), np.zeros((0, 2), np.float32), np.zeros(0, np.int64), 0, 10, 2.0, 0)
    assert np.isnan(_np(got[0])).all() and not _np(got[1]).any() and not _np(got[2]).any()
