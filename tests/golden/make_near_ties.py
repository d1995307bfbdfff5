"""Generate tests/golden/near_ties.npz and tests/golden/near_ties_any_ratio.npz: adversarial 2a-byte windows whose
reference sums land on or near an integer.

Run once from the repository root: `python tests/golden/make_near_ties.py` (a few minutes on 8 cores).  A re-run
writes both files again byte for byte.

The product's outputs must equal the reference's double-precision software path bit for bit
(full_TB.h:55-77: x = xx/SCALE, sum += in[i] * lanczos_kernel(x - i) in ascending taps, clamp, truncate).
On noise or image-like content a sum almost never falls close enough to an integer for the details of the
exact path to matter -- which weights it uses, the summation order, whether the multiply-add is fused, and
whether the fp32 guard really bounds the fast path's error.  This script finds windows where they do.

For every (N/D, a) that a kernel instance serves and a few output coordinates per phase (near the origin and
near 1024, 12288 and 27648 -- multiples of 256 output bytes for 1, 3 and 4 channels, so next to strip edges), it
stores the window bytes in three classes:
  * tie (0): the reference's sum is within 4e-12 of an integer 1..255 and its truncation changes under at least one
    wrong evaluation -- the phase-table weights instead of this coordinate's own, a fused multiply-add, or the
    reversed tap order -- or it is exactly integral;
  * wrong side (1): 1e-9 <= distance <= 3e-5, and an fp32 chain with the kernels' fp32 phase-table weights (fused
    multiply-adds from 0; outermost taps first as in the lanczos_v6 H pass, or ascending as everywhere else)
    truncates differently from the reference: only the guard can rescue these samples;
  * near (2): distance <= 1e-6: the exact path must always be taken.
Weights come from the oracle's oracle_kernel (glibc sin, as in the reference).  Ties are found by a
meet-in-the-middle search over every window for a <= 3 (a = 4: 2^48 of its 2^64 windows); the other two classes
by random windows.  The oracle stays the truth: this file only decides what the tests cover.

near_ties_any_ratio.npz holds windows for the generic kernel (lanczos_generic.cu), which serves every ratio and
(channels, a) without a kernel instance.  Its arithmetic differs from the instances': s = fmaf(b_k, (float)w_k, s) from
0 in ascending taps, each output coordinate with its own weights.  For every ratio N/D <= 16 the library accepts and
a = 1..4 (GENERIC_CONFIGS), at one coordinate near the origin and one near 1024, both on edges of the generic kernel's
64 x 32 output tiles, it stores
  * wrong side (1): 1e-9 <= distance <= 3e-5 and that chain truncates differently from the reference (flag
    F_WRONG_GENERIC; F_OFF_INTEGER when the fp32 result is not the integer itself, so that only a guard wider than
    half an ulp re-evaluates the sample);
  * near (2): distance <= 1e-6.
Classes that no window falls into are empty.  For 2/1 the weights of the one interpolated phase are symmetric, so
a sum is a combination of the pair sums b_k + b_{2a-1-k}: with a = 1 or 2 no window comes within 3e-5 of an integer
1..255 at all, and with a = 3 or 4 no tie discriminates.  The search found no discriminating tie either for 3/2 and 3/1
with a = 2 or for 4/1 with a = 3; those ratios keep their wrong-side and near windows.
"""
import math
import multiprocessing
import os
import sys
from fractions import Fraction

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle_py as O  # noqa: E402

OUT = os.path.join(HERE, "near_ties.npz")
OUT_ANY = os.path.join(HERE, "near_ties_any_ratio.npz")

# every (N, D, a) that a specialised kernel instance serves
CONFIGS = [(2, 1, 1), (2, 1, 2), (2, 1, 3), (2, 1, 4), (3, 2, 2), (3, 2, 3), (17, 10, 3), (3, 1, 2), (3, 1, 3),
           (4, 1, 3), (5, 3, 3), (7, 4, 3)]
MAGNITUDES = [36, 1024, 12288, 27648]
TIE, WRONG, NEAR = 0, 1, 2
# flag bits
F_PHASE, F_FMA, F_REV, F_INTEGRAL, F_WRONG_OUTER, F_WRONG_ASC = 1, 2, 4, 8, 16, 32
F_WRONG_GENERIC, F_OFF_INTEGER = 64, 128
TIE_TOL, WRONG_LO, WRONG_HI, NEAR_TOL = 4e-12, 1e-9, 3e-5, 1e-6
CAP_TIE_EACH, CAP_INTEGRAL, CAP_WRONG, CAP_NEAR = 4, 2, 4, 3


# ---- the reference's arithmetic --------------------------------------------------------------------

def weights(xx, n, d, a):
    """Weights of output coordinate xx, full_TB.h:57-60: x = (double)xx / ((double)N/D), w_k = L(x - (first + k))."""
    x = xx / (n / d)
    first = (xx * d) // n - a + 1
    L = O.lib().oracle_kernel
    return np.array([L(x - (first + k), a) for k in range(2 * a)], dtype=np.float64), first


def phase(xx, n, d):
    return (xx * d) % n


def phase_weights(ph, n, d, a):
    """The polyphase table row of phase ph: the weights of the first coordinate with that phase (plan.cpp build_plan)."""
    for xx in range(n):
        if phase(xx, n, d) == ph:
            return weights(xx, n, d, a)[0]
    raise ValueError(ph)


def quantise(s):
    """double_to_uint8 (full_TB.h:29-37): clamp, then truncate toward zero; works on numpy arrays and Fractions."""
    if isinstance(s, np.ndarray):
        return np.clip(np.trunc(np.clip(s, 0.0, 255.0)), 0, 255).astype(np.int64)
    if s > 255:
        return 255
    if s < 0:
        return 0
    return int(s)


def seq_sum(win, w, order=None):
    """Sequential double sum of (double)b_k * w_k, one rounding per multiply and per add (numpy, vectorised over rows)."""
    win = np.atleast_2d(win).astype(np.float64)
    s = np.zeros(win.shape[0])
    for k in (range(len(w)) if order is None else order):
        s = s + win[:, k] * w[k]
    return s


def fma_sum(win, w):
    """The same sum with every multiply-add fused (one rounding per tap), exactly."""
    s = 0.0
    for b, wk in zip(win, w):
        s = float(Fraction(int(b)) * Fraction(float(wk)) + Fraction(s))
    return s


def round_f32(q):
    """Round a Fraction to the nearest binary32 value (ties to even); normal range only."""
    if q == 0:
        return Fraction(0)
    sign = -1 if q < 0 else 1
    m = abs(q)
    e = m.numerator.bit_length() - m.denominator.bit_length()
    if Fraction(2) ** e > m:
        e -= 1
    while Fraction(2) ** (e + 1) <= m:
        e += 1
    scale = Fraction(2) ** (e - 23)
    t = m / scale                       # in [2^23, 2^24)
    fl = t.numerator // t.denominator
    rem = t - fl
    if rem > Fraction(1, 2) or (rem == Fraction(1, 2) and fl % 2 == 1):
        fl += 1
    return sign * fl * scale


def tap_order_outer(taps):
    """lanczos_v6.cu tap_order6: outermost (smallest) weights first, the two central taps last."""
    return [(i // 2) if i % 2 == 0 else taps - 1 - i // 2 for i in range(taps)]


def f32_chain(win, w32, order):
    """An fp32 chain of fused multiply-adds from 0 with fp32 weights, exactly (the kernels' fast path, shifted by guard)."""
    acc = Fraction(0)
    for k in order:
        acc = round_f32(Fraction(int(win[k])) * Fraction(float(w32[k])) + acc)
    return acc


def classify(win, xx, n, d, a):
    """Everything recorded about one window at output coordinate xx: (class or -1, flags, nearest integer, distance)."""
    taps = 2 * a
    w, _ = weights(xx, n, d, a)
    wp = phase_weights(phase(xx, n, d), n, d, a)
    win = np.asarray(win[:taps], dtype=np.int64)
    s = float(seq_sum(win, w)[0])
    k = int(np.rint(s))
    dist = abs(s - k)
    q = quantise(s)
    flags = 0
    if k < 1 or k > 255:
        return -1, 0, k, dist
    if dist <= TIE_TOL:              # the exact path's details only matter this close
        if quantise(seq_sum(win, wp)[0]) != q:
            flags |= F_PHASE
        if quantise(fma_sum(win, w)) != q:
            flags |= F_FMA
        if quantise(seq_sum(win, w, order=list(range(taps))[::-1])[0]) != q:
            flags |= F_REV
        if s == k:
            flags |= F_INTEGRAL
    if dist >= WRONG_LO:             # fp32 chains cannot resolve anything closer: the guard always flags it
        w32 = wp.astype(np.float32)
        if quantise(f32_chain(win, w32, tap_order_outer(taps))) != q:
            flags |= F_WRONG_OUTER
        if quantise(f32_chain(win, w32, list(range(taps)))) != q:
            flags |= F_WRONG_ASC
    if dist <= TIE_TOL and flags & (F_PHASE | F_FMA | F_REV | F_INTEGRAL):
        cls = TIE
    elif WRONG_LO <= dist <= WRONG_HI and flags & (F_WRONG_OUTER | F_WRONG_ASC):
        cls = WRONG
    elif dist <= NEAR_TOL:
        cls = NEAR
    else:
        cls = -1
    return cls, flags, k, dist


# ---- search ----------------------------------------------------------------------------------------

def coordinates(n, d, a):
    """A few output coordinates per interpolated phase and magnitude (phase 0 is the copy path, pinned elsewhere)."""
    phases = [p for p in range(1, n)]
    out = []
    for mi, t in enumerate(MAGNITUDES):
        sel = phases if len(phases) <= 4 else [phases[(mi * 5 + j * (len(phases) // 3)) % len(phases)] for j in range(3)]
        for ph in sel:
            xs = [xx for xx in range(t - 2 * n, t + 2 * n) if phase(xx, n, d) == ph]
            out.append(min(xs, key=lambda xx: (abs(xx - t), xx)))
    return out


def float_floor_ok(xx, n, d):
    """The reference's tap origin floor((double)xx / ((double)N/D)) equals the exact floor(xx*D/N) (plan.cpp)."""
    return math.floor(xx / (n / d)) == xx * d // n


def first_float_floor_miss(n, d, limit=1 << 12):
    """The first output coordinate below `limit` at which the library rejects N/D (LANCZOS_ERR_RATIO_FLOAT), or None."""
    return next((xx for xx in range(limit) if not float_floor_ok(xx, n, d)), None)


# every reduced N/D with D < N <= 16 that the library accepts up to 4096 output samples, with a = 1..4
GENERIC_CONFIGS = [(n, d, a) for n in range(2, 17) for d in range(1, n) if math.gcd(n, d) == 1
                   and first_float_floor_miss(n, d) is None for a in range(1, 5)]
GENERIC_BASES = [64, 1024]


def generic_coordinates(n, d):
    """Per base, the first interpolated coordinate among base - 1, base, base + 63, base + 64, ...: the last or first
    column of a 64-pixel tile and the last or first row of a 32-row tile of the generic kernel."""
    return [next(xx for j in range(n) for xx in (b + 64 * j - 1, b + 64 * j) if phase(xx, n, d) != 0)
            for b in GENERIC_BASES]


def generic_chain(win, w):
    """lanczos_generic.cu: s = fmaf((float)b_k, (float)w_k, s) from 0, ascending taps, this coordinate's own weights."""
    return f32_chain(win, np.asarray(w).astype(np.float32), list(range(len(w))))


def classify_generic(win, xx, n, d, a):
    """(class or -1, flags, nearest integer, distance) of one window for the generic kernel's arithmetic."""
    taps = 2 * a
    w, _ = weights(xx, n, d, a)
    win = np.asarray(win[:taps], dtype=np.int64)
    s = float(seq_sum(win, w)[0])
    k = int(np.rint(s))
    dist = abs(s - k)
    if k < 1 or k > 255:
        return -1, 0, k, dist
    flags = 0
    if dist >= WRONG_LO:
        g = generic_chain(win, w)
        if quantise(g) != quantise(s):
            flags |= F_WRONG_GENERIC | (F_OFF_INTEGER if g != k else 0)
    if WRONG_LO <= dist <= WRONG_HI and flags & F_WRONG_GENERIC:
        cls = WRONG
    elif dist <= NEAR_TOL:
        cls = NEAR
    else:
        cls = -1
    return cls, flags, k, dist


def half_sums(w, rng, limit):
    """All byte combinations of the taps with weights w (or `limit` random ones): (sums, bytes)."""
    h = len(w)
    if 256 ** h <= limit:
        grids = np.meshgrid(*[np.arange(256, dtype=np.float64)] * h, indexing="ij")
        byt = np.stack([g.reshape(-1) for g in grids], axis=1).astype(np.uint8)
    else:
        byt = rng.integers(0, 256, size=(limit, h), dtype=np.uint8)
    s = np.zeros(byt.shape[0])
    for k in range(h):
        s = s + byt[:, k].astype(np.float64) * w[k]
    return s, byt


def tie_candidates(w, rng):
    """Windows whose sum is within TIE_TOL (+ rounding) of an integer: meet in the middle over the two halves."""
    taps = len(w)
    if taps == 2:                                              # a = 1: every window
        g = np.stack(np.meshgrid(np.arange(256), np.arange(256), indexing="ij"), -1).reshape(-1, 2)
        s = seq_sum(g, w)
        return g[(np.abs(s - np.rint(s)) <= 2 * TIE_TOL) & (np.rint(s) >= 1) & (np.rint(s) <= 255)].astype(np.uint8)
    h = taps // 2
    A, abyt = half_sums(w[:h], rng, 1 << 24)
    B, bbyt = half_sums(w[h:], rng, 1 << 24)
    fb = B - np.floor(B)
    order = np.argsort(fb, kind="stable")
    fbs = fb[order]
    t = -A - np.floor(-A)
    idx = np.searchsorted(fbs, t)
    found = []
    for off in (-1, 0, 1):
        j = (idx + off) % len(fbs)
        diff = fbs[j] - t
        diff -= np.rint(diff)
        m = np.abs(diff) <= 2 * TIE_TOL
        ia = np.nonzero(m)[0]
        found.append(np.concatenate([abyt[ia], bbyt[order[j[ia]]]], axis=1))
    wins = np.unique(np.concatenate(found), axis=0)
    s = seq_sum(wins, w)
    return wins[(np.rint(s) >= 1) & (np.rint(s) <= 255)]       # sums near 0 or 256 are clamped either way


def random_candidates(w, rng, count=1 << 22):
    """Random windows whose reference sum is within WRONG_HI of an integer."""
    wins = rng.integers(0, 256, size=(count, len(w)), dtype=np.uint8)
    s = seq_sum(wins, w)
    dist = np.abs(s - np.rint(s))
    m = (dist <= WRONG_HI) & (np.rint(s) >= 1) & (np.rint(s) <= 255)
    wins, dist = wins[m], dist[m]
    return wins[np.argsort(dist, kind="stable")]


def one_coordinate(job):
    n, d, a, xx = job
    rng = np.random.default_rng(1000003 * n + 1009 * d + 101 * a + xx)
    w, _ = weights(xx, n, d, a)
    rows = []
    # ties: the discriminating ones first (fused, reversed, phase-table), then exactly integral ones
    ties = []
    for win in tie_candidates(w, rng):
        cls, flags, k, dist = classify(win, xx, n, d, a)
        if cls == TIE:
            ties.append((win, flags, k, dist))
    kept = set()
    for bit, cap in ((F_FMA, CAP_TIE_EACH), (F_REV, CAP_TIE_EACH), (F_PHASE, CAP_TIE_EACH), (F_INTEGRAL, CAP_INTEGRAL)):
        n_bit = 0
        for i, (win, flags, k, dist) in enumerate(ties):
            if n_bit >= cap:
                break
            if flags & bit:
                n_bit += 1
                if i not in kept:
                    kept.add(i)
                    rows.append((TIE, win, flags, k, dist))
    n_wrong = n_near = 0
    for win in random_candidates(w, rng):
        if n_wrong >= CAP_WRONG and n_near >= CAP_NEAR:
            break
        cls, flags, k, dist = classify(win, xx, n, d, a)
        if cls == WRONG and n_wrong < CAP_WRONG:
            n_wrong += 1
            rows.append((WRONG, win, flags, k, dist))
        elif cls == NEAR and n_near < CAP_NEAR:
            n_near += 1
            rows.append((NEAR, win, flags, k, dist))
    return (n, d, a, xx, len(ties), rows)


def one_generic_coordinate(job):
    n, d, a, xx = job
    rng = np.random.default_rng(1000003 * n + 1009 * d + 101 * a + xx + 7)
    w, _ = weights(xx, n, d, a)
    rows = []
    n_wrong = n_near = 0
    for win in random_candidates(w, rng):
        if n_wrong >= CAP_WRONG and n_near >= CAP_NEAR:
            break
        cls, flags, k, dist = classify_generic(win, xx, n, d, a)
        if cls == WRONG and n_wrong < CAP_WRONG:
            n_wrong += 1
            rows.append((WRONG, win, flags, k, dist))
        elif cls == NEAR and n_near < CAP_NEAR:
            n_near += 1
            rows.append((NEAR, win, flags, k, dist))
    return (n, d, a, xx, 0, rows)


def save(path, results):
    cols = {k: [] for k in ("n", "d", "a", "coord", "cls", "flags", "k", "dist", "win")}
    for (n, d, a, xx, n_ties, rows) in results:
        print(f"{n}/{d} a={a} x={xx}: {n_ties} ties found, kept " +
              ", ".join(f"{name} {sum(r[0] == c for r in rows)}" for c, name in ((TIE, "tie"), (WRONG, "wrong"), (NEAR, "near"))))
        for (cls, win, flags, k, dist) in rows:
            padded = np.zeros(8, np.uint8)
            padded[:2 * a] = win[:2 * a]
            for key, v in (("n", n), ("d", d), ("a", a), ("coord", xx), ("cls", cls), ("flags", flags), ("k", k),
                           ("dist", dist), ("win", padded)):
                cols[key].append(v)
    np.savez_compressed(path, **{k: np.array(v, dtype=np.float64 if k == "dist" else (np.uint8 if k == "win" else np.int32))
                                 for k, v in cols.items()})
    print("wrote", path, os.path.getsize(path), "bytes,", len(cols["n"]), "windows")


def main():
    jobs = [(n, d, a, xx) for (n, d, a) in CONFIGS for xx in coordinates(n, d, a)]
    any_jobs = [(n, d, a, xx) for (n, d, a) in GENERIC_CONFIGS for xx in generic_coordinates(n, d)]
    with multiprocessing.Pool(min(8, os.cpu_count() or 1)) as pool:
        save(OUT, pool.map(one_coordinate, jobs, chunksize=1))
        save(OUT_ANY, pool.map(one_generic_coordinate, any_jobs, chunksize=1))


if __name__ == "__main__":
    main()
