"""Shared content for the tests: synthetic images, the golden fixture list, the near-tie windows and their image
builders, and the table of the library's specialised kernel instances."""
import collections
import glob
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import make_near_ties as NT  # noqa: E402


def golden_files():
    return sorted(glob.glob(os.path.join(HERE, "golden", "ref_*.npz")))


def noise_hwc(oracle, h, w, c, seed=0):
    """Uniform xorshift noise, interleaved [H][W][C] (SURVEY.md 8d (i))."""
    return oracle.xorshift_bytes(h * w * c, oracle.SEED + seed).reshape(h, w, c)


def smooth_hwc(oracle, h, w, c, seed=0):
    """Smooth + noise (SURVEY.md 8d (ii)): 128 + 90 sin(0.05x+c) cos(0.037y) + U[-8,7]."""
    yy, xx = np.mgrid[0:h, 0:w]
    noise = (oracle.xorshift_bytes(h * w * c, oracle.SEED + 77 + seed).reshape(h, w, c).astype(np.int32) & 15) - 8
    img = np.stack([128 + 90 * np.sin(0.05 * xx + ch) * np.cos(0.037 * yy) for ch in range(c)], axis=-1)
    return np.clip(img + noise, 0, 255).astype(np.uint8)


def dark_hwc(oracle, h, w, c, seed=0):
    """Dark noise 0..15: the regime where the reference's sin(k*pi) residues flip phase-0 samples."""
    return (noise_hwc(oracle, h, w, c, seed) & 15).astype(np.uint8)


def patchwork_hwc(oracle, h, w, c, seed, band, col):
    """Image-like, uniform-noise and dark-noise patches side by side: `band` rows x `col` pixels each, in turn."""
    kinds = [smooth_hwc(oracle, h, w, c, seed), noise_hwc(oracle, h, w, c, seed + 1), dark_hwc(oracle, h, w, c, seed + 2)]
    yy, xx = np.mgrid[0:h, 0:w]
    sel = ((yy // band) + (xx // col)) % 3
    img = np.zeros((h, w, c), dtype=np.uint8)
    for k in range(3):
        img[sel == k] = kinds[k][sel == k]
    return img


PATCH_H = 120                 # input rows of a patchwork (a multiple of every D served)


def patch_width(c, n, d):
    """Input width of a patchwork: whole 32-bit input words, output rows a multiple of 8 bytes but not of a 256-byte
    strip (a partial last strip), at least three strips."""
    w = d
    while True:
        ob = w * n // d * c
        if w % d == 0 and (w * c) % 4 == 0 and ob % 8 == 0 and ob % 256 != 0 and ob >= 700:
            return w
        w += d


def patchwork(oracle, c, n, d, seed, w=None):
    w = w or patch_width(c, n, d)
    return patchwork_hwc(oracle, PATCH_H, w, c, seed=seed, band=13, col=37)


def planar(img_hwc):
    return np.ascontiguousarray(np.transpose(img_hwc, (2, 0, 1)))


def interleaved(img_chw):
    return np.ascontiguousarray(np.transpose(img_chw, (1, 2, 0)))


def diff_stats(a, b):
    d = np.abs(a.astype(np.int16) - b.astype(np.int16))
    return {"max": int(d.max()) if d.size else 0, "exact": float((d == 0).mean()) if d.size else 1.0,
            "n_diff": int((d != 0).sum())}


# ---- the specialised kernel instances ------------------------------------------------------------------

Instance = collections.namedtuple("Instance", "family kid c a n d ph km mask", defaults=(None, None, None))

INSTANCES = (
    # LZ6_CASE list of launch_v6 (lanczos_hls_b200/csrc/lanczos_v6.cu): kernel id, C, a, N, D, PH, KM
    [Instance("v6", *i) for i in [(1, 3, 3, 2, 1, 8, 17), (2, 4, 3, 2, 1, 6, 17), (3, 4, 3, 3, 2, 4, 17),
                                  (4, 3, 2, 2, 1, 8, 0), (8, 1, 3, 2, 1, 24, 17), (9, 1, 3, 3, 2, 16, 17),
                                  (10, 1, 2, 2, 1, 24, 0)]]
    # LZD_CASE list of launch_dyn (lanczos_dyn.cu): kernel id, C, a, N, D
    + [Instance("dyn", *i) for i in [(5, 3, 3, 17, 10), (6, 3, 3, 3, 2), (7, 3, 3, 3, 1), (11, 1, 3, 17, 10),
                                     (12, 3, 2, 3, 1), (13, 1, 2, 3, 1), (14, 3, 3, 4, 1), (15, 1, 3, 3, 1),
                                     (16, 3, 3, 5, 3), (17, 3, 3, 7, 4), (18, 2, 3, 2, 1), (19, 3, 4, 2, 1),
                                     (20, 3, 1, 2, 1), (21, 4, 3, 3, 1), (22, 4, 3, 4, 1), (23, 3, 2, 3, 2),
                                     (24, 1, 3, 4, 1)]]
    # HLS_CASE list of launch_hls (lanczos_hls.cu), bit precision 8: C, a, N, MASK
    + [Instance("hls_tile", 101, c, a, n, 1, mask=m) for (c, a, n, m) in [(3, 3, 2, 4), (4, 3, 2, 4), (1, 3, 2, 4),
                                                                          (3, 2, 2, 0), (3, 3, 4, 4), (3, 2, 4, 0)]])

# kernel id -> (C, a, N, D) of the v6 and dyn instances, and back
SPECIALISED = {i.kid: (i.c, i.a, i.n, i.d) for i in INSTANCES if i.family in ("v6", "dyn")}
KERNEL_OF = {v: k for k, v in SPECIALISED.items()}


# ---- near-tie windows (tests/golden/near_ties.npz) and images that plant them --------------------------

TIE, WRONG, NEAR = NT.TIE, NT.WRONG, NT.NEAR
V_TOP = 24            # V windows start below this output row: the in-place top rows (VERBATIM) read final values
BLOCK_GAP = 3         # noise pixels between V column blocks

# 2/1 with a = 1 or 2: the one interpolated phase has symmetric weights (w_k = w_{2a-1-k}), so a sum is a combination
# of a few pair sums b_k + b_{2a-1-k} and no window comes within 3e-5 of an integer 1..255
EMPTY = {(2, 1, 1), (2, 1, 2)}


def windows():
    z = np.load(os.path.join(HERE, "golden", "near_ties.npz"))
    return {k: z[k] for k in z.files}


WIN = windows()


def config_rows(n, d, a, win=WIN):
    return np.nonzero((win["n"] == n) & (win["d"] == d) & (win["a"] == a))[0]


def tap0(xx, n, d, a):
    return (xx * d) // n - a + 1


def up_len(in_len, n, d):
    return in_len * n // d


def h_image(oracle, n, d, a, c, seed=0, odd=False, win=WIN):
    """Wide, short image with every H window of (n, d, a) planted; returns (img, [(row, channel, idx)]).
    win: the windows (default near_ties.npz)."""
    idx = config_rows(n, d, a, win)
    taps = 2 * a
    need = max([tap0(int(win["coord"][i]), n, d, a) + taps for i in idx] + [64]) + 4
    step = 16 * d
    in_w = step * ((need + step - 1) // step) + (1 if odd else 0)
    slots = []                                      # per (row, channel): occupied [lo, hi) pixel intervals
    planted = []
    for i in idx:
        lo = tap0(int(win["coord"][i]), n, d, a)
        hi = lo + taps
        for s, iv in enumerate(slots):
            if all(hi <= l or lo >= h for (l, h) in iv):
                iv.append((lo, hi))
                break
        else:
            slots.append([(lo, hi)])
            s = len(slots) - 1
        planted.append((1 + s // c, s % c, int(i)))       # row 0 stays noise
    in_h = max(2 * taps, 2 + (len(slots) + c - 1) // c)
    img = noise_hwc(oracle, in_h, in_w, c, seed=seed)
    for (r, ch, i) in planted:
        lo = tap0(int(win["coord"][i]), n, d, a)
        img[r, lo:lo + taps, ch] = win["win"][i][:taps]
    return img, planted


def q_table(xx, n, d, a):
    """q_X(v): the horizontal result at output column xx of a row that is v across all its taps (reference arithmetic)."""
    w, _ = NT.weights(xx, n, d, a)
    return NT.quantise(NT.seq_sum(np.repeat(np.arange(256)[:, None], 2 * a, axis=1), w))


def v_image(oracle, n, d, a, c, seed=0, nblk=24, base=None, place=None, win=WIN):
    """Tall, narrow image with every V window of (n, d, a) planted; returns (img, [(block, channel, X, idx)]).
    A window goes to one channel of one block; windows whose bytes no q_X of the block reaches are skipped.
    base: plant into a copy of this [H][W][C] image instead; place(idx): the output row of window idx (None: leave it
    out), by default its stored coordinate when that lies below V_TOP."""
    idx = config_rows(n, d, a, win)
    taps = 2 * a
    wblk = taps + 4
    p0s = [4 + j * (wblk + BLOCK_GAP) for j in range(nblk)]
    if base is None:
        step = 16 * d
        in_w = step * ((p0s[-1] + wblk + 4 + step - 1) // step)
        in_h = max([tap0(int(win["coord"][i]), n, d, a) + taps for i in idx] + [64]) + 4
        img = noise_hwc(oracle, in_h, in_w, c, seed=seed + 1)
    else:
        img = base.copy()
        in_w = img.shape[1]
    if place is None:
        def place(i):
            return int(win["coord"][i]) if win["coord"][i] >= V_TOP else None
    # interior output columns of every block (all taps inside the block) and their q tables
    cols = []
    for p0 in p0s:
        xs = [X for X in range(up_len(in_w, n, d)) if tap0(X, n, d, a) >= p0 and tap0(X, n, d, a) + taps <= p0 + wblk]
        cols.append([(X, q_table(X, n, d, a)) for X in xs])
    used = {}                                       # (block, channel) -> occupied [lo, hi) input rows
    planted = []
    for i in idx:
        yy = place(i)
        if yy is None:
            continue
        lo = tap0(yy, n, d, a)
        bytes_ = win["win"][i][:taps]
        done = False
        for b, p0 in enumerate(p0s):
            for ch in range(c):
                if done or not all(lo + taps <= l or lo >= h for (l, h) in used.get((b, ch), [])):
                    continue
                for X, q in cols[b]:
                    pre = [np.nonzero(q == t)[0] for t in bytes_]
                    if all(len(v) for v in pre):
                        used.setdefault((b, ch), []).append((lo, lo + taps))
                        for k, v in enumerate(pre):
                            img[lo + k, p0:p0 + wblk, ch] = v[0]
                        planted.append((b, ch, X, int(i)))
                        done = True
                        break
    return img, planted


def planted_counts(planted, win=WIN):
    out = {TIE: 0, WRONG: 0, NEAR: 0}
    for p in planted:
        out[int(win["cls"][p[-1]])] += 1
    return out


def strict_floor(planted, win=WIN):
    """Samples the exact path must have evaluated: the planted near and wrong-side windows."""
    return sum(1 for p in planted if win["cls"][p[-1]] in (NEAR, WRONG))


# ---- a plain restatement of the reference (full_TB.h:29-96) -------------------------------------------

def axis_tables(out_len, in_len, n, d, a):
    taps = 2 * a
    w = np.zeros((out_len, taps))
    first = np.zeros(out_len, np.int64)
    for xx in range(out_len):
        w[xx], first[xx] = NT.weights(xx, n, d, a)
    idx = first[:, None] + np.arange(taps)[None, :]
    valid = (idx >= 0) & (idx < in_len)
    return w, np.clip(idx, 0, in_len - 1), valid


def restate_planar(img, out_w, out_h, a, n, d, clean, parts=False):
    """uint8 [C][H][W] -> [C][out_h][out_w]: sequential double sums in ascending taps over the clipped window, clamp,
    truncate; rows first, then columns bottom-up in place (clean=False) or from a copy of the row pass (clean=True).
    parts=True returns (out, row pass [C][H][out_w] uint8, column sums [C][out_h][out_w] before quantisation)."""
    c, h, w = img.shape
    wx, ix, vx = axis_tables(out_w, w, n, d, a)
    wy, iy, vy = axis_tables(out_h, h, n, d, a)
    out = np.zeros((c, out_h, out_w), np.uint8)
    src = img.astype(np.float64)
    s = np.zeros((c, h, out_w))
    for k in range(2 * a):
        term = src[:, :, ix[:, k]] * wx[:, k]
        s = np.where(vx[:, k], s + term, s)
    out[:, :h, :] = NT.quantise(s)
    mid = out.copy() if clean or parts else out
    sums = np.zeros((c, out_h, out_w)) if parts else None
    for yy in range(out_h - 1, -1, -1):
        s = np.zeros((c, out_w))
        for k in range(2 * a):
            if vy[yy, k]:
                s = s + (mid if clean else out)[:, iy[yy, k], :].astype(np.float64) * wy[yy, k]
        out[:, yy, :] = NT.quantise(s)
        if parts:
            sums[:, yy, :] = s
    return (out, mid, sums) if parts else out
