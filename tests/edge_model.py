"""A float64 model of the edge detector (step 1) and images that probe its threshold table at every boundary.

The 8-bit detector of the library does not evaluate the reference's FP64 expression (stereo.c:16-28) per pixel: it
tabulates the decision for every pair of 3-pixel sums (k_edge_lut), turns the table into one threshold hi[m] per
smaller sum (k_edge_thresholds) and decides max(L, R) > hi[min(L, R)] in integers.  It is right only if it reproduces
the FP64 rounding of the reference exactly, and that matters only at the boundary M = hi[m] / hi[m] + 1 of each m.
The probe images built here put every boundary entry of a threshold's table in front of one detector of one pixel
while the other three detectors of that pixel stay silent, so that a single wrong entry changes a single edge bit.
"""
import functools

import numpy as np

WRAP, GHOST = 0, 1
NSUM = 766  # 3-pixel sums of 8-bit pixels: 0 .. 765

# The stencil of a pixel as a 3 x 3 tile, (row, column) = (dy + 1, dx + 1):
#     tl tc tr
#     ml  c mr
#     bl bc br
# and the four detectors as the cells of their first and second 3-pixel sum, in the reference's order of addition
# (left_right stereo.c:16-28, top_bottom :30-42, upleft_downright :44-56, downleft_upright :58-70).
DETECTORS = (
    (((0, 0), (1, 0), (2, 0)), ((0, 2), (1, 2), (2, 2))),  # left_right: tl ml bl | tr mr br
    (((0, 0), (0, 1), (0, 2)), ((2, 0), (2, 1), (2, 2))),  # top_bottom: tl tc tr | bl bc br
    (((0, 0), (0, 1), (1, 0)), ((1, 2), (2, 1), (2, 2))),  # upleft_downright: tl tc ml | mr bc br
    (((2, 0), (2, 1), (1, 0)), ((0, 1), (0, 2), (1, 2))),  # downleft_upright: bl bc ml | tc tr mr
)
DIRECTIONS = ("left_right", "top_bottom", "upleft_downright", "downleft_upright")

# The thresholds the edge tests run at.  0 and the smallest subnormal: any difference fires; 1e-4 and 2.5e-3: the
# FP64 fallback of one-pixel-wide / one-pixel-high GHOST frames decides on |a - b| across its range; 0.15: the table
# built when a context is created; 0.5 has exact ties at (3k, 5k), 1.0 at (m, 3m).
THRESHOLDS = (0.0, 5e-324, 1e-4, 2.5e-3, 0.05, 0.15, 1 / 3, 0.4, 0.5, 2 / 3, 1.0)
NEAR_ZERO = (0.0, 5e-324, 1e-4, 2.5e-3)


def _decide(l, r, thr):
    """stereo.c:16-28 from the two averages on: (l + r) / 2.0, thr * overall, CLAMP to [0, 1] (util.h:24-26),
    fabs(l - r) > lim.  Numpy's float64 element-wise operations round to nearest and are never contracted."""
    ov = (l + r) / 2.0
    lim = np.minimum(np.maximum(thr * ov, 0.0), 1.0)
    return np.abs(l - r) > lim


@functools.lru_cache(maxsize=None)
def detect_table(thr):
    """The decision of one detector for every pair of 3-pixel sums, T[L, R] (766 x 766 bool).  The three cells of a
    sum are k / 256.0, exact, and so is their sum: ((a + b) + c) / 3.0 is (L / 256.0) / 3.0."""
    l = (np.arange(NSUM) / 256.0) / 3.0
    t = _decide(l[:, None], l[None, :], thr)
    t.flags.writeable = False
    return t


@functools.lru_cache(maxsize=None)
def hi(thr):
    """The thresholds as k_edge_thresholds derives them: for each smaller sum m the largest M >= m without an edge,
    765 when none fires."""
    t = detect_table(thr)
    idx = np.arange(NSUM)
    upper = t & (idx[None, :] >= idx[:, None])
    h = np.where(upper.any(1), upper.argmax(1), NSUM) - 1
    h.flags.writeable = False
    return h


def model_edges(img, thr, variant):
    """The four detectors over a whole u8 image in float64, as the reference evaluates them on img / 256.0: WRAP on
    the torus, GHOST with 128.0 ghost cells around the frame (stereo-ghost.c:384-385)."""
    h, w = img.shape
    b = img.astype(np.float64) / 256.0
    p = np.pad(b, 1, mode="wrap") if variant == WRAP else np.pad(b, 1, constant_values=128.0)

    def avg(cells):
        (r0, c0), (r1, c1), (r2, c2) = cells
        return ((p[r0:r0 + h, c0:c0 + w] + p[r1:r1 + h, c1:c1 + w]) + p[r2:r2 + h, c2:c2 + w]) / 3.0

    e = np.zeros((h, w), bool)
    for a, bb in DETECTORS:
        e |= _decide(avg(a), avg(bb), thr)
    return e.astype(np.uint8)


def boundary_pairs(thr):
    """Every ordered pair of sums (A, B) of a boundary entry: {min, max} = (m, hi[m]) or (m, hi[m] + 1) for each m
    with hi[m] < 765.  (m, m) occurs once."""
    h = hi(thr)
    out = set()
    for m in np.nonzero(h < NSUM - 1)[0]:
        for big in (int(h[m]), int(h[m]) + 1):
            out.add((int(m), big))
            out.add((big, int(m)))
    return np.array(sorted(out), np.int64).reshape(-1, 2)


def _sums(cells, det):
    """The two sums of detector `det` over stencils given as an (..., 3, 3) integer array."""
    a, b = DETECTORS[det]
    return sum(cells[..., r, c] for r, c in a), sum(cells[..., r, c] for r, c in b)


def _decisive(cells, thr, det):
    """Stencils (..., 3, 3) on which the three detectors other than `det` do not fire."""
    t = detect_table(thr)
    ok = np.ones(cells.shape[:-2], bool)
    for j in range(4):
        if j != det:
            a, b = _sums(cells, j)
            ok &= ~t[a, b]
    return ok


def _split3(rng, s):
    """Random decompositions of the sums s (any shape) into three values in [0, 255]."""
    a = rng.integers(np.maximum(0, s - 510), np.minimum(255, s) + 1)
    rest = s - a
    b = rng.integers(np.maximum(0, rest - 255), np.minimum(255, rest) + 1)
    return a, b, rest - b


def _search(thr, det, pairs, rng, tries=4000, chunk=250):
    """Random search: the probed detector's two sums split into three cells at random, the free cells drawn at
    random, the first decisive draw of `tries` per pair kept.  Returns stencils (P, 3, 3) and a found mask."""
    n = len(pairs)
    out = np.zeros((n, 3, 3), np.int64)
    found = np.zeros(n, bool)
    a_cells, b_cells = DETECTORS[det]
    free = [(r, c) for r in range(3) for c in range(3) if (r, c) not in a_cells + b_cells]
    for _ in range(tries // chunk):
        todo = np.nonzero(~found)[0]
        if len(todo) == 0:
            break
        cells = np.empty((len(todo), chunk, 3, 3), np.int64)
        for cells_of, s in ((a_cells, pairs[todo, 0]), (b_cells, pairs[todo, 1])):
            parts = _split3(rng, np.repeat(s[:, None], chunk, 1))
            for (r, c), v in zip(cells_of, parts):
                cells[:, :, r, c] = v
        for r, c in free:
            cells[:, :, r, c] = rng.integers(0, 256, (len(todo), chunk))
        ok = _decisive(cells, thr, det)
        hit = ok.any(1)
        first = ok.argmax(1)
        rows = todo[hit]
        out[rows] = cells[hit, first[hit]]
        found[rows] = True
    return out, found


def _constructed(det, A, B, free=128):
    """A stencil in which detector `det` compares the sums (A, B) and the other three compare equal sums, so that
    they cannot fire at any threshold; None when no such stencil of this form exists (it needs max <= 2 * min).

    left_right: top row = bottom row = (p, q, s), p + ml = s + mr = K, so A = p + K and B = s + K.
    upleft_downright: the stencil equal to its transpose (tc = ml, tr = bl, bc = mr), tl + ml = mr + br = K, so
    A = K + ml and B = K + mr.  top_bottom is the transpose of a left_right stencil, downleft_upright the left-right
    mirror of an upleft_downright stencil with the two sums exchanged."""
    if det == 1:
        s = _constructed(0, A, B, free)
        return None if s is None else s.T.copy()
    if det == 3:
        s = _constructed(2, B, A, free)
        return None if s is None else s[:, ::-1].copy()
    lo = max(max(A, B) - 255, (max(A, B) + 1) // 2)
    up = min(min(A, B), (min(A, B) + 255) // 2)
    if lo > up:
        return None
    k = (lo + up) // 2
    s = np.full((3, 3), free, np.int64)
    if det == 0:
        s[0, 0] = s[2, 0] = A - k
        s[0, 2] = s[2, 2] = B - k
        s[1, 0], s[1, 2] = 2 * k - A, 2 * k - B
    else:
        s[1, 0] = s[0, 1] = A - k
        s[1, 2] = s[2, 1] = B - k
        s[0, 0], s[2, 2] = 2 * k - A, 2 * k - B
    return s


@functools.lru_cache(maxsize=None)
def probes(thr, seed=0):
    """The decisive stencils of a threshold: for every direction, a (P, 3, 3) u8 array of stencils and the (P, 2)
    ordered sums (A, B) they put in front of that direction's detector.  Random search first (random cells exercise
    the detector more than constructed ones); near 0, where almost any difference fires and random draws rarely
    succeed, constructed stencils first.  Pairs with neither are left out: boundary_pairs(thr) minus these are the
    infeasible ones."""
    rng = np.random.default_rng(seed)
    pairs = boundary_pairs(thr)
    out = []
    for det in range(4):
        st = np.zeros((len(pairs), 3, 3), np.int64)
        found = np.zeros(len(pairs), bool)

        def construct():
            for i in np.nonzero(~found)[0]:
                s = _constructed(det, int(pairs[i, 0]), int(pairs[i, 1]))
                if s is not None and _decisive(s, thr, det):
                    st[i], found[i] = s, True

        if thr < 0.01:
            construct()
        todo = np.nonzero(~found)[0]
        st[todo], found[todo] = _search(thr, det, pairs[todo], rng)
        construct()
        out.append((st[found].astype(np.uint8), pairs[found]))
    return tuple(out)


def all_stencils(thr, seed=0):
    """Every probe stencil of the threshold, the four directions interleaved so that each frame gets some of each."""
    ps = [st for st, _ in probes(thr, seed)]
    n = max(len(s) for s in ps)
    order = [s[i] for i in range(n) for s in ps if i < len(s)]
    return np.stack(order) if order else np.zeros((0, 3, 3), np.uint8)


def filler(rng, h, w):
    """Smooth content plus noise: no tile of a frame sits in a flat area."""
    y, x = np.mgrid[0:h, 0:w]
    base = 128 + 70 * np.sin(x / 5.3 + 0.7 * np.sin(y / 11.0)) * np.cos(y / 7.1)
    return np.clip(base + rng.integers(-24, 25, (h, w)), 0, 255).astype(np.uint8)


def _centres(variant, w, h):
    """Where probe stencils go, in order.  WRAP: first along the four seams (x = 0, x = W - 1, y = 0, y = H - 1), so
    that stencils straddle them, then a grid of step 3, whose centres run through every residue of x mod 4 and
    mod 32.  GHOST: the interior only (the border rule is tested on its own)."""
    out = []
    if variant == WRAP:
        for y in range(1, h - 1, 6):
            out.append((0, y))
            out.append((w - 1, y + 3))
        for x in range(1, w - 1, 6):
            out.append((x, 0))
            out.append((x + 3, h - 1))
        out += [(x, y) for y in range(1, h - 1, 3) for x in range(1, w - 1, 3)]
    else:
        out += [(x, y) for y in range(1, h - 1, 3) for x in range(1, w - 1, 3)]
    return out


@functools.lru_cache(maxsize=None)
def _placement(variant, w, h):
    """The centres of _centres whose 3 x 3 tiles (wrapped) do not overlap, first come first served."""
    used = np.zeros((h, w), bool)
    placed = []
    for cx, cy in _centres(variant, w, h):
        ys = [(cy + d) % h for d in (-1, 0, 1)]
        xs = [(cx + d) % w for d in (-1, 0, 1)]
        if len(set(ys)) < 3 or len(set(xs)) < 3 or used[np.ix_(ys, xs)].any():
            continue
        used[np.ix_(ys, xs)] = True
        placed.append((cx, cy))
    assert placed, "frame too small for a stencil"
    return np.array(placed, np.int64)


def probe_frames(thr, variant, w, h, seed=0):
    """Frames (n, h, w) u8 that together hold every probe stencil of the threshold, one probe pixel per 3 x 3 tile,
    the remaining tiles filler.  Also returns each frame's probe centres."""
    assert w >= 3 and h >= 3
    st = all_stencils(thr)
    at = _placement(variant, w, h)
    rng = np.random.default_rng(seed + 1)
    d = np.arange(-1, 2)
    frames, where = [], []
    for k in range(0, max(len(st), 1), len(at)):
        img = filler(rng, h, w)
        c = at[:len(st) - k]
        ys, xs = (c[:, 1, None] + d) % h, (c[:, 0, None] + d) % w
        img[ys[:, :, None], xs[:, None, :]] = st[k:k + len(at)]
        frames.append(img)
        where.append([tuple(p) for p in c.tolist()])
    return np.stack(frames), where


def stencil_sums(img, variant):
    """The integer sums (4, 2, H, W) of the four detectors at every pixel (WRAP: on the torus), and for GHOST the
    mask of pixels whose stencil is inside the frame (the only ones the sums describe)."""
    h, w = img.shape
    p = np.pad(img.astype(np.int64), 1, mode="wrap")
    cells = np.stack([np.stack([p[r:r + h, c:c + w] for c in range(3)], -1) for r in range(3)], -2)
    sums = np.stack([np.stack(_sums(cells, d)) for d in range(4)])
    inside = np.ones((h, w), bool)
    if variant == GHOST:
        inside[[0, -1], :] = False
        inside[:, [0, -1]] = False
    return sums, inside


def decisive_hits(img, thr, variant):
    """For each direction, the set of ordered boundary pairs (A, B) that some pixel of the image puts in front of
    that detector while the other three do not fire."""
    t, h = detect_table(thr), hi(thr)
    sums, inside = stencil_sums(img, variant)
    fires = np.stack([t[sums[d, 0], sums[d, 1]] for d in range(4)])
    out = []
    for d in range(4):
        a, b = sums[d]
        mn, mx = np.minimum(a, b), np.maximum(a, b)
        quiet = ~(fires[[j for j in range(4) if j != d]].any(0))
        at = inside & quiet & (h[mn] < NSUM - 1) & ((mx == h[mn]) | (mx == h[mn] + 1))
        out.append(set(zip(a[at].tolist(), b[at].tolist())))
    return out
