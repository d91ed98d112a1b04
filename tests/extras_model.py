"""One reference for every output of the hot path's result families, on top of the oracle's score planes.

match_wta_all stacks the oracle's score planes of the shifts [m, m + D) once and derives from them what the int32 /
16-bit entries (best, web), the runner-up entries (runner_up, tests/runner_up_model.py) and the sub-pixel entries
(web_sub, tests/subpixel_model.py) report: winner-take-all with ties to the highest shift, the second-largest score of
each pixel's multiset of scores (0 with a single shift), and 16 * web + frac with frac from the scores beside the
winner (0 at both range ends).  So a test that compares several families on one input builds the planes only once."""
import numpy as np

from subpixel_model import sub_frac


def match_wta_all(orc, le, re, D, sw, variant, m=0, direct=False):
    """(best, web, runner_up, web_sub) as int32 arrays over the shifts [m, m + D) of the oracle's score planes."""
    H, W = le.shape
    scores = np.stack([orc.shift_planes(le, re, sw, m + i, variant, direct)[2] for i in range(D)])
    best = scores.max(axis=0)
    w = D - 1 - np.argmax(scores[::-1] == best[None], axis=0)  # the highest shift index that ties for best
    web = m + w + 1
    ru = np.partition(scores, D - 2, axis=0)[D - 2] if D > 1 else np.zeros((H, W), np.int32)
    frac = np.zeros((H, W), np.int64)
    inner = (w > 0) & (w < D - 1)
    if inner.any():
        take = lambda k: np.take_along_axis(scores, np.clip(k, 0, D - 1)[None], axis=0)[0]  # noqa: E731
        sm, sp = take(w - 1), take(w + 1)
        # outside `inner` (den may be 0 there) the triple is replaced by one whose frac is 0 and then discarded
        frac = np.where(inner, sub_frac(np.where(inner, best, 1), np.where(inner, sm, 0), np.where(inner, sp, 0)), 0)
    return tuple(a.astype(np.int32) for a in (best, web, ru, 16 * web + frac))


def reference_all(orc, name, le, re, D, sw, variant, m=0):
    """match_wta_all with the literal tap loop for saturated maps and small problems; maps whose rows are all equal
    are evaluated on 2*half+1 rows and expanded (as runner_up_model.reference_ru and subpixel_model.reference_sub
    do)."""
    H, W = le.shape
    half = sw // 2
    N = 2 * half + 1
    if H > N and (le == le[:1]).all() and (re == re[:1]).all():
        outs = reference_all(orc, name, le[:N], re[:N], D, sw, variant, m)
        ys = np.arange(H)
        src = np.where(ys < half, ys, np.where(ys >= H - half, ys - (H - N), half))
        return tuple(a[src] for a in outs)
    direct = name == "saturated" or W * H * D * N * N <= 10 ** 6
    return match_wta_all(orc, le, re, D, sw, variant, m=m, direct=direct)
