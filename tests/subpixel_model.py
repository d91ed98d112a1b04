"""The sub-pixel web's reference model, on top of the oracle's score planes.

match_wta_sub is the oracle's winner-take-all loop (ascending shifts, `score >= best` moves the winner, so ties go to
the highest shift) over the score planes of the shifts [m, m + D), followed by the contract of
sm_match_wta_dev_batch_sub16: with w = web - 1 the winning shift, frac = 0 where w == m or w == m + D - 1, else
s- = s(w - 1), s+ = s(w + 1), den = 2 * best - s- - s+ and frac = min(7, floor((16 * (s+ - s-) + den) / (2 * den)));
web_sub = 16 * web + frac.  All of it integer arithmetic on the oracle's exact counts."""
import numpy as np


def sub_frac(s0, sm, sp):
    """frac of the contract for arrays of (best, s-, s+) whose winner has both neighbours (den >= 1)."""
    s0, sm, sp = (np.asarray(v, np.int64) for v in (s0, sm, sp))
    den = 2 * s0 - sm - sp
    return np.minimum(7, (16 * (sp - sm) + den) // (2 * den))


def match_wta_sub(orc, le, re, D, sw, variant, direct=False, m=0):
    """(best, web, web_sub) as int32 arrays over the shifts [m, m + D) of the oracle's score planes."""
    H, W = le.shape
    scores = np.stack([orc.shift_planes(le, re, sw, m + i, variant, direct)[2] for i in range(D)]).astype(np.int64)
    best = scores.max(axis=0)
    w = D - 1 - np.argmax(scores[::-1] == best[None], axis=0)  # the highest shift index that ties for best
    web = m + w + 1
    inner = (w > 0) & (w < D - 1)
    wi = np.clip(w, 1, max(D - 2, 1))
    take = lambda k: np.take_along_axis(scores, np.clip(k, 0, D - 1)[None], axis=0)[0]
    frac = np.zeros((H, W), np.int64)
    if inner.any():
        sm, sp = take(wi - 1), take(wi + 1)
        den = np.where(inner, 2 * best - sm - sp, 1)
        frac = np.where(inner, np.minimum(7, (16 * (sp - sm) + den) // (2 * den)), 0)
    return best.astype(np.int32), web.astype(np.int32), (16 * web + frac).astype(np.int32)


def reference_sub(orc, name, le, re, D, sw, variant, m=0):
    """match_wta_sub with the literal tap loop for saturated maps and small problems; maps whose rows are all equal
    are evaluated on 2*half+1 rows and expanded (as runner_up_model.reference_ru does)."""
    H, W = le.shape
    half = sw // 2
    N = 2 * half + 1
    if H > N and (le == le[:1]).all() and (re == re[:1]).all():
        b, w, s = reference_sub(orc, name, le[:N], re[:N], D, sw, variant, m)
        ys = np.arange(H)
        src = np.where(ys < half, ys, np.where(ys >= H - half, ys - (H - N), half))
        return b[src], w[src], s[src]
    direct = name == "saturated" or W * H * D * N * N <= 10 ** 6
    return match_wta_sub(orc, le, re, D, sw, variant, direct=direct, m=m)
