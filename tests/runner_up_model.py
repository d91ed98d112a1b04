"""The runner-up score's reference model, on top of the oracle's score planes.

match_wta_ru is the oracle's winner-take-all loop (oracle_match_wta: ascending shifts, `score >= best` moves the
winner, so ties go to the highest shift) that also keeps the second order statistic: where a shift takes over,
the old best becomes the runner-up, else the runner-up is the larger of itself and the shift's score.  So
runner_up is the second-largest value of the multiset of a pixel's scores over the shifts [m, m + D): best again
where two shifts tie for best, 0 with a single shift."""
import numpy as np


def match_wta_ru(orc, le, re, D, sw, variant, direct=False, m=0):
    """(best, web, runner_up) as int32 arrays over the shifts [m, m + D) of the oracle's score planes."""
    H, W = le.shape
    best = np.zeros((H, W), np.int32)
    web = np.zeros((H, W), np.int32)
    ru = np.zeros((H, W), np.int32)
    for i in range(D):
        score = orc.shift_planes(le, re, sw, m + i, variant, direct)[2]
        win = score >= best
        ru = np.where(win, best, np.maximum(ru, score))
        web = np.where(win, m + i + 1, web)
        best = np.where(win, score, best)
    return best, web, ru


def reference_ru(orc, name, le, re, D, sw, variant, m=0):
    """match_wta_ru with the literal tap loop for saturated maps and small problems; maps whose rows are all equal
    are evaluated on 2*half+1 rows and expanded (the first and last `half` rows are those of the small frame's
    border rows, as tests/test_gpu_flavours.py's reference does)."""
    H, W = le.shape
    half = sw // 2
    N = 2 * half + 1
    if H > N and (le == le[:1]).all() and (re == re[:1]).all():
        b, w, r = reference_ru(orc, name, le[:N], re[:N], D, sw, variant, m)
        ys = np.arange(H)
        src = np.where(ys < half, ys, np.where(ys >= H - half, ys - (H - N), half))
        return b[src], w[src], r[src]
    direct = name == "saturated" or W * H * D * N * N <= 10 ** 6
    return match_wta_ru(orc, le, re, D, sw, variant, direct=direct, m=m)
