#!/usr/bin/env python
"""Cost weights of the tcgen05 contraction schedules (rae_decoder_tc.cu: tc_cost) from a per-CTA life table.

usage: fit_sched_cost.py CSV d [fwd rec dq]

CSV: pass, cta, life_cycles, segments, ends_tile, first_unit, end_unit per CTA of one step's forward, recompute and dq
kernels (profiles/r04_cta_life_before_*.csv: the -DRAE_TRACE build, profiles/trace_tc.py, at K = 100, B = 4096).  The
optional cadences are the steady-state cycles per unit of each pass; the defaults are the medians of the chunk-4 ->
chunk-12 (forward, recompute) and stage-8 -> stage-24 (dq) stamps of the T trace of the parent build.  A CTA's life less
its body units at the cadence is fitted by least squares to c0 + wt * tail units + h * (segments - 1); the weights are
printed in eighths of a body unit, the unit tc_cost uses.
"""
import csv
import sys

import numpy as np

path, d = sys.argv[1], int(sys.argv[2])
cadence = dict(zip(("fwd", "rec", "dq"), (float(v) for v in sys.argv[3:6]))) if len(sys.argv) > 5 else \
    {"fwd": 1735.0, "rec": 1740.0, "dq": 1584.0}
DP = 32 if d <= 32 else 64 if d <= 64 else 128
rps = 128 // DP
n_bil_rows = (d + rps - 1) // rps * rps * DP
n_bil_half, n_sp_half = n_bil_rows // 64, 2 * DP // 64
n_fwd, n_rec, n_st = (n_bil_half + n_sp_half + 1) // 2, n_bil_half // 2, (n_bil_rows + 2 * DP + 127) // 128
geom = {"fwd": (n_fwd, n_fwd - n_rec), "rec": (n_rec, 0), "dq": (n_st, n_st - n_bil_rows // 128)}   # units per tile, tail units

rows = list(csv.DictReader(open(path)))
for name, (upt, ntail) in geom.items():
    A, y = [], []
    for r in (r for r in rows if r["pass"] == name):
        u = np.arange(int(r["first_unit"]), int(r["end_unit"]))
        tail = int(np.count_nonzero(u % upt >= upt - ntail))
        A.append([1.0, tail, int(r["segments"]) - 1])
        y.append(int(r["life_cycles"]) - cadence[name] * (len(u) - tail))
    A, y = np.array(A), np.array(y)
    cols = [0, 1, 2] if ntail else [0, 2]
    coef = np.linalg.lstsq(A[:, cols], y, rcond=None)[0]
    fit = dict(zip(["c0", "wt", "h"] if ntail else ["c0", "h"], coef))
    resid = np.abs(y - A[:, cols] @ coef).max()
    wt = 8 * fit.get("wt", cadence[name]) / cadence[name]
    print("%-3s  DP=%d  c0 %.0f cycles, tail unit %.0f, segment switch %.0f cycles -> wt = %.1f, h = %.1f eighths "
          "(largest residual %.0f cycles)" % (name, DP, fit["c0"], fit.get("wt", cadence[name]), fit["h"], wt,
                                             8 * fit["h"] / cadence[name], resid))
