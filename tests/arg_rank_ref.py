"""Float64 argument ranker: the reference for rae_rank_arguments (CPU tests pin it to the oracle's cost, GPU tests
compare the kernel against it).

For example i with posterior q and the forward vectors v = M R, w = M^T L, c1 = C1 q, c2 = C2 q of
``oracle.rae_oracle.cost_and_grads`` (L = A[a1], R = A[a2], or A[a1] for model C under the args1 quirk), the candidate
scores of the two argument slots are
    s1(x) = A[x].(v + c1) + Ab[x]      s2(x) = A[x].(w + c2) + Ab[x]
and the oracle's negative-sample scores are n1 = s1(neg1) + c2.R, n2 = s2(neg2) + c1.L."""
from __future__ import annotations

import numpy as np

from oracle import rae_oracle as O


def forward(model, p, indptr, indices, a1, a2, fix_sp_quirk=False):
    """dict of float64 q, logq, L, R, v, w, c1, c2, U1 = v + c1, U2 = w + c2 (the oracle's forward pass)."""
    model = O.MODEL_ALIASES[model]
    A = np.asarray(p["A"], np.float64)
    z = O.encoder_scores_fast(np.asarray(p["W"], np.float64), np.asarray(p["Wb"], np.float64), np.asarray(indptr),
                              np.asarray(indices))
    q, logq = O.softmax_rows(z)
    n, d = len(a1), A.shape[1]
    L = A[a1]
    R = A[a1] if (model == O.MODEL_C and not fix_sp_quirk) else A[a2]
    zero = np.zeros((n, d))
    v = w = c1 = c2 = zero
    if model in (O.MODEL_A, O.MODEL_AC):
        M = np.tensordot(q, np.asarray(p["C"], np.float64), axes=[[1], [2]])
        v = np.einsum("bij,bj->bi", M, R)
        w = np.einsum("bij,bi->bj", M, L)
    if model in (O.MODEL_C, O.MODEL_AC):
        c1 = q @ np.asarray(p["C1"], np.float64).T
        c2 = q @ np.asarray(p["C2"], np.float64).T
    return dict(q=q, logq=logq, L=L, R=R, v=v, w=w, c1=c1, c2=c2, U1=v + c1, U2=w + c2)


def candidate_scores(p, U, ids):
    """s(x) = A[x].U + Ab[x] for every row of U and each entity id of ids ([n] or [n, m] per row)."""
    A = np.asarray(p["A"], np.float64)
    Ab = np.asarray(p["Ab"], np.float64)
    ids = np.asarray(ids)
    if ids.ndim == 1:
        return (A[ids] * U).sum(1) + Ab[ids]
    return np.einsum("bmj,bj->bm", A[ids], U) + Ab[ids]


def thresholds(p, U, true_ids):
    return candidate_scores(p, U, true_ids)


def counts_above(p, U, true_ids, t, chunk=256):
    """#{x != true : s(x) > t} per row (float64, all N entities)."""
    A = np.asarray(p["A"], np.float64)
    Ab = np.asarray(p["Ab"], np.float64)
    out = np.zeros(len(true_ids), np.int64)
    for s in range(0, len(true_ids), chunk):
        S = U[s:s + chunk] @ A.T + Ab[None, :]
        above = S > np.asarray(t)[s:s + chunk, None]
        above[np.arange(above.shape[0]), np.asarray(true_ids)[s:s + chunk]] = False
        out[s:s + chunk] = above.sum(1)
    return out


def tolerance(p, U):
    """tau per query: 1e-5 (sum_j |U_j| max_x |A_xj| + max |Ab|)."""
    A = np.asarray(p["A"], np.float64)
    Ab = np.asarray(p["Ab"], np.float64)
    return 1e-5 * (np.abs(U) @ np.abs(A).max(0) + np.abs(Ab).max())


def ranks(model, p, indptr, indices, a1, a2, fix_sp_quirk=False):
    """(rank1, rank2) int64: 1 + #{x != true : s(x) > s(true)} per slot."""
    f = forward(model, p, indptr, indices, a1, a2, fix_sp_quirk)
    out = []
    for U, t_ids in ((f["U1"], a1), (f["U2"], a2)):
        out.append(1 + counts_above(p, U, t_ids, thresholds(p, U, t_ids)))
    return out[0], out[1]


def bracket(model, p, indptr, indices, a1, a2):
    """Per slot, (lo, hi): the float64 ranks at thresholds t + tau and t - tau.  A rank computed with fp32-accurate
    scores lies in [lo, hi]."""
    f = forward(model, p, indptr, indices, a1, a2)
    out = []
    for U, t_ids in ((f["U1"], a1), (f["U2"], a2)):
        t, tau = thresholds(p, U, t_ids), tolerance(p, U)
        out.append((1 + counts_above(p, U, t_ids, t + tau), 1 + counts_above(p, U, t_ids, t - tau)))
    return out


def cost_from_candidates(model, p, indptr, indices, a1, a2, neg1, neg2, alpha, fix_sp_quirk=False):
    """The oracle's batch cost rebuilt from the candidate scores: positives, negatives and the entropy term."""
    model = O.MODEL_ALIASES[model]
    f = forward(model, p, indptr, indices, a1, a2, fix_sp_quirk)
    Ab = np.asarray(p["Ab"], np.float64)
    L, R, c1, c2 = f["L"], f["R"], f["c1"], f["c2"]
    k1 = (c2 * R).sum(1)                 # x-independent terms of slot 1 / slot 2
    k2 = (c1 * L).sum(1)
    u1 = candidate_scores(p, f["U1"], a1) + k1
    if model == O.MODEL_C and not fix_sp_quirk:
        # the quirk: the cost's slot-2 positive never reads A[a2] (SelectionalPreferences.py:35), u2 = pos + Ab[a2]
        u2 = (L * f["v"]).sum(1) + k2 + k1 + Ab[a2]
    else:
        u2 = candidate_scores(p, f["U2"], a2) + k2
    n1 = candidate_scores(p, f["U1"], np.asarray(neg1).T).T + k1[None, :]
    n2 = candidate_scores(p, f["U2"], np.asarray(neg2).T).T + k2[None, :]
    ent = alpha * -(f["logq"] * f["q"]).sum(1)
    S, B = np.asarray(neg1).shape
    total = (O._log_sigmoid(u1).sum() + O._log_sigmoid(u2).sum() + 2.0 * ent.sum()
             + O._log_sigmoid(-n1).sum() + O._log_sigmoid(-n2).sum())
    return -total / float(4 * B + 2 * B * S)
