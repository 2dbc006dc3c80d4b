"""Float64 argument predictor: the reference for rae_predict_arguments, built on the candidate scores of
tests/arg_rank_ref.py.  Per row and slot, the k entities with the highest s(x) = A[x].U + Ab[x], score descending, equal
scores by ascending entity id."""
from __future__ import annotations

import numpy as np

from tests import arg_rank_ref as R


def all_scores(p, U):
    """float64 [n, N]: s(x) for every row of U and every entity."""
    return U @ np.asarray(p["A"], np.float64).T + np.asarray(p["Ab"], np.float64)[None, :]


def topk(S, k):
    """(ids int64 [n, k], scores float64 [n, k]) of a score matrix: a stable sort of -S keeps the lower id first on ties."""
    ids = np.argsort(-S, axis=1, kind="stable")[:, :k]
    return ids, np.take_along_axis(S, ids, axis=1)


def slot_scores(model, p, indptr, indices, a1, a2, fix_sp_quirk=False):
    """((S1, tau1), (S2, tau2)): the full float64 score matrices of slot 1 (candidates for args1) and slot 2, with the
    per-row tolerance of arg_rank_ref.tolerance."""
    f = R.forward(model, p, indptr, indices, a1, a2, fix_sp_quirk)
    return tuple((all_scores(p, f[u]), R.tolerance(p, f[u])) for u in ("U1", "U2"))


def predictions(model, p, indptr, indices, a1, a2, k, fix_sp_quirk=False):
    """(ids1, scores1, ids2, scores2) float64 top-k per slot."""
    (S1, _), (S2, _) = slot_scores(model, p, indptr, indices, a1, a2, fix_sp_quirk)
    i1, s1 = topk(S1, k)
    i2, s2 = topk(S2, k)
    return i1, s1, i2, s2


def check_fp32_lists(ids, scores, S, tau, k):
    """Asserts that fp32-accurate lists (ids, scores) [n, k] are what the float64 scores S [n, N] allow within tau [n]:
    distinct ids in [0, N) ordered by (score descending, id ascending) exactly, |score - S[id]| <= tau, every entity
    above the k-th float64 score + 2 tau listed and every listed entity at least the k-th float64 score - 2 tau."""
    n, N = S.shape
    assert ids.shape == (n, k) and scores.shape == (n, k)
    assert ids.min() >= 0 and ids.max() < N
    assert all(len(set(r)) == k for r in ids.tolist())
    if k > 1:
        a, b = scores[:, :-1], scores[:, 1:]
        assert np.all((a > b) | ((a == b) & (ids[:, :-1] < ids[:, 1:])))
    got = np.take_along_axis(S, ids.astype(np.int64), axis=1)
    err = np.abs(scores.astype(np.float64) - got)
    assert np.all(err <= tau[:, None]), "score error %g > tau" % err.max()
    kth = np.sort(S, axis=1)[:, N - k]
    listed = np.zeros_like(S, dtype=bool)
    np.put_along_axis(listed, ids.astype(np.int64), True, axis=1)
    must = S > (kth + 2 * tau)[:, None]
    assert not np.any(must & ~listed), "an entity clearly in the top %d is missing" % k
    assert np.all(got >= (kth - 2 * tau)[:, None]), "a listed entity is clearly outside the top %d" % k
