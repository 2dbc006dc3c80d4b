"""Shared helpers for the test-suite: seeded random problem instances and an independent torch-float64
transcription of the reference's Theano graph (used to pin the NumPy oracle; Theano itself is not installable)."""
from __future__ import annotations

import numpy as np

from oracle import rae_oracle as O


def tc_eligible(model, K, d):
    """Shapes the tcgen05 contraction path takes (rae_decoder_tc.cu: tc_supported): a bilinear model, 16 < d <= 128, K <= 104."""
    return O.MODEL_ALIASES.get(model, model) != "sp" and 16 < d <= 128 and K <= 104


def record_err(test, name, value):
    """Measured parity errors, appended to $RAE_PARITY_LOG (one JSON line each) so a GPU run leaves the margins behind."""
    import json
    import os
    path = os.environ.get("RAE_PARITY_LOG")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps({"test": test, "what": name, "err": float(value)}) + "\n")


def make_problem(model, B=12, K=5, d=6, S=3, F=40, N=25, fbar=4, seed=0, dup_heavy=False, empty_rows=False, hot_rows=False):
    """Random tiny instance: params in reference init order + one batch with injected negatives.

    hot_rows: feature ids 0-4 and entity ids 0-4 get fixed shares of the batch on top of the random draws - id 0 in every
    example, id 1 in every 5th, ids 2-4 in every 14th each (at B = 512: 512, ~100 and ~37 occurrences), so that the
    sparse-row update sees rows cut by one chunk boundary, rows over a few chunks and rows over many chunks."""
    rng = np.random.RandomState(seed)
    p = O.init_params(rng, model, F, K, N, d)
    # make biases / W non-trivial so every term is exercised
    p["W"] = rng.uniform(-0.5, 0.5, size=(F, K))
    p["Wb"] = rng.uniform(-0.3, 0.3, size=K)
    p["A"] = rng.uniform(-0.8, 0.8, size=(N, d))
    p["Ab"] = rng.uniform(-0.3, 0.3, size=N)
    indptr = [0]
    indices = []
    for b in range(B):
        n = int(rng.randint(1, 2 * fbar))
        if empty_rows and b % 5 == 0:
            n = 0
        feats = np.sort(rng.choice(F, size=min(n, F), replace=False))
        if hot_rows:
            feats = np.union1d(feats, _hot_ids(b))
        indices.extend(feats.tolist())
        indptr.append(len(indices))
    hiN = max(2, N // 5) if dup_heavy else N
    a1 = rng.randint(0, hiN, size=B).astype(np.int32)
    a2 = rng.randint(0, hiN, size=B).astype(np.int32)
    neg1 = rng.randint(0, hiN, size=(S, B)).astype(np.int32)
    neg2 = rng.randint(0, hiN, size=(S, B)).astype(np.int32)
    if hot_rows:
        b = np.arange(B)
        a1[:] = 0
        a2[b % 5 == 0] = 1
        for k in range(3):
            neg1[0, b % 14 == k] = 2 + k
    return dict(p=p, indptr=np.asarray(indptr, dtype=np.int32), indices=np.asarray(indices, dtype=np.int32),
                a1=a1, a2=a2, neg1=neg1, neg2=neg2)


def _hot_ids(b):
    """The hot feature ids of example b (make_problem(hot_rows=True))."""
    return [0] + ([1] if b % 5 == 0 else []) + [2 + k for k in range(3) if b % 14 == k]


def torch_reference_cost(model, p, indptr, indices, a1, a2, neg1, neg2, alpha, l1, l2, adj, ext_reg):
    """Op-by-op torch float64 transcription of the Theano graph (independent of the oracle's closed forms).

    Encoder RelationClassifier.py:35-36; entropy OieModel.py:81; decoders Bilinear.py:28-79,
    SelectionalPreferences.py:30-51, BilinearPlusSP.py:34-102; -mean OieModel.py:90; regulariser
    OieModel.py:54-62 + OieInduction.py:134-135.  Returns (cost tensor, dict of leaf tensors).
    """
    import torch
    model = O.MODEL_ALIASES[model]
    t = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in p.items()}
    B = len(indptr) - 1
    F = p["W"].shape[0]
    X = torch.zeros(B, F, dtype=torch.float64)
    for b in range(B):
        X[b, torch.as_tensor(indices[indptr[b]:indptr[b + 1]], dtype=torch.long)] = 1.0
    scores = X @ t["W"] + t["Wb"]
    q = torch.softmax(scores, dim=1)
    entropy = alpha * -(torch.log(q) * q).sum(dim=1)
    A, Ab = t["A"], t["Ab"]
    a1t = torch.as_tensor(a1, dtype=torch.long)
    a2t = torch.as_tensor(a2, dtype=torch.long)
    n1t = torch.as_tensor(neg1, dtype=torch.long)
    n2t = torch.as_tensor(neg2, dtype=torch.long)
    S = neg1.shape[0]
    d = p["A"].shape[1]
    ls = torch.nn.functional.logsigmoid

    def bt(a, b_, *_):
        """T.batched_tensordot(a, b, axes=[[1],[1]]) for the four operand-rank combinations the decoders use."""
        if a.dim() == 3 and b_.dim() == 2:      # (l,r,r) x (l,r)   -> (l,r)
            return torch.einsum("bij,bi->bj", a, b_)
        if a.dim() == 3 and b_.dim() == 3:      # (l,r,r) x (l,r,s) -> (l,r,s)
            return torch.einsum("bij,bis->bjs", a, b_)
        if a.dim() == 2 and b_.dim() == 3:      # (l,r) x (l,r,s)   -> (l,s)
            return torch.einsum("bj,bjs->bs", a, b_)
        raise ValueError

    def bt32(a, b_):                            # (l,r,s) x (l,r) -> (l,s)   (Bilinear.py:69)
        return torch.einsum("bjs,bj->bs", a, b_)

    if model == O.MODEL_A:
        e1, e2 = A[a1t], A[a2t]
        wR = torch.tensordot(q, t["C"], dims=([1], [2]))
        afirst = bt(wR, e1)
        one = (afirst * e2).sum(1)
        u = torch.cat([one + Ab[a1t], one + Ab[a2t]])
        allS = torch.cat([ls(u), entropy, entropy])
        x = A[n1t.reshape(-1)].reshape(S, B, d)
        y = A[n2t.reshape(-1)].reshape(S, B, d)
        negOne = bt32(bt(wR, x.permute(1, 2, 0)), e2)
        negTwo = bt(afirst, y.permute(1, 2, 0))
        g = torch.cat([negOne + Ab[n1t].permute(1, 0), negTwo + Ab[n2t].permute(1, 0)])
        allS = torch.cat([allS, ls(-g).flatten()])
    elif model == O.MODEL_C:
        wC1 = q @ t["C1"].permute(1, 0)
        wC2 = q @ t["C2"].permute(1, 0)
        left = (wC1 * A[a1t.flatten()]).sum(1)
        right = (wC2 * A[a1t.flatten()]).sum(1)
        one = left + right
        u = torch.cat([one + Ab[a1t], one + Ab[a2t]])
        allS = torch.cat([ls(u), entropy, entropy])
        x = A[n1t.reshape(-1)].reshape(S, B, d)
        y = A[n2t.reshape(-1)].reshape(S, B, d)
        nl = bt(wC1, x.permute(1, 2, 0))
        nr = bt(wC2, y.permute(1, 2, 0))
        negOne = nl.permute(1, 0) + right
        negTwo = nr.permute(1, 0) + left
        g = torch.cat([negOne + Ab[n1t], negTwo + Ab[n2t]])
        allS = torch.cat([allS, ls(-g).flatten()])
    else:
        wC1 = q @ t["C1"].permute(1, 0)
        wC2 = q @ t["C2"].permute(1, 0)
        wC = torch.tensordot(q, t["C"], dims=([1], [2]))
        e1, e2 = A[a1t], A[a2t]
        afirst = bt(wC, e1)
        one = (afirst * e2).sum(1) + (wC1 * e1).sum(1) + (wC2 * e2).sum(1)
        u = torch.cat([one + Ab[a1t], one + Ab[a2t]])
        allS = torch.cat([ls(u), entropy, entropy])
        x = A[n1t.reshape(-1)].reshape(S, B, d)
        y = A[n2t.reshape(-1)].reshape(S, B, d)
        xt, yt = x.permute(1, 2, 0), y.permute(1, 2, 0)
        negOne = bt32(bt(wC, xt), e2) + bt(wC1, xt) + (wC2 * e2).sum(1).reshape(B, 1)
        negTwo = bt(afirst, yt) + bt(wC2, yt) + (wC1 * e1).sum(1).reshape(B, 1)
        g = torch.cat([negOne + Ab[n1t].permute(1, 0), negTwo + Ab[n2t].permute(1, 0)])
        allS = torch.cat([allS, ls(-g).flatten()])
    cost = -allS.mean()
    names = O.regularised_names(model, ext_reg)
    L1 = sum(t[n].abs().sum() for n in names)
    L2 = sum((t[n] ** 2).sum() for n in names)
    cost = cost + l1 * L1 * adj + l2 * L2 * adj
    return cost, t, q


def rel_err(a, b):
    """||a-b||_inf / max(||b||_inf, tiny): the tensor-relative error all parity tolerances are stated in."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    den = max(float(np.abs(b).max()) if b.size else 0.0, 1e-30)
    return float(np.abs(a - b).max() / den) if b.size else 0.0
