"""rae_label_topk (the fused top-k labelling kernel) against rae_label_shards on the same handle and inputs: ids[:, 0]
are the labels, probs are the full probabilities at ids bit for bit, and the chosen set agrees with float64 scores
except at rounding ties.  Every KT of the scalar body and every QT of the 16-byte body is reached."""
from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

EINVAL = -1


def _csr(n, F, fbar, seed, empty_every=0):
    rng = np.random.default_rng(seed)
    counts = rng.integers(1, 2 * fbar, size=n)
    if empty_every:
        counts[::empty_every] = 0
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum(counts, out=indptr[1:])
    indices = np.concatenate([np.sort(rng.choice(F, size=c, replace=False)) for c in counts]) if n else np.zeros(0)
    return indptr.astype(np.int32), indices.astype(np.int32)


class Case:
    """One engine handle with W [F, K] and Wb bound (world 1) and device copies of a CSR."""

    def __init__(self, K, F=600, n=3001, seed=0, zero=False, empty_every=7, fbar=8):
        import torch
        from relation_autoencoder_b200.engine import Engine
        self.torch = torch
        self.K, self.F, self.n = K, F, n
        rng = np.random.RandomState(seed)
        self.eng = Engine("rescal", K, 4, 1, 8, F, 8, 8)
        p = {"W": rng.uniform(-1, 1, (F, K)), "Wb": rng.uniform(-0.5, 0.5, K), "A": rng.uniform(-1, 1, (8, 4)),
             "Ab": np.zeros(8), "C": rng.normal(0, 0.3, (4, 4, K))}
        # a few exact ties inside rows: equal W columns and Wb entries
        if K > 8:
            p["W"][:, 7] = p["W"][:, 3]
            p["Wb"][7] = p["Wb"][3]
        if zero:
            p["W"][:] = 0
            p["Wb"][:] = 0
        self.eng.set_params_numpy({k_: v.astype(np.float32) for k_, v in p.items()})
        self.W64 = self.eng.params["W"].double().cpu().numpy()
        self.Wb64 = self.eng.params["Wb"].double().cpu().numpy()
        self.indptr, self.indices = _csr(n, F, fbar, seed + 1, empty_every)
        self.ip = torch.as_tensor(self.indptr).cuda()
        self.ix = torch.as_tensor(self.indices if self.indices.size else np.zeros(1, np.int32)).cuda()
        self.lib, self.h = self.eng.lib, self.eng._h

    def shards(self, world, W=None):
        W = self.eng.params["W"] if W is None else W
        if world == 1:
            bufs = [W]
        else:
            bufs = [W[r::world].contiguous() for r in range(world)]
        self._keep = bufs
        return (C.c_void_p * world)(*[b.data_ptr() for b in bufs])

    def full(self, w, off=0, n=None):
        t = self.torch
        n = self.n - off if n is None else n
        labels = t.empty(max(n, 1), dtype=t.int64, device="cuda")
        probs = t.empty((max(n, 1), self.K), dtype=t.float32, device="cuda")
        rc = self.lib.rae_label_shards(self.h, w, len(w), C.c_void_p(self.ip.data_ptr() + 4 * off), C.c_void_p(self.ix.data_ptr()),
                                       n, C.c_void_p(labels.data_ptr()), C.c_void_p(probs.data_ptr()), None)
        assert rc == 0, self.lib.rae_last_error(self.h)
        t.cuda.synchronize()
        return labels[:n].cpu().numpy(), probs[:n].cpu().numpy()

    def topk(self, w, k, off=0, n=None, with_probs=True, world=None):
        t = self.torch
        n = self.n - off if n is None else n
        ids = t.full((max(n, 1), k), -7, dtype=t.int32, device="cuda")
        probs = t.full((max(n, 1), k), -7.0, dtype=t.float32, device="cuda") if with_probs else None
        rc = self.lib.rae_label_topk(self.h, w, len(w) if world is None else world, C.c_void_p(self.ip.data_ptr() + 4 * off),
                                     C.c_void_p(self.ix.data_ptr()), n, k, C.c_void_p(ids.data_ptr()),
                                     C.c_void_p(probs.data_ptr() if probs is not None else 0), None)
        t.cuda.synchronize()
        if rc != 0:
            return rc, None, None
        return rc, ids[:n].cpu().numpy(), (probs[:n].cpu().numpy() if probs is not None else None)

    def close(self):
        self.eng.close()


def _check(case, ids, probs, labels, full, k, off=0):
    n = len(labels)
    assert ids.shape == (n, k)
    assert np.array_equal(ids[:, 0], labels.astype(np.int32))
    got = probs.view(np.uint32)
    want = np.take_along_axis(full, ids.astype(np.int64), axis=1).view(np.uint32)
    assert np.array_equal(got, want)                                      # bit for bit
    assert np.all(np.diff(probs, axis=1) <= 0)
    assert np.all((ids >= 0) & (ids < case.K))
    assert all(len(set(r)) == k for r in ids[:2000].tolist())
    # float64 agreement except at rounding ties (the rule of the full-size label test)
    m = min(n, 3000)
    ip = case.indptr[off:off + m + 1]
    from oracle import rae_oracle as O
    z = O.encoder_scores_fast(case.W64, case.Wb64, ip - ip[0], case.indices[ip[0]:ip[-1]])
    order = np.argsort(-z, axis=1, kind="stable")
    zs = np.take_along_axis(z, order, axis=1)
    tol = 1e-5 * max(np.abs(z).max(), 1e-30)
    for j in range(k):
        gap = (zs[:, j] - zs[:, j + 1] > tol) if j + 1 < case.K else np.ones(m, bool)
        assert np.array_equal(np.sort(ids[:m][gap, :j + 1], axis=1), np.sort(order[gap, :j + 1], axis=1)), j


SCALAR_K = [5, 50, 101, 130, 300, 1000, 1024]        # KT 1, 2, 4, 8, 16, 32, 32
VEC_K = [100, 256, 512]                               # QT 1, 2, 4


@pytest.mark.parametrize("K", SCALAR_K + VEC_K)
def test_topk_matches_label_shards(K):
    case = Case(K, F=max(600, 2 * K))
    try:
        for world in (1, 3):
            w = case.shards(world)
            labels, full = case.full(w)
            for k in sorted({1, 3, min(K, 16)}):
                rc, ids, probs = case.topk(w, k)
                assert rc == 0
                _check(case, ids, probs, labels, full, k)
                rc, ids2, none = case.topk(w, k, with_probs=False)
                assert rc == 0 and none is None and np.array_equal(ids2, ids)
            # indptr starting at an offset
            off = 11
            labels_o, full_o = case.full(w, off=off)
            rc, ids, probs = case.topk(w, 3, off=off)
            assert rc == 0
            _check(case, ids, probs, labels_o, full_o, 3, off=off)
        rows = np.diff(case.indptr) == 0
        assert rows.any()
        w = case.shards(1)
        _, ids, _ = case.topk(w, 3)
        assert np.array_equal(ids[rows], np.tile(np.argsort(-case.Wb64, kind="stable")[:3], (rows.sum(), 1)))
    finally:
        case.close()


@pytest.mark.parametrize("K", [100, 1000])
def test_topk_many_rows(K):
    case = Case(K, F=3000, n=200_003, empty_every=13)
    try:
        w = case.shards(1)
        labels, full = case.full(w)
        k = 16
        rc, ids, probs = case.topk(w, k)
        assert rc == 0
        _check(case, ids, probs, labels, full, k)
    finally:
        case.close()


@pytest.mark.parametrize("K", [5, 100, 1000])
def test_topk_all_zero_parameters(K):
    case = Case(K, zero=True)
    try:
        w = case.shards(1)
        labels, full = case.full(w)
        k = min(K, 16)
        rc, ids, probs = case.topk(w, k)
        assert rc == 0
        assert np.array_equal(ids, np.tile(np.arange(k, dtype=np.int32), (case.n, 1)))
        assert np.array_equal(probs.view(np.uint32), full[:, :k].view(np.uint32))
    finally:
        case.close()


def test_topk_misaligned_w_takes_the_scalar_path():
    """A W base 4 bytes off 16-byte alignment at K = 100: both entry points take the scalar body, whose exp-sum order
    differs from the 16-byte body's, so the reference is rae_label_shards on the same base."""
    case = Case(100)
    try:
        t = case.torch
        flat = t.empty(case.F * 100 + 4, dtype=t.float32, device="cuda")
        Wm = flat[1:1 + case.F * 100].view(case.F, 100)
        Wm.copy_(case.eng.params["W"])
        assert Wm.data_ptr() % 16 == 4
        w = (C.c_void_p * 1)(Wm.data_ptr())
        labels, full = case.full(w)
        for k in (1, 3, 16):
            rc, ids, probs = case.topk(w, k)
            assert rc == 0
            _check(case, ids, probs, labels, full, k)
    finally:
        case.close()


def test_topk_refusals():
    case = Case(5, n=20)
    try:
        w = case.shards(1)
        for k in (0, 17, 6):                  # K = 5
            assert case.topk(w, k)[0] == EINVAL
        assert b"k = 6" in case.lib.rae_last_error(case.h)
        assert case.topk(w, 3, world=0)[0] == EINVAL
        w17 = (C.c_void_p * 17)(*([case.eng.params["W"].data_ptr()] * 17))
        assert case.topk(w17, 3)[0] == EINVAL
        wnull = (C.c_void_p * 2)(case.eng.params["W"].data_ptr(), 0)
        assert case.topk(wnull, 3)[0] == EINVAL
        assert b"null W shard" in case.lib.rae_last_error(case.h)
        rc, ids, _ = case.topk(w, 3, n=0)
        assert rc == 0 and ids.shape == (0, 3)
    finally:
        case.close()


def test_engine_label_topk_covers_every_row():
    case = Case(100, n=1234)
    try:
        ids, probs = case.eng.label_topk(case.indptr, case.indices, 5)
        labels, full = case.full(case.shards(1))
        _check(case, ids, probs, labels, full, 5)
        ids2, none = case.eng.label_topk(case.ip, case.ix[:len(case.indices)], 5, probs=False)
        assert none is None and np.array_equal(ids2, ids)
        with pytest.raises(RuntimeError, match="k = 0"):
            case.eng.label_topk(case.indptr, case.indices, 0)
    finally:
        case.close()
