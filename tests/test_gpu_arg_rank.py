"""rae_rank_arguments (fused tcgen05 argument-ranking kernel) against the float64 ranker of tests/arg_rank_ref.py.

Scores are fp32-accurate, so a GPU rank must lie in the float64 bracket: 1 + #{x != true : s(x) > t + tau} <= rank <=
1 + #{x != true : s(x) > t - tau}, tau = 1e-5 (sum_j |U_j| max_x |A_xj| + max |Ab|) per query.  Covered: models A, C, AC;
d = 10 and 256 (SIMT forward), d = 30 and 128 (tcgen05 forward) and d = 128 under RAE_FLAG_FORCE_SIMT; N and n_rows
that are multiples of no tile and of no batch, an offset indptr, empty rows, args1 == args2, true entities at both ends
of the id range and at both ends of the ranking, run-to-run identity, the refusals, a trained model and the export."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import pytest

from tests import arg_rank_ref as R

pytestmark = pytest.mark.gpu

EINVAL, ENOTBOUND = -1, -3
FORCE_SIMT = 4


def _params(model, K, d, F, N, seed):
    rng = np.random.RandomState(seed)
    p = {"W": rng.uniform(-1, 1, (F, K)), "Wb": rng.uniform(-0.5, 0.5, K), "A": rng.uniform(-1, 1, (N, d)),
         "Ab": rng.uniform(-0.3, 0.3, N), "C": rng.normal(0, 0.8 / np.sqrt(d), (d, d, K)),
         "C1": rng.normal(0, 0.5, (d, K)), "C2": rng.normal(0, 0.5, (d, K))}
    return {k: v.astype(np.float32) for k, v in p.items()}


def _csr(n, F, seed, empty_every=5, lead=0):
    rng = np.random.default_rng(seed)
    counts = rng.integers(1, 12, size=n)
    counts[::empty_every] = 0
    indptr = np.zeros(n + 1, np.int64)
    np.cumsum(counts, out=indptr[1:])
    indptr += lead
    body = [np.sort(rng.choice(F, size=c, replace=False)) for c in counts]
    indices = np.concatenate([rng.integers(0, F, size=lead)] + body) if n else rng.integers(0, F, size=lead)
    return indptr.astype(np.int32), indices.astype(np.int32)


class Case:
    def __init__(self, model, d, K=20, F=700, N=3001, B=96, n=301, seed=0, flags=0, lead=13):
        from relation_autoencoder_b200.engine import Engine
        self.model, self.N = model, N
        self.eng = Engine(model, K, d, 3, B, F, N, B, flags=flags)
        self.eng.set_params_numpy(_params(model, K, d, F, N, seed))
        self.p = {k: v.detach().double().cpu().numpy() for k, v in self.eng.params.items()}
        rng = np.random.RandomState(seed + 1)
        self.indptr, self.indices = _csr(n, F, seed + 2, lead=lead)
        self.a1 = rng.randint(0, N, n).astype(np.int32)
        self.a2 = rng.randint(0, N, n).astype(np.int32)
        self.a2[::7] = self.a1[::7]                  # args1 == args2
        if n > 4:                                    # true entities at both ends of the id range
            self.a1[1], self.a2[2], self.a1[3], self.a2[4] = 0, 0, N - 1, N - 1

    def rank(self):
        return self.eng.rank_arguments(self.indptr, self.indices, self.a1, self.a2)

    def check(self, r1, r2):
        ip = self.indptr - self.indptr[0]
        ix = self.indices[self.indptr[0]:]
        (lo1, hi1), (lo2, hi2) = R.bracket(self.model, self.p, ip, ix, self.a1, self.a2)
        for r, lo, hi, s in ((r1, lo1, hi1, 1), (r2, lo2, hi2, 2)):
            bad = np.flatnonzero((r < lo) | (r > hi))
            assert bad.size == 0, "slot %d rows %s: gpu %s, bracket %s..%s" % (s, bad[:8], r[bad[:8]], lo[bad[:8]], hi[bad[:8]])
        # the bracket is tight: almost every rank is the float64 rank itself
        f1, f2 = R.ranks(self.model, self.p, ip, ix, self.a1, self.a2)
        assert np.mean(r1 == f1) > 0.97 and np.mean(r2 == f2) > 0.97


@pytest.mark.parametrize("model", ["rescal", "sp", "rescal+sp"])
@pytest.mark.parametrize("d,flags", [(10, 0), (30, 0), (128, 0), (128, FORCE_SIMT), (256, 0)])
def test_ranks_in_float64_bracket(model, d, flags):
    c = Case(model, d, flags=flags, seed=d + flags)
    r1, r2 = c.rank()
    assert r1.dtype == np.int32 and r1.shape == (301,) and r2.shape == (301,)
    assert r1.min() >= 1 and r1.max() <= c.N and r2.min() >= 1 and r2.max() <= c.N
    c.check(r1, r2)


def test_rows_beyond_one_pass_and_repeatable():
    # more rows than one B-row chunk many times over, a K that is not a multiple of 16 and a tiny N (one candidate chunk)
    c = Case("rescal+sp", 64, K=37, N=77, B=128, n=1000, seed=5)
    r1, r2 = c.rank()
    c.check(r1, r2)
    s1, s2 = c.rank()
    assert np.array_equal(r1, s1) and np.array_equal(r2, s2)


def test_true_entity_first_and_last():
    c = Case("rescal+sp", 30, N=1000, n=200, seed=9)
    p = c.eng.params
    p["Ab"][0] = 100.0                     # entity 0 beats everything, entity N-1 loses to everything
    p["Ab"][c.N - 1] = -100.0
    c.p = {k: v.detach().double().cpu().numpy() for k, v in p.items()}
    r1, r2 = c.rank()
    c.check(r1, r2)
    assert r1[1] == 1 and r2[2] == 1
    assert r1[3] == c.N and r2[4] == c.N


def test_zero_rows_and_no_features():
    c = Case("rescal", 30, n=0)
    r1, r2 = c.eng.rank_arguments(np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32))
    assert r1.shape == (0,) and r2.shape == (0,)
    # rows without any feature: ranked under the posterior of Wb alone
    n = 50
    c.indptr, c.indices = np.zeros(n + 1, np.int32), np.zeros(0, np.int32)
    rng = np.random.RandomState(3)
    c.a1, c.a2 = rng.randint(0, c.N, n).astype(np.int32), rng.randint(0, c.N, n).astype(np.int32)
    c.check(*c.rank())


def test_refusals():
    import torch
    from relation_autoencoder_b200.engine import Engine
    eng = Engine("rescal", 8, 16, 2, 32, 50, 40, 32)
    lib, h = eng.lib, eng._h
    buf = torch.zeros(64, dtype=torch.int32, device="cuda")
    ptr = C.c_void_p(buf.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.rae_rank_arguments(h, ptr, ptr, ptr, ptr, 4, ptr, ptr, stream) == ENOTBOUND
    eng.set_params_numpy(_params("rescal", 8, 16, 50, 40, 0))
    null = C.c_void_p(0)
    for args in ((null, ptr, ptr, ptr, 4, ptr, ptr), (ptr, ptr, ptr, null, 4, ptr, ptr), (ptr, ptr, ptr, ptr, 4, null, ptr),
                 (ptr, ptr, ptr, ptr, -1, ptr, ptr)):
        assert lib.rae_rank_arguments(h, *args, stream) == EINVAL
    assert lib.rae_rank_arguments(h, ptr, ptr, ptr, ptr, 0, ptr, ptr, stream) == 0
    with pytest.raises(ValueError, match="entity ids outside"):
        eng.rank_arguments([0, 1], [3], [40], [0])
    with pytest.raises(ValueError, match="feature ids outside"):
        eng.rank_arguments([0, 1], [50], [0], [0])


def test_trained_model(tmp_path, monkeypatch):
    """A model trained by the CUDA driver for a few epochs: Engine.rank_arguments and export --rank-arguments agree with
    the float64 ranker on the checkpoint."""
    from relation_autoencoder_b200 import export as X
    from relation_autoencoder_b200 import induction as I
    from relation_autoencoder_b200 import preprocess as P
    from relation_autoencoder_b200.data import entity_index, unpickle_objects
    from tests.test_export import _line, _write
    train = _write(tmp_path / "train.txt", [_line(i) for i in range(400)])
    held = _write(tmp_path / "held.txt", [_line(i + 1000) for i in range(150)])
    pk = str(tmp_path / "d.pk")
    for b, src in (("train", train), ("dev", held), ("test", held)):
        P.preprocess(src, pk, batch=b, verbose=False)
    monkeypatch.setattr(I, "models_path", str(tmp_path / "products"))
    ind = I.main([pk, "--model-name", "m", "--decoder", "rescal+sp", "--epochs", "3", "--batch-size", "32", "--relations",
                  "10", "--embed-size", "30", "--neg-samples", "5", "--seed", "2"])
    ind._release()
    ckpt = os.path.join(str(tmp_path / "products"), "m.npz")
    ck = I.load_model(ckpt)
    p = {k: np.asarray(v, np.float64) for k, v in ck["params"].items()}
    _, lex, data, _ = unpickle_objects(pk)
    _, _, arg2id = entity_index(data)
    ex = data["test"]
    indptr, indices, _ = X.csr_of(ex, lex.get_feature_space_dimensionality())
    a1 = np.array([arg2id[e.arg1] for e in ex], np.int32)
    a2 = np.array([arg2id[e.arg2] for e in ex], np.int32)
    (lo1, hi1), (lo2, hi2) = R.bracket("rescal+sp", p, indptr, indices, a1, a2)
    ranker, close = X.cuda_ranker(ck)
    try:
        r1, r2 = ranker(indptr, indices, a1, a2)
    finally:
        close()
    assert np.all((lo1 <= r1) & (r1 <= hi1)) and np.all((lo2 <= r2) & (r2 <= hi2))
    s = X.export(ckpt, pk, str(tmp_path / "out"), rank_arguments=True)
    z = np.load(str(tmp_path / "out" / "test.argranks.npz"))
    assert np.array_equal(z["rank1"], r1) and np.array_equal(z["rank2"], r2)
    assert s["sets"]["test"]["arguments"]["rows_ranked"] == len(ex)
    assert s["sets"]["test"]["arguments"]["both"] == X.rank_metrics(np.concatenate([r1, r2]))


def test_readme_run_model():
    """The README run (data-sample.txt, README flags) for 3 epochs through the CUDA engine, then Engine.rank_arguments on
    its test split: within the float64 bracket of the trained parameters, and the training's q is what rae_get_probs
    shows before the call only."""
    from relation_autoencoder_b200 import data as D
    from tests.golden.make_readme_run import run_readme
    idx = D.IndexedDataset.load_npz(os.path.join(os.path.dirname(__file__), "golden", "data_sample_indexed.npz"))
    _, ind = run_readme(idx, None, epochs=3)
    eng = ind.engine
    p = {k: np.asarray(v, np.float64) for k, v in eng.get_params_numpy().items()}
    sp = idx.split["test"]
    ip, ix = np.asarray(sp.indptr), np.asarray(sp.indices)
    a1, a2 = np.asarray(sp.args1, np.int32), np.asarray(sp.args2, np.int32)
    r1, r2 = eng.rank_arguments(ip, ix, a1, a2)
    (lo1, hi1), (lo2, hi2) = R.bracket("rescal+sp", p, ip, ix, a1, a2)
    assert np.all((lo1 <= r1) & (r1 <= hi1)) and np.all((lo2 <= r2) & (r2 <= hi2))
    ind._release()
