"""rae_predict_arguments (top-k epilogue of the tcgen05 ranking GEMM) against the float64 top-k of tests/arg_predict_ref.py.

Scores are fp32-accurate, so per slot a GPU list must be ordered exactly by (score descending, id ascending), each score
within tau of its float64 value, and its set inside the float64 bracket of the k-th score +- 2 tau
(arg_predict_ref.check_fp32_lists).  Bit-exact properties: shorter lists are prefixes of the k = 16 list, reruns are
identical, a slot never reads the argument it predicts, and the lists do not depend on how the candidates were split."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import pytest

from tests import arg_predict_ref as P
from tests import arg_rank_ref as R
from tests.test_gpu_arg_rank import FORCE_SIMT, Case, _params

pytestmark = pytest.mark.gpu

EINVAL, ENOTBOUND = -1, -3


def _ref(c):
    ip = c.indptr - c.indptr[0]
    ix = c.indices[c.indptr[0]:]
    return P.slot_scores(c.model, c.p, ip, ix, c.a1, c.a2)


def _predict(c, k):
    return c.eng.predict_arguments(c.indptr, c.indices, c.a1, c.a2, k)


@pytest.mark.parametrize("model", ["rescal", "sp", "rescal+sp"])
@pytest.mark.parametrize("d,flags", [(10, 0), (30, 0), (128, 0), (128, FORCE_SIMT), (256, 0)])
def test_lists_in_float64_bracket(model, d, flags):
    c = Case(model, d, flags=flags, seed=d + flags)
    # true arguments inside the top 16 for a third of the rows per slot.  Slot 1 never reads args1, so args1 of rows
    # 0 mod 3 can be taken from slot 1's float64 top 16 without changing it (slot 2 likewise on rows 1 mod 3).
    (S1, _), (S2, _) = _ref(c)
    rows = np.arange(len(c.a1))
    for S, a, m in ((S1, c.a1, 0), (S2, c.a2, 1)):
        top = P.topk(S, 16)[0]
        sel = rows[rows % 3 == m]
        a[sel] = top[sel, (sel // 3) % 16]
    (S1, tau1), (S2, tau2) = _ref(c)
    out = _predict(c, 16)
    i1, s1, i2, s2 = out
    assert i1.dtype == np.int32 and s1.dtype == np.float32 and i1.shape == (301, 16)
    P.check_fp32_lists(i1, s1, S1, tau1, 16)
    P.check_fp32_lists(i2, s2, S2, tau2, 16)
    for k in (1, 3, 10):                       # k rounds up to a top-kt list: its first k entries are the top-k list
        short = _predict(c, k)
        for a, b in zip(short, out):
            assert np.array_equal(a, b[:, :k])
    again = _predict(c, 16)
    assert all(np.array_equal(a, b) for a, b in zip(out, again))
    # agreement with the ranking kernel: where rank r <= 16 and no other float64 score is within 2 tau of the true one,
    # the true entity sits at position r - 1
    r1, r2 = c.eng.rank_arguments(c.indptr, c.indices, c.a1, c.a2)
    for ids, S, tau, r, t in ((i1, S1, tau1, r1, c.a1), (i2, S2, tau2, r2, c.a2)):
        st = S[np.arange(len(t)), t]
        near = (np.abs(S - st[:, None]) <= 2 * tau[:, None]).sum(1) > 1
        sel = np.flatnonzero((r <= 16) & ~near)
        assert sel.size > 50
        assert np.array_equal(ids[sel, r[sel] - 1], t[sel])


@pytest.mark.parametrize("model,d", [("rescal", 30), ("sp", 30), ("rescal+sp", 128), ("rescal+sp", 10)])
def test_slot_never_reads_the_argument_it_predicts(model, d):
    c = Case(model, d, seed=40 + d)
    base = _predict(c, 8)
    rng = np.random.RandomState(3)
    a1, a2 = c.a1.copy(), c.a2.copy()
    c.a1 = ((a1 + rng.randint(1, c.N, a1.size)) % c.N).astype(np.int32)
    x1, y1, _, _ = _predict(c, 8)
    assert np.array_equal(x1, base[0]) and np.array_equal(y1, base[1])
    c.a1, c.a2 = a1, ((a2 + rng.randint(1, c.N, a2.size)) % c.N).astype(np.int32)
    _, _, x2, y2 = _predict(c, 8)
    assert np.array_equal(x2, base[2]) and np.array_equal(y2, base[3])


def test_lists_do_not_depend_on_the_candidate_split():
    """The first B rows alone (2 query tiles: the candidates are split over several CTAs) equal the same rows predicted in
    front of about 10 k further rows (more query tiles than SMs: no split)."""
    B = 96
    c = Case("rescal+sp", 128, N=5003, B=B, n=B + 10000, seed=11)
    full = _predict(c, 10)
    ip, ix, a1, a2 = c.indptr, c.indices, c.a1, c.a2
    c.indptr, c.a1, c.a2 = ip[:B + 1], a1[:B], a2[:B]
    alone = _predict(c, 10)
    for a, b in zip(alone, full):
        assert np.array_equal(a, b[:B])
    c.indptr, c.a1, c.a2 = ip, a1, a2
    (S1, tau1), (S2, tau2) = _ref_rows(c, B)
    P.check_fp32_lists(alone[0], alone[1], S1, tau1, 10)
    P.check_fp32_lists(alone[2], alone[3], S2, tau2, 10)


def _ref_rows(c, m, lo=0):
    ip = c.indptr[lo:m + 1] - c.indptr[lo]
    ix = c.indices[c.indptr[lo]:]
    return P.slot_scores(c.model, c.p, ip, ix, c.a1[lo:m], c.a2[lo:m])


def test_rows_beyond_one_pass():
    """More rows than one ranking pass (131 040 rows at B = 96): the second pass's lists land at their own rows (output
    offset row0 * k, partial-list workspace reused), equal to those rows predicted alone and inside the float64 bracket."""
    B, tail = 96, 300
    n = (131072 // B) * B + tail
    c = Case("rescal+sp", 30, N=3001, B=B, n=n, seed=21)
    full = _predict(c, 5)
    lo = n - tail - 20                               # the last 20 rows of the first pass and the whole second pass
    ip, a1, a2 = c.indptr, c.a1, c.a2
    c.indptr, c.a1, c.a2 = ip[lo:], a1[lo:], a2[lo:]
    alone = _predict(c, 5)
    for a, b in zip(alone, full):
        assert np.array_equal(a, b[lo:])
    c.indptr, c.a1, c.a2 = ip, a1, a2
    (S1, tau1), (S2, tau2) = _ref_rows(c, n, lo)
    P.check_fp32_lists(full[0][lo:], full[1][lo:], S1, tau1, 5)
    P.check_fp32_lists(full[2][lo:], full[3][lo:], S2, tau2, 5)
    (S1, tau1), _ = _ref_rows(c, 40)                 # the first rows of the first pass
    P.check_fp32_lists(full[0][:40], full[1][:40], S1, tau1, 5)


def test_exact_ties_ordered_by_id_across_threads_groups_and_splits():
    """Entities with identical rows of A and Ab score identically.  A tied group at the top of every list, placed in the same
    epilogue thread (columns 128 apart), in the other column group (64 apart) and in other candidate ranges (N >= 2048 and
    few rows: the candidates are split), must come out in ascending id order, and k = 3 must keep its three lowest ids."""
    c = Case("rescal+sp", 128, N=5003, n=50, seed=13)
    src = 700
    group = [src, src - 640, src + 64, src + 128, src + 2048, src + 4096]
    A, Ab = c.eng.params["A"], c.eng.params["Ab"]
    Ab[src] = 50.0                                     # far above every other score
    for x in group[1:]:
        A[x] = A[src]
        Ab[x] = Ab[src]
    want = sorted(group)
    for k in (16, 3):
        i1, s1, i2, s2 = _predict(c, k)
        m = min(k, len(group))
        for ids, sc in ((i1, s1), (i2, s2)):
            assert np.all(ids[:, :m] == np.array(want[:m])), ids[:3]
            assert np.all(sc[:, :m] == sc[:, :1])


def test_zero_rows_no_features_and_k_equal_n():
    c = Case("rescal", 30, n=0)
    out = c.eng.predict_arguments(np.zeros(1, np.int32), np.zeros(0, np.int32), np.zeros(0, np.int32),
                                  np.zeros(0, np.int32), 4)
    assert all(o.shape == (0, 4) for o in out)
    n = 50
    c.indptr, c.indices = np.zeros(n + 1, np.int32), np.zeros(0, np.int32)
    rng = np.random.RandomState(3)
    c.a1, c.a2 = rng.randint(0, c.N, n).astype(np.int32), rng.randint(0, c.N, n).astype(np.int32)
    (S1, tau1), (S2, tau2) = _ref(c)
    i1, s1, i2, s2 = _predict(c, 5)
    P.check_fp32_lists(i1, s1, S1, tau1, 5)
    P.check_fp32_lists(i2, s2, S2, tau2, 5)
    # N < 128 (one candidate chunk, -inf padding rows) with k = N: every entity listed once
    c = Case("rescal+sp", 30, N=13, n=40, seed=4)
    (S1, tau1), (S2, tau2) = _ref(c)
    i1, s1, i2, s2 = _predict(c, 13)
    P.check_fp32_lists(i1, s1, S1, tau1, 13)
    P.check_fp32_lists(i2, s2, S2, tau2, 13)
    assert np.all(np.sort(i1, 1) == np.arange(13)) and np.all(np.isfinite(s1)) and np.all(np.isfinite(s2))


def test_refusals():
    import torch
    from relation_autoencoder_b200.engine import Engine
    eng = Engine("rescal", 8, 16, 2, 32, 50, 40, 32)
    lib, h = eng.lib, eng._h
    buf = torch.zeros(256, dtype=torch.int32, device="cuda")
    ptr = C.c_void_p(buf.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.rae_predict_arguments(h, ptr, ptr, ptr, ptr, 4, 2, ptr, ptr, ptr, ptr, stream) == ENOTBOUND
    eng.set_params_numpy(_params("rescal", 8, 16, 50, 40, 0))
    null = C.c_void_p(0)
    for i in (0, 1, 2, 3, 4, 5, 6, 7):                  # each pointer argument null in turn
        a = [ptr] * 8
        a[i] = null
        assert lib.rae_predict_arguments(h, a[0], a[1], a[2], a[3], 4, 2, a[4], a[5], a[6], a[7], stream) == EINVAL
    for n, k in ((-1, 2), (4, 0), (4, 17), (4, -3)):
        assert lib.rae_predict_arguments(h, ptr, ptr, ptr, ptr, n, k, ptr, ptr, ptr, ptr, stream) == EINVAL
    assert lib.rae_predict_arguments(h, ptr, ptr, ptr, ptr, 0, 2, ptr, ptr, ptr, ptr, stream) == 0
    small = Engine("rescal", 8, 16, 2, 32, 50, 12, 32)
    small.set_params_numpy(_params("rescal", 8, 16, 50, 12, 0))
    assert small.lib.rae_predict_arguments(small._h, ptr, ptr, ptr, ptr, 4, 13, ptr, ptr, ptr, ptr, stream) == EINVAL
    from relation_autoencoder_b200 import _lib as L
    emit = Engine("rescal", 8, 16, 2, 32, 50, 40, 32, flags=L.RAE_FLAG_EMIT_ONLY)
    emit.set_params_numpy(_params("rescal", 8, 16, 50, 40, 0))
    assert emit.lib.rae_predict_arguments(emit._h, ptr, ptr, ptr, ptr, 4, 2, ptr, ptr, ptr, ptr, stream) == EINVAL
    assert b"emit-only" in emit.lib.rae_last_error(emit._h)
    with pytest.raises(ValueError, match="outside"):
        small.predict_arguments([0, 1], [3], [0], [0], 13)
    with pytest.raises(ValueError, match="entity ids outside"):
        eng.predict_arguments([0, 1], [3], [40], [0], 2)
    with pytest.raises(ValueError, match="feature ids outside"):
        eng.predict_arguments([0, 1], [50], [0], [0], 2)


def test_trained_model(tmp_path, monkeypatch):
    """A model trained by the CUDA driver: Engine.predict_arguments and export --predict-arguments agree with each other
    and with the float64 reference on the checkpoint."""
    from relation_autoencoder_b200 import export as X
    from relation_autoencoder_b200 import induction as I
    from relation_autoencoder_b200 import preprocess as PP
    from relation_autoencoder_b200.data import entity_index, unpickle_objects
    from tests.test_export import _line, _write
    train = _write(tmp_path / "train.txt", [_line(i) for i in range(400)])
    held = _write(tmp_path / "held.txt", [_line(i + 1000) for i in range(150)])
    pk = str(tmp_path / "d.pk")
    for b, src in (("train", train), ("dev", held), ("test", held)):
        PP.preprocess(src, pk, batch=b, verbose=False)
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
    k = min(5, len(arg2id))
    predictor, close = X.cuda_predictor(ck)
    try:
        i1, s1, i2, s2 = predictor(indptr, indices, a1, a2, k)
    finally:
        close()
    (S1, tau1), (S2, tau2) = P.slot_scores("rescal+sp", p, indptr, indices, a1, a2)
    P.check_fp32_lists(i1, s1, S1, tau1, k)
    P.check_fp32_lists(i2, s2, S2, tau2, k)
    s = X.export(ckpt, pk, str(tmp_path / "out"), predict_arguments=k)
    z = np.load(str(tmp_path / "out" / "test.argpreds.npz"))
    assert np.array_equal(z["ids1"], i1) and np.array_equal(z["ids2"], i2)
    assert np.array_equal(z["scores1"], s1) and np.array_equal(z["scores2"], s2)
    assert s["sets"]["test"]["predictions"]["arg1"]["rows_predicted"] == len(ex)
    r1, _ = R.ranks("rescal+sp", p, indptr, indices, a1, a2)
    assert s["sets"]["test"]["predictions"]["arg1"]["share_in_list"] == pytest.approx(np.mean(r1 <= k), abs=0.05)
