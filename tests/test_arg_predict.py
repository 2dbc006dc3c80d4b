"""Argument prediction, CPU tier: the float64 top-k reference, its independence of the argument it predicts, the export's
--predict-arguments path with an injected predictor, and the library's new entry point and kernels."""
from __future__ import annotations

import json
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import rae_oracle as O
from relation_autoencoder_b200 import data as D
from relation_autoencoder_b200 import export as X
from relation_autoencoder_b200 import induction as I
from tests import arg_predict_ref as P
from tests import arg_rank_ref as R
from tests.test_export import _line, _train, _write, corpora, f64_labeller  # noqa: F401  (fixture)


def _case(model, seed, F=30, K=5, N=17, d=6, n=7):
    rng = np.random.RandomState(seed)
    p = O.init_params(rng, model, F, K, N, d)
    for k in ("Ab", "C1", "C2"):
        if k in p:
            p[k] = p[k] + rng.normal(0, 0.3, p[k].shape)
    counts = rng.randint(0, 5, n)
    indptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    indices = np.concatenate([np.sort(rng.choice(F, c, replace=False)) for c in counts] + [[]]).astype(np.int32)
    return p, indptr, indices, rng.randint(0, N, n), rng.randint(0, N, n)


def test_reference_top_k_by_brute_force_with_ties():
    p, indptr, indices, a1, a2 = _case("AC", 1)
    for src, dst in ((2, 5), (2, 11), (9, 0)):       # exact ties: equal rows of A and Ab, ordered by ascending id
        p["A"][dst], p["Ab"][dst] = p["A"][src], p["Ab"][src]
    f = R.forward("AC", p, indptr, indices, a1, a2)
    for k in (1, 4, 17):
        i1, s1, i2, s2 = P.predictions("AC", p, indptr, indices, a1, a2, k)
        for ids, sc, U in ((i1, s1, f["U1"]), (i2, s2, f["U2"])):
            S = P.all_scores(p, U)
            for i in range(len(a1)):
                assert np.allclose(S[i], p["A"] @ U[i] + p["Ab"], rtol=0, atol=1e-12)
                want = sorted(range(17), key=lambda x: (-S[i, x], x))[:k]
                assert list(ids[i]) == want and np.array_equal(sc[i], S[i, want])
    S = P.all_scores(p, f["U1"])
    assert S[0, 2] == S[0, 5] == S[0, 11]
    order = list(P.topk(S, 17)[0][0])
    assert order.index(2) < order.index(5) < order.index(11)


@pytest.mark.parametrize("fix", [False, True])
@pytest.mark.parametrize("model", ["A", "C", "AC"])
def test_reference_slot_never_reads_the_argument_it_predicts(model, fix):
    p, indptr, indices, a1, a2 = _case(model, 3)
    i1, s1, i2, s2 = P.predictions(model, p, indptr, indices, a1, a2, 5, fix)
    b1, b2 = (a1 + 3) % 17, (a2 + 5) % 17
    j1, t1, _, _ = P.predictions(model, p, indptr, indices, b1, a2, 5, fix)       # slot 1 predicts args1
    _, _, j2, t2 = P.predictions(model, p, indptr, indices, a1, b2, 5, fix)       # slot 2 predicts args2
    assert np.array_equal(i1, j1) and np.array_equal(s1, t1)
    assert np.array_equal(i2, j2) and np.array_equal(s2, t2)
    if model == "C":                                                            # model C reads neither argument
        k1, u1, k2, u2 = P.predictions(model, p, indptr, indices, b1, b2, 5, fix)
        assert np.array_equal(i1, k1) and np.array_equal(i2, k2) and np.array_equal(s2, u2)


def f64_predictor(ck):
    p = {k: np.asarray(v, np.float64) for k, v in ck["params"].items()}
    model = ck["config"]["decoder"]
    calls = []

    def predict(indptr, indices, a1, a2, k):
        calls.append((np.asarray(a1).copy(), np.asarray(a2).copy(), k))
        i1, s1, i2, s2 = P.predictions(model, p, np.asarray(indptr), np.asarray(indices), np.asarray(a1), np.asarray(a2), k)
        return i1.astype(np.int32), s1.astype(np.float32), i2.astype(np.int32), s2.astype(np.float32)
    predict.calls = calls
    return predict


def _export(tmp_path, ckpt, pk, out, **kw):
    ck = I.load_model(ckpt)
    return X.export(ckpt, pk, str(tmp_path / out), labeller=f64_labeller(ck), **kw)


# unseen arg2, known arg1 (and the reverse): predicted in the slot whose conditioning argument is known
HALF1 = _line(3).replace("Beta3 Inc", "Nowhere Ltd")
HALF2 = _line(8).replace("Alpha1 Corp", "Nobody Co")


def test_export_predictions_files_and_summary(tmp_path, monkeypatch, corpora):  # noqa: F811
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")
    ck = I.load_model(ckpt)
    pred = f64_predictor(ck)
    half = _write(tmp_path / "half.txt", [HALF1, HALF2])
    k = 3
    s = _export(tmp_path, ckpt, corpora["mode2"], "out", tsv=[corpora["new"], half], predict_arguments=k, predictor=pred)
    _, lex, data, _ = D.unpickle_objects(corpora["mode2"])
    _, id2arg, arg2id = D.entity_index(data)
    p = {kk: np.asarray(v, np.float64) for kk, v in ck["params"].items()}
    F = lex.get_feature_space_dimensionality()
    out = tmp_path / "out"
    # a split: every row predicted in both slots, against the float64 reference on DatasetManager's entity ids
    dm = D.DatasetManager(data, lex, np.random.RandomState(0))
    sp = dm.split["test"]
    z = np.load(str(out / "test.argpreds.npz"))
    i1, s1, i2, s2 = P.predictions("sp", p, sp.indptr, sp.indices, sp.args1, sp.args2, k)
    assert np.array_equal(z["ids1"], i1) and np.array_equal(z["ids2"], i2)
    assert np.array_equal(z["scores1"], s1.astype(np.float32)) and np.array_equal(z["scores2"], s2.astype(np.float32))
    lab = np.load(str(out / "test.labels.npz"))["ids"][:, 0]
    rows = open(str(out / "test.argpreds.tsv"), encoding="utf-8").read().splitlines()
    assert rows[0].split("\t") == ["index", "arg1", "arg2", "trigger", "relation", "predicted_arg1", "predicted_arg2",
                                   "position1", "position2"]
    ex = data["test"]
    pos1 = []
    for i, line in enumerate(rows[1:]):
        c = line.split("\t")
        assert c[:5] == [str(i), ex[i].arg1, ex[i].arg2, ex[i].trigger, str(lab[i])]
        assert c[5] == " ".join("%s:%.6g" % (id2arg[x], v) for x, v in zip(z["ids1"][i], z["scores1"][i]))
        assert c[6] == " ".join("%s:%.6g" % (id2arg[x], v) for x, v in zip(z["ids2"][i], z["scores2"][i]))
        want1 = list(z["ids1"][i]).index(sp.args1[i]) + 1 if sp.args1[i] in z["ids1"][i] else 0
        want2 = list(z["ids2"][i]).index(sp.args2[i]) + 1 if sp.args2[i] in z["ids2"][i] else 0
        assert (int(c[7]), int(c[8])) == (want1, want2)
        pos1.append(want1)
    e = s["sets"]["test"]["predictions"]
    assert e["k"] == k and e["arg1"]["rows_predicted"] == len(ex) == e["arg2"]["rows_predicted"]
    assert e["arg1"]["rows_with_known_argument"] == len(ex)
    assert e["arg1"]["share_in_list"] == pytest.approx(np.mean(np.array(pos1) > 0), rel=1e-15)
    assert json.load(open(str(out / "summary.json")))["sets"]["test"]["predictions"] == e
    # new sentences: PARTIAL and UNKNOWN know neither entity -> not sent, -1 / NaN in both slots
    z = np.load(str(out / "new_sentences.argpreds.npz"))
    for r in (0, 2):
        assert np.all(z["ids1"][r] == -1) and np.all(z["ids2"][r] == -1)
        assert np.all(np.isnan(z["scores1"][r])) and np.all(np.isnan(z["scores2"][r]))
    assert np.all(z["ids1"][[1, 3]] >= 0) and np.all(z["ids2"][[1, 3]] >= 0)
    c = open(str(out / "new_sentences.argpreds.tsv"), encoding="utf-8").read().splitlines()[1].split("\t")
    assert c[5:] == ["", "", "-1", "-1"]
    e = s["sets"]["new_sentences"]["predictions"]
    assert e["arg1"]["rows_predicted"] == 2 and e["arg2"]["rows_predicted"] == 2
    assert len(pred.calls[-2][0]) == 2                         # only the rows with a known entity reach the predictor
    # one unknown entity: the slot that predicts it is still predicted (from the known one), the other is not
    z = np.load(str(out / "half.argpreds.npz"))
    ex, _ = X.featurize(half, lex, D.unpickle_objects(corpora["mode2"])[0])
    indptr, indices, _ = X.csr_of(ex, F)
    known1, known2 = arg2id[ex[0].arg1], arg2id[ex[1].arg2]
    w1, v1, w2, v2 = P.predictions("sp", p, indptr, indices, np.array([known1, 0]), np.array([0, known2]), k)
    assert np.array_equal(z["ids2"][0], w2[0]) and np.all(z["ids1"][0] == -1)   # row 0: arg2 unseen, predicted from arg1
    assert np.array_equal(z["ids1"][1], w1[1]) and np.all(z["ids2"][1] == -1)   # row 1: arg1 unseen, predicted from arg2
    assert np.all(np.isnan(z["scores1"][0])) and np.array_equal(z["scores2"][0], v2[0].astype(np.float32))
    c = [ln.split("\t") for ln in open(str(out / "half.argpreds.tsv"), encoding="utf-8").read().splitlines()[1:]]
    assert c[0][5] == "" and c[0][6] != "" and c[0][7:] == ["-1", "-1"]
    assert c[1][5] != "" and c[1][6] == "" and c[1][7:] == ["-1", "-1"]
    e = s["sets"]["half"]["predictions"]
    assert e["arg1"] == {"rows_predicted": 1, "rows_with_known_argument": 0, "share_in_list": None}
    assert e["arg2"]["rows_predicted"] == 1
    assert list(pred.calls[-1][0]) == [known1, 0] and list(pred.calls[-1][1]) == [0, known2]   # unknown ids sent as 0


def test_export_without_the_flag_is_unchanged(tmp_path, monkeypatch, corpora):  # noqa: F811
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")
    ck = I.load_model(ckpt)
    s0 = _export(tmp_path, ckpt, corpora["mode2"], "off", tsv=[corpora["new"]])
    s1 = _export(tmp_path, ckpt, corpora["mode2"], "on", tsv=[corpora["new"]], predict_arguments=2,
                 predictor=f64_predictor(ck))
    off, on = sorted(os.listdir(str(tmp_path / "off"))), sorted(os.listdir(str(tmp_path / "on")))
    assert sorted(set(on) - set(off)) == sorted(n + e for n in s0["sets"] for e in (".argpreds.npz", ".argpreds.tsv"))
    for f in off:
        if f != "summary.json":
            assert open(str(tmp_path / "off" / f), "rb").read() == open(str(tmp_path / "on" / f), "rb").read(), f
    for e in s1["sets"].values():
        del e["predictions"]
    assert s0 == s1


def test_export_refusals(tmp_path, monkeypatch, corpora):  # noqa: F811
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")

    def never(*a):
        raise AssertionError("no prediction before the checks")
    n = I.load_model(ckpt)["params"]["A"].shape[0]
    assert n < 16
    for k in (-1, 17, n + 1):
        with pytest.raises(ValueError, match=r"--predict-arguments %d is outside \[1, min\(N, 16\)\] = \[1, %d\]" % (k, n)):
            _export(tmp_path, ckpt, corpora["mode2"], "out", predict_arguments=k, predictor=never)
    _export(tmp_path, ckpt, corpora["mode2"], "ok", predict_arguments=n, predictor=f64_predictor(I.load_model(ckpt)))
    z = dict(np.load(ckpt))
    z["param_A"] = z["param_A"][:-1]
    bad = str(tmp_path / "bad.npz")
    np.savez(bad, **z)
    with pytest.raises(ValueError, match=r"A has %d rows, but the dataset has %d entities" % (n - 1, n)):
        _export(tmp_path, bad, corpora["mode2"], "out", predict_arguments=2, predictor=never)
    assert not os.path.exists(str(tmp_path / "out"))


def test_export_command_line_flag(tmp_path, monkeypatch, corpora):  # noqa: F811
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")
    ck = I.load_model(ckpt)
    monkeypatch.setattr(X, "cuda_labeller", lambda ck_, device=0: (f64_labeller(ck), lambda: None))
    monkeypatch.setattr(X, "cuda_predictor", lambda ck_, device=0: (f64_predictor(ck), lambda: None))
    for bad in ("0", "17"):
        with pytest.raises((SystemExit, ValueError)):
            X.main([ckpt, corpora["mode2"], "--out", str(tmp_path / "no"), "--predict-arguments", bad])
    assert not os.path.exists(str(tmp_path / "no"))
    s = X.main([ckpt, corpora["mode2"], "--out", str(tmp_path / "cli"), "--split", "test", "--predict-arguments", "4"])
    assert s["sets"]["test"]["predictions"]["k"] == 4
    z = np.load(str(tmp_path / "cli" / "test.argpreds.npz"))
    assert z["ids1"].shape == (len(D.unpickle_objects(corpora["mode2"])[2]["test"]), 4)
    assert os.path.exists(str(tmp_path / "cli" / "test.argpreds.tsv"))


def test_library_has_the_entry_point_and_tcgen05_kernels():
    from relation_autoencoder_b200 import _lib as L
    from relation_autoencoder_b200.build import LIB, OBJ
    lib = L.load()
    assert hasattr(lib, "rae_predict_arguments")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(OBJ, "rae_decoder_tc.o")
    if not (os.path.exists(cuobjdump) and os.path.exists(obj)):
        pytest.skip("cuobjdump or the object files are not available")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    funcs = {}
    for part in sass.split("Function : ")[1:]:
        funcs[part.split("\n", 1)[0].strip()] = part
    for kt in (1, 2, 4, 8, 16):
        pred = [f for f in funcs if "k_tc_predictILi%dE" % kt in f]
        merge = [f for f in funcs if "k_predict_mergeILi%dE" % kt in f]
        assert len(pred) == 1 and len(merge) == 1, (pred, merge)
        body = funcs[pred[0]]
        assert "UTCHMMA" in body and "LDTM" in body and "UBLKCP" in body
        assert "STL" not in body and "LDL" not in body              # no local-memory spills
    assert os.path.exists(LIB)
