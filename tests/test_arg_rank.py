"""Argument ranking, CPU tier: the float64 reference ranker pinned to the oracle's cost, the export's --rank-arguments
path with an injected ranker, and the library's new entry point and kernels."""
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
from tests import arg_rank_ref as R
from tests.test_export import _train, corpora  # noqa: F401  (fixture)


@pytest.mark.parametrize("fix", [False, True])
@pytest.mark.parametrize("model", ["A", "C", "AC"])
def test_candidate_scores_reproduce_the_oracle_cost(model, fix):
    """Positive, negative and entropy terms rebuilt from s1 / s2 give oracle.train_cost (the quirk's slot-2 positive of
    model C from the oracle's own formula)."""
    rng = np.random.RandomState(7)
    F, K, N, d, B, S = 40, 6, 25, 7, 9, 4
    p = O.init_params(rng, model, F, K, N, d)
    for k in ("Ab", "C1", "C2"):
        if k in p:
            p[k] = p[k] + rng.normal(0, 0.3, p[k].shape)
    counts = rng.randint(0, 6, B)
    indptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.int32)
    indices = np.concatenate([np.sort(rng.choice(F, c, replace=False)) for c in counts]).astype(np.int32)
    a1, a2 = rng.randint(0, N, B), rng.randint(0, N, B)
    neg1, neg2 = rng.randint(0, N, (S, B)), rng.randint(0, N, (S, B))
    got = R.cost_from_candidates(model, p, indptr, indices, a1, a2, neg1, neg2, 0.3, fix_sp_quirk=fix)
    if fix:
        want = O.cost_and_grads(model, p, indptr, indices, a1, a2, neg1, neg2, 0.3, fix_sp_quirk=True)[0]
    else:
        want = O.train_cost(model, p, indptr, indices, a1, a2, neg1, neg2, 0.3)[0]
    assert abs(got - want) <= 1e-12 * max(1.0, abs(want))
    # the ranks do not depend on the quirk: it changes only x-independent terms
    assert all(np.array_equal(x, y) for x, y in zip(R.ranks(model, p, indptr, indices, a1, a2, False),
                                                    R.ranks(model, p, indptr, indices, a1, a2, True)))


def test_reference_ranks_by_brute_force():
    rng = np.random.RandomState(1)
    p = O.init_params(rng, "AC", 30, 5, 17, 6)
    p["Ab"] = rng.normal(0, 0.5, 17)
    indptr = np.array([0, 2, 2, 5], np.int32)
    indices = np.array([1, 4, 0, 7, 9], np.int32)
    a1, a2 = np.array([3, 16, 0]), np.array([3, 5, 2])
    r1, r2 = R.ranks("AC", p, indptr, indices, a1, a2)
    f = R.forward("AC", p, indptr, indices, a1, a2)
    for i in range(3):
        for U, t, r in ((f["U1"][i], a1[i], r1[i]), (f["U2"][i], a2[i], r2[i])):
            s = p["A"] @ U + p["Ab"]
            assert r == 1 + sum(1 for x in range(17) if x != t and s[x] > s[t])


def f64_ranker(ck):
    p = {k: np.asarray(v, np.float64) for k, v in ck["params"].items()}
    model = ck["config"]["decoder"]
    calls = []

    def rank(indptr, indices, a1, a2):
        calls.append((np.asarray(indptr).copy(), np.asarray(a1).copy(), np.asarray(a2).copy()))
        r1, r2 = R.ranks(model, p, np.asarray(indptr), np.asarray(indices), np.asarray(a1), np.asarray(a2))
        return r1.astype(np.int32), r2.astype(np.int32)
    rank.calls = calls
    return rank


def _export(tmp_path, ckpt, pk, out, **kw):
    from tests.test_export import f64_labeller
    ck = I.load_model(ckpt)
    return X.export(ckpt, pk, str(tmp_path / out), labeller=f64_labeller(ck), **kw)


def test_export_ranks_and_metrics(tmp_path, monkeypatch, corpora):  # noqa: F811
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")
    ck = I.load_model(ckpt)
    ranker = f64_ranker(ck)
    s = _export(tmp_path, ckpt, corpora["mode2"], "out", tsv=[corpora["new"]], rank_arguments=True, ranker=ranker)
    _, lex, data, _ = D.unpickle_objects(corpora["mode2"])
    _, _, arg2id = D.entity_index(data)
    dm = D.DatasetManager(data, lex, np.random.RandomState(0))
    p = {k: np.asarray(v, np.float64) for k, v in ck["params"].items()}
    for name in ("train", "test"):
        sp = dm.split[name]
        z = np.load(str(tmp_path / "out" / (name + ".argranks.npz")))
        r1, r2 = R.ranks("sp", p, sp.indptr, sp.indices, sp.args1, sp.args2)
        assert np.array_equal(z["rank1"], r1) and np.array_equal(z["rank2"], r2)      # DatasetManager's entity ids
        a = s["sets"][name]["arguments"]
        assert a["rows_ranked"] == len(sp.args1) and a["rows_skipped"] == 0
        both = np.concatenate([r1, r2]).astype(np.float64)
        assert a["both"]["mrr"] == pytest.approx(np.mean(1 / both), rel=1e-15)
        assert a["arg1"]["mean_rank"] == pytest.approx(np.mean(r1), rel=1e-15)
        assert a["arg2"]["hits@3"] == np.mean(r2 <= 3)
        assert set(a["both"]) == {"mrr", "mean_rank", "hits@1", "hits@3", "hits@10"}
    # TSV: PARTIAL and UNKNOWN name entities the dataset never saw -> -1, left out of the metrics
    z = np.load(str(tmp_path / "out" / "new_sentences.argranks.npz"))
    assert list(z["rank1"][[0, 2]]) == [-1, -1] and list(z["rank2"][[0, 2]]) == [-1, -1]
    assert np.all(z["rank1"][[1, 3]] >= 1) and np.all(z["rank2"][[1, 3]] >= 1)
    a = s["sets"]["new_sentences"]["arguments"]
    assert a["rows_ranked"] == 2 and a["rows_skipped"] == 2
    assert a["both"]["mean_rank"] == pytest.approx(np.mean(np.concatenate([z["rank1"][[1, 3]], z["rank2"][[1, 3]]])))
    assert json.load(open(str(tmp_path / "out" / "summary.json")))["sets"]["new_sentences"]["arguments"] == a
    # only the rankable rows reach the ranker
    assert len(ranker.calls[-1][1]) == 2


def test_export_refuses_a_model_of_another_entity_count(tmp_path, monkeypatch, corpora):  # noqa: F811
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")
    z = dict(np.load(ckpt))
    n = z["param_A"].shape[0]
    z["param_A"] = z["param_A"][:-1]
    bad = str(tmp_path / "bad.npz")
    np.savez(bad, **z)

    def never(*a):
        raise AssertionError("no ranking before the checks")
    with pytest.raises(ValueError, match=r"A has %d rows, but the dataset has %d entities" % (n - 1, n)):
        _export(tmp_path, bad, corpora["mode2"], "out", rank_arguments=True, ranker=never)
    assert not os.path.exists(str(tmp_path / "out"))
    # without the flag the entity count is not checked
    _export(tmp_path, bad, corpora["mode2"], "out2")


def test_export_without_the_flag_is_unchanged(tmp_path, monkeypatch, corpora):  # noqa: F811
    """Flag off: no argranks file and no 'arguments' entry; the label files are byte-identical to those of a run with the
    flag, and summary.json equals that run's with the 'arguments' entries removed."""
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")
    ck = I.load_model(ckpt)
    s0 = _export(tmp_path, ckpt, corpora["mode2"], "off", tsv=[corpora["new"]])
    s1 = _export(tmp_path, ckpt, corpora["mode2"], "on", tsv=[corpora["new"]], rank_arguments=True, ranker=f64_ranker(ck))
    off, on = sorted(os.listdir(str(tmp_path / "off"))), sorted(os.listdir(str(tmp_path / "on")))
    assert not any(f.endswith(".argranks.npz") for f in off)
    assert sorted(set(on) - set(off)) == sorted(n + ".argranks.npz" for n in s0["sets"])
    for f in off:
        if f != "summary.json":
            assert open(str(tmp_path / "off" / f), "rb").read() == open(str(tmp_path / "on" / f), "rb").read(), f
    for e in s1["sets"].values():
        del e["arguments"]
    assert s0 == s1
    assert json.load(open(str(tmp_path / "off" / "summary.json"))) == s0


def test_export_command_line_flag(tmp_path, monkeypatch, corpora, capsys):  # noqa: F811
    ckpt = _train(tmp_path, monkeypatch, corpora["mode2"], "m")
    ck = I.load_model(ckpt)
    from tests.test_export import f64_labeller
    monkeypatch.setattr(X, "cuda_labeller", lambda ck_, device=0: (f64_labeller(ck), lambda: None))
    monkeypatch.setattr(X, "cuda_ranker", lambda ck_, device=0: (f64_ranker(ck), lambda: None))
    s = X.main([ckpt, corpora["mode2"], "--out", str(tmp_path / "cli"), "--split", "test", "--rank-arguments"])
    out = capsys.readouterr().out
    assert "argument MRR %.4f" % s["sets"]["test"]["arguments"]["both"]["mrr"] in out
    assert os.path.exists(str(tmp_path / "cli" / "test.argranks.npz"))


def test_library_has_the_entry_point_and_tcgen05_kernels():
    from relation_autoencoder_b200 import _lib as L
    from relation_autoencoder_b200.build import LIB, OBJ
    lib = L.load()
    assert hasattr(lib, "rae_rank_arguments")
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(OBJ, "rae_decoder_tc.o")
    if not (os.path.exists(cuobjdump) and os.path.exists(obj)):
        pytest.skip("cuobjdump or the object files are not available")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    funcs = {}
    for part in sass.split("Function : ")[1:]:
        funcs[part.split("\n", 1)[0].strip()] = part
    names = {n: [f for f in funcs if n in f] for n in ("k_rank_prep_a", "k_rank_queries", "k_tc_rank")}
    assert all(len(v) == 1 for v in names.values()), names
    rank = funcs[names["k_tc_rank"][0]]
    assert "UTCHMMA" in rank and "LDTM" in rank and "UBLKCP" in rank
    assert os.path.exists(LIB)
