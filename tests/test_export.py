"""Export of the induced relations (relation_autoencoder_b200/export.py) and the frozen-lexicon featuriser.

CPU: models trained with the float64 oracle backend are exported through a float64 top-k labeller (scores of
``oracle.rae_oracle.encoder_scores_fast``, the function the oracle driver labels with), so the driver's logged B-cubed is
reproduced exactly.  GPU: a model trained through the CUDA engine is exported through ``rae_label_topk``."""
from __future__ import annotations

import hashlib
import json
import os
from collections import Counter

import numpy as np
import pytest

from oracle import rae_oracle as O
from relation_autoencoder_b200 import data as D
from relation_autoencoder_b200 import evaluation as E
from relation_autoencoder_b200 import export as X
from relation_autoencoder_b200 import induction as I
from relation_autoencoder_b200 import preprocess as P
from tests.oracle_backend import oracle_backend

N_TRAIN, BATCH = 43, 10            # a tail of 3 rows the driver never labels


def _line(i, rel=None):
    rel = ("/r/%d" % (i % 3) if i % 4 else "") if rel is None else rel
    return ("->nsubj->word%d->dobj->\tAlpha%d Corp\tBeta%d Inc\tORG-ORG\tTRIGGER:word%d\t./d%d.xml\tAlpha%d Corp likes word%d "
            "of Beta%d Inc today .\tNNP NNP VBZ NN IN NNP NNP NN .\t%s\n" % (i % 5, i % 7, i % 6, i % 5, i, i % 7, i % 5, i % 6, rel))


# every string unseen: its row has no features
UNKNOWN = ("->qq->zz->\tUnk1 Thing\tUnk2 Stuff\tAAA-BBB\tTRIGGER:nothingness\t./x.xml\tUnk1 Thing zork Unk2 Stuff\t"
           "QQ QQ QQ QQ QQ\t/r/1\n")
# unseen entities and words, known trigger, types and path
PARTIAL = ("->nsubj->word1->dobj->\tGamma Ltd\tDelta Co\tORG-ORG\tTRIGGER:word1\t./y.xml\tGamma Ltd likes word1 of Delta Co "
           "today .\tNNP NNP VBZ NN IN NNP NNP NN .\t\n")


def _write(path, lines):
    path.write_text("".join(lines), encoding="utf-8")
    return str(path)


def f64_labeller(ck):
    """Top-k of the float64 scores: score descending, then relation id ascending; softmax probabilities."""
    W = np.asarray(ck['params']['W'], dtype=np.float64)
    Wb = np.asarray(ck['params']['Wb'], dtype=np.float64)

    def lab(indptr, indices, k):
        z = O.encoder_scores_fast(W, Wb, np.asarray(indptr), np.asarray(indices))
        ids = np.argsort(-z, axis=1, kind='stable')[:, :k]
        q, _ = O.softmax_rows(z)
        return ids.astype(np.int32), np.take_along_axis(q, ids, axis=1).astype(np.float32)
    return lab


def _train(tmp_path, monkeypatch, pk, name, backend=oracle_backend, relations=4):
    monkeypatch.setattr(I, "models_path", str(tmp_path / "products"))
    ind = I.main([pk, "--model-name", name, "--decoder", "sp", "--epochs", "2", "--batch-size", str(BATCH), "--relations",
                  str(relations), "--embed-size", "6", "--neg-samples", "3", "--seed", "2"], backend=backend)
    if backend is None:
        ind._release()
    return os.path.join(str(tmp_path / "products"), name + ".npz")


@pytest.fixture
def corpora(tmp_path):
    train = _write(tmp_path / "train.txt", [_line(i) for i in range(N_TRAIN)])
    held = _write(tmp_path / "held.txt", [_line(i + 100) for i in range(23)])
    mode1 = str(tmp_path / "mode1.pk")
    P.preprocess(train, mode1, batch='train', verbose=False)
    mode2 = str(tmp_path / "mode2.pk")
    for b, src in (('train', train), ('dev', held), ('test', held)):
        P.preprocess(src, mode2, batch=b, verbose=False)
    new = _write(tmp_path / "new_sentences.txt", [PARTIAL, _line(3), UNKNOWN, _line(7)])
    return dict(train=train, held=held, mode1=mode1, mode2=mode2, new=new)


# ----------------------------------------------------------------------------------------------------------------------
# frozen featuriser
# ----------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("threshold", [0, 1])
def test_featurize_reproduces_stored_examples_and_leaves_the_lexicon_alone(tmp_path, threshold):
    train = _write(tmp_path / "c.txt", [_line(i) for i in range(N_TRAIN)])
    pk = str(tmp_path / "c.pk")
    P.preprocess(train, pk, batch='train', threshold=threshold, verbose=False)
    before = hashlib.sha256(open(pk, 'rb').read()).hexdigest()
    feats, lex, data, gold = D.unpickle_objects(pk)
    F = lex.get_feature_space_dimensionality()
    ex, g = P.featurize(train, lex, feats)
    assert len(ex) == N_TRAIN and g == gold['train']
    for a, b in zip(ex, data['train']):
        assert sorted(set(a.features)) == sorted(set(b.features))
        assert (a.arg1, a.arg2, a.trigger) == (b.arg1, b.arg2, b.trigger)
    assert lex.get_feature_space_dimensionality() == F

    new = _write(tmp_path / "n.txt", [PARTIAL, UNKNOWN])
    ex, g = P.featurize(new, lex, [f.__name__ for f in feats])
    known = {lex.str2IdPruned[s] for s in ('trigger#word1', 'entityTypes#ORG-ORG', 'entity1Type#ORG', 'entity2Type#ORG',
                                           'lexicalPattern#word1') if s in lex.str2IdPruned}
    assert known and known <= set(ex[0].features)
    assert set(ex[0].features) <= set(range(F))
    assert not any(s in lex.str2IdPruned for s in ('arg1_lower#gamma ltd', 'arg2_lower#delta co'))
    assert ex[1].features == [] and g[1] == ['/r/1'] and g[0] == ['']
    indptr, indices, n_features = X.csr_of(ex, F)
    assert n_features[1] == 0 and indptr[2] == indptr[1] and n_features[0] == len(set(ex[0].features))
    assert lex.get_feature_space_dimensionality() == F
    assert hashlib.sha256(open(pk, 'rb').read()).hexdigest() == before


def test_featurize_refuses_an_unknown_extractor(tmp_path):
    train = _write(tmp_path / "c.txt", [_line(0)])
    pk = str(tmp_path / "c.pk")
    P.preprocess(train, pk, batch='train', verbose=False)
    feats, lex, _, _ = D.unpickle_objects(pk)
    with pytest.raises(ValueError, match="skiptrigrams"):
        P.featurize(train, lex, [f.__name__ for f in feats] + ['skiptrigrams'])


# ----------------------------------------------------------------------------------------------------------------------
# end to end (float64 labeller)
# ----------------------------------------------------------------------------------------------------------------------
def _read_tsv(path):
    with open(path, encoding='utf-8') as f:
        rows = [ln.rstrip('\n').split('\t') for ln in f]
    return rows[0], rows[1:]


def _check_set(out, name, examples, gold, lab_out, k):
    ids, probs = lab_out
    z = np.load(os.path.join(out, name + '.labels.npz'))
    assert np.array_equal(z['ids'], ids) and np.array_equal(z['probs'], probs)
    assert z['ids'].dtype == np.int32 and z['probs'].dtype == np.float32 and z['n_features'].dtype == np.int32
    n = len(examples)
    assert z['ids'].shape == (n, k) and z['n_features'].shape == (n,)
    head, rows = _read_tsv(os.path.join(out, name + '.examples.tsv'))
    assert head == ['index', 'arg1', 'arg2', 'trigger', 'gold', 'relation', 'prob', 'n_features', 'topk']
    assert len(rows) == n
    assert [int(r[5]) for r in rows] == ids[:, 0].tolist()
    assert [int(r[7]) for r in rows] == z['n_features'].tolist()
    assert [[int(p.split(':')[0]) for p in r[8].split()] for r in rows] == ids.tolist()
    assert [r[4] for r in rows] == [gold[i][0] for i in range(n)]
    head, crow = _read_tsv(os.path.join(out, name + '.clusters.tsv'))
    assert head == ['relation', 'size', 'mean_prob', 'triggers', 'gold']
    sizes = [int(r[1]) for r in crow]
    assert sum(sizes) == n and sizes == sorted(sizes, reverse=True)
    for r in crow:
        members = np.flatnonzero(ids[:, 0] == int(r[0]))
        assert len(members) == int(r[1])
        want = Counter(examples[i].trigger for i in members)
        got = {t.rsplit(':', 1)[0]: int(t.rsplit(':', 1)[1]) for t in r[3].split()}
        assert len(got) == min(len(want), X.TRIGGERS_PER_CLUSTER) and all(want[t] == c for t, c in got.items())
        assert abs(float(r[2]) - probs[members, 0].mean()) <= 1e-5
    return z


def _b3_all(gold, ids0, n, label):
    ev = E.SingleLabelClusterEvaluation(gold, label)
    cl = {}
    for i in range(n):
        cl.setdefault(int(ids0[i]), set()).add(i)
    ev.feed_induced_clusters(cl)
    return list(ev.compute_metrics())


@pytest.mark.parametrize("mode", [1, 2])
def test_export_end_to_end_reproduces_the_driver(tmp_path, monkeypatch, corpora, mode):
    pk = corpora['mode%d' % mode]
    ckpt = _train(tmp_path, monkeypatch, pk, "m%d" % mode)
    ck = I.load_model(ckpt)
    lab = f64_labeller(ck)
    out = str(tmp_path / "out")
    k = 3
    s = X.export(ckpt, pk, out, tsv=[corpora['new']], k=k, labeller=lab)
    feats, lex, data, gold = D.unpickle_objects(pk)
    F = lex.get_feature_space_dimensionality()
    on_disk = json.load(open(os.path.join(out, 'summary.json')))
    assert on_disk == json.loads(json.dumps(s))
    assert s['k'] == k and s['config']['K'] == 4 and s['config']['decoder'] == 'sp' and s['config']['epochs_done'] == 2
    splits = ['train'] if mode == 1 else ['train', 'valid', 'test']
    assert list(s['sets']) == splits + ['new_sentences']
    logged = ['train'] if mode == 1 else ['valid', 'test']
    for split in splits:
        exs = data[split]
        n = len(exs)
        indptr, indices, _ = X.csr_of(exs, F)
        want = lab(indptr, indices, k)
        z = _check_set(out, split, exs, gold[split], want, k)
        e = s['sets'][split]
        assert e['rows'] == n and e['rows_without_features'] == int((z['n_features'] == 0).sum())
        assert e['clusters'] == len(set(want[0][:, 0].tolist()))
        assert [e['b3']['f1'], e['b3']['precision'], e['b3']['recall']] == _b3_all(gold[split], want[0][:, 0], n, split)
        drv = e['b3_driver_rows']
        if split in logged:           # the rows and labels the training log scored: the same numbers, exactly
            assert [drv['f1'], drv['precision'], drv['recall']] == list(ck['config']['metrics'][split][-1])
    if mode == 1:
        assert N_TRAIN % BATCH != 0 and s['sets']['train']['rows'] == N_TRAIN
    ex, g = P.featurize(corpora['new'], lex, feats)
    indptr, indices, _ = X.csr_of(ex, F)
    z = _check_set(out, 'new_sentences', ex, g, lab(indptr, indices, k), k)
    e = s['sets']['new_sentences']
    assert e['rows'] == 4 and e['rows_without_features'] == 1 and z['n_features'][2] == 0
    assert 'b3' in e and 'b3_driver_rows' not in e
    # the row without features scores Wb alone
    Wb = np.asarray(ck['params']['Wb'], dtype=np.float64)
    assert z['ids'][2].tolist() == np.argsort(-Wb, kind='stable')[:k].tolist()


def test_export_command_line(tmp_path, monkeypatch, corpora, capsys):
    ckpt = _train(tmp_path, monkeypatch, corpora['mode2'], "cli")
    ck = I.load_model(ckpt)
    lab = f64_labeller(ck)
    monkeypatch.setattr(X, "cuda_labeller", lambda ck_, device=0: (lab, lambda: None))
    out = str(tmp_path / "cli_out")
    X.main([ckpt, corpora['mode2'], '--out', out, '--split', 'test', '--tsv', corpora['new'], '--top-k', '2'])
    s = json.load(open(os.path.join(out, 'summary.json')))
    assert list(s['sets']) == ['test', 'new_sentences'] and s['k'] == 2
    assert sorted(os.listdir(out)) == sorted(['summary.json'] + ['%s.%s' % (n, e) for n in ('test', 'new_sentences')
                                                                  for e in ('labels.npz', 'examples.tsv', 'clusters.tsv')])
    assert "Wrote" in capsys.readouterr().out


# ----------------------------------------------------------------------------------------------------------------------
# refusals, all before any GPU work
# ----------------------------------------------------------------------------------------------------------------------
def test_export_refusals(tmp_path, monkeypatch, corpora):
    ckpt = _train(tmp_path, monkeypatch, corpora['mode1'], "ref")
    lab = f64_labeller(I.load_model(ckpt))
    out = str(tmp_path / "o")
    pk = corpora['mode1']
    with pytest.raises(ValueError, match="checkpoint"):
        X.export(str(tmp_path / "missing.npz"), pk, out, labeller=lab)
    for k in (0, 17, 5):                  # K = 4
        with pytest.raises(ValueError, match=r"top-k %d is outside \[1, min\(K, 16\)\] = \[1, 4\]" % k):
            X.export(ckpt, pk, out, k=k, labeller=lab)
    with pytest.raises(ValueError, match="'valid'"):
        X.export(ckpt, pk, out, splits=['valid'], labeller=lab)
    clash = _write(tmp_path / "train.tsv", [_line(1)])
    with pytest.raises(ValueError, match="'train'"):
        X.export(ckpt, pk, out, tsv=[clash], labeller=lab)
    with pytest.raises(ValueError, match="'new_sentences'"):
        X.export(ckpt, pk, out, splits=[], tsv=[corpora['new'], corpora['new']], labeller=lab)
    assert not os.path.exists(out)
    # appending a split with new features grows F: W no longer matches the dataset
    F0 = D.unpickle_objects(pk)[1].get_feature_space_dimensionality()
    extra = _write(tmp_path / "extra.txt", [_line(i + 500).replace('word', 'verb') for i in range(5)])
    P.preprocess(extra, pk, batch='test', verbose=False)
    F1 = D.unpickle_objects(pk)[1].get_feature_space_dimensionality()
    assert F1 > F0
    with pytest.raises(ValueError, match=r"\(%d, 4\).*F = %d.*\(%d, 4\)" % (F0, F1, F1)):
        X.export(ckpt, pk, out, labeller=lab)


def test_export_without_gpu_or_labeller_raises(tmp_path, monkeypatch, corpora):
    import torch
    if torch.cuda.is_available():
        pytest.skip("checks the refusal to run without a GPU")
    ckpt = _train(tmp_path, monkeypatch, corpora['mode1'], "nogpu")
    with pytest.raises(RuntimeError):
        X.export(ckpt, corpora['mode1'], str(tmp_path / "o"))


# ----------------------------------------------------------------------------------------------------------------------
# GPU: export through the CUDA engine
# ----------------------------------------------------------------------------------------------------------------------
def _tie_free_agreement(ids, probs_gpu, z, k):
    """The GPU top-k set agrees with the float64 scores wherever consecutive float64 scores are farther apart than
    1e-5 max|z| (rounding ties excepted)."""
    order = np.argsort(-z, axis=1, kind='stable')
    zs = np.take_along_axis(z, order, axis=1)
    tol = 1e-5 * max(np.abs(z).max(), 1e-30)
    for j in range(k):
        gap = zs[:, j] - zs[:, j + 1] > tol if j + 1 < z.shape[1] else np.ones(len(z), bool)
        a = np.sort(ids[gap, :j + 1], axis=1)
        b = np.sort(order[gap, :j + 1], axis=1)
        assert np.array_equal(a, b), j


@pytest.mark.gpu
def test_export_through_the_cuda_engine(tmp_path, monkeypatch, corpora):
    from relation_autoencoder_b200.engine import Engine
    pk = corpora['mode2']
    ckpt = _train(tmp_path, monkeypatch, pk, "gpu", backend=None)
    ck = I.load_model(ckpt)
    out = str(tmp_path / "gout")
    k = 3
    s = X.export(ckpt, pk, out, tsv=[corpora['new']], k=k)
    for split in ('valid', 'test'):
        drv = s['sets'][split]['b3_driver_rows']
        assert [drv['f1'], drv['precision'], drv['recall']] == list(ck['config']['metrics'][split][-1])
    feats, lex, data, gold = D.unpickle_objects(pk)
    F = lex.get_feature_space_dimensionality()
    cfg, p = ck['config'], ck['params']
    eng = Engine(cfg['decoder'], 4, 6, 3, BATCH, F, p['A'].shape[0], BATCH)
    eng.set_params_numpy(p)
    lab64 = f64_labeller(ck)
    for split in ('train', 'valid', 'test'):
        z = np.load(os.path.join(out, split + '.labels.npz'))
        indptr, indices, _ = X.csr_of(data[split], F)
        zeros = np.zeros(len(data[split]), np.int32) if split == 'train' else None    # entity ids: labelling reads none
        eng.bind_split(split, indptr, indices, zeros, zeros)
        nb = len(data[split]) // BATCH
        drv = np.concatenate([eng.label(split, b)[0] for b in range(nb)])
        assert np.array_equal(z['ids'][:nb * BATCH, 0], drv.astype(np.int32))
        zz = O.encoder_scores_fast(np.asarray(p['W'], np.float64), np.asarray(p['Wb'], np.float64), indptr, indices)
        _tie_free_agreement(z['ids'], z['probs'], zz, k)
        assert np.all(np.diff(z['probs'], axis=1) <= 0)
    eng.close()
