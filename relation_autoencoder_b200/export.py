"""The induced relations of a trained model: which relation each example gets, how confident the model is, and what each
cluster holds.  This is what the reference's ``learn(debug=True)`` pickles (``OieInduction.py:230-234,395-402``),
``compute_posteriors`` returns (``:240-250``) and ``Visualizator.print_clusters`` prints (``evaluation/Visuals.py:8-30``).

    python -m relation_autoencoder_b200.export train_products/m.npz sample.pk --out exported/ \\
        [--split train --split test ...] [--tsv new_sentences.txt ...] [--top-k 3] [--rank-arguments]
        [--predict-arguments 5] [--device 0]

Every row of every labelled set is labelled, the tail batch included, by one ``rae_label_topk`` call on one GPU (the
checkpoint does not depend on the world size it was trained on).  New sentences (``--tsv``) are featurised through the
dataset's lexicon without changing it, so W still matches.  Per set NAME (a split, or a TSV file's stem) the output
directory gets ``NAME.labels.npz``, ``NAME.examples.tsv`` and ``NAME.clusters.tsv``, and ``summary.json`` holds the
checkpoint's configuration and per-set counts and B-cubed scores.

With ``--rank-arguments`` the decoder is measured as well, without gold labels: every example's true arguments are
ranked against all entities (``rae_rank_arguments``: rank 1 + the number of entities whose score in that argument slot
beats the true one's).  Per set, ``NAME.argranks.npz`` holds ``rank1`` and ``rank2`` (-1 for a row whose entity strings
the dataset never saw: such rows cannot be ranked and are left out of the metrics), and ``summary.json`` gets
``sets[NAME]['arguments']``: rows ranked and skipped, and MRR, mean rank and Hits@1/3/10 per slot and over both slots.

With ``--predict-arguments K`` the decoder is asked what it was trained to answer: for each example, the K entities it
scores highest in each argument slot (``rae_predict_arguments``).  A slot is predicted whenever the argument it is
conditioned on (the other one) is an entity the dataset knows, even if the argument it predicts is not: that is the case
``--rank-arguments`` has to skip.  Per set, ``NAME.argpreds.npz`` holds ``ids1, scores1, ids2, scores2`` ([n, K]; ids -1
and scores NaN for a slot that was not predicted), ``NAME.argpreds.tsv`` lists them as ``entity:score`` with the 1-based
position of the true argument in each list (0: not in the list, -1: unknown or not predicted), and ``summary.json`` gets
``sets[NAME]['predictions']``: rows predicted per slot and the share of those with a known true argument that list it.
Scores order one row's candidates; they are not comparable across rows.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
from collections import Counter
from typing import Callable, Dict, Optional, Sequence

import numpy as np

from .data import SPLIT_LABELS, entity_index, unpickle_objects
from .evaluation import SingleLabelClusterEvaluation
from .induction import load_model
from .preprocess import featurize

TRIGGERS_PER_CLUSTER = 10        # settings.py elems_to_visualize: the triggers print_clusters shows per cluster
GOLD_PER_CLUSTER = 5
MAX_TOP_K = 16                   # RAE_MAX_TOPK (include/rae.h)
HITS_AT = (1, 3, 10)


def csr_of(examples, F: int):
    """Binary CSR of the examples' feature ids (duplicates collapse, ascending within a row, as DatasetManager builds it)
    -> (indptr int32 [n+1], indices int32 [nnz], n_features int32 [n])."""
    rows = [np.unique(np.asarray(ex.features, dtype=np.int64)) for ex in examples]
    for i, u in enumerate(rows):
        if u.size and (u[0] < 0 or u[-1] >= F):
            raise IndexError("feature id out of range [0, %d) in example %d" % (F, i))
    n_features = np.array([u.size for u in rows], dtype=np.int32)
    indptr = np.zeros(len(rows) + 1, dtype=np.int64)
    np.cumsum(n_features, out=indptr[1:])
    if indptr[-1] >= 2 ** 31:
        raise ValueError("%d features in one set: more than an int32 CSR holds" % indptr[-1])
    indices = np.concatenate(rows).astype(np.int32) if rows else np.zeros(0, np.int32)
    return indptr.astype(np.int32), indices, n_features


def _engine(ck: dict, device: int):
    """An Engine bound to the checkpoint's parameters, with the checkpoint's batch size as the forward pass's chunk."""
    from .engine import Engine
    cfg, p = ck['config'], ck['params']
    F, K = p['W'].shape
    N, d = p['A'].shape
    B = int(cfg.get('batch_size', 1))
    eng = Engine(cfg['decoder'], K, d, int(cfg.get('neg_samples', 1)), B, F, N, B, device=device)
    eng.set_params_numpy(p)
    return eng


def cuda_labeller(ck: dict, device: int = 0):
    """(labeller, close): ``labeller(indptr, indices, k) -> (ids, probs)`` through :meth:`Engine.label_topk` on the
    checkpoint's parameters.  Only W and Wb are read, but the engine binds every parameter of the decoder."""
    eng = _engine(ck, device)
    return (lambda indptr, indices, k: eng.label_topk(indptr, indices, k, probs=True)), eng.close


def cuda_ranker(ck: dict, device: int = 0):
    """(ranker, close): ``ranker(indptr, indices, args1, args2) -> (rank1, rank2)`` through :meth:`Engine.rank_arguments`
    on the checkpoint's parameters, with the checkpoint's batch size as the forward pass's chunk."""
    eng = _engine(ck, device)
    return eng.rank_arguments, eng.close


def cuda_predictor(ck: dict, device: int = 0):
    """(predictor, close): ``predictor(indptr, indices, args1, args2, k) -> (ids1, scores1, ids2, scores2)`` through
    :meth:`Engine.predict_arguments` on the checkpoint's parameters, as :func:`cuda_ranker`."""
    eng = _engine(ck, device)
    return eng.predict_arguments, eng.close


def rank_metrics(ranks: np.ndarray) -> dict:
    """MRR, mean rank and Hits@1/3/10 of 1-based ranks (float64 means)."""
    r = np.asarray(ranks, dtype=np.float64)
    m = {'mrr': float(np.mean(1.0 / r)), 'mean_rank': float(np.mean(r))}
    for k in HITS_AT:
        m['hits@%d' % k] = float(np.mean(r <= k))
    return m


def _rank_set(out_dir: str, name: str, examples, arg2id: Dict[str, int], F: int, ranker) -> dict:
    """Ranks the arguments of the rows whose two entity strings are in the dataset, writes NAME.argranks.npz and returns
    the summary entry."""
    n = len(examples)
    a1 = np.array([arg2id.get(ex.arg1, -1) for ex in examples], dtype=np.int64)
    a2 = np.array([arg2id.get(ex.arg2, -1) for ex in examples], dtype=np.int64)
    ok = np.flatnonzero((a1 >= 0) & (a2 >= 0))
    rank1 = np.full(n, -1, dtype=np.int32)
    rank2 = np.full(n, -1, dtype=np.int32)
    if ok.size:
        indptr, indices, _ = csr_of([examples[i] for i in ok], F)
        r1, r2 = ranker(indptr, indices, a1[ok].astype(np.int32), a2[ok].astype(np.int32))
        r1 = np.asarray(r1, dtype=np.int32)
        r2 = np.asarray(r2, dtype=np.int32)
        if r1.shape != (ok.size,) or r2.shape != (ok.size,):
            raise RuntimeError("the ranker returned %s / %s for %d rows" % (r1.shape, r2.shape, ok.size))
        rank1[ok], rank2[ok] = r1, r2
    np.savez(os.path.join(out_dir, name + '.argranks.npz'), rank1=rank1, rank2=rank2)
    entry = {'rows_ranked': int(ok.size), 'rows_skipped': int(n - ok.size)}
    if ok.size:
        entry['arg1'] = rank_metrics(rank1[ok])
        entry['arg2'] = rank_metrics(rank2[ok])
        entry['both'] = rank_metrics(np.concatenate([rank1[ok], rank2[ok]]))
    return entry


def _position(ids: np.ndarray, true: np.ndarray, known: np.ndarray) -> np.ndarray:
    """1-based position of true[i] in ids[i] (0: not listed), -1 where known[i] is False."""
    hit = ids == true[:, None]
    pos = np.where(hit.any(1), hit.argmax(1) + 1, 0)
    return np.where(known, pos, -1).astype(np.int64)


def _predict_set(out_dir: str, name: str, examples, arg2id: Dict[str, int], id2arg, F: int, predictor, k: int,
                 relation: np.ndarray) -> dict:
    """Predicts each slot whose conditioning argument is known, writes NAME.argpreds.npz / .tsv and returns the summary
    entry."""
    n = len(examples)
    a1 = np.array([arg2id.get(ex.arg1, -1) for ex in examples], dtype=np.int64)
    a2 = np.array([arg2id.get(ex.arg2, -1) for ex in examples], dtype=np.int64)
    k1, k2 = a1 >= 0, a2 >= 0
    send = np.flatnonzero(k1 | k2)
    ids = [np.full((n, k), -1, np.int32), np.full((n, k), -1, np.int32)]
    scores = [np.full((n, k), np.nan, np.float32), np.full((n, k), np.nan, np.float32)]
    if send.size:
        indptr, indices, _ = csr_of([examples[i] for i in send], F)
        got = predictor(indptr, indices, np.maximum(a1[send], 0).astype(np.int32), np.maximum(a2[send], 0).astype(np.int32), k)
        got = [np.asarray(g) for g in got]
        if len(got) != 4 or any(g.shape != (send.size, k) for g in got):
            raise RuntimeError("the predictor returned %s for %d rows and k = %d" % ([g.shape for g in got], send.size, k))
        # slot 1 predicts arg1 from arg2, slot 2 predicts arg2 from arg1: keep a slot only where its condition is known
        for s, cond in ((0, k2), (1, k1)):
            rows = send[cond[send]]
            ids[s][rows] = got[2 * s][cond[send]]
            scores[s][rows] = got[2 * s + 1][cond[send]]
    np.savez(os.path.join(out_dir, name + '.argpreds.npz'), ids1=ids[0], scores1=scores[0], ids2=ids[1], scores2=scores[1])
    pos1 = _position(ids[0], a1, k1 & k2)
    pos2 = _position(ids[1], a2, k1 & k2)

    def listing(i, s):
        return ' '.join('%s:%.6g' % (id2arg[x], v) for x, v in zip(ids[s][i], scores[s][i]) if x >= 0)
    with open(os.path.join(out_dir, name + '.argpreds.tsv'), 'w', encoding='utf-8') as f:
        f.write('index\targ1\targ2\ttrigger\trelation\tpredicted_arg1\tpredicted_arg2\tposition1\tposition2\n')
        for i, ex in enumerate(examples):
            f.write('%d\t%s\t%s\t%s\t%d\t%s\t%s\t%d\t%d\n' % (i, ex.arg1, ex.arg2, ex.trigger, relation[i], listing(i, 0),
                                                              listing(i, 1), pos1[i], pos2[i]))
    entry = {'k': k}
    for slot, pos, cond in (('arg1', pos1, k2), ('arg2', pos2, k1)):
        known = pos >= 0
        entry[slot] = {'rows_predicted': int(cond.sum()), 'rows_with_known_argument': int(known.sum()),
                       'share_in_list': float(np.mean(pos[known] > 0)) if known.any() else None}
    return entry


def _b3(gold: Dict[int, list], label: str, ids0: np.ndarray, n_rows: int):
    """B-cubed of the clustering ids0[:n_rows] against the whole set's gold labels, as the driver scores a split; None
    when no row of the set has a gold label."""
    ev = SingleLabelClusterEvaluation(gold, label if label in SPLIT_LABELS else 'test')
    if not ev.assessableElemSet:
        return None
    clusters: Dict[int, set] = {}
    for i in range(n_rows):
        clusters.setdefault(int(ids0[i]), set()).add(i)
    ev.feed_induced_clusters(clusters)
    f1, pre, rec = ev.compute_metrics()
    return {'f1': f1, 'precision': pre, 'recall': rec}


def _first_gold(gold: Dict[int, list], i: int) -> str:
    g = gold.get(i) or ['']
    return g[0]


def _top(counter: Counter, n: int) -> str:
    return ' '.join('%s:%d' % (s, c) for s, c in sorted(counter.items(), key=lambda t: (-t[1], t[0]))[:n])


def _write_set(out_dir: str, name: str, examples, gold, ids, probs, n_features):
    n, k = ids.shape
    np.savez(os.path.join(out_dir, name + '.labels.npz'), ids=ids, probs=probs, n_features=n_features)
    with open(os.path.join(out_dir, name + '.examples.tsv'), 'w', encoding='utf-8') as f:
        f.write('index\targ1\targ2\ttrigger\tgold\trelation\tprob\tn_features\ttopk\n')
        for i, ex in enumerate(examples):
            topk = ' '.join('%d:%.6g' % (ids[i, j], probs[i, j]) for j in range(k))
            f.write('%d\t%s\t%s\t%s\t%s\t%d\t%.6g\t%d\t%s\n' % (i, ex.arg1, ex.arg2, ex.trigger, _first_gold(gold, i),
                                                              ids[i, 0], probs[i, 0], n_features[i], topk))
    members: Dict[int, list] = {}
    for i in range(n):
        members.setdefault(int(ids[i, 0]), []).append(i)
    order = sorted(members, key=lambda r: (-len(members[r]), r))
    with open(os.path.join(out_dir, name + '.clusters.tsv'), 'w', encoding='utf-8') as f:
        f.write('relation\tsize\tmean_prob\ttriggers\tgold\n')
        for r in order:
            m = members[r]
            trig = Counter(examples[i].trigger for i in m)
            gl = Counter(g for g in (_first_gold(gold, i) for i in m) if g != '')
            f.write('%d\t%d\t%.6g\t%s\t%s\n' % (r, len(m), float(np.mean(probs[m, 0], dtype=np.float64)),
                                                _top(trig, TRIGGERS_PER_CLUSTER), _top(gl, GOLD_PER_CLUSTER)))
    return len(order)


def export(checkpoint: str, dataset: str, out_dir: str, splits: Optional[Sequence[str]] = None, tsv: Sequence[str] = (),
           k: int = 3, device: int = 0, labeller: Optional[Callable] = None, rank_arguments: bool = False,
           ranker: Optional[Callable] = None, predict_arguments: int = 0, predictor: Optional[Callable] = None) -> dict:
    """Labels the requested splits of ``dataset`` (default: all of them) and the sentences of each ``tsv`` file with the
    k most probable relations of the model in ``checkpoint``, writes the files the module docstring lists into
    ``out_dir`` and returns the summary.  ``labeller(indptr, indices, k) -> (ids int32 [n, k], probs float32 [n, k])``
    replaces the CUDA engine (there is no CPU fallback: without a GPU and without a labeller this raises).  With
    ``rank_arguments`` every set's arguments are ranked as well (module docstring); ``ranker(indptr, indices, args1,
    args2) -> (rank1 int32 [n], rank2 int32 [n])`` replaces the CUDA engine there in the same way.  With
    ``predict_arguments = K > 0`` the K most likely entities of each argument slot are written (module docstring);
    ``predictor(indptr, indices, args1, args2, K) -> (ids1, scores1, ids2, scores2)`` replaces the CUDA engine there.
    The arguments are checked before any GPU work."""
    try:
        ck = load_model(checkpoint)
    except Exception as e:
        raise ValueError("cannot load the checkpoint %s: %s" % (checkpoint, e)) from e
    cfg = ck['config']
    feats, lex, data, gold = unpickle_objects(dataset)
    F = lex.get_feature_space_dimensionality()
    W = ck['params'].get('W')
    K = int(cfg['relations'])
    if W is None or W.ndim != 2 or W.shape != (F, K):
        raise ValueError("the checkpoint's W has shape %s, but the dataset's lexicon has F = %d features and the model K = %d "
                         "relations: W must be (F, K) = (%d, %d); was the dataset extended after training?"
                         % (None if W is None else tuple(W.shape), F, K, F, K))
    k = int(k)
    if not 1 <= k <= min(K, MAX_TOP_K):
        raise ValueError("top-k %d is outside [1, min(K, %d)] = [1, %d]" % (k, MAX_TOP_K, min(K, MAX_TOP_K)))
    splits = [s for s in SPLIT_LABELS if s in data] if splits is None else list(splits)
    missing = [s for s in splits if s not in data]
    if missing:
        raise ValueError("split(s) %s are not in %s, which has %s" % (missing, dataset, [s for s in SPLIT_LABELS if s in data]))
    names = list(splits)
    for path in tsv:
        stem = os.path.splitext(os.path.basename(path))[0]
        if stem in names:
            raise ValueError("the TSV file %s would be written as set %r, which is already a set of this export" % (path, stem))
        names.append(stem)
    arg2id = id2arg = None
    predict_arguments = int(predict_arguments)
    if rank_arguments or predict_arguments:
        _, id2arg, arg2id = entity_index(data)
        A = ck['params'].get('A')
        if A is None or A.ndim != 2 or A.shape[0] != len(arg2id):
            raise ValueError("the checkpoint's A has %s rows, but the dataset has %d entities: the model was not trained on "
                             "this dataset" % (None if A is None else A.shape[0], len(arg2id)))
    if predict_arguments and not 1 <= predict_arguments <= min(len(arg2id), MAX_TOP_K):
        raise ValueError("--predict-arguments %d is outside [1, min(N, %d)] = [1, %d]"
                         % (predict_arguments, MAX_TOP_K, min(len(arg2id), MAX_TOP_K)))
    sets = [(s, data[s], gold.get(s, {}), True) for s in splits]
    for path, name in zip(tsv, names[len(splits):]):
        ex, g = featurize(path, lex, feats)
        sets.append((name, ex, g, False))

    close = None
    if labeller is None:
        labeller, close = cuda_labeller(ck, device)
    close_ranker = None
    if rank_arguments and ranker is None:
        ranker, close_ranker = cuda_ranker(ck, device)
    close_predictor = None
    if predict_arguments and predictor is None:
        predictor, close_predictor = cuda_predictor(ck, device)
    os.makedirs(out_dir, exist_ok=True)
    B = int(cfg.get('batch_size', 1))
    summary = {'checkpoint': os.path.abspath(checkpoint),
               'config': {'decoder': cfg.get('decoder'), 'K': K, 'd': int(ck['params']['A'].shape[1]),
                          'epochs_done': cfg.get('epochs_done'), 'model_id': cfg.get('model_id')},
               'k': k, 'sets': {}}
    try:
        for name, examples, g, is_split in sets:
            indptr, indices, n_features = csr_of(examples, F)
            ids, probs = labeller(indptr, indices, k)
            ids = np.ascontiguousarray(ids, dtype=np.int32)
            probs = np.ascontiguousarray(probs, dtype=np.float32)
            n = len(examples)
            if ids.shape != (n, k) or probs.shape != (n, k):
                raise RuntimeError("the labeller returned %s / %s for %d rows and k = %d" % (ids.shape, probs.shape, n, k))
            n_clusters = _write_set(out_dir, name, examples, g, ids, probs, n_features)
            entry = {'rows': n, 'rows_without_features': int((n_features == 0).sum()), 'clusters': n_clusters}
            b3 = _b3(g, name, ids[:, 0], n)
            if b3 is not None:
                entry['b3'] = b3
                if is_split:         # the rows the training log scores: whole batches only (OieInduction.py:96-98)
                    entry['b3_driver_rows'] = _b3(g, name, ids[:, 0], (n // B) * B)
            if rank_arguments:
                entry['arguments'] = _rank_set(out_dir, name, examples, arg2id, F, ranker)
            if predict_arguments:
                entry['predictions'] = _predict_set(out_dir, name, examples, arg2id, id2arg, F, predictor, predict_arguments,
                                                    ids[:, 0])
            summary['sets'][name] = entry
    finally:
        if close is not None:
            close()
        if close_ranker is not None:
            close_ranker()
        if close_predictor is not None:
            close_predictor()
    with open(os.path.join(out_dir, 'summary.json'), 'w') as f:
        json.dump(summary, f, indent=1)
    return summary


def main(argv=None):
    p = argparse.ArgumentParser(prog='export', description='Exports the relations a trained model induces for a dataset '
                                'and for new sentences: top-k labels, per-example table, cluster summaries, B-cubed.')
    p.add_argument('checkpoint', help='the .npz checkpoint written by the training command')
    p.add_argument('dataset', help='the pickled dataset the model was trained on')
    p.add_argument('--out', required=True, help='output directory')
    p.add_argument('--split', action='append', default=None, help='a split to label (repeatable; default: every split)')
    p.add_argument('--tsv', action='append', default=[], help='a file of new sentences in the dataset format (repeatable)')
    p.add_argument('--top-k', dest='k', type=int, default=3, help='relations kept per example (1 to min(K, 16))')
    p.add_argument('--rank-arguments', action='store_true',
                   help='also rank every example\'s true arguments against all entities (MRR, mean rank, Hits@1/3/10)')
    p.add_argument('--predict-arguments', dest='predict_arguments', type=int, default=None, metavar='K',
                   help='also list the K most likely entities of each argument slot of every example (1 to min(N, 16))')
    p.add_argument('--device', type=int, default=0, help='CUDA device index')
    a = p.parse_args(argv)
    if a.predict_arguments is not None and a.predict_arguments < 1:
        p.error('--predict-arguments %d: K must be at least 1' % a.predict_arguments)
    summary = export(a.checkpoint, a.dataset, a.out, splits=a.split, tsv=a.tsv, k=a.k, device=a.device,
                     rank_arguments=a.rank_arguments, predict_arguments=a.predict_arguments or 0)
    for name, s in summary['sets'].items():
        b3 = s.get('b3')
        args = s.get('arguments', {}).get('both')
        print('%s: %d rows, %d without features, %d clusters%s%s' % (name, s['rows'], s['rows_without_features'], s['clusters'],
              '' if b3 is None else ', B3 f1 %.4f' % b3['f1'], '' if args is None else ', argument MRR %.4f' % args['mrr']))
    print('Wrote', os.path.join(a.out, 'summary.json'))
    return summary


if __name__ == '__main__':
    main(sys.argv[1:])
