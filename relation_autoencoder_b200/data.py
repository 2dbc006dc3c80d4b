"""The pickled OiePreprocessor dataset format and its indexing, drop-in compatible with the reference.

File format (``processing/OiePreprocessor.py:317-320`` writer, ``:344-359`` reader): FOUR consecutive pickles
  1. list of feature-extraction functions           (``definitions.OieFeatures.<name>`` globals)
  2. ``FeatureLexicon``                              (``processing.OiePreprocessor.FeatureLexicon``, or
                                                     ``__main__.FeatureLexicon`` when the preprocessor ran as a script)
  3. ``{split: [OieExample, ...]}``                  (``definitions.OieExample.OieExample``)
  4. ``{split: {example index: [label tokens]}}``
written by Python 2 with ``HIGHEST_PROTOCOL`` (= 2).  :func:`unpickle_objects` reads such files under Python 3 (class
paths are remapped in ``find_class``; py2 ``str`` is decoded as UTF-8, falling back to latin-1) and
:func:`pickle_objects` writes protocol-2 files whose globals carry the REFERENCE's module paths, so the reference's own
``unpickle_objects`` can read them back.

``DatasetManager`` / ``DatasetSplit`` restate ``learning/OieData.py:8-155``: entity <-> id maps, the freq**0.75
cumulative negative-sampling distribution (``:57-59``) and, per split, int32 ``args1/args2`` plus the binary CSR feature
matrix (``:83-90``; duplicate feature ids of one example collapse as the reference's ``dok`` assignment does).
One stated divergence: the reference numbers entities in Python-2 ``dict`` iteration order of a ``Counter``
(``OieData.py:54,139-144``, hash order, not reproducible across interpreters); here ids follow first appearance.
"""
from __future__ import annotations

import io
import os
import pickle
import sys
import types
from collections import Counter
from typing import Dict, List

import numpy as np

SPLIT_LABELS = ['train', 'valid', 'test']           # settings.py:26

REF_LEXICON_MODULE = 'processing.OiePreprocessor'
REF_EXAMPLE_MODULE = 'definitions.OieExample'
REF_FEATURES_MODULE = 'definitions.OieFeatures'
# every extractor the reference defines (OieFeatures.py:294); the nine defaults are restated in preprocess.py
REF_FEATURE_NAMES = frozenset("""bow bow_clean before_arg1 after_arg2 bigrams trigrams skiptrigrams skipfourgrams trigger
entityTypes entity1Type entity2Type arg1 arg1_lower arg1unigrams arg2 arg2_lower arg2unigrams lexicalPattern
dependencyParsing rightDep leftDep posPatternPath""".split())


class OieExample(object):
    """One sentence datapoint: thresholded feature ids + the two entity strings, trigger and gold label
    (``definitions/OieExample.py:1-20``; attribute names are part of the pickle format)."""

    def __init__(self, arg1, arg2, features, trigger, relation=''):
        self.features = features
        self.arg1 = arg1
        self.arg2 = arg2
        self.relation = relation
        self.trigger = trigger


class FeatureLexicon(object):
    """Feature string <-> id maps with frequencies and the thresholded ("pruned") id space
    (``processing/OiePreprocessor.py:9-110``; attribute names are part of the pickle format)."""

    def __init__(self):
        self.nextId = 0
        self.id2Str = {}
        self.str2Id = {}
        self.id2freq = {}
        self.nextIdPruned = 0
        self.id2StrPruned = {}
        self.str2IdPruned = {}

    def get_or_add(self, s):
        if s not in self.str2Id:
            self.id2Str[self.nextId] = s
            self.str2Id[s] = self.nextId
            self.id2freq[self.nextId] = 1
            self.nextId += 1
        else:
            self.id2freq[self.str2Id[s]] += 1
        return self.str2Id[s]

    def get_or_add_pruned(self, s):
        if s not in self.str2IdPruned:
            self.id2StrPruned[self.nextIdPruned] = s
            self.str2IdPruned[s] = self.nextIdPruned
            self.nextIdPruned += 1
        return self.str2IdPruned[s]

    def get_id(self, a_string):
        return self.str2Id.get(a_string)

    def get_str(self, idx):
        return self.id2Str.get(idx)

    def get_str_pruned(self, idx):
        return self.id2StrPruned.get(idx)

    def get_freq(self, idx):
        return self.id2freq.get(idx)

    def get_feature_space_dimensionality(self):
        return self.nextIdPruned


class _FeatureFunctionStub(object):
    """Stands in for a ``definitions.OieFeatures`` function this package does not restate (the pickle stores the
    extractors by global name only; training never calls them)."""

    def __init__(self, name):
        self.__name__ = name

    def __call__(self, info, arg1, arg2):
        raise NotImplementedError("feature extractor %r is not available (only its name travelled in the pickle)" % self.__name__)

    def __reduce__(self):
        return (_FeatureFunctionStub, (self.__name__,))


def _feature_function(name):
    from . import preprocess
    fn = getattr(preprocess, name, None)
    if callable(fn) and name in preprocess.FEATURE_FUNCTION_NAMES:
        return fn
    return _FeatureFunctionStub(name)


_SAFE_GLOBALS = frozenset(
    [(m, n) for m in ('builtins', '__builtin__') for n in ('set', 'frozenset', 'list', 'dict', 'tuple', 'object', 'int', 'long',
                                                          'float', 'str', 'unicode', 'bytes', 'bool', 'complex')]
    + [('copy_reg', '_reconstructor'), ('copyreg', '_reconstructor'), ('collections', 'OrderedDict'),
       ('collections', 'defaultdict'), ('collections', 'Counter')])


class _RefUnpickler(pickle.Unpickler):
    def find_class(self, module, name):
        if name == 'FeatureLexicon' and module in ('__main__', REF_LEXICON_MODULE, 'OiePreprocessor', __name__):
            return FeatureLexicon
        if name == 'OieExample' and module in (REF_EXAMPLE_MODULE, 'OieExample', '__main__', __name__):
            return OieExample
        if module in (REF_FEATURES_MODULE, 'OieFeatures'):
            return _feature_function(name)
        if module == __name__ and name == '_FeatureFunctionStub':
            return _FeatureFunctionStub
        # the format needs nothing else beyond a few harmless builtins (py2 names included): anything else - os.system
        # through REDUCE, say - is refused instead of imported, so a dataset file from an untrusted source cannot run code
        if (module, name) in _SAFE_GLOBALS:
            return super().find_class(module, name)
        raise pickle.UnpicklingError("dataset pickle refers to %s.%s, which the dataset format does not need" % (module, name))


class _RefPickler(pickle._Pickler):
    """Protocol-2 pickler that names this package's classes / extractor functions by the REFERENCE's module paths."""

    def save_global(self, obj, name=None):
        ref = None
        if obj is FeatureLexicon:
            ref = (REF_LEXICON_MODULE, 'FeatureLexicon')
        elif obj is OieExample:
            ref = (REF_EXAMPLE_MODULE, 'OieExample')
        elif (callable(obj) and getattr(obj, '__name__', None) in REF_FEATURE_NAMES
              and getattr(obj, '__module__', '') in (__package__ + '.preprocess', '__main__')):
            ref = (REF_FEATURES_MODULE, obj.__name__)
        if ref is None:
            return super().save_global(obj, name)
        self.write(pickle.GLOBAL + ref[0].encode('ascii') + b'\n' + ref[1].encode('ascii') + b'\n')
        self.memoize(obj)

    def save(self, obj, save_persistent_id=True):
        if isinstance(obj, _FeatureFunctionStub):
            self.write(pickle.GLOBAL + REF_FEATURES_MODULE.encode('ascii') + b'\n' + obj.__name__.encode('ascii') + b'\n')
            self.memoize(obj)
            return
        return super().save(obj, save_persistent_id)

    dispatch = dict(pickle._Pickler.dispatch)


# plain functions reach save_global through the dispatch table, which holds the BASE class's function
_RefPickler.dispatch[types.FunctionType] = _RefPickler.save_global


def _load_all(raw: bytes, encoding: str):
    f = io.BytesIO(raw)
    out = []
    for _ in range(4):
        out.append(_RefUnpickler(f, encoding=encoding).load())
    return out


def unpickle_objects(a_file, verbose=False):
    """(feature functions, FeatureLexicon, {split: [OieExample]}, {split: {idx: [tokens]}})  - OiePreprocessor.py:323-364."""
    with open(a_file, 'rb') as f:
        raw = f.read()
    try:
        feats, lex, data, gold = _load_all(raw, 'utf-8')
    except UnicodeDecodeError:
        feats, lex, data, gold = _load_all(raw, 'latin-1')
    # the four objects of a dataset file, in file order (validated like pickle_objects validates what it writes)
    for pos, obj, want in ((1, feats, list), (2, lex, FeatureLexicon), (3, data, dict), (4, gold, dict)):
        if not isinstance(obj, want):
            raise AssertionError('%s: object %d of the dataset file is a %s, expected %s'
                                 % (a_file, pos, type(obj).__name__, want.__name__))
    if verbose:
        print('  loaded feature extractors:', ', '.join("'" + str(getattr(_, '__name__', _)) + "'" for _ in feats))
        print('  loaded dataset with {} splits'.format(', '.join("'" + _ + "'" for _ in data.keys())))
    return feats, lex, data, gold


def pickle_objects(feat_extrs, feat_lex, dataset_splits, goldstandard_splits, a_file):
    """Writes the four pickles (protocol 2, reference module paths) in the order OiePreprocessor.py:290-320 defines:
    [feature functions], FeatureLexicon, {split: [OieExample]}, {split: {index: [label tokens]}}.  The arguments are
    validated first (the reference does the same before it opens the file)."""
    splits_allowed = ('train', 'test', 'valid')
    if not isinstance(feat_extrs, list) or not all(callable(f) for f in feat_extrs):
        raise AssertionError('object 1 of the dataset file must be a list of feature callables, got %r' % (feat_extrs,))
    if not isinstance(feat_lex, FeatureLexicon):
        raise AssertionError('object 2 of the dataset file must be a FeatureLexicon, got %s' % type(feat_lex).__name__)
    for pos, obj in ((3, dataset_splits), (4, goldstandard_splits)):
        if not isinstance(obj, dict):
            raise AssertionError('object %d of the dataset file must be a dict keyed by split, got %s' % (pos, type(obj).__name__))
        unknown = [k for k in obj if k not in splits_allowed]
        if unknown:
            raise AssertionError('object %d of the dataset file has split keys %r outside %r' % (pos, unknown, splits_allowed))
    with open(a_file, 'wb') as pkl_file:
        for obj in (feat_extrs, feat_lex, dataset_splits, goldstandard_splits):
            _RefPickler(pkl_file, protocol=2).dump(obj)


# ----------------------------------------------------------------------------------------------------------------------
# indexing  (learning/OieData.py)
# ----------------------------------------------------------------------------------------------------------------------
class DatasetSplit(object):
    """args1/args2 int32 [l] + binary CSR features [l, F] (OieData.py:8-26).  ``xFeats`` is a scipy CSR matrix as in the
    reference; ``indptr``/``indices`` are the int32 arrays the engine binds."""

    def __init__(self, arguments1, arguments2, arg_features):
        self.args1 = arguments1
        self.args2 = arguments2
        self.xFeats = arg_features

    def get_size(self):
        return len(self.args1)

    @property
    def indptr(self):
        return np.asarray(self.xFeats.indptr, dtype=np.int32)

    @property
    def indices(self):
        return np.asarray(self.xFeats.indices, dtype=np.int32)


def generate_args(oie_dataset):
    """arg1, arg2 of every example of every split, train -> valid -> test (OieData.py:158-171)."""
    for split in ('train', 'valid', 'test'):
        if split in oie_dataset:
            for ex in oie_dataset[split]:
                yield ex.arg1
                yield ex.arg2


def entity_index(oie_dataset):
    """(entity_freqs, id2Arg, arg2Id) of a dataset's entity strings (OieData.py:54,139-144): ids in the order of the strings'
    first occurrence in ``generate_args``.  The one indexing of entities: DatasetManager trains with it and the export
    ranks arguments with it."""
    entity_freqs = Counter(generate_args(oie_dataset))
    id2_arg, arg2_id = DatasetManager._index_elements(entity_freqs)
    return entity_freqs, id2_arg, arg2_id


class DatasetManager(object):
    def __init__(self, oie_dataset, feature_lex, rng, neg_sampling_distr_power=0.75, verbose=False):
        if 'train' not in oie_dataset:
            raise Exception("Dataset manager requires that the provided dataset contains a 'train' split.")
        self.negSamplingDistrPower = neg_sampling_distr_power
        self.rng = rng
        self.featureLex = feature_lex
        self.split: Dict[str, DatasetSplit] = {}
        entity_freqs, self.id2Arg, self.arg2Id = entity_index(oie_dataset)
        if verbose:
            print('  feature space size: {}\n  number of unique entities: {}'.format(self.get_dimensionality(), len(entity_freqs)))
        powered = [entity_freqs[self.id2Arg[i]] ** self.negSamplingDistrPower for i in range(len(self.id2Arg))]
        norm1 = float(sum(powered))                                   # OieData.py:57 (left-to-right python sum)
        self.negSamplingDistr = [x / norm1 for x in powered]          # :58
        self.negSamplingCum = np.cumsum(self.negSamplingDistr)        # :59
        for split in SPLIT_LABELS:
            if split in oie_dataset:
                self.split[split] = self._produce_dataset_split(oie_dataset, split)
                if verbose:
                    print("  initialized '{}' split with {} number of examples".format(split, len(self.split[split].args1)))

    def _produce_dataset_split(self, oie_examples, split):
        """OieData.py:71-90: entity ids + binary CSR (row i has a 1.0 at every id in ``example.features``)."""
        import scipy.sparse as sp
        exs = oie_examples[split]
        l = len(exs)
        F = self.featureLex.get_feature_space_dimensionality()
        args1 = np.zeros(l, dtype=np.int32)
        args2 = np.zeros(l, dtype=np.int32)
        indptr = np.zeros(l + 1, dtype=np.int64)
        cols: List[np.ndarray] = []
        for i, ex in enumerate(exs):
            args1[i] = self.arg2Id[ex.arg1]
            args2[i] = self.arg2Id[ex.arg2]
            u = np.unique(np.asarray(ex.features, dtype=np.int64))    # dok assignment de-duplicates; ascending within row
            if u.size and (u[0] < 0 or u[-1] >= F):
                raise IndexError("feature id out of range in split %r, example %d" % (split, i))
            cols.append(u)
            indptr[i + 1] = indptr[i] + u.size
        indices = np.concatenate(cols).astype(np.int32) if cols else np.zeros(0, np.int32)
        data = np.ones(indices.shape[0], dtype=np.float32)
        x = sp.csr_matrix((data, indices, indptr.astype(np.int32)), shape=(l, F), dtype=np.float32)
        return DatasetSplit(args1, args2, x)

    def get_arg_voc_size(self):
        return len(self.arg2Id)

    def get_dimensionality(self):
        return self.featureLex.get_feature_space_dimensionality()

    def get_example_feature(self, an_id, a_split, feature):
        for e in self.split[a_split].xFeats[an_id].nonzero()[1]:
            feat = self.featureLex.get_str_pruned(e)
            if feat is not None and feat.find(feature) > -1:
                return feat
        return None

    def get_neg_sampling_cum(self):
        return self.negSamplingCum

    def generate_split_keys(self):
        for _ in SPLIT_LABELS:
            if _ in self.split:
                yield _

    @staticmethod
    def _index_elements(elements):
        id2_elem, elem2_id = {}, {}
        for idx, x in enumerate(elements):
            id2_elem[idx] = x
            elem2_id[x] = idx
        return id2_elem, elem2_id


def load_data(pickled_dataset, rng, verbose=False):
    """(DatasetManager, goldstandard) from a pickled dataset file (OieInduction.py:416-436)."""
    if not os.path.exists(pickled_dataset):
        print("Pickled '{}' dataset not found".format(pickled_dataset), file=sys.stderr)
        sys.exit(1)
    if verbose:
        print('Loading data from pickled file')
    _, relation_lexicon, data, gold_standard = unpickle_objects(pickled_dataset)
    return DatasetManager(data, relation_lexicon, rng, verbose=verbose), gold_standard


class IndexedDataset(object):
    """The indexed form of a dataset (what ``DatasetManager`` produces) without the strings: per split int32
    ``args1/args2`` + binary CSR, the negative-sampling cumulative distribution and the gold labels' first tokens.
    Offers the part of the ``DatasetManager`` interface the driver uses, and a compact ``.npz`` round trip."""

    def __init__(self, splits: Dict[str, DatasetSplit], neg_sampling_cum, n_features: int, n_entities: int,
                 gold: Dict[str, Dict[int, List[str]]]):
        self.split = splits
        self.negSamplingCum = np.asarray(neg_sampling_cum, dtype=np.float64)
        self._F = int(n_features)
        self._N = int(n_entities)
        self.goldStandard = gold

    @classmethod
    def from_manager(cls, dm: DatasetManager, gold):
        return cls(dict(dm.split), dm.negSamplingCum, dm.get_dimensionality(), dm.get_arg_voc_size(),
                   {s: {i: [g[i][0]] for i in g} for s, g in gold.items()})

    def get_arg_voc_size(self):
        return self._N

    def get_dimensionality(self):
        return self._F

    def get_neg_sampling_cum(self):
        return self.negSamplingCum

    def generate_split_keys(self):
        for _ in SPLIT_LABELS:
            if _ in self.split:
                yield _

    def save_npz(self, path):
        arrays = dict(neg_cum=self.negSamplingCum, F=np.int64(self._F), N=np.int64(self._N))
        for s, sp_ in self.split.items():
            arrays[s + '_indptr'] = sp_.indptr
            arrays[s + '_indices'] = sp_.indices
            arrays[s + '_args1'] = np.asarray(sp_.args1, dtype=np.int32)
            arrays[s + '_args2'] = np.asarray(sp_.args2, dtype=np.int32)
            g = self.goldStandard.get(s, {})
            arrays[s + '_gold'] = np.array([g.get(i, [''])[0] for i in range(sp_.get_size())], dtype='U')
        np.savez_compressed(path, **arrays)

    @classmethod
    def load_npz(cls, path):
        import scipy.sparse as sp
        z = np.load(path, allow_pickle=False)
        F, N = int(z['F']), int(z['N'])
        splits, gold = {}, {}
        for s in SPLIT_LABELS:
            if s + '_indptr' not in z.files:
                continue
            indptr, indices = z[s + '_indptr'], z[s + '_indices']
            x = sp.csr_matrix((np.ones(len(indices), dtype=np.float32), indices, indptr), shape=(len(indptr) - 1, F))
            splits[s] = DatasetSplit(z[s + '_args1'], z[s + '_args2'], x)
            gold[s] = {i: [str(t)] for i, t in enumerate(z[s + '_gold'])}
        return cls(splits, z['neg_cum'], F, N, gold)
