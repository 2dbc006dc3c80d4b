"""Tab-separated corpus -> pickled dataset, same command line and file format as the reference's
``processing/OiePreprocessor.py`` (run once per split; the pickle is extended in place).

    python -m relation_autoencoder_b200.preprocess --batch train data-sample.txt sample.pk
    python -m relation_autoencoder_b200.preprocess --batch valid data-sample.txt sample.pk
    python -m relation_autoencoder_b200.preprocess --batch test  data-sample.txt sample.pk

Restated here (not on the GPU path; pure string work):
  * ``read_examples``            OiePreprocessor.py:211-241   (9 tab-separated fields per line)
  * the nine default extractors  OieFeatures.py:247-263 -> trigger, entityTypes, arg1_lower, arg2_lower, bow_clean,
                                 entity1Type, entity2Type, lexicalPattern, posPatternPath  (OieFeatures.py:27-44,132-245)
  * lexicon build + thresholding OiePreprocessor.py:113-208,244-287
  * ``featurize``                new sentences through a trained model's frozen lexicon (export.py; no reference
                                 counterpart: the reference's preprocessor only grows the lexicon)
Stated divergences: (1) the reference takes its English stop-word list from NLTK (``OieFeatures.py:19``), which is not
installed here - the list is embedded below (NLTK's 153-word list of that era); (2) Python 3 strings: ``lower()`` also
lowers non-ASCII letters, Python 2 byte strings did not; (3) ``--batch-name`` (README.md:33-35 spelling) is accepted next
to ``--batch`` and ``dev`` is stored as ``valid`` (the reference's own writer rejects the README's ``dev`` key,
OiePreprocessor.py:312-316).
"""
from __future__ import annotations

import argparse
import os
import re
import string
import time

from .data import FeatureLexicon, OieExample, pickle_objects, unpickle_objects

parsing, entities, trig, sentence, pos, docPath = 0, 1, 2, 3, 4, 5      # OieFeatures.py:9-14

STOPWORDS = frozenset("""i me my myself we our ours ourselves you your yours yourself yourselves he him his himself she her
hers herself it its itself they them their theirs themselves what which who whom this that these those am is are was
were be been being have has had having do does did doing a an the and but if or because as until while of at by for
with about against between into through during before after above below to from up down in out on off over under again
further then once here there when where why how all any both each few more most other some such no nor not only own
same so than too very s t can will just don should now d ll m o re ve y ain aren couldn didn doesn hadn hasn haven isn
ma mightn mustn needn shan shouldn wasn weren won wouldn""".split())
_digits = re.compile(r'\d')


def _strip_punctuation(word):
    # one strip per punctuation character, in string.punctuation order (OieFeatures.py:37-38): NOT strip(all at once)
    for pun in string.punctuation:
        word = word.strip(pun)
    return word


def _between(info, arg1, arg2):
    s = info[sentence]
    return s[s.find(arg1):s.rfind(arg2) + len(arg2)].split()


def bow_clean(info, arg1, arg2):
    """Lower-cased words from entity 1 to entity 2 (inclusive) without stop words and numbers (OieFeatures.py:27-44)."""
    tmp = []
    for word in _between(info, arg1, arg2):
        word = _strip_punctuation(word)
        if word != '':
            tmp.append(word.lower())
    return [w for w in tmp if w not in STOPWORDS and not _digits.search(w) and not w[0].isupper()]


def trigger(info, arg1, arg2):
    return info[trig].replace('TRIGGER:', '')


def entityTypes(info, arg1, arg2):
    return info[entities]


def entity1Type(info, arg1, arg2):
    return info[entities].split('-')[0]


def entity2Type(info, arg1, arg2):
    return info[entities].split('-')[1]


def arg1_lower(info, arg1, arg2):
    return arg1.lower()


def arg2_lower(info, arg1, arg2):
    return arg2.lower()


def lexicalPattern(info, arg1, arg2):
    """Words of the dependency path (every second token once the arrows are blanked), joined by '_' (OieFeatures.py:177-189)."""
    p = info[parsing].replace('->', ' ').replace('<-', ' ').split()
    return '_'.join(x for num, x in enumerate(p) if num % 2 != 0)


def posPatternPath(info, arg1, arg2):
    """POS tags strictly between the first occurrence of entity 1's last token and the first occurrence of entity 2's
    first token, joined by '_' (OieFeatures.py:207-232)."""
    words = info[sentence].split()
    postags = info[pos].split()
    assert len(postags) == len(words), 'error'
    if not words:
        return ''
    last1, first2 = arg1.split()[-1], arg2.split()[0]
    begin = next((i for i, w in enumerate(words) if w == last1), None)
    end = next((i for i, w in enumerate(words) if w == first2), None)
    if begin is None or end is None:
        return ''
    return '_'.join(postags[begin + 1:end]) if end > begin else ''


def getBasicCleanFeatures():
    """The reference's default extractor list, in its order (OieFeatures.py:247-263)."""
    return [trigger, entityTypes, arg1_lower, arg2_lower, bow_clean, entity1Type, entity2Type, lexicalPattern, posPatternPath]


FEATURE_FUNCTION_NAMES = frozenset(f.__name__ for f in getBasicCleanFeatures())


# ----------------------------------------------------------------------------------------------------------------------
def generate_feature_element(extractor_output):
    if type(extractor_output) == list:
        for _ in extractor_output:
            yield _
    else:
        yield extractor_output


def get_features(lexicon, feature_extractors, info, arg1=None, arg2=None, expand=False):
    """Ids of every extracted 'name#value' string; ``expand`` adds unseen strings and counts frequencies
    (OiePreprocessor.py:120-150,189-196)."""
    feats = []
    for f in feature_extractors:
        res = f(info, arg1, arg2)
        if res is not None:
            for feat_el in generate_feature_element(res):
                key = f.__name__ + "#" + feat_el
                if expand:
                    feats.append(lexicon.get_or_add(key))
                else:
                    feat_id = lexicon.get_id(key)
                    if feat_id is not None:
                        feats.append(feat_id)
    return feats


def get_thresholded_features(lexicon, feature_extractors, info, arg1, arg2, threshold, expand=False):
    """Pruned ids of the extracted strings whose frequency exceeds ``threshold`` (OiePreprocessor.py:153-177,199-208)."""
    feats = []
    for f in feature_extractors:
        res = f(info, arg1, arg2)
        if res is not None:
            for feat_el in generate_feature_element(res):
                key = f.__name__ + "#" + feat_el
                feat_id = lexicon.get_id(key)
                if expand:
                    if lexicon.id2freq[feat_id] > threshold:        # KeyError(None) on an unseen string, as the reference
                        feats.append(lexicon.get_or_add_pruned(key))
                elif feat_id is not None and lexicon.id2freq[feat_id] > threshold:
                    feats.append(lexicon.get_or_add_pruned(key))
    return feats


def read_examples(file_name, verbose=True):
    """[[counter, field_1 .. field_9], ...] from a tab-separated file (OiePreprocessor.py:211-241)."""
    start = time.time()
    relation_examples = []
    with open(file_name, 'r', encoding='utf-8', errors='replace') as fp:
        for count, line in enumerate(fp):
            if len(line) == 0 or len(line.split()) == 0:
                raise IOError("empty line %d in %s" % (count, file_name))
            fields = line.split('\t')
            assert len(fields) == 9, "a problem with the file format (# fields is wrong) len is " + str(len(fields)) + "instead of 9"
            relation_examples.append([str(count)] + fields)
    if verbose:
        print('  File contained {} lines'.format(len(relation_examples)))
        print('  Done in {:.2f} sec'.format(time.time() - start))
    return relation_examples


def _info(feats):
    return [feats[1], feats[4], feats[5], feats[7], feats[8], feats[6]]


def build_feature_lexicon(raw_features, feature_extractors, lexicon, verbose=True):
    """First pass: every feature string gets an id and a frequency (OiePreprocessor.py:113-118)."""
    for ex_f in raw_features:
        get_features(lexicon, feature_extractors, _info(ex_f), ex_f[2], ex_f[3], expand=True)
    if verbose:
        print('  Lexicon now has {} unique entries'.format(lexicon.nextId))


def load_features(raw_features_struct, lexicon, feature_extractors, examples_list, labels_dict, threshold, verbose=True):
    """Second pass: thresholded ids -> OieExample, gold label tokens -> labels_dict (OiePreprocessor.py:244-287)."""
    index = 0
    for feats in raw_features_struct:
        feat_ids = get_thresholded_features(lexicon, feature_extractors, _info(feats), feats[2], feats[3],
                                            expand=True, threshold=threshold)
        examples_list.append(OieExample(feats[2], feats[3], feat_ids, feats[5], relation=feats[9]))
        labels_dict[index] = feats[-1].strip().split(' ')
        index += 1
    if verbose:
        print('  Unique thresholded feature keys: {}'.format(lexicon.nextIdPruned))


def featurize(input_file, feature_lex, feature_names, verbose=False):
    """New sentences through a trained model's FROZEN lexicon -> ([OieExample], {index: [gold tokens]}).

    Same 9-field file as :func:`read_examples`; the extractors are the defaults named by the dataset's object 1
    (``feature_names``: names or the stored extractor objects).  Every extracted 'name#value' string keeps the pruned id
    the lexicon gave it and is dropped when it has none, so the feature space (F) stays the one the model was trained
    on.  The lexicon is only read.  A line whose strings are all unknown gives an example without features."""
    names = [getattr(f, '__name__', f) for f in feature_names]
    unknown = [n for n in names if n not in FEATURE_FUNCTION_NAMES]
    if unknown:
        raise ValueError('feature extractors %r are not among the defaults %s: new text cannot be featurised like the dataset'
                         % (unknown, sorted(FEATURE_FUNCTION_NAMES)))
    by_name = {f.__name__: f for f in getBasicCleanFeatures()}
    extractors = [by_name[n] for n in names]
    examples, gold = [], {}
    for index, feats in enumerate(read_examples(input_file, verbose=verbose)):
        ids = []
        for f in extractors:
            res = f(_info(feats), feats[2], feats[3])
            if res is not None:
                for feat_el in generate_feature_element(res):
                    feat_id = feature_lex.str2IdPruned.get(f.__name__ + "#" + feat_el)
                    if feat_id is not None:
                        ids.append(feat_id)
        examples.append(OieExample(feats[2], feats[3], ids, feats[5], relation=feats[9]))
        gold[index] = feats[-1].strip().split(' ')
    return examples, gold


def preprocess(input_file, pickled_dataset, batch='train', threshold=0, verbose=True):
    """One run of the reference's ``__main__`` (OiePreprocessor.py:377-414)."""
    if batch == 'dev':
        batch = 'valid'
    exs_raw_features = read_examples(input_file, verbose=verbose)
    feat_extractors = getBasicCleanFeatures()
    relation_lexicon = FeatureLexicon()
    dataset, goldstandard = {}, {}
    if os.path.exists(pickled_dataset):
        _, relation_lexicon, dataset, goldstandard = unpickle_objects(pickled_dataset)
    if batch in dataset:
        examples, relation_labels = dataset[batch], goldstandard[batch]
    else:
        examples, relation_labels = [], {}
        dataset[batch], goldstandard[batch] = examples, relation_labels
    build_feature_lexicon(exs_raw_features, feat_extractors, relation_lexicon, verbose=verbose)
    load_features(exs_raw_features, relation_lexicon, feat_extractors, examples, relation_labels, threshold, verbose=verbose)
    pickle_objects(feat_extractors, relation_lexicon, dataset, goldstandard, pickled_dataset)
    return relation_lexicon, dataset, goldstandard


def get_cmd_arguments(argv=None):
    p = argparse.ArgumentParser(description='Processes an Oie file and add its representations to a Python pickled file.')
    p.add_argument('input_file', metavar='input-file', help='input file in the Yao format, like data-sample.txt')
    p.add_argument('pickled_dataset', metavar='pickled-dataset', help='pickle file to be used to store output (created if empty)')
    p.add_argument('--batch', '--batch-name', dest='batch', metavar='batch-name', default="train", nargs="?",
                   help="name used as a reference in the pickled file, default is 'train'")
    p.add_argument('--thres', metavar='threshold-value', default="0", nargs="?", type=int, help='minimum feature frequency')
    p.add_argument('--test-mode', action='store_true', help='accepted for compatibility (unused by the reference as well)')
    return p.parse_args(argv)


def main(argv=None):
    args = get_cmd_arguments(argv)
    preprocess(args.input_file, args.pickled_dataset, batch=args.batch, threshold=int(args.thres))


if __name__ == '__main__':
    main()
