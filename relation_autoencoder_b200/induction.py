"""The training driver and command line of the reference (``learning/OieInduction.py``) on top of the CUDA engine.

    python -m relation_autoencoder_b200.induction sample.pk --model-name m --decoder rescal+sp --epochs 10 \
        --batch-size 100 --relations 10 --neg-samples 5 --l2 0.1 --alpha 0.1 --seed 2 --embed-size 10 --learning-rate 0.1

Both flag spellings are accepted: this fork's argparse names (``OieInduction.py:461-491``, incl. unique prefixes such as
``--ep 2 --emb 10 --dec rescal+sp`` used by ``test.py:20``) and the README's (``README.md:44``: ``--pickled_dataset
--model_name --model A|C|AC --optimization 1 --batch_size --relations_number --negative_samples_number
--l2_regularization --embed_size --learning_rate``).

``ReconstructInducer`` keeps the reference's constructor, ``compile_function`` / ``train`` / ``learn`` / ``save``
protocol and touches the model only through ``self.func['train'](batch_index, neg1, neg2) -> cost`` and
``self.func['label_'+split](batch_index) -> (labels, probs)`` (``OieInduction.py:146-155,189,207,216``), which are bound
to :class:`relation_autoencoder_b200.engine.Engine` (hand-written sm_100a kernels behind librae.so).  There is no CPU
fallback: without a CUDA device ``compile_function`` raises.  ``backend`` exists so the host logic (epoch loop, sampler
order, clustering, B-cubed) can be exercised by the CPU test-suite with an injected checker.

Parameter initialisation draws from the run's single ``RandomState`` in the reference's order: W (RelationClassifier.py:24),
A (OieModel.py:105), then the decoder normals (Bilinear.py:14 / SelectionalPreferences.py:13-14 / BilinearPlusSP.py:14-17).
Out of scope (stated in DESIGN.md): word2vec initialisation (``--ext-emb``, gensim) and the matplotlib plots.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import time
from collections import Counter
from typing import Callable, Dict, Optional

import numpy as np

from .data import SPLIT_LABELS, load_data
from .evaluation import construct_split_evaluator, get_clusters_sets
from .sampler import NegativeExampleGenerator

INIT_LOW, INIT_HIGH = -1.e-3, 1.e-3                  # settings.py:23-24
MODEL_ALIASES = {'A': 'rescal', 'C': 'sp', 'AC': 'rescal+sp', 'rescal': 'rescal', 'sp': 'sp', 'rescal+sp': 'rescal+sp'}
PARAM_ORDER = {'rescal': ['W', 'Wb', 'C', 'A', 'Ab'],                 # RelationClassifier.py:26 + Bilinear.py:20
               'sp': ['W', 'Wb', 'A', 'C1', 'C2', 'Ab'],             # SelectionalPreferences.py:22
               'rescal+sp': ['W', 'Wb', 'C', 'A', 'Ab', 'C1', 'C2']}  # BilinearPlusSP.py:32

models_path = os.path.join(os.getcwd(), 'train_products')            # settings.py:5 (relative to the run directory here)


def init_parameters(rng, model, F, K, N, d, dtype=np.float32) -> Dict[str, np.ndarray]:
    """Reference initialisation, in the reference's RNG draw order (see module docstring)."""
    p = {}
    p['W'] = np.asarray(rng.uniform(low=INIT_LOW, high=INIT_HIGH, size=(F, K)), dtype=dtype)
    p['Wb'] = np.zeros(K, dtype=dtype)
    p['A'] = np.asarray(rng.uniform(-0.01, 0.01, size=(N, d)), dtype=dtype)
    sd = math.sqrt(0.1)
    if model in ('rescal', 'rescal+sp'):
        p['C'] = np.asarray(rng.normal(0, sd, size=(d, d, K)), dtype=dtype)
    if model in ('sp', 'rescal+sp'):
        p['C1'] = np.asarray(rng.normal(0, sd, size=(d, K)), dtype=dtype)
        p['C2'] = np.asarray(rng.normal(0, sd, size=(d, K)), dtype=dtype)
    p['Ab'] = np.zeros(N, dtype=dtype)
    return p


def cuda_backend(inducer: "ReconstructInducer") -> Dict[str, Callable]:
    """func['train'] / func['label_<split>'] bound to the CUDA engine (the product path)."""
    from .engine import Engine
    data = inducer.data
    tr = data.split['train']
    eng = Engine(inducer.decoder_type, inducer.relationNum, inducer.embedSize, inducer.neg_sample_num, inducer.batch_size,
                 data.get_dimensionality(), data.get_arg_voc_size(), tr.get_size(), lr=inducer.learningRate,
                 l1=inducer.lambdaL1, l2=inducer.lambdaL2, alpha=inducer.alpha, optimizer=inducer.optimization,
                 ext_reg=inducer.extendedReg, device=inducer.device)
    eng.set_params_numpy(inducer.initial_params, inducer.initial_acc)     # initial_acc: AdaGrad state of a resumed run, else None
    func = {}
    for split in data.generate_split_keys():
        sp = data.split[split]
        eng.bind_split(split, sp.indptr, sp.indices, sp.args1 if split == 'train' else None, sp.args2 if split == 'train' else None)
        func['label_' + split] = (lambda b, _s=split: eng.label(_s, b))
    func['train'] = eng.train
    inducer.engine = eng
    inducer.get_parameters = eng.get_params_numpy
    inducer.get_accumulators = eng.get_acc_numpy
    return func


def check_global_batch(batch_size: int, world: int):
    """--batch-size is the GLOBAL batch: every rank trains batch_size / world examples of it."""
    if batch_size % world != 0:
        raise ValueError("--batch-size %d is not divisible by the world size %d: each of the %d ranks trains batch-size / "
                         "world examples of every global batch" % (batch_size, world, world))


class _RankEngine(object):
    """The inducer's handle on this rank's :class:`relation_autoencoder_b200.dist.DistributedEngine`: ``learn()`` hands it
    the epoch's full negative arrays and global-batch slices, it passes on this rank's columns.  ``version`` counts the
    parameter changes (steps, loads), so labels gathered for one state are reused until the next change."""

    def __init__(self, de, rows, rank, B):
        self.de, self.rows, self.rank, self.B = de, rows, rank, B
        self._rows_dev = None
        self.version = 0

    def _cols(self, neg):
        if isinstance(neg, np.ndarray):
            return neg[:, self.rows]
        if self._rows_dev is None or self._rows_dev.device != neg.device:
            import torch
            self._rows_dev = torch.as_tensor(self.rows, device=neg.device)
        return neg[:, self._rows_dev]

    def bind_epoch_negatives(self, neg1, neg2):
        """Collective: the epoch's [S, n_train] arrays, identical on every rank; this rank's columns are bound."""
        self.de.bind_epoch_negatives(self._cols(neg1), self._cols(neg2))

    def train(self, batch_index, neg1, neg2):
        """func['train'] on the global batch's [S, Bg] slices: this rank's columns go to the engine, the GLOBAL cost returns."""
        lo, hi = self.rank * self.B, (self.rank + 1) * self.B
        self.version += 1
        return self.de.train(batch_index, neg1[:, lo:hi], neg2[:, lo:hi])

    def train_device(self, batch_index, want_cost=True):
        self.version += 1
        return self.de.train_device(batch_index, want_cost)

    def set_params_numpy(self, params, acc=None):
        self.version += 1
        self.de.set_params_numpy(params, acc)

    def get_params_numpy(self):
        return self.de.get_params_numpy()

    def get_acc_numpy(self):
        return self.de.get_acc_numpy()

    def close(self):
        self.de.close()


def distributed_backend(inducer: "ReconstructInducer", backend_factory=None, group=None) -> Dict[str, Callable]:
    """The contract of :func:`cuda_backend` on the ranks of a process group (one process per GPU of one node), through
    :class:`relation_autoencoder_b200.dist.DistributedEngine`.  Collective: every rank calls it, and then the driver, with
    the same arguments and the same seeded generator.

    The reference's global-batch semantics at any world size: ``batch_size`` is the global batch Bg, each rank trains
    B = Bg / world rows of it - global batch g is rows [g*Bg, (g+1)*Bg) and rank r trains rows [g*Bg + r*B, g*Bg + (r+1)*B).
    The tail is dropped as in the reference, adj = Bg / N_train and Z is global.  Every rank draws the same epoch negatives
    and binds its own columns.  ``func['label_<split>']`` returns the labels of the global batch (probs: None); the first
    call after a parameter change labels the split's batch_reps * Bg rows, a share per rank (``label_rows``, no collective
    with the CUDA backend), and all-gathers them into global order, so clustering and B-cubed see the single-process
    vector.  ``backend_factory``: the local-compute backend of the engine (the CPU tests inject a float64 NumPy one)."""
    import torch
    import torch.distributed as dist

    from .dist import DistributedEngine
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    Bg = inducer.batch_size
    check_global_batch(Bg, world)
    B = Bg // world
    data = inducer.data
    tr = data.split['train']
    nb = inducer.batch_reps['train']
    rows = (np.arange(nb, dtype=np.int64)[:, None] * Bg + rank * B + np.arange(B, dtype=np.int64)[None, :]).reshape(-1)
    ip = np.asarray(tr.indptr, dtype=np.int64)
    counts = ip[rows + 1] - ip[rows]
    loc_ip = np.zeros(rows.size + 1, dtype=np.int64)
    loc_ip[1:] = np.cumsum(counts)
    loc_ix = np.asarray(tr.indices)[np.repeat(ip[rows] - loc_ip[:-1], counts) + np.arange(loc_ip[-1], dtype=np.int64)]
    de = DistributedEngine(inducer.decoder_type, inducer.relationNum, inducer.embedSize, inducer.neg_sample_num, B,
                           data.get_dimensionality(), data.get_arg_voc_size(), tr.get_size(), lr=inducer.learningRate,
                           l1=inducer.lambdaL1, l2=inducer.lambdaL2, alpha=inducer.alpha, optimizer=inducer.optimization,
                           ext_reg=inducer.extendedReg, device=inducer.device, backend_factory=backend_factory, group=group)
    de.set_params_numpy(inducer.initial_params, inducer.initial_acc)
    de.bind_split('train', loc_ip, loc_ix, np.asarray(tr.args1)[rows], np.asarray(tr.args2)[rows])
    for split in data.generate_split_keys():
        if split != 'train':
            de.bind_split(split, data.split[split].indptr, data.split[split].indices)
    eng = _RankEngine(de, rows, rank, B)

    def gather_labels(split):
        """This split's labels of rows [0, batch_reps * Bg) in global order, on every rank (collective)."""
        n_share = inducer.batch_reps[split] * B
        if split == 'train':                  # this rank's own bound rows: the layout above gives their global order
            mine, _ = de.label_rows('train', 0, n_share, probs=False)
        else:
            mine, _ = de.label_rows(split, rank * n_share, (rank + 1) * n_share, probs=False)
        parts = [torch.empty_like(mine) for _ in range(world)] if world > 1 else [mine]
        if world > 1:
            dist.all_gather(parts, mine, group=group)
        out = torch.stack(parts)              # [world, n_share]
        if split == 'train':
            out = out.reshape(world, -1, B).transpose(0, 1)
        return out.reshape(-1).cpu().numpy()

    cache = {}

    def label(split, b):
        if cache.get(split, (None,))[0] != eng.version:
            cache[split] = (eng.version, gather_labels(split))
        return cache[split][1][b * Bg:(b + 1) * Bg], None

    func = {'label_' + split: (lambda b, _s=split: label(_s, b)) for split in data.generate_split_keys()}
    func['train'] = eng.train
    inducer.engine = eng
    inducer.get_parameters = eng.get_params_numpy
    inducer.get_accumulators = eng.get_acc_numpy
    inducer.sharded, inducer.rank, inducer.world, inducer.dist_group = True, rank, world, group
    return func


class ReconstructInducer(object):
    def __init__(self, data, gold_standard, rng, nb_epochs, learning_rate, batch_size, embed_size, nb_relations,
                 nb_neg_samples, lambda1, lambda2, optimization, model_name, decoder_model, external_embeddings,
                 extended_regularizer, frequent_eval, alpha, backend: Optional[Callable] = None, device: int = 0,
                 out=None, device_sampler: bool = False):
        if decoder_model not in MODEL_ALIASES:
            raise ValueError("unknown decoder %r (expected rescal | sp | rescal+sp)" % (decoder_model,))
        self.data = data
        self.goldStandard = gold_standard
        self.rng = rng
        self.nb_epochs = nb_epochs
        self.learningRate = learning_rate
        self.batch_size = batch_size
        self.embedSize = embed_size
        self.relationNum = nb_relations
        self.neg_sample_num = nb_neg_samples
        self.lambdaL1 = lambda1
        self.lambdaL2 = lambda2
        self.optimization = optimization
        self.modelName = model_name
        self.decoder_type = MODEL_ALIASES[decoder_model]
        self.extEmb = external_embeddings
        self.extendedReg = extended_regularizer
        self.frequentEval = frequent_eval
        self.alpha = alpha
        self.device = device
        # distributed_backend: the ranks of a process group (at any world size, 1 included), this process's rank of `world`
        self.sharded, self.rank, self.world, self.dist_group = False, 0, 1, None
        self.out = out if out is not None else sys.stdout
        self._backend = backend if backend is not None else cuda_backend
        if self.extEmb:
            raise NotImplementedError("--ext-emb (word2vec initialisation through gensim, OieModel.py:112-128) is out of scope")
        if optimization not in ('adagrad', 'sgd'):
            raise Exception("Optimizer '{}' not implemented".format(optimization))          # OieInduction.py:269
        # OieInduction.py:82.  device_sampler: same ids (same MT19937 stream), drawn and kept on the GPU; the epoch then
        # binds them once and steps with rae_train_step instead of passing host slices (cuda backend only)
        self.device_sampler = bool(device_sampler)
        if self.device_sampler:
            from .sampler import DeviceNegativeExampleGenerator
            self.negativeSampler = DeviceNegativeExampleGenerator(rng, data.negSamplingCum, device=device)
        else:
            self.negativeSampler = NegativeExampleGenerator(rng, data.negSamplingCum)
        self.modelID = decoder_model + '_' + model_name + '_maxepoch' + str(nb_epochs) + '_lr' + str(learning_rate) + \
            '_embedsize' + str(embed_size) + '_l1' + str(lambda1) + '_l2' + str(lambda2) + '_opt' + str(optimization) + \
            '_rel_num' + str(self.relationNum) + '_batch' + str(batch_size) + '_negs' + str(self.neg_sample_num)
        self.initial_params = init_parameters(rng, self.decoder_type, data.get_dimensionality(), nb_relations,
                                              data.get_arg_voc_size(), embed_size)           # OieInduction.py:88
        self.func = dict(zip([SPLIT_LABELS[0]] + ['label_' + s for s in SPLIT_LABELS], [None] * (1 + len(SPLIT_LABELS))))
        self.cur_epoch = 0
        self.initial_acc = None              # AdaGrad accumulators restored by load() before the functions are compiled
        self.evaluator = dict(zip(SPLIT_LABELS, [None] * len(SPLIT_LABELS)))
        for split in self.data.generate_split_keys():
            self.evaluator[split] = construct_split_evaluator(self.goldStandard[split], split)
        self.batch_reps = dict(zip(SPLIT_LABELS, [None] * len(SPLIT_LABELS)))
        for split in self.data.generate_split_keys():
            self.batch_reps[split] = self.data.split[split].args1.shape[0] // self.batch_size   # tail dropped, :96-98
        self.cluster = dict(zip(SPLIT_LABELS, [None] * len(SPLIT_LABELS)))
        self.train_error_series = []
        self.metrics = {s: [] for s in SPLIT_LABELS}
        self.engine = None
        self.get_parameters = lambda: {k: v.copy() for k, v in self.initial_params.items()}
        self.get_accumulators = lambda: {k: np.zeros_like(v) for k, v in self.initial_params.items()}

    def _print(self, *a):
        print(*a, file=self.out)

    def initialize(self):
        """Re-draws the parameters from the run's generator (OieInduction.py:104-108) and forgets the compiled functions."""
        self.initial_params = init_parameters(self.rng, self.decoder_type, self.data.get_dimensionality(), self.relationNum,
                                              self.data.get_arg_voc_size(), self.embedSize)
        self._release()
        self.func = dict(zip([SPLIT_LABELS[0]] + ['label_' + s for s in SPLIT_LABELS], [None] * (1 + len(SPLIT_LABELS))))

    def _release(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None

    def compile_function(self):
        """Binds ``self.func`` (OieInduction.py:118-155): dataset resident on the device, sliced by ``batch_index``."""
        self._print('Compiling...')
        self.func.update(self._backend(self))

    def train(self):
        t0 = time.perf_counter()
        if not self._check_for_compiled_functions():
            self.compile_function()
        compile_duration = time.perf_counter() - t0
        t0 = time.perf_counter()
        self.learn(debug=False)
        train_duration = time.perf_counter() - t0
        if self.rank == 0:
            print('Compiling completed in {:.1f}s'.format(compile_duration), file=sys.stderr)
            print('Training completed in {:.1f}s'.format(train_duration), file=sys.stderr)
        self._print('Trained for {} epochs. Avg epoch duration: {:.1f}s'.format(self.cur_epoch, train_duration / float(max(1, self.cur_epoch))))

    def learn(self, debug=True):
        """The epoch loop of OieInduction.py:172-222: two sampler calls per epoch (side 1, then side 2), one
        ``func['train']`` call per batch on the [S, B] column slices, per-epoch labelling + B-cubed."""
        n_train = self.data.split['train'].get_size()
        self._print('Training model on {} examples'.format(n_train))
        epoch = self.cur_epoch               # 0 for a fresh run; load() restores the epochs a resumed run has already done
        while epoch < self.nb_epochs:
            t_epoch = time.perf_counter()
            err = 0
            epoch += 1
            self.cur_epoch = epoch
            self._print('\nEPOCH', epoch)
            neg_samples1 = self.negativeSampler.get_negative_samples(self.data.split['train'].args1.shape[0], self.neg_sample_num)
            neg_samples2 = self.negativeSampler.get_negative_samples(self.data.split['train'].args2.shape[0], self.neg_sample_num)
            B = self.batch_size
            if self.device_sampler or self.sharded:
                # sharded: every rank drew the same arrays and binds its own columns, whichever the sampler
                self.engine.bind_epoch_negatives(neg_samples1, neg_samples2)
            for batch_ind in range(self.batch_reps['train']):
                if self.device_sampler:
                    err += self.engine.train_device(batch_ind)
                else:
                    neg1 = neg_samples1[:, batch_ind * B:(batch_ind + 1) * B]
                    neg2 = neg_samples2[:, batch_ind * B:(batch_ind + 1) * B]
                    err += self.func['train'](batch_ind, neg1, neg2)
                if self.frequentEval:
                    if self._mode() == 1:
                        self._print(batch_ind * B, batch_ind, '############################################################')
                        self._print(self.get_clusters_size(self.func['label_train'], self.batch_reps['train']), '\n')
                    elif self._mode() == 2:
                        self._print(batch_ind * B, batch_ind, '############################################################')
                        for split in SPLIT_LABELS[1:]:
                            self.cluster[split] = get_clusters_sets(self.func['label_' + split], self.batch_reps[split], self.relationNum)
                            self._evaluate(split, store=False)
            self.train_error_series.append(float(err))
            self._print('Training error: {:.4f}'.format(err))
            self._print('Epoch duration: {:.1f}s'.format(time.perf_counter() - t_epoch))
            if self._mode() == 1:
                self._print('Training Set')
                self.cluster['train'] = get_clusters_sets(self.func['label_train'], self.batch_reps['train'], self.relationNum)
                self._evaluate('train', store=True)
            if self._mode() == 2:
                for split in SPLIT_LABELS[1:]:
                    self.cluster[split] = get_clusters_sets(self.func['label_' + split], self.batch_reps[split], self.relationNum)
                    self._evaluate(split, store=True)

    def _evaluate(self, split, store=False):
        self.evaluator[split].feed_induced_clusters(self.cluster[split])
        f1, pre, rec = self.evaluator[split].compute_metrics()
        self._print('{} f1: {:.4f} pre: {:.4f} rec: {:.4f}'.format(split, f1, pre, rec))
        if store:
            self.metrics[split].append((f1, pre, rec))

    @staticmethod
    def compute_posteriors(labeling_func, batch_reps):
        """Rows of q(r|x) for every example of a split (OieInduction.py:240-250)."""
        return [row for i in range(batch_reps) for row in labeling_func(i)[1]]

    @staticmethod
    def get_clusters_size(labeling_func, nb_batches):
        """cluster id -> population (OieInduction.py:252-263)."""
        return Counter(int(item) for i in range(nb_batches) for item in labeling_func(i)[0])

    def _check_for_compiled_functions(self):
        if self.func.get('train') is None:
            return False
        return all(self.func.get('label_' + s) is not None for s in self.data.generate_split_keys())

    def _mode(self):
        """1: only 'train'; 2: 'train', 'valid' and 'test' (OieInduction.py:298-310)."""
        sp = self.data.split
        if len(sp) == 1 and 'train' in sp:
            return 1
        if len(sp) == 3 and 'train' in sp and 'valid' in sp and 'test' in sp:
            return 2
        raise Exception("Either 'train' split or 'train', 'valid' and 'test' splits should be defined")

    def save(self, directory: Optional[str] = None) -> str:
        """Portable checkpoint ``<models_path>/<model name>.npz``: parameters, AdaGrad accumulators (which the reference's
        pickle of ``self`` loses, OieInduction.py:110-116 + Optimizers.py:12-15) and the run configuration.  The format
        does not depend on the world size.  Several ranks: collective (the shards are gathered), rank 0 writes, and every
        rank returns once the file is complete."""
        directory = directory if directory is not None else models_path
        path = os.path.join(directory, self.modelName + '.npz')
        params, acc = self.get_parameters(), self.get_accumulators()
        if self.rank != 0:
            self._barrier()
            return path
        os.makedirs(directory, exist_ok=True)
        cfg = dict(decoder=self.decoder_type, relations=self.relationNum, embed_size=self.embedSize, batch_size=self.batch_size,
                   neg_samples=self.neg_sample_num, l1=self.lambdaL1, l2=self.lambdaL2, alpha=self.alpha, optimizer=self.optimization,
                   learning_rate=self.learningRate, epochs_done=self.cur_epoch, model_id=self.modelID, ext_reg=bool(self.extendedReg),
                   train_error=self.train_error_series, metrics=self.metrics)
        arrays = {'param_' + k: v for k, v in params.items()}
        arrays.update({'acc_' + k: v for k, v in acc.items()})
        # the run's generator feeds the negative sampler (OieInduction.py:183-184): its state is part of the run
        kind, keys, pos, has_gauss, cached = self.rng.get_state()
        arrays.update(rng_keys=np.asarray(keys, dtype=np.uint32), rng_pos=np.int64(pos), rng_has_gauss=np.int64(has_gauss),
                      rng_cached_gaussian=np.float64(cached))
        np.savez(path, config=np.array(json.dumps(cfg)), **arrays)
        self._barrier()
        return path

    def _barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier(group=self.dist_group)

    def load(self, path: str):
        """Resume from a checkpoint written by :meth:`save`: parameters, AdaGrad accumulators, the epoch counter, the
        error / metric series and the generator state, so that training continues exactly where the saved run stopped
        (works before or after the functions are compiled).  Any world size resumes a checkpoint of any other: each rank
        keeps its own rows (collective once compiled on several ranks)."""
        ck = load_model(path)
        if self.engine is None and getattr(self, 'oracle_model', None) is None:
            self.initial_params = {k: v for k, v in ck['params'].items()}
            self.initial_acc = {k: v for k, v in ck['acc'].items()} if ck['acc'] else None
        elif self.engine is not None:
            self.engine.set_params_numpy(ck['params'], ck['acc'])
        else:
            self.oracle_model.params = {k: np.asarray(v, dtype=np.float64) for k, v in ck['params'].items()}
            self.oracle_model.acc = {k: np.asarray(v, dtype=np.float64) for k, v in ck['acc'].items()}
        cfg = ck['config']
        self.cur_epoch = int(cfg.get('epochs_done', 0))
        self.train_error_series = list(cfg.get('train_error', []))
        for split, series in (cfg.get('metrics') or {}).items():
            self.metrics[split] = [tuple(m) for m in series]
        if ck.get('rng') is not None:
            self.rng.set_state(ck['rng'])
        return ck


def load_model(path: str):
    """{'config': dict, 'params': {...}, 'acc': {...}} from a checkpoint written by ``ReconstructInducer.save``."""
    if not os.path.exists(path) and os.path.exists(os.path.join(models_path, path)):
        path = os.path.join(models_path, path)
    z = np.load(path, allow_pickle=False)
    params = {k[len('param_'):]: z[k] for k in z.files if k.startswith('param_')}
    acc = {k[len('acc_'):]: z[k] for k in z.files if k.startswith('acc_')}
    rng = None
    if 'rng_keys' in z.files:
        rng = ('MT19937', z['rng_keys'], int(z['rng_pos']), int(z['rng_has_gauss']), float(z['rng_cached_gaussian']))
    return {'config': json.loads(str(z['config'])), 'params': params, 'acc': acc, 'rng': rng}


# ----------------------------------------------------------------------------------------------------------------------
# command line
# ----------------------------------------------------------------------------------------------------------------------
class _Parser(argparse.ArgumentParser):
    def _get_option_tuples(self, option_string):
        # a unique-prefix abbreviation that matches several spellings of the SAME option is not ambiguous
        found = super()._get_option_tuples(option_string)
        if len(found) > 1 and all(t[0] is found[0][0] for t in found):
            return found[:1]
        return found


def fix_parsing(bool_flag):
    if bool_flag == 'False' or bool_flag == 'True':
        return bool_flag == 'True'
    if type(bool_flag) == bool:
        return bool_flag
    raise Exception("Failed to parse '{}' of type '{}'".format(bool_flag, type(bool_flag)))


def get_command_args(program_name, argv=None):
    p = _Parser(prog=program_name, description='Trains a basic Open Information Extraction Model',
                formatter_class=argparse.ArgumentDefaultsHelpFormatter)
    p.add_argument('dataset', nargs='?', help='the pickled dataset file (produced by the preprocessor)')
    p.add_argument('--pickled_dataset', dest='dataset_opt', default=None, help='README.md:44 spelling of the dataset argument')
    p.add_argument('--epochs', type=int, default=100, help='the number of training epochs')
    p.add_argument('--learning-rate', '--learning_rate', dest='learning_rate', type=float, default=0.1, help='the initial learning rate')
    p.add_argument('--batch-size', '--batch_size', dest='batch_size', type=int, default=50, help='the size of the minibatches')
    p.add_argument('--embed-size', '--embed_size', dest='embed_size', type=int, default=30, help='the embedding space dimensionality')
    p.add_argument('--relations', '--relations_number', dest='relations', type=int, default=3, help='the number of semantic relation to induce')
    p.add_argument('--neg-samples', '--negative_samples_number', dest='neg_samples', type=int, default=5,
                   help='the number of negative samples to take per entity')
    p.add_argument('--l1', '--l1_regularization', dest='l1', metavar='lambda_1', type=float, default=0.0, help='the L1 coefficient')
    p.add_argument('--l2', '--l2_regularization', dest='l2', metavar='lambda_2', type=float, default=0.0, help='the L2 coefficient')
    p.add_argument('--optimizer', choices=['adagrad', 'sgd'], type=str, default='adagrad', help='the optimization algorithm')
    p.add_argument('--optimization', type=int, default=None, help='README.md:44 spelling: 0 = sgd, 1 = adagrad')
    p.add_argument('--model-name', '--model_name', dest='model_name', required=True, type=str, help='a name for the trained model')
    p.add_argument('--decoder', choices=['rescal', 'sp', 'rescal+sp'], type=str, default=None,
                   help='the factorization model used as the decoder (sp: selectional preferences)')
    p.add_argument('--model', choices=['A', 'C', 'AC'], default=None, help='README.md:44 spelling of --decoder')
    p.add_argument('--ext-emb', dest='ext_emb', action='store_true', default='False', help='use external embeddings')
    p.add_argument('--ext-reg', dest='ext_reg', action='store_true', default='True', help='regularize the decoder parameters as well')
    p.add_argument('--freq-eval', dest='freq_eval', action='store_true', default='False', help='use frequent evaluation')
    p.add_argument('--alpha', type=float, default=1.0, help='the alpha coefficient for scaling the entropy term')
    p.add_argument('--seed', type=int, default=2, help='a seed number')
    p.add_argument('--device', type=int, default=None, help='CUDA device index (default 0; several ranks use LOCAL_RANK)')
    p.add_argument('--device-sampler', dest='device_sampler', action='store_true',
                   help='draw the negative samples on the GPU (bit-identical ids, same random stream)')
    if argv is None:
        argv = sys.argv[1:]
    if len(argv) == 0:
        p.print_help()
        sys.exit(1)
    a = p.parse_args(argv)
    a.ext_emb = fix_parsing(a.ext_emb)
    a.ext_reg = fix_parsing(a.ext_reg)
    a.freq_eval = fix_parsing(a.freq_eval)
    if a.dataset is None:
        a.dataset = a.dataset_opt
    if a.dataset is None:
        p.error('the pickled dataset is required (positional, or --pickled_dataset)')
    if a.optimization is not None:
        if a.optimization not in (0, 1):
            raise Exception("Optimizer '{}' not implemented".format(a.optimization))
        a.optimizer = 'adagrad' if a.optimization == 1 else 'sgd'
    if a.decoder is None:
        a.decoder = MODEL_ALIASES[a.model] if a.model is not None else None
    if a.decoder is None:
        p.error('a decoder is required (--decoder rescal|sp|rescal+sp, or --model A|C|AC)')
    return a


def main(argv=None, backend=None):
    """The command line.  Under ``torchrun --nproc-per-node N`` (WORLD_SIZE > 1) every process trains on GPU LOCAL_RANK
    through :func:`distributed_backend`: NCCL is initialised here (unless the caller already formed the process group),
    ``--batch-size`` is the global batch, only rank 0 prints the training log and writes the checkpoint, and the process
    group is destroyed on the way out.  ``backend`` replaces the binding (cuda_backend, or distributed_backend on several
    ranks).  With WORLD_SIZE unset or 1 this is the single-GPU driver."""
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if world <= 1:
        return _run(argv, backend)
    import torch
    import torch.distributed as dist
    rank, local = int(os.environ['RANK']), int(os.environ.get('LOCAL_RANK', '0'))
    out = sys.stdout if rank == 0 else open(os.devnull, 'w')
    own_group = False
    try:
        args = get_command_args('induction', argv)
        if args.device is not None:
            raise ValueError("--device cannot be combined with several ranks: rank %d uses GPU LOCAL_RANK = %d" % (rank, local))
        check_global_batch(args.batch_size, world)
        if not dist.is_initialized():
            torch.cuda.set_device(local)
            dist.init_process_group('nccl', device_id=torch.device('cuda', local))
            own_group = True
        return _run(argv, backend if backend is not None else distributed_backend, out=out, device=local, rank=rank)
    finally:
        if own_group:
            dist.destroy_process_group()
        if out is not sys.stdout:
            out.close()


def _run(argv, backend, out=None, device=None, rank=0):
    out = out if out is not None else sys.stdout
    print("Relation Learner", file=out)
    args = get_command_args('induction', argv)
    rand = np.random.RandomState(seed=args.seed)
    indexed_data, gold_standard = load_data(args.dataset, rand, verbose=rank == 0)
    inducer = ReconstructInducer(indexed_data, gold_standard, rand, args.epochs, args.learning_rate, args.batch_size,
                                 args.embed_size, args.relations, args.neg_samples, args.l1, args.l2, args.optimizer,
                                 args.model_name, args.decoder, args.ext_emb, args.ext_reg, args.freq_eval, args.alpha,
                                 backend=backend, device=device if device is not None else (args.device or 0), out=out,
                                 device_sampler=args.device_sampler)
    inducer.train()
    path = inducer.save()
    print('Saved', path, file=out)
    if inducer.sharded:
        inducer._release()                # collective: the peer mappings go before the process group
    return inducer


if __name__ == '__main__':
    main()
