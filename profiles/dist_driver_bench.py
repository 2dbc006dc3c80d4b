"""Per-epoch time of the training driver on several GPUs (``distributed_backend``) at cfg2 sizes: AC, K = 100, d = 30, S = 5,
global batch 4096, 2M training examples of ~30 features, 1M feature rows, 500k entities, valid / test of 200k examples.

    python -m torch.distributed.run --nproc-per-node W profiles/dist_driver_bench.py OUT.json [--epochs 2]

``ReconstructInducer`` is built with ``distributed_backend``; the epoch is then run phase by phase as ``learn()`` runs it
(mode 2: train, then label valid and test and score them), each phase between two barriers and max-reduced over the ranks:
negative draw (host sampler, both sides), ``bind_epoch_negatives``, the steps, labelling (label_rows + all-gather + copy to
the host, both splits), B-cubed.  For labelling the ``rae_label_shards`` kernel alone is also timed with CUDA events on
each rank's share, with its bytes: nnz * K * 4 of W rows + the CSR slice + 8 B per label.  The last epoch is reported.
Rank 0 writes OUT.json with the card, its power limit and clocks, read in the same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import scipy.sparse as sp
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from relation_autoencoder_b200 import induction as I  # noqa: E402
from relation_autoencoder_b200 import synthetic as SY  # noqa: E402
from relation_autoencoder_b200.data import DatasetSplit, IndexedDataset  # noqa: E402
from relation_autoencoder_b200.evaluation import get_clusters_sets  # noqa: E402


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.sm,clocks.max.sm,clocks.mem",
                        "--format=csv,noheader"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip().splitlines()


def _split(n, wl, seed):
    d = SY.make_dataset(n, wl["F"], wl["N"], wl["fbar"], seed=seed)
    x = sp.csr_matrix((np.ones(d.indices.size, np.float32), d.indices, d.indptr), shape=(n, wl["F"]))
    return DatasetSplit(d.args1, d.args2, x), d.neg_cum


def dataset(n_train, n_eval):
    wl = dict(SY.WORKLOADS["cfg2"])
    splits, cum = {}, None
    for i, (name, n) in enumerate((("train", n_train), ("valid", n_eval), ("test", n_eval))):
        splits[name], c = _split(n, wl, 1234 + i)
        cum = c if name == "train" else cum
    rng = np.random.RandomState(5)
    gold = {}
    for name, s in splits.items():                   # 20 relations, a third of the examples unlabelled
        lab = rng.randint(0, 30, size=s.get_size())
        gold[name] = {i: ["" if lab[i] >= 20 else "/r/%d" % lab[i]] for i in range(s.get_size())}
    return IndexedDataset(splits, cum, wl["F"], wl["N"], gold), wl


def main():
    out_path = sys.argv[1]
    epochs = int(sys.argv[sys.argv.index("--epochs") + 1]) if "--epochs" in sys.argv else 2
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    t0 = time.perf_counter()
    data, wl = dataset(2_000_000, 200_000)
    t_data = time.perf_counter() - t0
    args = dict(nb_epochs=epochs, learning_rate=0.1, batch_size=4096, embed_size=wl["d"], nb_relations=wl["K"],
                nb_neg_samples=wl["S"], lambda1=0.0, lambda2=0.0, optimization="adagrad", model_name="bench",
                decoder_model=wl["model"], external_embeddings=False, extended_regularizer=True, frequent_eval=False, alpha=1.0)
    ind = I.ReconstructInducer(data, data.goldStandard, np.random.RandomState(2), backend=I.distributed_backend,
                               out=open(os.devnull, "w"), device=local, **args)
    t0 = time.perf_counter()
    ind.compile_function()
    t_compile = time.perf_counter() - t0
    de = ind.engine.de
    dev = torch.device("cuda", local)

    def phase(fn):
        torch.cuda.synchronize(dev)
        dist.barrier()
        t = time.perf_counter()
        r = fn()
        torch.cuda.synchronize(dev)
        dt = torch.tensor([time.perf_counter() - t], dtype=torch.float64, device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        return r, float(dt.item())

    Bg, n_train = ind.batch_size, data.split["train"].get_size()
    rows = []
    for epoch in range(epochs):
        (n1, n2), t_neg = phase(lambda: (ind.negativeSampler.get_negative_samples(n_train, ind.neg_sample_num),
                                         ind.negativeSampler.get_negative_samples(n_train, ind.neg_sample_num)))
        _, t_bind = phase(lambda: ind.engine.bind_epoch_negatives(n1, n2))

        def steps():
            err = 0.0
            for b in range(ind.batch_reps["train"]):
                err += ind.func["train"](b, n1[:, b * Bg:(b + 1) * Bg], n2[:, b * Bg:(b + 1) * Bg])
            return err
        err, t_steps = phase(steps)
        _, t_label = phase(lambda: [ind.func["label_" + s](0) for s in ("valid", "test")])

        def b3():
            for s in ("valid", "test"):
                ind.cluster[s] = get_clusters_sets(ind.func["label_" + s], ind.batch_reps[s], ind.relationNum)
                ind.evaluator[s].feed_induced_clusters(ind.cluster[s])
                ind.evaluator[s].compute_metrics()
        _, t_b3 = phase(b3)
        rows.append(dict(epoch=epoch + 1, training_error=err, negative_draw_s=t_neg, bind_epoch_negatives_s=t_bind,
                         steps_s=t_steps, n_steps=ind.batch_reps["train"], labelling_s=t_label, b3_s=t_b3))

    # the labelling kernel alone on this rank's share of one split
    s = "valid"
    n_share = ind.batch_reps[s] * de.B
    lo, hi = rank * n_share, (rank + 1) * n_share
    ip = data.split[s].indptr
    nnz = int(ip[hi] - ip[lo])
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    times = []
    for _ in range(5):
        ev[0].record()
        de.label_rows(s, lo, hi, probs=False)
        ev[1].record()
        torch.cuda.synchronize(dev)
        times.append(ev[0].elapsed_time(ev[1]) * 1e-3)
    t_k = float(np.median(times))
    bytes_k = nnz * wl["K"] * 4 + (hi - lo + 1) * 4 + nnz * 4 + (hi - lo) * 8
    kern = torch.tensor([t_k, bytes_k / t_k / 1e9], dtype=torch.float64, device=dev)
    gathered = [torch.empty_like(kern) for _ in range(world)]
    dist.all_gather(gathered, kern)
    if rank == 0:
        res = dict(world=world, config="cfg2 sizes: AC K=100 d=30 S=5, global batch 4096, 2M train / 200k valid / 200k test",
                   gpus=_card()[:world], dataset_build_s=t_data, compile_s=t_compile, epochs=rows,
                   label_kernel_per_rank=[dict(rank=r, rows=n_share, seconds=float(g[0]), gb_per_s=float(g[1]))
                                          for r, g in enumerate(gathered)],
                   label_kernel_bytes_per_rank_valid_share=bytes_k)
        json.dump(res, open(out_path, "w"), indent=1)
        last = rows[-1]
        print("world %d: neg %.2fs bind %.2fs steps %.2fs (%d) label %.3fs b3 %.2fs | label kernel %.2f ms %.0f GB/s"
              % (world, last["negative_draw_s"], last["bind_epoch_negatives_s"], last["steps_s"], last["n_steps"],
                 last["labelling_s"], last["b3_s"], t_k * 1e3, bytes_k / t_k / 1e9))
    ind._release()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
