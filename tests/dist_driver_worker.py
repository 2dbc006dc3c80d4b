"""Worker for tests/test_dist_driver.py: the training driver (ReconstructInducer) on several ranks through
``distributed_backend``, run under torch.distributed.run - gloo + the float64 NumPy backend of tests/dist_worker_reg.py on
CPU, NCCL + librae on GPUs.

    dist_driver_worker.py readme                               README run, 3 epochs, both golden traces (CPU)
    dist_driver_worker.py ckpt DIR ORACLE_CKPT                 world-N checkpoint after epoch 1 -> DIR/dist; the oracle's
                                                               epoch-1 checkpoint resumed here to epoch 3 -> DIR/resumed (CPU)
    dist_driver_worker.py labels                               label_rows of a split wider than the compact table (CPU)
    dist_driver_worker.py cli DIR ARGS...                      the command line (relation_autoencoder_b200.induction.main)
    dist_driver_worker.py cuda-readme                          README run, 10 epochs, against the golden traces' bounds
    dist_driver_worker.py cuda-labels                          rae_label_shards against a single-GPU Engine on the gathered W
    dist_driver_worker.py cuda-between-steps                   labels between steps against the gathered parameters
    dist_driver_worker.py cuda-repro DIR                       two identical runs and a --device-sampler run: checkpoints

Rank 0 prints DRIVER_OK or DRIVER_MISMATCH (the ranks agree through an all-reduce of the verdict)."""
import io
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from relation_autoencoder_b200 import data as D  # noqa: E402
from relation_autoencoder_b200 import induction as I  # noqa: E402
from tests.dist_worker_reg import RegNumpyBackend  # noqa: E402
from tests.golden.make_readme_run import README_ARGS, SEED, run_readme  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
CUDA = False


def _indexed():
    return D.IndexedDataset.load_npz(os.path.join(GOLD, "data_sample_indexed.npz"))


def backend(ind):
    return I.distributed_backend(ind, backend_factory=None if CUDA else RegNumpyBackend)


def _device():
    return int(os.environ.get("LOCAL_RANK", "0")) if CUDA else 0


def _traced(ind):
    costs = []
    train = ind.func["train"]

    def traced(b, n1, n2):
        c = train(b, n1, n2)
        costs.append(float(c))
        return c
    ind.func["train"] = traced
    return costs


def _close(a, b, rtol):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and bool(np.all(np.abs(a - b) <= rtol * np.abs(b)))


# ---------------------------------------------------------------------------------------------------------------- CPU
def readme(fails):
    """The README run (global batch 100) at this world size, 3 epochs: the single-process oracle driver's golden trace."""
    for name in ("readme_run.json", "readme_run_l2_0.json"):
        gold = json.load(open(os.path.join(GOLD, name)))
        res, ind = run_readme(_indexed(), backend, epochs=3, lambda2=gold["config"]["lambda2"])
        if ind.batch_reps != {"train": 10, "valid": 10, "test": 10} or ind.world != dist.get_world_size():
            fails.append("%s: batch_reps %s world %d" % (name, ind.batch_reps, ind.world))
        if not _close(res["batch_costs"], gold["batch_costs"][:30], 1e-12):
            fails.append("%s: batch costs" % name)
        if not _close(res["train_error"], gold["train_error"][:3], 1e-12):
            fails.append("%s: training error" % name)
        for split in ("valid", "test"):
            if not _close(res["metrics"][split], gold["metrics"][split][:3], 1e-12):
                fails.append("%s: %s B-cubed %s vs %s" % (name, split, res["metrics"][split], gold["metrics"][split][:3]))
        ind._release()


def ckpt(fails, directory, oracle_ckpt):
    """World N -> file (after epoch 1), and the oracle's file -> world N (epochs 2 and 3).  The test compares both with the
    uninterrupted oracle run."""
    _, ind = run_readme(_indexed(), backend, epochs=1, lambda2=0.1)
    ind.save(os.path.join(directory, "dist"))
    ind._release()
    idx = _indexed()
    args = dict(README_ARGS, nb_epochs=3, lambda2=0.1)
    ind2 = I.ReconstructInducer(idx, idx.goldStandard, np.random.RandomState(SEED + 99), backend=backend, out=io.StringIO(),
                                device=_device(), **args)
    ind2.load(oracle_ckpt)
    ind2.compile_function()
    costs = _traced(ind2)
    ind2.learn(debug=False)
    ind2.save(os.path.join(directory, "resumed"))
    if ind2.rank == 0:
        json.dump(dict(batch_costs=costs, train_error=ind2.train_error_series, metrics=ind2.metrics),
                  open(os.path.join(directory, "resumed", "trace.json"), "w"))
    ind2._release()


def labels(fails):
    """label_rows through the generic fallback (GranularStep) on a valid split whose batches hold more distinct features
    than the compact table: chunked, and equal to the float64 oracle's labels on the full W."""
    from oracle import rae_oracle as O
    from relation_autoencoder_b200.dist import DistributedEngine
    from tests.helpers import make_problem
    rank, world = dist.get_rank(), dist.get_world_size()
    B, K, d, S, F, N, nb = 6, 5, 4, 2, 300, 30, 2
    tr = make_problem("rescal+sp", B=B * world * nb, K=K, d=d, S=S, F=F, N=N, fbar=3, seed=3)
    va = make_problem("rescal+sp", B=37, K=K, d=d, S=S, F=F, N=N, fbar=8, seed=4)    # rows of <= 15 features, batches of ~50
    p = {k: v.astype(np.float32).astype(np.float64) for k, v in tr["p"].items()}
    rows = np.concatenate([np.arange(g * B * world + rank * B, g * B * world + (rank + 1) * B) for g in range(nb)])
    ip = tr["indptr"]
    loc_ix = np.concatenate([tr["indices"][ip[r]:ip[r + 1]] for r in rows])
    loc_ip = np.concatenate([[0], np.cumsum(ip[rows + 1] - ip[rows])])
    de = DistributedEngine("rescal+sp", K, d, S, B, F, N, n_train=B * world * nb, rank=rank, world=world,
                           backend_factory=RegNumpyBackend)
    de.set_params_numpy(p)
    de.bind_split("train", loc_ip, loc_ix, tr["a1"][rows], tr["a2"][rows])
    de.bind_split("valid", va["indptr"], va["indices"])
    cap = de.backend.compact["W"].shape[0]
    vip = va["indptr"]
    widest = max(np.unique(va["indices"][vip[b * B]:vip[(b + 1) * B]]).size for b in range(37 // B))
    if widest <= cap:
        fails.append("the valid batches fit the compact table (%d <= %d)" % (widest, cap))
    om = O.OracleModel("rescal+sp", p, K=K, d=d, S=S, B=37)
    om.bind_split("valid", va["indptr"], va["indices"], va["a1"], va["a2"])
    lab_ref, q_ref = om.label("valid", 0)
    lo, hi = (3, 37) if rank == 0 else (0, 29)          # different row ranges, so different chunk counts per rank
    lab, q = de.label_rows("valid", lo, hi)
    if not (np.array_equal(lab.numpy(), lab_ref[lo:hi]) and np.abs(q.numpy() - q_ref[lo:hi]).max() < 1e-12):
        fails.append("label_rows(valid, %d, %d) vs oracle" % (lo, hi))
    lab2, q2 = de.label_rows("valid", lo, hi, probs=False)
    if q2 is not None or not np.array_equal(lab2.numpy(), lab.numpy()):
        fails.append("label_rows without probs")
    for b in range(37 // B):
        lb, qb = de.label("valid", b)
        if not np.array_equal(lb, lab_ref[b * B:(b + 1) * B]):
            fails.append("label(valid, %d)" % b)
    de.close()


def cli(fails, directory, argv):
    I.models_path = directory
    I.main(argv, backend=backend)


# ---------------------------------------------------------------------------------------------------------------- GPU
def cuda_readme(fails):
    """tests/test_driver.py::test_readme_run_on_cuda_matches_oracle_trace's bounds, through the sharded driver."""
    for name in ("readme_run.json", "readme_run_l2_0.json"):
        gold = json.load(open(os.path.join(GOLD, name)))
        res, ind = run_readme(_indexed(), backend, lambda2=gold["config"]["lambda2"], device=_device())
        c0 = abs(res["batch_costs"][0] - gold["batch_costs"][0]) / abs(gold["batch_costs"][0])
        e10 = (np.abs(np.array(res["batch_costs"][:10]) - np.array(gold["batch_costs"][:10])) / np.abs(gold["batch_costs"][:10])).max()
        te = (np.abs(np.array(res["train_error"]) - np.array(gold["train_error"])) / np.abs(gold["train_error"])).max()
        f1 = abs(res["metrics"]["test"][-1][0] - gold["metrics"]["test"][-1][0])
        if dist.get_rank() == 0:
            print("%s world %d: first cost rel %.3g, first 10 max rel %.3g, epoch error max rel %.3g, test F1 diff %.4f"
                  % (name, ind.world, c0, e10, te, f1))
        if not (c0 <= 1e-5 and e10 <= 1e-3 and te <= 2e-3 and f1 <= 0.03):
            fails.append("%s bounds" % name)
        if res["metrics"]["valid"] != res["metrics"]["test"]:
            fails.append("%s: valid != test" % name)
        ind._release()


def _problem(K, world, rank):
    """A train split of narrow rows (small compact table) and a valid split of wide ones."""
    from tests.helpers import make_problem
    B, d, S, F, N, nb = 32, 16, 3, 5000, 400, 3
    tr = make_problem("rescal+sp", B=B * world * nb, K=K, d=d, S=S, F=F, N=N, fbar=3, seed=7)
    va = make_problem("rescal+sp", B=1000, K=K, d=d, S=S, F=F, N=N, fbar=40, seed=8)
    rows = np.concatenate([np.arange(g * B * world + rank * B, g * B * world + (rank + 1) * B) for g in range(nb)])
    ip = tr["indptr"]
    loc_ix = np.concatenate([tr["indices"][ip[r]:ip[r + 1]] for r in rows])
    loc_ip = np.concatenate([[0], np.cumsum(ip[rows + 1] - ip[rows])])
    return dict(B=B, d=d, S=S, F=F, N=N, nb=nb, tr=tr, va=va, rows=rows, loc_ip=loc_ip, loc_ix=loc_ix)


def _sharded(model, K, pb, rank, world):
    from relation_autoencoder_b200.dist import DistributedEngine
    tr = pb["tr"]
    de = DistributedEngine(model, K, pb["d"], pb["S"], pb["B"], pb["F"], pb["N"], n_train=pb["B"] * world * pb["nb"], l2=0.1,
                           rank=rank, world=world, device=_device())
    de.set_params_numpy({k: v.astype(np.float32) for k, v in tr["p"].items()})
    de.bind_split("train", pb["loc_ip"], pb["loc_ix"], tr["a1"][pb["rows"]], tr["a2"][pb["rows"]])
    de.bind_split("valid", pb["va"]["indptr"], pb["va"]["indices"])
    return de


def _single_labels(model, K, pb, params, lo, hi):
    """Rows [lo, hi) of the valid split labelled by a single-GPU Engine holding the full W (one batch of hi - lo rows)."""
    from relation_autoencoder_b200.engine import Engine
    va = pb["va"]
    ip = va["indptr"]
    sub_ip = (ip[lo:hi + 1] - ip[lo]).astype(np.int32)
    sub_ix = va["indices"][ip[lo]:ip[hi]]
    eng = Engine(model, K, pb["d"], pb["S"], hi - lo, pb["F"], pb["N"], hi - lo, device=_device())
    eng.set_params_numpy(params)
    eng.bind_split("valid", sub_ip, sub_ix)
    lab, q = eng.label("valid", 0)
    eng.close()
    return lab, q


def cuda_labels(fails):
    rank, world = dist.get_rank(), dist.get_world_size()
    for K in (100, 10):                      # 16-byte rows, scalar rows
        pb = _problem(K, world, rank)
        de = _sharded("rescal+sp", K, pb, rank, world)
        tr = pb["tr"]
        de.bind_epoch_negatives(tr["neg1"][:, pb["rows"]], tr["neg2"][:, pb["rows"]])
        de.train_device(0)                   # labels of a trained W, not only of the initial one
        params = de.get_params_numpy()
        B = pb["B"]
        cap = de.backend.compact["W"].shape[0]
        vip, vix = pb["va"]["indptr"], pb["va"]["indices"]
        widest = max(np.unique(vix[vip[b * B]:vip[(b + 1) * B]]).size for b in range(1000 // B))
        if widest <= cap:
            fails.append("K=%d: the valid batches fit the compact table (%d <= %d)" % (K, widest, cap))
        for lo, hi in ((0, 1000), (37 + rank, 913)):         # n_rows > B; an indptr offset != 0
            lab_ref, q_ref = _single_labels("rescal+sp", K, pb, params, lo, hi)
            lab, q = de.label_rows("valid", lo, hi)
            if not (np.array_equal(lab.cpu().numpy(), lab_ref) and np.array_equal(q.cpu().numpy(), q_ref)):
                fails.append("K=%d rows [%d, %d): not bit-identical (labels %d differ, max |dq| %.3g)"
                             % (K, lo, hi, int((lab.cpu().numpy() != lab_ref).sum()), np.abs(q.cpu().numpy() - q_ref).max()))
            lab2, q2 = de.label_rows("valid", lo, hi, probs=False)
            if q2 is not None or not np.array_equal(lab2.cpu().numpy(), lab_ref):
                fails.append("K=%d rows [%d, %d) without probs" % (K, lo, hi))
        # func['label_valid'](b) on batches wider than the compact table (the parent commit raised here)
        lab_ref, q_ref = _single_labels("rescal+sp", K, pb, params, 0, 1000)
        for b in range(1000 // B):
            lb, qb = de.label("valid", b)
            if not (np.array_equal(lb, lab_ref[b * B:(b + 1) * B]) and np.array_equal(qb, q_ref[b * B:(b + 1) * B])):
                fails.append("K=%d label(valid, %d)" % (K, b))
                break
        de.close()


def cuda_between_steps(fails):
    """The --freq-eval pattern: labels taken between steps equal the labels of the parameters gathered after each step."""
    rank, world = dist.get_rank(), dist.get_world_size()
    K = 100
    pb = _problem(K, world, rank)
    de = _sharded("rescal+sp", K, pb, rank, world)
    tr = pb["tr"]
    de.bind_epoch_negatives(tr["neg1"][:, pb["rows"]], tr["neg2"][:, pb["rows"]])
    for g in range(pb["nb"]):
        if g == 1:
            B = pb["B"]
            cols = pb["rows"][g * B:(g + 1) * B]
            de.train(g, tr["neg1"][:, cols], tr["neg2"][:, cols])
        else:
            de.train_device(g)
        lab, q = de.label_rows("valid", 0, 1000)
        lab_ref, q_ref = _single_labels("rescal+sp", K, pb, de.get_params_numpy(), 0, 1000)
        if not (np.array_equal(lab.cpu().numpy(), lab_ref) and np.array_equal(q.cpu().numpy(), q_ref)):
            fails.append("after step %d" % g)
    de.close()


def cuda_repro(fails, directory):
    """Two identical world-N runs give bit-identical checkpoints; the --device-sampler run reproduces them."""
    paths = []
    for i, dev_smp in enumerate((False, False, True)):
        idx = _indexed()
        args = dict(README_ARGS, nb_epochs=2, lambda2=0.1, model_name="run%d" % i)
        ind = I.ReconstructInducer(idx, idx.goldStandard, np.random.RandomState(SEED), backend=backend, out=io.StringIO(),
                                   device=_device(), device_sampler=dev_smp, **args)
        ind.compile_function()
        ind.learn(debug=False)
        paths.append(ind.save(directory))
        ind._release()
    if dist.get_rank() == 0:
        z = [I.load_model(p) for p in paths]
        for i in (1, 2):
            for part in ("params", "acc"):
                for k, v in z[0][part].items():
                    if not np.array_equal(z[i][part][k], v):
                        fails.append("run %d: %s %s differs (max %.3g)" % (i, part, k, np.abs(z[i][part][k] - v).max()))
            if z[i]["config"]["train_error"] != z[0]["config"]["train_error"] or z[i]["config"]["metrics"] != z[0]["config"]["metrics"]:
                fails.append("run %d: training error / metrics differ" % i)


def main():
    global CUDA
    mode, rest = sys.argv[1], sys.argv[2:]
    CUDA = mode.startswith("cuda")
    if mode == "cli":
        dist.init_process_group("gloo")
    elif CUDA:
        lr_ = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(lr_)
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr_))
    else:
        dist.init_process_group("gloo")
    rank = dist.get_rank()
    fails = []
    try:
        if mode == "readme":
            readme(fails)
        elif mode == "ckpt":
            ckpt(fails, rest[0], rest[1])
        elif mode == "labels":
            labels(fails)
        elif mode == "cli":
            try:
                cli(fails, rest[0], rest[1:])
            except ValueError as e:          # a refused configuration: every rank reports it, nothing else runs
                print("rank %d refused: %s" % (rank, e), flush=True)
                dist.barrier()               # both messages are out before torchrun sees a rank fail
                dist.destroy_process_group()
                sys.exit(3)
        elif mode == "cuda-readme":
            cuda_readme(fails)
        elif mode == "cuda-labels":
            cuda_labels(fails)
        elif mode == "cuda-between-steps":
            cuda_between_steps(fails)
        elif mode == "cuda-repro":
            cuda_repro(fails, rest[0])
        else:
            raise SystemExit("unknown mode " + mode)
    except Exception as e:                   # reported through the verdict instead of leaving the peers waiting
        import traceback
        traceback.print_exc()
        fails.append("rank %d raised %r" % (rank, e))
    if fails:
        print("rank %d:" % rank, "; ".join(fails), flush=True)
    flag = torch.tensor([0 if fails else 1], device="cuda" if CUDA else "cpu")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("DRIVER_OK" if int(flag) == 1 else "DRIVER_MISMATCH", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 1 else 1)


if __name__ == "__main__":
    main()
