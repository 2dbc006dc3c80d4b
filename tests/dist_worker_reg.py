"""Worker for tests/test_dist_regulariser.py: the row-sharded step with the L1/L2 regulariser, run under
torch.distributed.run (gloo + a float64 NumPy backend on CPU, NCCL + librae on GPUs), against the float64 oracle on the
global batch.

    dist_worker_reg.py MODEL OPTIMIZER L1 L2 EXT_REG [cuda] [--determinism]

On CPU one (optimizer, l1, l2, ext_reg) setting runs; with ``cuda`` the given setting and the two others of SETTINGS run,
each at K = 100 (16-byte rows) and K = 10 (scalar rows).  Every step also checks that some W row was touched by no rank,
that such rows moved, and that they moved by the regulariser alone.  ``--determinism`` runs the same two steps twice
from the same state and requires bit-identical shards and accumulators."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import rae_oracle as O  # noqa: E402
from relation_autoencoder_b200.dist import DistributedEngine  # noqa: E402
from tests.dist_numpy_backend import NumpyBackend  # noqa: E402
from tests.helpers import make_problem  # noqa: E402

# (optimizer, l1, l2, ext_reg): the reference's README / test.py setting, an L1-only setting without the decoder terms, SGD
SETTINGS = [("adagrad", 0.0, 0.1, True), ("adagrad", 0.01, 0.0, False), ("sgd", 0.0, 0.1, True)]


class RegNumpyBackend(NumpyBackend):
    """The owner-side passes of the regularised step in float64: the local regulariser value (own W shard, and the decoder
    tensors on rank 0), the decoder tensors' term added to the summed dense gradient, and W applied over the whole shard."""

    def _decoder(self):
        return [n for n in ("C", "C1", "C2") if n in self.order] if self.de.ext_reg else []

    def add_local_regulariser(self):
        de = self.de
        ts = [self.shards["W"].numpy()] + ([self.dense[n].numpy() for n in self._decoder()] if de.rank == 0 else [])
        L1 = sum(float(np.abs(t).sum()) for t in ts)
        L2 = sum(float(np.square(t).sum()) for t in ts)
        self._cost[0] += de.adj * (de.l1 * L1 + de.l2 * L2)

    def dense_apply(self):
        de = self.de
        off = 0
        for n in self.order:
            k = self.dense[n].numel()
            if n in self._decoder():
                p = self.dense[n].reshape(-1)
                self.dense_grad[off:off + k] += de.adj * (de.l1 * torch.sign(p) + 2.0 * de.l2 * p)
            off += k
        super().dense_apply()

    def shard_apply(self, name, table, acc, rows_local, ent_off, ent_src, ent_slot):
        de = self.de
        grads = self._all(self.grads[name])          # collective, as pull_apply
        t, a = table.numpy(), acc.numpy()
        g = np.zeros_like(t)
        rl, eo, es, el = rows_local.numpy(), ent_off.numpy(), ent_src.numpy(), ent_slot.numpy()
        for i in range(len(rl)):
            for e in range(eo[i], eo[i + 1]):        # rank order
                g[rl[i]] = g[rl[i]] + grads[es[e]][el[e]].numpy()
        g += de.adj * (de.l1 * np.sign(t) + 2.0 * de.l2 * t)
        if de.optimizer == "adagrad":
            a += g * g
            t -= de.lr * g / (np.sqrt(a) + 1e-6)
        else:
            t -= de.lr * g


def _untouched_w_rows(pr, g, Bg, F):
    ip = pr["indptr"]
    touched = np.unique(pr["indices"][ip[g * Bg]:ip[(g + 1) * Bg]])
    return np.setdiff1d(np.arange(F), touched)


def run(model, optimizer, l1, l2, ext_reg, cuda, K, rank, world, determinism=False):
    B, d, S, F, N, nb = (64, 32, 5, 3000, 900, 3) if cuda else (6, 4, 3, 40, 23, 3)
    Bg = B * world
    lr, alpha = 0.1, 0.7
    pr = make_problem(model, B=Bg * nb, K=K, d=d, S=S, F=F, N=N, seed=5, dup_heavy=True)
    p0 = {k: v.astype(np.float32).astype(np.float64) for k, v in pr["p"].items()}
    rows = np.concatenate([np.arange(g * Bg + rank * B, g * Bg + (rank + 1) * B) for g in range(nb)])
    ip = pr["indptr"]
    loc_ip = [0]
    loc_ix = []
    for r in rows:
        loc_ix.extend(pr["indices"][ip[r]:ip[r + 1]].tolist())
        loc_ip.append(len(loc_ix))
    de = DistributedEngine(model, K, d, S, B, F, N, n_train=Bg * nb, lr=lr, l1=l1, l2=l2, alpha=alpha, optimizer=optimizer,
                           ext_reg=ext_reg, rank=rank, world=world, device=int(os.environ.get("LOCAL_RANK", "0")),
                           backend_factory=None if cuda else RegNumpyBackend,
                           peer_dense_max_bytes=int(os.environ.get("RAE_TEST_PEER_DENSE_MAX", str(16 << 20))))
    de.set_params_numpy(p0)
    de.bind_split("train", np.asarray(loc_ip), np.asarray(loc_ix), pr["a1"][rows], pr["a2"][rows])
    de.bind_epoch_negatives(pr["neg1"][:, rows], pr["neg2"][:, rows])
    ok = True
    what = "%s %s l1=%g l2=%g ext_reg=%d K=%d world=%d" % (model, optimizer, l1, l2, ext_reg, K, world)

    if determinism:
        runs = []
        for _ in range(2):
            de.set_params_numpy(p0)
            for g in range(2):
                de.train_device(g)
            runs.append((de.get_params_numpy(), de.get_acc_numpy()))
        for n in O.param_names(model):
            ok &= np.array_equal(runs[0][0][n], runs[1][0][n]) and np.array_equal(runs[0][1][n], runs[1][1][n])
        if not ok and rank == 0:
            print("not bit-identical:", what)
        de.close()
        return ok

    om = O.OracleModel(model, {k: v.copy() for k, v in p0.items()}, K=K, d=d, S=S, B=Bg, lr=lr, l1=l1, l2=l2, alpha=alpha,
                       optimizer=optimizer, ext_reg=ext_reg)
    om.bind_split("train", pr["indptr"], pr["indices"], pr["a1"], pr["a2"])
    adj = de.adj
    assert abs(adj - om.adj) < 1e-15
    for g in range(nb):
        before = {k: v.astype(np.float64) for k, v in de.get_params_numpy().items()}
        acc_before = {k: v.astype(np.float64) for k, v in de.get_acc_numpy().items()}
        if cuda:     # fp32 path: every step is checked from the GPUs' current state (see tests/dist_worker.py)
            om.params = {k: v.copy() for k, v in before.items()}
            om.acc = {k: v.copy() for k, v in acc_before.items()}
        if g == 1:   # the reference-style call with host negatives
            c = de.train(g, pr["neg1"][:, rows[g * B:(g + 1) * B]], pr["neg2"][:, rows[g * B:(g + 1) * B]])
        else:
            c = de.train_device(g)
        c_ref = om.train(g, pr["neg1"][:, g * Bg:(g + 1) * Bg], pr["neg2"][:, g * Bg:(g + 1) * Bg])
        got = de.get_params_numpy()
        acc = de.get_acc_numpy()
        fails = []

        def check(cond, name):
            if not bool(cond):
                fails.append(name)
        if cuda:
            check(abs(c - c_ref) <= 1e-5 * max(1.0, abs(c_ref)), "cost %r vs %r" % (c, c_ref))
            for n in O.param_names(model):
                ea = np.abs(acc[n] - om.acc[n]).max() / max(np.abs(om.acc[n]).max(), 1e-30)
                check(ea <= 1e-4, "acc %s rel %.3g" % (n, ea))
                diff = np.abs(got[n] - om.params[n])
                tol = 1e-5 * max(1.0, np.abs(om.params[n]).max())
                frac = np.mean(diff <= tol)
                # AdaGrad's step lr*g/(sqrt(a + g^2) + 1e-6) is sign-like for |g| near 1e-6 from a small accumulator: there
                # it magnifies the gradient's fp32 rounding by |dp'/dg|.  "99.9 % within tol" allows for that in large
                # tensors; in a tensor of a few hundred elements (K = 10) each element beyond tol must instead be
                # explained by that magnification of a gradient error of 1e-5 * max|g|
                out = diff > tol
                if out.any() and optimizer == "adagrad":
                    gr = om.last_grads[n][out]
                    sq = np.sqrt(om.acc[n][out])
                    sens = lr * ((om.acc[n][out] - gr * gr) / np.maximum(sq, 1e-30) + 1e-6) / (sq + 1e-6) ** 2
                    explained = bool(np.all(diff[out] <= tol + sens * 1e-5 * np.abs(om.last_grads[n]).max()))
                else:
                    explained = not out.any()
                check((frac > 0.999 or explained) and diff.max() < 5e-3, "param %s within %.5f, max %.3g" % (n, frac, diff.max()))
        else:
            check(abs(c - c_ref) < 1e-12 * max(1.0, abs(c_ref)), "cost %r vs %r" % (c, c_ref))
            for n in O.param_names(model):
                check(np.abs(got[n] - om.params[n]).max() < 1e-12, "param " + n)
                check(np.abs(acc[n] - om.acc[n]).max() < 1e-12, "acc " + n)
        # a W row no rank touched has data gradient 0: it moves, by the regulariser alone
        un = _untouched_w_rows(pr, g, Bg, F)
        check(un.size > 0, "no untouched W row")
        w0, w1 = before["W"][un], got["W"][un].astype(np.float64)
        check(np.all(np.any(w1 != w0, axis=1)), "an untouched W row did not move")
        check(np.abs(w1 - om.params["W"][un]).max() <= (1e-5 if cuda else 1e-12), "untouched W rows vs oracle")
        g_reg = adj * (l1 * np.sign(w0) + 2.0 * l2 * w0)
        if optimizer == "adagrad":
            a1 = acc["W"][un].astype(np.float64)
            check(np.all(np.abs(a1 - (acc_before["W"][un] + g_reg * g_reg)) <= 1e-6 * np.abs(a1)), "untouched W acc rule")
        else:
            check(np.all(np.abs(w1 - (w0 - lr * g_reg)) <= 1e-6 * np.abs(w1) + 1e-12), "untouched W SGD rule")
        if fails and rank == 0:
            print("mismatch at step", g, what, "|", "; ".join(fails))
        ok &= not fails
    de.close()
    return ok


def main():
    args = [a for a in sys.argv[1:] if not a.startswith("--")]
    determinism = "--determinism" in sys.argv
    model, optimizer, l1, l2, ext_reg = args[0], args[1], float(args[2]), float(args[3]), args[4] == "1"
    cuda = len(args) > 5 and args[5] == "cuda"
    if cuda:
        lr_ = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(lr_)
        dist.init_process_group("nccl", device_id=torch.device("cuda", lr_))
    else:
        dist.init_process_group("gloo")
    rank, world = dist.get_rank(), dist.get_world_size()
    first = (optimizer, l1, l2, ext_reg)
    if not cuda:
        cases = [(first, 5)]
    elif determinism:
        cases = [(first, 100)]
    else:
        cases = [(s, K) for s in [first] + [s for s in SETTINGS if s != first] for K in (100, 10)]
    ok = True
    for (opt, a, b, e), K in cases:
        ok &= run(model, opt, a, b, e, cuda, K, rank, world, determinism)
    flag = torch.tensor([1 if ok else 0], device="cuda" if cuda else "cpu")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print("DIST_REG_OK" if int(flag) == 1 else "DIST_REG_MISMATCH")
    dist.destroy_process_group()
    sys.exit(0 if int(flag) == 1 else 1)


if __name__ == "__main__":
    main()
