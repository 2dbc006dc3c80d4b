"""Row-sharded multi-GPU training with the L1/L2 regulariser (OieModel.py:54-62, OieInduction.py:131-135).

CPU: the sharded step under gloo with a float64 NumPy backend against the float64 oracle on the global batch, and the
ctypes layout of rae_dist_step.  GPU: the same worker on librae (worlds 1, 2, 4; 16-byte and scalar W rows), the NCCL dense
path, world 1 against the single-GPU engine, determinism at world 2, and rae_shard_apply on crafted plans against an fp32
NumPy emulation of the rule."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from relation_autoencoder_b200 import _lib as L
from tests.test_dist_cpu import ROOT, _free_port

WORKER = os.path.join(ROOT, "tests", "dist_worker_reg.py")


def _run_worker(world, args, env=None, timeout=900):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), WORKER] + args
    env = dict(os.environ, OMP_NUM_THREADS="1", **(env or {}))
    r = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    assert r.returncode == 0 and "DIST_REG_OK" in r.stdout, r.stdout[-3000:]


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("setting", [("adagrad", "0", "0.1", "1"), ("adagrad", "0.01", "0", "0")], ids=["l2_ext", "l1_noext"])
@pytest.mark.parametrize("model", ["rescal", "sp", "rescal+sp"])
def test_two_rank_gloo_regularised_matches_oracle(model, setting):
    _run_worker(2, [model, *setting], timeout=600)


def test_two_rank_gloo_regularised_sgd_matches_oracle():
    _run_worker(2, ["rescal+sp", "sgd", "0", "0.1", "1"], timeout=600)


def test_dist_step_layout_matches_c(tmp_path):
    src = tmp_path / "sz.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "rae.h"\nint main(){printf("%zu %zu %zu\\n",'
                   'sizeof(rae_dist_step),offsetof(rae_dist_step,global_cost),offsetof(rae_dist_step,w_rows));return 0;}\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)]).decode().split()
    got = [C.sizeof(L.RaeDistStep), L.RaeDistStep.global_cost.offset, L.RaeDistStep.w_rows.offset]
    assert [int(x) for x in out] == got


# ---------------------------------------------------------------------------------------------------------------- GPU
def _ngpu():
    import torch
    return torch.cuda.device_count()


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4])
@pytest.mark.parametrize("model", ["rescal", "sp", "rescal+sp"])
def test_sharded_regularised_step_matches_oracle(model, world):
    """AdaGrad (l2 with ext_reg, l1 without) and SGD, each at K = 100 and K = 10, inside one worker run."""
    if _ngpu() < world:
        pytest.skip("needs %d GPUs" % world)
    _run_worker(world, [model, "adagrad", "0", "0.1", "1", "cuda"])


@pytest.mark.gpu
def test_sharded_regularised_step_with_nccl_dense_allreduce():
    """The decoder tensors' regulariser through rae_train_step_end's dense update (NCCL all-reduce of the gradient)."""
    if _ngpu() < 2:
        pytest.skip("needs 2 GPUs")
    _run_worker(2, ["rescal+sp", "adagrad", "0", "0.1", "1", "cuda"], env={"RAE_TEST_PEER_DENSE_MAX": "0"})


@pytest.mark.gpu
def test_sharded_regularised_step_is_deterministic():
    if _ngpu() < 2:
        pytest.skip("needs 2 GPUs")
    _run_worker(2, ["rescal+sp", "adagrad", "0", "0.1", "1", "cuda", "--determinism"])


@pytest.mark.gpu
@pytest.mark.parametrize("model", ["rescal+sp", "sp"])
def test_world1_sharded_matches_single_gpu_engine(model):
    """The world-1 sharded engine and the single-GPU engine on the same inputs at l2 = 0.1, every parameter to 1e-6
    relative after each of two steps."""
    from relation_autoencoder_b200.dist import DistributedEngine
    from relation_autoencoder_b200.engine import Engine
    from tests.helpers import make_problem, rel_err
    K, d, S, B, F, N = 100, 32, 5, 64, 3000, 900
    pr = make_problem(model, B=2 * B, K=K, d=d, S=S, F=F, N=N, seed=11, dup_heavy=True)
    p0 = {k: v.astype(np.float32) for k, v in pr["p"].items()}
    kw = dict(lr=0.1, l2=0.1, alpha=0.7, ext_reg=True)
    single = Engine(model, K, d, S, B, F, N, 2 * B, **kw)
    sharded = DistributedEngine(model, K, d, S, B, F, N, 2 * B, rank=0, world=1, **kw)
    for e in (single, sharded):
        e.set_params_numpy(p0)
        e.bind_split("train", pr["indptr"], pr["indices"], pr["a1"], pr["a2"])
        e.bind_epoch_negatives(pr["neg1"], pr["neg2"])
    identical = {}
    for b in range(2):
        c1 = single.train_device(b)
        c2 = sharded.train_device(b)
        assert abs(c1 - c2) <= 1e-6 * max(1.0, abs(c1)), (b, c1, c2)
        ps, pd = single.get_params_numpy(), sharded.get_params_numpy()
        acs, acd = single.get_acc_numpy(), sharded.get_acc_numpy()
        for n in ps:
            assert rel_err(pd[n], ps[n]) <= 1e-6, (b, n)
            assert rel_err(acd[n], acs[n]) <= 1e-6, (b, n, "acc")
            identical[n] = bool(np.array_equal(pd[n], ps[n]) and np.array_equal(acd[n], acs[n]))
    print("bit-identical after 2 steps:", identical)
    single.close()
    sharded.close()


def _emulate(table, acc, rows, ent_off, ent_src, ent_slot, grads, lr, r1, r2, adagrad):
    """fp32 NumPy statement of rae_shard_apply: summed contributions in entry order, + r1 sgn w + 2 r2 w, then the rule."""
    f = np.float32
    w, a = table.copy(), acc.copy()
    g = np.zeros_like(w)
    for i, r in enumerate(rows):
        for e in range(ent_off[i], ent_off[i + 1]):
            g[r] = (g[r] + grads[ent_src[e]][ent_slot[e]]).astype(f)
    g = (g + (f(r1) * np.sign(w) + f(2.0) * f(r2) * w).astype(f)).astype(f)
    if adagrad:
        a = (a + g * g).astype(f)
        w = (w - f(lr) * g / (np.sqrt(a) + f(1e-6))).astype(f)
    else:
        w = (w - f(lr) * g).astype(f)
    return w, a


@pytest.mark.gpu
@pytest.mark.parametrize("optimizer", ["adagrad", "sgd"])
@pytest.mark.parametrize("width", [7, 100])
@pytest.mark.parametrize("plan", ["empty", "all", "edges"])
def test_shard_apply_on_crafted_plans(plan, width, optimizer):
    import torch

    from relation_autoencoder_b200.engine import Engine
    l1, l2, adj, lr, world = 0.01, 0.1, 0.25, 0.1, 3
    eng = Engine("rescal+sp", 5, 6, 2, 8, 20, 10, 32, lr=lr, l1=l1, l2=l2, optimizer=optimizer, adj=adj)
    # the kernel gives each CTA min(1024, 16384 // width) rows: the shard spans several CTAs
    rpc = min(1024, 16384 // width)
    n_shard = 2 * rpc + rpc // 2 + 3
    if plan == "empty":
        rows = np.zeros(0, np.int64)
    elif plan == "all":
        rows = np.arange(n_shard)
    else:
        rows = np.unique([0, 1, rpc - 1, rpc, rpc + 1, 2 * rpc - 1, 2 * rpc, n_shard - 2, n_shard - 1])
    rng = np.random.RandomState(width + len(rows))
    cap = max(len(rows), 1)
    grads = [rng.uniform(-1, 1, size=(cap, width)).astype(np.float32) for _ in range(world)]
    cnt = rng.randint(1, world + 1, size=len(rows))
    ent_off = np.zeros(len(rows) + 1, np.int64)
    ent_off[1:] = np.cumsum(cnt)
    ent_src, ent_slot = [], []
    for i, c in enumerate(cnt):
        src = np.sort(rng.choice(world, size=c, replace=False))
        ent_src.extend(src.tolist())
        ent_slot.extend([i] * c)                  # slot i of every source holds row i's contribution
    ent_src, ent_slot = np.asarray(ent_src, np.int64), np.asarray(ent_slot, np.int64)
    table = rng.uniform(-0.5, 0.5, size=(n_shard, width)).astype(np.float32)
    table[3] = 0.0                                 # sgn(0) = 0
    acc = rng.uniform(0, 0.2, size=(n_shard, width)).astype(np.float32)
    dev = torch.device("cuda")
    i32 = lambda x: torch.as_tensor(np.asarray(x, np.int32)).to(dev)
    t_tab, t_acc = torch.from_numpy(table).to(dev), torch.from_numpy(acc).to(dev)
    t_grads = [torch.from_numpy(g).to(dev) for g in grads]
    t_rows, t_off, t_src, t_slot = i32(rows), i32(ent_off), i32(ent_src), i32(ent_slot)
    ptrs = (C.c_void_p * world)(*[g.data_ptr() for g in t_grads])
    rc = eng.lib.rae_shard_apply(eng._h, t_tab.data_ptr(), t_acc.data_ptr(), width, t_rows.data_ptr(), t_off.data_ptr(),
                                 t_src.data_ptr(), t_slot.data_ptr(), len(rows), ptrs, world, n_shard, eng._stream)
    assert rc == 0, eng.lib.rae_last_error(eng._h)
    torch.cuda.synchronize()
    w_ref, a_ref = _emulate(table, acc, rows, ent_off, ent_src, ent_slot, grads, lr, adj * l1, adj * l2, optimizer == "adagrad")
    w, a = t_tab.cpu().numpy(), t_acc.cpu().numpy()
    # AdaGrad's sqrt / reciprocal are the 1-ulp approximations (rae_common.cuh): a few ulp of the step
    assert np.all(np.abs(w - w_ref) <= 2e-6 * np.abs(w_ref) + 1e-7), np.abs(w - w_ref).max()
    if optimizer == "adagrad":
        assert np.all(np.abs(a - a_ref) <= 1e-6 * np.abs(a_ref) + 1e-12)
    else:
        assert np.array_equal(a, acc)                                  # SGD keeps no accumulator
    untouched = np.setdiff1d(np.arange(n_shard), rows)
    if untouched.size:
        moved = np.any(w[untouched] != table[untouched], axis=1)
        assert moved[np.any(table[untouched] != 0, axis=1)].all()     # the regulariser moves every non-zero row
    eng.close()
