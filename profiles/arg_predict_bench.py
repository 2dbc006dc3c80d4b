"""Times rae_predict_arguments (top-k epilogue of the tcgen05 ranking GEMM) against rae_rank_arguments on the same inputs
and against a torch fp32 top-k baseline, on one GPU.

    python profiles/arg_predict_bench.py --out profiles/arg_predict_b200.json [--rows 200000] [--rounds 3]

Inputs: those of profiles/arg_rank_bench.py (model AC, K = 100, N = 500 k entities, F = 1 M features, 200 k rows,
B = 4096, d = 128 and d = 30).  Timed with CUDA events, median over alternating rounds after one warm-up:
  rae_predict_arguments at k = 1, 10 and 16; rae_rank_arguments; and torch fp32 (TF32 off): the forward of
  arg_rank_bench.torch_queries, then per chunk of 2048 queries the [2048, N] scores A U + Ab and torch.topk.
The predict call's kernels are split in a separate torch.profiler run (k_tc_predict, k_predict_merge, the rest).
Agreement, per slot against the baseline's fp32 scores S with tau = 1e-5 (sum_j |U_j| max_x |A_xj| + max |Ab|) per
query: every listed score within tau of S[id], every entity with S > (k-th score) + 2 tau listed, every listed entity with
S >= (k-th score) - 2 tau (the bracket of tests/test_gpu_arg_predict.py).  The card's name, power limit and maximum SM
clock are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import arg_rank_bench as RB  # noqa: E402
from relation_autoencoder_b200.engine import Engine  # noqa: E402
from relation_autoencoder_b200.synthetic import make_dataset  # noqa: E402

KS = (1, 10, 16)


def torch_topk(p, U, k):
    ids = torch.empty(U.shape[0], k, dtype=torch.int64, device="cuda")
    for lo in range(0, U.shape[0], RB.CHUNK):
        hi = min(U.shape[0], lo + RB.CHUNK)
        ids[lo:hi] = torch.topk(U[lo:hi] @ p["A"].T + p["Ab"], k, dim=1).indices
    return ids


def violations(p, U, ids, sc, tau):
    """(score errors > tau, entities above k-th + 2 tau missing, listed entities below k-th - 2 tau) over all queries."""
    k = ids.shape[1]
    bad = [0, 0, 0]
    for lo in range(0, U.shape[0], RB.CHUNK):
        hi = min(U.shape[0], lo + RB.CHUNK)
        S = U[lo:hi] @ p["A"].T + p["Ab"]
        t = tau[lo:hi, None]
        i = ids[lo:hi].long()
        got = torch.gather(S, 1, i)
        kth = torch.topk(S, k, dim=1).values[:, -1:]
        bad[0] += int((sc[lo:hi] - got).abs().gt(t).sum())
        above = (S > kth + 2 * t).sum(1)
        listed_above = (got > kth + 2 * t).sum(1)
        bad[1] += int((above - listed_above).sum())
        bad[2] += int((got < kth - 2 * t).sum())
    return bad


def run_shape(d, rows, F, N, K, B, rounds):
    data = make_dataset(rows, F, N, 30)
    p = RB.params(K, d, F, N)
    eng = Engine("rescal+sp", K, d, 5, B, F, N, B)
    eng.bind_params(p)
    ip = torch.as_tensor(data.indptr).cuda()
    ix = torch.as_tensor(data.indices).cuda()
    g = torch.Generator(device="cuda").manual_seed(11)
    a1 = torch.randint(0, N, (rows,), generator=g, device="cuda", dtype=torch.int32)
    a2 = torch.randint(0, N, (rows,), generator=g, device="cuda", dtype=torch.int32)
    r1 = torch.empty(rows, dtype=torch.int32, device="cuda")
    r2 = torch.empty(rows, dtype=torch.int32, device="cuda")
    out = {k: [torch.empty(rows, k, dtype=dt, device="cuda") for dt in (torch.int32, torch.float32) * 2] for k in KS}
    lib, h = eng.lib, eng._h
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)  # noqa: E731

    def predict(k):
        def fn():
            assert lib.rae_predict_arguments(h, P(ip), P(ix), P(a1), P(a2), rows, k, *[P(t) for t in out[k]], st()) == 0
        return fn

    def rank():
        assert lib.rae_rank_arguments(h, P(ip), P(ix), P(a1), P(a2), rows, P(r1), P(r2), st()) == 0

    base = {}

    def baseline():
        U1, U2 = RB.torch_queries(p, ip, ix, a1, a2, F)
        base["ids"] = (torch_topk(p, U1, 10), torch_topk(p, U2, 10))
        base["U"] = (U1, U2)

    torch.backends.cuda.matmul.allow_tf32 = False
    variants = [("predict_k%d" % k, predict(k)) for k in KS] + [("rank", rank), ("torch_fp32_topk10", baseline)]
    for _, fn in variants:
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name, _ in variants}
    for _ in range(rounds):
        for name, fn in variants:
            times[name].append(RB.timed(fn))
    U1, U2 = base["U"]
    Amax = p["A"].abs().max(0).values
    abmax = p["Ab"].abs().max()
    agree = {}
    for k in KS:
        i1, s1, i2, s2 = out[k]
        for s, (U, ids, sc) in enumerate(((U1, i1, s1), (U2, i2, s2)), 1):
            tau = 1e-5 * (U.abs() @ Amax + abmax)
            e, miss, low = violations(p, U, ids, sc, tau)
            agree["k%d_slot%d" % (k, s)] = {"score_error_over_tau": e, "missing_above_bracket": miss, "listed_below_bracket": low}
        agree["k%d_prefix_of_k16" % k] = all(bool(torch.equal(a, b[:, :k])) for a, b in zip(out[k], out[16]))
    agree["k10_ids_equal_to_torch"] = [float((out[10][2 * s] == base["ids"][s]).all(1).double().mean()) for s in (0, 1)]
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        predict(10)()
        torch.cuda.synchronize()
    split = {"predict_kernel_us": 0.0, "merge_us": 0.0, "rest_us": 0.0, "kernels": {}}
    for e in prof.key_averages():
        if e.device_type is None or "Memset" in e.key or e.self_device_time_total <= 0:
            continue
        us = float(e.self_device_time_total)
        split["kernels"][e.key[:80]] = us
        key = "predict_kernel_us" if "k_tc_predict" in e.key else "merge_us" if "k_predict_merge" in e.key else "rest_us"
        split[key] += us
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {"d": d, "K": K, "N": N, "F": F, "rows": rows, "B": B, "rounds": rounds, "ms_median": med, "ms_all": times,
           "predict_over_rank": {k: med["predict_k%d" % k] / med["rank"] for k in KS},
           "torch_over_predict_k10": med["torch_fp32_topk10"] / med["predict_k10"],
           "split_k10_us_profiled": split, "agreement": agree}
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rows", type=int, default=200_000)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("arg_predict_bench needs a CUDA device")
    res = {"hardware": RB.hardware(), "shapes": []}
    for d in (128, 30):
        r = run_shape(d, a.rows, 1_000_000, 500_000, 100, 4096, a.rounds)
        print(json.dumps({k: r[k] for k in ("d", "ms_median", "predict_over_rank", "torch_over_predict_k10", "agreement")}),
              flush=True)
        print(json.dumps(r["split_k10_us_profiled"]), flush=True)
        res["shapes"].append(r)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["hardware"]))


if __name__ == "__main__":
    main()
