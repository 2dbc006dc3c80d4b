"""Times rae_rank_arguments (fused tcgen05 argument ranking) against a torch fp32 baseline that computes the same ranks,
on one GPU.

    python profiles/arg_rank_bench.py --out profiles/arg_rank_b200.json [--rows 200000] [--rounds 3]

Inputs: model AC, K = 100, N = 500 k entities, F = 1 M features (synthetic CSR of ``synthetic.make_dataset``, fbar = 30),
200 k rows, batch B = 4096, at d = 128 (the target shape) and d = 30 (cfg2), parameters drawn on the device from a seeded
generator.  A alone is 256 MB (d = 128) / 60 MB, its FP16-pair image twice that, the score matrix of the baseline 800 GB:
no round starts warm in the 126 MB L2.  Timed with CUDA events, median over alternating rounds after one warm-up:
  (a) the whole rae_rank_arguments call; its kernels are split in a separate torch.profiler run into the A image
      (k_tc_absmax, k_rank_prep_a), query preparation (encoder, forward contraction, k_rank_queries) and ranking
      (k_tc_rank);
  (b) torch fp32 (TF32 off): the same forward in torch (sparse CSR x W, softmax, M = sum_r q_r C_r, v, w, c1, c2), then
      per chunk of 2048 queries a [2048, N] score matrix A U + Ab, the comparison with the thresholds and a row sum.
Agreement: every fused rank lies between the baseline's counts at thresholds t + tau and t - tau, tau = 1e-5
(sum_j |U_j| max_x |A_xj| + max |Ab|), the bracket of tests/test_gpu_arg_rank.py.  Flop: algorithmic 2 x rows x N x d x 2;
issued by the tensor cores 3 MMAs per product on padded shapes (rows and N to 128, d to 16), whose floor at the data
sheet's 2250 TFLOP/s dense FP16 is a bound from shapes, not a measurement.  The card's name, power limit and maximum SM
clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from relation_autoencoder_b200.engine import Engine  # noqa: E402
from relation_autoencoder_b200.synthetic import make_dataset  # noqa: E402

CHUNK = 2048
FP16_DENSE_TFLOPS = 2250.0


def hardware():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"torch_device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else None}


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def params(K, d, F, N, seed=7):
    g = torch.Generator(device="cuda").manual_seed(seed)
    u = lambda *s: torch.rand(s, generator=g, device="cuda") * 2 - 1  # noqa: E731
    n = lambda *s: torch.randn(s, generator=g, device="cuda")        # noqa: E731
    return {"W": u(F, K), "Wb": u(K) * 0.5, "A": u(N, d), "Ab": u(N) * 0.3, "C": n(d, d, K) * (0.8 / d ** 0.5),
            "C1": n(d, K) * 0.5, "C2": n(d, K) * 0.5}


def torch_queries(p, ip, ix, a1, a2, F):
    """U1 = v + c1, U2 = w + c2 in fp32 torch."""
    n = ip.numel() - 1
    X = torch.sparse_csr_tensor(ip.long(), ix.long(), torch.ones(ix.numel(), device="cuda"), size=(n, F))
    q = torch.softmax(X @ p["W"] + p["Wb"], dim=1)
    d, K = p["C1"].shape
    Cf = p["C"].reshape(d * d, K)
    U1 = torch.empty(n, d, device="cuda")
    U2 = torch.empty(n, d, device="cuda")
    for lo in range(0, n, 4096):
        hi = min(n, lo + 4096)
        M = (q[lo:hi] @ Cf.T).reshape(-1, d, d)
        L, R = p["A"][a1[lo:hi].long()], p["A"][a2[lo:hi].long()]
        U1[lo:hi] = torch.bmm(M, R[:, :, None])[:, :, 0] + q[lo:hi] @ p["C1"].T
        U2[lo:hi] = torch.bmm(M.transpose(1, 2), L[:, :, None])[:, :, 0] + q[lo:hi] @ p["C2"].T
    return U1, U2


def torch_counts(p, U, true_ids, shift=None):
    """#{x != true : A[x].U + Ab[x] > t (+ shift)} per query, in chunks of CHUNK queries."""
    A, Ab = p["A"], p["Ab"]
    t = (A[true_ids.long()] * U).sum(1) + Ab[true_ids.long()]
    if shift is not None:
        t = t + shift
    out = torch.empty(U.shape[0], dtype=torch.int64, device="cuda")
    for lo in range(0, U.shape[0], CHUNK):
        hi = min(U.shape[0], lo + CHUNK)
        S = U[lo:hi] @ A.T + Ab
        S[torch.arange(hi - lo, device="cuda"), true_ids[lo:hi].long()] = -float("inf")
        out[lo:hi] = (S > t[lo:hi, None]).sum(1)
    return out


def run_shape(d, rows, F, N, K, B, rounds):
    data = make_dataset(rows, F, N, 30)
    p = params(K, d, F, N)
    eng = Engine("rescal+sp", K, d, 5, B, F, N, B)
    eng.bind_params(p)
    ip = torch.as_tensor(data.indptr).cuda()
    ix = torch.as_tensor(data.indices).cuda()
    g = torch.Generator(device="cuda").manual_seed(11)
    a1 = torch.randint(0, N, (rows,), generator=g, device="cuda", dtype=torch.int32)
    a2 = torch.randint(0, N, (rows,), generator=g, device="cuda", dtype=torch.int32)
    r1 = torch.empty(rows, dtype=torch.int32, device="cuda")
    r2 = torch.empty(rows, dtype=torch.int32, device="cuda")
    lib, h = eng.lib, eng._h
    import ctypes as C
    P = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def fused():
        assert lib.rae_rank_arguments(h, P(ip), P(ix), P(a1), P(a2), rows, P(r1), P(r2),
                                      C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0

    base = {}

    def baseline():
        U1, U2 = torch_queries(p, ip, ix, a1, a2, F)
        base["r1"] = torch_counts(p, U1, a1) + 1
        base["r2"] = torch_counts(p, U2, a2) + 1
        base["U"] = (U1, U2)

    torch.backends.cuda.matmul.allow_tf32 = False
    variants = [("a_fused_call", fused), ("b_torch_fp32", baseline)]
    for _, fn in variants:
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name, _ in variants}
    for _ in range(rounds):
        for name, fn in variants:
            times[name].append(timed(fn))
    # agreement: the fused ranks inside the bracket of the baseline's scores
    U1, U2 = base["U"]
    Amax = p["A"].abs().max(0).values
    abmax = p["Ab"].abs().max()
    agree = {}
    for s, (U, tru, r) in enumerate(((U1, a1, r1), (U2, a2, r2)), 1):
        tau = 1e-5 * (U.abs() @ Amax + abmax)
        lo = torch_counts(p, U, tru, tau) + 1
        hi = torch_counts(p, U, tru, -tau) + 1
        rr = r.long()
        agree["slot%d_outside_bracket" % s] = int(((rr < lo) | (rr > hi)).sum())
        agree["slot%d_equal_to_torch" % s] = float((rr == base["r%d" % s]).double().mean())
    # kernel split (separate run, profiler on)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fused()
        torch.cuda.synchronize()
    split = {"a_image_us": 0.0, "query_prep_us": 0.0, "rank_kernel_us": 0.0, "kernels": {}}
    for e in prof.key_averages():
        if e.device_type is None or "Memset" in e.key or e.self_device_time_total <= 0:
            continue
        us = float(e.self_device_time_total)
        split["kernels"][e.key[:80]] = us
        if "k_tc_rank" in e.key:
            split["rank_kernel_us"] += us
        elif "k_rank_prep_a" in e.key or "k_tc_absmax" in e.key:
            split["a_image_us"] += us
        else:
            split["query_prep_us"] += us
    DH = (d + 15) // 16 * 16
    rp = (rows + 127) // 128 * 128
    Np = (N + 127) // 128 * 128
    algo = 2.0 * rows * N * d * 2
    issued = 2.0 * rp * Np * DH * 2 * 3
    med = {k: float(np.median(v)) for k, v in times.items()}
    res = {"d": d, "K": K, "N": N, "F": F, "rows": rows, "B": B, "rounds": rounds, "ms_median": med, "ms_all": times,
           "split_us_profiled": split, "agreement": agree,
           "algorithmic_flop": algo, "issued_flop": issued,
           "issued_floor_ms_at_datasheet": issued / (FP16_DENSE_TFLOPS * 1e12) * 1e3,
           "issued_share_of_fp16_dense_rate_rank_kernel": issued / (FP16_DENSE_TFLOPS * 1e12) / (split["rank_kernel_us"] * 1e-6)
           if split["rank_kernel_us"] > 0 else None,
           "issued_share_of_fp16_dense_rate_whole_call": issued / (FP16_DENSE_TFLOPS * 1e12) / (med["a_fused_call"] * 1e-3),
           "speedup_vs_torch": med["b_torch_fp32"] / med["a_fused_call"]}
    eng.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rows", type=int, default=200_000)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("arg_rank_bench needs a CUDA device")
    out = {"hardware": hardware(), "shapes": []}
    for d in (128, 30):
        r = run_shape(d, a.rows, 1_000_000, 500_000, 100, 4096, a.rounds)
        print(json.dumps({k: r[k] for k in ("d", "ms_median", "agreement", "speedup_vs_torch",
                                            "issued_share_of_fp16_dense_rate_rank_kernel")}), flush=True)
        print(json.dumps(r["split_us_profiled"]), flush=True)
        out["shapes"].append(r)
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["hardware"]))


if __name__ == "__main__":
    main()
