"""Times the fused top-k labelling kernel (rae_label_topk) against the labels-only floor and against full probabilities
followed by torch.topk, on one GPU.

    python profiles/label_topk_bench.py --out profiles/label_topk_b200.json [--rows 2000000] [--rounds 5]

Inputs: synthetic CSR from ``synthetic.make_dataset`` (F = 1 M, fbar = 30, Zipf feature ids) at the cfg2 (K = 100) and
cfg5 (K = 1000) sizes, W uniform in [-1, 1) drawn on the device, Wb = 0.  What is timed, CUDA events around each call,
median over alternating rounds (every call streams all of W's touched rows and the whole CSR, 0.6-4 GB, far beyond the
126 MB L2, so no round starts warm):
  (a) rae_label_shards, probs NULL: the labels-only floor;
  (b) rae_label_topk at k = 1, 3, 16 with probs;
  (c) rae_label_shards with probs, then torch.topk, in chunks of 256 k rows so that the [rows, K] probabilities fit.
Bytes of (b): 4 nnz K (W rows) + 4 nnz (indices) + 4 n (indptr) + 8 n k (ids and probs).  The card's name, power
limit and maximum SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import ctypes as C
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

CHUNK = 256 * 1024


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


def run_shape(K, n, F, fbar, rounds):
    d = make_dataset(n, F, 1000, fbar)
    nnz = int(d.indptr[-1])
    eng = Engine("rescal", K, 4, 1, 8, F, 8, 8)
    g = torch.Generator(device="cuda").manual_seed(7)
    W = torch.rand((F, K), generator=g, device="cuda") * 2 - 1
    eng.bind_params({"W": W, "Wb": torch.zeros(K, device="cuda"), "A": torch.zeros((8, 4), device="cuda"),
                     "Ab": torch.zeros(8, device="cuda"), "C": torch.zeros((4, 4, K), device="cuda")})
    ip = torch.as_tensor(d.indptr).cuda()
    ix = torch.as_tensor(d.indices).cuda()
    lib, h = eng.lib, eng._h
    w = (C.c_void_p * 1)(W.data_ptr())
    labels = torch.empty(n, dtype=torch.int64, device="cuda")
    full = torch.empty((CHUNK, K), dtype=torch.float32, device="cuda")
    ks = [1, 3, 16]
    ids = {k: torch.empty((n, k), dtype=torch.int32, device="cuda") for k in ks}
    probs = {k: torch.empty((n, k), dtype=torch.float32, device="cuda") for k in ks}
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731

    def floor():
        assert lib.rae_label_shards(h, w, 1, p(ip), p(ix), n, p(labels), C.c_void_p(0), None) == 0

    def fused(k):
        assert lib.rae_label_topk(h, w, 1, p(ip), p(ix), n, k, p(ids[k]), p(probs[k]), None) == 0

    def unfused(k):
        for lo in range(0, n, CHUNK):
            m = min(CHUNK, n - lo)
            assert lib.rae_label_shards(h, w, 1, C.c_void_p(ip.data_ptr() + 4 * lo), p(ix), m, p(labels[lo:]), p(full), None) == 0
            v, i = torch.topk(full[:m], k, dim=1)
            probs[k][lo:lo + m] = v
            ids[k][lo:lo + m] = i

    variants = [("a_labels_only", floor)] + [("b_topk_k%d" % k, (lambda k=k: fused(k))) for k in ks] + \
               [("c_probs_then_torch_topk_k%d" % k, (lambda k=k: unfused(k))) for k in ks]
    for _, fn in variants:            # warm-up: module load, torch.topk's kernel choice
        fn()
    torch.cuda.synchronize()
    times = {name: [] for name, _ in variants}
    for _ in range(rounds):
        for name, fn in variants:
            times[name].append(timed(fn))
    # the fused top-1 is the labels-only argmax, and its probabilities are those of the full softmax
    fused(16)
    floor()
    torch.cuda.synchronize()
    same_top1 = bool(torch.equal(ids[16][:, 0].long(), labels))
    unfused(16)
    ref_probs = probs[16].clone()
    fused(16)
    torch.cuda.synchronize()
    same_probs = bool(torch.equal(probs[16], ref_probs))
    res = {"K": K, "rows": n, "F": F, "fbar": fbar, "nnz": nnz, "rounds": rounds, "same_top1_as_labels": same_top1,
           "fused_probs_equal_torch_topk_values_k16": same_probs, "ms_median": {}, "ms_all": times, "topk_GBps": {}}
    for name, t in times.items():
        res["ms_median"][name] = float(np.median(t))
    for k in ks:
        byts = 4.0 * nnz * K + 4.0 * nnz + 4.0 * n + 8.0 * n * k
        res["topk_GBps"]["k%d" % k] = byts / (res["ms_median"]["b_topk_k%d" % k] * 1e-3) / 1e9
    res["floor_GBps"] = (4.0 * nnz * K + 4.0 * nnz + 4.0 * n + 8.0 * n) / (res["ms_median"]["a_labels_only"] * 1e-3) / 1e9
    eng.close()
    del W, full, ids, probs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--rows", type=int, default=2_000_000)
    ap.add_argument("--features", type=int, default=1_000_000)
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("label_topk_bench needs a CUDA device")
    out = {"hardware": hardware(), "shapes": []}
    for K in (100, 1000):
        r = run_shape(K, a.rows, a.features, 30, a.rounds)
        print(json.dumps({k: r[k] for k in ("K", "ms_median", "topk_GBps", "floor_GBps", "same_top1_as_labels",
                                            "fused_probs_equal_torch_topk_values_k16")}), flush=True)
        out["shapes"].append(r)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out["hardware"]))


if __name__ == "__main__":
    main()
