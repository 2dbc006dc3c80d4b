"""Cost of the regulariser in the row-sharded multi-GPU step at the north-star shape T (AC, K = 100, d = 128, S = 20,
B = 4096 per GPU, F = 1M, N = 500k).

    python -m torch.distributed.run --nproc-per-node W profiles/sharded_regulariser_bench.py OUT.json [--steps 20 --rounds 5]

Two sharded engines on the same inputs, l2 = 0 and l2 = 0.1 (ext_reg, AdaGrad), timed in alternating rounds of --steps
steps (CUDA events around each round, every rank's time max-reduced; the median round is reported).  Then, in timeline
mode, the marks of the owner-side W pass of the regularised engine (w_shard_begin -> apply_W) and of its norms + cost re-run
(end -> reg_cost), median over 5 steps, and the pass's bytes: 16 B per shard element (w and acc read and written) plus the
batch's contribution rows (4 B per element), over its time.  Rank 0 writes OUT.json with the card and its power limit,
read in the same run."""
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from relation_autoencoder_b200 import synthetic as SY  # noqa: E402
from relation_autoencoder_b200.dist import DistributedEngine  # noqa: E402


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    return q.stdout.strip().splitlines()


def _peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "MEASURED_PEAKS.json"
    return None, "not available on this machine"


def main():
    out = sys.argv[1]
    steps = int(sys.argv[sys.argv.index("--steps") + 1]) if "--steps" in sys.argv else 20
    n_rounds = int(sys.argv[sys.argv.index("--rounds") + 1]) if "--rounds" in sys.argv else 5
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if world_env > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        rank, world = dist.get_rank(), dist.get_world_size()
    else:
        rank, world = 0, 1
    wl = SY.WORKLOADS["T"]
    B, K = wl["B"], wl["K"]
    nb = steps * n_rounds + 40
    data = SY.make_dataset(nb * B, wl["F"], wl["N"], wl["fbar"], seed=1234 + rank)
    rng = np.random.RandomState(2)
    params = SY.init_params(rng, wl["model"], wl["F"], K, wl["N"], wl["d"])
    neg1, neg2 = SY.draw_negatives(rng, data.neg_cum, data.n, wl["S"])
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    engs = {}
    for l2 in (0.0, 0.1):
        e = DistributedEngine(wl["model"], K, wl["d"], wl["S"], B, wl["F"], wl["N"], wl["N_train"], lr=0.1, l2=l2,
                              alpha=wl.get("alpha", 1.0), device=local, rank=rank, world=world)
        e.set_params_numpy(params)
        e.bind_split("train", data.indptr, data.indices, data.args1, data.args2)
        e.bind_epoch_negatives(neg1, neg2)
        engs[l2] = e
    del params
    nb = engs[0.0].nb
    for e in engs.values():                      # warm-up
        for s in range(5):
            e.train_device(s % nb, want_cost=False)
    barrier()
    times = {0.0: [], 0.1: []}
    nxt = 5
    for r in range(n_rounds):
        for l2, e in engs.items():               # alternating
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for s in range(steps):
                e.train_device((nxt + s) % nb, want_cost=False)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1)
            if world > 1:
                t = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms = float(t[0])
            times[l2].append(ms / steps)
        nxt += steps

    # timeline of the regularised engine: the W pass and the norms + cost re-run, median over 5 steps
    e = engs[0.1]
    fp = e.fplan
    e.set_timeline(True)
    pass_us, cost_us, pass_bytes = [], [], []
    w_rows = int(e.shard["W"].shape[0])
    for r in range(5):
        for s in range(6):
            b = (nxt + 6 * r + s) % nb
            e.train_device(b, want_cost=False)
        tl = {(n, sid): t for n, sid, t in e.timeline()}
        pass_us.append(tl[("apply_W", 0)] - tl[("w_shard_begin", 0)])
        cost_us.append(tl[("reg_cost", 0)] - tl[("end", 0)])
        lo, hi = fp.r_off[b], fp.r_off[b + 1]
        n_ent = int(fp.ent_off[hi].item() - fp.ent_off[lo].item())
        pass_bytes.append(16.0 * w_rows * K + 4.0 * n_ent * K)
    e.set_timeline(False)
    e0_ = engs[0.0]
    e0_.set_timeline(True)
    for s in range(6):
        e0_.train_device((nxt + s) % nb, want_cost=False)
    tl0 = e0_.timeline()
    e0_.set_timeline(False)
    barrier()
    for x in engs.values():
        x.close()
    # every rank's pass time: the slowest rank sets the step
    vals = torch.tensor([float(np.median(pass_us)), float(np.median(cost_us)), float(np.median(pass_bytes))], dtype=torch.float64,
                        device=dev)
    allv = [torch.zeros_like(vals) for _ in range(world)]
    if world > 1:
        dist.all_gather(allv, vals)
    else:
        allv = [vals]
    if rank == 0:
        peak, peak_src = _peak()
        per_rank = [[float(v) for v in a.tolist()] for a in allv]
        worst = max(per_rank, key=lambda v: v[0])
        gbs = worst[2] / (worst[0] * 1e-6) / 1e9
        res = {
            "workload": "T: " + wl["desc"], "world": world, "batch_per_gpu": B, "steps_per_round": steps, "rounds": n_rounds,
            "card": _card(), "measured_at": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()),
            "ms_per_step": {"l2=0": float(np.median(times[0.0])), "l2=0.1": float(np.median(times[0.1]))},
            "ms_per_step_rounds": {"l2=0": times[0.0], "l2=0.1": times[0.1]},
            "w_rows_rank0": w_rows,
            "w_pass": {"us_per_rank": [v[0] for v in per_rank], "bytes_per_rank": [v[2] for v in per_rank],
                       "slowest_rank_GBs": gbs, "peak_GBs": peak, "peak_source": peak_src,
                       "frac_of_peak": (gbs / peak) if peak else None,
                       "bytes_model": "16 B per shard element (w, acc read + written) + 4 B per contribution element"},
            "reg_cost_us_per_rank": [v[1] for v in per_rank],
            "timeline_l2_0_last_step": tl0,
        }
        with open(out, "w") as f:
            json.dump(res, f, indent=1)
        print(json.dumps({k: res[k] for k in ("world", "card", "ms_per_step")}), json.dumps(res["w_pass"]))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
