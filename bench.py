#!/usr/bin/env python
"""bench.py - training examples/sec of the relation-autoencoder hot path on B200 (BASELINE.json's metric).

One "step" = one fused forward/backward/update pass of the hot path over one batch of synthetic input
(SURVEY 8d).  Default workload: ``T``, the shape BASELINE.json's target sentence is quoted on (AC, K=100, d=128,
20 negatives, batch 4096 per GPU, ~30 features/example, 1M feature vocab, 500k entities); ``--workload
cfg2|cfg3|cfg4|cfg5|cfg1`` select BASELINE.json's configs.  At N=1 a short cfg2 (configs[1]) measurement rides along as
``extra.cfg2``.

Timing: W warm-up steps, then one round of EXACTLY K timed steps (CUDA events on the launching stream, barrier +
synchronize on both sides, max over ranks).  ``--min-time S`` repeats the K-step round until S seconds of device time have
been timed and reports the MEDIAN round.  ``--check`` (default on) runs one step of a small sharded problem outside the
timed region and compares cost and every parameter's gradient with the float64 oracle (``parity_ok``).
``--dump-outputs DIR`` writes the parameters after the last timed step as DIR/<name>.npy (see ``_dump_outputs``); the
inputs depend on the arguments only, so two builds run with the same arguments can be compared array for array.

  python bench.py --gpus N --steps K --warmup W            our arm  (N>1: launched by torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K ...  reference arm: the reference's CPU path (NumPy float64 port of
                                                           the Theano graph with the reference's DENSE AdaGrad sweep;
                                                           Theano itself is not installable) on the box's host cores

Prints ONE JSON line (rank 0).  `value` = whole-job examples/sec with inputs resident in HBM; `e2e` = the same through
Engine.train(batch_index, neg1, neg2) with HOST negatives copied in and the cost read back every step (the reference's
func['train'] call, OieInduction.py:189).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from relation_autoencoder_b200 import synthetic as SY  # noqa: E402

METRIC = "AC-model train examples/sec"
UNIT = "examples/s"


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        pk = json.load(open(path))
        return dict(hbm_gbs=float(pk["hbm_gbs"]), bf16_burst=float(pk["bf16_tflops"]),
                    bf16_sustained=float(pk.get("bf16_tflops_sustained", pk["bf16_tflops"])), source="measured")
    return dict(hbm_gbs=6650.0, bf16_burst=1590.0, bf16_sustained=1400.0, source="fallback")   # B200_PROFILING.md:17-20


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (B200_PROFILING.md:70-72): NVML polled from a thread
    every ~2 ms (nvidia-smi -lms as a fallback, which is too slow for short regions)."""
    REASONS = (("hw_slowdown", 0x8), ("sw_power_cap", 0x4), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, device_index=0, period_s=0.002):
        self.dev = device_index
        self.period = period_s
        self.sm, self.mask = [], 0
        self.max_sm = None
        self._stop = threading.Event()
        self._t = None
        self._nvml = None
        self._h = None
        self._smi = None

    def _handle(self):
        import pynvml
        pynvml.nvmlInit()
        self._nvml = pynvml
        try:
            import torch
            uuid = str(torch.cuda.get_device_properties(self.dev).uuid)
            return pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid).encode())
        except Exception:
            return pynvml.nvmlDeviceGetHandleByIndex(self.dev)

    def start(self):
        try:
            self._h = self._handle()
            self.max_sm = float(self._nvml.nvmlDeviceGetMaxClockInfo(self._h, self._nvml.NVML_CLOCK_SM))
            self._t = threading.Thread(target=self._poll, daemon=True)
            self._t.start()
        except Exception:
            self._h = None
            try:
                q = "clocks.sm,clocks.max.sm,clocks_event_reasons.active"
                self._smi = subprocess.Popen(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                              "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self._t = threading.Thread(target=self._read_smi, daemon=True)
                self._t.start()
            except Exception:
                self._smi = None

    def _poll(self):
        n = self._nvml
        while not self._stop.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)))
                self.mask |= int(n.nvmlDeviceGetCurrentClocksEventReasons(self._h))
            except Exception:
                pass
            time.sleep(self.period)

    def _read_smi(self):
        for line in self._smi.stdout:
            f = [x.strip() for x in line.split(",")]
            try:
                self.sm.append(float(f[0]))
                self.max_sm = float(f[1])
                self.mask |= int(f[2], 16)
            except Exception:
                continue

    def stop(self):
        self._stop.set()
        if self._smi is not None:
            time.sleep(0.05)
            self._smi.terminate()
        if self._t is not None:
            self._t.join(timeout=2)
        if not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_sm, "samples": 0, "reasons": ["no clock samples"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_min_mhz": float(min(self.sm)), "sm_max_mhz": self.max_sm,
                "samples": len(self.sm), "reasons": sorted(name for name, bit in self.REASONS if self.mask & bit)}


def _needed_examples(wl, steps, warmup, extra):
    return (steps + warmup + extra) * wl["B"]


def _make_inputs(wl, n_examples, rank=0, uniform=False):
    data = SY.make_dataset(n_examples, wl["F"], wl["N"], wl["fbar"], seed=1234 + rank, uniform=uniform)
    rng = np.random.RandomState(2)
    params = SY.init_params(rng, wl["model"], wl["F"], wl["K"], wl["N"], wl["d"])
    neg1, neg2 = SY.draw_negatives(rng, data.neg_cum, data.n, wl["S"])
    return data, params, neg1, neg2


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle port of the reference's CPU path (the ONLY place bench.py executes oracle/)
# ----------------------------------------------------------------------------------------------------------------------
def cpu_reference_steps(wl, data, params32, neg1, neg2, steps, warmup, budget_s, sparse_rows=False):
    from oracle import rae_oracle as O
    p = {k: v.astype(np.float64) for k, v in params32.items()}
    om = O.OracleModel(wl["model"], p, K=wl["K"], d=wl["d"], S=wl["S"], B=wl["B"], lr=0.1, l1=0.0, l2=wl.get("l2", 0.0),
                       alpha=wl.get("alpha", 1.0), sparse_rows=sparse_rows)
    om.bind_split("train", data.indptr, data.indices, data.args1, data.args2)
    B = wl["B"]
    nb = data.n // B
    times = []
    t_begin = time.perf_counter()
    done = 0
    for s in range(warmup + steps):
        b = s % nb
        t0 = time.perf_counter()
        om.train(b, neg1[:, b * B:(b + 1) * B], neg2[:, b * B:(b + 1) * B])
        t1 = time.perf_counter()
        if s >= warmup:
            times.append(t1 - t0)
            done += 1
        if time.perf_counter() - t_begin > budget_s and done >= 1:
            break
    sec = float(np.mean(times))
    return B / sec, sec, done


def _host_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [i.get("num_threads", 1) for i in threadpool_info() if i.get("user_api") == "blas"]
        return max(n) if n else 1
    except Exception:
        return os.cpu_count() or 1


def run_reference(args, wl, rank, world):
    if rank != 0:
        return
    steps, warmup = args.steps, args.warmup
    n_ex = min(wl["N_train"], max(4, min(steps + warmup, 8)) * wl["B"])
    data, params, neg1, neg2 = _make_inputs(wl, n_ex)
    eps, sec, done = cpu_reference_steps(wl, data, params, neg1, neg2, steps, min(warmup, 1), budget_s=args.cpu_budget)
    cores = _host_threads()
    sample = ("%d of %d requested steps of batch %d on the same synthetic workload; NumPy float64 port of the Theano graph "
              "with the reference's dense AdaGrad sweep over every parameter (Optimizers.py:29-32); Theano is not "
              "installable offline" % (done, steps, wl["B"]))
    line = {
        "impl": "reference", "metric": METRIC, "value": eps, "unit": UNIT, "n_gpus": args.gpus, "steps": done,
        "warmup": min(warmup, 1), "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": _config(wl, args, world),
        "cpu_baseline": {"value": eps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": eps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def _config(wl, args, world, name=None):
    return {"workload": "%s: %s" % (name or args.workload, wl["desc"]), "decoder": wl["model"], "K": wl["K"], "d": wl["d"],
            "S": wl["S"], "batch_per_gpu": wl["B"], "global_batch": wl["B"] * world, "fbar": wl["fbar"], "F": wl["F"],
            "N": wl["N"], "N_train_nominal": wl["N_train"], "optimizer": "adagrad", "lr": 0.1,
            "l2": wl.get("l2", 0.0), "alpha": wl.get("alpha", 1.0), "feature_distribution": "zipf(1.0)" if not args.uniform else "uniform",
            "parallelism": "dp%d" % world,
            "l2_cache_policy": "inputs larger than L2: W+acc %.0f MB, A+acc %.0f MB, a different batch every step"
                               % (2 * 4e-6 * wl["F"] * wl["K"], 2 * 4e-6 * wl["N"] * wl["d"])}


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
def run_ours(args, wl, rank, world, local_rank):
    # libraries (NCCL's version banner, ...) must not write to stdout: only the JSON line does
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = _run_ours(args, wl, rank, world, local_rank)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if line is not None:
        print(json.dumps(line))
        sys.stdout.flush()


def _measure_tf32_peak(dev):
    """TF32 tensor-core denominator (SURVEY 8d: 'measure a TF32 cuBLAS GEMM once on the box'): torch.matmul fp32 8192^3
    with TF32 allowed, best of 10 (burst) - the contraction kernels are timed alone, per launch."""
    import torch
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev, dtype=torch.float32)
        b = torch.randn(n, n, device=dev, dtype=torch.float32)
        for _ in range(3):
            torch.matmul(a, b)
        best = 1e30
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            torch.matmul(a, b)
            e1.record()
            e1.synchronize()
            best = min(best, e0.elapsed_time(e1))
        del a, b
        return 2.0 * n ** 3 / (best * 1e-3) / 1e12
    except Exception:
        return None
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def _parity_check(args, rank, world, local_rank, dist):
    """One step of a small sharded problem (outside every timed region) against the float64 oracle run on the GLOBAL
    batch: cost within 1e-5 and, from the AdaGrad accumulators of a first step from zero (acc' = g^2), |g| of EVERY
    element of every parameter within 1e-5 of ||g_ref||_inf - the check tests/dist_worker.py does, on the driver's own
    multi-GPU box.  The oracle is the checker here, never the thing measured."""
    import torch
    from oracle import rae_oracle as O
    from relation_autoencoder_b200.engine import Engine
    model, K, d, S, B, F, N, fbar = "rescal+sp", 100, 128, 4, 128, 3000, 900, 12
    Bg = B * world
    data = SY.make_dataset(Bg, F, N, fbar, seed=77)
    rng = np.random.RandomState(5)
    p0 = {k: v.astype(np.float32) for k, v in SY.init_params(rng, model, F, K, N, d).items()}
    p0["W"] = rng.uniform(-0.3, 0.3, size=(F, K)).astype(np.float32)         # away from the flat-softmax start
    p0["A"] = rng.uniform(-0.5, 0.5, size=(N, d)).astype(np.float32)
    neg1, neg2 = SY.draw_negatives(rng, data.neg_cum, Bg, S)
    rows = np.arange(rank * B, (rank + 1) * B)
    ip = data.indptr
    lo, hi = int(ip[rows[0]]), int(ip[rows[-1] + 1])
    loc_ip = (ip[rows[0]:rows[-1] + 2] - lo).astype(np.int32)
    loc_ix = data.indices[lo:hi]
    if world > 1:
        from relation_autoencoder_b200.dist import DistributedEngine
        eng = DistributedEngine(model, K, d, S, B, F, N, n_train=Bg, lr=0.1, alpha=0.7, rank=rank, world=world, device=local_rank)
    else:
        eng = Engine(model, K, d, S, B, F, N, Bg, lr=0.1, alpha=0.7, device=local_rank)
    eng.set_params_numpy(p0)
    eng.bind_split("train", loc_ip, loc_ix, data.args1[rows], data.args2[rows])
    eng.bind_epoch_negatives(np.ascontiguousarray(neg1[:, rows]), np.ascontiguousarray(neg2[:, rows]))
    cost = eng.train_device(0, want_cost=True)
    acc = eng.get_acc_numpy()              # collective gather for N > 1
    tensor_path = int(eng.stats().get("tensor_path", -1))
    eng.close()
    res = None
    if rank == 0:
        om = O.OracleModel(model, {k: v.astype(np.float64) for k, v in p0.items()}, K=K, d=d, S=S, B=Bg, lr=0.1, alpha=0.7)
        om.bind_split("train", data.indptr, data.indices, data.args1, data.args2)
        c_ref = om.train(0, neg1, neg2)
        worst, worst_name = 0.0, ""
        for n in O.param_names(model):
            g = np.abs(om.last_grads[n])
            e = float(np.abs(np.sqrt(acc[n].astype(np.float64)) - g).max() / max(g.max(), 1e-300))
            if e > worst:
                worst, worst_name = e, n
        cost_err = abs(cost - c_ref) / max(1.0, abs(c_ref))
        res = {"parity_ok": bool(cost_err <= 1e-5 and worst <= 1e-5), "max_rel_err": worst, "max_rel_err_param": worst_name,
               "cost_rel_err": cost_err, "tensor_path": tensor_path,
               "parity_check": "one sharded step, AC K=100 d=128 S=4, %d examples per rank x %d ranks, cost and |grad| of every "
                               "parameter element vs the float64 oracle on the global batch (tolerances 1e-5 / 1e-5)" % (B, world)}
    if dist is not None:
        dist.barrier()
    return res


DUMP_MAX_ELEMS = 2 << 20       # per array: 8 MB of float32; at most 7 parameters, so a dump stays under 64 MB


def _dump_outputs(out_dir, params, data, neg1, neg2, b, B):
    """The parameters after the last timed step (what the caller of the training step gets back: they are updated in
    place) as ``out_dir/<name>.npy``, float32.  Of the row tables only the rows batch ``b`` (the last step's) touched are
    kept: its feature rows of W, its argument and negative rows of A and Ab.  An array of more than DUMP_MAX_ELEMS
    elements is cut to a fixed, seeded sample of those rows (tables) or of its elements (dense parameters)."""
    os.makedirs(out_dir, exist_ok=True)
    lo, hi = b * B, (b + 1) * B
    ent = np.concatenate([data.args1[lo:hi], data.args2[lo:hi], neg1[:, lo:hi].ravel(), neg2[:, lo:hi].ravel()])
    rows = {"W": np.unique(data.indices[data.indptr[lo]:data.indptr[hi]]), "A": np.unique(ent), "Ab": np.unique(ent)}
    for name, a in params.items():
        if name in rows:
            r = rows[name]
            width = int(np.prod(a.shape[1:]))
            if r.size * width > DUMP_MAX_ELEMS:
                r = np.sort(np.random.default_rng(0).choice(r, DUMP_MAX_ELEMS // width, replace=False))
            a = a[r]
        elif a.size > DUMP_MAX_ELEMS:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, DUMP_MAX_ELEMS, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def _measure(args, wl, wl_name, rank, world, local_rank, dist, steps, warmup, min_time, with_e2e=True, with_phases=True,
             dump_dir=None):
    """Throughput of one workload: device-resident, end to end, per-phase.  Returns (line fragment dict, engine params for
    the CPU leg or None, data tuple).  With ``dump_dir`` the parameters after the device-resident timed steps are written
    there (``_dump_outputs``)."""
    import torch

    from relation_autoencoder_b200.engine import Engine
    dev = torch.device("cuda", local_rank)
    prof_steps = 5
    B = wl["B"]
    n_ex = min(wl["N_train"], _needed_examples(wl, 2 * steps, 2 * warmup, prof_steps))
    n_ex = (n_ex // B) * B
    data, params, neg1, neg2 = _make_inputs(wl, n_ex, rank=rank, uniform=args.uniform)
    nb = data.n // B

    if world > 1:
        from relation_autoencoder_b200.dist import DistributedEngine
        eng = DistributedEngine(wl["model"], wl["K"], wl["d"], wl["S"], B, wl["F"], wl["N"], wl["N_train"], lr=0.1,
                                l2=wl.get("l2", 0.0), alpha=wl.get("alpha", 1.0), device=local_rank, rank=rank, world=world,
                                peer_dense_max_bytes=int(args.peer_dense_max_mb * (1 << 20)))
    else:
        eng = Engine(wl["model"], wl["K"], wl["d"], wl["S"], B, wl["F"], wl["N"], wl["N_train"], lr=0.1,
                     l2=wl.get("l2", 0.0), alpha=wl.get("alpha", 1.0), device=local_rank, flags=(128 if args.no_pdl else 0) | args.engine_flags)
    eng.set_params_numpy(params)
    del params

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # bind-time work (static features: per-batch sort / routing plans, once per run) and per-epoch work (negatives are
    # redrawn every epoch, OieInduction.py:183-184: device copy + multi-GPU routing plans) - reported, then amortised
    barrier()
    t0 = time.perf_counter()
    eng.bind_split("train", data.indptr, data.indices, data.args1, data.args2)
    barrier()
    t_bind = time.perf_counter() - t0
    t0 = time.perf_counter()
    eng.bind_epoch_negatives(neg1, neg2)
    barrier()
    t_epoch = time.perf_counter() - t0
    pinned1 = torch.from_numpy(neg1).pin_memory()
    pinned2 = torch.from_numpy(neg2).pin_memory()

    def timed(fn, first_batch, min_time_s):
        """Rounds of exactly `steps` steps; every rank takes the same decisions (they see the max-reduced times)."""
        for s in range(warmup):
            fn((first_batch + s) % nb)
        rounds, walls = [], []
        nxt = first_batch + warmup
        while True:
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0 = time.perf_counter()
            e0.record()
            for s in range(steps):
                fn((nxt + s) % nb)
            e1.record()
            barrier()
            wall = time.perf_counter() - t0
            ms = e0.elapsed_time(e1)
            if dist is not None:
                t = torch.tensor([ms, wall * 1e3], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms, wall = float(t[0]), float(t[1]) / 1e3
            rounds.append(ms)
            walls.append(wall)
            nxt += steps
            if sum(rounds) >= min_time_s * 1e3 or len(rounds) >= args.max_rounds:
                break
        k = int(np.argsort(rounds)[len(rounds) // 2])       # the median round
        return rounds[k], walls[k], rounds

    # ---- (1) device-resident throughput ----
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_dev, _, rounds_dev = timed(lambda b: eng.train_device(b, want_cost=False), 0, min_time)
    clocks = sampler.stop() if rank == 0 else None
    st = eng.stats()
    if dump_dir:
        params_after = eng.get_params_numpy()          # collective for N > 1
        if rank == 0:
            _dump_outputs(dump_dir, params_after, data, neg1, neg2, (warmup + len(rounds_dev) * steps - 1) % nb, B)
        del params_after
    # ---- (2) end to end through the reference-facing call: host negatives in, cost out, every step ----
    ms_e2e = None
    if with_e2e:
        n1np, n2np = pinned1.numpy(), pinned2.numpy()

        def e2e_step(b):
            eng.train(b, n1np[:, b * B:(b + 1) * B], n2np[:, b * B:(b + 1) * B])
        ms_e2e, wall_e2e, _ = timed(e2e_step, (warmup + steps) % nb, min_time / 2)
        ms_e2e = max(ms_e2e, wall_e2e * 1e3)       # host-side staging counts
    # ---- (3) per-phase device times for the roofline of the dominant kernel ----
    phase_ms = None
    dist_phase_ms = None
    timeline = None
    if with_phases and world > 1:
        eng.set_profiling(True)
        for s in range(20):
            eng.train_device((2 * (warmup + steps) + s) % nb, want_cost=False)
        dist_phase_ms = eng.phase_times_ms()
        eng.set_profiling(False)
        if hasattr(eng, "set_timeline"):
            eng.set_timeline(True)
            tls = []
            for r in range(5):
                for s in range(6):
                    eng.train_device((2 * (warmup + steps) + 20 + 6 * r + s) % nb, want_cost=False)
                tls.append(eng.timeline())
            eng.set_timeline(False)
            timeline = [[tls[0][i][0], tls[0][i][1], round(float(np.median([t[i][2] for t in tls])), 1)] for i in range(len(tls[0]))]
    if with_phases and world == 1:
        eng.set_profiling(True)
        acc = {}
        for s in range(prof_steps):
            eng.train_device((2 * (warmup + steps) + s) % nb, want_cost=False)
            for k, v in eng.phase_times_ms().items():
                acc[k] = acc.get(k, 0.0) + v / prof_steps
        eng.set_profiling(False)
        phase_ms = acc
        st = eng.stats()
        # the overlapped step's real schedule: an event behind every kernel group on its own stream (median of 9 steps)
        eng.set_profiling(2)
        tls = []
        for r in range(7):
            # several steps back to back, the LAST one read: the host runs ahead as in the timed loop (a step read right
            # after a synchronise starts with ~40 us of launch latency that the steady state does not have)
            for s in range(6):
                eng.train_device((2 * (warmup + steps) + prof_steps + 6 * r + s) % nb, want_cost=False)
            tls.append(eng.timeline())
        eng.set_profiling(False)
        timeline = [[tls[0][i][0], tls[0][i][1], round(float(np.median([t[i][2] for t in tls])), 1)] for i in range(len(tls[0]))]

    p_cpu = eng.get_params_numpy() if (world == 1 and not args.no_cpu_baseline and with_e2e) else None
    eng.close()                      # collective for N > 1 (nobody unmaps peer memory while a peer may still read it)
    pk = _peaks()
    ms_step = ms_dev / steps
    value = world * B * steps / (ms_dev * 1e-3)
    alg_bytes = st["algorithmic_bytes"]
    nnz = st["nnz"]
    flops = SY.algorithmic_flops(wl["model"], wl["K"], wl["d"], wl["S"], B, nnz)
    # epoch-level throughput: the bind / per-epoch costs measured on this run's n_ex examples, scaled to the nominal epoch
    scale = wl["N_train"] / float(max(n_ex, 1))
    epoch_steps_s = (wl["N_train"] / float(B)) * ms_step * 1e-3
    frag = {
        "value": value, "ms_per_step": ms_step, "rounds": len(rounds_dev), "timed_region_s": sum(rounds_dev) * 1e-3,
        "round_ms_min_med_max": [min(rounds_dev) / steps, ms_step, max(rounds_dev) / steps],
        "clocks": clocks,
        "gpu_launches": int(st["kernel_launches"]) * steps,
        "step_stats": {"nnz": int(nnz), "unique_w_rows": int(st["unique_w_rows"]), "unique_e_rows": int(st["unique_e_rows"]),
                       "entity_occ": int(st["entity_occ"]), "kernel_launches_per_step": int(st["kernel_launches"]),
                       "tensor_path": int(st["tensor_path"]), "algorithmic_bytes": alg_bytes, "algorithmic_flops": flops},
        "step_roofline": {"bound": "hbm", "achieved": alg_bytes / (ms_step * 1e-3) / 1e9, "peak": pk["hbm_gbs"], "unit": "GB/s",
                          "frac": alg_bytes / (ms_step * 1e-3) / 1e9 / pk["hbm_gbs"], "of": pk["source"],
                          "note": "whole step: SURVEY 8(d) algorithmic bytes / device time per step"},
        "setup_s": {"bind_split": t_bind, "bind_epoch_negatives": t_epoch, "examples_bound": int(n_ex),
                    "note": "bind_split = per-batch feature sort (1 GPU) / feature routing plans (N GPUs), once per run; "
                            "bind_epoch_negatives = negatives to the device (+ entity routing plans at N GPUs), once per EPOCH"},
        "epoch_level": {"value": world * wl["N_train"] / (epoch_steps_s + t_epoch * scale), "unit": UNIT,
                        "note": "nominal epoch of N_train examples per GPU: steps + the per-epoch setup scaled from the bound sample"},
    }
    if ms_e2e is not None:
        frag["e2e"] = {"value": world * B * steps / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 2 * wl["S"] * B * 4,
                       "d2h_bytes_per_step": 8, "ms_per_step": ms_e2e / steps,
                       "api": "Engine.train(batch_index, neg1, neg2) == func['train'] (OieInduction.py:189): dataset bound on the "
                              "device once, host negatives copied per step, cost read back per step"}
    if dist_phase_ms:
        frag["dist_phase_ms"] = {k: round(v, 5) for k, v in dist_phase_ms.items()}
    if phase_ms is not None:
        frag["phase_ms"] = {k: round(v, 5) for k, v in phase_ms.items()}
    if timeline is not None:
        frag["timeline_us"] = timeline
    return frag, st, phase_ms, p_cpu, (data, neg1, neg2)


def _run_ours(args, wl, rank, world, local_rank):
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the hot path has no CPU fallback (use --impl reference for the CPU arm)")
    dist = None
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    steps, warmup = args.steps, args.warmup
    parity = _parity_check(args, rank, world, local_rank, dist) if args.check else None
    tf32_peak = _measure_tf32_peak(dev) if rank == 0 else None
    frag, st, phase_ms, p_cpu, (data, neg1, neg2) = _measure(args, wl, args.workload, rank, world, local_rank, dist, steps, warmup,
                                                             args.min_time, dump_dir=args.dump_outputs)
    extra = {}
    if world == 1 and args.workload != "cfg2" and not args.no_extra:
        wl2 = dict(SY.WORKLOADS["cfg2"])
        f2, st2, ph2, _, _ = _measure(args, wl2, "cfg2", rank, world, local_rank, dist, steps, warmup, args.min_time / 2,
                                      with_e2e=False, with_phases=True)
        extra["cfg2"] = {"config": _config(wl2, args, world, "cfg2"), "value": f2["value"], "unit": UNIT, "ms_per_step": f2["ms_per_step"],
                         "rounds": f2["rounds"], "step_roofline": f2["step_roofline"], "phase_ms": f2.get("phase_ms"), "timeline_us": f2.get("timeline_us"),
                         "step_stats": f2["step_stats"]}
    if dist is not None:
        dist.destroy_process_group()
    if rank != 0:
        return None
    pk = _peaks()
    B = wl["B"]
    line = {
        "metric": METRIC, "value": frag["value"], "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": frag["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": _config(wl, args, world, args.workload),
    }
    for k in ("rounds", "timed_region_s", "round_ms_min_med_max", "clocks", "e2e", "gpu_launches", "step_stats", "step_roofline",
              "setup_s", "epoch_level", "dist_phase_ms", "phase_ms", "timeline_us"):
        if k in frag:
            line[k] = frag[k]
    if parity is not None:
        line.update(parity)
    if tf32_peak is not None:
        line["tf32_peak_tflops_measured"] = tf32_peak
    if phase_ms is not None:
        line["roofline"] = _roofline(wl, st, phase_ms, pk, args.workload, frag["step_roofline"], tf32_peak)
        try:
            line["tensor_kernels"] = _tensor_kernels(wl, st, phase_ms, pk, tf32_peak)
        except Exception as e:          # a reporting extra must never cost the bench line
            line["tensor_kernels"] = {"error": repr(e)}
    if extra:
        line["extra"] = extra
    if world == 1 and not args.no_cpu_baseline:
        n_cpu = min(data.n // B, 3) * B
        sub = SY.SyntheticData(data.indptr[: n_cpu + 1], data.indices[: data.indptr[n_cpu]], data.args1[:n_cpu],
                               data.args2[:n_cpu], data.neg_cum, n_cpu)
        eps, sec, done = cpu_reference_steps(wl, sub, p_cpu, neg1[:, :n_cpu], neg2[:, :n_cpu], steps=4, warmup=1,
                                             budget_s=args.cpu_budget)
        eps_sp, sec_sp, done_sp = cpu_reference_steps(wl, sub, p_cpu, neg1[:, :n_cpu], neg2[:, :n_cpu], steps=4, warmup=1,
                                                      budget_s=args.cpu_budget / 2, sparse_rows=True)
        line["cpu_baseline"] = {
            "value": eps, "unit": UNIT, "cores": _host_threads(), "kind": "port",
            "sample": "%d steps of batch %d of the same workload, NumPy float64 port of the reference graph with its dense "
                      "AdaGrad sweep (Theano not installable offline); %.2f s/step" % (done, B, sec),
            "sparse_row_variant": {"value": eps_sp, "sec_per_step": sec_sp,
                                   "note": "same math, touched rows only (what a tuned CPU port would do)"}}
    return line


PHASE_KERNELS = {      # phase -> the kernel it times (rae.h: one phase = one kernel of the step plus small helpers)
    "encoder_forward": "k_encoder_forward_v4", "entity_sort": "k_radix_sort<1> (own cooperative radix sort)",
    "operand_prep": "k_tc_prep_c + k_tc_prep_qt", "contract_forward": "k_tc_bilinear (forward)", "score": "k_score",
    "entity_update": "k_rows_chunk<1> + k_entity_long2", "w_update": "k_rows_chunk<0> + k_w_long2",
    "contract_recompute": "k_tc_bilinear (recompute)", "contract_dq": "k_tc_transpose_al + k_tc_dq", "backward_finish": "k_tc_bwd_finish",
    "contract_dc": "k_tc_dc", "dense_finalize": "k_dense_finalize (+ fused optimiser rule)", "cost": "k_cost", "dense_apply": "k_dense_apply (regulariser path only)",
}


def _traffic(workload, phase):
    """DRAM bytes per launch of the phase's kernel from the committed `ncu --set full` capture (profiles/r02_traffic.json,
    made by profiles/make_traffic.py; the round-1 file as a fallback); None when that kernel was not captured."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", name)))
            v = t.get(workload, {}).get(phase, {}).get("dram_bytes_per_launch")
            if v is not None:
                return v
        except Exception:
            continue
    return None


def _tensor_kernels(wl, st, phase_ms, pk, tf32_peak):
    """Tensor roofline of the four contraction phases (always reported, whichever kernel dominates the step): algorithmic
    2*B*(d+2)*d*K flop of one contraction / the phase's device time (the phase includes the small transposed-view / combine
    helpers beside the tcgen05 kernel, so the kernel itself is slightly faster) against the TF32 cuBLAS GEMM measured in
    this run (`frac`).  The kernels ISSUE 3x the algorithmic flops as kind::f16 MMAs (hi.hi + hi.lo + lo.hi on FP16 pairs),
    whose rate is the bf16 one: `issued_frac` = 3 x achieved / the measured bf16 burst peak (MEASURED_PEAKS.json)."""
    if not int(st.get("tensor_path", 0)):
        return None
    K, d, B = wl["K"], wl["d"], wl["B"]
    units = (d if wl["model"] in ("rescal", "rescal+sp") else 0) + (2 if wl["model"] in ("sp", "rescal+sp") else 0)
    gemm = 2.0 * B * units * d * K
    peak = tf32_peak if tf32_peak else pk["bf16_burst"] / 2.0
    out = {"issued_peak_tflops": pk["bf16_burst"], "peak_tflops": peak, "peak_is": "TF32 cuBLAS GEMM 8192^3 measured in this run" if tf32_peak else "bf16 burst / 2 (fallback)",
           "algorithmic_flops_per_launch": gemm}
    for ph in ("contract_forward", "contract_recompute", "contract_dq", "contract_dc"):
        ms = phase_ms.get(ph)
        if ms and ms > 0:
            ach = gemm / (ms * 1e-3) / 1e12
            out[ph] = {"ms": round(ms, 5), "tflops": round(ach, 1), "frac": round(ach / peak, 4),
                       "issued_frac": round(3.0 * ach / pk["bf16_burst"], 4)}
    return out


def _roofline(wl, st, phase_ms, pk, workload, step_roofline, tf32_peak):
    """Roofline of the kernel with the largest share of the step: SURVEY 8(d) algorithmic bytes / flops of ONE launch
    divided by its duration (CUDA events around the kernel on its stream, averaged over the profiled steps).  The bytes
    of a kernel are the 8(d) terms that kernel is the one to move: the W-row gather (4 nnz K) belongs to the encoder, the
    entity-row gather (4 (2+2S) B (d+1)) to the scoring kernel; the update kernels get the row read-modify-writes and the
    sorted occurrence ids only.  When no kernel holds 30 % of the step, the whole-step figure is the primary roofline."""
    K, d, S, B = wl["K"], wl["d"], wl["S"], wl["B"]
    nnz, UW, UE = st["nnz"], st["unique_w_rows"], st["unique_e_rows"]
    hasM = wl["model"] in ("rescal", "rescal+sp")
    hasSP = wl["model"] in ("sp", "rescal+sp")
    units = (d if hasM else 0) + (2 if hasSP else 0)
    occ = (2 + 2 * S) * B
    bytes_of = {
        "encoder_forward": 4.0 * nnz * K + 4.0 * nnz + 8.0 * B * K,
        "w_update": 16.0 * UW * K + 8.0 * nnz,
        "entity_update": 16.0 * UE * (d + 1) + 8.0 * occ,
        "score": 4.0 * (2 * S) * B * (d + 1) + 4.0 * 2 * S * B,
        "dense_apply": 16.0 * (units * d * K + K),
        "dense_finalize": 8.0 * (units * d * K + K),
    }
    gemm = 2.0 * B * units * d * K
    flops_of = {"contract_forward": gemm, "contract_recompute": gemm, "contract_dq": gemm, "contract_dc": gemm}
    cand = {k: v for k, v in phase_ms.items() if k in bytes_of or k in flops_of}
    name = max(cand, key=lambda k: cand[k])
    t = phase_ms[name] * 1e-3
    total = sum(phase_ms.values())
    share = phase_ms[name] / total
    common = {"kernel": PHASE_KERNELS.get(name, name), "phase": name, "ms_per_launch": phase_ms[name],
              "share_of_step": share, "of": pk["source"], "traffic": _traffic(workload, name)}
    if name in flops_of:
        ach = flops_of[name] / t / 1e12
        if tf32_peak:
            peak, what = tf32_peak, "TF32 cuBLAS GEMM 8192^3 measured in this run (burst)"
        else:
            peak, what = pk["bf16_burst"] / 2.0, "half the measured bf16 burst peak (no TF32 measurement available)"
        kern = dict(common, bound="tensor", achieved=ach, peak=peak, unit="TFLOP/s", frac=ach / peak,
                    algorithmic_flops_per_launch=flops_of[name], issued_frac=3.0 * ach / peak,
                    note="algorithmic flops 2*B*(d+2)*d*K per launch over " + what + "; the kernel issues 3x that in TF32 "
                         "(hi.hi + hi.lo + lo.hi), so the ceiling of `frac` is 1/3 and `issued_frac` is the tensor-pipe share")
    else:
        ach = bytes_of[name] / t / 1e9
        kern = dict(common, bound="hbm", achieved=ach, peak=pk["hbm_gbs"], unit="GB/s", frac=ach / pk["hbm_gbs"],
                    algorithmic_bytes_per_launch=bytes_of[name])
    if share >= 0.30:
        return kern
    return dict(step_roofline, kernel="whole step (no kernel holds 30 % of it)", traffic=None, dominant_kernel=kern)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--workload", choices=sorted(SY.WORKLOADS), default="T")
    ap.add_argument("--min-time", type=float, default=0.0, help="repeat the K-step round until this many seconds are timed "
                    "(0: one round, exactly K timed steps)")
    ap.add_argument("--max-rounds", type=int, default=400)
    ap.add_argument("--check", dest="check", action="store_true", default=True, help="parity check of one small sharded step (default)")
    ap.add_argument("--no-check", dest="check", action="store_false")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra cfg2 record")
    ap.add_argument("--uniform", action="store_true", help="uniform instead of Zipf feature ids")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--peer-dense-max-mb", type=float, default=16.0, help="N GPUs: remote dense-gradient bytes per rank up to which the "
                    "dense update sums the peers' buffers itself; above it NCCL's all-reduce runs beside the sparse-row applies")
    ap.add_argument("--engine-flags", type=int, default=0, help="extra RAE_FLAG_* bits for the 1-GPU engine (4 = force the SIMT contraction)")
    ap.add_argument("--no-pdl", action="store_true", help="RAE_FLAG_NO_PDL: plain stream-order launches (A/B of programmatic dependent launch)")
    ap.add_argument("--cpu-budget", type=float, default=45.0, help="seconds of CPU work allowed for the CPU legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the parameters after the last timed step as "
                    "DIR/<name>.npy (float32, a fixed sample of the rows the last step touched; under 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the timed GPU path computed: --impl ours only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world == 1 and args.gpus > 1 and args.impl == "ours":
        raise SystemExit("launch with: python -m torch.distributed.run --nnodes=1 --nproc-per-node %d --master-addr 127.0.0.1 "
                         "bench.py --gpus %d ..." % (args.gpus, args.gpus))
    wl = dict(SY.WORKLOADS[args.workload])
    if args.impl == "reference":
        run_reference(args, wl, rank, world)
    else:
        run_ours(args, wl, rank, world, local_rank)


if __name__ == "__main__":
    main()
