"""bench.py's pure-Python reporting logic (no GPU): the roofline of the dominant kernel follows SURVEY 8(d)'s byte terms, the
tensor table reports the four contraction phases against the measured TF32 peak, the reference arm prints a complete line."""
import importlib.util
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


PHASES_T = {"encoder_forward": 0.021, "entity_sort": 0.032, "feature_sort": 0.003, "operand_prep": 0.033, "contract_forward": 0.0747,
            "score": 0.038, "entity_update": 0.083, "w_update": 0.0485, "contract_recompute": 0.0725, "contract_dq": 0.0574,
            "backward_finish": 0.013, "contract_dc": 0.0748, "dense_finalize": 0.021, "cost": 0.011, "dense_apply": 0.003}


def test_roofline_terms_and_tensor_table():
    b = _bench()
    from relation_autoencoder_b200 import synthetic as SY
    wl = dict(SY.WORKLOADS["T"])
    st = {"nnz": 120000, "unique_w_rows": 45000, "unique_e_rows": 48000, "tensor_path": 1}
    pk = {"hbm_gbs": 6537.3, "bf16_burst": 1660.8, "bf16_sustained": 1377.6, "source": "measured"}
    step = {"bound": "hbm", "achieved": 850.0, "peak": 6537.3, "unit": "GB/s", "frac": 0.13, "of": "measured", "note": ""}
    r = b._roofline(wl, st, PHASES_T, pk, "T", step, 740.0)
    # no kernel holds 30 % of the step: the whole-step figure is primary, the largest kernel is named beside it
    assert r["kernel"].startswith("whole step") and r["dominant_kernel"]["phase"] == "entity_update"
    d, S, B = wl["d"], wl["S"], wl["B"]
    want = 16.0 * st["unique_e_rows"] * (d + 1) + 8.0 * (2 + 2 * S) * B      # row RMWs + sorted ids, no gather term
    assert abs(r["dominant_kernel"]["algorithmic_bytes_per_launch"] - want) < 1e-6
    t = b._tensor_kernels(wl, st, PHASES_T, pk, 740.0)
    gemm = 2.0 * B * (d + 2) * d * wl["K"]
    assert t["algorithmic_flops_per_launch"] == gemm
    for ph in ("contract_forward", "contract_recompute", "contract_dq", "contract_dc"):
        ach = gemm / (PHASES_T[ph] * 1e-3) / 1e12
        assert abs(t[ph]["tflops"] - ach) < 0.06 and abs(t[ph]["frac"] - ach / 740.0) < 1e-3
        assert abs(t[ph]["issued_frac"] - 3 * ach / 1660.8) < 1e-3
    assert b._tensor_kernels(dict(SY.WORKLOADS["cfg4"]), {"tensor_path": 0}, PHASES_T, pk, 740.0) is None


def test_dump_outputs_keeps_the_last_batch_rows_under_the_cap(tmp_path, monkeypatch):
    """--dump-outputs: float32 arrays named after the parameters; the row tables keep the rows the given batch touched,
    cut to a fixed sample when an array would exceed the per-array cap; two dumps of the same state are identical."""
    import numpy as np
    b = _bench()
    from relation_autoencoder_b200 import synthetic as SY
    F, N, K, d, S, B = 3000, 700, 6, 5, 3, 40
    data = SY.make_dataset(4 * B, F, N, 10, seed=3)
    rng = np.random.RandomState(2)
    params = SY.init_params(rng, "rescal+sp", F, K, N, d)
    params["Ab"] = np.arange(N, dtype=np.float32)            # a row's value is its id
    neg1, neg2 = SY.draw_negatives(rng, data.neg_cum, data.n, S)
    monkeypatch.setattr(b, "DUMP_MAX_ELEMS", 100)
    for out in ("a", "b"):
        b._dump_outputs(str(tmp_path / out), params, data, neg1, neg2, 2, B)
    lo, hi = 2 * B, 3 * B
    w_rows = np.unique(data.indices[data.indptr[lo]:data.indptr[hi]])
    e_rows = np.unique(np.concatenate([data.args1[lo:hi], data.args2[lo:hi], neg1[:, lo:hi].ravel(), neg2[:, lo:hi].ravel()]))
    assert w_rows.size * K > 100 and e_rows.size > 100
    got = {n: np.load(str(tmp_path / "a" / (n + ".npy"))) for n in params}
    for n, a in got.items():
        assert a.dtype == np.float32 and a.size <= 100, n
        assert np.array_equal(a, np.load(str(tmp_path / "b" / (n + ".npy")))), n
    assert got["W"].shape == (100 // K, K) and got["A"].shape == (100 // d, d) and got["Ab"].shape == (100,)
    # every dumped table row is one the batch touched
    w_table = {tuple(r) for r in params["W"][w_rows]}
    assert all(tuple(r) in w_table for r in got["W"])
    assert set(got["Ab"].astype(np.int64).tolist()) <= set(e_rows.tolist())
    assert np.array_equal(got["Wb"], params["Wb"]) and got["C"].shape == (100,)
    assert set(got["C"].tolist()) <= set(params["C"].ravel().tolist())


def test_reference_arm_prints_a_complete_line():
    """`bench.py --impl reference` (the NumPy float64 port of the reference's CPU path; the README-size config keeps it short)."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "cfg1", "--steps", "2",
                        "--warmup", "1"], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "examples/s" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["e2e"]["h2d_bytes_per_step"] == 0
    for k in ("metric", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "dtype", "data", "config"):
        assert k in line, k
