"""Multi-GPU training from the driver and the command line: ``distributed_backend`` and ``torchrun ... -m
relation_autoencoder_b200.induction``, with the splits labelled straight from the row-sharded W.

CPU (gloo + the float64 NumPy backend, tests/dist_driver_worker.py): the README run at 2 and 4 ranks against the
single-process oracle driver's golden traces, checkpoints across world sizes, the chunked labelling fallback, the command
line.  GPU (NCCL + librae): the README run's bounds at every world size present, rae_label_shards bit-identical to a
single-GPU engine on the gathered W, labels between steps, reproducible checkpoints and the device sampler."""
import io
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from relation_autoencoder_b200 import induction as I
from relation_autoencoder_b200 import preprocess as P
from tests.oracle_backend import oracle_backend
from tests.test_dist_cpu import ROOT, _free_port

WORKER = os.path.join(ROOT, "tests", "dist_driver_worker.py")


def _run_worker(world, args, timeout=900, expect_ok=True):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr",
           "127.0.0.1", "--master-port", str(_free_port()), WORKER] + list(args)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    r = subprocess.run(cmd, cwd=ROOT, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    if expect_ok:
        assert r.returncode == 0 and "DRIVER_OK" in r.stdout, r.stdout[-4000:]
    return r


def _indexed():
    from relation_autoencoder_b200 import data as D
    return D.IndexedDataset.load_npz(os.path.join(ROOT, "tests", "golden", "data_sample_indexed.npz"))


# ---------------------------------------------------------------------------------------------------------------- CPU
@pytest.mark.parametrize("world", [1, 2, 4])
def test_readme_run_on_ranks_reproduces_golden_trace(world):
    """--batch-size 100 is the global batch (B = 50 at 2 ranks, 25 at 4): batch costs, training error and valid / test
    B-cubed of 3 epochs equal the single-process oracle driver's to 1e-12, for l2 = 0.1 and l2 = 0."""
    _run_worker(world, ["readme"])


def test_checkpoints_move_between_world_sizes(tmp_path):
    """A 2-rank checkpoint after epoch 1, resumed by the single-process oracle driver, and the oracle's epoch-1 checkpoint
    resumed on 2 ranks: both end where the uninterrupted 3-epoch oracle run ends (costs, metrics, parameters,
    accumulators to 1e-12)."""
    from tests.golden.make_readme_run import README_ARGS, SEED, run_readme
    full, ind_full = run_readme(_indexed(), oracle_backend, epochs=3, lambda2=0.1)
    _, ind1 = run_readme(_indexed(), oracle_backend, epochs=1, lambda2=0.1)
    oracle_ck = ind1.save(str(tmp_path / "oracle"))
    _run_worker(2, ["ckpt", str(tmp_path), oracle_ck])

    def same(a, b):
        return np.allclose(a, b, rtol=1e-12, atol=1e-12)
    p_full, a_full = ind_full.get_parameters(), ind_full.get_accumulators()
    # world 2 -> single process
    ck = I.load_model(str(tmp_path / "dist" / (README_ARGS["model_name"] + ".npz")))
    assert ck["config"]["epochs_done"] == 1 and ck["config"]["batch_size"] == 100
    idx = _indexed()
    ind2 = I.ReconstructInducer(idx, idx.goldStandard, np.random.RandomState(SEED + 99), backend=oracle_backend,
                                out=io.StringIO(), **dict(README_ARGS, nb_epochs=3, lambda2=0.1))
    ind2.load(str(tmp_path / "dist" / (README_ARGS["model_name"] + ".npz")))
    ind2.compile_function()
    costs = []
    train = ind2.func["train"]
    ind2.func["train"] = lambda b, n1, n2: costs.append(float(train(b, n1, n2))) or costs[-1]
    ind2.learn(debug=False)
    assert same(costs, full["batch_costs"][10:30])
    assert same(ind2.train_error_series, full["train_error"])
    for split in ("valid", "test"):
        assert same(ind2.metrics[split], full["metrics"][split])
    for k, v in p_full.items():
        assert same(ind2.get_parameters()[k], v), k
        assert same(ind2.get_accumulators()[k], a_full[k]), k
    # single process -> world 2
    ck = I.load_model(str(tmp_path / "resumed" / (README_ARGS["model_name"] + ".npz")))
    tr = json.load(open(str(tmp_path / "resumed" / "trace.json")))
    assert ck["config"]["epochs_done"] == 3
    assert same(tr["batch_costs"], full["batch_costs"][10:30])
    assert same(tr["train_error"], full["train_error"])
    for split in ("valid", "test"):
        assert same(tr["metrics"][split], full["metrics"][split])
    for k, v in p_full.items():
        assert same(ck["params"][k], v), k
        assert same(ck["acc"][k], a_full[k]), k


@pytest.mark.parametrize("world", [1, 2])
def test_label_rows_fallback_chunks_a_split_wider_than_the_compact_table(world):
    _run_worker(world, ["labels"], timeout=300)


def _pickle(tmp_path):
    lines = []
    for i in range(40):
        rel = "/r/%d" % (i % 3) if i % 4 else ""
        lines.append("->nsubj->word%d->dobj->\tAlpha%d Corp\tBeta%d Inc\tORG-ORG\tTRIGGER:word%d\t./d%d.xml\tAlpha%d Corp likes word%d "
                     "of Beta%d Inc today .\tNNP NNP VBZ NN IN NNP NNP NN .\t%s\n" % (i % 5, i % 7, i % 6, i % 5, i, i % 7, i % 5, i % 6, rel))
    src = tmp_path / "c.txt"
    src.write_text("".join(lines), encoding="utf-8")
    pk = str(tmp_path / "c.pk")
    P.main(["--batch-name", "train", str(src), pk])
    return pk


CLI = ["--model-name", "t", "--decoder", "sp", "--epochs", "2", "--relations", "4", "--embed-size", "6", "--neg-samples", "3",
       "--seed", "2", "--l2", "0.1"]


def test_command_line_on_two_ranks_end_to_end(tmp_path, monkeypatch, capsys):
    """preprocess -> pickle -> torchrun with 2 ranks -> main(): one training log (rank 0), one checkpoint, and the same
    checkpoint as the single-process command line with the oracle bound."""
    pk = _pickle(tmp_path)
    r = _run_worker(2, ["cli", str(tmp_path / "dist"), pk, "--batch-size", "10"] + CLI, timeout=600)
    out = r.stdout
    assert out.count("Relation Learner") == 1 and out.count("EPOCH 2") == 1 and out.count("Saved") == 1, out[-3000:]
    assert out.count("train f1:") == 2
    assert os.listdir(str(tmp_path / "dist")) == ["t.npz"]
    monkeypatch.setattr(I, "models_path", str(tmp_path / "single"))
    ind = I.main([pk, "--batch-size", "10"] + CLI, backend=oracle_backend)
    capsys.readouterr()
    assert ind._mode() == 1
    a, b = I.load_model(str(tmp_path / "dist" / "t.npz")), I.load_model(str(tmp_path / "single" / "t.npz"))
    for part in ("params", "acc"):
        for k, v in b[part].items():
            assert np.allclose(a[part][k], v, rtol=1e-12, atol=1e-12), (part, k)
    assert np.allclose(a["config"]["train_error"], b["config"]["train_error"], rtol=1e-12, atol=0)
    assert np.allclose(a["config"]["metrics"]["train"], b["config"]["metrics"]["train"], rtol=1e-12, atol=0)


def test_command_line_refuses_a_batch_size_the_world_does_not_divide(tmp_path):
    pk = _pickle(tmp_path)
    r = _run_worker(2, ["cli", str(tmp_path / "dist"), pk, "--batch-size", "9"] + CLI, timeout=300, expect_ok=False)
    assert r.returncode != 0
    for rank in (0, 1):
        assert ("rank %d refused: --batch-size 9 is not divisible by the world size 2" % rank) in r.stdout, r.stdout[-3000:]
    assert not os.path.exists(str(tmp_path / "dist"))


def test_command_line_refuses_an_explicit_device_on_several_ranks(tmp_path):
    pk = _pickle(tmp_path)
    r = _run_worker(2, ["cli", str(tmp_path / "dist"), pk, "--batch-size", "10", "--device", "1"] + CLI, timeout=300,
                    expect_ok=False)
    assert r.returncode != 0 and r.stdout.count("--device cannot be combined with several ranks") == 2, r.stdout[-3000:]


def test_single_rank_main_is_the_single_gpu_driver(monkeypatch):
    """WORLD_SIZE unset or 1: main() never touches torch.distributed."""
    import torch.distributed as dist
    calls = []
    monkeypatch.setattr(dist, "init_process_group", lambda *a, **k: calls.append(a))
    monkeypatch.setenv("WORLD_SIZE", "1")
    with pytest.raises(SystemExit):
        I.main([])                           # no arguments: the help text and exit(1), as before
    assert calls == []


def test_global_batch_check_names_both_numbers():
    I.check_global_batch(100, 4)
    with pytest.raises(ValueError, match="--batch-size 100 is not divisible by the world size 3"):
        I.check_global_batch(100, 3)


# ---------------------------------------------------------------------------------------------------------------- GPU
def _ngpu():
    import torch
    return torch.cuda.device_count()


def _need(world):
    if _ngpu() < world:
        pytest.skip("needs %d GPUs" % world)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4])
def test_readme_run_through_sharded_driver_meets_cuda_bounds(world):
    """test_readme_run_on_cuda_matches_oracle_trace's bounds on both traces: first batch cost 1e-5, first 10 batches 1e-3,
    per-epoch error 2e-3, test F1 0.03."""
    _need(world)
    r = _run_worker(world, ["cuda-readme"])
    print(r.stdout[-2000:])


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2, 4])
def test_label_shards_bit_identical_to_single_gpu_engine(world):
    """K = 100 (16-byte rows) and K = 10 (scalar rows); n_rows > B, an indptr offset != 0, probs = NULL, and a valid split
    whose batches exceed the compact table."""
    _need(world)
    _run_worker(world, ["cuda-labels"])


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
def test_labels_between_steps_equal_gathered_parameters(world):
    _need(world)
    _run_worker(world, ["cuda-between-steps"])


@pytest.mark.gpu
@pytest.mark.parametrize("world", [1, 2])
def test_sharded_runs_are_reproducible_and_device_sampler_matches(world, tmp_path):
    _need(world)
    _run_worker(world, ["cuda-repro", str(tmp_path)])
