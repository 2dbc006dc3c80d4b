"""GPU parity tests: the CUDA path, called through the C ABI (librae.so), against the float64 oracle on identical
inputs, weights and injected negative-sample indices.

Tolerances (north_star: 1e-5 relative, fp32 storage vs the float64 run), stated per quantity:
  * index work (sort-by-row layout, segment boundaries, labels)           : bit-exact
  * cost, q(r|x)                                                          : |x - ref| <= 1e-5 * max|ref|
  * per-parameter gradients (dense, what T.grad would return)             : ||g - ref||_inf <= 1e-5 * ||ref||_inf
  * the optimiser step itself: p_after vs AdaGrad(p_before, g_gpu) in f64 : <= 2e-6 * max(|p|, lr)
"""
import numpy as np
import pytest

from oracle import rae_oracle as O
from tests.helpers import make_problem, record_err, rel_err, tc_eligible

pytestmark = pytest.mark.gpu

TOL_COST = 1e-5
TOL_Q = 1e-5
TOL_GRAD = 1e-5          # the north star's tolerance; measured margins are logged through tests.helpers.record_err
FLAG_FORCE_SIMT = 4
FLAG_FORCE_TENSOR = 8
FLAG_DENSE = 2

SHAPES = {
    "tiny": dict(B=12, K=5, d=6, S=3, F=40, N=25, fbar=4),
    "readme": dict(B=100, K=10, d=10, S=5, F=300, N=150, fbar=14),     # config 1 sizes (README run)
    "odd": dict(B=37, K=7, d=33, S=2, F=90, N=60, fbar=5),             # nothing a multiple of 4 / 32
    "k100d30": dict(B=64, K=100, d=30, S=5, F=500, N=300, fbar=30),    # config 2 per-example shape
    "k100d128": dict(B=40, K=100, d=128, S=4, F=400, N=200, fbar=20),  # config 3 / target per-example shape
    "k130d70": dict(B=24, K=130, d=70, S=3, F=200, N=100, fbar=8),     # K chunked, d between tiles
    "b512d128": dict(B=512, K=100, d=128, S=4, F=3000, N=900, fbar=20),  # 4 example tiles: cluster of 4, operand multicast
    "b256d30": dict(B=256, K=100, d=30, S=5, F=2000, N=700, fbar=30),    # 2 example tiles: cluster of 2
}
HOT_SHAPES = {      # batches for make_problem(hot_rows=True)
    "k100d128": dict(B=512, K=100, d=128, S=4, F=3000, N=900, fbar=20),  # row widths multiples of 4: 16-byte row accesses
    "k7d33": dict(B=512, K=7, d=33, S=4, F=3000, N=900, fbar=20),        # neither width a multiple of 4
}


def _engine(model, sh, flags=FLAG_DENSE, **kw):
    from relation_autoencoder_b200.engine import Engine
    return Engine(model, sh["K"], sh["d"], sh["S"], sh["B"], sh["F"], sh["N"], kw.pop("n_train", sh["B"]), flags=flags, **kw)


def _to32(p):
    # the GPU stores fp32: the oracle must start from the same (fp32-representable) values
    return {k: v.astype(np.float32).astype(np.float64) for k, v in p.items()}


def _check_step(model, sh, seed=0, dup_heavy=False, empty_rows=False, l1=0.0, l2=0.0, ext_reg=True, alpha=1.0,
                optimizer="adagrad", lr=0.1, steps=1, flags=FLAG_DENSE, hot_rows=False):
    pr = make_problem(model, seed=seed, dup_heavy=dup_heavy, empty_rows=empty_rows, hot_rows=hot_rows, **sh)
    p0 = _to32(pr["p"])
    names = O.param_names(model)
    adj = 0.37
    om = O.OracleModel(model, {k: v.copy() for k, v in p0.items()}, K=sh["K"], d=sh["d"], S=sh["S"], B=sh["B"], lr=lr,
                       l1=l1, l2=l2, alpha=alpha, optimizer=optimizer, ext_reg=ext_reg)
    eng = _engine(model, sh, flags=flags, lr=lr, l1=l1, l2=l2, alpha=alpha, optimizer=optimizer, ext_reg=ext_reg, adj=adj)
    eng.set_params_numpy(p0)
    rng = np.random.RandomState(seed + 100)
    for step in range(steps):
        neg1 = pr["neg1"] if step == 0 else rng.randint(0, sh["N"], size=pr["neg1"].shape).astype(np.int32)
        neg2 = pr["neg2"] if step == 0 else rng.randint(0, sh["N"], size=pr["neg2"].shape).astype(np.int32)
        before = eng.get_params_numpy()
        acc_before = eng.get_acc_numpy()
        # the oracle step is evaluated at the GPU's current parameters so each step is an independent check
        om.params = {k: before[k].astype(np.float64) for k in names}
        om.acc = {k: acc_before[k].astype(np.float64) for k in names}
        c_ref = om.train_explicit(pr["indptr"], pr["indices"], pr["a1"], pr["a2"], neg1, neg2, adj=adj)
        c_gpu = eng.train_explicit(pr["indptr"], pr["indices"], pr["a1"], pr["a2"], neg1, neg2)
        assert abs(c_gpu - c_ref) <= TOL_COST * max(1.0, abs(c_ref)), (step, c_gpu, c_ref)
        assert rel_err(eng.last_probs(), om.last_q) <= TOL_Q
        g_gpu = eng.dense_grads()
        for n in names:
            e = rel_err(g_gpu[n], om.last_grads[n])
            record_err("step:%s:K%dd%dB%d:flags%d" % (model, sh["K"], sh["d"], sh["B"], flags), n, e)
            assert e <= TOL_GRAD, (step, n, e)
        # the contraction path that ran is the one the shape calls for: a silent SIMT fallback must not pass
        want_tc = tc_eligible(model, sh["K"], sh["d"]) and not (flags & FLAG_FORCE_SIMT)
        assert int(eng.stats()["tensor_path"]) == (1 if want_tc else 0), (model, sh, flags)
        # optimiser rule applied to the GPU's own gradient (Optimizers.py:29-32 / :51)
        after = eng.get_params_numpy()
        acc_after = eng.get_acc_numpy()
        for n in names:
            g = g_gpu[n].astype(np.float64)
            if optimizer == "adagrad":
                acc = acc_before[n].astype(np.float64) + g * g
                exp = before[n].astype(np.float64) - lr * g / (np.sqrt(acc) + 1e-6)
                assert np.abs(acc_after[n] - acc).max() <= 2e-6 * max(acc.max(), 1e-30), n
            else:
                exp = before[n].astype(np.float64) - lr * g
            scale = max(float(np.abs(exp).max()), lr)
            assert np.abs(after[n] - exp).max() <= 2e-6 * scale, (step, n)
    eng.close()


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("model", O.MODELS)
def test_step_matches_oracle(model, shape):
    _check_step(model, SHAPES[shape], seed=1)


@pytest.mark.parametrize("shape", ["b512d128", "b256d30"])
def test_cluster_flag_is_accepted(shape):
    """RAE_FLAG_CLUSTER_MULTICAST (64) is still accepted (the multicast variant was removed: no gain on B200)."""
    _check_step("rescal+sp", SHAPES[shape], seed=2, flags=FLAG_DENSE | 64)


@pytest.mark.parametrize("shape", ["k100d30", "k100d128", "b512d128", "b256d30"])
@pytest.mark.parametrize("model", ["rescal", "rescal+sp"])
def test_tensor_and_simt_paths_both_match_oracle(model, shape):
    """The same problem through the tcgen05 contraction (RAE_FLAG_FORCE_TENSOR) and through the SIMT contraction
    (RAE_FLAG_FORCE_SIMT): each is held to the oracle, and _check_step asserts which path ran."""
    _check_step(model, SHAPES[shape], seed=3, flags=FLAG_DENSE | FLAG_FORCE_TENSOR)
    _check_step(model, SHAPES[shape], seed=3, flags=FLAG_DENSE | FLAG_FORCE_SIMT)


def test_force_tensor_rejects_unsupported_shape():
    with pytest.raises(RuntimeError):
        _engine("rescal+sp", SHAPES["k130d70"], flags=FLAG_FORCE_TENSOR)


@pytest.mark.parametrize("model", O.MODELS)
def test_duplicate_rows_are_summed_before_squaring(model):
    """Duplicates (same entity as e1, e2 and several negatives) accumulate first (AdvancedIncSubtensor1), then AdaGrad
    squares the SUM - SURVEY 7.3-4."""
    _check_step(model, SHAPES["tiny"], seed=4, dup_heavy=True, steps=3)
    _check_step(model, SHAPES["readme"], seed=5, dup_heavy=True, steps=2)


@pytest.mark.parametrize("model", O.MODELS)
def test_empty_feature_rows(model):
    _check_step(model, SHAPES["tiny"], seed=6, empty_rows=True)


@pytest.mark.parametrize("model", O.MODELS)
@pytest.mark.parametrize("reg", [(0.0, 0.1, True), (0.02, 0.05, True), (0.0, 0.1, False)])
def test_regulariser_makes_w_gradient_dense(model, reg):
    """README/test.py configs use l2 = 0.1 (README.md:44, test.py:16,33): every row of W moves every step."""
    l1, l2, ext = reg
    _check_step(model, SHAPES["readme"], seed=7, l1=l1, l2=l2, ext_reg=ext, alpha=0.1, steps=2)


@pytest.mark.parametrize("model", O.MODELS)
def test_sgd(model):
    _check_step(model, SHAPES["tiny"], seed=8, optimizer="sgd", steps=2)


def _chunk_spans(keys):
    """Chunks of 32 positions that each row's segment covers in the stable sort by row (the row-update kernels' layout)."""
    s = np.sort(keys, kind="stable")
    starts = np.flatnonzero(np.r_[True, s[1:] != s[:-1]])
    ends = np.r_[starts[1:], len(s)]
    return (ends - 1) // 32 - starts // 32 + 1


@pytest.mark.parametrize("optimizer", ["adagrad", "sgd"])
@pytest.mark.parametrize("shape", list(HOT_SHAPES))
@pytest.mark.parametrize("model", O.MODELS)
def test_hot_rows_take_every_row_update_path(model, shape, optimizer):
    """Rows of 2 chunks (feature rows: absorbed by level 1), of 3-9 chunks (level 2, one warp) and of 10 or more chunks
    (level 2, the whole CTA), on both feature and entity rows, held to the oracle."""
    sh = HOT_SHAPES[shape]
    pr = make_problem(model, seed=13, hot_rows=True, **sh)
    feature_keys = pr["indices"]
    entity_keys = np.concatenate([pr["a1"], pr["a2"], pr["neg1"].reshape(-1), pr["neg2"].reshape(-1)])
    for keys in (feature_keys, entity_keys):
        spans = _chunk_spans(keys)
        assert (spans == 2).any() and ((spans >= 3) & (spans <= 9)).any() and (spans >= 10).any(), np.bincount(spans)
    _check_step(model, sh, seed=13, hot_rows=True, optimizer=optimizer)


@pytest.mark.parametrize("model", O.MODELS)
def test_production_path_without_dense_grads_matches_debug_path(model):
    """The flag that materialises dense gradients must not change the update (bitwise)."""
    for sh, pr in ((SHAPES["k100d30"], make_problem(model, seed=9, dup_heavy=True, **SHAPES["k100d30"])),
                   (HOT_SHAPES["k7d33"], make_problem(model, seed=13, hot_rows=True, **HOT_SHAPES["k7d33"]))):
        res = []
        for flags in (FLAG_DENSE, 0, 16):       # debug, production (cached feature index n/a for explicit), no cache
            eng = _engine(model, sh, flags=flags)
            eng.set_params_numpy(_to32(pr["p"]))
            c = eng.train_explicit(pr["indptr"], pr["indices"], pr["a1"], pr["a2"], pr["neg1"], pr["neg2"])
            res.append((c, eng.get_params_numpy(), eng.get_acc_numpy()))
            eng.close()
        for c, p, a in res[1:]:
            assert c == res[0][0]
            for n in p:
                assert np.array_equal(p[n], res[0][1][n]) and np.array_equal(a[n], res[0][2][n]), n


def test_sort_segment_layout_is_bit_exact():
    """sort-by-row layout == np.argsort(kind='stable'), segments == np.unique boundaries (SURVEY 8c)."""
    sh = SHAPES["readme"]
    pr = make_problem("AC", seed=10, dup_heavy=True, **sh)
    eng = _engine("AC", sh)
    eng.set_params_numpy(_to32(pr["p"]))
    eng.train_explicit(pr["indptr"], pr["indices"], pr["a1"], pr["a2"], pr["neg1"], pr["neg2"])
    rows, occ, seg = eng.entity_segments()
    keys = np.concatenate([pr["a1"], pr["a2"], pr["neg1"].reshape(-1), pr["neg2"].reshape(-1)])
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(occ, order.astype(np.int32))
    assert np.array_equal(rows, keys[order])
    uniq, first = np.unique(keys[order], return_index=True)
    assert np.array_equal(seg[:-1], first.astype(np.int32)) and seg[-1] == len(keys)
    assert eng.stats()["unique_e_rows"] == len(uniq)
    assert eng.stats()["unique_w_rows"] == len(np.unique(pr["indices"]))
    eng.close()


@pytest.mark.parametrize("model", O.MODELS)
def test_bitwise_reproducible(model):
    sh = SHAPES["k100d30"]
    pr = make_problem(model, seed=11, dup_heavy=True, **sh)
    outs = []
    for _ in range(2):
        eng = _engine(model, sh, flags=0)
        eng.set_params_numpy(_to32(pr["p"]))
        costs = [eng.train_explicit(pr["indptr"], pr["indices"], pr["a1"], pr["a2"], pr["neg1"], pr["neg2"]) for _ in range(3)]
        outs.append((costs, eng.get_params_numpy()))
        eng.close()
    assert outs[0][0] == outs[1][0]
    for n in outs[0][1]:
        assert np.array_equal(outs[0][1][n], outs[1][1][n]), n


@pytest.mark.parametrize("model", O.MODELS)
def test_bound_split_api_matches_reference_callables(model):
    """func['train'](batch_index, neg1, neg2) and func['label_train'](batch_index) on a bound split, several batches,
    trailing partial batch dropped (OieInduction.py:96-98,146-155,186-189)."""
    sh = dict(SHAPES["readme"])
    B = sh["B"]
    n_rows = 3 * B + 17
    pr = make_problem(model, seed=12, **{**sh, "B": n_rows})
    p0 = _to32(pr["p"])
    S = sh["S"]
    for flags in (0, 16):
        om = O.OracleModel(model, {k: v.copy() for k, v in p0.items()}, K=sh["K"], d=sh["d"], S=S, B=B, lr=0.1, alpha=1.0)
        om.bind_split("train", pr["indptr"], pr["indices"], pr["a1"], pr["a2"])
        eng = _engine(model, sh, flags=flags, n_train=n_rows)
        eng.set_params_numpy(p0)
        eng.bind_split("train", pr["indptr"], pr["indices"], pr["a1"], pr["a2"])
        assert eng.n_batches() == 3
        eng.bind_epoch_negatives(pr["neg1"], pr["neg2"])
        for b in range(3):
            n1 = pr["neg1"][:, b * B:(b + 1) * B]
            n2 = pr["neg2"][:, b * B:(b + 1) * B]
            om.params = {k: v.astype(np.float64) for k, v in eng.get_params_numpy().items()}
            om.acc = {k: v.astype(np.float64) for k, v in eng.get_acc_numpy().items()}
            c_ref = om.train(b, n1, n2)
            if b == 1:
                c_gpu = eng.train_device(b)            # device-resident epoch negatives, strided in place
            else:
                c_gpu = eng.train(b, n1, n2)           # the reference call: host [S,B] slices
            assert abs(c_gpu - c_ref) <= TOL_COST * max(1.0, abs(c_ref)), (b, c_gpu, c_ref)
            assert rel_err(eng.last_probs(), om.last_q) <= TOL_Q
        om.params = {k: v.astype(np.float64) for k, v in eng.get_params_numpy().items()}
        for b in range(3):
            lab, probs = eng.label("train", b)
            lab_ref, q_ref = om.label("train", b)
            assert lab.dtype == np.int64 and np.array_equal(lab, lab_ref)
            assert rel_err(probs, q_ref) <= TOL_Q
        with pytest.raises(RuntimeError):
            eng.train_device(3)                        # the trailing partial batch does not exist
        eng.close()


@pytest.mark.parametrize("model", ["rescal", "rescal+sp"])
def test_host_negatives_pinned_pageable_and_pipelined_steps_agree(model):
    """func['train'] returns the cost as soon as the forward pass has it and the next call is issued behind the running
    backward pass.  Page-locked column slices (strided DMA, no staging), pageable slices (pinned staging) and
    contiguous copies with a full synchronisation between steps must give bit-identical costs and parameters."""
    import torch
    sh = dict(SHAPES["readme"])
    B, S = sh["B"], sh["S"]
    nb = 6
    pr = make_problem(model, seed=21, **{**sh, "B": nb * B})
    p0 = _to32(pr["p"])
    neg = [np.ascontiguousarray(pr[k], dtype=np.int32) for k in ("neg1", "neg2")]
    pinned = [torch.from_numpy(a.copy()).pin_memory().numpy() for a in neg]
    outs = []
    for mode in ("pinned", "pageable", "synchronised"):
        eng = _engine(model, sh, flags=0, n_train=nb * B)
        eng.set_params_numpy(p0)
        eng.bind_split("train", pr["indptr"], pr["indices"], pr["a1"], pr["a2"])
        src = pinned if mode == "pinned" else neg
        costs = []
        for e in range(2):
            for b in range(nb):
                n1, n2 = (a[:, b * B:(b + 1) * B] for a in src)
                if mode == "synchronised":
                    n1, n2 = n1.copy(), n2.copy()
                costs.append(eng.train(b, n1, n2))
                if mode == "synchronised":
                    torch.cuda.synchronize()
        outs.append((costs, eng.get_params_numpy(), eng.get_acc_numpy()))
        eng.close()
    for costs, p, acc in outs[1:]:
        assert costs == outs[0][0]
        for n in p:
            assert np.array_equal(p[n], outs[0][1][n]), n
            assert np.array_equal(acc[n], outs[0][2][n]), n


def test_label_ties_first_max_wins():
    from relation_autoencoder_b200.engine import Engine
    K, F, B = 40, 8, 4
    eng = Engine("rescal", K, 4, 1, B, F, 5, B)
    W = np.zeros((F, K), dtype=np.float32)
    W[0, 7] = W[0, 33] = 2.0          # tie between 7 and 33 -> 7
    W[1, 39] = 1.0
    p = dict(W=W, Wb=np.zeros(K, np.float32), A=np.zeros((5, 4), np.float32), Ab=np.zeros(5, np.float32),
             C=np.zeros((4, 4, K), np.float32))
    eng.set_params_numpy(p)
    indptr = np.array([0, 1, 2, 2, 4], dtype=np.int32)
    indices = np.array([0, 1, 0, 1], dtype=np.int32)
    eng.bind_split("test", indptr, indices)
    lab, probs = eng.label("test", 0)
    assert lab.tolist() == [7, 39, 0, 7]
    assert np.allclose(probs[2], 1.0 / K, rtol=1e-6)
    eng.close()


def test_errors_are_reported_not_thrown_across_the_abi():
    from relation_autoencoder_b200.engine import Engine
    eng = Engine("rescal+sp", 4, 4, 2, 8, 16, 16, 8)
    with pytest.raises(RuntimeError, match="not bound"):
        eng.train_device(0)
    with pytest.raises(Exception, match="not implemented"):
        Engine("rescal+sp", 4, 4, 2, 8, 16, 16, 8, optimizer="adam")
    with pytest.raises(RuntimeError, match="unsupported sizes"):
        Engine("rescal+sp", 4, 300, 2, 8, 16, 16, 8)
    eng.close()


def test_step_timeline_marks_follow_the_streams():
    """rae_set_profiling(h, 2): the step keeps its three-stream overlap and records an event behind every kernel group on the
    stream it ran on; per stream the marks are ordered in time, the step ends after all of them (bench.py: timeline_us)."""
    sh = SHAPES["k100d128"]
    pr = make_problem("AC", seed=21, **sh)
    eng = _engine("AC", sh, flags=0)
    eng.set_params_numpy(_to32(pr["p"]))
    eng.set_profiling(2)
    for _ in range(2):
        eng.train_explicit(pr["indptr"], pr["indices"], pr["a1"], pr["a2"], pr["neg1"], pr["neg2"])
    tl = eng.timeline()
    eng.set_profiling(0)
    names = [n for n, _, _ in tl]
    assert names[0] == "start" and names[-1] == "end"
    for want in ("encoder", "contract_forward", "score", "contract_dq", "backward_finish", "contract_dc", "dense_finalize",
                 "entity_sort", "entity_update", "w_update"):
        assert want in names, (want, names)
    for stream in (0, 1, 2):
        t = [us for _, s, us in tl if s == stream]
        assert all(b >= a for a, b in zip(t, t[1:])), (stream, tl)
    assert tl[-1][2] >= max(us for _, _, us in tl) - 1e-3
    assert int(eng.stats()["tensor_path"]) == 1
    eng.close()


@pytest.mark.parametrize("model", O.MODELS)
def test_programmatic_dependent_launch_changes_no_bit(model):
    """The step's kernels are launched with programmatic stream serialization (griddepcontrol.wait before their first global
    access); RAE_FLAG_NO_PDL launches them in plain stream order.  Same data dependencies, so the same bits."""
    sh = SHAPES["b512d128"]
    pr = make_problem(model, seed=22, dup_heavy=True, **sh)
    outs = []
    for flags in (0, 128):
        eng = _engine(model, sh, flags=flags)
        eng.set_params_numpy(_to32(pr["p"]))
        costs = [eng.train_explicit(pr["indptr"], pr["indices"], pr["a1"], pr["a2"], pr["neg1"], pr["neg2"]) for _ in range(3)]
        outs.append((costs, eng.get_params_numpy(), eng.get_acc_numpy()))
        eng.close()
    assert outs[0][0] == outs[1][0]
    for n in outs[0][1]:
        assert np.array_equal(outs[0][1][n], outs[1][1][n]), n
        assert np.array_equal(outs[0][2][n], outs[1][2][n]), n
