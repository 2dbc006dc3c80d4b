"""Segments of the balanced tcgen05 schedule: CTAs whose range crosses an example-tile boundary run two or three segments,
each with its own P operand (forward / recompute) or X/Y register cache (dq).

CPU tier: a Python mirror of make_sched / TcSegIter / tc_init (rae_decoder_tc.cu, rae_internal.h) shows that the shapes of
the GPU tier really hold one-, two- and three-segment CTAs and CTAs that end a tile.
GPU tier: at the three-segment shape one full-size step matches the float64 oracle within the tolerances of
test_scale_fullsize (which checks T and cfg2 the same way), and the same step run twice is bit-identical.
"""
import collections

import numpy as np
import pytest

NUM_SMS = 148                 # B200
TC_DQ_MAX_STAGES = 64

# name -> (B, K, d): the segments depend on these only
SHAPES = {
    "T": dict(B=4096, K=100, d=128),        # the flagship shape
    "cfg2": dict(B=4096, K=100, d=30),      # nine 128-row chunks per tile
    "wide": dict(B=20480, K=100, d=128),    # 160 example tiles over 148 SMs: three segments
}


def make_sched(ntile, upt, num_sms, max_share):
    T = ntile * upt
    G = min(T, num_sms)
    if max_share > 0 and (T + G - 1) // G > max_share:
        waves = (T + num_sms * max_share - 1) // (num_sms * max_share)
        G = min(T, waves * num_sms)
    return max(G, 1), upt, ntile


def segments(sched, x):
    """TcSegIter: the (tile, u0, u1) pieces of CTA x's range [floor(x T / G), floor((x + 1) T / G))."""
    G, upt, ntile = sched
    cur, end = x * upt * ntile // G, (x + 1) * upt * ntile // G
    out = []
    while cur < end:
        tile = cur // upt
        u0 = cur - tile * upt
        n = min(upt - u0, end - cur)
        out.append((tile, u0, u0 + n))
        cur += n
    return out


def schedules(B, K, d, sp=True, num_sms=NUM_SMS):
    """The forward, recompute and dq schedules tc_init builds."""
    DP = 32 if d <= 32 else 64 if d <= 64 else 128
    rps = 128 // DP
    n_bil_rows = (d + rps - 1) // rps * rps * DP
    n_bil_half = n_bil_rows // 64
    n_sp_half = 2 * DP // 64 if sp else 0
    n_rows_total = (n_bil_rows + (2 * DP if sp else 0) + 127) // 128 * 128
    ntile = (B + 127) // 128
    return {
        "fwd": make_sched(ntile, (n_bil_half + n_sp_half + 1) // 2, num_sms, 0),
        "rec": make_sched(ntile, n_bil_half // 2, num_sms, 0),
        "dq": make_sched(ntile, n_rows_total // 128, num_sms, TC_DQ_MAX_STAGES),
    }


def test_segment_mirror_covers_every_unit_once():
    for sh in SHAPES.values():
        for sched in schedules(sh["B"], sh["K"], sh["d"]).values():
            G, upt, ntile = sched
            seen = np.zeros((ntile, upt), np.int32)
            for x in range(G):
                for tile, u0, u1 in segments(sched, x):
                    seen[tile, u0:u1] += 1
            assert (seen == 1).all()


@pytest.mark.parametrize("name,counts", [
    ("T", {1, 2}),
    ("cfg2", {1, 2}),
    ("wide", {2, 3}),
])
def test_gpu_shapes_hold_multi_segment_and_tile_end_ctas(name, counts):
    sh = SHAPES[name]
    for kernel, sched in schedules(sh["B"], sh["K"], sh["d"]).items():
        segs = [segments(sched, x) for x in range(sched[0])]
        n = collections.Counter(len(s) for s in segs)
        tile_end = sum(any(u1 == sched[1] for _, _, u1 in s) for s in segs)
        if kernel != "dq":
            assert set(n) == counts, (name, kernel, n)
        else:
            assert max(n) >= 2, (name, kernel, n)
        assert tile_end >= min(sched[0], sched[2]) - 1, (name, kernel, tile_end)


def test_wide_shape_has_three_segment_ctas_in_both_bilinear_passes():
    sh = SHAPES["wide"]
    for kernel in ("fwd", "rec"):
        sched = schedules(sh["B"], sh["K"], sh["d"])[kernel]
        assert any(len(segments(sched, x)) == 3 for x in range(sched[0])), kernel


# T and cfg2 are the full-size shapes of test_scale_fullsize.py, which checks one step of each against the oracle and
# twice for bit-identity; "wide" adds the CTAs with three segments and the tiles shared by two CTAs' ends.
WIDE_FULL = ("rescal+sp", 100, 128, 5, 20480, 1_000_000, 500_000, 30)


@pytest.mark.gpu
def test_three_segment_step_matches_oracle():
    from oracle import rae_oracle as O
    from tests.helpers import rel_err
    from tests.test_scale_fullsize import TOL_COST, TOL_Q, _gpu_first_step, check_first_step, make_full_problem, touched_rows
    model, K, d, S, B, F, N, fbar = WIDE_FULL
    data, p, neg1, neg2 = make_full_problem(model, K, d, S, B, F, N, fbar)
    out = _gpu_first_step(model, K, d, S, B, F, N, data, p, neg1, neg2)
    assert int(out["stats"]["tensor_path"]) == 1
    p64 = {k: v.astype(np.float64) for k, v in p.items()}
    ip = data.indptr[:B + 1]
    c_ref, q_ref, g = O.cost_and_grads(model, p64, ip, data.indices[:ip[-1]], data.args1[:B], data.args2[:B], neg1[:, :B],
                                       neg2[:, :B], alpha=1.0)
    del p64
    assert abs(out["cost"] - c_ref) <= TOL_COST * max(1.0, abs(c_ref)), (out["cost"], c_ref)
    assert rel_err(out["q"], q_ref) <= TOL_Q
    check_first_step(p, out["p1"], out["acc1"], g, touched_rows(data, neg1, neg2, B))


@pytest.mark.gpu
def test_three_segment_step_is_bitwise_reproducible():
    from tests.test_scale_fullsize import _gpu_first_step, make_full_problem
    model, K, d, S, B, F, N, fbar = WIDE_FULL
    data, p, neg1, neg2 = make_full_problem(model, K, d, S, B, F, N, fbar, seed=78)
    a = _gpu_first_step(model, K, d, S, B, F, N, data, p, neg1, neg2)
    b = _gpu_first_step(model, K, d, S, B, F, N, data, p, neg1, neg2)
    assert a["cost"] == b["cost"]
    for n in a["p1"]:
        assert np.array_equal(a["p1"][n], b["p1"][n]) and np.array_equal(a["acc1"][n], b["acc1"][n]), n
