"""The cost-weighted schedule of the tcgen05 contractions (TcSched, rae_internal.h; make_sched / tc_plan, rae_decoder_tc.cu).

CPU tier: librae's own schedule code, through the host-only `rae_debug_tc_schedule` export (no device needed), over a
sweep of the shapes the tensor path takes.  Every unit is owned exactly once, no CTA is empty, the CTAs that overlap a
tile are consecutive and their count is the tile's partial-slot count, no dq CTA takes more than TC_DQ_MAX_STAGES stages,
and no CTA's weighted cost exceeds its share of the virtual time by more than one unit.
GPU tier: full-size steps at odd batch sizes (a partial last example tile) and at a shape with three-segment CTAs in
every pass against the float64 oracle with the checker of test_scale_fullsize.py.  That file checks T and cfg2 and their
bit-identity across two runs, and test_tc_segments.py checks B = 20 480; all of them run on this schedule.
"""
import ctypes as C

import numpy as np
import pytest

from relation_autoencoder_b200 import _lib as L
from relation_autoencoder_b200.build import build

NUM_SMS = 148                 # B200
TC_DQ_MAX_STAGES = 64         # rae_decoder_tc.cu: stages per dq segment (accuracy bound of the MMA chain)
PASSES = ("fwd", "rec", "dq")


@pytest.fixture(scope="module")
def lib():
    build()
    lib = C.CDLL(L.LIB_PATH)
    f = lib.rae_debug_tc_schedule
    f.restype = C.c_int
    f.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
    return lib


def schedule(lib, B, K, d, sp, p, num_sms=NUM_SMS):
    """(fields dict, CTA starts [G + 1], partial slots per tile) of pass p as tc_init builds it."""
    f = np.zeros(7, np.int32)
    G = lib.rae_debug_tc_schedule(B, K, d, int(sp), num_sms, p, f.ctypes.data, None, 0, None, 0)
    assert G > 0
    starts = np.zeros(G + 1, np.int64)
    nslots = np.zeros(int(f[2]), np.int32)
    assert lib.rae_debug_tc_schedule(B, K, d, int(sp), num_sms, p, f.ctypes.data, starts.ctypes.data, G + 1,
                                      nslots.ctypes.data, len(nslots)) == G
    s = dict(zip(("G", "upt", "ntile", "ntail", "wb", "wt", "h"), (int(v) for v in f)))
    return s, starts, nslots


def cta_costs(s, starts):
    """Weighted cost of every CTA: its units' weights plus h for each segment after its first."""
    upt, ntail = s["upt"], s["ntail"]
    costs = []
    for x in range(s["G"]):
        u = np.arange(starts[x], starts[x + 1])
        i = u % upt
        w = np.where(i >= upt - ntail, s["wt"], s["wb"]).sum()
        costs.append(int(w) + s["h"] * int(np.count_nonzero((i == 0) & (u != starts[x]))))
    return np.array(costs)


@pytest.mark.parametrize("sp", [True, False])
@pytest.mark.parametrize("K", [10, 100, 104])
@pytest.mark.parametrize("d", [17, 30, 64, 128])
@pytest.mark.parametrize("B", [128, 1000, 4096, 20480])
def test_schedule_invariants(lib, B, K, d, sp):
    for p, name in enumerate(PASSES):
        s, starts, nslots = schedule(lib, B, K, d, sp, p)
        G, upt, ntile = s["G"], s["upt"], s["ntile"]
        T = upt * ntile
        assert ntile == (B + 127) // 128
        assert 1 <= G <= T and s["wb"] > 0 and s["wt"] >= s["wb"] and s["h"] >= 0
        # contiguous ranges that cover [0, T), none empty: every unit owned exactly once
        assert starts[0] == 0 and starts[-1] == T
        assert (np.diff(starts) >= 1).all(), (name, s)
        if name == "dq":
            assert np.diff(starts).max() <= TC_DQ_MAX_STAGES, (name, s)
        # the CTAs that overlap tile t are consecutive, from the owner of its first unit to the owner of its last, and
        # their count is the tile's partial-slot count (k_tc_combine, k_tc_bwd_finish, wT, dqT)
        owner = np.repeat(np.arange(G), np.diff(starts))
        for t in range(ntile):
            o = owner[t * upt:(t + 1) * upt]
            assert (np.diff(o) >= 0).all()
            assert nslots[t] == o[-1] - o[0] + 1 == len(np.unique(o)), (name, t)
        # the closed form cuts at the unit that holds x V / G: no CTA costs more than its share plus one unit
        V = ntile * (s["h"] + (upt - s["ntail"]) * s["wb"] + s["ntail"] * s["wt"])
        assert cta_costs(s, starts).max() < V / G + max(s["wb"], s["wt"]), (name, s)


def test_flagship_shape_is_balanced_within_one_tail_unit(lib):
    # T (B = 4096, K = 100, d = 128, selectional preferences): the weights are in force (not capped) and no CTA's cost is
    # more than one tail unit (one body unit for the recompute pass, which has no tail) above the mean.  The CTAs whose
    # range starts on a tile boundary save the switch the model charges there, which lowers the mean by h per such CTA
    # over all G CTAs; the bound allows for that.
    for p, name in enumerate(PASSES):
        s, starts, _ = schedule(lib, 4096, 100, 128, True, p)
        assert s["G"] == NUM_SMS and s["h"] > 0
        assert s["ntail"] == (0 if name == "rec" else 2)
        c = cta_costs(s, starts)
        on_boundary = int(np.count_nonzero(starts[1:-1] % s["upt"] == 0))
        bound = (s["wt"] if s["ntail"] else s["wb"]) + s["h"] * on_boundary / s["G"]
        assert c.max() - c.mean() <= bound, (name, s, c.max(), c.mean(), on_boundary)


@pytest.fixture(scope="module")
def make_sched(lib):
    f = lib.rae_debug_tc_make_sched
    f.restype = C.c_int
    f.argtypes = [C.c_int] * 8 + [C.c_void_p, C.c_void_p, C.c_int]

    def run(ntile, upt, max_share, num_sms=NUM_SMS, cost=(0, 0, 0, 0)):
        fields = np.zeros(7, np.int32)
        G = f(ntile, upt, num_sms, max_share, *cost, fields.ctypes.data, None, 0)
        assert G > 0
        starts = np.zeros(G + 1, np.int64)
        assert f(ntile, upt, num_sms, max_share, *cost, fields.ctypes.data, starts.ctypes.data, G + 1) == G
        return dict(zip(("G", "upt", "ntile", "ntail", "wb", "wt", "h"), (int(v) for v in fields))), starts
    return run


@pytest.mark.parametrize("max_share", [0, 16, 32, 64])
def test_default_weights_give_the_plain_split(make_sched, max_share):
    # the dC schedules take the default (uniform) weights: the split must stay floor(x T / G), with the wave count the
    # max_share bound asks for
    for ntile in (1, 2, 3, 17, 64, 65, 130):
        for upt in (1, 7, 16, 64, 65, 320):
            s, starts = make_sched(ntile, upt, max_share)
            T = ntile * upt
            G = min(T, NUM_SMS)
            if max_share > 0 and -(-T // G) > max_share:
                G = min(T, -(-T // (NUM_SMS * max_share)) * NUM_SMS)
            assert (s["G"], s["h"], s["ntail"], s["wb"], s["wt"]) == (G, 0, 0, 1, 1)
            assert (starts == np.arange(G + 1) * T // G).all(), (ntile, upt, max_share)


def test_one_unit_per_cta_caps_the_weights(lib):
    # one unit per CTA leaves no room for weights: make_sched caps them, and the split is one unit per CTA
    s, starts, _ = schedule(lib, 128, 100, 128, True, 0, num_sms=130)
    assert s["G"] == 130 and s["h"] == 0 and s["wt"] == s["wb"]
    assert (starts == np.arange(131)).all()


def max_segments(s, starts):
    upt = s["upt"]
    return max((e - 1) // upt - b // upt + 1 for b, e in zip(starts[:-1], starts[1:]))


def test_three_segment_shape_holds_three_segment_ctas(lib):
    # Under the weighted schedules B = 20 480 (test_tc_segments.py's full-size step) holds one- and two-segment CTAs only.
    # B = 24 576 at d = 64 holds CTAs whose range crosses two tile boundaries in all three passes: the GPU tier below runs
    # that shape against the oracle.
    for p, name in enumerate(PASSES):
        assert max_segments(*schedule(lib, 20480, 100, 128, True, p)[:2]) == 2, name
        assert max_segments(*schedule(lib, 24576, 100, 64, True, p)[:2]) == 3, name


# odd batch sizes (a partial last example tile), DP = 64 (the interpolated weights), and three-segment CTAs in every pass
ODD_FULL = {
    "B1000": ("rescal+sp", 100, 128, 20, 1000, 1_000_000, 500_000, 30),
    "B1000_d64": ("rescal+sp", 100, 64, 20, 1000, 1_000_000, 500_000, 30),
    "B24576_d64": ("rescal+sp", 100, 64, 5, 24576, 1_000_000, 500_000, 30),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(ODD_FULL))
def test_odd_batch_step_matches_oracle(name):
    from oracle import rae_oracle as O
    from tests.helpers import rel_err
    from tests.test_scale_fullsize import TOL_COST, TOL_Q, _gpu_first_step, check_first_step, make_full_problem, touched_rows
    model, K, d, S, B, F, N, fbar = ODD_FULL[name]
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
