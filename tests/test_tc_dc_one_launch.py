"""dC in one launch: the two-tile FP16 kernel (k_tc_dc2) takes every 128-row tile of the operand rows, the C1 / C2 tiles as
one more tile pair (the selectional-preference pair) at the end of its schedule; the one-tile TF32 kernel (k_tc_dc) is
the whole-dC fallback for B % 4 != 0.

CPU tier: librae's own dC plan, through the host-only `rae_debug_tc_dc_plan` export (no device needed), over a sweep of
the shapes the tensor path takes.  Every (row tile of [bilinear | C1 | C2], stage of 64 examples) is owned exactly once,
no segment exceeds the chain bound, the per-tile partial-slot table agrees with the schedule, and the flagship shape
needs at most 4 slots (the partial buffer is slots x (d^2 K + 2 d K) floats).
GPU tier: full-size production steps against the float64 oracle with the checker of test_scale_fullsize.py, with the
C1 / C2 gradients (the rows that moved from TF32 to FP16 pairs) checked by name; the same step twice is bit-identical;
the step issues as many launches as the one-kernel fallback does.
"""
import ctypes as C

import numpy as np
import pytest

from relation_autoencoder_b200 import _lib as L
from relation_autoencoder_b200.build import build

NUM_SMS = 148                 # B200
MAX_SMEM_OPTIN = 232448       # B200: 227 KB of shared memory per block (opt-in)
TC_DC2_MAX_STAGES = 32        # rae_decoder_tc.cu: stages per accumulator and segment of the two-tile kernel
TC_DC_MAX_STAGES = 16         # ... of the one-tile kernel, per accumulator (two accumulators)


@pytest.fixture(scope="module")
def lib():
    build()
    lib = C.CDLL(L.LIB_PATH)
    f = lib.rae_debug_tc_dc_plan
    f.restype = C.c_int
    f.argtypes = [C.c_int] * 6 + [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int]
    return lib


def dc_plan(lib, B, K, d, sp, num_sms=NUM_SMS):
    """(info dict, schedule fields, CTA starts [G + 1], partial slots per row tile) of the dC plan tc_init builds."""
    info = np.zeros(4, np.int32)
    f = np.zeros(7, np.int32)
    G = lib.rae_debug_tc_dc_plan(B, K, d, int(sp), num_sms, MAX_SMEM_OPTIN, info.ctypes.data, f.ctypes.data, None, 0, None, 0)
    assert G > 0
    starts = np.zeros(G + 1, np.int64)
    slots = np.zeros(int(info[2]), np.int32)
    assert lib.rae_debug_tc_dc_plan(B, K, d, int(sp), num_sms, MAX_SMEM_OPTIN, info.ctypes.data, f.ctypes.data,
                                    starts.ctypes.data, G + 1, slots.ctypes.data, len(slots)) == G
    inf = dict(zip(("dc2", "n_bil_tiles", "n_ntiles", "slots_dc"), (int(v) for v in info)))
    s = dict(zip(("G", "upt", "ntile", "ntail", "wb", "wt", "h"), (int(v) for v in f)))
    return inf, s, starts, slots


def expected_tiles(d, sp):
    """(bilinear 128-row tiles, all row tiles) of rae_decoder_tc.cu's operand rows [C rows (i, j) | C1 rows | C2 rows]."""
    DP = 32 if d <= 32 else 64 if d <= 64 else 128
    rps = 128 // DP
    n_bil_rows = -(-d // rps) * rps * DP
    n_rows = n_bil_rows + (2 * DP if sp else 0)
    return n_bil_rows // 128, -(-n_rows // 128)


def tiles_of_unit_tile(t, inf):
    """Row tiles schedule tile t covers: a pair of bilinear tiles, the SP pair (every C1 / C2 tile), or, in the one-tile
    kernel, tile t itself."""
    nb, nt = inf["n_bil_tiles"], inf["n_ntiles"]
    if not inf["dc2"]:
        return [t]
    n_pairs = (nb + 1) // 2
    if t < n_pairs:
        return [r for r in (2 * t, 2 * t + 1) if r < nb]
    assert t == n_pairs
    return list(range(nb, nt))


def check_plan(inf, s, starts, slots, B):
    G, upt, ntile = s["G"], s["upt"], s["ntile"]
    T = upt * ntile
    assert upt == -(-B // 64)
    assert (s["h"], s["ntail"], s["wb"], s["wt"]) == (0, 0, 1, 1)          # uniform weights
    assert starts[0] == 0 and starts[-1] == T and (np.diff(starts) >= 1).all()
    bound = TC_DC2_MAX_STAGES if inf["dc2"] else 2 * TC_DC_MAX_STAGES
    owner = np.repeat(np.arange(G), np.diff(starts))
    # every (row tile, stage) owned exactly once; no segment longer than the chain bound
    own = np.zeros((inf["n_ntiles"], upt), np.int32)
    for t in range(ntile):
        o = owner[t * upt:(t + 1) * upt]
        seg_len = np.bincount(o - o[0])
        assert seg_len.max() <= bound, (t, seg_len.max())
        for r in tiles_of_unit_tile(t, inf):
            own[r] += 1
            # the partial slots of the row tile: the CTAs that overlap its schedule tile
            assert slots[r] == o[-1] - o[0] + 1 == len(np.unique(o)), (r, t)
    assert (own == 1).all()
    assert inf["slots_dc"] == slots.max()


@pytest.mark.parametrize("sp", [True, False])
@pytest.mark.parametrize("K", [10, 100, 104])
@pytest.mark.parametrize("d", [17, 30, 64, 128])
@pytest.mark.parametrize("B", [128, 1000, 4096, 20480])
def test_dc_plan_invariants(lib, B, K, d, sp):
    inf, s, starts, slots = dc_plan(lib, B, K, d, sp)
    nb, nt = expected_tiles(d, sp)
    assert (inf["n_bil_tiles"], inf["n_ntiles"]) == (nb, nt)
    # B % 4 == 0 and the stages fit: one kernel, bilinear pairs then the SP pair
    assert inf["dc2"] == 1
    assert s["ntile"] == (nb + 1) // 2 + (1 if sp else 0)
    check_plan(inf, s, starts, slots, B)


@pytest.mark.parametrize("sp", [True, False])
@pytest.mark.parametrize("d", [30, 128])
@pytest.mark.parametrize("B", [37, 1001, 4094])
def test_batch_not_multiple_of_4_plans_the_fallback(lib, B, d, sp):
    inf, s, starts, slots = dc_plan(lib, B, 100, d, sp)
    assert inf["dc2"] == 0
    assert s["ntile"] == inf["n_ntiles"] == expected_tiles(d, sp)[1]
    check_plan(inf, s, starts, slots, B)


def test_flagship_shape_needs_few_partial_slots(lib):
    # T (B = 4096, K = 100, d = 128, selectional preferences): 64 bilinear pairs + the SP pair over one CTA per SM.  The C1 /
    # C2 tiles used to take 64 slots of their own, and the partial buffer is sized by the largest slot count.
    inf, s, _, slots = dc_plan(lib, 4096, 100, 128, True)
    assert inf["dc2"] == 1 and s["ntile"] == 65 and s["G"] == NUM_SMS
    assert inf["slots_dc"] <= 4 and slots[-2:].max() <= 4
    d, K = 128, 100
    assert inf["slots_dc"] * (d * d * K + 2 * d * K) * 4 < 28e6


def test_plan_export_rejects_shapes_off_the_tensor_path(lib):
    info, f = np.zeros(4, np.int32), np.zeros(7, np.int32)
    for B, K, d in ((0, 100, 128), (4096, 105, 128), (4096, 100, 16), (4096, 100, 129)):
        assert lib.rae_debug_tc_dc_plan(B, K, d, 1, NUM_SMS, MAX_SMEM_OPTIN, info.ctypes.data, f.ctypes.data, None, 0, None, 0) == -1


# ----------------------------------------------------------------------------------------------------------------------
# GPU tier
# ----------------------------------------------------------------------------------------------------------------------
FULL = {
    "T": ("rescal+sp", 100, 128, 20, 4096, 1_000_000, 500_000, 30),
    "cfg2": ("rescal+sp", 100, 30, 5, 4096, 1_000_000, 500_000, 30),
    "d64": ("rescal+sp", 100, 64, 20, 4096, 1_000_000, 500_000, 30),
}
TOL_GRAD = 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(FULL))
def test_one_launch_step_matches_oracle_and_repeats_bitwise(name):
    from oracle import rae_oracle as O
    from tests.helpers import rel_err
    from tests.test_scale_fullsize import TOL_COST, TOL_Q, _gpu_first_step, check_first_step, make_full_problem, touched_rows
    model, K, d, S, B, F, N, fbar = FULL[name]
    data, p, neg1, neg2 = make_full_problem(model, K, d, S, B, F, N, fbar)
    out = _gpu_first_step(model, K, d, S, B, F, N, data, p, neg1, neg2)
    again = _gpu_first_step(model, K, d, S, B, F, N, data, p, neg1, neg2)
    assert int(out["stats"]["tensor_path"]) == 1
    assert out["cost"] == again["cost"]
    for n in out["p1"]:
        assert np.array_equal(out["p1"][n], again["p1"][n]) and np.array_equal(out["acc1"][n], again["acc1"][n]), n
    p64 = {k: v.astype(np.float64) for k, v in p.items()}
    ip = data.indptr[:B + 1]
    c_ref, q_ref, g = O.cost_and_grads(model, p64, ip, data.indices[:ip[-1]], data.args1[:B], data.args2[:B], neg1[:, :B],
                                       neg2[:, :B], alpha=1.0)
    del p64
    assert abs(out["cost"] - c_ref) <= TOL_COST * max(1.0, abs(c_ref)), (out["cost"], c_ref)
    assert rel_err(out["q"], q_ref) <= TOL_Q
    # dC, dC1, dC2 by name: |g| from the accumulators of the first AdaGrad step, within 1e-5 of the tensor's ||g||_inf
    for n in ("C", "C1", "C2"):
        ref = np.abs(np.asarray(g[n], np.float64))
        e = np.abs(np.sqrt(out["acc1"][n].astype(np.float64)) - ref).max()
        assert e <= TOL_GRAD * ref.max(), (n, e / ref.max())
    check_first_step(p, out["p1"], out["acc1"], g, touched_rows(data, neg1, neg2, B))


@pytest.mark.gpu
def test_step_launches_as_many_kernels_as_the_fallback():
    # B = 4096 runs the two-tile kernel alone; B = 4092 (not a multiple of 4) runs the one-tile kernel alone.  Every other
    # launch of the step is the same, so the counts agree (with the C1 / C2 tiles in a kernel of their own they did not).
    from tests.test_scale_fullsize import _gpu_first_step, make_full_problem
    launches = []
    for B in (4096, 4092):
        model, K, d, S, F, N, fbar = "rescal+sp", 100, 128, 5, 200_000, 100_000, 30
        data, p, neg1, neg2 = make_full_problem(model, K, d, S, B, F, N, fbar)
        out = _gpu_first_step(model, K, d, S, B, F, N, data, p, neg1, neg2)
        assert int(out["stats"]["tensor_path"]) == 1
        launches.append(int(out["stats"]["kernel_launches"]))
    assert launches[0] == launches[1], launches
