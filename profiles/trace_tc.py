#!/usr/bin/env python
"""In-kernel timeline of the tcgen05 contraction kernels (needs librae_trace.so: `python -m relation_autoencoder_b200.build --trace`).

Slots per CTA (SM clock64 values, printed relative to the kernel's entry stamp):
  forward (slots 0..) and recompute (the same slots + 64)
     0 entry | 1 setup done | 12 R (c) loads issued | 13 P image in shared memory | 2 first P rows in TMEM | 6/7 MMA chunk 4 operands ready / issued | 10/11 same, chunk 12 |
     9 epilogue of the first segment done | 3 all MMAs issued | 4 epilogue done | 5 exit |
     segment 2: 58 epilogue starts it | 63 its P rows in TMEM | 59 MMA thread sees them | 60 its first chunk issued |
     61 its R (c) rows loaded | values: 57 segment count, 62 the CTA ends a tile
  dq   16 entry | 17 setup | 22/23 MMA stage 8 ready / issued | 27/28 same, stage 24 | 24/25/26 generator warp 0 stage 8:
        computed / slot acquired / published | 19 all MMAs issued | 20 generators + drain done | 21 exit |
        102 drain of the first segment starts | 100 / 101 first selectional-preference stage starts / last one published |
        segment 2: 97 X/Y loads start | 98 X/Y loaded | 99 MMA thread sees the drained accumulator | 104 its first stage
        published | values: 96 segment count, 103 the CTA ends a tile
  dC   32 entry | 33 staging + setup | 38/39 MMA stage 8 ready / issued | 43/44 same, stage 24 | 40/41/42 generator warp 0
        stage 8 | 35 all MMAs issued | 36 generators + drain done | 37 exit |
        values: 80 segment count, 81 the CTA's range holds stages of the selectional-preference pair (the last tile pair)
"""
import ctypes as C, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from relation_autoencoder_b200 import _lib as L
L.LIB_PATH = os.path.join(ROOT, "librae_trace.so")
from relation_autoencoder_b200 import synthetic as SY
from relation_autoencoder_b200.engine import Engine
import bench

wlname = sys.argv[1] if len(sys.argv) > 1 else "T"
wl = dict(SY.WORKLOADS[wlname]); B = wl["B"]
data, params, neg1, neg2 = bench._make_inputs(wl, 8 * B)
eng = Engine(wl["model"], wl["K"], wl["d"], wl["S"], B, wl["F"], wl["N"], wl["N_train"])
eng.set_params_numpy(params); eng.bind_split("train", data.indptr, data.indices, data.args1, data.args2)
eng.bind_epoch_negatives(neg1, neg2)
for b in range(4): eng.train_device(b, want_cost=False)
torch.cuda.synchronize()
NCTA, STRIDE = 320, 128
buf = torch.zeros(NCTA * STRIDE, dtype=torch.int64, device="cuda")
lib = C.CDLL(L.LIB_PATH)
lib.rae_debug_set_trace.argtypes = [C.c_void_p]
assert lib.rae_debug_set_trace(C.c_void_p(buf.data_ptr())) == 0
# knock-out runs (measurement build only; results are garbage, timing is the point): per-kernel wall time and median CTA cycles
if os.environ.get("TRACE_KNOCK"):
    print("knock-out runs: 1 = no operand copies after the first fills, 2 = no MMAs, 4 = no epilogue / generator arithmetic")
    for bits in (0, 1, 2, 4, 3, 6, 7):
        lib.rae_debug_set_knock(bits)
        buf.zero_()
        eng.train_device(4, want_cost=False)
        torch.cuda.synchronize()
        tk = buf.cpu().numpy().reshape(NCTA, STRIDE)
        row = []
        for kname, base in (("fwd", 0), ("rec", 64), ("dq", 16), ("dC", 32)):
            live = [c for c in range(NCTA) if tk[c, base] != 0]
            if live:
                wall = (max(tk[c, base + 15] for c in live) - min(tk[c, base + 14] for c in live)) / 1e3
                med = int(np.median([tk[c, base + 5] - tk[c, base] for c in live]))
                row.append("%s %.1f us / %d cyc" % (kname, wall, med))
        print("  knock %d: %s" % (bits, "; ".join(row)))
    lib.rae_debug_set_knock(0)
    buf.zero_()
    # the knocked-out steps leave garbage in the parameters: timing only from here on
eng.train_device(4, want_cost=False)
torch.cuda.synchronize()
t = buf.cpu().numpy().reshape(NCTA, STRIDE)
FWD = {0: "entry", 1: "setup done", 12: "R loads issued", 13: "P image in smem", 8: "R loads done", 2: "first P in TMEM", 6: "mma c4 ready", 7: "mma c4 issued", 10: "mma c12 ready",
                    11: "mma c12 issued", 51: "mma c8 start", 48: "mma c8 mid: wait next t_empty", 49: "mma c8 mid: t_empty ok",
                    50: "mma c8 mid: b_full ok", 52: "mma c9 start", 53: "epi c8 wait t_full", 54: "epi c8 t_full ok",
                    55: "epi c8 arrived t_empty", 56: "epi c8 done", 9: "first segment epilogue done", 3: "all MMAs issued", 4: "epilogue done", 5: "exit",
       58: "seg 2: epilogue starts", 63: "seg 2: P in TMEM", 59: "seg 2: MMA sees P", 60: "seg 2: first chunk issued",
       61: "seg 2: R loaded"}
KERNELS = {
    "fwd": (0, FWD, 57, 62),
    "rec": (64, {k + 64: v for k, v in FWD.items()}, 121, 126),
    "dq": (16, {16: "entry", 17: "setup done", 29: "X/Y loads done", 18: "stage 0 published", 22: "mma s8 ready", 23: "mma s8 issued", 27: "mma s24 ready", 28: "mma s24 issued",
                24: "gen s8 computed", 25: "gen s8 slot acquired", 26: "gen s8 published", 19: "all MMAs issued", 20: "gen+drain done", 21: "exit",
                102: "first segment drain starts", 100: "SP stages start", 101: "SP stages published", 97: "seg 2: X/Y loads start",
                98: "seg 2: X/Y loaded", 99: "seg 2: MMA sees drained acc", 104: "seg 2: first stage published"}, 96, 103),
    "dC": (32, {32: "entry", 33: "staging+setup done", 38: "mma s8 ready", 39: "mma s8 issued", 43: "mma s24 ready", 44: "mma s24 issued",
                40: "gen s8 wait slot", 41: "gen s8 slot acquired", 42: "gen s8 published", 35: "all MMAs issued", 36: "gen+drain done", 37: "exit"}, 80, 81),
}
# what the second per-CTA value says (CTAs are grouped by segment count and by it)
FLAG = {"dC": ("holds SP-pair stages", "bilinear pairs only")}
for kname, (base, names, s_nseg, s_end) in KERNELS.items():
    live = [c for c in range(NCTA) if t[c, base] != 0]
    if not live:
        continue
    t0 = min(t[c, base] for c in live)
    ex = base + 5
    life = {c: int(t[c, ex] - t[c, base]) for c in live}
    dur = list(life.values())
    print("== %s: %d CTAs, per-CTA cycles entry->exit min/median/max = %d / %d / %d (max / median %.3f)"
          % (kname, len(live), min(dur), int(np.median(dur)), max(dur), max(dur) / np.median(dur)))
    ns0, ns1 = base + 14, base + 15
    k_ns = max(t[c, ns1] for c in live) - min(t[c, ns0] for c in live)
    mhz = [1e3 * (t[c, ex] - t[c, base]) / max(1, t[c, ns1] - t[c, ns0]) for c in live]
    print("   kernel wall time (globaltimer, first entry -> last exit) = %.1f us; SM clock held per CTA min/median/max = %.0f / %.0f / %.0f MHz"
          % (k_ns / 1e3, min(mhz), float(np.median(mhz)), max(mhz)))
    if s_nseg is not None:
        # CTA life by segment count and by whether the CTA's range ends a tile
        groups = {}
        for c in live:
            groups.setdefault((int(t[c, s_nseg]), int(t[c, s_end])), []).append(c)
        for (n, e), cs in sorted(groups.items()):
            d = [life[c] for c in cs]
            yes, no = FLAG.get(kname, ("ends a tile", "no tile end"))
            print("   %d segment(s), %s: %3d CTAs, life min/median/max = %d / %d / %d"
                  % (n, yes if e else no, len(cs), min(d), int(np.median(d)), max(d)))
    slowest = max(live, key=lambda c: life[c])
    median_cta = sorted(live, key=lambda c: life[c])[len(live) // 2]
    for tag, cta in (("first", live[0]), ("median life", median_cta), ("slowest", slowest)):
        r = t[cta]
        extra = "" if s_nseg is None else ", %d segment(s)%s" % (r[s_nseg], ", " + FLAG.get(kname, ("ends a tile",))[0] if r[s_end] else "")
        print("  CTA %d, %s (entry at +%d%s)" % (cta, tag, r[base] - t0, extra))
        for slot in sorted(names, key=lambda s: r[s]):
            if r[slot]:
                print("    %8d  %s" % (r[slot] - r[base], names[slot]))
eng.close()
