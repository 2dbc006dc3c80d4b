"""Data-parallel training step over the GPUs of one node (SURVEY 8e).  The reference is single-process and has no
counterpart; the partitioning follows from its objective: examples are independent given the parameters and the cost is
a sum over examples divided by the global Z (learning/OieModel.py:90).

* batch: every rank owns B examples of each global batch of world*B; Z and adj are global.
* dense parameters C/R, C1, C2, Wb: replicated; every rank applies the identical optimiser step (Optimizers.py:29-32) to
  the SUM of the ranks' dense gradients, which the dense-update kernel reads from the peers' flat gradient buffers in
  rank order (above 16 MB of remote reads per rank one NCCL all-reduce of the flat buffer is used instead).
* sparse tables W[F,K], A[N,d], Ab[N] (+ AdaGrad accumulators): row-sharded, owner(row) = row mod world, local index =
  row // world, in CUDA-IPC memory every rank of the node maps.  The steady-state step issues NO collective:
    (1) fetch   - a rank's kernel reads the distinct rows its batch touches straight from their owners' HBM over
                  NVLink into compact tables (``rae_fetch_rows``); ids are remapped to compact slots (ascending id);
    (2) step    - the fused step runs on the compact tables with RAE_FLAG_EMIT_ONLY: one reduced gradient row per compact
                  row (duplicates inside the rank already summed, in sorted order);
    (3) barrier - flag words in peer memory (``rae_peer_barrier``, bounded spin) order "every rank has emitted"; the
                  ranks' costs are summed over peer memory behind it and handed to ``train()`` before the pulls finish;
    (4) pull    - each OWNER reads the gradient rows of its rows from all ranks' compact gradient buffers, sums them in
                  rank order and applies ONE optimiser read-modify-write per row (``rae_pull_apply``);
    (5) barrier - "every owner has applied", before the next step's fetch.
* regulariser (l1 / l2 != 0, OieModel.py:54-62, OieInduction.py:131-135): it reaches every element of W (and of C | C1 | C2
  when ext_reg), touched or not.  The local step emits data gradients only.  Before (3) each rank adds
  adj*(l1*L1 + l2*L2) of its own pre-update W shard to its local cost, rank 0 also that of the decoder tensors, so the
  rank-order sum of the local costs is the global batch's cost.  The dense update adds the decoder tensors' term to the
  summed gradient.  In (4) the owner applies W over its WHOLE shard (``rae_shard_apply``): per element the summed
  contributions (0 for a row no rank touched), then adj*(l1*sgn + 2*l2*w), then the rule - the order of the single-GPU
  dense update.
* labelling (``label_rows``): any rows of a split are labelled straight from the owners' W shards with one
  ``rae_label_shards`` call (no collective), in the single-GPU summation order; it is issued on the caller's stream behind
  the step's "every owner has applied" barrier, and the next step's applies wait behind its first barrier.
  Fixed orders everywhere: bitwise reproducible for a given world size.  (Backends without peer memory - the NumPy
  backend of the CPU tests - order (3) and (5) with the dense all-reduce and a one-element cost all-reduce.)
* routing (which rows, which slots, who owns what) depends only on the ids: the plans of ALL batches are built at bind
  time (features) / once per epoch (entities) with a handful of vectorised tensor ops and two all-gathers, so the step
  itself needs no host synchronisation and no id exchange.

torch.distributed is the plumbing (NCCL on GPUs, gloo in the CPU tests); the numerical work is done by a backend:
:class:`CudaBackend` (librae.so) in production.  The CPU tests inject a NumPy backend to check the routing logic.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional

import numpy as np
import torch
import torch.distributed as dist

SPARSE = ("W", "A", "Ab")


def shard_rows(full: np.ndarray, rank: int, world: int) -> np.ndarray:
    return np.ascontiguousarray(full[rank::world])


# ----------------------------------------------------------------------------------------------------------------------
# routing plans
# ----------------------------------------------------------------------------------------------------------------------
@dataclass
class EpochPlan:
    """Routing of one table family (features -> W, entities -> A/Ab) for every batch of a split / epoch."""
    nb: int
    u_ids: torch.Tensor        # int32 [sum U_b]  distinct global row ids of each batch, ascending within the batch
    u_off: List[int]           # [nb+1] offsets into u_ids
    compact: torch.Tensor      # int32 [n_occ]    compact slot (position in the batch's u_ids) of every occurrence
    rows_local: torch.Tensor   # int32 [sum R_b]  owner side: local row index of every row this rank owns and any rank touches
    r_off: List[int]           # [nb+1] offsets into rows_local (and into ent_off)
    ent_off: torch.Tensor      # int32 [sum R_b + 1] absolute offsets into ent_src / ent_slot
    ent_src: torch.Tensor      # int32 [E] source rank of each contribution (ascending within a row)
    ent_slot: torch.Tensor     # int32 [E] compact slot of the row in the source rank's gradient buffer
    max_u: int

    def ids_of(self, b):
        return self.u_ids[self.u_off[b]:self.u_off[b + 1]]


def _excl_cumsum(cnt: torch.Tensor) -> torch.Tensor:
    off = torch.zeros(cnt.numel() + 1, dtype=torch.int64, device=cnt.device)
    off[1:] = torch.cumsum(cnt, 0)
    return off


def _owned_entries(keys: List[torch.Tensor], nb: int, stride: int, rank: int, world: int):
    """Owner-side view of every rank's distinct (batch, row) keys: for the rows this rank owns, (batch, local row, source rank,
    compact slot of the row in that source's batch list).  One vectorised pass over the concatenated keys (no per-source
    loop, no host synchronisation): a key's slot is its position inside its source's list minus the number of that
    source's keys in earlier batches."""
    dev = keys[0].device
    sizes = torch.tensor([k.numel() for k in keys], dtype=torch.int64, device=dev)
    allk = torch.cat(keys)
    src = torch.repeat_interleave(torch.arange(world, dtype=torch.int64, device=dev), sizes)
    b = torch.div(allk, stride, rounding_mode="floor")
    idd = allk - b * stride
    start_of_src = _excl_cumsum(sizes)[:-1]
    pos = torch.arange(allk.numel(), dtype=torch.int64, device=dev) - start_of_src[src]
    cnt = torch.bincount(src * nb + b, minlength=world * nb).reshape(world, nb)
    off = torch.cumsum(cnt, 1) - cnt                       # [world, nb] keys of the source in earlier batches
    slot = pos - off.reshape(-1)[src * nb + b]
    own = (idd % world) == rank
    return b[own], torch.div(idd[own], world, rounding_mode="floor"), src[own], slot[own]


def build_epoch_plan(ids: torch.Tensor, batch_of: torch.Tensor, nb: int, n_rows_total: int, rank: int, world: int,
                     group=None) -> EpochPlan:
    """Collective.  ``ids`` int64 [n]: global row id of every occurrence this rank has in the epoch; ``batch_of`` int64 [n]:
    the batch each occurrence belongs to."""
    dev = ids.device
    stride = int(n_rows_total)
    n_local = (stride + world - 1) // world
    key = batch_of * stride + ids
    ukey, inverse = torch.unique(key, sorted=True, return_inverse=True)
    ub = torch.div(ukey, stride, rounding_mode="floor")
    u_off_t = _excl_cumsum(torch.bincount(ub, minlength=nb))
    compact = (inverse - u_off_t[batch_of]).to(torch.int32)
    u_ids = (ukey - ub * stride).to(torch.int32)
    # every rank learns every rank's distinct (batch, row) keys
    if world > 1:
        n_mine = torch.tensor([ukey.numel()], dtype=torch.int64, device=dev)
        sizes = [torch.zeros_like(n_mine) for _ in range(world)]
        dist.all_gather(sizes, n_mine, group=group)
        sizes = [int(s.item()) for s in sizes]
        mx = max(max(sizes), 1)
        padded = torch.zeros(mx, dtype=torch.int64, device=dev)
        padded[: ukey.numel()] = ukey
        gathered = [torch.empty_like(padded) for _ in range(world)]
        dist.all_gather(gathered, padded, group=group)
        keys = [gathered[s][: sizes[s]] for s in range(world)]
    else:
        keys = [ukey]
    eb, erow, esrc, eslot = _owned_entries(keys, nb, stride, rank, world)
    key2 = (eb * n_local + erow) * world + esrc            # distinct by construction: any sort gives the same order
    order = torch.argsort(key2)
    rowkey = torch.div(key2[order], world, rounding_mode="floor")
    uniq, counts = torch.unique_consecutive(rowkey, return_counts=True)
    rb = torch.div(uniq, n_local, rounding_mode="floor")
    rows_local = (uniq - rb * n_local).to(torch.int32)
    r_off_t = _excl_cumsum(torch.bincount(rb, minlength=nb))
    ent_off = _excl_cumsum(counts).to(torch.int32)
    return EpochPlan(nb=nb, u_ids=u_ids.contiguous(), u_off=u_off_t.tolist(), compact=compact.contiguous(),
                     rows_local=rows_local.contiguous(), r_off=r_off_t.tolist(), ent_off=ent_off.contiguous(),
                     ent_src=esrc[order].to(torch.int32).contiguous(), ent_slot=eslot[order].to(torch.int32).contiguous(),
                     max_u=int((u_off_t[1:] - u_off_t[:-1]).max().item()) if nb > 0 else 0)


# ----------------------------------------------------------------------------------------------------------------------
# CUDA backend: librae.so + CUDA-IPC peer memory
# ----------------------------------------------------------------------------------------------------------------------
class _DevArray:
    """Raw device allocation exposed to torch through ``__cuda_array_interface__`` (zero copy)."""

    def __init__(self, ptr: int, shape, typestr="<f4"):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (ptr, False), "version": 3,
                                         "strides": None}


class PeerBuffer:
    """fp32 device buffer allocated by librae (cudaMalloc, zeroed) whose IPC handle the other ranks can open."""

    def __init__(self, lib, shape, device):
        self.lib = lib
        self.shape = tuple(int(x) for x in shape)
        n = int(np.prod(self.shape)) if len(self.shape) else 1
        self.nbytes = max(4 * n, 4)
        ptr = C.c_void_p(0)
        self.handle = (C.c_ubyte * 64)()
        rc = lib.rae_peer_alloc(self.nbytes, C.byref(ptr), self.handle)
        if rc != 0:
            raise RuntimeError("rae_peer_alloc failed (%d): %s" % (rc, lib.rae_last_error(None).decode()))
        self.ptr = int(ptr.value)
        self.tensor = torch.as_tensor(_DevArray(self.ptr, self.shape if n > 0 else (0,)), device=device)
        self.peers: List[int] = [self.ptr]       # device pointers of this buffer on every rank (own rank included)
        self._opened: List[int] = []

    def handle_bytes(self) -> bytes:
        return bytes(self.handle)

    def open_peers(self, handles: List[bytes], rank: int):
        self.peers = []
        for r, hb in enumerate(handles):
            if r == rank:
                self.peers.append(self.ptr)
                continue
            buf = (C.c_ubyte * 64).from_buffer_copy(hb)
            p = C.c_void_p(0)
            rc = self.lib.rae_peer_open(buf, C.byref(p))
            if rc != 0:
                raise RuntimeError("rae_peer_open failed (%d): %s" % (rc, self.lib.rae_last_error(None).decode()))
            self.peers.append(int(p.value))
            self._opened.append(int(p.value))

    def peer_array(self):
        return (C.c_void_p * len(self.peers))(*self.peers)

    def close(self):
        for p in self._opened:
            self.lib.rae_peer_close(C.c_void_p(p))
        self._opened = []
        if self.ptr:
            self.tensor = None
            self.lib.rae_peer_free(C.c_void_p(self.ptr))
            self.ptr = 0


class GranularStep:
    """``run_begin`` / ``run_end`` of a step spelled out call by call (the order is the contract; CudaBackend issues the same
    sequence inside librae with one C call each)."""

    def run_begin(self, de, b, a1c, a2c, n1c, n2c, neg_ld):
        e_ids = de.eplan.ids_of(b)
        self.fetch("W", de.fplan.ids_of(b))
        self.fetch("A", e_ids)
        self.fetch("Ab", e_ids)
        self.local_step(b, a1c, a2c, n1c, n2c, neg_ld)

    def run_end(self, de, b):
        # a regularised step (backends implement add_local_regulariser / shard_apply): the regulariser's value is taken
        # from the parameters before any apply of this step, and W moves over the whole shard, touched rows or not
        reg = de.l1 != 0.0 or de.l2 != 0.0
        if reg:
            self.add_local_regulariser()
        self.dense_apply()
        for name, plan in (("W", de.fplan), ("A", de.eplan), ("Ab", de.eplan)):
            lo, hi = plan.r_off[b], plan.r_off[b + 1]
            apply = self.shard_apply if (reg and name == "W") else self.pull_apply
            apply(name, de.shard[name], de.shard_acc[name], plan.rows_local[lo:hi], plan.ent_off[lo:hi + 1], plan.ent_src,
                  plan.ent_slot)
        return self.local_cost_tensor()

    def plans_changed(self, de):
        pass

    def label_rows(self, de, indptr, indices, lo, hi, probs=True):
        """Rows [lo, hi) of a split (int32 CSR, global feature ids) labelled on the compact table: per chunk, fetch the
        chunk's distinct W rows, then label on their compact slots (backends implement fetch / label).  A chunk is at most
        B rows whose distinct features fit the compact table, so no split is too wide for it.  A backend without peer
        memory fetches collectively, so every rank issues as many fetches as the rank with the most chunks."""
        cap = self.compact["W"].shape[0]
        ip = indptr.to(torch.int64)
        chunks = []
        r = lo
        while r < hi:
            e = min(r + de.B, hi)
            while True:
                u, inv = torch.unique(indices[ip[r]:ip[e]], sorted=True, return_inverse=True)
                if u.numel() <= cap:
                    break
                if e == r + 1:
                    raise RuntimeError("label: row %d has %d distinct features, more than the %d rows of the compact table"
                                       % (r, u.numel(), cap))
                e = r + (e - r) // 2
            chunks.append((r, e, u, inv))
            r = e
        n_fetch = len(chunks)
        if de.world > 1:
            t = torch.tensor([n_fetch], dtype=torch.int64, device=de.dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=de.group)
            n_fetch = int(t.item())
        labels, q = [], []
        for i in range(n_fetch):
            if i >= len(chunks):
                self.fetch("W", torch.zeros(0, dtype=torch.int32, device=de.dev))
                continue
            r, e, u, inv = chunks[i]
            self.fetch("W", u.to(torch.int32).contiguous())
            lab, pr = self.label((ip[r:e + 1] - ip[r]).to(torch.int32).contiguous(), inv.to(torch.int32).contiguous())
            labels.append(torch.as_tensor(lab).to(de.dev, torch.int64))
            q.append(torch.as_tensor(pr).to(de.dev))
        if not chunks:
            return torch.zeros(0, dtype=torch.int64, device=de.dev), (torch.zeros((0, de.K), device=de.dev) if probs else None)
        return torch.cat(labels), (torch.cat(q) if probs else None)


class CudaBackend(GranularStep):
    """Local numerical work on one GPU through librae.so (emit-only engine on compact tables) and the peer-memory
    fetch / pull kernels."""

    def __init__(self, de: "DistributedEngine"):
        from . import _lib as L
        self.L = L
        self.lib = L.load()
        self.de = de
        self.device = de.dev
        torch.cuda.set_device(self.device)
        self.eng = None
        self.shard_buf: Dict[str, PeerBuffer] = {}
        self.grad_buf: Dict[str, PeerBuffer] = {}
        self.compact: Dict[str, torch.Tensor] = {}
        self.dense_grad = None
        self.cost_t = torch.zeros(1, dtype=torch.float64, device=self.device)

    @staticmethod
    def _p(t):
        return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)

    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _exchange(self, bufs: Dict[str, PeerBuffer]):
        de = self.de
        if de.world == 1:
            return
        mine = {n: b.handle_bytes() for n, b in bufs.items()}
        allh = [None] * de.world
        dist.all_gather_object(allh, mine, group=de.group)
        for n, b in bufs.items():
            b.open_peers([allh[r][n] for r in range(de.world)], de.rank)

    # -- tables
    def alloc_tables(self, shapes: Dict[str, tuple]) -> Dict[str, torch.Tensor]:
        """Collective: the row shards of W / A / Ab in peer-visible memory."""
        for b in self.shard_buf.values():
            b.close()
        self.shard_buf = {n: PeerBuffer(self.lib, shp, self.device) for n, shp in shapes.items()}
        self._exchange(self.shard_buf)
        return {n: b.tensor for n, b in self.shard_buf.items()}

    def setup(self, f_cap: int, n_cap: int):
        """Collective: emit-only engine on compact tables of capacity f_cap / n_cap, peer-visible gradient buffers."""
        from .engine import Engine
        de = self.de
        L = self.L
        self.eng = Engine(de.model, de.K, de.d, de.S, de.B, f_cap, n_cap, de.n_train, lr=de.lr, alpha=de.alpha,
                          optimizer=de.optimizer, device=self.device.index, flags=L.RAE_FLAG_EMIT_ONLY, z_total=de.z_total,
                          adj=de.adj, l1=de.l1, l2=de.l2, ext_reg=de.ext_reg)
        self.h = self.eng._h
        f32 = dict(dtype=torch.float32, device=self.device)
        self.compact = {"W": torch.zeros(f_cap, de.K, **f32), "A": torch.zeros(n_cap, de.d, **f32), "Ab": torch.zeros(n_cap, **f32)}
        # gradient PUSH: every rank owns RECEIVE buffers with one region per source rank, [world][cap][width]; the emit-only
        # row-update kernels of rank s store the reduced gradient row of compact slot j into region [s][j] of the row's
        # owner (posted stores over NVLink beside the dense contraction), and the owner applies from local memory
        self.f_cap, self.n_cap = int(f_cap), int(n_cap)
        W_ = de.world
        self.grad_buf = {"W": PeerBuffer(self.lib, (W_ * f_cap, de.K), self.device), "A": PeerBuffer(self.lib, (W_ * n_cap, de.d), self.device),
                         "Ab": PeerBuffer(self.lib, (W_ * n_cap,), self.device)}
        # the flat dense gradient and the barrier flags are peer-visible too: with them the step needs NO collective
        n_dense = int(self.lib.rae_dense_grad_size(self.h))
        self.grad_buf["dense"] = PeerBuffer(self.lib, (n_dense,), self.device)
        self.grad_buf["flags"] = PeerBuffer(self.lib, (L.RAE_FLAG_WORDS,), self.device)   # barrier epochs + local cost, zeroed
        self._exchange(self.grad_buf)
        self.dense_grad = self.grad_buf["dense"].tensor
        self.peer_sync = True
        gb = self.grad_buf
        self.eng._check(self.lib.rae_bind_push_targets(self.h, gb["W"].peer_array(), gb["A"].peer_array(), gb["Ab"].peer_array(),
                                                       de.world, de.rank, self.f_cap, self.n_cap), "rae_bind_push_targets")
        # the owner-side apply reads the `world` regions of the OWN receive buffers
        def regions(buf, cap, width):
            base = buf.tensor.data_ptr()
            return (C.c_void_p * de.world)(*[base + 4 * r * cap * width for r in range(de.world)])
        self._recv_regions = {"W": regions(gb["W"], self.f_cap, de.K), "A": regions(gb["A"], self.n_cap, de.d),
                              "Ab": regions(gb["Ab"], self.n_cap, 1)}
        # small dense gradients are summed straight from the peers' buffers inside the dense update; large ones (d = 128:
        # 6.6 MB) go through NCCL's all-reduce, which moves 2(n-1)/n of the bytes instead of (n-1)
        self.peer_dense = (de.world - 1) * n_dense * 4 <= de.peer_dense_max_bytes

    def bind_dense(self, dense: Dict[str, torch.Tensor], dense_acc: Dict[str, torch.Tensor]):
        g = lambda m, n: self._p(m.get(n))
        e = self.eng
        e._check(self.lib.rae_bind_params(self.h, self._p(self.compact["W"]), g(dense, "Wb"), self._p(self.compact["A"]),
                                          self._p(self.compact["Ab"]), g(dense, "C"), g(dense, "C1"), g(dense, "C2")), "rae_bind_params")
        e._check(self.lib.rae_bind_accumulators(self.h, None, g(dense_acc, "Wb"), None, None, g(dense_acc, "C"),
                                                g(dense_acc, "C1"), g(dense_acc, "C2")), "rae_bind_accumulators")
        gb = self.grad_buf
        e._check(self.lib.rae_bind_grad_buffers(self.h, self._p(gb["W"].tensor), self._p(gb["A"].tensor), self._p(gb["Ab"].tensor),
                                                self._p(self.dense_grad)), "rae_bind_grad_buffers")

    def bind_train_csr(self, indptr: torch.Tensor, indices_compact: torch.Tensor, a1: torch.Tensor, a2: torch.Tensor):
        """The local train rows with COMPACT feature slots as column ids: the engine caches the per-batch transposed index."""
        self.eng.bind_split("train", indptr, indices_compact, a1, a2)

    # -- the step
    def fetch(self, name: str, ids: torch.Tensor):
        t = self.compact[name]
        width = 1 if t.dim() == 1 else t.shape[1]
        self.eng._check(self.lib.rae_fetch_rows(self.h, self.shard_buf[name].peer_array(), self.de.world, width, self._p(ids),
                                                ids.numel(), self._p(t), self._stream), "rae_fetch_rows")

    def local_step(self, batch_index, a1c, a2c, n1c, n2c, neg_ld):
        self.eng._check(self.lib.rae_train_step_begin(self.h, int(batch_index), self._p(a1c), self._p(a2c), self._p(n1c),
                                                      self._p(n2c), int(neg_ld), self._stream), "rae_train_step_begin")

    def dense_apply(self):
        self.eng._check(self.lib.rae_train_step_end(self.h, self._stream), "rae_train_step_end")

    def pull_apply(self, name: str, table, acc, rows_local, ent_off, ent_src, ent_slot):
        if name == "W" and (self.de.l1 != 0.0 or self.de.l2 != 0.0):
            return self.shard_apply(name, table, acc, rows_local, ent_off, ent_src, ent_slot)   # every row moves
        width = 1 if table.dim() == 1 else table.shape[1]
        n_rows = rows_local.numel()
        if n_rows == 0:
            return
        self.eng._check(self.lib.rae_pull_apply(self.h, self._p(table), self._p(acc), width, self._p(rows_local), self._p(ent_off),
                                                self._p(ent_src), self._p(ent_slot), n_rows, self._recv_regions[name],
                                                self.de.world, self._stream), "rae_pull_apply")

    def shard_apply(self, name: str, table, acc, rows_local, ent_off, ent_src, ent_slot):
        """The regularised owner-side pass over every row of the shard ``table`` (``rae_shard_apply``)."""
        width = 1 if table.dim() == 1 else table.shape[1]
        self.eng._check(self.lib.rae_shard_apply(self.h, self._p(table), self._p(acc), width, self._p(rows_local), self._p(ent_off),
                                                 self._p(ent_src), self._p(ent_slot), rows_local.numel(), self._recv_regions[name],
                                                 self.de.world, table.shape[0], self._stream), "rae_shard_apply")

    def local_cost_tensor(self) -> torch.Tensor:
        self.eng._check(self.lib.rae_copy_cost(self.h, self._p(self.cost_t), self._stream), "rae_copy_cost")
        return self.cost_t

    # -- fused step: one descriptor per batch, built when the plans change, two C calls per step
    def plans_changed(self, de):
        L = self.L
        fp, ep = de.fplan, de.eplan
        self.descs = []
        if fp is None or ep is None:
            return
        self._peer_arrays = {k: b.peer_array() for k, b in list(self.shard_buf.items())}
        self._grad_arrays = {k: b.peer_array() for k, b in list(self.grad_buf.items())}
        vp = lambda arr: C.cast(arr, C.c_void_p)
        el = lambda t, off: C.c_void_p(t.data_ptr() + 4 * int(off))
        B, n_used = de.B, de.nb * de.B
        for b in range(de.nb):
            d = L.RaeDistStep()
            d.world = de.world
            d.w_shards, d.a_shards, d.ab_shards = vp(self._peer_arrays["W"]), vp(self._peer_arrays["A"]), vp(self._peer_arrays["Ab"])
            d.gw_bufs, d.ga_bufs, d.gab_bufs = (vp(self._recv_regions[k]) for k in ("W", "A", "Ab"))
            d.Wc, d.Ac, d.Abc = (self.compact[k].data_ptr() for k in ("W", "A", "Ab"))
            d.f_ids, d.n_f = el(fp.u_ids, fp.u_off[b]), fp.u_off[b + 1] - fp.u_off[b]
            d.e_ids, d.n_e = el(ep.u_ids, ep.u_off[b]), ep.u_off[b + 1] - ep.u_off[b]
            d.batch_index = b
            d.a1c, d.a2c = el(de.a1c, b * B), el(de.a2c, b * B)
            d.n1c, d.n2c, d.neg_ld = el(de.n1c, b * B), el(de.n2c, b * B), n_used
            d.W, d.accW = de.shard["W"].data_ptr(), de.shard_acc["W"].data_ptr()
            d.A, d.accA = de.shard["A"].data_ptr(), de.shard_acc["A"].data_ptr()
            d.Ab, d.accAb = de.shard["Ab"].data_ptr(), de.shard_acc["Ab"].data_ptr()
            d.fr_rows, d.fr_off, d.n_fr = el(fp.rows_local, fp.r_off[b]), el(fp.ent_off, fp.r_off[b]), fp.r_off[b + 1] - fp.r_off[b]
            d.f_src, d.f_slot = fp.ent_src.data_ptr(), fp.ent_slot.data_ptr()
            d.er_rows, d.er_off, d.n_er = el(ep.rows_local, ep.r_off[b]), el(ep.ent_off, ep.r_off[b]), ep.r_off[b + 1] - ep.r_off[b]
            d.e_src, d.e_slot = ep.ent_src.data_ptr(), ep.ent_slot.data_ptr()
            d.cost_dev = self.cost_t.data_ptr()
            d.flag_bufs = vp(self._grad_arrays["flags"])
            d.dense_bufs = vp(self._grad_arrays["dense"]) if self.peer_dense else None
            d.rank = de.rank
            d.global_cost = 1                     # the ranks' costs are summed over peer memory too: no collective in the step
            d.w_rows = de.shard["W"].shape[0]     # the handle's F is the compact capacity: the shard's rows come from here
            self.descs.append(d)

    def run_begin(self, de, b, a1c, a2c, n1c, n2c, neg_ld):
        d = self.descs[b]
        if n1c is not None:                       # explicit compact negatives (train() with host ids): patched copy
            d2 = self.L.RaeDistStep()
            C.memmove(C.byref(d2), C.byref(d), C.sizeof(d))
            d2.n1c, d2.n2c, d2.neg_ld = n1c.data_ptr(), n2c.data_ptr(), int(neg_ld)
            self._keep_step = (d2, n1c, n2c)
            d = d2
        self.eng._check(self.lib.rae_dist_step_begin(self.h, C.byref(d), self._stream), "rae_dist_step_begin")

    def run_begin_host(self, de, b, neg1, neg2):
        """func['train'] form: this rank's host negatives are copied and checked against the plan inside the C call."""
        n1, p1, ld1 = self.eng._host_negatives(neg1)
        n2, p2, ld2 = self.eng._host_negatives(neg2)
        self.eng._check(self.lib.rae_dist_step_begin_host(self.h, C.byref(self.descs[b]), p1, ld1, p2, ld2, self._stream),
                        "rae_dist_step_begin_host")

    def dense_allreduce_aside(self, group):
        cur = torch.cuda.current_stream(self.device)
        if getattr(self, "_ar_stream", None) is None:
            self._ar_stream = torch.cuda.Stream(device=self.device)
            self._ar_event = torch.cuda.Event()
        self._ar_stream.wait_stream(cur)
        with torch.cuda.stream(self._ar_stream):
            dist.all_reduce(self.dense_grad, group=group)
            self._ar_event.record(self._ar_stream)
        self.eng._check(self.lib.rae_dist_set_dense_wait(self.h, C.c_void_p(self._ar_event.cuda_event)), "rae_dist_set_dense_wait")

    def run_end(self, de, b):
        self.eng._check(self.lib.rae_dist_step_end(self.h, C.byref(self.descs[b]), self._stream), "rae_dist_step_end")
        return self.cost_t

    def read_global_cost(self) -> float:
        """The sum of the ranks' costs of the last step, as soon as every rank has emitted (the pulls keep running)."""
        self.eng._check(self.lib.rae_dist_read_cost(self.h, self.eng._cost_ref), "train()")
        return self.eng._cost.value

    def label_rows(self, de, indptr, indices, lo, hi, probs=True):
        """One rae_label_shards call: rows [lo, hi) read their W rows straight from the owners' shards (no collective, no
        host synchronisation, no capacity limit)."""
        n = hi - lo
        labels = torch.empty(n, dtype=torch.int64, device=self.device)
        q = torch.empty((n, de.K), dtype=torch.float32, device=self.device) if probs else None
        self.eng._check(self.lib.rae_label_shards(self.h, self.shard_buf["W"].peer_array(), de.world, C.c_void_p(indptr.data_ptr() + 4 * lo),
                                                  self._p(indices), n, self._p(labels), self._p(q), self._stream), "rae_label_shards")
        return labels, q

    def close(self):
        if self.eng is not None:
            self.eng._check(self.lib.rae_peer_status(self.h, self._stream), "peer barrier")
            torch.cuda.synchronize(self.device)
            if self.de.world > 1:
                dist.barrier(group=self.de.group)      # nobody unmaps while a peer may still read
            self.eng.close()
            self.eng = None
        for b in list(self.grad_buf.values()) + list(self.shard_buf.values()):
            b.close()
        self.grad_buf, self.shard_buf = {}, {}


# ----------------------------------------------------------------------------------------------------------------------
class DistributedEngine:
    """Same calls as :class:`relation_autoencoder_b200.engine.Engine`, one instance per rank."""

    def __init__(self, model: str, K: int, d: int, S: int, B: int, F: int, N: int, n_train: int, lr: float = 0.1,
                 l1: float = 0.0, l2: float = 0.0, alpha: float = 1.0, optimizer: str = "adagrad", ext_reg: bool = True,
                 device=0, rank: Optional[int] = None, world: Optional[int] = None, backend_factory=None, group=None,
                 peer_dense_max_bytes: int = 16 << 20):
        self.peer_dense_max_bytes = int(peer_dense_max_bytes)
        from .engine import MODEL_IDS, MODEL_PARAMS
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        if self.world > 16:
            raise ValueError("at most 16 ranks (RAE_MAX_PEERS)")
        self.group = group
        self.model, self.K, self.d, self.S, self.B, self.F, self.N = model, K, d, S, B, F, N
        self.n_train = n_train
        self.lr, self.alpha, self.optimizer = lr, alpha, optimizer
        self.l1, self.l2, self.ext_reg = float(l1), float(l2), bool(ext_reg)
        self.names = list(MODEL_PARAMS[MODEL_IDS[model]])
        self.dense_names = [n for n in self.names if n not in SPARSE]
        self.z_total = self.world * (4 * B + 2 * B * S)                       # global Z (OieModel.py:90)
        self.adj = float(self.world * B) / float(max(1, n_train))              # OieInduction.py:131 with the global batch
        self.dev = torch.device("cpu") if backend_factory is not None else torch.device("cuda", device)
        self.backend = backend_factory(self) if backend_factory is not None else CudaBackend(self)
        self.shard: Dict[str, torch.Tensor] = {}
        self.shard_acc: Dict[str, torch.Tensor] = {}
        self.dense: Dict[str, torch.Tensor] = {}
        self.dense_acc: Dict[str, torch.Tensor] = {}
        self.fplan: Optional[EpochPlan] = None
        self.eplan: Optional[EpochPlan] = None
        self.nb = 0
        self._ready = False
        self._label_split = {}
        self._train_csr32 = None
        self._profiling = False
        self._phase_log = []

    def _rows_total(self, name):
        return self.F if name == "W" else self.N

    def _width(self, name):
        return {"W": (self.K,), "A": (self.d,), "Ab": ()}[name]

    # ------------------------------------------------------------------ parameters
    def set_params_numpy(self, params: Dict[str, np.ndarray], acc: Optional[Dict[str, np.ndarray]] = None):
        """``params`` are the FULL tables (every rank passes the same arrays); each rank keeps its own rows.  Collective."""
        dt = self.backend.dtype if hasattr(self.backend, "dtype") else torch.float32
        shapes = {n: (len(range(self.rank, self._rows_total(n), self.world)),) + self._width(n) for n in SPARSE}
        self.shard = self.backend.alloc_tables(shapes)
        for n in self.names:
            if n in SPARSE:
                self.shard[n].copy_(torch.as_tensor(shard_rows(np.asarray(params[n]), self.rank, self.world)).to(self.dev, dt))
                self.shard_acc[n] = (torch.zeros_like(self.shard[n]) if acc is None else
                                     torch.as_tensor(shard_rows(np.asarray(acc[n]), self.rank, self.world)).to(self.dev, dt).contiguous())
            else:
                self.dense[n] = torch.as_tensor(np.ascontiguousarray(params[n])).to(self.dev, dt).contiguous()
                self.dense_acc[n] = (torch.zeros_like(self.dense[n]) if acc is None else
                                     torch.as_tensor(np.ascontiguousarray(acc[n])).to(self.dev, dt).contiguous())
        if self._ready:
            self.backend.bind_dense(self.dense, self.dense_acc)
            self.backend.plans_changed(self)          # shard / accumulator addresses are part of the step descriptors
        self._sync_all()

    def _sync_all(self):
        if self.dev.type == "cuda":
            torch.cuda.synchronize(self.dev)
        if self.world > 1:
            dist.barrier(group=self.group)

    def _gather_full(self, shards: Dict[str, torch.Tensor], dense: Dict[str, torch.Tensor]) -> Dict[str, np.ndarray]:
        out = {}
        for n in self.names:
            if n in SPARSE:
                total = self._rows_total(n)
                width = tuple(shards[n].shape[1:])
                full = torch.zeros((total,) + width, dtype=shards[n].dtype, device=self.dev)
                rows = (total + self.world - 1) // self.world
                pad = torch.zeros((rows,) + width, dtype=shards[n].dtype, device=self.dev)
                pad[: shards[n].shape[0]] = shards[n]
                if self.world > 1:
                    parts = [torch.empty_like(pad) for _ in range(self.world)]
                    dist.all_gather(parts, pad, group=self.group)
                else:
                    parts = [pad]
                for r in range(self.world):
                    cnt = len(range(r, total, self.world))
                    full[r::self.world] = parts[r][:cnt]
                out[n] = full.cpu().numpy()
            else:
                out[n] = dense[n].cpu().numpy()
        return out

    def get_params_numpy(self) -> Dict[str, np.ndarray]:
        return self._gather_full(self.shard, self.dense)

    def get_acc_numpy(self) -> Dict[str, np.ndarray]:
        return self._gather_full(self.shard_acc, self.dense_acc)

    # ------------------------------------------------------------------ data
    def _i64(self, x):
        if isinstance(x, torch.Tensor):
            return x.to(self.dev, torch.int64)
        return torch.as_tensor(np.ascontiguousarray(x)).to(self.dev, torch.int64)

    def _i32(self, x):
        if isinstance(x, torch.Tensor):
            return x.to(self.dev, torch.int32).contiguous()
        return torch.as_tensor(np.ascontiguousarray(x)).to(self.dev, torch.int32).contiguous()

    def bind_split(self, split: str, indptr, indices, args1=None, args2=None):
        """Local rows of the split.  For 'train' (collective): routing plan of the feature rows of every batch."""
        if split != "train":
            # every row of the split (labels are per example: any partition of the rows gives the same labels)
            self._label_split[split] = (self._i32(indptr), self._i32(indices))
            return
        ip, ix = self._i64(indptr), self._i64(indices)
        self._train_csr32 = None
        B = self.B
        nb = (ip.numel() - 1) // B
        if self.world > 1:
            nbt = torch.tensor([nb], device=self.dev)
            dist.all_reduce(nbt, op=dist.ReduceOp.MIN, group=self.group)
            nb = int(nbt.item())                                               # every rank steps the same number of batches
        self.nb = nb
        n_used = nb * B
        ip = ip[: n_used + 1].contiguous()
        base = int(ip[0].item())
        ix = ix[base:int(ip[-1].item())].contiguous()
        ip = ip - base
        self.ip, self.ix = ip, ix
        self.a1, self.a2 = self._i64(args1)[:n_used].contiguous(), self._i64(args2)[:n_used].contiguous()
        counts = ip[1:] - ip[:-1]
        row_of = torch.repeat_interleave(torch.arange(n_used, device=self.dev, dtype=torch.int64), counts)
        self.fplan = build_epoch_plan(ix, torch.div(row_of, B, rounding_mode="floor"), nb, self.F, self.rank, self.world, self.group)
        f_cap = max(self.fplan.max_u, 1)
        if self.world > 1:
            cap = torch.tensor([f_cap], device=self.dev)
            dist.all_reduce(cap, op=dist.ReduceOp.MAX, group=self.group)
            f_cap = int(cap.item())
        n_cap = (2 + 2 * self.S) * B
        self.backend.setup(f_cap, n_cap)
        self.backend.bind_dense(self.dense, self.dense_acc)
        self._ready = True
        # placeholders for the entity ids: the compact slots are per epoch (bind_epoch_negatives)
        zeros = torch.zeros(n_used, dtype=torch.int32, device=self.dev)
        self.backend.bind_train_csr(ip.to(torch.int32).contiguous(), self.fplan.compact, zeros, zeros)
        self._sync_all()

    def n_batches(self, split: str = "train") -> int:
        return self.nb

    def bind_epoch_negatives(self, neg1, neg2):
        """The epoch's negatives [S, n_local] (OieInduction.py:183-184).  Collective: routing plan of the entity rows of
        every batch (args1, args2 and the 2S negatives of each example)."""
        B, S, nb = self.B, self.S, self.nb
        n_used = nb * B
        n1 = self._i64(neg1)[:, :n_used]
        n2 = self._i64(neg2)[:, :n_used]
        col_batch = torch.div(torch.arange(n_used, device=self.dev, dtype=torch.int64), B, rounding_mode="floor")
        ids = torch.cat([self.a1, self.a2, n1.reshape(-1), n2.reshape(-1)])
        batch_of = torch.cat([col_batch, col_batch, col_batch.repeat(S), col_batch.repeat(S)])
        self.eplan = build_epoch_plan(ids, batch_of, nb, self.N, self.rank, self.world, self.group)
        c = self.eplan.compact
        self.a1c = c[:n_used].contiguous()
        self.a2c = c[n_used:2 * n_used].contiguous()
        self.n1c = c[2 * n_used:(2 + S) * n_used].reshape(S, n_used).contiguous()
        self.n2c = c[(2 + S) * n_used:].reshape(S, n_used).contiguous()
        self.backend.plans_changed(self)
        self._sync_all()

    # ------------------------------------------------------------------ the step
    def _step(self, b, n1c, n2c, neg_ld, want_cost, host_neg=None):
        """n1c / n2c None: the epoch's bound negatives (compact slots planned at bind time); host_neg: the caller's host
        arrays, checked against that plan on the device (CUDA backend)."""
        bk = self.backend
        B = self.B
        if n1c is None and not hasattr(bk, "descs"):
            n1c, n2c, neg_ld = self.n1c[:, b * B:], self.n2c[:, b * B:], self.nb * B
        ev = self._phase_events() if self._profiling else None
        if host_neg is not None:
            bk.run_begin_host(self, b, host_neg[0], host_neg[1])
        else:
            bk.run_begin(self, b, self.a1c[b * B:(b + 1) * B], self.a2c[b * B:(b + 1) * B], n1c, n2c, neg_ld)
        if ev: ev[1].record()
        peer_sync = getattr(bk, "peer_sync", False)               # CUDA backend: flag barriers over peer memory inside run_end
        if self.world > 1 and not getattr(bk, "peer_dense", False):
            if peer_sync and hasattr(bk, "dense_allreduce_aside"):
                # NCCL's all-reduce of the dense gradient runs on its own stream BESIDE the flag barrier and the sparse-row
                # applies of run_end (they do not need the sum); the dense update inside run_end waits for its event
                bk.dense_allreduce_aside(self.group)
            else:
                dist.all_reduce(bk.dense_grad, group=self.group)  # sum of the ranks' dense gradients (C | C1 | C2 | Wb);
        if ev: ev[2].record()                                     # without peer_sync it also orders "every rank has emitted"
        cost = bk.run_end(self, b)
        if ev: ev[3].record()
        if peer_sync and hasattr(bk, "read_global_cost"):
            # the ranks' costs were summed over peer memory inside run_end: nothing collective, nothing to wait for but the sum
            if ev:
                ev[4].record()
                self._phase_log.append(ev)
            return bk.read_global_cost() if (want_cost or host_neg is not None) else None
        if self.world > 1 and (want_cost or not peer_sync):
            dist.all_reduce(cost, group=self.group)               # global cost; without peer_sync: "every owner has applied"
        if ev:
            ev[4].record()
            self._phase_log.append(ev)
        return float(cost.item()) if want_cost else None

    def _phase_events(self):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        ev[0].record()
        return ev

    def set_profiling(self, on: bool):
        """Per-phase CUDA-event timing of the distributed step (fetch+local step | dense all-reduce | dense apply + pulls |
        cost all-reduce / barrier).  Adds event records: never on for a timed run."""
        self._profiling = bool(on) and self.dev.type == "cuda"
        self._phase_log = []

    def set_timeline(self, on: bool):
        """Timeline mode of this rank's handle (rae_set_profiling(h, 2)): events behind every kernel group of the sharded
        step on the stream it ran on, overlap kept."""
        self.backend.eng.set_profiling(2 if on else 0)

    def timeline(self):
        return self.backend.eng.timeline()

    def phase_times_ms(self) -> Dict[str, float]:
        names = ("fetch_and_local_step", "dense_allreduce", "dense_apply_and_pull", "cost_allreduce_barrier")
        if not self._phase_log:
            return {}
        torch.cuda.synchronize(self.dev)
        acc = {n: 0.0 for n in names}
        for ev in self._phase_log:
            for i, n in enumerate(names):
                acc[n] += ev[i].elapsed_time(ev[i + 1]) / len(self._phase_log)
        return acc

    def train_device(self, batch_index: int, want_cost: bool = True):
        b, B = int(batch_index), self.B
        if not (0 <= b < self.nb):
            raise RuntimeError("batch_index %d out of range [0,%d)" % (b, self.nb))
        if self.eplan is None:
            raise RuntimeError("epoch negatives are not bound (bind_epoch_negatives)")
        return self._step(b, None, None, 0, want_cost)

    def train(self, batch_index: int, neg1, neg2) -> float:
        """func['train'](batch_index, neg1, neg2) with this rank's HOST negatives [S,B] (the columns of the bound epoch
        negatives, as the reference's driver passes them, OieInduction.py:187-189); returns the GLOBAL batch cost."""
        b, B = int(batch_index), self.B
        if not (0 <= b < self.nb):
            raise RuntimeError("batch_index %d out of range [0,%d)" % (b, self.nb))
        if self.eplan is None:
            raise RuntimeError("epoch negatives are not bound (bind_epoch_negatives)")
        if hasattr(self.backend, "run_begin_host") and getattr(self.backend, "descs", None):
            return self._step(b, None, None, 0, True, host_neg=(neg1, neg2))
        u = self.eplan.ids_of(b).to(torch.int64)
        out = []
        ok = torch.ones((), dtype=torch.bool, device=self.dev)
        for x in (neg1, neg2):
            t = self._i64(x).contiguous()
            c = torch.searchsorted(u, t.reshape(-1)).clamp_(max=max(u.numel() - 1, 0))
            ok = ok & (u[c] == t.reshape(-1)).all()
            out.append(c.to(torch.int32).reshape(t.shape).contiguous())
        cost = self._step(b, out[0], out[1], B, True)
        if not bool(ok.item()):
            raise RuntimeError("train(): the negatives passed for batch %d are not the columns of the bound epoch negatives" % b)
        return cost

    def _label_csr(self, split: str):
        if split != "train":
            return self._label_split[split]
        if self._train_csr32 is None:
            self._train_csr32 = (self.ip.to(torch.int32).contiguous(), self.ix.to(torch.int32).contiguous())
        return self._train_csr32

    def label_rows(self, split: str, lo: int, hi: int, probs: bool = True):
        """Labels (device int64 [hi-lo]) and q(r|x) ([hi-lo, K], or None with ``probs=False``) of rows [lo, hi) of the bound
        split: every row of 'valid' / 'test', this rank's bound rows of 'train'.  The W rows are read from their owners;
        the CUDA backend needs no collective (one rae_label_shards call)."""
        ip, ix = self._label_csr(split)
        lo, hi = int(lo), int(hi)
        if not (0 <= lo <= hi <= ip.numel() - 1):
            raise RuntimeError("label_rows(%r, %d, %d): the split has %d rows" % (split, lo, hi, ip.numel() - 1))
        return self.backend.label_rows(self, ip, ix, lo, hi, probs)

    def label(self, split: str, batch_index: int):
        """func['label_<split>'](batch_index) for this rank's rows [b*B, (b+1)*B) of the bound split (label_rows)."""
        B = self.B
        labels, q = self.label_rows(split, batch_index * B, (batch_index + 1) * B)
        return labels.cpu().numpy(), q.cpu().numpy()

    # ------------------------------------------------------------------ misc
    def stats(self) -> dict:
        eng = getattr(self.backend, "eng", None)
        return eng.stats() if eng is not None else {}

    def close(self):
        self.backend.close()
