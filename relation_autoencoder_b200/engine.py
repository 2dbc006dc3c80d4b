"""Host-side mirror of the reference's run-time boundary on top of librae.so.

The reference driver touches its model only through ``self.func['train'](batch_index, neg1, neg2) -> cost`` and
``self.func['label_'+split](batch_index) -> (labels, probs)`` (learning/OieInduction.py:146-155, used at :189 and
:207/:216/:321-340) plus ``modelFunc.params`` for pickling (:114-116).  :class:`Engine` offers exactly these calls;
PyTorch is used only to own device memory and to provide the CUDA stream.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional

import numpy as np
import torch

from . import _lib as L

MODEL_IDS = {"rescal": L.RAE_MODEL_A, "sp": L.RAE_MODEL_C, "rescal+sp": L.RAE_MODEL_AC,
             "A": L.RAE_MODEL_A, "C": L.RAE_MODEL_C, "AC": L.RAE_MODEL_AC}     # README.md:44 / Decoder.py:85-93
MODEL_PARAMS = {L.RAE_MODEL_A: ["W", "Wb", "C", "A", "Ab"],                     # Bilinear.py:20
                L.RAE_MODEL_C: ["W", "Wb", "A", "C1", "C2", "Ab"],              # SelectionalPreferences.py:22
                L.RAE_MODEL_AC: ["W", "Wb", "C", "A", "Ab", "C1", "C2"]}        # BilinearPlusSP.py:32
_ORDER = ["W", "Wb", "A", "Ab", "C", "C1", "C2"]


def _ptr(t: Optional[torch.Tensor]):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class Engine:
    """One handle per GPU / rank.  Not thread-safe; all work is ordered on the current torch CUDA stream."""

    def __init__(self, model: str, K: int, d: int, S: int, B: int, F: int, N: int, n_train: int, lr: float = 0.1,
                 l1: float = 0.0, l2: float = 0.0, alpha: float = 1.0, optimizer: str = "adagrad", ext_reg: bool = True,
                 device: int = 0, flags: int = 0, z_total: int = 0, adj: Optional[float] = None):
        if model not in MODEL_IDS:
            raise ValueError("unknown decoder %r (expected rescal | sp | rescal+sp)" % (model,))
        if optimizer not in ("adagrad", "sgd"):
            raise Exception("Optimizer '{}' not implemented".format(optimizer))       # OieInduction.py:269
        self.lib = L.load()
        if not torch.cuda.is_available():
            raise RuntimeError("no CUDA device: the relation-autoencoder hot path has no CPU fallback")
        self.model_id = MODEL_IDS[model]
        self.K, self.d, self.S, self.B, self.F, self.N = int(K), int(d), int(S), int(B), int(F), int(N)
        self.n_train = int(n_train)
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        cfg = L.RaeConfig()
        cfg.abi_version = L.RAE_ABI_VERSION
        cfg.model = self.model_id
        cfg.K, cfg.d, cfg.S, cfg.B, cfg.F, cfg.N = self.K, self.d, self.S, self.B, self.F, self.N
        cfg.optimizer = L.RAE_OPT_ADAGRAD if optimizer == "adagrad" else L.RAE_OPT_SGD
        cfg.ext_reg = 1 if ext_reg else 0
        cfg.flags = int(flags)
        cfg.device = int(device)
        cfg.lr, cfg.l1, cfg.l2, cfg.alpha = float(lr), float(l1), float(l2), float(alpha)
        cfg.adj = float(adj) if adj is not None else float(B) / float(max(1, n_train))   # OieInduction.py:131
        cfg.z_total = int(z_total)
        self.cfg = cfg
        self.flags = int(flags)
        self._h = C.c_void_p(0)
        rc = self.lib.rae_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            raise RuntimeError("rae_create failed (%d): %s" % (rc, self.lib.rae_last_error(None).decode()))
        self.params: Dict[str, torch.Tensor] = {}
        self.acc: Dict[str, torch.Tensor] = {}
        self._keep = {}          # device tensors borrowed by the library
        self._cost = C.c_double(0.0)
        self._cost_ref = C.byref(self._cost)

    # ------------------------------------------------------------------ lifetime
    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            torch.cuda.synchronize(self.device)
            self.lib.rae_destroy(self._h)
            self._h = C.c_void_p(0)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise RuntimeError("%s failed (%d): %s" % (what, rc, self.lib.rae_last_error(self._h).decode()))

    @property
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def param_names(self):
        return list(MODEL_PARAMS[self.model_id])

    def param_shape(self, name):
        K, d, F, N = self.K, self.d, self.F, self.N
        return {"W": (F, K), "Wb": (K,), "A": (N, d), "Ab": (N,), "C": (d, d, K), "C1": (d, K), "C2": (d, K)}[name]

    # ------------------------------------------------------------------ bindings
    def bind_params(self, params: Dict[str, torch.Tensor], acc: Optional[Dict[str, torch.Tensor]] = None):
        """Borrow fp32 CUDA tensors as the model parameters (theano.shared equivalents) and their AdaGrad
        accumulators (zeros when not given, Optimizers.py:12-15)."""
        for n in self.param_names():
            t = params[n]
            if not (t.is_cuda and t.dtype == torch.float32 and t.is_contiguous() and tuple(t.shape) == self.param_shape(n)):
                raise ValueError("parameter %s must be a contiguous fp32 CUDA tensor of shape %s" % (n, self.param_shape(n)))
        self.params = {n: params[n] for n in self.param_names()}
        if acc is None:
            acc = {n: torch.zeros_like(t) for n, t in self.params.items()}
        self.acc = {n: acc[n] for n in self.param_names()}
        a = [_ptr(self.params.get(n)) for n in _ORDER]
        self._check(self.lib.rae_bind_params(self._h, *a), "rae_bind_params")
        a = [_ptr(self.acc.get(n)) for n in _ORDER]
        self._check(self.lib.rae_bind_accumulators(self._h, *a), "rae_bind_accumulators")

    def set_params_numpy(self, params: Dict[str, np.ndarray], acc: Optional[Dict[str, np.ndarray]] = None):
        dev = {n: torch.as_tensor(np.ascontiguousarray(params[n], dtype=np.float32)).to(self.device) for n in self.param_names()}
        dacc = None
        if acc is not None:
            dacc = {n: torch.as_tensor(np.ascontiguousarray(acc[n], dtype=np.float32)).to(self.device) for n in self.param_names()}
        self.bind_params(dev, dacc)

    def get_params_numpy(self) -> Dict[str, np.ndarray]:
        torch.cuda.synchronize(self.device)
        return {n: t.detach().cpu().numpy() for n, t in self.params.items()}

    def get_acc_numpy(self) -> Dict[str, np.ndarray]:
        torch.cuda.synchronize(self.device)
        return {n: t.detach().cpu().numpy() for n, t in self.acc.items()}

    def _dev_i32(self, x):
        if isinstance(x, torch.Tensor):
            t = x.to(device=self.device, dtype=torch.int32)
        else:
            t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.int32)).to(self.device)
        return t.contiguous()

    def bind_split(self, split: str, indptr, indices, args1=None, args2=None):
        """``make_shared(DatasetSplit)`` (OieInduction.py:439-449): binary CSR + int32 entity ids, device resident."""
        sid = L.RAE_SPLIT[split]
        ip, ix = self._dev_i32(indptr), self._dev_i32(indices)
        a1 = self._dev_i32(args1) if args1 is not None else None
        a2 = self._dev_i32(args2) if args2 is not None else None
        n_rows = ip.numel() - 1
        self._keep[("split", sid)] = (ip, ix, a1, a2)
        self._check(self.lib.rae_bind_split(self._h, sid, _ptr(ip), _ptr(ix), n_rows, _ptr(a1), _ptr(a2), self._stream),
                    "rae_bind_split")

    def n_batches(self, split: str = "train") -> int:
        ip = self._keep[("split", L.RAE_SPLIT[split])][0]
        return (ip.numel() - 1) // self.B        # trailing partial batch dropped, OieInduction.py:96-98

    def bind_epoch_negatives(self, neg1, neg2):
        """The epoch's negative ids [S, N_train] (OieInduction.py:183-184) kept on the device."""
        n1, n2 = self._dev_i32(neg1), self._dev_i32(neg2)
        if n1.dim() != 2 or n1.shape != n2.shape or n1.shape[0] != self.S:
            raise ValueError("negatives must be int32 [S, n] arrays")
        self._keep["neg"] = (n1, n2)
        self._check(self.lib.rae_bind_epoch_negatives(self._h, _ptr(n1), _ptr(n2), n1.shape[1]), "rae_bind_epoch_negatives")

    # ------------------------------------------------------------------ func['train']
    def _host_negatives(self, neg):
        """(array kept alive, address, row stride in elements) of an int32 [S, B] host array; column slices of the
        epoch's [S, n] arrays (what the driver passes, OieInduction.py:187-188) are used in place."""
        if not (isinstance(neg, np.ndarray) and neg.dtype == np.int32 and neg.ndim == 2):
            neg = np.ascontiguousarray(neg, dtype=np.int32)
        if neg.shape != (self.S, self.B):
            raise ValueError("neg1/neg2 must have shape (S, B) = (%d, %d)" % (self.S, self.B))
        s0, s1 = neg.strides
        if self.S and self.B and (s1 != 4 or s0 % 4 or s0 < 4 * self.B):
            neg = np.ascontiguousarray(neg)
            s0 = 4 * self.B
        return neg, neg.__array_interface__["data"][0], s0 // 4

    def train(self, batch_index: int, neg1: np.ndarray, neg2: np.ndarray) -> float:
        """Drop-in for ``func['train'](batch_index, neg1, neg2)`` (OieInduction.py:146-149,189): host int32 [S,B]
        negatives in, regularised batch cost out, parameters updated in place (the cost is returned as soon as the
        forward pass has produced it; the updates complete in stream order before anything else reads them)."""
        n1, p1, ld1 = self._host_negatives(neg1)
        n2, p2, ld2 = self._host_negatives(neg2)
        self._check(self.lib.rae_train_step_host_ld(self._h, int(batch_index), p1, ld1, p2, ld2, self._cost_ref, self._stream),
                    "rae_train_step_host")
        return self._cost.value

    def train_device(self, batch_index: int, want_cost: bool = True) -> Optional[float]:
        """Same step with the epoch negatives already bound on the device; asynchronous when ``want_cost`` is False."""
        cp = C.byref(self._cost) if want_cost else C.POINTER(C.c_double)()
        self._check(self.lib.rae_train_step(self._h, int(batch_index), cp, self._stream), "rae_train_step")
        return float(self._cost.value) if want_cost else None

    def train_explicit(self, indptr, indices, a1, a2, neg1, neg2) -> float:
        """One step on injected inputs (parity tests): everything is copied to the device first."""
        ip, ix = self._dev_i32(indptr), self._dev_i32(indices)
        t1, t2 = self._dev_i32(a1), self._dev_i32(a2)
        n1, n2 = self._dev_i32(neg1), self._dev_i32(neg2)
        if ip.numel() != self.B + 1:
            raise ValueError("indptr must have B+1 entries")
        self._keep["explicit"] = (ip, ix, t1, t2, n1, n2)
        self._check(self.lib.rae_train_step_explicit(self._h, _ptr(ip), _ptr(ix), _ptr(t1), _ptr(t2), _ptr(n1), _ptr(n2),
                                                     n1.shape[1] if n1.dim() == 2 else self.B, C.byref(self._cost),
                                                     self._stream), "rae_train_step_explicit")
        return float(self._cost.value)

    # ------------------------------------------------------------------ func['label_<split>']
    def label(self, split: str, batch_index: int):
        """Drop-in for ``func['label_'+split](batch_index)`` -> (labels int64[B], probs float32[B,K])."""
        labels = np.empty(self.B, dtype=np.int64)
        probs = np.empty((self.B, self.K), dtype=np.float32)
        self._check(self.lib.rae_label_host(self._h, L.RAE_SPLIT[split], int(batch_index),
                                            labels.ctypes.data_as(C.c_void_p), probs.ctypes.data_as(C.c_void_p),
                                            self._stream), "rae_label_host")
        return labels, probs

    def label_topk(self, indptr, indices, k: int, probs: bool = True):
        """The k most probable relations of every row of a host or device int32 CSR (any number of rows, none dropped),
        from the bound W and Wb in one ``rae_label_topk`` call -> (ids int32 [n, k], probs float32 [n, k] or None).
        ids run by score descending, equal scores by ascending relation id, so ``ids[:, 0]`` is the argmax label."""
        if not self.params:
            raise RuntimeError("label_topk needs bound parameters (bind_params / set_params_numpy)")
        ip, ix = self._dev_i32(indptr), self._dev_i32(indices)
        n, k = ip.numel() - 1, int(k)
        if ix.numel() == 0:                  # rows without features only: the library wants a non-null array
            ix = torch.zeros(1, dtype=torch.int32, device=self.device)
        size = max(n * k, 1)                 # non-null outputs for n == 0 too (the call then launches nothing)
        ids = torch.empty(size, dtype=torch.int32, device=self.device)
        q = torch.empty(size, dtype=torch.float32, device=self.device) if probs else None
        w = (C.c_void_p * 1)(self.params["W"].data_ptr())
        self._check(self.lib.rae_label_topk(self._h, w, 1, _ptr(ip), _ptr(ix), n, k, _ptr(ids), _ptr(q), self._stream),
                    "rae_label_topk")
        torch.cuda.synchronize(self.device)
        ids = ids[:n * k].reshape(n, k).cpu().numpy()
        return ids, (q[:n * k].reshape(n, k).cpu().numpy() if q is not None else None)

    def _argument_inputs(self, what, indptr, indices, args1, args2):
        """Host checks shared by rank_arguments / predict_arguments -> (n, indptr, indices, args1, args2) on the device
        (non-null arrays for n == 0 and for rows without features)."""
        if not self.params:
            raise RuntimeError("%s needs bound parameters (bind_params / set_params_numpy)" % what)
        ip_h = np.asarray(indptr.cpu() if isinstance(indptr, torch.Tensor) else indptr, dtype=np.int64)
        ix_h = np.asarray(indices.cpu() if isinstance(indices, torch.Tensor) else indices, dtype=np.int64)
        a1_h = np.asarray(args1.cpu() if isinstance(args1, torch.Tensor) else args1, dtype=np.int64)
        a2_h = np.asarray(args2.cpu() if isinstance(args2, torch.Tensor) else args2, dtype=np.int64)
        n = ip_h.size - 1
        if n < 0 or a1_h.shape != (n,) or a2_h.shape != (n,):
            raise ValueError("%s: indptr has %d entries, args1 %s and args2 %s; expected n+1, (n,), (n,)"
                             % (what, ip_h.size, a1_h.shape, a2_h.shape))
        if n > 0 and (np.any(np.diff(ip_h) < 0) or ip_h[0] < 0 or ip_h[-1] > ix_h.size):
            raise ValueError("%s: indptr is not a non-decreasing offset array into %d indices" % (what, ix_h.size))
        for name, a in (("args1", a1_h), ("args2", a2_h)):
            if a.size and (a.min() < 0 or a.max() >= self.N):
                raise ValueError("%s: %s holds entity ids outside [0, N = %d): min %d, max %d"
                                 % (what, name, self.N, a.min(), a.max()))
        used = ix_h[ip_h[0]:ip_h[-1]] if n > 0 else ix_h[:0]
        if used.size and (used.min() < 0 or used.max() >= self.F):
            raise ValueError("%s: indices hold feature ids outside [0, F = %d): min %d, max %d"
                             % (what, self.F, used.min(), used.max()))
        ip, ix = self._dev_i32(indptr), self._dev_i32(indices)
        a1, a2 = self._dev_i32(args1), self._dev_i32(args2)
        if ix.numel() == 0:                  # rows without features only: the library wants a non-null array
            ix = torch.zeros(1, dtype=torch.int32, device=self.device)
        if n == 0:
            a1 = a2 = torch.zeros(1, dtype=torch.int32, device=self.device)
        return n, ip, ix, a1, a2

    def rank_arguments(self, indptr, indices, args1, args2):
        """Entity ranks of every row's true arguments under the bound model, from one ``rae_rank_arguments`` call ->
        (rank1 int32 [n], rank2 int32 [n]).  rank_s = 1 + the number of other entities whose candidate score in slot s
        (the decoder's negative-sample score with that argument replaced) exceeds the true one's.  Host or device int32
        CSR and argument ids of any length; entity ids must lie in [0, N) and feature ids in [0, F).  The call reuses the
        handle's per-batch scratch, so ``last_probs`` afterwards no longer shows the last training step."""
        n, ip, ix, a1, a2 = self._argument_inputs("rank_arguments", indptr, indices, args1, args2)
        r1 = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        r2 = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        self._check(self.lib.rae_rank_arguments(self._h, _ptr(ip), _ptr(ix), _ptr(a1), _ptr(a2), n, _ptr(r1), _ptr(r2),
                                                self._stream), "rae_rank_arguments")
        torch.cuda.synchronize(self.device)
        return r1[:n].cpu().numpy(), r2[:n].cpu().numpy()

    def predict_arguments(self, indptr, indices, args1, args2, k: int):
        """The k most likely entities of each argument slot of every row, from one ``rae_predict_arguments`` call ->
        (ids1 int32 [n, k], scores1 float32 [n, k], ids2, scores2).  Slot 1 lists candidates for args1 (it reads args2,
        never args1), slot 2 candidates for args2 (it reads args1, never args2); per row, score descending, equal scores by
        ascending entity id.  Scores order a row's candidates but are not comparable across rows.  Inputs and checks as
        :meth:`rank_arguments`, and 1 <= k <= min(N, 16).  The call reuses the handle's per-batch scratch, so
        ``last_probs`` afterwards no longer shows the last training step."""
        k = int(k)
        if not 1 <= k <= min(self.N, L.RAE_MAX_TOPK):
            raise ValueError("predict_arguments: k = %d is outside [1, min(N = %d, %d)]" % (k, self.N, L.RAE_MAX_TOPK))
        n, ip, ix, a1, a2 = self._argument_inputs("predict_arguments", indptr, indices, args1, args2)
        size = max(n * k, 1)
        out = [torch.empty(size, dtype=dt, device=self.device) for dt in (torch.int32, torch.float32) * 2]
        self._check(self.lib.rae_predict_arguments(self._h, _ptr(ip), _ptr(ix), _ptr(a1), _ptr(a2), n, k,
                                                   *[_ptr(t) for t in out], self._stream), "rae_predict_arguments")
        torch.cuda.synchronize(self.device)
        return tuple(t[:n * k].reshape(n, k).cpu().numpy() for t in out)

    # ------------------------------------------------------------------ introspection
    def last_probs(self) -> np.ndarray:
        out = torch.empty(self.B, self.K, dtype=torch.float32, device=self.device)
        self._check(self.lib.rae_get_probs(self._h, _ptr(out), self._stream), "rae_get_probs")
        return out.cpu().numpy()

    def dense_grads(self) -> Dict[str, np.ndarray]:
        res = {}
        for n in self.param_names():
            out = torch.empty(self.param_shape(n), dtype=torch.float32, device=self.device)
            self._check(self.lib.rae_get_dense_grad(self._h, L.PARAM_IDS[n], _ptr(out), self._stream), "rae_get_dense_grad")
            res[n] = out.cpu().numpy()
        return res

    def entity_segments(self):
        n_occ = (2 + 2 * self.S) * self.B
        rows = torch.empty(n_occ, dtype=torch.int32, device=self.device)
        occ = torch.empty(n_occ, dtype=torch.int32, device=self.device)
        seg = torch.empty(n_occ + 1, dtype=torch.int32, device=self.device)
        a, b = C.c_int64(0), C.c_int64(0)
        self._check(self.lib.rae_get_entity_segments(self._h, _ptr(rows), _ptr(occ), _ptr(seg), C.byref(a), C.byref(b),
                                                     self._stream), "rae_get_entity_segments")
        torch.cuda.synchronize(self.device)
        return rows.cpu().numpy(), occ.cpu().numpy(), seg.cpu().numpy()[: b.value + 1]

    def set_profiling(self, on):
        """False / 0 = off, True / 1 = per-phase (serialised), 2 = timeline of the overlapped step (``timeline()``)."""
        self._check(self.lib.rae_set_profiling(self._h, int(on)), "rae_set_profiling")

    def timeline(self):
        """[(mark, stream, microseconds since the step's start)] of the last step run under ``set_profiling(2)``."""
        buf = C.create_string_buffer(8192)
        self._check(self.lib.rae_get_timeline(self._h, buf, len(buf)), "rae_get_timeline")
        out = []
        for ln in buf.value.decode().splitlines():
            n, s, t = ln.split()
            out.append((n, int(s), float(t)))
        return out

    def phase_times_ms(self) -> Dict[str, float]:
        buf = (C.c_float * L.RAE_NUM_PHASES)()
        self._check(self.lib.rae_get_phase_times(self._h, buf), "rae_get_phase_times")
        return {self.lib.rae_phase_name(i).decode(): float(buf[i]) for i in range(L.RAE_NUM_PHASES)}

    def stats(self) -> dict:
        st = L.RaeStepStats()
        self._check(self.lib.rae_get_step_stats(self._h, C.byref(st)), "rae_get_step_stats")
        return {f: getattr(st, f) for f, _ in st._fields_}
