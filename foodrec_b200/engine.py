"""Device engine: owns the tables (torch CUDA tensors = device memory + streams only)
and drives libfoodrec_b200.so through the C ABI.  No compute happens in Python or
torch; without the CUDA library every entry point raises."""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib as L


@dataclass
class Hyper:
    """The ``args`` fields ``Model.__init__`` reads (Model_Recommender.py:6-24) plus the
    TF-1.x optimizer defaults the reference inherits."""
    learner: str = "adam"
    lr: float = 0.001
    high_level_score_coefficient: float = 0.99
    beta_1: float = 0.01
    beta_2: float = 0.01
    alpha: float = 0.01
    clip_norm: float = 5.0
    adam_beta1: float = 0.9
    adam_beta2: float = 0.999
    adam_eps: float = 1e-8
    adagrad_init: float = 0.1
    rms_decay: float = 0.9
    rms_eps: float = 1e-10

    @classmethod
    def from_args(cls, args):
        return cls(learner=args.learner, lr=float(args.lr),
                   high_level_score_coefficient=float(args.high_level_score_coefficient),
                   beta_1=float(args.beta_1), beta_2=float(args.beta_2), alpha=float(args.alpha))


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def exclusion_csr(exclude, n):
    """Per-query-row exclusion lists as a CSR ``(offsets int32 [n+1], ids int32 [nnz])``.

    ``exclude`` is either a tuple ``(offsets, ids)`` (numpy / torch / sequences) or a list of ``n`` per-row sequences
    of recipe ids.  Host offsets are validated: ``n+1`` entries, the first 0, non-decreasing, the last ``len(ids)``.
    CUDA tensors are passed through after a length check (validating them would wait for the device).  Ids may be
    anything in int32: ids the table cannot return are ignored by the kernels."""
    if isinstance(exclude, tuple):
        if len(exclude) != 2:
            raise ValueError("exclude=(offsets, ids) takes two arrays")
        off, ids = exclude
        if torch.is_tensor(off) and off.is_cuda and torch.is_tensor(ids) and ids.is_cuda:
            if off.numel() != n + 1:
                raise ValueError(f"exclusion offsets: {off.numel()} entries for {n} query rows (want {n + 1})")
            return off.to(torch.int32).contiguous().reshape(-1), ids.to(torch.int32).contiguous().reshape(-1)
        off = (off.cpu().numpy() if torch.is_tensor(off) else np.asarray(off)).reshape(-1)
        ids = (ids.cpu().numpy() if torch.is_tensor(ids) else np.asarray(ids)).reshape(-1)
    else:
        rows = [np.asarray(r.cpu().numpy() if torch.is_tensor(r) else r).reshape(-1) for r in exclude]
        rows = [r if r.size else r.astype(np.int64) for r in rows]          # an empty list is float64 to numpy
        if len(rows) != n:
            raise ValueError(f"exclude has {len(rows)} lists for {n} query rows")
        off = np.zeros(n + 1, np.int64)
        off[1:] = np.cumsum([r.size for r in rows])
        ids = np.concatenate(rows) if rows else np.zeros(0, np.int64)
    if off.size and not np.issubdtype(off.dtype, np.integer) or ids.size and not np.issubdtype(ids.dtype, np.integer):
        raise TypeError("exclusion offsets and ids must be integers")
    off = off.astype(np.int64); ids = ids.astype(np.int64)
    if off.shape != (n + 1,):
        raise ValueError(f"exclusion offsets: {off.size} entries for {n} query rows (want {n + 1})")
    if off[0] != 0 or off[-1] != ids.size or (np.diff(off) < 0).any():
        raise ValueError(f"exclusion offsets must start at 0, be non-decreasing and end at len(ids) = {ids.size}")
    if ids.size and (ids.min() < -2**31 or ids.max() >= 2**31):
        raise ValueError("exclusion ids must fit int32")
    return off.astype(np.int32), ids.astype(np.int32)


class Engine:
    def __init__(self, hyper: Hyper, P, R, Cat, G, device="cuda:0", max_rows=1 << 16,
                 max_label_entries=None, adam_mode="lazy", item_cats=None, user_labels=None,
                 user_label_csr=None, adopt=False, single_pass=None, table_dtype="float32"):
        self.lib = L.lib()                       # raises if the .so is missing
        if not torch.cuda.is_available():
            raise RuntimeError("foodrec_b200 needs a CUDA device (no CPU fallback)")
        self.device = torch.device(device)
        torch.cuda.set_device(self.device)
        self.h = hyper
        # adopt=True: float32 tensors that already live on the device are used in place (no second copy of a
        # table that fills a third of the HBM: cfg3 shards)
        def dev(x):
            if adopt and torch.is_tensor(x) and x.device == self.device and x.is_contiguous() and (
                    x.dtype == torch.float32 or (x.dtype == torch.bfloat16 and table_dtype == "bf16")):
                return x
            return torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x,
                                   dtype=torch.float32).to(self.device).contiguous().clone()
        self.P, self.R, self.Cat, self.G = dev(P), dev(R), dev(Cat), dev(G)
        # bf16 tables (BASELINE configs[4]): Personal_Memory / Recipe_Embedding are STORED in bfloat16 (fp32 arithmetic,
        # round to nearest even on store: fr_set_table_format); Cat, G and the optimizer slots stay fp32
        if table_dtype not in ("float32", "bf16"):
            raise ValueError("table_dtype must be 'float32' or 'bf16'")
        self.table_bf16 = table_dtype == "bf16"
        if self.table_bf16:
            if L.learner_code(hyper.learner) == L.FR_ADAM:
                raise L.FoodRecError("bf16 tables are offered for SGD / Adagrad / RMSProp (TF-1.x Adam moves every row every "
                                     "step: see include/foodrec_b200.h:fr_set_table_format)")
            self.P, self.R = self.P.to(torch.bfloat16), self.R.to(torch.bfloat16)     # torch rounds to nearest even
            self.Cat, self.G = self.Cat.float(), self.G.float()
        self.U, five, self.D = self.P.shape
        assert five == 5 and self.Cat.shape == (4, self.D) and self.R.shape[1] == self.D
        self.I, self.Lb = self.R.shape[0], self.G.shape[0]
        self.learner = L.learner_code(hyper.learner)
        modes = {"dense": L.FR_ADAM_DENSE, "lazy_exact": L.FR_ADAM_LAZY_EXACT,
                 "lazy": L.FR_ADAM_LAZY_SERIES, "lazy_series": L.FR_ADAM_LAZY_SERIES}
        if adam_mode not in modes:
            raise ValueError(f"adam_mode must be one of {sorted(modes)}")
        self.adam_mode = modes[adam_mode]
        z = lambda t: torch.zeros(t.shape, dtype=torch.float32, device=t.device)
        self.s1 = {}; self.s2 = {}
        tabs = {"P": self.P, "R": self.R, "Cat": self.Cat}
        if self.learner == L.FR_ADAM:
            self.s1 = {k: z(v) for k, v in tabs.items()}; self.s2 = {k: z(v) for k, v in tabs.items()}
        elif self.learner == L.FR_ADAGRAD:
            self.s1 = {k: torch.full(v.shape, hyper.adagrad_init, dtype=torch.float32, device=v.device) for k, v in tabs.items()}
        elif self.learner == L.FR_RMSPROP:
            self.s1 = {k: z(v) + 1.0 for k, v in tabs.items()}; self.s2 = {k: z(v) for k, v in tabs.items()}
        self.last_P = torch.zeros(self.U, dtype=torch.int32, device=self.device)
        self.last_R = torch.zeros(self.I, dtype=torch.int32, device=self.device)
        self.item_cats = None
        self.lab_off = self.lab_idx = None
        self.max_labels_per_user = self.Lb
        if item_cats is not None:
            # [I,4] for this table's recipes -- or, for a row-sharded engine, the GLOBAL map
            self.item_cats = torch.as_tensor(np.asarray(item_cats, np.float32).reshape(-1, 4)).to(self.device).contiguous()
        if user_labels is not None:     # dense [U, L] multi-hot -> CSR (weights must be 0/1)
            ul = np.asarray(user_labels)
            assert ul.shape == (self.U, self.Lb)
            if not np.isin(ul, (0, 1)).all():
                raise ValueError("resident user-label table must be 0/1 (use the dense feed for weights)")
            rows, cols = np.nonzero(ul)
            cnt = np.bincount(rows, minlength=self.U)
            off = np.zeros(self.U + 1, np.int32); off[1:] = np.cumsum(cnt)
            self.lab_off = torch.as_tensor(off).to(self.device)
            self.lab_idx = torch.as_tensor(cols.astype(np.int32)).to(self.device)
            self.max_labels_per_user = int(cnt.max()) if cnt.size else 1
        elif user_label_csr is not None:   # (offsets [U+1], label ids [nnz]) built by the caller
            off, idx = (np.asarray(x, np.int32) for x in user_label_csr)
            assert off.shape == (self.U + 1,) and off[-1] == idx.shape[0]
            if idx.size and (idx.min() < 0 or idx.max() >= self.Lb) or (np.diff(off) < 0).any():
                raise IndexError(f"user-label CSR: label ids must lie in [0, {self.Lb}) and offsets be non-decreasing")
            self.lab_off = torch.as_tensor(off).to(self.device)
            self.lab_idx = torch.as_tensor(idx).to(self.device)
            self.max_labels_per_user = int(np.diff(off).max())
        self.max_rows = int(max_rows)
        if max_label_entries is None:
            max_label_entries = self.max_rows * (self.max_labels_per_user if self.lab_off is not None else min(self.Lb, 16))
        self.max_label_entries = int(min(max_label_entries, 2**31 - 1))
        cfg = L.fr_config(self.D, self.U, self.I, self.Lb, self.learner, self.adam_mode, self.max_rows,
                          self.max_label_entries, hyper.lr, hyper.high_level_score_coefficient,
                          hyper.beta_1, hyper.beta_2, hyper.alpha, hyper.clip_norm,
                          hyper.adam_beta1, hyper.adam_beta2, hyper.adam_eps, hyper.rms_decay, hyper.rms_eps)
        self.handle = C.c_void_p()
        rc = self.lib.fr_create(C.byref(cfg), C.byref(self.handle))
        if rc == L.FR_ERR_UNSUPPORTED and adam_mode == "lazy":
            # "lazy" = the fastest exact-to-fp32 scheme: the closed-form catch-up where its truncation bound covers
            # the configured betas (fr_create checks), else the step-by-step replay (bit-identical to the dense sweep)
            import warnings
            warnings.warn("foodrec_b200: " + self.lib.fr_last_error(self.handle).decode() + " -- falling back to lazy_exact")
            self.lib.fr_destroy(self.handle); self.handle = C.c_void_p()
            self.adam_mode = cfg.adam_mode = L.FR_ADAM_LAZY_EXACT
            rc = self.lib.fr_create(C.byref(cfg), C.byref(self.handle))
        if rc != L.FR_OK:
            msg = self.lib.fr_last_error(self.handle).decode() if self.handle else "fr_create failed"
            self.lib.fr_destroy(self.handle); self.handle = None
            raise L.FoodRecError(msg)
        if self.table_bf16:
            L.check(self.handle, self.lib.fr_set_table_format(self.handle, L.FR_TABLE_BF16))
            single_pass = False
        self._set_tables()
        # Single-pass step (fr_set_shadow): a second copy of Personal_Memory + its Adam slots lets the library score and
        # update a user's rows in ONE kernel (the two-pass step reads them twice: 6.1 -> 4.0 GB of DRAM traffic per
        # cfg2 step).  Default: on for lazy Adam when the extra 3 x |P| bytes leave half of the free memory untouched.
        lazy_adam = self.learner == L.FR_ADAM and self.adam_mode != L.FR_ADAM_DENSE
        if single_pass is None:
            need = 3 * self.P.numel() * 4
            single_pass = lazy_adam and need < 0.5 * torch.cuda.mem_get_info(self.device)[0]
        self.single_pass = bool(single_pass) and lazy_adam
        self._shadow = None
        if self.single_pass:
            self._shadow = [torch.empty_like(self.P) for _ in range(3)]
            L.check(self.handle, self.lib.fr_set_shadow(self.handle, *[_ptr(t) for t in self._shadow]))
        self.out = torch.zeros(L.FR_OUT_COUNT, dtype=torch.float32, device=self.device)
        self.out_host = torch.zeros(L.FR_OUT_COUNT, dtype=torch.float32).pin_memory()
        self._dirty = False          # lazy Adam rows pending a flush
        self._keep = []

    # ------------------------------------------------------------------ plumbing
    def _set_tables(self):
        t = L.fr_tables()
        t.P, t.R, t.Cat, t.G = _ptr(self.P), _ptr(self.R), _ptr(self.Cat), _ptr(self.G)
        g = lambda d, k: _ptr(d.get(k))
        t.s1_P, t.s2_P = g(self.s1, "P"), g(self.s2, "P")
        t.s1_R, t.s2_R = g(self.s1, "R"), g(self.s2, "R")
        t.s1_Cat, t.s2_Cat = g(self.s1, "Cat"), g(self.s2, "Cat")
        t.last_P, t.last_R = _ptr(self.last_P), _ptr(self.last_R)
        t.item_cats, t.user_label_off, t.user_label_idx = _ptr(self.item_cats), _ptr(self.lab_off), _ptr(self.lab_idx)
        L.check(self.handle, self.lib.fr_set_tables(self.handle, C.byref(t)))

    def close(self):
        if getattr(self, "handle", None):
            torch.cuda.synchronize(self.device)
            self.lib.fr_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @property
    def step(self) -> int:
        s = C.c_int64()
        L.check(self.handle, self.lib.fr_get_step(self.handle, C.byref(s)))
        return s.value

    def _i32(self, x):
        if torch.is_tensor(x):
            return x.to(self.device, torch.int32).contiguous().reshape(-1)
        return torch.as_tensor(np.ascontiguousarray(np.asarray(x).astype(np.int32)).reshape(-1)).to(self.device)

    def _check_ids(self, x, n, what):
        """Host-side range check of ids that arrive as host data (lists / numpy / CPU tensors): the reference's
        tf.gather raises for an id outside its table.  Device tensors are checked on the device by the kernels
        (train step: FR_OUT_OVERFLOW = 3 -> read_scalars raises; inference: NaN score / empty rank list)."""
        if torch.is_tensor(x):
            if x.is_cuda or x.numel() == 0:
                return
            lo, hi = int(x.min()), int(x.max())
        else:
            a = np.asarray(x)
            if a.size == 0:
                return
            a = a.astype(np.int64)
            lo, hi = int(a.min()), int(a.max())
        if lo < 0 or hi >= n:
            raise IndexError(f"{what}: ids must lie in [0, {n}), got [{lo}, {hi}]")

    def _f32(self, x, shape=None):
        if x is None:
            return None
        if torch.is_tensor(x):
            t = x.to(self.device, torch.float32).contiguous()
        else:
            t = torch.as_tensor(np.ascontiguousarray(np.asarray(x, dtype=np.float32))).to(self.device)
        return t.reshape(shape) if shape is not None else t

    # ------------------------------------------------------------------ hot path
    def train_step(self, users, items, labels=None, categories=None, write_sign=None,
                   user_one_hot_label=None, neg_items=None, neg_categories=None,
                   write_personal=False, return_scores=False):
        """One optimizer step on device-resident (or host, copied here) feed tensors.
        Pointwise when ``neg_items`` is None, else BPR.  Returns the device scalar
        vector (FR_OUT_*); nothing is synchronised."""
        self._check_ids(users, self.U, "user_input"); self._check_ids(items, self.I, "item_input")
        u = self._i32(users)
        B = u.numel()
        bpr = neg_items is not None
        if bpr:
            self._check_ids(neg_items, self.I, "neg_item_input")
            it = torch.stack([self._i32(items), self._i32(neg_items)], 1).reshape(-1).contiguous()
            cats = None
            if categories is not None:
                if neg_categories is None:
                    raise ValueError("BPR step: `categories` was given without `neg_categories` (pass both, or neither "
                                     "to use the resident dish_to_category table)")
                cats = torch.stack([self._f32(categories, (B, 4)), self._f32(neg_categories, (B, 4))], 1).reshape(-1, 4).contiguous()
        else:
            it = self._i32(items)
            cats = self._f32(categories, (B, 4))
        S = it.numel()
        ws = self._f32(write_sign, (-1,))
        if ws is not None and ws.numel() != S:
            if bpr and ws.numel() == B:
                # one sign per TRIPLE: the C ABI wants one per item row (S = 2B, interleaved pos/neg); the sign of a
                # triple applies to its positive row and is negated for its negative row (the +1/-1 default pattern)
                ws = torch.stack([ws, -ws], 1).reshape(-1).contiguous()
            else:
                raise ValueError(f"write_sign has {ws.numel()} entries; the step has {S} item rows"
                                 + (f" ({B} triples)" if bpr else ""))
        lab = self._f32(labels, (-1,))
        if not bpr and (lab is None or lab.numel() != B):
            raise ValueError(f"labels must have one entry per row ({B})")
        return self._step_dev(L.FR_BPR if bpr else L.FR_POINTWISE, B, u, it, cats, lab,
                              ws, self._f32(user_one_hot_label, (B, self.Lb)),
                              write_personal, return_scores)

    def _step_dev(self, mode, B, users, items, cats, labels, ws, ulab, write_personal=False, return_scores=False):
        b = L.fr_batch(mode, B, _ptr(users), _ptr(items), _ptr(cats), _ptr(labels), _ptr(ws), _ptr(ulab))
        scores = torch.empty(items.numel(), dtype=torch.float32, device=self.device) if return_scores else None
        L.check(self.handle, self.lib.fr_train_step(self.handle, C.byref(b), int(bool(write_personal)),
                                                    _ptr(self.out), _ptr(scores), self._stream()))
        self._dirty = True
        self._catalog_ready = False                             # the catalog index follows Recipe_Embedding
        self._keep = [users, items, cats, labels, ws, ulab]    # alive until the next step is queued
        return (self.out, scores) if return_scores else self.out

    def train_step_host(self, mode, B, users, items, cats=None, labels=None, ws=None, ulab=None,
                        write_personal=False):
        """fr_train_step_host: host (ideally pinned) torch/numpy buffers; H2D + step +
        D2H of the scalars are queued on the current stream.  Returns the pinned
        host scalar tensor (valid after a stream sync)."""
        hp = lambda x: C.c_void_p(0) if x is None else C.c_void_p(x.data_ptr() if torch.is_tensor(x) else x.ctypes.data)
        b = L.fr_batch(mode, B, hp(users), hp(items), hp(cats), hp(labels), hp(ws), hp(ulab))
        L.check(self.handle, self.lib.fr_train_step_host(self.handle, C.byref(b), int(bool(write_personal)),
                                                         C.c_void_p(self.out_host.data_ptr()), self._stream()))
        self._dirty = True
        self._catalog_ready = False
        self._keep = [users, items, cats, labels, ws, ulab]
        return self.out_host

    def feed_prefetch(self, mode, B, users, items, cats=None, labels=None, ws=None, ulab=None):
        """fr_feed_prefetch: start the H2D copy of a FUTURE batch (same host buffers later passed to
        train_step_host) on the library's copy stream, overlapping the step in flight."""
        hp = lambda x: C.c_void_p(0) if x is None else C.c_void_p(x.data_ptr() if torch.is_tensor(x) else x.ctypes.data)
        b = L.fr_batch(mode, B, hp(users), hp(items), hp(cats), hp(labels), hp(ws), hp(ulab))
        L.check(self.handle, self.lib.fr_feed_prefetch(self.handle, C.byref(b)))
        self._keep_prefetch = [users, items, cats, labels, ws, ulab]

    def read_scalars(self):
        v = self.out.cpu().numpy()       # synchronises
        if v[L.FR_OUT_OVERFLOW] == 3:
            raise IndexError("train step: a user or recipe id of the batch lies outside its table (tf.gather would "
                             "raise); the offending rows were redirected to row 0, the step's results are invalid")
        if v[L.FR_OUT_OVERFLOW] == 2:
            raise L.FoodRecError("row-sharded step: a rank needed more distinct recipes from one owner than "
                                 "fr_shard.cap; raise ShardedEngine(cap=...)")
        if v[L.FR_OUT_OVERFLOW] != 0:
            raise L.FoodRecError(f"label feed has {int(v[L.FR_OUT_LABEL_ENTRIES])} non-zeros > "
                                 f"max_label_entries={self.max_label_entries}; General_Memory write truncated")
        return v

    def timing_enable(self, on=True):
        L.check(self.handle, self.lib.fr_timing_enable(self.handle, int(bool(on))))

    def timing_read(self, reset=True):
        """{phase: mean ms per step} from CUDA events recorded on the step's stream."""
        ms = (C.c_double * L.FR_T_COUNT)()
        n = C.c_int64()
        L.check(self.handle, self.lib.fr_timing_read(self.handle, ms, C.byref(n), int(bool(reset))))
        k = max(n.value, 1)
        return {name: ms[i] / k for i, name in enumerate(L.FR_T_NAMES)}, n.value

    def flush(self):
        """Lazy-exact Adam: bring every row to the current step before the tables are read."""
        if self._dirty and self.learner == L.FR_ADAM and self.adam_mode != L.FR_ADAM_DENSE:
            L.check(self.handle, self.lib.fr_adam_flush(self.handle, self._stream()))
        self._dirty = False

    def set_health_blend(self, on=True):
        """Score users as P[u] + alpha * mean G[labels(u)] at inference (score, eval_sampled_topk, catalog_topk)."""
        L.check(self.handle, self.lib.fr_set_health_blend(self.handle, int(bool(on))))

    def score(self, users, items, categories=None):
        self.flush()
        self._check_ids(users, self.U, "user_input"); self._check_ids(items, self.I, "item_input")
        u, it = self._i32(users), self._i32(items)
        cats = self._f32(categories, (u.numel(), 4))
        out = torch.empty(u.numel(), dtype=torch.float32, device=self.device)
        L.check(self.handle, self.lib.fr_fwd_score(self.handle, _ptr(u), _ptr(it), _ptr(cats), u.numel(), _ptr(out), self._stream()))
        self._keep = [u, it, cats]
        return out

    def eval_sampled_topk(self, users, cand, n_cand, K, cand_cats=None, return_scores=False):
        self.flush()
        self._check_ids(users, self.U, "test users"); self._check_ids(cand, self.I, "candidates")
        u = self._i32(users)
        n = u.numel()
        cand = torch.as_tensor(np.asarray(cand, np.int32)) if not torch.is_tensor(cand) else cand
        stride = cand.shape[1]
        cand_d = cand.to(self.device, torch.int32).contiguous()
        nc = self._i32(n_cand)
        cc = self._f32(cand_cats, (n, stride, 4))
        ids = torch.empty((n, K), dtype=torch.int32, device=self.device)
        rank = torch.empty(n, dtype=torch.int32, device=self.device)
        sc = torch.zeros((n, stride), dtype=torch.float32, device=self.device) if return_scores else None
        L.check(self.handle, self.lib.fr_eval_sampled_topk(self.handle, _ptr(u), _ptr(cand_d), _ptr(nc), n, stride,
                                                           _ptr(cc), K, _ptr(ids), _ptr(rank), _ptr(sc), self._stream()))
        self._keep = [u, cand_d, nc, cc]
        return (ids, rank, sc) if return_scores else (ids, rank)

    def set_item_cats(self, item_cats):
        """(Re)place the resident dish_to_category table [I,4] (compact feed, catalog scoring)."""
        ic = torch.as_tensor(np.asarray(item_cats, np.float32).reshape(-1, 4)).to(self.device).contiguous()
        torch.cuda.synchronize(self.device)          # kernels in flight may still read the old table
        self.item_cats = ic
        self._set_tables()
        self._catalog_ready = False

    # ------------------------------------------------------------------ full-catalog top-K
    def catalog_prepare(self, cta_group=0, max_pass_rows=0, splits=0, epi_sets=0, tile_n=0, a_split=0, item_cats=None):
        """Build the recipe-side index of the catalog kernel from the current R / item_cats
        (call again after training changed R).  ``item_cats`` [I,4]: the masks of THIS table's
        rows when the resident table is a global map (row-sharded engines).  Synchronises."""
        if item_cats is not None:
            self._catalog_cats = torch.as_tensor(np.asarray(item_cats, np.float32).reshape(-1, 4)).to(self.device).contiguous()
            assert self._catalog_cats.shape[0] == self.I
        elif self.item_cats is None:
            raise L.FoodRecError("catalog scoring needs the item_cats (dish_to_category) table")
        else:
            self._catalog_cats = None
        self.flush()
        o = L.fr_catalog_opts(int(cta_group), int(max_pass_rows), int(splits), int(epi_sets), int(tile_n), int(a_split))
        L.check(self.handle, self.lib.fr_catalog_prepare(self.handle, C.byref(o), _ptr(self._catalog_cats), self._stream()))
        self._catalog_ready = True

    def catalog_topk(self, users=None, K=100, P_rows=None, n_users=None, id_mul=1, id_add=0, return_scores=True,
                     exclude=None):
        """The K best recipes of the whole catalog per query user by (score desc, id asc):
        ``ids`` int32 [n,K] (-1 padded), ``scores`` float64 [n,K].  Query rows are
        ``P_rows`` [n,5,D] (device) if given, else ``users`` into Personal_Memory
        (None = the first ``n_users`` users).  ``exclude``: recipe ids each query row must not get
        back (e.g. its training positives), as ``(offsets, ids)`` or a list of per-row sequences
        (:func:`exclusion_csr`), in the output id space (``local row * id_mul + id_add``).
        Asynchronous on the current stream."""
        if not getattr(self, "_catalog_ready", False):
            self.catalog_prepare()
        self.flush()
        pr = u = None
        if P_rows is not None:
            pr = self._f32(P_rows, (-1, 5, self.D))
            n = pr.shape[0]
        elif users is not None:
            self._check_ids(users, self.U, "catalog_topk users")
            u = self._i32(users)
            n = u.numel()
        else:
            n = self.U if n_users is None else int(n_users)
        ids = torch.empty((n, K), dtype=torch.int32, device=self.device)
        sc = torch.empty((n, K), dtype=torch.float64, device=self.device) if return_scores else None
        if exclude is None:
            L.check(self.handle, self.lib.fr_catalog_topk(self.handle, _ptr(u), _ptr(pr), n, int(K), int(id_mul), int(id_add),
                                                          _ptr(ids), _ptr(sc), self._stream()))
            self._keep = [u, pr]
        else:
            off, xi = exclusion_csr(exclude, n)
            off = self._i32(off)
            xi = self._i32(xi) if xi.shape[0] else torch.zeros(1, dtype=torch.int32, device=self.device)   # never NULL
            L.check(self.handle, self.lib.fr_catalog_topk_excluding(self.handle, _ptr(u), _ptr(pr), n, int(K), _ptr(off), _ptr(xi),
                                                                    int(id_mul), int(id_add), _ptr(ids), _ptr(sc), self._stream()))
            self._keep = [u, pr, off, xi]
        return (ids, sc) if return_scores else ids

    def catalog_merge(self, ids, scores):
        """Merge per-shard lists [W,n,K] into the K best of their union."""
        ids = ids.to(self.device, torch.int32).contiguous(); scores = scores.to(self.device, torch.float64).contiguous()
        W, n, K = ids.shape
        oi = torch.empty((n, K), dtype=torch.int32, device=self.device)
        os_ = torch.empty((n, K), dtype=torch.float64, device=self.device)
        L.check(self.handle, self.lib.fr_catalog_merge(self.handle, _ptr(ids), _ptr(scores), W, n, K, _ptr(oi), _ptr(os_),
                                                       self._stream()))
        self._keep = [ids, scores]
        return oi, os_

    def catalog_timing_read(self, reset=True):
        ms = (C.c_double * 4)()
        n = C.c_int64()
        L.check(self.handle, self.lib.fr_catalog_timing_read(self.handle, ms, C.byref(n), int(bool(reset))))
        return dict(zip(("user_operand", "gemm_filter", "rerank", "exact_fallback"), list(ms))), n.value

    def catalog_cycle_counters(self):
        v = (C.c_uint64 * 8)()
        L.check(self.handle, self.lib.fr_catalog_cycle_counters(self.handle, v, self._stream()))
        v = list(v)
        out = {}
        if v[3]:
            out.update(mma_cycles=v[0] / v[3], mma_wait_accumulator=v[1] / v[3], mma_wait_operands=v[2] / v[3])
        if v[6]:
            out.update(epilogue_cycles=v[4] / v[6], epilogue_wait_accumulator=v[5] / v[6])
        return out

    def catalog_fallback_rows(self):
        v = C.c_int32()
        L.check(self.handle, self.lib.fr_catalog_fallback_rows(self.handle, C.byref(v), self._stream()))
        return v.value

    def catalog_info(self):
        v = (C.c_int32 * 8)()
        L.check(self.handle, self.lib.fr_catalog_info(self.handle, v))
        return dict(zip(("cta_group", "k_padded", "tiles", "present_masks", "recipes_with_category", "epi_sets",
                         "list_capacity", "fallback_blocks"), list(v)))

    # ------------------------------------------------------------------ 1:N negative sampling
    def sample_negatives(self, pos_items, n_neg, seed, sample_offset=0):
        """int32 [n, n_neg] device: counter-based (Philox4x32-10) uniform negatives != positive;
        the same ids oracle/sampler_oracle.sample_negatives draws for (seed, sample index)."""
        pos = self._i32(pos_items)
        out = torch.empty((pos.numel(), int(n_neg)), dtype=torch.int32, device=self.device)
        L.check(self.handle, self.lib.fr_sample_negatives(self.handle, _ptr(pos), pos.numel(), int(n_neg), int(seed) & (2**64 - 1),
                                                          int(sample_offset), _ptr(out), self._stream()))
        self._keep = [pos]
        return out

    def sample_bpr_batch(self, users, pos_items, n_neg, seed, sample_offset=0, num_items=0):
        """(users [n*n_neg], items [2*n*n_neg]) int32 device: the 1:n_neg BPR batch of n positives -- every (user,
        positive) repeated against n_neg sampled negatives (the draws of ``sample_negatives``), laid out as the step
        consumes it.  ``num_items``: catalog size to draw from (0 = this engine's; a row-sharded rank passes the global one)."""
        u, pos = self._i32(users), self._i32(pos_items)
        n = pos.numel()
        ou = torch.empty(n * int(n_neg), dtype=torch.int32, device=self.device)
        oi = torch.empty(2 * n * int(n_neg), dtype=torch.int32, device=self.device)
        L.check(self.handle, self.lib.fr_sample_bpr_batch(self.handle, _ptr(u), _ptr(pos), n, int(n_neg), int(seed) & (2**64 - 1),
                                                          int(sample_offset), int(num_items), _ptr(ou), _ptr(oi), self._stream()))
        self._keep = [u, pos]
        return ou, oi

    def train_step_sampled(self, users, pos_items, n_neg, seed, sample_offset=0, **kw):
        """One BPR step with n_neg sampled negatives per positive: the batch of B positives becomes
        B*n_neg triples (u, i+, i-_j) drawn on the device (resident side tables required)."""
        uu, items = self.sample_bpr_batch(users, pos_items, n_neg, seed, sample_offset)
        return self._step_dev(L.FR_BPR, uu.numel(), uu, items, None, None, None, None, **kw)

    def philox(self, ctr_key):
        ck = torch.as_tensor(np.ascontiguousarray(np.asarray(ctr_key, np.uint32)).view(np.int32)).to(self.device)
        n = ck.numel() // 6
        out = torch.empty(4 * n, dtype=torch.int32, device=self.device)
        L.check(self.handle, self.lib.fr_philox4x32_10(self.handle, _ptr(ck), n, _ptr(out), self._stream()))
        return out.cpu().numpy().view(np.uint32).reshape(n, 4)

    def sort_pairs(self, keys, nbits):
        k = torch.as_tensor(np.asarray(keys, np.int64).astype(np.uint32).view(np.int32)).to(self.device)
        ok = torch.empty_like(k); oi = torch.empty_like(k)
        L.check(self.handle, self.lib.fr_sort_pairs(self.handle, _ptr(k), k.numel(), nbits, _ptr(ok), _ptr(oi), self._stream()))
        return ok.cpu().numpy().view(np.uint32), oi.cpu().numpy().view(np.uint32)

    # ------------------------------------------------------------------ state
    def tables(self):
        """Host copies of the four tables at the current step (flushes lazy Adam)."""
        self.flush()
        return {k: getattr(self, k).detach().float().cpu().numpy() for k in ("P", "R", "Cat", "G")}

    def state_dict(self):
        self.flush()
        sd = {k: getattr(self, k).detach().float().cpu().numpy() for k in ("P", "R", "Cat", "G")}
        for name, d in (("s1", self.s1), ("s2", self.s2)):
            for k, v in d.items():
                sd[f"{name}_{k}"] = v.detach().cpu().numpy()
        sd["step"] = np.int64(self.step)
        return sd

    def load_state_dict(self, sd):
        for k in ("P", "R", "Cat", "G"):
            getattr(self, k).copy_(torch.as_tensor(sd[k]))
        for name, d in (("s1", self.s1), ("s2", self.s2)):
            for k, v in d.items():
                v.copy_(torch.as_tensor(sd[f"{name}_{k}"]))
        step = int(sd["step"])
        self.last_P.fill_(step); self.last_R.fill_(step)
        L.check(self.handle, self.lib.fr_set_step(self.handle, step))
        self._dirty = False
        self._catalog_ready = False      # the catalog index (bf16 operand, norms, filter bound) was built from the OLD R

    def tables_modified(self):
        """Call after writing P / R / Cat / G (the tensors this engine holds: ``adopt=True`` shares them with the
        caller) outside train_step / load_state_dict: derived state (the catalog index) is rebuilt on next use."""
        self._catalog_ready = False
