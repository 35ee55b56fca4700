"""Row-sharded training over W GPUs (one process per GPU, torch.distributed/NCCL for the
plumbing).  SURVEY 8(e): Personal_Memory (+ optimizer slots) is sharded by ``user % W`` and
every sample is routed to the GPU that owns its user when it is loaded, so the 5*D-float
user rows and their updates never move; Recipe_Embedding is sharded by ``recipe % W`` and
the looked-up rows / their gradient rows travel in fixed-capacity all-to-alls; loss,
sum|g|^2, dCat and dG travel in ONE packed all-reduce.  The reference has none of this
(single ``tf.Session``).

Two runners drive the five C-ABI phases (``fr_shard_*``):
  * :class:`DistRunner`   -- this process is one rank; collectives via torch.distributed.
  * :class:`LocalRunner`  -- all W ranks live in THIS process on one GPU and the collectives
    are tensor shuffles: the same kernels and protocol, used by the parity tests.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L
from .engine import Engine, Hyper, _ptr, exclusion_csr


# ---------------------------------------------------------------------------- host-side layout
def local_rows(n: int, world: int) -> int:
    return (n + world - 1) // world


def shard_rows(x: np.ndarray, rank: int, world: int) -> np.ndarray:
    """rows r, r+W, r+2W, ... (local row k <-> global row r + k*W), zero-padded to ceil(n/W)."""
    part = np.ascontiguousarray(x[rank::world])
    need = local_rows(x.shape[0], world)
    if part.shape[0] < need:
        part = np.concatenate([part, np.zeros((need - part.shape[0],) + x.shape[1:], x.dtype)])
    return part


def unshard_rows(parts, n: int) -> np.ndarray:
    world = len(parts)
    out = np.zeros((n,) + parts[0].shape[1:], parts[0].dtype)
    for r, p in enumerate(parts):
        cnt = len(range(r, n, world))
        out[r::world] = p[:cnt]
    return out


def route_batch(users: np.ndarray, world: int):
    """Index lists (stable, i.e. batch order) of the groups each rank owns: user % W."""
    users = np.asarray(users)
    return [np.nonzero(users % world == r)[0] for r in range(world)]


def shard_label_csr(off: np.ndarray, idx: np.ndarray, rank: int, world: int, n_users: int):
    """CSR over the rank's local user rows."""
    us = np.arange(rank, n_users, world)
    cnt = off[us + 1] - off[us]
    need = local_rows(n_users, world)
    loff = np.zeros(need + 1, np.int32)
    loff[1:len(us) + 1] = np.cumsum(cnt)
    loff[len(us) + 1:] = loff[len(us)]
    src = np.concatenate([np.arange(off[u], off[u + 1]) for u in us]) if len(us) < 20000 else \
        (np.repeat(off[us], cnt) + (np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)))
    return loff, idx[src].astype(np.int32)


# ---------------------------------------------------------------------------- one rank
class ShardedEngine:
    """The tables of one rank + the five phases of a sharded step."""

    def __init__(self, hyper: Hyper, P_loc, R_loc, Cat, G, rank, world, device="cuda:0", max_rows=1 << 16,
                 cap=None, adam_mode="lazy", item_cats_global=None, user_label_csr_local=None,
                 max_label_entries=None, adopt=False, single_pass=None, table_dtype="float32"):
        if not (1 <= world <= 8):
            raise ValueError("1 <= world <= 8")
        self.rank, self.world = rank, world
        self.e = Engine(hyper, P_loc, R_loc, Cat, G, device=device, max_rows=max_rows, adam_mode=adam_mode,
                        item_cats=item_cats_global, user_label_csr=user_label_csr_local,
                        max_label_entries=max_label_entries, adopt=adopt, single_pass=single_pass, table_dtype=table_dtype)
        e = self.e
        self.device = e.device
        self.I_global = None if item_cats_global is None else int(len(item_cats_global))
        if cap is None:
            # unique recipes per (source, owner).  A batch has at most max_rows distinct recipes,
            # spread over the owners by id % W: max_rows/W on average even when every row is
            # distinct; 10 % head-room + 256 for the imbalance.  Overflow is detected on device
            # (FR_OUT_OVERFLOW = 2) and raised by read_scalars(), never silent.
            cap = min(max_rows, e.I) if world == 1 else min(max_rows, e.I, int(1.1 * max_rows / world) + 256)
        self.cap = int(cap)
        n = world * self.cap
        dev = self.device
        # two plan slots (fr_shard_plan of step k+1 may overlap update / apply of step k): request buffers and batch
        # descriptors are per slot; slot of a step = its index & 1 (counters mirror the library's)
        self._req = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(2)]
        self._rreq = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(2)]
        self._n_plan = self._n_apply = 0
        self._slots = [None, None]
        self._pending = None
        self.rows = torch.empty((n, e.D), dtype=torch.float32, device=dev)
        self.rbuf = torch.empty((n, e.D), dtype=torch.float32, device=dev)
        self.grows = torch.empty((n, e.D), dtype=torch.float32, device=dev)
        self.rgrows = torch.empty((n, e.D), dtype=torch.float32, device=dev)
        self.packed = torch.zeros(int(e.lib.fr_shard_packed_len(e.handle)), dtype=torch.float32, device=dev)

    # the request buffers of the step being planned / the step being executed
    @property
    def req(self): return self._req[(self._n_plan - 1) & 1] if self._n_plan > self._n_apply else self._req[self._n_plan & 1]
    @property
    def rreq(self): return self._rreq[self._n_apply & 1]
    @property
    def _b(self): return self._slots[self._n_apply & 1][0]
    @property
    def _sh(self): return self._slots[self._n_apply & 1][1]
    def planned(self): return self._n_plan > self._n_apply

    def _shard(self, global_batch):
        return L.fr_shard(self.world, self.rank, self.cap, self.e.I, int(global_batch))

    def set_batch(self, users_local, items_global, labels=None, neg_items=None, categories=None, neg_categories=None,
                  write_sign=None, user_one_hot_label=None, global_batch=None):
        e = self.e
        u = e._i32(users_local)
        B = u.numel()
        bpr = neg_items is not None
        if bpr:
            it = torch.stack([e._i32(items_global), e._i32(neg_items)], 1).reshape(-1).contiguous()
            cats = None if categories is None else torch.stack(
                [e._f32(categories, (B, 4)), e._f32(neg_categories, (B, 4))], 1).reshape(-1, 4).contiguous()
        else:
            it = e._i32(items_global)
            cats = e._f32(categories, (B, 4))
        lab, ws = e._f32(labels, (-1,)), e._f32(write_sign, (-1,))
        ul = e._f32(user_one_hot_label, (B, e.Lb))
        self._pending = (L.fr_batch(L.FR_BPR if bpr else L.FR_POINTWISE, B, _ptr(u), _ptr(it), _ptr(cats), _ptr(lab), _ptr(ws), _ptr(ul)),
                         self._shard(global_batch if global_batch is not None else B), [u, it, cats, lab, ws, ul])

    def set_batch_dev(self, mode, B, users_local, items, labels=None, global_batch=None):
        """Device tensors already in the C-ABI layout (int32 users [B]; int32 items [S],
        BPR rows interleaved pos/neg): nothing is copied or reshaped."""
        self._pending = (L.fr_batch(mode, B, _ptr(users_local), _ptr(items), _ptr(None), _ptr(labels), _ptr(None), _ptr(None)),
                         self._shard(global_batch if global_batch is not None else B), [users_local, items, labels])

    def set_batch_sampled(self, users_local, pos_items_global, n_neg, seed, sample_offset=0, global_batch=None, num_items=None):
        """1:n_neg BPR batch drawn on the device (fr_sample_bpr_batch): n (user, positive) pairs of THIS rank's users ->
        n*n_neg triples, negatives uniform over the GLOBAL catalog.  ``sample_offset`` = the global index of this
        rank's first pair, so the draws do not depend on how the pairs are spread over the ranks."""
        ni = num_items if num_items is not None else self.I_global
        if ni is None:
            raise ValueError("set_batch_sampled needs the global recipe count (num_items= or item_cats_global)")
        uu, items = self.e.sample_bpr_batch(users_local, pos_items_global, n_neg, seed, sample_offset, num_items=ni)
        B = uu.numel()
        self.set_batch_dev(L.FR_BPR, B, uu, items, global_batch=global_batch if global_batch is not None else B)

    def set_batch_raw(self, batch, keep, global_batch):
        """An fr_batch built by the caller (device pointers) -- e.g. the reference's dense feed."""
        self._pending = (batch, self._shard(global_batch), keep)

    # un-routed batches ------------------------------------------------------------------
    def route(self, mode, users_global, items, labels=None, rcap=None):
        """fr_shard_route: bucket a batch that arrived on THIS rank (global user ids, any owner) by owner rank into
        one fixed-capacity block per destination.  Returns the send buffer [W, block] for ONE all-to-all."""
        e = self.e
        u = e._i32(users_global)
        B = u.numel()
        group = 2 if mode == L.FR_BPR else 1
        it = e._i32(items)
        assert it.numel() == B * group
        lab = e._f32(labels, (-1,)) if mode == L.FR_POINTWISE else None
        if rcap is None:
            rcap = max(getattr(self, "_rcap", 0), int(1.25 * B / self.world) + 256)
        b = L.fr_batch(mode, B, _ptr(u), _ptr(it), _ptr(None), _ptr(lab), _ptr(None), _ptr(None))
        blk = int(e.lib.fr_shard_route_block(C.byref(b), int(rcap)))
        if getattr(self, "_rcap", None) != rcap or getattr(self, "_rmode", None) != mode:
            self._rcap, self._rmode, self._rblk = rcap, mode, blk
            self._rsend = torch.empty((self.world, blk), dtype=torch.int32, device=self.device)
            self._rrecv = torch.empty_like(self._rsend)
            cap_out = e.max_rows // group
            # (two sets: the routed batch of step k+1 is written while step k may still read its own)
            self._rus = [torch.empty(cap_out, dtype=torch.int32, device=self.device) for _ in range(2)]
            self._ris = [torch.empty(cap_out * group, dtype=torch.int32, device=self.device) for _ in range(2)]
            self._rys = [torch.empty(cap_out, dtype=torch.float32, device=self.device) for _ in range(2)]
            self._rn = torch.zeros(1, dtype=torch.int32, device=self.device)
            self._rflag = torch.zeros(1, dtype=torch.float32, device=self.device)
        self._rflag.zero_()
        L.check(e.handle, e.lib.fr_shard_route(e.handle, C.byref(b), self.world, int(rcap), _ptr(self._rsend), _ptr(self._rflag), e._stream()))
        self._keep_route = [u, it, lab]
        return self._rsend

    def unroute(self, global_batch):
        """fr_shard_unroute on the received blocks (self._rrecv) + set_batch_dev with what arrived.  Reads the routed
        batch size on the host (one 8-byte device->host copy: the phases take the row count as a host integer)."""
        e = self.e
        mode = self._rmode
        group = 2 if mode == L.FR_BPR else 1
        k = self._n_plan & 1
        self._ru, self._ri, self._ry = self._rus[k], self._ris[k], self._rys[k]
        L.check(e.handle, e.lib.fr_shard_unroute(e.handle, mode, self.world, int(self._rcap), _ptr(self._rrecv), self._ru.numel(),
                                                 _ptr(self._ru), _ptr(self._ri), _ptr(self._ry), _ptr(self._rn), _ptr(self._rflag),
                                                 e._stream()))
        n, flag = (int(x) for x in torch.stack([self._rn.float().squeeze(0), self._rflag.squeeze(0)]).cpu())
        if flag:
            raise L.FoodRecError("routing: more groups for one destination than the block capacity (raise rcap) or more "
                                 "arrived than max_rows holds")
        self.set_batch_dev(mode, n, self._ru[:n], self._ri[:n * group], self._ry[:n] if mode == L.FR_POINTWISE else None,
                           global_batch=global_batch)
        return n

    # the five phases ------------------------------------------------------------------
    def plan(self):
        """fr_shard_plan of the batch last given to set_batch*.  May be called while the previous step's update / apply
        are still queued (on another stream): it writes only its own plan slot."""
        e = self.e
        if self._pending is None:
            raise L.FoodRecError("plan(): no batch was set")
        if self._n_plan - self._n_apply >= 2:
            raise L.FoodRecError("plan(): both plan slots are in use")
        slot = self._n_plan & 1
        b, sh, keep = self._pending
        L.check(e.handle, e.lib.fr_shard_plan(e.handle, C.byref(b), C.byref(sh), _ptr(self._req[slot]), e._stream()))
        self._slots[slot] = (b, sh, keep)
        self._pending = None
        self._n_plan += 1
        return self._req[slot]

    def set_peers(self, rbuf_ptrs, rgrows_ptrs):
        """fr_shard_set_peers: device pointers of every rank's rbuf / rgrows as mapped into THIS process (own
        buffers at index rank).  From then on serve() / update() store rows straight into the consumer's buffer
        over NVLink and the runner replaces the two row all-to-alls by barriers."""
        W = self.world
        assert len(rbuf_ptrs) == W and len(rgrows_ptrs) == W
        a = (C.c_void_p * W)(*[C.c_void_p(int(x)) for x in rbuf_ptrs])
        b = (C.c_void_p * W)(*[C.c_void_p(int(x)) for x in rgrows_ptrs])
        sh = self._shard(1)
        L.check(self.e.handle, self.e.lib.fr_shard_set_peers(self.e.handle, C.byref(sh), a, b))
        self.p2p = True

    def serve_prepare(self):
        """fr_shard_serve_prepare for the step planned last (its received requests must be in place): the owner-side
        sort of the request list, which serve / apply of that step then find done.  Like plan(), it may be queued on
        another stream while the previous step's update / apply are still running."""
        e = self.e
        slot = (self._n_plan - 1) & 1
        L.check(e.handle, e.lib.fr_shard_serve_prepare(e.handle, C.byref(self._slots[slot][1]), _ptr(self._rreq[slot]), e._stream()))

    def serve(self):
        e = self.e
        rows = None if getattr(self, "p2p", False) else self.rows
        L.check(e.handle, e.lib.fr_shard_serve(e.handle, C.byref(self._sh), _ptr(self.rreq), _ptr(rows), e._stream()))
        return self.rows

    def forward(self):
        e = self.e
        L.check(e.handle, e.lib.fr_shard_forward(e.handle, C.byref(self._b), C.byref(self._sh), _ptr(self.rbuf),
                                                 _ptr(self.packed), e._stream()))
        return self.packed

    def update(self, write_personal=False):
        e = self.e
        grows = None if getattr(self, "p2p", False) else self.grows
        L.check(e.handle, e.lib.fr_shard_update(e.handle, C.byref(self._b), C.byref(self._sh), int(bool(write_personal)),
                                                _ptr(self.rbuf), _ptr(self.packed), _ptr(grows), _ptr(e.out), e._stream()))
        return self.grows

    def apply(self):
        e = self.e
        L.check(e.handle, e.lib.fr_shard_apply(e.handle, C.byref(self._sh), _ptr(self.rreq), _ptr(self.rgrows), _ptr(e.out),
                                               e._stream()))
        self._n_apply += 1
        e._dirty = True
        e._catalog_ready = False
        return e.out


    # checkpoint (SURVEY 8f.2): one .npz per rank, the layout tf.train.Saver's single file would have had ------
    def save(self, path_prefix):
        """``<prefix>.rank<r>of<W>.npz``: this rank's rows of P / R (+ optimizer slots), the replicated Cat / G and
        the step.  Every rank writes its own file; rank 0's Cat / G are the ones restore() trusts."""
        sd = self.e.state_dict()
        sd["rank"], sd["world"] = np.int64(self.rank), np.int64(self.world)
        f = f"{path_prefix}.rank{self.rank}of{self.world}.npz"
        np.savez(f, **sd)
        return f

    def restore(self, path_prefix):
        sd = dict(np.load(f"{path_prefix}.rank{self.rank}of{self.world}.npz"))
        if int(sd.pop("world")) != self.world or int(sd.pop("rank")) != self.rank:
            raise ValueError("checkpoint was written for a different sharding")
        self.e.load_state_dict(sd)

    # full-catalog top-K, item-sharded (SURVEY 8e) -------------------------------------------
    def catalog_prepare(self, **opts):
        """Index of THIS rank's recipe shard (local row k = recipe rank + k*W; rows past the
        catalog end carry no category and are never returned)."""
        e = self.e
        cats = e.item_cats.cpu().numpy() if e.item_cats is not None else None
        if cats is None:
            raise L.FoodRecError("catalog scoring needs the global item_cats map")
        e.catalog_prepare(item_cats=shard_rows(cats, self.rank, self.world), **opts)

    def catalog_query_rows(self, users_local):
        """This rank's query users as dense [n,5,D] rows (what the all-gather moves)."""
        e = self.e
        e.flush()
        u = e._i32(users_local)
        rows = torch.empty((u.numel(), 5, e.D), dtype=torch.float32, device=e.device)
        L.check(e.handle, e.lib.fr_gather_user_rows(e.handle, _ptr(u), u.numel(), _ptr(rows), e._stream()))
        e._keep = [u]
        return rows

    def catalog_local(self, P_rows_all, K, exclude=None):
        """Top-K of THIS rank's recipe shard for every gathered query row, ids global.  ``exclude``: the
        gathered rows' lists of GLOBAL recipe ids; ids of other shards are ignored by the kernels."""
        if exclude is None:
            return self.e.catalog_topk(P_rows=P_rows_all, K=K, id_mul=self.world, id_add=self.rank)
        return self.e.catalog_topk(P_rows=P_rows_all, K=K, id_mul=self.world, id_add=self.rank, exclude=exclude)

    def catalog_merge(self, ids, scores):
        return self.e.catalog_merge(ids, scores)


# ---------------------------------------------------------------------------- runners
class DistRunner:
    """This process is rank `dist.get_rank()`; NCCL (or gloo on CPU tensors in tests)."""

    def __init__(self, engine: ShardedEngine):
        import torch.distributed as dist
        self.dist, self.eng = dist, engine
        assert dist.get_world_size() == engine.world and dist.get_rank() == engine.rank

    def enable_p2p(self):
        """Fuse the two row exchanges into the producing kernels: rbuf / rgrows are re-allocated as symmetric
        memory (torch.distributed._symmetric_memory: one CUDA IPC rendezvous over the group), every rank learns the
        peers' device pointers, and gather / gradient kernels store rows straight into the consumer's buffer over
        NVLink.  The all-to-alls become barriers.  Same results bit for bit (same rows in the same places)."""
        import torch.distributed._symmetric_memory as symm
        g = self.eng
        n = g.world * g.cap
        group = self.dist.group.WORLD
        bufs = []
        for name in ("rbuf", "rgrows"):
            t = symm.empty((n, g.e.D), dtype=torch.float32, device=g.device)
            hdl = symm.rendezvous(t, group.group_name)
            setattr(g, name, t)
            bufs.append(hdl)
        self._symm = bufs
        g.set_peers(list(bufs[0].buffer_ptrs), list(bufs[1].buffer_ptrs))
        self._sync = torch.zeros(1, device=g.device)
        self._symm_barrier = hasattr(bufs[0], "barrier") and os.environ.get("FOODREC_P2P_NCCL_BARRIER") is None

    def _barrier(self):
        # stream-ordered: when it completes every rank has finished the phase before it.  The symmetric-memory
        # handle offers a signal-pad barrier (a few microseconds, no NCCL launch); fall back to a 1-element all-reduce.
        if self._symm_barrier:
            self._symm[0].barrier(channel=0)
        else:
            self.dist.all_reduce(self._sync)

    def set_batch_unrouted(self, mode, users_global, items, labels=None, global_batch=None, rcap=None):
        """A batch whose groups were NOT loaded at their users' owners: bucket by owner, ONE all-to-all of the blocks,
        compact what arrives.  ``global_batch`` = groups summed over all ranks (the loss mean divides by it)."""
        g = self.eng
        send = g.route(mode, users_global, items, labels, rcap)
        self.dist.all_to_all_single(g._rrecv, send)
        return g.unroute(global_batch)

    def step(self, write_personal=False, phase_events=None, next_batch=None):
        """One training step.  ``phase_events`` (a list) receives (name, torch.cuda.Event) marks recorded on the
        step's stream before every phase and after the last one -- bench.py's per-phase timing; None: no overhead.

        ``next_batch`` (a callable that gives the NEXT step's batch to ``set_batch*``): its fr_shard_plan and the id
        all-to-all are issued on a side stream, so they execute under this step's kernels (they depend only on the
        batch ids; the library keeps two plan slots).  The next call to step() then starts at ``serve``."""
        d, g = self.dist, self.eng
        p2p = getattr(g, "p2p", False)
        cuda = torch.device(getattr(g, "device", "cpu")).type == "cuda"     # (the gloo wiring test drives CPU stubs)
        main = torch.cuda.current_stream(g.device) if cuda else None

        def mark(name):
            if phase_events is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record()
                phase_events.append((name, ev))

        if g.planned():                                  # planned one step ahead on the side stream
            mark("plan")
            if cuda:
                main.wait_stream(self._side)
            mark("ids_all_to_all")
        else:
            mark("plan"); req = g.plan()
            mark("ids_all_to_all"); d.all_to_all_single(g._rreq[g._n_apply & 1], req)          # requests -> owners
        mark("serve"); g.serve()                         # p2p: rows land in the requesters' rbuf from inside the kernel
        mark("rows_exchange")
        if p2p:
            self._barrier()
        else:
            d.all_to_all_single(g.rbuf, g.rows)          # recipe rows -> requesters (NVLink)
        mark("forward"); g.forward()
        mark("all_reduce"); d.all_reduce(g.packed)       # loss, sum|g|^2, dCat, dG
        mark("update"); g.update(write_personal)         # p2p: gradient rows land in the owners' rgrows
        mark("grads_exchange")
        if p2p:
            self._barrier()
        else:
            d.all_to_all_single(g.rgrows, g.grows)       # finished gradient rows -> owners
        mark("apply"); out = g.apply()
        mark("end")
        prev_end = getattr(self, "_step_end", None)
        if cuda:
            self._step_end = torch.cuda.Event(); self._step_end.record(main)
        # The next step's plan + id all-to-all, issued on the side stream once THIS step is fully queued (the host runs
        # ahead of the device, so they still execute under this step's kernels; a next_batch that has to wait for the
        # device -- an un-routed batch reads its routed size -- then blocks the host while the device is busy).
        if next_batch is not None and cuda:
            if getattr(self, "_side", None) is None:
                self._side = torch.cuda.Stream(device=g.device)
            # the slot plan(k+1) writes (and its rreq) were last read by step k-1, which ended before this step began
            if prev_end is not None:
                self._side.wait_event(prev_end)
            with torch.cuda.stream(self._side):
                next_batch()
                req = g.plan()
                d.all_to_all_single(g._rreq[(g._n_plan - 1) & 1], req)
                if hasattr(g, "serve_prepare"):
                    g.serve_prepare()                     # owner-side request sort: depends on the requests only
        elif next_batch is not None:
            next_batch()
            req = g.plan()
            d.all_to_all_single(g._rreq[(g._n_plan - 1) & 1], req)
            if hasattr(g, "serve_prepare"):
                g.serve_prepare()
        return out


    def catalog_topk(self, users_local, K=100, exclude=None):
        """Item-sharded full-catalog top-K for this rank's ``users_local`` (same count on every rank):
        all-gather of the query rows, local top-K per recipe shard, all-to-all of the (id, score)
        lists back to the user owners, exact merge.  Returns ids int32 [n,K], scores float64 [n,K].
        ``exclude``: per-user lists of global recipe ids to leave out (``Engine.catalog_topk``); they
        travel with the query rows (all-gather of the list lengths, then of the ids padded to the
        longest rank's total)."""
        d, g = self.dist, self.eng
        W = g.world
        rows = g.catalog_query_rows(users_local)
        n = rows.shape[0]
        allrows = torch.empty((W * n,) + tuple(rows.shape[1:]), dtype=rows.dtype, device=rows.device)
        d.all_gather_into_tensor(allrows, rows)
        if exclude is None:
            ids, sc = g.catalog_local(allrows, K)             # [W*n, K]: block s = users of rank s
        else:
            ids, sc = g.catalog_local(allrows, K, exclude=self._gather_exclusion(exclude, n, rows.device))
        rid, rsc = torch.empty_like(ids), torch.empty_like(sc)
        d.all_to_all_single(rid, ids)                         # block w <- rank w's list for MY users
        d.all_to_all_single(rsc, sc)
        return g.catalog_merge(rid.view(W, n, K), rsc.view(W, n, K))


    def _gather_exclusion(self, exclude, n, dev):
        """This rank's lists for its n query rows -> the CSR of all W*n gathered rows (rank order)."""
        d, W = self.dist, self.eng.world
        off, ids = (torch.as_tensor(x).to(dev) for x in exclusion_csr(exclude, n))
        lens = (off[1:] - off[:-1]).to(torch.int32).contiguous()
        all_lens = torch.empty(W * n, dtype=torch.int32, device=dev)
        d.all_gather_into_tensor(all_lens, lens)
        per_rank = all_lens.view(W, n).sum(1).cpu()
        m = max(int(per_rank.max()), 1)
        pad = torch.zeros(m, dtype=torch.int32, device=dev)
        pad[:ids.numel()] = ids
        all_ids = torch.empty(W * m, dtype=torch.int32, device=dev)
        d.all_gather_into_tensor(all_ids, pad)
        return concat_csr([all_lens[s * n:(s + 1) * n] for s in range(W)],
                          [all_ids[s * m:s * m + int(per_rank[s])] for s in range(W)])


def concat_csr(lens, ids):
    """CSR (offsets [sum n_s + 1], ids) of the row blocks s = (row lengths lens[s], ids[s]) stacked in order."""
    lens = torch.cat(lens).to(torch.int64)
    off = torch.zeros(lens.numel() + 1, dtype=torch.int32, device=lens.device)
    off[1:] = torch.cumsum(lens, 0).to(torch.int32)
    return off, torch.cat(ids).to(torch.int32)


class LocalRunner:
    """All W ranks in one process on one GPU: the collectives become tensor shuffles."""

    def __init__(self, engines):
        self.engs = list(engines)
        self.W = len(self.engs)
        assert all(g.world == self.W and g.rank == r for r, g in enumerate(self.engs))

    def _all_to_all(self, src_attr, dst_attr):
        W = self.W
        for r, g in enumerate(self.engs):
            dst = getattr(g, dst_attr).view(W, g.cap, -1)
            for s, gs in enumerate(self.engs):
                dst[s].copy_(getattr(gs, src_attr).view(W, gs.cap, -1)[r])

    def enable_p2p(self):
        """Same kernels and peer tables as DistRunner.enable_p2p; here every "peer" is another engine of this
        process, so the pointers are plain device pointers and the barriers are stream order."""
        rb = [g.rbuf.data_ptr() for g in self.engs]
        rg = [g.rgrows.data_ptr() for g in self.engs]
        for g in self.engs:
            g.set_peers(rb, rg)

    def set_batches_unrouted(self, mode, batches, global_batch, rcap=None):
        """batches[r] = (users_global, items, labels) as they arrived on rank r.  Same kernels as DistRunner."""
        sends = [g.route(mode, *b, rcap=rcap) for g, b in zip(self.engs, batches)]
        for r, g in enumerate(self.engs):
            for s_, gs in enumerate(self.engs):
                g._rrecv[s_].copy_(sends[s_][r])
        return [g.unroute(global_batch) for g in self.engs]

    def step(self, write_personal=False, plan_ahead=None):
        """``plan_ahead`` (a callable that sets the NEXT batch on every engine): the next step's plan + request exchange
        are issued after this step's forward, before its update -- the order DistRunner's side stream allows."""
        p2p = getattr(self.engs[0], "p2p", False)
        if not self.engs[0].planned():
            for g in self.engs: g.plan()
            self._exchange_requests()
        self._step_tail(write_personal, p2p, plan_ahead)
        return self._outs

    def _exchange_requests(self):
        W = self.W
        for r, g in enumerate(self.engs):
            dst = g._rreq[(g._n_plan - 1) & 1].view(W, g.cap)
            for s_, gs in enumerate(self.engs):
                dst[s_].copy_(gs._req[(gs._n_plan - 1) & 1].view(W, gs.cap)[r])

    def _step_tail(self, write_personal, p2p, plan_ahead):
        for g in self.engs: g.serve()
        if not p2p: self._all_to_all("rows", "rbuf")
        for g in self.engs: g.forward()
        total = torch.stack([g.packed for g in self.engs]).sum(0)       # rank order, like a ring on W=2
        for g in self.engs: g.packed.copy_(total)
        if plan_ahead is not None:
            plan_ahead()
            for g in self.engs: g.plan()
            self._exchange_requests()
            for g in self.engs: g.serve_prepare()
        for g in self.engs: g.update(write_personal)
        if not p2p: self._all_to_all("grows", "rgrows")
        self._outs = [g.apply() for g in self.engs]

    def catalog_topk(self, users_local_per_rank, K=100, exclude=None):
        """Same protocol as DistRunner.catalog_topk with the collectives as tensor shuffles.  ``exclude``:
        one entry per rank, that rank's per-user lists of global recipe ids (or None)."""
        W = self.W
        rows = [g.catalog_query_rows(u) for g, u in zip(self.engs, users_local_per_rank)]
        n = rows[0].shape[0]
        assert all(r.shape[0] == n for r in rows)
        allrows = torch.cat(rows, 0)
        if exclude is None:
            lists = [g.catalog_local(allrows, K) for g in self.engs]      # per recipe shard: [W*n, K]
        else:
            csr = [tuple(torch.as_tensor(x) for x in exclusion_csr(ex, n)) for ex in exclude]
            ex = concat_csr([off[1:] - off[:-1] for off, _ in csr], [ids for _, ids in csr])
            lists = [g.catalog_local(allrows, K, exclude=ex) for g in self.engs]
        out = []
        for r, g in enumerate(self.engs):
            ids = torch.stack([lists[w][0][r * n:(r + 1) * n] for w in range(W)])
            sc = torch.stack([lists[w][1][r * n:(r + 1) * n] for w in range(W)])
            out.append(g.catalog_merge(ids, sc))
        return out
