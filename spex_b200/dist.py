"""Row-partitioned propagation across the GPUs of one NVSwitch box (SURVEY §8e).

The reference has no distributed code; its only scale-out hook is the serial row folding
``A_split`` (/root/reference/LightGCN_SPEX/code/utility1/dataloader.py:167-177, model.py:84-89):
cut the adjacency into row blocks, multiply each block by the full table, concatenate.  This module
is that partition with one process per GPU: rank p owns the contiguous node range
[bounds[p], bounds[p+1]) (balanced by nnz), holds the CSR row block of those rows, and every layer

    1. assembles the full E^(k) [N, D] on every rank (the exchange),
    2. runs the local CSR SpMM over its rows, accumulating the layer mean in its own slice.

Three exchange modes:
  "nccl"  one all-gather of the [rows_p, D] slices per layer (torch.distributed over NCCL/NVLink);
  "push"  the SpMM epilogue itself stores every output row into all peers' next-layer tables with
          P2P stores over NVLink (spex_spmm_csr_f32_push): transfer overlaps the gather-bound
          math row by row; layers are separated by a stream-ordered 4-byte all-reduce (barrier).
          E^(0) has no producing kernel to fuse with and travels by NCCL all-gather (measured
          faster than P2P stores or copy engines, which stay selectable: e0_exchange).

  "mcast" the same fusion with ONE store per row to an NVSwitch multicast mapping of the tables
          (NVLS; torch symmetric memory provides the mapping): a row leaves the GPU once instead of
          P-1 times, which removes the NVLink egress bound of "push" (spex_spmm_csr_f32_mcast,
          spex_mcast_rows_f32 for E^(0)).

In the two fused modes the tables are a ring of THREE buffers: E^(0) of a call lives in slot a, layer k
reads slot a+k and writes slot a+k+1 (mod 3), the next call's E^(0) goes to slot a+K.  That slot is idle
while the LAST layer runs (which stores nothing over NVLink), so `propagate(E0, next_E0_local=...)`
publishes the next call's table DURING the last layer - from that layer's own epilogue (the warp that
finishes output row r also multicasts row r of the next table: spex_spmm_csr_f32_publish), or from a
small high-priority side-stream kernel (fuse_publish = False): the E^(0) exchange (5.4 ms + 2.5 ms of
skew at 8 GPUs in round 1, un-overlapped) disappears from the critical path, and the ring makes the "everybody is done reading the buffer" barrier of round 1
unnecessary (every slot's previous readers are separated from its next writer by a barrier that
already exists).

The local multiply is injectable (``local_spmm``) so the orchestration can be tested on CPU with the
oracle's SpMM under the gloo backend; the default is the CUDA kernel and there is no fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional, Sequence

import numpy as np
import torch
import torch.distributed as dist


def slice_bounds(bounds: Sequence[int], rank: int):
    return int(bounds[rank]), int(bounds[rank + 1])


class _CudaArray:
    """Expose a raw device allocation to torch through __cuda_array_interface__."""

    def __init__(self, ptr: int, shape, typestr="<f4"):
        self.__cuda_array_interface__ = {"data": (int(ptr), False), "shape": tuple(shape),
                                         "typestr": typestr, "version": 3, "strides": None}


class PartitionedPropagator:
    """K-layer propagation + layer mean over a row partition; returns this rank's rows of the mean."""

    def __init__(self, local_graph, bounds: Sequence[int], D: int, K: int, group=None,
                 mode: str = "nccl", local_spmm: Optional[Callable] = None, device=None):
        self.g = local_graph
        self.bounds = [int(b) for b in bounds]
        self.D, self.K = int(D), int(K)
        self.group = group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        if len(self.bounds) != self.world + 1:
            raise ValueError("bounds must have world_size + 1 entries")
        self.N = self.bounds[-1]
        self.r0, self.r1 = slice_bounds(self.bounds, self.rank)
        self.mode = mode
        self.local_spmm = local_spmm
        self.device = device if device is not None else getattr(local_graph, "device", torch.device("cpu"))
        self._X: List[torch.Tensor] = []
        self.n_tables = 3         # ring of table buffers (module docstring)
        self._peer_ptrs = None
        self._raw = []
        self._flag = None
        # push mode: how E^(0) travels: "nccl" (all-gather; NVLS multicast makes it the fastest on an
        # NVSwitch box: 6.2 ms for 3.84 GB at 8 GPUs), "push" (SM stores, 10.5 ms) or "copy" (copy
        # engines, 13.2 ms)
        self.e0_exchange = "nccl"
        self._copy_streams = []
        self.timing = None        # set to [] to collect per-phase CUDA-event pairs (bring-up)
        self._mc = None           # multicast pointers of the tables (mode "mcast")
        self._symm = []
        self._nnz_global = None   # nnz of the whole matrix (receptive_sets)
        self._slot = 0            # ring slot that holds / receives E^(0) of the next propagate()
        self._staged = None       # (key, event): E^(0) already published into slot self._slot
        self._side = None         # high-priority stream of the background publish
        self.bg_ctas = 148        # CTAs of the background publish kernel (it must not crowd out the SpMM)
        # publish the next table from the last layer's own epilogue instead of a side-stream kernel
        # (8 GPUs: layer 3 + background kernel 10.7 ms, against 8.2 ms for a layer that pushes its Y rows)
        self.fuse_publish = True
        if mode == "push":
            if local_spmm is not None:
                raise ValueError("push mode is CUDA-only")
            self._setup_push()
        elif mode == "mcast":
            if local_spmm is not None:
                raise ValueError("mcast mode is CUDA-only")
            self._setup_mcast()
            self.e0_exchange = "mcast"
        elif mode == "nccl":
            self._X = [torch.empty(self.N, self.D, dtype=torch.float32, device=self.device)
                       for _ in range(self.n_tables)]
        else:
            raise ValueError("mode must be 'nccl', 'push' or 'mcast'")

    # ---- push mode: IPC-mapped double-buffered tables --------------------------------------------
    def _setup_push(self):
        from ._capi import call

        nbytes = self.N * self.D * 4
        handles = []
        for _ in range(self.n_tables):
            p = C.c_void_p()
            h = C.create_string_buffer(64)
            call("spex_ipc_alloc", nbytes, C.byref(p), h)
            self._raw.append(p)
            handles.append(h.raw)
            self._X.append(torch.as_tensor(_CudaArray(p.value, (self.N, self.D)), device=self.device))
        gathered = [None] * self.world
        dist.all_gather_object(gathered, handles, group=self.group)
        self._peer_ptrs = []  # [buf][rank] raw pointers of every rank's table (own included)
        self._opened = []
        for b in range(self.n_tables):
            ptrs = []
            for r in range(self.world):
                if r == self.rank:  # our own table is just one more destination of the epilogue
                    ptrs.append(self._raw[b].value)
                    continue
                q = C.c_void_p()
                call("spex_ipc_open", gathered[r][b], C.byref(q))
                self._opened.append(q)
                ptrs.append(q.value)
            self._peer_ptrs.append((C.c_void_p * max(len(ptrs), 1))(*ptrs))
        self._flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        dist.barrier(group=self.group)

    # ---- mcast mode: symmetric-memory tables with an NVSwitch multicast mapping -------------------
    def _setup_mcast(self):
        import torch.distributed._symmetric_memory as symm

        group = self.group if self.group is not None else dist.group.WORLD
        self._mc = []
        for _ in range(self.n_tables):
            t = symm.empty(self.N * self.D, dtype=torch.float32, device=self.device)
            h = symm.rendezvous(t, group)
            if not h.multicast_ptr:
                raise RuntimeError("this box has no NVLS multicast support: use mode='push'")
            self._symm.append((t, h))
            self._X.append(t.view(self.N, self.D))
            self._mc.append(int(h.multicast_ptr))
        self._flag = torch.zeros(1, dtype=torch.int32, device=self.device)
        dist.barrier(group=self.group)

    def close(self):
        if self.mode == "mcast" and self._symm:
            torch.cuda.synchronize()
            dist.barrier(group=self.group)
            self._X, self._symm, self._mc = [], [], None
        if self.mode == "push" and self._raw:
            from ._capi import call

            torch.cuda.synchronize()
            dist.barrier(group=self.group)
            for q in self._opened:
                call("spex_ipc_close", q)
            self._X = []
            for p in self._raw:
                call("spex_ipc_free", p)
            self._raw = []

    # ---- exchange ---------------------------------------------------------------------------------
    def _all_gather_rows(self, X_full: torch.Tensor, local: torch.Tensor):
        if self.world == 1:
            X_full[self.r0: self.r1].copy_(local)
            return
        outs = [X_full[self.bounds[r]: self.bounds[r + 1]] for r in range(self.world)]
        if dist.get_backend(self.group) == "nccl":
            # uneven slices: NCCL issues one grouped broadcast per rank straight into the views
            dist.all_gather(outs, local.contiguous(), group=self.group)
        else:  # gloo (CPU tests): all_gather needs equal sizes, so broadcast slice by slice
            outs[self.rank].copy_(local)
            for r in range(self.world):
                dist.broadcast(outs[r], src=dist.get_global_rank(self.group, r) if self.group else r,
                               group=self.group)

    def _stream_barrier(self):
        if self.world > 1:
            dist.all_reduce(self._flag, group=self.group)

    # ---- one layer --------------------------------------------------------------------------------
    def _layer(self, X_full, Y_local, addend, Z_local, z_scale, push_buf=None, publish=None, subset=None,
               x_nonzero=None):
        if subset is not None or x_nonzero is not None:
            # restricted to a row list (receptive field of a mini-batch) and / or reading a table that is zero
            # outside the rows x_nonzero marks; same fused exchange
            from ._capi import call, ptr, stream_ptr

            rows, slots, segs = subset if subset is not None else (None, None, None)
            mc = C.c_void_p(self._mc[push_buf]) if (push_buf is not None and self.mode == "mcast") else None
            peers = self._peer_ptrs[push_buf] if (push_buf is not None and self.mode == "push") else None
            call("spex_spmm_csr_rows_exchange_f32", ptr(self.g.rowptr), ptr(self.g.col), ptr(self.g.val), ptr(X_full),
                 self.g.n_rows, self.D, ptr(rows), -1 if rows is None else rows.numel(), ptr(slots),
                 0 if slots is None else slots.numel(), ptr(segs), 0 if segs is None else segs.numel(),
                 ptr(x_nonzero), self.r0, mc, peers,
                 self.world if peers is not None else 0, ptr(addend), 1.0, ptr(Z_local), float(z_scale),
                 self.g.plan(self.D), stream_ptr())
            return
        if self.local_spmm is not None:
            acc = self.local_spmm(self.g, X_full)
            if Y_local is not None:
                Y_local.copy_(acc)
            Z_local.copy_((addend + acc) * z_scale)
            return
        from . import ops
        from ._capi import call, ptr, stream_ptr

        if publish is not None:   # last layer + the next call's E^(0) on its epilogue
            src, slot = publish
            mc = C.c_void_p(self._mc[slot]) if self.mode == "mcast" else None
            peers = None if self.mode == "mcast" else self._peer_ptrs[slot]
            call("spex_spmm_csr_f32_publish", ptr(self.g.rowptr), ptr(self.g.col), ptr(self.g.val), ptr(X_full),
                 self.g.n_rows, self.D, self.r0, ptr(addend), 1.0, ptr(Z_local), float(z_scale), ptr(src), mc,
                 peers, 0 if self.mode == "mcast" else self.world, self.g.plan(self.D), stream_ptr())
            return
        if push_buf is None:
            ops.spmm(self.g, X_full, Y=Y_local, addend=addend, addend_scale=1.0, Z=Z_local, z_scale=z_scale)
            return
        if self.mode == "mcast":   # fused SpMM + all-gather, one multicast store per row
            call("spex_spmm_csr_f32_mcast", ptr(self.g.rowptr), ptr(self.g.col), ptr(self.g.val), ptr(X_full),
                 self.g.n_rows, self.D, self.r0, C.c_void_p(self._mc[push_buf]),
                 ptr(addend), 1.0, ptr(Z_local), float(z_scale), self.g.plan(self.D), stream_ptr())
            return
        # fused SpMM + all-gather: rows go to every peer's (and our own) next-layer table
        call("spex_spmm_csr_f32_push", ptr(self.g.rowptr), ptr(self.g.col), ptr(self.g.val), ptr(X_full),
             self.g.n_rows, self.D, self.r0, self._peer_ptrs[push_buf], self.world,
             ptr(addend), 1.0, ptr(Z_local), float(z_scale), self.g.plan(self.D), stream_ptr())

    def _layer_adam(self, X_full, addend, z_scale, adam, slot):
        """Last layer of the backward propagation + dense Adam on the owned rows + publish of the updated
        rows into ring slot `slot` of every rank (spex_spmm_csr_f32_adam)."""
        from ._capi import call, ptr, stream_ptr

        mc = C.c_void_p(self._mc[slot]) if self.mode == "mcast" else None
        peers = None if self.mode == "mcast" else self._peer_ptrs[slot]
        call("spex_spmm_csr_f32_adam", ptr(self.g.rowptr), ptr(self.g.col), ptr(self.g.val), ptr(X_full),
             self.g.n_rows, self.D, self.r0, ptr(addend), 1.0, None, float(z_scale), ptr(adam["p"]), ptr(adam["m"]),
             ptr(adam["v"]), float(adam["lr"]), float(adam["beta1"]), float(adam["beta2"]), float(adam["eps"]),
             int(adam["step"]), mc, peers, 0 if self.mode == "mcast" else self.world, self.g.plan(self.D),
             stream_ptr())

    def _mark(self, name):
        if self.timing is not None:
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.timing.append((name, ev))

    def phase_ms(self):
        """[(phase, ms)] between consecutive marks of the last propagate() (timing enabled)."""
        torch.cuda.synchronize()
        t = self.timing or []
        return [(t[i + 1][0], t[i][1].elapsed_time(t[i + 1][1])) for i in range(len(t) - 1)]

    def _exchange_e0(self, E0_local, slot: int = 0, background: bool = False):
        """All-gather this rank's rows of E^(0) into ring slot `slot` of every rank.  No barrier is
        needed before it in the fused modes: the ring guarantees that the slot's last readers finished
        before a barrier every rank has already passed (module docstring)."""
        if self.mode == "mcast" and self.e0_exchange == "mcast":
            from ._capi import call, ptr, stream_ptr

            call("spex_mcast_rows_f32_ex", ptr(E0_local), E0_local.shape[0], self.D, self.r0,
                 C.c_void_p(self._mc[slot]), self.bg_ctas if background else 0, stream_ptr())
        elif self.mode == "push" and self.e0_exchange in ("push", "copy"):
            from ._capi import call, ptr, stream_ptr

            if self.e0_exchange == "push":   # SM stores: one read, P stores per element
                call("spex_push_rows_f32_ex", ptr(E0_local), E0_local.shape[0], self.D, self.r0,
                     self._peer_ptrs[slot], self.world, self.bg_ctas if background else 0, stream_ptr())
                return
            # copy engines: one cudaMemcpyAsync per peer on its own stream, peers visited in
            # rotated order so that the ranks do not all target the same GPU at the same time
            main = torch.cuda.current_stream()
            if not self._copy_streams:
                self._copy_streams = [torch.cuda.Stream() for _ in range(self.world - 1)]
            start = torch.cuda.Event()
            start.record(main)
            nbytes = E0_local.numel() * 4
            off = self.r0 * self.D * 4
            E0c = E0_local.contiguous()
            done = []
            for j, st in enumerate(self._copy_streams):
                peer = (self.rank + 1 + j) % self.world
                st.wait_event(start)
                call("spex_memcpy_peer_async", C.c_void_p(self._peer_ptrs[slot][peer] + off), ptr(E0c), nbytes,
                     C.c_void_p(st.cuda_stream))
                ev = torch.cuda.Event()
                ev.record(st)
                done.append(ev)
            self._X[slot][self.r0: self.r1].copy_(E0c)
            for ev in done:
                main.wait_event(ev)
        else:
            self._all_gather_rows(self._X[slot], E0_local)

    @staticmethod
    def _key(t: torch.Tensor):
        return (t.data_ptr(), t._version, tuple(t.shape))

    def can_prefetch(self) -> bool:
        """Can the next call's E^(0) be published during this call's last layer?  In the fused modes that
        needs one of our own exchange kernels (NCCL on a side stream would race the stream-ordered
        barriers on the same communicator); in "nccl" mode the publish is a plain all-gather issued
        before the last layer (same ring bookkeeping, no overlap)."""
        if self.mode == "nccl":
            return True
        return (self.mode == "mcast" and self.e0_exchange == "mcast") or \
               (self.mode == "push" and self.e0_exchange == "push")

    # ---- receptive field of a mini-batch (training forward) ------------------------------------------
    def _own(self, rows_global: torch.Tensor) -> torch.Tensor:
        m = (rows_global >= self.r0) & (rows_global < self.r1)
        return rows_global[m] - self.r0

    def _sum_over_ranks(self, x: int) -> int:
        t = torch.tensor([int(x)], dtype=torch.int64, device=self.device)
        if self.world > 1:
            dist.all_reduce(t, group=self.group)
        return int(t.item())

    def _all_gather_var(self, t: torch.Tensor) -> torch.Tensor:
        """Concatenation of every rank's 1-D int64 tensor (lengths differ)."""
        if self.world == 1:
            return t
        n = torch.tensor([t.numel()], dtype=torch.int64, device=self.device)
        sizes = [torch.zeros_like(n) for _ in range(self.world)]
        dist.all_gather(sizes, n, group=self.group)
        sizes = [int(x.item()) for x in sizes]
        pad = torch.zeros(max(max(sizes), 1), dtype=torch.int64, device=self.device)
        pad[: t.numel()] = t
        bufs = [torch.empty_like(pad) for _ in range(self.world)]
        dist.all_gather(bufs, pad, group=self.group)
        return torch.cat([b[:k] for b, k in zip(bufs, sizes)])

    def zero_slot(self, j: int):
        """Zero this rank's copy of the ring slot that layer j of the NEXT propagate() writes (a restricted layer
        stores only its rows; the rest of a gradient table must read as zero).  Call it before a collective that
        every rank passes before that propagate(): peers push into the slot only afterwards."""
        self._X[(self._slot + j) % self.n_tables].zero_()

    def receptive_sets(self, S: torch.Tensor):
        """ops.receptive_rows over the partition: R[k] (global row ids, identical on every rank) = the rows of
        E^(k) that the rows S of the layer mean depend on, or None = all rows.  Every rank expands the rows it
        owns through its own CSR block (the columns are global ids); the lists are all-gathered."""
        from . import ops

        K = self.K
        R = [None] * (K + 1)
        if (K < 1 or self.mode not in ("push", "mcast") or self.local_spmm is not None
                or self.D not in (32, 64, 128)):
            return R
        if self._nnz_global is None:
            self._nnz_global = self._sum_over_ranks(self.g.nnz)
        nnz = self._nnz_global
        d = self._sum_over_ranks(self.g.degree_sum(self._own(S)))
        if d > ops.SUBSET_MAX_EDGE_FRAC * nnz:
            return R
        R[K] = S
        cur = S
        for k in range(K - 1, 0, -1):
            if d > ops.EXPAND_MAX_EDGE_FRAC * nnz:
                break
            cand = torch.unique(torch.cat([S, self._all_gather_var(self.g.neighbors(self._own(cur)))]))
            d = self._sum_over_ranks(self.g.degree_sum(self._own(cand)))
            if d > ops.SUBSET_MAX_EDGE_FRAC * nnz:
                break
            R[k] = cur = cand
        return R

    def propagate(self, E0_local: torch.Tensor, out: torch.Tensor = None,
                  next_E0_local: torch.Tensor = None, next_ready=None, first_full: torch.Tensor = None,
                  adam: dict = None, row_sets=None, x_masks=None) -> torch.Tensor:
        """E0_local: this rank's rows [r0, r1) of the fused table.  Returns mean_k E^(k)[r0:r1]
        (written into `out` if given).  `next_E0_local`: this rank's rows of the table of the NEXT
        call, if the caller already has it (an inference / evaluation sweep over many tables, or
        the optimiser's output): it is published to all ranks while the last layer of this call runs
        (`next_ready`: CUDA event after which next_E0_local may be read, e.g. the end of its upload).
        `first_full` (fused modes): a full [N, D] table every rank has already assembled locally, whose rows
        [r0, r1) are E0_local - the first layer reads it instead of an exchange (the gradient table of the
        training step: zero but for the batch's rows, which every rank can compute).
        `adam` (fused modes): {p, m, v, lr, beta1, beta2, eps, step} - the result is not returned but consumed
        as the gradient of `p` by a dense Adam fused into the last layer's epilogue, and the updated rows of
        `p` are published as the next call's table (spex_spmm_csr_f32_adam).
        `row_sets` (fused modes; from receptive_sets(S)): layer k computes - and exchanges - only the rows
        row_sets[k] (None = all); only the rows S = row_sets[K] of the result are then valid.
        `x_masks` (fused modes): x_masks[k] = uint8 [N] marking the rows of layer k's INPUT table that may be
        non-zero (None = dense): gathers of the other rows are skipped (bit-identical, see spmm_rows)."""
        K = self.K
        if out is None:
            out = torch.empty_like(E0_local)
        if K == 0:
            out.copy_(E0_local)
            return out
        inv = 1.0 / (K + 1)
        if self.timing is not None:
            self.timing = []
        fused = self.mode in ("push", "mcast")
        nt = self.n_tables
        a = self._slot
        self._mark("start")
        staged, self._staged = self._staged, None
        if staged is not None and staged[1] is not None:
            torch.cuda.current_stream().wait_event(staged[1])   # the publish of the last call (even a stale one
                                                                # must be over before this slot is written again)
        if first_full is not None:
            if not fused:
                raise ValueError("first_full needs a fused exchange mode")
        elif staged is None or staged[0] != self._key(E0_local):
            self._exchange_e0(E0_local, slot=a)
        self._mark("e0_exchange")
        if fused and first_full is None:
            self._stream_barrier()  # E^(0) complete everywhere
        self._mark("barrier")
        Y = None
        for k in range(K):
            last = k == K - 1
            X_full = self._X[(a + k) % nt] if (k > 0 or first_full is None) else first_full
            addend = E0_local if k == 0 else out
            if last and adam is not None:
                if not fused:
                    raise ValueError("the fused Adam epilogue needs a fused exchange mode")
                self._layer_adam(X_full, addend, inv, adam, (a + K) % nt)
                self._mark(f"layer{k + 1}")
                done = torch.cuda.Event()
                done.record()
                self._staged = (self._key(adam["p"]), done)
                self._slot = (a + K) % nt
                return None
            publish = None
            if last and next_E0_local is not None and self.can_prefetch():
                if fused and self.fuse_publish and self.D in (32, 64, 128) and next_E0_local.is_contiguous():
                    # the next table rides on this layer's epilogue (spex_spmm_csr_f32_publish)
                    if next_ready is not None:
                        torch.cuda.current_stream().wait_event(next_ready)
                    publish = (next_E0_local, (a + K) % nt)
                else:
                    self._publish_next(next_E0_local, (a + K) % nt, next_ready)
            if fused:
                subset = None
                if row_sets is not None and row_sets[k + 1] is not None:
                    if publish is not None:
                        raise ValueError("row_sets cannot be combined with a published next table")
                    subset = self.g.row_subset(self._own(row_sets[k + 1]))
                xm = x_masks[k + 1] if x_masks is not None else None
                if xm is not None and publish is not None:
                    raise ValueError("x_masks cannot be combined with a published next table")
                self._layer(X_full, None, addend, out, inv if last else 1.0,
                            push_buf=None if last else (a + k + 1) % nt, publish=publish, subset=subset,
                            x_nonzero=xm)
                if publish is not None:
                    done = torch.cuda.Event()
                    done.record()
                    self._staged = (self._key(next_E0_local), done)
                self._mark(f"layer{k + 1}")
                if not last:
                    self._stream_barrier()
                    self._mark("barrier")
            else:
                if not last and Y is None:
                    Y = torch.empty_like(E0_local)
                self._layer(X_full, None if last else Y, addend, out, inv if last else 1.0)
                self._mark(f"layer{k + 1}")
                if not last:
                    self._all_gather_rows(self._X[(a + k + 1) % nt], Y)
                    self._mark("all_gather")
        self._slot = (a + K) % nt
        return out

    def _publish_next(self, next_E0_local, slot, next_ready=None):
        """Exchange of the next call's E^(0) into ring slot `slot`.  Fused modes: on the high-priority
        side stream; it starts once everything enqueued so far on the main stream (the barrier before
        the last layer) is done and runs next to the last layer, which stores nothing over NVLink."""
        if self.mode == "nccl":
            if next_ready is not None:
                torch.cuda.current_stream().wait_event(next_ready)
            self._all_gather_rows(self._X[slot], next_E0_local)
            self._staged = (self._key(next_E0_local), None)
            return
        main = torch.cuda.current_stream()
        if self._side is None:
            self._side = torch.cuda.Stream(priority=-1)
        ready = torch.cuda.Event()
        ready.record(main)
        self._side.wait_event(ready)
        if next_ready is not None:
            self._side.wait_event(next_ready)
        with torch.cuda.stream(self._side):
            self._exchange_e0(next_E0_local, slot=slot, background=True)
            done = torch.cuda.Event()
            done.record(self._side)
        self._staged = (self._key(next_E0_local), done)


# ---------------------------------------------------------------------------------------------------
# Row-partitioned TRAINING (SURVEY §8e rows 2-3): the step of main_rec.py:30-37 with the table, its
# gradient and the Adam moments split by owner rank.
#
#   forward   out_p  = propagate(W_p)                      (the exchange above; rows [r0, r1) of the mean)
#   batch     every rank holds the whole mini-batch (256 samples: replicated host-side sampling with a
#             shared seed, no communication).  The <= 2B rows of `out` the batch touches are assembled
#             on every rank: each rank fills the rows it owns into a compact [2B, D] buffer, zeros
#             elsewhere, one sum all-reduce (a single non-zero term per row: exact, order-free)
#   loss      BCE on the compact rows, replicated: bit-identical to the single-GPU loss
#   backward  dL/d(out) rows are scattered by the same deterministic segmented reduction, each rank
#             keeping only the rows it owns (row window), into its [rows_p, D] gradient slice;
#             dL/dW = (1/(K+1)) sum_k (A^T)^k dL/d(out) = propagate(dL/d(out)) because the normalised
#             adjacency is symmetric: the SAME partitioned propagation, exchange included, on gradients
#             (sum-of-powers instead of the single-GPU kernel's Horner form: <= 1e-6 relative, not
#             bit-equal).  Edge dropout (non-symmetric values) is not supported in this mode.
#   optimiser row-owned dense Adam (spex_adam_f32 on the local slice): no collective.
# With a fused exchange (push / mcast) the tail of the step is ONE kernel per rank: the last backward layer
# applies Adam to each owned row in its epilogue and stores the updated row into every rank's table
# (spex_spmm_csr_f32_adam), so the next forward starts without an E^(0) exchange; and the first backward
# layer reads a gradient table every rank assembles locally (all batch rows are known everywhere): of the
# four exchanges of round-partitioned step only the per-layer ones remain.
# ---------------------------------------------------------------------------------------------------
class _CudaTrainOps:
    """The CUDA entry points behind PartitionedTrainer (no fallback: CPU tensors are rejected)."""

    def gather_owned(self, local, rows, r0, r1):
        from ._capi import call, ptr, stream_ptr

        R = torch.empty(rows.numel(), local.shape[1], dtype=torch.float32, device=local.device)
        call("spex_gather_owned_rows_f32", ptr(local), ptr(rows), rows.numel(), local.shape[1], r0, r1, ptr(R),
             stream_ptr())
        return R

    def bce(self, Ru, Ri, labels):
        from ._capi import call, ptr, stream_ptr

        B, D = Ru.shape
        ar = torch.arange(B, device=Ru.device)
        gamma = torch.empty(B, dtype=torch.float32, device=Ru.device)
        dgamma = torch.empty_like(gamma)
        loss = torch.empty(1, dtype=torch.float32, device=Ru.device)
        call("spex_bce_fwd_f32", ptr(Ru), ptr(Ri), D, ptr(ar), ptr(ar), ptr(labels), B, ptr(gamma), ptr(loss),
             ptr(dgamma), stream_ptr())
        return loss, dgamma

    def scatter(self, dst_rows, src, coef, out_local, r0, r1):
        from . import ops
        from ._capi import call, ptr, stream_ptr

        B, D = src.shape
        ar = torch.arange(B, device=src.device)
        work, wb = ops._scatter_workspace(B, src.device)
        call("spex_scatter_rows_f32", ptr(dst_rows), ptr(ar), ptr(coef), None, 1.0, B, ptr(src), D, ptr(out_local),
             r0, r1, ptr(work), wb, stream_ptr())

    def clear_rows(self, table_local, rows_local):
        from ._capi import call, ptr, stream_ptr

        if rows_local.numel():
            call("spex_clear_rows_f32", ptr(table_local), ptr(rows_local), rows_local.numel(), table_local.shape[1],
                 stream_ptr())

    def adam(self, W, g, m, v, lr, b1, b2, eps, step):
        from . import ops

        ops.adam_step(W, g, m, v, lr, b1, b2, eps, step)


class _TorchTrainOps:
    """The same five operations in plain torch: used by the gloo CPU test of the orchestration (the
    oracle's arithmetic; never selected on a GPU)."""

    def gather_owned(self, local, rows, r0, r1):
        R = torch.zeros(rows.numel(), local.shape[1], dtype=local.dtype)
        own = (rows >= r0) & (rows < r1)
        R[own] = local[rows[own] - r0]
        return R

    def bce(self, Ru, Ri, labels):
        gamma = (Ru * Ri).sum(1)
        loss = torch.nn.functional.binary_cross_entropy_with_logits(gamma, labels).reshape(1)
        return loss, (torch.sigmoid(gamma) - labels) / labels.numel()

    def scatter(self, dst_rows, src, coef, out_local, r0, r1):
        own = (dst_rows >= r0) & (dst_rows < r1)
        out_local.index_add_(0, dst_rows[own] - r0, src[own] * coef[own, None])

    def clear_rows(self, table_local, rows_local):
        table_local[rows_local] = 0

    def adam(self, W, g, m, v, lr, b1, b2, eps, step):
        m.lerp_(g, 1 - b1)
        v.mul_(b2).addcmul_(g, g, value=1 - b2)
        denom = v.sqrt() / (1 - b2 ** step) ** 0.5 + eps
        W.addcdiv_(m, denom, value=-lr / (1 - b1 ** step))


class PartitionedTrainer:
    """main_rec.py:30-37 over a row partition: this rank owns rows [r0, r1) of the fused table `W_local`,
    of its gradient and of the Adam moments.  `prop` is the PartitionedPropagator of the same partition."""

    def __init__(self, prop: PartitionedPropagator, W_local: torch.Tensor, n_user_rows: int, lr: float = 1e-3,
                 betas=(0.9, 0.999), eps: float = 1e-8, train_ops=None, fused_tail: bool = True):
        self.prop = prop
        self.W = W_local
        self.nur = int(n_user_rows)
        self.lr, self.betas, self.eps = lr, betas, eps
        self.m = torch.zeros_like(W_local)
        self.v = torch.zeros_like(W_local)
        # fused path (push / mcast exchange on GPUs, K >= 1, D with a vector kernel): see step()
        self.fused = (train_ops is None and prop.mode in ("push", "mcast") and prop.K >= 1
                      and prop.D in (32, 64, 128) and fused_tail)
        if self.fused:
            self.G_full = torch.zeros(prop.N, W_local.shape[1], dtype=W_local.dtype, device=W_local.device)
            self.g = None
        else:
            self.g = torch.zeros_like(W_local)    # dL/d(out), zero except the batch's owned rows
        self.dW = torch.empty_like(W_local)
        self.out = torch.empty_like(W_local)
        self._dirty = None
        self.t = 0
        self.receptive_field = True
        self.receptive_backward = True
        self.ops = train_ops if train_ops is not None else _CudaTrainOps()

    def step(self, users: torch.Tensor, items: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        p, r0, r1 = self.prop, self.prop.r0, self.prop.r1
        B = users.numel()
        rows = torch.cat([users, items + self.nur]).to(torch.int64)
        # forward restricted to the batch's receptive field (fused modes; every computed row is bit-identical to
        # the full computer(), so loss, gradients and weights are unchanged): layer K on the batch's rows, layer
        # K-1 on their neighbours, ...; the backward mirrors it (below)
        sets = p.receptive_sets(torch.unique(rows)) if (self.receptive_field and self.fused) else None
        out = p.propagate(self.W, out=self.out, row_sets=sets)
        R = self.ops.gather_owned(out, rows, r0, r1)
        # backward mirror of the receptive field: H_j = g + A^T H_{j-1} is non-zero only on sets[K - j], so layer j
        # (j < K) computes and exchanges those rows into a zeroed table (zeroed here, before the all-reduce that
        # orders it ahead of every peer's stores)
        bsets = bmasks = None
        if sets is not None and self.fused and self.receptive_backward:
            from . import ops

            bsets = [None] * (p.K + 1)
            bmasks = [None] * (p.K + 1)
            x_rows = sets[p.K]                       # layer 1 reads the gradient table: non-zero on the batch rows
            for j in range(1, p.K):                  # (the last layer is the fused Adam kernel: dense)
                if x_rows is not None:
                    d = p._sum_over_ranks(p.g.degree_sum(p._own(x_rows)))
                    if d <= ops.SPARSE_INPUT_MAX_EDGE_FRAC * p._nnz_global:
                        bmasks[j] = ops.nonzero_mask(p.N, x_rows)
                if sets[p.K - j] is not None:
                    bsets[j] = sets[p.K - j]
                    p.zero_slot(j)
                    x_rows = sets[p.K - j]           # the next layer reads a zeroed table holding these rows
                else:
                    x_rows = None
        if p.world > 1:
            dist.all_reduce(R, group=p.group)
        Ru, Ri = R[:B], R[B:]
        loss, dgamma = self.ops.bce(Ru, Ri, labels.to(torch.float32))
        self.t += 1
        if self.fused:
            # Every rank holds all rows of the batch, so every rank can write ALL gradient rows into its own
            # full-size gradient table (zero elsewhere: zero-filled once, the touched rows cleared per step):
            # the first backward layer needs no exchange.  The last one applies Adam to the owned rows in its
            # epilogue and publishes the updated rows as the next forward's table (one kernel for
            # main_rec.py:35-37's backward tail, the optimiser and the next all-gather).
            if self._dirty is not None:
                self.ops.clear_rows(self.G_full, self._dirty)
            self.ops.scatter(rows[:B], Ri, dgamma, self.G_full, 0, 0)
            self.ops.scatter(rows[B:], Ru, dgamma, self.G_full, 0, 0)
            self._dirty = rows
            if bsets is not None and any(b is not None for b in bsets):
                self.dW.zero_()     # a restricted first layer writes g + A g on its rows only; the rest is 0
            p.propagate(self.G_full[r0:r1], out=self.dW, first_full=self.G_full, row_sets=bsets, x_masks=bmasks,
                        adam={"p": self.W, "m": self.m, "v": self.v, "lr": self.lr, "beta1": self.betas[0],
                              "beta2": self.betas[1], "eps": self.eps, "step": self.t})
            return loss
        if self._dirty is not None:
            self.ops.clear_rows(self.g, self._dirty)
        self.ops.scatter(rows[:B], Ri, dgamma, self.g, r0, r1)      # gU[users] = sum dgamma * I[items]
        self.ops.scatter(rows[B:], Ru, dgamma, self.g, r0, r1)      # gI[items] = sum dgamma * U[users]
        own = (rows >= r0) & (rows < r1)
        self._dirty = (rows[own] - r0).contiguous()
        dW = p.propagate(self.g, out=self.dW)                        # (1/(K+1)) sum_k A^k g
        self.ops.adam(self.W, dW, self.m, self.v, self.lr, self.betas[0], self.betas[1], self.eps, self.t)
        return loss

    def gather_table(self, local: torch.Tensor) -> torch.Tensor:
        """The full [N, D] table from the ranks' slices (evaluation: every rank ranks its own users
        against all items)."""
        full = torch.empty(self.prop.N, local.shape[1], dtype=local.dtype, device=local.device)
        self.prop._all_gather_rows(full, local)
        return full


# ---------------------------------------------------------------------------------------------------
# Evaluation sharded by user (SURVEY §8e row 4): no data-path communication, one all-reduce of sums.
# ---------------------------------------------------------------------------------------------------
def shard_range(n: int, rank: int, world: int):
    return (n * rank) // world, (n * (rank + 1)) // world


class ShardedEvaluator:
    """Full-ranking top-k + Recall/NDCG over a user shard per rank.  The propagated item table is
    replicated (5 M x 64 fp16 = 640 MB), every rank ranks users [lo, hi) of the list it is given with the
    tcgen05 scorer, metrics are summed over ranks with ONE all-reduce of three numbers."""

    def __init__(self, U_all, I_all, mask_rowptr=None, mask_col=None, k: int = 20, group=None, scorer: str = "f16"):
        from . import ops

        self.U, self.I = U_all, I_all
        self.mrp, self.mcol = mask_rowptr, mask_col
        self.k, self.group, self.scorer = int(k), group, scorer
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        if scorer == "f16" and not ops.f16_filter_is_selective(U_all, I_all, torch.arange(U_all.shape[0], device=I_all.device)):
            scorer = self.scorer = "fp32"      # near-equal scores: the exact scorer is the faster exact path
        self.ranker = ops.FullRanker(I_all, scorer)

    def rank_topk(self, users: torch.Tensor, block: int = 148 * 2 * 128 * 4):
        """(idx int32 [n_local, k], val fp32 [n_local, k], (lo, hi)) for this rank's shard of `users`."""
        lo, hi = shard_range(users.numel(), self.rank, self.world)
        mine = users[lo:hi].to(torch.int64).contiguous()
        idx, val = self.ranker.topk(self.U, mine, self.k, self.mrp, self.mcol, block)
        return idx, val, (lo, hi)

    def recall_ndcg(self, users: torch.Tensor, truth_rowptr, truth_col):
        """Mean Recall@k / NDCG@k over ALL of `users` (truth: CSR over the positions of `users`): local
        metrics on the host, one all-reduce of (sum recall, sum ndcg, count)."""
        from . import metrics

        idx, _, (lo, hi) = self.rank_topk(users)
        trp = np.asarray(truth_rowptr)
        rec, ndcg = metrics.fullrank_recall_ndcg(idx.cpu().numpy(), trp[lo: hi + 1] - trp[lo],
                                                 np.asarray(truth_col)[trp[lo]: trp[hi]], self.k)
        s = torch.tensor([float(rec.sum()), float(ndcg.sum()), float(hi - lo)], dtype=torch.float64,
                         device=self.I.device if dist.is_initialized() and dist.get_backend(self.group) == "nccl"
                         else "cpu")
        if self.world > 1:
            dist.all_reduce(s, group=self.group)
        n = max(float(s[2]), 1.0)
        return {"recall": float(s[0]) / n, "ndcg": float(s[1]) / n, "users": int(s[2])}
