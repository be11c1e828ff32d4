"""Row-partitioned iterated product (power method, BASELINE.json config 5) over torch.distributed.

One process per GPU.  The matrix is split into contiguous row ranges balanced by nnz with the
reference's greedy rule (partition.py <- reference src/csr_matrix.c:167-266); every rank keeps its
rows (global column ids) and a full-length replica of x.  One iteration is

    y_loc = A_loc x ;  s = sum_ranks |y_loc|^2 (1-double all-reduce) ;  x[rows_loc] = y_loc / sqrt(s)
    refresh of the replicas of x   <- the only data-path exchange

Two refresh strategies, same numerical result (the exchange only copies doubles):
  * "allgather": every rank receives every other rank's slice (the literal "NCCL allgather of x");
    slices differ by a few rows, so it is issued as one broadcast per owner;
  * "halo": a rank receives only the part of x its rows actually reference -- the contiguous column
    range [min col, max col] of its local matrix -- from the ranks that own it (for the 7-point
    Laplacian: one n^2 plane from each neighbour instead of the whole vector).

The exchange plan is pure host logic and backend agnostic (NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import torch
import torch.distributed as dist


@dataclass
class ExchangePlan:
    """Who owns which rows and who needs which columns."""
    parts: List[Tuple[int, int]]                 # owned row range of every rank
    needs: List[Tuple[int, int]]                 # referenced column range [lo, hi) of every rank
    rank: int
    sends: List[Tuple[int, int, int]] = field(default_factory=list)   # (peer, lo, hi) of MY rows to ship
    recvs: List[Tuple[int, int, int]] = field(default_factory=list)   # (peer, lo, hi) of THEIR rows I need

    @classmethod
    def build(cls, parts, needs, rank):
        plan = cls(list(parts), list(needs), rank)
        my_lo, my_hi = parts[rank]
        for peer, (p_lo, p_hi) in enumerate(parts):
            if peer == rank:
                continue
            lo, hi = max(my_lo, needs[peer][0]), min(my_hi, needs[peer][1])   # what the peer needs of mine
            if hi > lo:
                plan.sends.append((peer, lo, hi))
            lo, hi = max(p_lo, needs[rank][0]), min(p_hi, needs[rank][1])     # what I need of the peer's
            if hi > lo:
                plan.recvs.append((peer, lo, hi))
        return plan

    def halo_doubles_received(self) -> int:
        return sum(hi - lo for _, lo, hi in self.recvs)

    def allgather_doubles_received(self) -> int:
        return sum(e - s for r, (s, e) in enumerate(self.parts) if r != self.rank)


def exchange_allgather(x: torch.Tensor, plan: ExchangePlan, group=None) -> None:
    """Refresh every replica of x completely: slice p is broadcast by its owner p."""
    if len(plan.parts) == 1:
        return
    works = [dist.broadcast(x[s:e], src=dist.get_global_rank(group, p) if group is not None else p, group=group, async_op=True)
             for p, (s, e) in enumerate(plan.parts)]
    for w in works:
        w.wait()


def exchange_halo(x: torch.Tensor, plan: ExchangePlan, group=None) -> None:
    """Refresh only the referenced column range of every replica (point-to-point)."""
    ops = []
    for peer, lo, hi in plan.recvs:
        ops.append(dist.P2POp(dist.irecv, x[lo:hi], peer, group))
    for peer, lo, hi in plan.sends:
        ops.append(dist.P2POp(dist.isend, x[lo:hi], peer, group))
    if not ops:
        return
    for w in dist.batch_isend_irecv(ops):
        w.wait()


def gather_needs(local_need: Tuple[int, int], world: int, device, group=None) -> List[Tuple[int, int]]:
    t = torch.tensor(local_need, dtype=torch.int64, device=device)
    if world == 1:
        return [tuple(int(v) for v in t.tolist())]
    out = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(out, t, group=group)
    return [tuple(int(v) for v in o.tolist()) for o in out]


# ---- the padded rank-major layout of x behind the one-collective all-gather (host logic; the device twin of
# remap_columns_host is spmv_b200_csr_remap_columns) ---------------------------------------------------------------
def padded_layout(parts: List[Tuple[int, int]]) -> Tuple[List[int], int]:
    """(starts, stride): part p's entries live at [p*stride, p*stride + rows_p); stride = largest part rounded up to 32."""
    rows_max = max(e - s for s, e in parts)
    return [s for s, _ in parts] + [parts[-1][1]], (rows_max + 31) // 32 * 32


def remap_columns_host(cols, starts, stride):
    """Column c owned by part p (starts[p] <= c < starts[p+1]) -> p*stride + (c - starts[p])."""
    import numpy as np
    st = np.asarray(starts, dtype=np.int64)
    owner = np.searchsorted(st, np.asarray(cols, dtype=np.int64), side="right") - 1
    return (owner * stride + np.asarray(cols, dtype=np.int64) - st[owner]).astype(np.int32)


def unpad(xg: torch.Tensor, parts: List[Tuple[int, int]], stride: int) -> torch.Tensor:
    return torch.cat([xg[p * stride: p * stride + (e - s)] for p, (s, e) in enumerate(parts)])


class _CudaView:
    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": typestr, "data": (ptr, False), "version": 2}


class PowerIteration:
    """Power method on a synthetic matrix, row-partitioned over the ranks of ``group``."""

    def __init__(self, kind, p0, p1=0, p2=0, seed=0x5EED, exchange="halo", group=None, parts=None, single=False,
                 hack_aligned=False):
        import ctypes as C

        from . import _native as N
        from . import device, partition, synth
        self.dev = device
        self.group = group
        distributed = dist.is_initialized() and not single  # single=True: the whole matrix on this rank alone
        self.world = dist.get_world_size(group) if distributed else 1
        self.rank = dist.get_rank(group) if distributed else 0
        self.exchange = exchange
        self.parts = parts if parts is not None else partition.synth_partition(kind, p0, p1, p2, self.world)
        if hack_aligned:   # HLL work is cut on 32-row block boundaries (reference src/hll_matrix.c:471-498)
            self.parts = partition.hack_aligned(self.parts, self.parts[-1][1])
        if len(self.parts) != self.world:
            raise ValueError(f"the nnz-balanced partition produced {len(self.parts)} parts for {self.world} ranks")
        self.row_begin, self.row_end = self.parts[self.rank]
        self.A = device.DeviceCSR.synth(kind, p0, p1, p2, seed=seed, row_begin=self.row_begin, row_end=self.row_end)
        info = self.A.info()
        self.N, self.rows, self.nnz_local = info.N, info.M, info.nnz
        self.nnz_global = synth.row_offset(kind, p0, p1, p2, self.parts[-1][1])
        self.algorithmic_bytes_local = info.algorithmic_bytes
        cu = torch.device("cuda", torch.cuda.current_device())
        # referenced column range of the local rows
        ptrs = [C.c_void_p() for _ in range(3)]
        N.check(N.lib().spmv_b200_csr_device_arrays(self.A._h, *[C.byref(p) for p in ptrs]))
        if info.nnz:
            cols = torch.as_tensor(_CudaView(ptrs[1].value, info.nnz, "<i4"), device=cu)
            lo, hi = torch.aminmax(cols)
            need = (int(lo.item()), int(hi.item()) + 1)
        else:
            need = (self.row_begin, self.row_begin)
        self.plan = ExchangePlan.build(self.parts, gather_needs(need, self.world, cu, group), self.rank)
        # algorithmic bytes of the LOCAL product: the rank streams its rows and reads only the referenced part of x
        self.algorithmic_bytes_local = 12 * info.nnz + 4 * (info.M + 1) + 8 * info.M + 8 * (need[1] - need[0])
        self.x = torch.ones(self.N, dtype=torch.float64, device=cu)
        self.y = torch.zeros(max(self.rows, 1), dtype=torch.float64, device=cu)
        self.ws = torch.empty(device.vec_ws_doubles(), dtype=torch.float64, device=cu)
        self.ss = torch.zeros(1, dtype=torch.float64, device=cu)
        self.launches_per_step = 4 + (2 if info.num_long_rows else 0)

    def reset(self, value=1.0):
        self.dev.vec_fill(self.x, value)

    def step(self):
        """One iteration; everything is enqueued on the current stream, nothing synchronises the host."""
        d = self.dev
        self.A.spmv(self.x, self.y)
        d.vec_sumsq(self.y, self.ws, self.ss, n=self.rows)
        if self.world > 1:
            dist.all_reduce(self.ss, group=self.group)
        d.vec_scale_by_inv_norm(self.x[self.row_begin:self.row_end], self.y, self.ss, n=self.rows)
        if self.world > 1:
            if self.exchange == "allgather":
                exchange_allgather(self.x, self.plan, self.group)
            else:
                exchange_halo(self.x, self.plan, self.group)

    def eigenvalue_estimate(self) -> float:
        return float(self.ss.item()) ** 0.5


class FusedPowerIteration(PowerIteration):
    """The same iteration with everything but an 8-byte all-reduce folded into the product kernel.

    Lazy normalisation: the stored vector is w_k = A v_{k-1} (not normalised); the next launch computes
    w_{k+1} = (A w_k) / |w_k| in its epilogue (algebraically A v_k), together with the per-CTA partial sums of
    |w_{k+1}|^2.  So there is no separate norm pass and no scale pass, and y IS the next x: the kernel writes
    the owned slice of the next x in place.
    peer_stores=True (needs NVLink peer access, one process per GPU on one node): the kernel also stores the
    rows a neighbour references straight into that neighbour's next-x buffer (cudaIpc-mapped peer memory), so
    the refresh of x costs no extra launch and no extra pass; the all-reduce of |w|^2 is the only collective
    and doubles as the barrier that orders those peer stores before the next product.
    peer_stores=False: the boundary rows travel with NCCL point-to-point messages instead.
    mailbox=True (implies peer stores): the all-reduce goes too.  The last CTA of every launch writes the rank's
    |w|^2 and an iteration tag into a mailbox slot of every rank (NVLink peer stores, release at system scope); the
    next launch starts by waiting for the tags of all ranks in its own mailbox, which also proves that the boundary
    rows have landed, and adds the sums in rank order (identical on every rank).  ONE launch per iteration, no
    collective library call in the loop (include/spmv_b200.h: spmv_b200_csr_spmv_fused_mail)."""

    def __init__(self, kind, p0, p1=0, p2=0, seed=0x5EED, group=None, parts=None, single=False, peer_stores=True,
                 mailbox=False, fmt="csr", hack_aligned=None, split=False):
        """split=True (implies mailbox): TWO launches per iteration -- the FLAT fused product, which never waits (grid as
        large as the matrix, the block scheduler balances the SMs), and a one-CTA exchange kernel that adds the partials,
        publishes |w|^2 + tag into every rank's mailbox and waits for all ranks (spmv_b200_*_spmv_fused_flat +
        spmv_b200_mail_exchange).  Same mailboxes, same numerics as mailbox=True.
        fmt="hll": the same iteration on the column-major HLL image (hll_row_fused_kernel); the row ranges are then cut
        on 32-row hack boundaries as the reference cuts HLL work.  hack_aligned=True with fmt="csr" gives the CSR iteration
        on exactly that partition (its results are bitwise those of the HLL iteration)."""
        if hack_aligned is None:
            hack_aligned = fmt == "hll"
        super().__init__(kind, p0, p1, p2, seed=seed, exchange="halo", group=group, parts=parts, single=single,
                         hack_aligned=hack_aligned)
        from . import _native as N
        d = self.dev
        self.A.set_image(0)   # the fused products never read the private image
        if self.A.info().num_long_rows:
            raise ValueError("FusedPowerIteration needs a matrix without long rows")
        self.fmt = fmt
        self.csr = self.A
        if fmt == "hll":
            if self.row_begin % 32:
                raise ValueError("the HLL iteration needs row ranges that start on a hack boundary")
            self.H = self.csr.to_hll()
            hi = self.H.info()
            self.algorithmic_bytes_local += 12 * hi.slots + 8 * (hi.num_hacks + 1) - 12 * self.nnz_local - 4 * (self.rows + 1)
            self.csr.close()          # only the HLL image stays resident
            self.csr = None
            self.A = self.H           # same fused entry points (DeviceHLL.spmv_fused / spmv_fused_mail / partials_count)
        elif fmt != "csr":
            raise ValueError(f"unknown format {fmt!r}")
        self.split = bool(split)
        self.mailbox = bool(mailbox) or self.split
        self.peer_stores = (bool(peer_stores) or self.mailbox) and self.world > 1
        cu = self.x.device
        del self.x, self.y
        nbytes = 8 * self.N
        if self.peer_stores:
            self.buf = [d.PeerBuffer(nbytes), d.PeerBuffer(nbytes)]
            self.xs = [b.as_tensor() for b in self.buf]
            handles = [None] * self.world
            dist.all_gather_object(handles, [b.handle_bytes() for b in self.buf], group=self.group)
            self.peers = []
            for parity in (0, 1):
                ps = N.Peers()
                ps.count = len(self.plan.sends)
                assert ps.count <= 7
                for i, (peer, lo, hi) in enumerate(self.plan.sends):
                    base = self.buf[parity].open_peer(handles[peer][parity])
                    ps.dst[i] = base + 8 * self.row_begin      # the peer's slot for MY local row 0
                    ps.lo[i], ps.hi[i] = lo - self.row_begin, hi - self.row_begin
                self.peers.append(ps)
        else:
            self.buf = None
            self.xs = [torch.empty(self.N, dtype=torch.float64, device=cu) for _ in range(2)]
            self.peers = [None, None]
        self.partials = torch.zeros(self.A.flat_partials_count() if self.split else self.A.partials_count(),
                                    dtype=torch.float64, device=cu)
        self.sumsq = [torch.zeros(1, dtype=torch.float64, device=cu) for _ in range(2)]
        self.scale = torch.ones(2, dtype=torch.float64, device=cu)   # split form: {|w|^2, 1/|w|} written by the exchange kernel
        self.k = 0
        self.box = None
        if self.mailbox:
            self.box = d.PeerBuffer(N.MAILBOX_BYTES)
            self.box_t = self.box.as_tensor("<i8", 8)
            self.box_t.zero_()
            self.sync = torch.zeros(2, dtype=torch.int32, device=cu)   # [0] CTA counter, [1] status
            self.mail = N.Mail()
            self.mail.world, self.mail.rank = self.world, self.rank
            self.mail.counter = self.sync.data_ptr()
            self.mail.status = self.sync.data_ptr() + 4
            if self.world > 1:
                handles = [None] * self.world
                dist.all_gather_object(handles, self.box.handle_bytes(), group=self.group)
                for r in range(self.world):
                    self.mail.box[r] = self.box.ptr.value if r == self.rank else self.box.open_peer(handles[r])
            else:
                self.mail.box[0] = self.box.ptr.value
        self.reset(1.0)
        self.launches_per_step = 2 if (self.split or not self.mailbox) else 1
        if self.world > 1:
            dist.barrier(group=self.group)

    def reset(self, value=1.0):
        for t in self.xs:
            self.dev.vec_fill(t, value)
        self.k = 0
        if self.box is not None:
            torch.cuda.synchronize()
            if self.world > 1:
                dist.barrier(group=self.group)   # nobody may still be writing tags of the previous run
            self.box_t.zero_()
            self.sync.zero_()
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)

    def step(self):
        cur, nxt = self.k & 1, (self.k & 1) ^ 1
        x, y = self.xs[cur], self.xs[nxt]
        if self.split:
            self.A.spmv_fused_flat(x.data_ptr(), y.data_ptr() + 8 * self.row_begin,
                                   inv_norm=self.scale.data_ptr() + 8 if self.k > 0 else None, partials=self.partials,
                                   peers=self.peers[nxt])
            self.mail.iteration = self.k
            self.dev.mail_exchange(self.partials, self.partials.numel(), self.mail, self.scale)
            self.k += 1
            return
        if self.mailbox:
            self.mail.iteration = self.k
            self.A.spmv_fused_mail(x.data_ptr(), y.data_ptr() + 8 * self.row_begin, self.partials, self.mail,
                                   peers=self.peers[nxt])
            self.k += 1
            return
        self.A.spmv_fused(x.data_ptr(), y.data_ptr() + 8 * self.row_begin,
                          prev_sumsq=self.sumsq[cur] if self.k > 0 else None, partials=self.partials,
                          peers=self.peers[nxt])
        self.dev.vec_sum(self.partials, self.partials.numel(), self.sumsq[nxt])
        if self.world > 1:
            dist.all_reduce(self.sumsq[nxt], group=self.group)  # |w|^2; also orders the peer stores
            if not self.peer_stores:
                exchange_halo(y, self.plan, self.group)
        self.k += 1

    def _mail_total(self) -> float:
        """|w_k|^2 as the next launch will see it: the slots of parity (k-1)&1 of MY mailbox, added in rank order."""
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)   # every rank's last launch has finished, so every tag has landed
        if int(self.sync[1].item()) != 0:
            raise RuntimeError("a mailbox wait timed out: a peer rank did not finish its launch")
        first = 2 * ((self.k - 1) & 1) * self.world
        slots = self.box_t[first: first + 2 * self.world].view(self.world, 2)
        tags = slots[:, 1].tolist()
        if any(t != self.k for t in tags):
            raise RuntimeError(f"mailbox tags {tags} do not match iteration {self.k}")
        total = 0.0
        for v in slots[:, 0].contiguous().view(torch.float64).tolist():
            total += v
        return total

    def eigenvalue_estimate(self) -> float:
        if self.split:
            torch.cuda.synchronize()
            if int(self.sync[1].item()) != 0:
                raise RuntimeError("a mailbox wait timed out: a peer rank did not finish its launch")
            return float(self.scale[0].item()) ** 0.5
        if self.mailbox:
            return self._mail_total() ** 0.5
        return float(self.sumsq[self.k & 1].item()) ** 0.5

    def normalized_x(self) -> torch.Tensor:
        """v_k = w_k / |w_k| (valid on the owned rows and on the referenced halo)."""
        if self.split:
            return self.xs[self.k & 1] / (self.eigenvalue_estimate())
        if self.mailbox:
            return self.xs[self.k & 1] / (self._mail_total() ** 0.5)
        return self.xs[self.k & 1] / self.sumsq[self.k & 1].sqrt()

    def close(self):
        if self.buf:
            torch.cuda.synchronize()
            if self.world > 1:
                dist.barrier(group=self.group)
            self.xs = []
            for b in self.buf:
                b.close()
            self.buf = None
        if self.box is not None:
            torch.cuda.synchronize()
            if self.world > 1:
                dist.barrier(group=self.group)
            self.box_t = None
            self.box.close()
            self.box = None


class AsyncPowerIteration(PowerIteration):
    """The fused iteration without any per-iteration rendezvous (include/spmv_b200.h: spmv_b200_csr_spmv_fused_async).

    x lives in a ring of three peer-mappable buffers; a launch computes the rows its neighbours reference first and
    raises a halo tag in their mailboxes as soon as those rows are stored; the scale factor lags one launch
    (launch k multiplies by 1/sqrt(S[k-2]), S[j] = |output of launch j|^2 over all ranks), so a launch only ever waits
    for things that finished a whole launch ago.  The iterate keeps the direction of the power method and stays bounded:
        lambda_K = sqrt(S[K-1] * S[K-3] / S[K-2]),   v_K = x_K / sqrt(S[K-1])        (K >= 3 launches)
    One launch per iteration, no collective call, no rank-to-rank wait on the critical path."""

    def __init__(self, kind, p0, p1=0, p2=0, seed=0x5EED, group=None, parts=None, single=False):
        super().__init__(kind, p0, p1, p2, seed=seed, exchange="halo", group=group, parts=parts, single=single)
        from . import _native as N
        d = self.dev
        self.A.set_image(0)   # the fused products never read the private image
        cu = self.x.device
        del self.x, self.y
        nbytes = 8 * self.N
        self.buf = [d.PeerBuffer(nbytes) for _ in range(3)]
        self.xs = [b.as_tensor() for b in self.buf]
        self.box = d.PeerBuffer(N.ASYNC_MAILBOX_BYTES)
        self.box_t = self.box.as_tensor("<i8", 8)
        self.sync = torch.zeros(4, dtype=torch.int32, device=cu)   # [0] CTA counter, [1] boundary counter, [2] status
        self.ex = N.Async()
        self.ex.world, self.ex.rank = self.world, self.rank
        self.ex.counter = self.sync.data_ptr()
        self.ex.bcounter = self.sync.data_ptr() + 4
        self.ex.status = self.sync.data_ptr() + 8
        senders = sorted({peer for peer, _, _ in self.plan.recvs})
        self.ex.num_recv = len(senders)
        for i, peer in enumerate(senders):
            self.ex.recv_from[i] = peer
        self.peers = [N.Peers() for _ in range(3)]
        if self.world > 1:
            handles = [None] * self.world
            dist.all_gather_object(handles, ([b.handle_bytes() for b in self.buf], self.box.handle_bytes()), group=self.group)
            for r in range(self.world):
                self.ex.box[r] = self.box.ptr.value if r == self.rank else self.box.open_peer(handles[r][1])
            assert len(self.plan.sends) <= 7
            for slot in range(3):
                ps = self.peers[slot]
                ps.count = len(self.plan.sends)
                for i, (peer, lo, hi) in enumerate(self.plan.sends):
                    base = self.buf[slot].open_peer(handles[peer][0][slot])
                    ps.dst[i] = base + 8 * self.row_begin
                    ps.lo[i], ps.hi[i] = lo - self.row_begin, hi - self.row_begin
                    self.ex.send_to[i] = peer
        else:
            self.ex.box[0] = self.box.ptr.value
        self.partials = torch.zeros(self.A.partials_count(), dtype=torch.float64, device=cu)
        self.k = 0
        self.launches_per_step = 1
        self.reset(1.0)

    def reset(self, value=1.0):
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)   # nobody may still be writing tags or rows of the previous run
        for t in self.xs:
            self.dev.vec_fill(t, value)
        self.box_t.zero_()
        self.sync.zero_()
        self.k = 0
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)

    def step(self):
        cur, nxt = self.k % 3, (self.k + 1) % 3
        self.ex.iteration = self.k
        self.A.spmv_fused_async(self.xs[cur].data_ptr(), self.xs[nxt].data_ptr() + 8 * self.row_begin, self.partials, self.ex,
                                peers=self.peers[nxt])
        self.k += 1

    def _sums(self):
        """S[K-1], S[K-2], S[K-3] (0.0 where K is too small), each added in rank order from MY mailbox."""
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)
        if int(self.sync[2].item()) != 0:
            raise RuntimeError("an exchange wait timed out: a peer rank did not finish its launch")
        flat = self.box_t.tolist()
        out = []
        for back in (1, 2, 3):
            j = self.k - back
            if j < 0:
                out.append(0.0)
                continue
            total = 0.0
            for r in range(self.world):
                at = 2 * ((j & 3) * self.world + r)
                if flat[at + 1] != j + 1:
                    raise RuntimeError(f"mailbox slot of launch {j}, rank {r} carries tag {flat[at + 1]}")
                total += torch.tensor(flat[at], dtype=torch.int64).view(torch.float64).item()
            out.append(total)
        return out

    def eigenvalue_estimate(self) -> float:
        s1, s2, s3 = self._sums()
        if self.k >= 3:
            return (s1 * s3 / s2) ** 0.5
        if self.k == 2:
            return (s1 / s2) ** 0.5       # no scaling yet: |u_2| / |u_1|
        raise ValueError("eigenvalue_estimate needs at least two iterations")

    def normalized_x(self) -> torch.Tensor:
        s1, _, _ = self._sums()
        return self.xs[self.k % 3] / (s1 ** 0.5)

    def close(self):
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)
        self.xs = []
        self.box_t = None
        for b in self.buf:
            b.close()
        self.box.close()
        self.buf = []


class AllgatherPowerIteration(PowerIteration):
    """The literal reading of BASELINE config 5: x refreshed by ONE NCCL all-gather per iteration.

    ncclAllGather needs equal slices while the nnz-balanced row ranges differ by a few rows (0.2 % at 512^3), so x is
    kept in a padded rank-major layout: part p's entries live at [p*stride, p*stride + rows_p), stride = the largest
    part rounded up to 32, and the column indices of the resident matrix are rewritten once on the device
    (spmv_b200_csr_remap_columns).  The collective is then in place (every rank's send buffer is its own slice of the
    receive buffer) and moves exactly (world-1)*stride doubles into every GPU -- the NVLink floor of a whole-vector
    refresh.  Overlap: the rows whose columns all lie in the rank's own slice (everything but the two boundary planes
    of a stencil) are multiplied WHILE the all-gather is in flight; the boundary rows follow once it has landed.

        step k:   [NCCL stream] all-gather of x_k           |  [compute stream] y = A x_k on the interior rows
                  boundary rows of y; |y|^2 -> 1-double all-reduce; own slice of x_{k+1} = y / |y|

    Rows are summed by the thread-per-row kernel in index order, so y, lambda and x match the other exchange modes
    bit for bit apart from the association of the N-rank sum of |y|^2."""

    def __init__(self, kind, p0, p1=0, p2=0, seed=0x5EED, group=None, parts=None, overlap=True):
        super().__init__(kind, p0, p1, p2, seed=seed, exchange="allgather", group=group, parts=parts)
        cu = self.x.device
        starts, self.stride = padded_layout(self.parts)
        # interior rows first (on the ORIGINAL column ids: own slice = [row_begin, row_end))
        self.interior = self.A.interior_rows(self.row_begin, self.row_end) if overlap and self.world > 1 else (0, self.rows)
        self.A.remap_columns(starts, self.stride)
        del self.x
        self.xg = torch.ones(self.world * self.stride, dtype=torch.float64, device=cu)   # padded, rank-major
        self.own = self.xg[self.rank * self.stride: (self.rank + 1) * self.stride]        # send buffer == its slot of xg
        self.launches_per_step = 5 if self.world > 1 else 3
        self.recv_bytes = 8 * (self.world - 1) * self.stride
        # The all-gather must run WHILE the interior product runs.  Both are ready at the same moment and the product's
        # grid (hundreds of thousands of small CTAs) keeps refilling every SM slot that frees up, so NCCL's few large CTAs
        # only got onto the SMs when the product had drained (measured on 2 GPUs: step = all-gather + product, no
        # overlap).  A communicator of its own on a HIGH-PRIORITY stream makes the block scheduler place NCCL's CTAs first.
        self.ag_group = group
        if self.world > 1 and dist.get_backend(group) == "nccl":
            try:
                opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
                ranks = dist.get_process_group_ranks(group) if group is not None else list(range(dist.get_world_size()))
                self.ag_group = dist.new_group(ranks=ranks, backend="nccl", pg_options=opts)
            except Exception:   # older torch: keep the default communicator (correct, just not overlapped)
                self.ag_group = group

    def reset(self, value=1.0):
        self.dev.vec_fill(self.xg, value)

    def step(self):
        d = self.dev
        lo, hi = self.interior
        if self.world > 1:
            work = dist.all_gather_into_tensor(self.xg, self.own, group=self.ag_group, async_op=True)
            if hi > lo:
                self.A.spmv_rows(lo, hi, self.xg, self.y)          # reads the own slice only: overlaps the collective
            work.wait()                                            # compute stream waits for the NCCL stream (no host block)
            if lo > 0:
                self.A.spmv_rows(0, lo, self.xg, self.y)
            if hi < self.rows:
                self.A.spmv_rows(hi, self.rows, self.xg, self.y)
        else:
            self.A.spmv(self.xg, self.y)
        d.vec_sumsq(self.y, self.ws, self.ss, n=self.rows)
        if self.world > 1:
            dist.all_reduce(self.ss, group=self.group)
        d.vec_scale_by_inv_norm(self.own[:self.rows], self.y, self.ss, n=self.rows)

    def normalized_x(self) -> torch.Tensor:
        """x in the ORIGINAL (unpadded) index space.  After a step only the own slice is current (the other slices are
        refreshed by the next step's all-gather), so they are gathered here."""
        if self.world > 1:
            dist.all_gather_into_tensor(self.xg, self.own, group=self.group)
        return unpad(self.xg, self.parts, self.stride)


class PeerAllgatherPowerIteration(PowerIteration):
    """The whole-vector refresh of BASELINE config 5 written against peer memory instead of calling NCCL ("allgather_peer").

    Every rank keeps two full replicas of x in peer-mappable buffers (x_k, x_{k+1}; original index space, no padding --
    peer stores do not need equal slices).  The all-gather is the own slice written into the same rows of every other
    rank's replica -- one DMA copy per peer (copy engines; the default), or ONE kernel per rank (spmv_b200_vec_push:
    256-bit loads, 256-bit NVLink stores) -- followed by the one-CTA
    mailbox kernel (spmv_b200_mail_exchange on a mailbox of its own) whose tags prove that every rank's slice has landed
    here.  It runs on a high-priority stream WHILE the interior rows -- a matrix handle of their own, columns inside the
    rank's slice -- are multiplied; the boundary rows (two more handles) follow once the replica is complete.  Lazy
    normalisation as in FusedPowerIteration(split=True): the product kernels are the FLAT fused ones (w = (A w_prev) /
    |w_prev|, written straight into the own slice of the next replica, one |w|^2 partial per CTA), a second mailbox
    exchange adds the partials of all ranks in rank order and leaves 1/|w| for the next launches.

        step k:   [push stream]    own slice of x_k -> all replicas ; tags            (started at the end of step k-1)
                  [compute stream] interior rows | wait for the tags | boundary rows | |w|^2 exchange -> start push k+1

    No collective library call in the loop; 5 + 2 launches per iteration."""

    def __init__(self, kind, p0, p1=0, p2=0, seed=0x5EED, group=None, parts=None, push_ctas=0, copy_engine=True, copy_streams=1,
                 kernel_peers=0):
        """copy_engine=True (default, the faster one measured): the slice travels as one cudaMemcpyAsync per peer -- the
        DMA engines drive NVLink and every SM stays with the product; copy_streams > 1 spreads the peers over that many
        streams.  copy_engine=False: spmv_b200_vec_push, the same transfer as ONE kernel of peer stores.
        kernel_peers=k with copy_engine=True: the LAST k peers of the rotation are served by the push kernel on a stream
        of its own while the copy engines serve the others (both drive the links at the same time)."""
        super().__init__(kind, p0, p1, p2, seed=seed, exchange="allgather", group=group, parts=parts)
        from . import _native as N
        d = self.dev
        cu = self.x.device
        if self.A.info().num_long_rows:
            raise ValueError("PeerAllgatherPowerIteration needs a matrix without long rows")
        lo, hi = self.A.interior_rows(self.row_begin, self.row_end) if self.world > 1 else (0, self.rows)
        self.interior = (lo, hi)
        self.A.close()
        self.A = None
        del self.x, self.y
        rb = self.row_begin
        # (local first row, handle) of the interior block and the two boundary blocks; empty blocks are skipped
        self.blocks = []
        for b_lo, b_hi in ((lo, hi), (0, lo), (hi, self.rows)):
            if b_hi > b_lo:
                self.blocks.append((b_lo, d.DeviceCSR.synth(kind, p0, p1, p2, seed=seed, row_begin=rb + b_lo, row_end=rb + b_hi)
                                    .set_image(0)))   # only the fused products run on these blocks
        self.has_interior = hi > lo
        counts = [A.flat_partials_count() for _, A in self.blocks]
        self.partials = torch.zeros(max(sum(counts), 1), dtype=torch.float64, device=cu)
        self.partial_views, at = [], 0
        for c in counts:
            self.partial_views.append(self.partials[at: at + c])
            at += c
        self.n_partials = max(at, 1)
        self.scale = torch.ones(2, dtype=torch.float64, device=cu)      # {|w|^2, 1/|w|} written by the norm exchange
        self.one = torch.ones(4, dtype=torch.float64, device=cu)        # the push barrier's dummy partial
        self.junk = torch.zeros(4, dtype=torch.float64, device=cu)
        nbytes = 8 * self.N
        self.buf = [d.PeerBuffer(nbytes), d.PeerBuffer(nbytes)]
        self.xs = [b.as_tensor() for b in self.buf]
        self.boxes = [d.PeerBuffer(N.MAILBOX_BYTES), d.PeerBuffer(N.MAILBOX_BYTES)]   # [0] |w|^2, [1] "my slice has landed"
        self.box_t = [b.as_tensor("<i8", 8) for b in self.boxes]
        self.sync = torch.zeros(4, dtype=torch.int32, device=cu)
        self.mails = []
        for i in range(2):
            m = N.Mail()
            m.world, m.rank = self.world, self.rank
            m.counter = self.sync.data_ptr() + 8 * i
            m.status = self.sync.data_ptr() + 8 * i + 4
            self.mails.append(m)
        self.push_targets = [[], []]          # per replica: the other ranks' slot for MY rows, nearest successor first
        self.push_views = [[], []]
        if self.world > 1:
            handles = [None] * self.world
            dist.all_gather_object(handles, ([b.handle_bytes() for b in self.buf], [b.handle_bytes() for b in self.boxes]),
                                   group=self.group)
            for i in range(2):
                for r in range(self.world):
                    self.mails[i].box[r] = self.boxes[i].ptr.value if r == self.rank else self.boxes[i].open_peer(handles[r][1][i])
            for parity in (0, 1):
                for step in range(1, self.world):
                    peer = (self.rank + step) % self.world
                    base = self.buf[parity].open_peer(handles[peer][0][parity])
                    self.push_targets[parity].append(base + 8 * rb)
                    self.push_views[parity].append(torch.as_tensor(_CudaView(base + 8 * rb, max(self.rows, 1), "<f8"), device=cu))
        else:
            for i in range(2):
                self.mails[i].box[0] = self.boxes[i].ptr.value
        self.push_ctas = int(push_ctas)
        self.copy_engine = bool(copy_engine)
        self.kernel_peers = max(0, min(int(kernel_peers), self.world - 1)) if self.copy_engine else 0
        self.kernel_stream = torch.cuda.Stream(device=cu, priority=-1)
        self.kernel_event = torch.cuda.Event()
        self.push_stream = torch.cuda.Stream(device=cu, priority=-1)
        self.copy_streams = [self.push_stream] + [torch.cuda.Stream(device=cu, priority=-1)
                                                  for _ in range(max(1, min(int(copy_streams), self.world - 1)) - 1)]
        self.copy_events = [torch.cuda.Event() for _ in self.copy_streams]
        self.ev_own = torch.cuda.Event()
        self.ev_landed = torch.cuda.Event()
        self.recv_bytes = 8 * (self.N - self.rows)
        self.launches_per_step = len(self.blocks) + 1 + (2 if self.world > 1 else 0)
        self.k = 0
        self.reset(1.0)

    def reset(self, value=1.0):
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)   # nobody may still be pushing rows or tags of the previous run
        for t in self.xs:
            self.dev.vec_fill(t, value)      # every replica starts complete: step 0 waits for nothing
        for t in self.box_t:
            t.zero_()
        self.sync.zero_()
        self.k = 0
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)

    def _push(self, nxt):
        """Own slice of xs[nxt] -> every other replica, then the tags (push stream; the caller recorded ev_own)."""
        ps = self.push_stream
        ps.wait_event(self.ev_own)
        own = self.xs[nxt][self.row_begin: self.row_end]
        if self.copy_engine:     # one cudaMemcpyAsync per peer, nearest successor first (every rank targets another one)
            for st in self.copy_streams[1:]:
                st.wait_event(self.ev_own)
            by_copy = len(self.push_views[nxt]) - self.kernel_peers
            if self.kernel_peers:
                self.kernel_stream.wait_event(self.ev_own)
                self.dev.vec_push(own, self.rows, self.push_targets[nxt][by_copy:], ctas=self.push_ctas, stream=self.kernel_stream)
                self.kernel_event.record(self.kernel_stream)
            for j, v in enumerate(self.push_views[nxt][:by_copy]):
                with torch.cuda.stream(self.copy_streams[j % len(self.copy_streams)]):
                    v[: self.rows].copy_(own, non_blocking=True)
            for st, ev in zip(self.copy_streams[1:], self.copy_events[1:]):
                ev.record(st)
                ps.wait_event(ev)
            if self.kernel_peers:
                ps.wait_event(self.kernel_event)
        else:
            self.dev.vec_push(own, self.rows, self.push_targets[nxt], ctas=self.push_ctas, stream=ps)
        self.mails[1].iteration = self.k
        self.dev.mail_exchange(self.one, 1, self.mails[1], self.junk, stream=ps)
        self.ev_landed.record(ps)

    def step(self):
        cur, nxt = self.k & 1, (self.k & 1) ^ 1
        x, y = self.xs[cur], self.xs[nxt]
        cs = torch.cuda.current_stream()
        inv = self.scale.data_ptr() + 8 if self.k > 0 else None
        waited = self.k == 0 or self.world == 1
        for i, (first, A) in enumerate(self.blocks):
            if not waited and (i > 0 or not self.has_interior):
                cs.wait_event(self.ev_landed)      # boundary rows read the other ranks' slices
                waited = True
            A.spmv_fused_flat(x.data_ptr(), y.data_ptr() + 8 * (self.row_begin + first), inv_norm=inv, partials=self.partial_views[i])
        if not waited:
            cs.wait_event(self.ev_landed)          # keeps the replicas two-deep even if no row needs the other slices
        self.mails[0].iteration = self.k
        self.dev.mail_exchange(self.partials, self.n_partials, self.mails[0], self.scale)
        if self.world > 1:
            self.ev_own.record(cs)
            self._push(nxt)
        self.k += 1

    def _settle(self):
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)
        if int(self.sync[1].item()) != 0 or int(self.sync[3].item()) != 0:
            raise RuntimeError("a mailbox wait timed out: a peer rank did not finish its launch")

    def eigenvalue_estimate(self) -> float:
        self._settle()
        return float(self.scale[0].item()) ** 0.5

    def normalized_x(self) -> torch.Tensor:
        """v_k = w_k / |w_k| on the WHOLE replica (the last step's push has landed: _settle synchronises all ranks)."""
        lam = self.eigenvalue_estimate()
        return self.xs[self.k & 1] / lam

    def close(self):
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier(group=self.group)
        self.xs, self.box_t, self.push_views = [], [], [[], []]
        for _, A in self.blocks:
            A.close()
        self.blocks = []
        for b in self.buf + self.boxes:
            b.close()
        self.buf, self.boxes = [], []
