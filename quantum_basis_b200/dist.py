"""Row-sharded H*v and Lanczos over several GPUs of one box: one process per GPU, torch.distributed for the plumbing.

The reference has no distributed mode (SURVEY section 5); this follows SURVEY section 8(e): H is partitioned into
contiguous row blocks, each rank holds the complete rows of the expanded Hermitian matrix for its block (no cross-GPU
writes), vectors are sharded by the same row ranges, and per product the Krylov vector is all-gathered over
NVLink (NCCL).  The two Lanczos scalars are all-reduced as device-resident doubles between the fused passes
(include/qbgpu.h: qbgpu_lanczos_step_a/b/c), so the step needs no host synchronisation.

The orchestration is written against a small `kernels` provider so that the same code runs
  - on GPUs: DeviceKernels (C-ABI calls on torch-allocated device buffers, NCCL collectives), and
  - in the CPU tests: any object with the same methods (tests/test_dist_gloo.py supplies an oracle-backed one over gloo).
"""
import ctypes as C
import json
import os
import time

import numpy as np


# Rows per owner are a multiple of this.  32: no 32-byte sector of a vector and no 32-row slice of the layout straddles two
# owners.  Species-order shards (whole up configurations, csrc/species.cu) set it to a multiple of D_dn before the operators
# are built -- species_row_align() -- and restore it afterwards.
ROW_ALIGN = 32


def species_row_align(d_dn):
    """Alignment for shards of a species-order handle: whole up configurations (multiples of D_dn rows) and, for fp64
    vectors, a multiple of 4 rows so that no 32-byte sector straddles two owners."""
    from math import gcd
    return d_dn * 4 // gcd(d_dn, 4)


def equal_row_bounds(n, parts, align=None):
    """Contiguous row partition with equal row counts (the last block may be shorter); chunk = rows per block, a multiple
    of `align` (default: the module's ROW_ALIGN)."""
    align = ROW_ALIGN if align is None else align
    chunk = (n + parts - 1) // parts
    if parts > 1:
        chunk = (chunk + align - 1) // align * align
    return [min(n, p * chunk) for p in range(parts + 1)], chunk


class ShardedOperator:
    """y_local = H[rows, :] x with x assembled from every rank's slice."""

    def __init__(self, kernels, n, rank, world, comm):
        self.k, self.n, self.rank, self.world, self.comm = kernels, n, rank, world, comm
        self.bounds, self.chunk = equal_row_bounds(n, world)
        self.lo, self.hi = self.bounds[rank], self.bounds[rank + 1]
        self.nloc = self.hi - self.lo
        self.x_full = kernels.alloc(self.chunk * world)      # padded so every rank contributes `chunk` entries

    def gather(self, x_local_padded):
        """all-gather the padded local slices into x_full (entries [p*chunk, p*chunk + n_p) are rank p's rows)."""
        self.comm.all_gather_into_tensor(self.x_full, x_local_padded)
        return self.x_full

    def matvec(self, x_local_padded, y_local):
        self.gather(x_local_padded)
        self.k.multmv(self.x_full, y_local)


def sharded_lanczos(op, u0, u1, maxit, steps, state, a_dev, b_dev):
    """`steps` fused Lanczos steps (src/lanczos.cc:167-214) on the shards.  u0/u1: padded local buffers (chunk entries),
    u0 holds this rank's slice of the normalised start vector.  state: 8 device doubles initialised to
    [1,0,0,0,0,0,0,0]; a_dev/b_dev: device arrays of maxit doubles.  Returns after `steps` steps without any host
    synchronisation; the caller reads a_dev/b_dev."""
    k, comm = op.k, op.comm
    U = [u0, u1]
    for m in range(1, steps + 1):
        ux, uz = U[(m - 1) % 2], U[m % 2]
        op.gather(ux)
        k.lanczos_step_a(op.x_full, uz, state)                # w = sx*H*ux - b*sz*uz ; state[3] = partial <v,w>
        comm.all_reduce(k.slot(state, 3))
        k.lanczos_step_b(ux, uz, state)                       # w -= a*v ; state[6] = partial |w|^2
        comm.all_reduce(k.slot(state, 6))
        k.lanczos_step_c(state, a_dev, b_dev, m)              # b = sqrt(.), rotate the scales
    return U


class PipelinedOperator(ShardedOperator):
    """The same product with the exchange overlapped: x travels as one broadcast per owner (issued asynchronously, in
    rank order), the shard is split into one column block per owner (qbgpu_split_columns), and block p is multiplied
    as soon as p's slice has arrived -- the own block first, while the first transfers are in flight."""

    def __init__(self, kernels, n, rank, world, comm):
        super().__init__(kernels, n, rank, world, comm)
        self.order = [rank] + [p for p in range(world) if p != rank]
        self.col_bounds = [min(n, p * self.chunk) for p in range(world)] + [n]

    def gather_async(self, x_local_padded):
        works = []
        for p in range(self.world):
            seg = self.k.segment(self.x_full, p * self.chunk, self.chunk)
            if p == self.rank:
                seg.copy_(x_local_padded)
            works.append(self.comm.broadcast_async(seg, p))
        return works

    def matvec(self, x_local_padded, y_local):
        works = self.gather_async(x_local_padded)
        for idx, p in enumerate(self.order):
            if p != self.rank:
                works[p].wait()
            self.k.multmv_part(p, self.x_full, y_local, accumulate=(idx > 0))
        works[self.rank].wait()

    def lanczos_step_a(self, ux, uz, state):
        works = self.gather_async(ux)
        last = len(self.order) - 1
        for idx, p in enumerate(self.order):
            if p != self.rank:
                works[p].wait()
            self.k.lanczos_step_a_part(p, self.x_full, uz, state, idx == 0, idx == last)
        works[self.rank].wait()


def pipelined_lanczos(op, u0, u1, maxit, steps, state, a_dev, b_dev):
    """sharded_lanczos with the overlapped exchange of PipelinedOperator."""
    k, comm = op.k, op.comm
    U = [u0, u1]
    for m in range(1, steps + 1):
        ux, uz = U[(m - 1) % 2], U[m % 2]
        op.lanczos_step_a(ux, uz, state)
        comm.all_reduce(k.slot(state, 3))
        k.lanczos_step_b(ux, uz, state)
        comm.all_reduce(k.slot(state, 6))
        k.lanczos_step_c(state, a_dev, b_dev, m)
    return U


class RawBuf:
    """A device buffer owned by libqbgpu (cudaMalloc, hence exportable through CUDA IPC) with the two methods the
    kernels provider needs from a tensor."""

    def __init__(self, qb, nbytes):
        self.qb, self.L, self.nbytes = qb, qb.lib(), int(nbytes)
        p = C.c_void_p()
        assert self.L.qbgpu_malloc(C.byref(p), self.nbytes) == 0, self.L.qbgpu_last_error()
        self.ptr = p.value
        assert self.L.qbgpu_memset0(C.c_void_p(self.ptr), self.nbytes) == 0

    def data_ptr(self):
        return self.ptr

    def view(self, byte_offset):
        v = object.__new__(RawBuf)
        v.qb, v.L, v.ptr, v.nbytes = self.qb, self.L, self.ptr + byte_offset, self.nbytes - byte_offset
        return v

    def upload(self, arr, byte_offset=0):
        arr = np.ascontiguousarray(arr)
        assert self.L.qbgpu_memcpy_h2d(C.c_void_p(self.ptr + byte_offset), C.c_void_p(arr.ctypes.data), arr.nbytes) == 0

    def download(self, dtype, count, byte_offset=0):
        out = np.empty(count, dtype=dtype)
        assert self.L.qbgpu_memcpy_d2h(C.c_void_p(out.ctypes.data), C.c_void_p(self.ptr + byte_offset), out.nbytes) == 0
        return out


class PeerExchangeOperator:
    """The sharded product with the exchange done by peer-memory pulls over NVLink instead of a collective.

    Every rank owns two full-length vector buffers X[0], X[1] (ping-pong) allocated by libqbgpu and exported through
    CUDA IPC; its own slice of the current vector lives in X[b][lo:hi].  A product on buffer b
      1. passes a barrier (a 1-element all-reduce, or -- inside Lanczos -- the scalar all-reduce that is there anyway),
         after which every rank's slice of X[b] is final,
      2. enqueues, on one copy stream per peer, the pull of that peer's slice from the peer's X[b] into the local X[b],
      3. multiplies the own column block at once and each other block as soon as its slice has arrived (event wait).
    The ping-pong plus the barrier make the pulls race-free: a slice is overwritten only two products later, after a
    barrier that every puller has passed."""

    def __init__(self, qb, kernels, n, rank, world, comm, torch_mod, lanes=None, mode=None, ctas=None, groups=None):
        self.qb, self.L, self.k, self.n, self.rank, self.world, self.comm, self.torch = qb, qb.lib(), kernels, n, rank, world, comm, torch_mod
        # copy streams in use.  One lane: the pulls run back to back, each at the full single-flow NVLink rate (measured
        # 718-726 GB/s), and arrive in ring order -- the order the blocks are multiplied, and at ring distance d every
        # GPU serves exactly one reader.  Measured on 8 B200 (profiles/r01_peer_variants_n8.jsonl): the exchange alone
        # takes 3.2-3.3 ms with 1 or 7 lanes, but with 7 lanes every slice arrives at the end and nothing overlaps:
        # 6.58 ms per product against 5.08 ms with one lane.
        self.lanes = int(os.environ.get("QB_PEER_LANES", "1")) if lanes is None else lanes
        # "ce": copy-engine transfers (cudaMemcpyAsync); "sm": qbgpu_peer_pull_sm, `ctas` thread blocks per transfer
        self.mode = (mode or os.environ.get("QB_PEER_MODE", "ce")).lower()
        self.ctas = int(os.environ.get("QB_PEER_CTAS", "16")) if ctas is None else ctas
        self.bounds, self.chunk = equal_row_bounds(n, world)
        self.lo, self.hi = self.bounds[rank], self.bounds[rank + 1]
        self.esize = 8 * kernels.ncomp
        self.configure(kernels, groups)
        self.col_bounds = [min(n, p * self.chunk) for p in range(world)] + [n]
        nbytes = self.chunk * world * self.esize
        self.X = [RawBuf(qb, nbytes), RawBuf(qb, nbytes)]
        import torch.distributed as dist
        handles = []
        for b in range(2):
            h = (C.c_ubyte * 64)()
            assert self.L.qbgpu_ipc_export(C.c_void_p(self.X[b].ptr), h) == 0, self.L.qbgpu_last_error()
            handles.append(bytes(h))
        allh = [None] * world
        dist.all_gather_object(allh, handles)
        self.peer = [[None] * world for _ in range(2)]
        for p in range(world):
            if p == rank:
                continue
            for b in range(2):
                out = C.c_void_p()
                hb = (C.c_ubyte * 64).from_buffer_copy(allh[p][b])
                assert self.L.qbgpu_ipc_open(hb, C.byref(out)) == 0, self.L.qbgpu_last_error()
                self.peer[b][p] = out.value
        self.token = torch_mod.zeros(1, dtype=torch_mod.float64, device="cuda")

    def configure(self, kernels, groups=None, mode=None, ctas=None, lanes=None, schedule=None):
        """(Re)select the column blocks -- kernels.parts[g] covers the owners groups[g] = (first, last+1), default one
        block per owner -- and optionally the transfer mode, on the same exported buffers."""
        rank, world = self.rank, self.world
        assert 8 * kernels.ncomp == self.esize
        self.k = kernels
        self.groups = groups if groups is not None else [(p, p + 1) for p in range(world)]
        self.own_group = next(g for g, (a, b) in enumerate(self.groups) if a <= rank < b)
        assert self.groups[self.own_group] == (rank, rank + 1), "the own slice must be a block of its own"
        # A column block without a single stored entry needs no product (Hubbard 4x4 on 8 ranks: two of the seven remote
        # blocks of every rank -- one hop cannot change the top site's occupation by two).  Its slices are still pulled:
        # dropping them was measured (profiles/r01_peer_variants_n8.jsonl, "skipped_empty_blocks") and is SLOWER, 6.43 ms
        # against 5.06 ms, because the ring schedule -- at step d every GPU serves exactly one reader -- falls out of
        # step and sources end up serving two or three readers at once (exchange alone 5.4 ms instead of 3.2 ms).
        # The saving is collected by the "matching" schedule below (conflict-free rounds over the needed transfers only:
        # 4.74 ms); QB_PEER_SCHEDULE=ring with QB_PEER_SKIP_PULLS=1 reproduces the unbalanced measurement.
        empty = set()
        if kernels.parts is not None and os.environ.get("QB_PEER_KEEP_EMPTY", "0") != "1":
            empty = {g for g in range(len(self.groups)) if kernels.parts[g].info.nnz_stored == 0}
        ring = lambda g: (self.groups[g][0] - rank) % world                                       # noqa: E731
        others = sorted((g for g in range(len(self.groups)) if g != self.own_group), key=ring)
        self.group_order = [g for g in others if g not in empty]
        pulled = self.group_order if os.environ.get("QB_PEER_SKIP_PULLS", "0") == "1" else others
        self.order = [p for g in pulled for p in range(*self.groups[g])]
        self.skipped_blocks = len(empty)
        self.schedule = "ring"
        if schedule is None:
            # measured on 8 ranks only (4.74 ms against 5.13 ms for the ring); smaller worlds keep the ring they were
            # measured with unless QB_PEER_SCHEDULE asks otherwise
            schedule = os.environ.get("QB_PEER_SCHEDULE", "matching" if world >= 8 else "ring")
        if schedule == "matching" and len(self.groups) == world and world > 2:
            # conflict-free rounds for the NEEDED transfers only: every rank publishes which owners it needs, the
            # reader/source graph is split into matchings (in a round every source serves at most one reader and every
            # reader pulls from at most one source), and each rank pulls its sources in round order
            import torch.distributed as dist
            mine = [g not in empty and g != self.own_group for g in range(world)]
            allneeds = [None] * world
            dist.all_gather_object(allneeds, mine)
            rounds = matching_rounds(allneeds)
            seq = [rd[rank] for rd in rounds if rd[rank] is not None]
            self.group_order = seq
            self.order = list(seq)
            self.schedule = f"matching ({len(rounds)} rounds)"
        if mode is not None:
            self.mode = mode
        if ctas is not None:
            self.ctas = ctas
        if lanes is not None:
            self.lanes = lanes

    def own(self, b):
        """this rank's slice of buffer b (where the caller writes its part of the vector)"""
        return self.X[b].view(self.lo * self.esize)

    def pull(self, b):
        for idx, p in enumerate(self.order):
            off = self.bounds[p] * self.esize
            nb = (self.bounds[p + 1] - self.bounds[p]) * self.esize
            if nb:
                dst, src = C.c_void_p(self.X[b].ptr + off), C.c_void_p(self.peer[b][p] + off)
                if self.mode == "sm":
                    rc = self.L.qbgpu_peer_pull_sm(idx % self.lanes, p, dst, src, nb, self.ctas)
                else:
                    rc = self.L.qbgpu_peer_pull_async(idx % self.lanes, p, dst, src, nb)
                assert rc == 0, self.L.qbgpu_last_error()

    def _wait_group(self, g):
        for p in range(*self.groups[g]):
            if self.bounds[p + 1] > self.bounds[p]:
                assert self.L.qbgpu_peer_wait(p) == 0, self.L.qbgpu_last_error()

    # ---- ring-fused product: ONE kernel over the unsplit shard that consumes the slices as they land (sjds.cu) ----
    def enable_ring(self, ring_kernels):
        """ring_kernels: DeviceKernels over the view returned by ring_view() (rows in ring order, waiting kernel)"""
        self.kr = ring_kernels

    @staticmethod
    def ring_view(qb, matrix, rank, world, chunk):
        h = C.c_void_p()
        rc = qb.lib().qbgpu_ring_prepare(matrix.handle, rank, world, chunk, C.byref(h))
        assert rc == 0, qb.lib().qbgpu_last_error()
        return qb.csr_mat._adopt(h, True)

    def pull_ring(self, b):
        assert self.L.qbgpu_peer_ring_reset() == 0, self.L.qbgpu_last_error()
        for d in range(1, self.world):
            p = (self.rank + d) % self.world
            off = self.bounds[p] * self.esize
            nb = (self.bounds[p + 1] - self.bounds[p]) * self.esize
            rc = self.L.qbgpu_peer_pull_flag((d - 1) % self.lanes, p, C.c_void_p(self.X[b].ptr + off), C.c_void_p(self.peer[b][p] + off), nb, d)
            assert rc == 0, self.L.qbgpu_last_error()

    def matvec_ring(self, b, y_local, barrier=True):
        if barrier:
            self.comm.all_reduce(self.token)
        self.pull_ring(b)
        self.kr.multmv(self.X[b], y_local)

    def lanczos_step_a_ring(self, b, uz, state):
        self.pull_ring(b)
        self.kr.lanczos_step_a(self.X[b], uz, state)

    def ring_timed_out(self):
        t = C.c_int(0)
        assert self.L.qbgpu_peer_ring_status(C.byref(t)) == 0, self.L.qbgpu_last_error()
        return bool(t.value)

    def pull_only(self, b):
        """the exchange alone (for measuring it): all pulls, then the compute stream waits for every arrival"""
        self.comm.all_reduce(self.token)
        self.pull(b)
        for g in self.group_order:
            self._wait_group(g)

    def matvec(self, b, y_local, barrier=True):
        if barrier:
            self.comm.all_reduce(self.token)
        self.pull(b)
        self.k.multmv_part(self.own_group, self.X[b], y_local, accumulate=False)
        for g in self.group_order:
            self._wait_group(g)
            self.k.multmv_part(g, self.X[b], y_local, accumulate=True)

    def lanczos_step_a(self, b, uz, state):
        """x = X[b] (all slices final: the caller's previous all-reduce is the barrier), w accumulated into uz"""
        self.pull(b)
        last = len(self.group_order)
        self.k.lanczos_step_a_part(self.own_group, self.X[b], uz, state, True, last == 0)
        for idx, g in enumerate(self.group_order):
            self._wait_group(g)
            self.k.lanczos_step_a_part(g, self.X[b], uz, state, False, idx == last - 1)


class SpeciesPeerOperator(PeerExchangeOperator):
    """The sharded product of a STORED species-order Hubbard handle (csrc/species.cu) with the peer-pull exchange: rows are
    whole up configurations, vectors are in the internal order, and the shard comes as two parts (qbgpu_species_parts):

        local  = diagonal + hops of the down electrons: gathers stay inside the rank's own rows -> needs NO remote data
        cross  = hops of the up electrons: gathers from every rank's rows

    so one product is: start every pull; local part (y = ...) while the slices travel; wait; cross part (y += ...) -- two
    kernels, instead of one column block per owner with its own pass over the row metadata and over y.  kernels.parts =
    [local, cross] (DeviceKernels over the two views)."""

    def __init__(self, qb, kernels, n, rank, world, comm, torch_mod, d_dn, lanes=None, mode=None, ctas=None):
        global ROW_ALIGN
        saved = ROW_ALIGN
        ROW_ALIGN = species_row_align(d_dn)
        try:
            super().__init__(qb, kernels, n, rank, world, comm, torch_mod, lanes=lanes, mode=mode, ctas=ctas)
        finally:
            ROW_ALIGN = saved

    def configure(self, kernels, groups=None, mode=None, ctas=None, lanes=None, schedule=None):
        rank, world = self.rank, self.world
        self.k = kernels
        self.groups = [(p, p + 1) for p in range(world)]
        self.own_group = rank
        # every slice is needed by the cross part; ring order, one reader per source at every step
        self.order = [(rank + d) % world for d in range(1, world)]
        self.group_order = list(self.order)
        self.skipped_blocks = 0
        self.schedule = "ring (all slices; local part overlaps the pulls)"
        if mode is not None:
            self.mode = mode
        if ctas is not None:
            self.ctas = ctas
        if lanes is not None:
            self.lanes = lanes

    def _wait_all(self):
        for p in self.order:
            if self.bounds[p + 1] > self.bounds[p]:
                assert self.L.qbgpu_peer_wait(p) == 0, self.L.qbgpu_last_error()

    def matvec(self, b, y_local, barrier=True):
        if barrier:
            self.comm.all_reduce(self.token)
        self.pull(b)
        self.k.multmv_part(0, self.X[b], y_local, accumulate=False)       # local part: own rows only
        self._wait_all()
        self.k.multmv_part(1, self.X[b], y_local, accumulate=True)        # cross part

    def lanczos_step_a(self, b, uz, state):
        self.pull(b)
        self.k.lanczos_step_a_part(0, self.X[b], uz, state, True, False)
        self._wait_all()
        self.k.lanczos_step_a_part(1, self.X[b], uz, state, False, True)


def matching_rounds(needs):
    """needs[r][p]: reader r needs the slice of owner p.  Returns rounds; rounds[k][r] = the owner r pulls from in round k
    (or None).  Repeated maximum bipartite matching (Kuhn's augmenting paths, deterministic): for a regular graph every
    round is a perfect matching, so the number of rounds equals the degree."""
    world = len(needs)
    adj = [[p for p in range(world) if needs[r][p]] for r in range(world)]
    rounds = []
    while any(adj):
        match_src = [None] * world                      # source -> reader

        def augment(r, seen):
            # try the sources in ring order from r, so that the rounds resemble the ring when everything is needed
            for p in sorted(adj[r], key=lambda q: (q - r) % world):
                if p in seen:
                    continue
                seen.add(p)
                if match_src[p] is None or augment(match_src[p], seen):
                    match_src[p] = r
                    return True
            return False

        for r in sorted(range(world), key=lambda q: -len(adj[q])):
            if adj[r]:
                augment(r, set())
        rd = [None] * world
        for p, r in enumerate(match_src):
            if r is not None:
                rd[r] = p
                adj[r].remove(p)
        rounds.append(rd)
    return rounds


def peer_groups(world, rank, size):
    """Column blocks for PeerExchangeOperator: the own slice alone, the other owners in runs of `size` neighbours growing
    away from it -> [(first, last+1), ...] in column order."""
    out = [(rank, rank + 1)]
    p = rank
    while p > 0:
        out.append((max(0, p - size), p))
        p = max(0, p - size)
    p = rank + 1
    while p < world:
        out.append((p, min(world, p + size)))
        p = min(world, p + size)
    return sorted(out)


def peer_lanczos(op, steps, state, a_dev, b_dev, start_buffer=0, ring=False):
    """Fused Lanczos on the shards with the peer-pull exchange.  The normalised start slice is in op.own(start_buffer)
    and must already be visible to the peers (call op.comm.all_reduce(op.token) after writing it).  ring=True: the
    ring-fused single-kernel product (op.enable_ring) instead of one product per column block."""
    k, comm = (op.kr if ring else op.k), op.comm
    for m in range(1, steps + 1):
        bx, bz = (start_buffer + m - 1) % 2, (start_buffer + m) % 2
        ux, uz = op.own(bx), op.own(bz)
        if ring:
            op.lanczos_step_a_ring(bx, uz, state)
        else:
            op.lanczos_step_a(bx, uz, state)
        comm.all_reduce(k.slot(state, 3))
        k.lanczos_step_b(ux, uz, state)
        comm.all_reduce(k.slot(state, 6))                      # also the barrier that makes X[bz] final everywhere
        k.lanczos_step_c(state, a_dev, b_dev, m)


# ----------------------------------------------------------------------------------------------- GPU provider
class TorchComm:
    def __init__(self):
        import torch.distributed as dist
        self.dist = dist

    def all_gather_into_tensor(self, out, inp):
        self.dist.all_gather_into_tensor(out, inp)

    def all_reduce(self, t):
        self.dist.all_reduce(t)

    def broadcast_async(self, t, src):
        return self.dist.broadcast(t, src=src, async_op=True)

    def barrier(self):
        self.dist.barrier()


class DeviceKernels:
    """C-ABI calls on torch device tensors.  real=False: complex128 vectors stored as float64 pairs (z entry points);
    real=True: float64 vectors through qbgpu_real_view handles (d entry points) -- for Krylov loops that stay real."""

    def __init__(self, qb, matrix, real=False, parts=None):
        import torch
        self.torch, self.qb, self.L = torch, qb, qb.lib()
        self.real, self.ncomp = real, (1 if real else 2)
        self.owner = matrix
        self.M = matrix.real_view() if real else matrix
        self.parts = None
        if parts is not None:
            self.parts = [p.real_view() for p in parts] if real else parts

    def alloc(self, nentries):
        return self.torch.zeros(self.ncomp * nentries, dtype=self.torch.float64, device="cuda")

    def slot(self, state, i):
        return state[i:i + 1]

    def segment(self, t, first_entry, nentries):
        return t[self.ncomp * first_entry: self.ncomp * (first_entry + nentries)]

    def _p(self, t):
        return C.c_void_p(t.data_ptr())             # torch tensor or RawBuf

    @staticmethod
    def split(qb, matrix, col_bounds, flags=0):
        """one handle per column owner (qbgpu_split_columns) of a complex-API shard"""
        L = qb.lib()
        nparts = len(col_bounds) - 1
        b = np.array(col_bounds, dtype=np.int64)
        hs = (C.c_void_p * nparts)()
        rc = L.qbgpu_split_columns(matrix.handle, nparts, b.ctypes.data, hs, flags)
        assert rc == 0, L.qbgpu_last_error()
        return [qb.csr_mat._adopt(C.c_void_p(hs[p]), True) for p in range(nparts)]

    def _mv(self, handle, x, beta, y):
        if self.real:
            rc = self.L.qbgpu_dmv(handle, 1.0, self._p(x), float(beta), self._p(y), 1)
        else:
            one = (C.c_double * 2)(1.0, 0.0); b = (C.c_double * 2)(float(beta), 0.0)
            rc = self.L.qbgpu_zmv(handle, one, self._p(x), b, self._p(y), 1)
        assert rc == 0, self.L.qbgpu_last_error()

    def multmv(self, x_full, y_local):
        self._mv(self.M.handle, x_full, 0.0, y_local)

    def multmv_part(self, p, x_full, y_local, accumulate):
        self._mv(self.parts[p].handle, x_full, 1.0 if accumulate else 0.0, y_local)

    def lanczos_step_a(self, x_full, uz, state):
        assert self.L.qbgpu_lanczos_step_a(self.M.handle, self._p(x_full), self._p(uz), self._p(state)) == 0, self.L.qbgpu_last_error()

    def lanczos_step_a_part(self, p, x_full, uz, state, first, last):
        rc = self.L.qbgpu_lanczos_step_a_part(self.parts[p].handle, self._p(x_full), self._p(uz), self._p(state), int(first), int(last))
        assert rc == 0, self.L.qbgpu_last_error()

    def lanczos_step_b(self, ux, uz, state):
        assert self.L.qbgpu_lanczos_step_b(self.M.handle, self._p(ux), self._p(uz), self._p(state)) == 0, self.L.qbgpu_last_error()

    def lanczos_step_c(self, state, a_dev, b_dev, m):
        assert self.L.qbgpu_lanczos_step_c(self._p(state), self._p(a_dev), self._p(b_dev), m) == 0, self.L.qbgpu_last_error()


# ----------------------------------------------------------------------------------------------- native drivers
class NativeDist:
    """ctypes face of csrc/dist.cu: the multi-GPU Krylov drivers behind the C ABI (qbgpu_dist_*).  One process per GPU; the
    vector slices and the scalars travel through peer memory (CUDA IPC), nothing in the loops touches NCCL or the host side of
    torch.distributed -- `exchange` is only used ONCE, to hand the 64-byte handles around (any all-gather of bytes will do:
    here torch.distributed.all_gather_object; a C++ host would use files, pipes or MPI, see INTEGRATION.md)."""

    def __init__(self, qb, n, bounds, rank, world, complex_vectors, exchange):
        self.qb, self.L, self.n, self.rank, self.world = qb, qb.lib(), n, rank, world
        self.bounds = [int(b) for b in bounds]
        self.complex = bool(complex_vectors)
        self.dtype = np.complex128 if self.complex else np.float64
        self.h = C.c_void_p()
        b = np.array(self.bounds, dtype=np.int64)
        self._chk(self.L.qbgpu_dist_create(C.byref(self.h), rank, world, n, b.ctypes.data, int(self.complex)))
        hb = (C.c_ubyte * 64)()
        self._chk(self.L.qbgpu_dist_export(self.h, hb))
        allh = exchange(bytes(hb))
        blob = (C.c_ubyte * (64 * world)).from_buffer_copy(b"".join(allh))
        self._chk(self.L.qbgpu_dist_connect(self.h, blob))

    def _chk(self, rc):
        if rc != 0:
            raise RuntimeError(f"libqbgpu status {rc}: {self.L.qbgpu_last_error().decode(errors='replace')}")

    @property
    def nloc(self):
        return self.bounds[self.rank + 1] - self.bounds[self.rank]

    def own(self, b):
        p, nl = C.c_void_p(), C.c_int64()
        self._chk(self.L.qbgpu_dist_own(self.h, b, C.byref(p), C.byref(nl)))
        return p.value

    def full(self, b):
        p = C.c_void_p()
        self._chk(self.L.qbgpu_dist_full(self.h, b, C.byref(p)))
        return p.value

    def upload_own(self, b, arr):
        arr = np.ascontiguousarray(arr, dtype=self.dtype)
        assert arr.size == self.nloc
        if arr.size:
            self._chk(self.L.qbgpu_memcpy_h2d(C.c_void_p(self.own(b)), C.c_void_p(arr.ctypes.data), arr.nbytes))

    def download_own(self, b):
        out = np.empty(self.nloc, dtype=self.dtype)
        if out.size:
            self._chk(self.L.qbgpu_memcpy_d2h(C.c_void_p(out.ctypes.data), C.c_void_p(self.own(b)), out.nbytes))
        return out

    def barrier(self):
        self._chk(self.L.qbgpu_dist_barrier(self.h))

    def randomize(self, b, seed, ref_rows_ptr=None):
        self._chk(self.L.qbgpu_dist_randomize(self.h, b, seed, C.c_void_p(ref_rows_ptr) if ref_rows_ptr else None))

    @staticmethod
    def _hp(m):
        return m.handle if m is not None else None

    def mv(self, local, rest, b, y_ptr, barrier=True):
        """barrier: True / 1 = before the pulls; 3 = also after the product (the own slice of X[b] may then be rewritten)"""
        self._chk(self.L.qbgpu_dist_mv(self.h, self._hp(local), rest.handle, b, C.c_void_p(y_ptr), int(barrier)))

    def lanczos(self, local, rest, np_, maxit, purpose="sr_val0", stop_on_breakdown=True):
        hess = np.zeros(2 * maxit)
        m = C.c_int64(0)
        self._chk(self.L.qbgpu_dist_lanczos(self.h, self._hp(local), rest.handle, np_, maxit, C.byref(m), C.c_void_p(hess.ctypes.data),
                                            purpose.encode(), int(stop_on_breakdown)))
        return int(m.value), hess

    def energy_scale(self, local, rest, extend=0.1, iters=128, ref_rows_ptr=None):
        lo, hi = C.c_double(), C.c_double()
        self._chk(self.L.qbgpu_dist_energy_scale(self.h, self._hp(local), rest.handle, C.c_void_p(ref_rows_ptr) if ref_rows_ptr else None,
                                                 C.byref(lo), C.byref(hi), extend, iters))
        return lo.value, hi.value

    def kpm_moments(self, local, rest, lo, hi, nmom):
        mu = np.zeros(nmom)
        self._chk(self.L.qbgpu_dist_kpm_moments(self.h, self._hp(local), rest.handle, lo, hi, nmom, C.c_void_p(mu.ctypes.data)))
        return mu

    def eigenvec_cg(self, local, rest, E0, v_ptr, r_ptr, p_ptr, pp_ptr, maxit=1000):
        m, accu = C.c_int64(0), C.c_double(0.0)
        e0 = (C.c_double * 2)(float(np.real(E0)), float(np.imag(E0)))
        self._chk(self.L.qbgpu_dist_eigenvec_cg(self.h, self._hp(local), rest.handle, maxit, C.byref(m), e0, C.byref(accu),
                                                C.c_void_p(v_ptr), C.c_void_p(r_ptr), C.c_void_p(p_ptr), C.c_void_p(pp_ptr)))
        return int(m.value), accu.value

    def lanczos_val1(self, local, rest, phi0_ptr, np_, maxit, stop_on_breakdown=True):
        """sr_val1 Lanczos (re-orthogonalised against phi0 in every step) from the normalised start vector in the own slice of
        X[0], orthogonal to phi0; phi0_ptr: this rank's rows of phi0 (device).  Returns (m, hess) like lanczos()."""
        hess = np.zeros(2 * maxit)
        m = C.c_int64(0)
        self._chk(self.L.qbgpu_dist_lanczos_val1(self.h, self._hp(local), rest.handle, C.c_void_p(phi0_ptr), np_, maxit, C.byref(m),
                                                 C.c_void_p(hess.ctypes.data), int(stop_on_breakdown)))
        return int(m.value), hess

    def locate_E0_lanczos(self, local, rest, nev=1, ncv=1, maxit=1000, ref_rows_ptr=None):
        """model<T>::locate_E0_lanczos (src/model.cc:1124-1316) on the shards: the keys of csr.locate_E0_lanczos, with the
        eigenvectors as this rank's rows in the shard's order (the internal order for species-order shards)."""
        import torch
        if not (0 < nev <= 2 and nev - 1 <= ncv <= nev):
            raise ValueError("need 0 < nev <= 2 and nev-1 <= ncv <= nev")          # the reference's assert, :1141
        w = np.zeros(2)
        steps = np.zeros(4, dtype=np.int64)
        accu = np.zeros(4)
        comps = 2 if self.complex else 1
        phi = torch.zeros(max(ncv * self.nloc * comps, 1), dtype=torch.float64, device="cuda") if ncv > 0 else None
        self._chk(self.L.qbgpu_dist_locate_e0_lanczos(self.h, self._hp(local), rest.handle, C.c_void_p(ref_rows_ptr) if ref_rows_ptr else None,
                                                      nev, ncv, maxit, C.c_void_p(w.ctypes.data), C.c_void_p(phi.data_ptr()) if phi is not None else None,
                                                      C.c_void_p(steps.ctypes.data), C.c_void_p(accu.ctypes.data)))
        out = {"eigenvals": [float(w[0])], "eigenvecs": [], "lanczos_steps": int(steps[0]), "lanczos_accuracy": float(accu[0])}
        if ncv == 0:
            return out
        out["cg_steps"], out["cg_accuracy"] = int(steps[1]), float(accu[1])
        vecs = phi.cpu().numpy()[:ncv * self.nloc * comps]
        vecs = (vecs.view(np.complex128) if self.complex else vecs).reshape(ncv, self.nloc)
        if nev == 2:
            out["eigenvals"].append(float(w[1]))
            out["gap"] = float(w[1] - w[0])
            out["lanczos_steps_E1"] = int(steps[2])
        out["eigenvecs"].append(vecs[0].copy())
        if ncv == 2:
            out["cg_steps_E1"], out["cg_accuracy_E1"] = int(steps[3]), float(accu[3])
            out["eigenvecs"].append(vecs[1].copy())
        return out

    def destroy(self):
        if self.h:
            self.L.qbgpu_dist_destroy(self.h)
            self.h = None


def species_order_key(words, nsites):
    """the order of the configurations of one species in csrc/species.cu (build_host_tables): odd-site bits major"""
    words = np.asarray(words, dtype=np.int64)
    odd = np.zeros_like(words)
    even = np.zeros_like(words)
    for s_ in range(nsites):
        bit = (words >> s_) & 1
        if s_ % 2:
            odd |= bit << (s_ // 2)
        else:
            even |= bit << (s_ // 2)
    return (odd << nsites) | even


def species_nnz_balanced_bounds(nsites, nup, ndn, bonds, world):
    """Row bounds (multiples of D_dn: whole up configurations) that balance the STORED ENTRIES of the species-order shards:
    rows of one up configuration u hold D_dn * (1 + h_dn) local entries (the same for every u) plus D_dn * h_up(u) cross
    entries, h_up(u) = number of hops available to the up electrons in u.  Returns (bounds, D_dn)."""
    from math import comb
    allw = np.arange(1 << nsites, dtype=np.int64)
    pc = np.zeros_like(allw)
    for s_ in range(nsites):
        pc += (allw >> s_) & 1
    ups = allw[pc == nup]
    ups = ups[np.argsort(species_order_key(ups, nsites), kind="stable")]
    hops = np.zeros(ups.size, dtype=np.int64)
    seen = set()
    for (i, j) in bonds:
        key = (min(i, j), max(i, j))
        if key in seen:
            continue
        seen.add(key)
        hops += (((ups >> i) & 1) != ((ups >> j) & 1)).astype(np.int64)
    dd = comb(nsites, ndn)
    dns = allw[pc == ndn]
    hd = 0
    for (i, j) in seen:
        hd += int((((dns >> i) & 1) != ((dns >> j) & 1)).sum())
    w = dd + hd + dd * hops                                  # stored entries of the rows of each up configuration
    cum = np.concatenate([[0], np.cumsum(w)])
    total = cum[-1]
    cuts = [0]
    for r in range(1, world):
        cuts.append(int(np.searchsorted(cum, total * r / world)))
    cuts.append(ups.size)
    cuts = [min(max(c, cuts[k - 1] if k else 0), ups.size) for k, c in enumerate(cuts)]
    return [c * dd for c in cuts], dd


def _species_up_configs(nsites, nup):
    allw = np.arange(1 << nsites, dtype=np.int64)
    pc = np.zeros_like(allw)
    for s_ in range(nsites):
        pc += (allw >> s_) & 1
    ups = allw[pc == nup]
    ups = ups[np.argsort(species_order_key(ups, nsites), kind="stable")]
    rank_of = np.full(1 << nsites, -1, dtype=np.int64)
    rank_of[ups] = np.arange(ups.size)
    return ups, rank_of


def species_needed_mask(nsites, nup, bonds, u_lo, u_hi, own=None):
    """need[u'] = the up-hops of the configurations [u_lo, u_hi) reach configuration u' (those inside `own` = (lo, hi) excluded)"""
    ups, rank_of = _species_up_configs(nsites, nup)
    mine = ups[u_lo:u_hi]
    need = np.zeros(ups.size, dtype=bool)
    seen = set()
    for (i, j) in bonds:
        key = (min(i, j), max(i, j))
        if key in seen:
            continue
        seen.add(key)
        act = mine[((mine >> i) & 1) != ((mine >> j) & 1)]
        need[rank_of[act ^ ((1 << i) | (1 << j))]] = True
    o = own if own is not None else (u_lo, u_hi)
    need[o[0]:o[1]] = False
    return need


def _mask_to_segments(need, world_bounds_u, dd, me, gap):
    """(owner, first_row, nrows) per run of needed configurations (runs closer than `gap` merged, never across owners), ring order"""
    world = len(world_bounds_u) - 1
    segs = []
    covered = np.zeros(need.size, dtype=bool)
    for p in range(world):
        a, b = world_bounds_u[p], world_bounds_u[p + 1]
        idx = np.nonzero(need[a:b])[0] + a
        if idx.size == 0:
            continue
        breaks = np.nonzero(np.diff(idx) - 1 > gap)[0]
        starts = np.concatenate([[idx[0]], idx[breaks + 1]])
        ends = np.concatenate([idx[breaks], [idx[-1]]])
        for s0, e0 in zip(starts, ends):
            segs.append((p, int(s0) * dd, int(e0 - s0 + 1) * dd))
            covered[s0:e0 + 1] = True
    segs.sort(key=lambda t: ((t[0] - me) % world, t[1]))
    return segs, covered


def species_needed_rows(nsites, nup, ndn, bonds, u_lo, u_hi, world_bounds_u, gap=8, row_cuts=None):
    """Row ranges of the OTHER ranks' slices that the cross part of the shard [u_lo, u_hi) (units: up configurations) references:
    the targets of the up-hops of its configurations.  Neighbouring targets closer than `gap` configurations are fetched as one
    range (fewer transfers).  Returns (segments, wait_after): segments = [(owner, first_row, nrows)] ordered by ring distance
    from the shard's rank; with row_cuts = [u_lo, c1, ..., u_hi] the segments the rows [u_lo, c1) need come first, then what
    [c1, c2) needs in addition, ..., and wait_after[j] = number of segments that must have arrived before row block j starts."""
    from math import comb
    dd = comb(nsites, ndn)
    world = len(world_bounds_u) - 1
    me = next((r for r in range(world) if world_bounds_u[r] <= u_lo < world_bounds_u[r + 1]), 0) if u_hi > u_lo else 0
    cuts = row_cuts if row_cuts else [u_lo, u_hi]
    segs, wait_after = [], []
    have = None
    for k in range(len(cuts) - 1):
        need = species_needed_mask(nsites, nup, bonds, cuts[k], cuts[k + 1], own=(u_lo, u_hi))
        if have is not None:
            need &= ~have
        sg, cov = _mask_to_segments(need, world_bounds_u, dd, me, gap)
        have = cov if have is None else (have | cov)
        segs += sg
        wait_after.append(len(segs))
    return segs, wait_after


class SpeciesShard:
    """A stored species-order row shard prepared for the native drivers (csrc/dist.cu).  Ways to run it (`install`):

      plain_whole_slices   local part while every peer's whole slice travels, then the cross part
      plain_needed_rows    the same, fetching only the row ranges the cross part references
      rows<k>_needed_rows  the cross part cut into k row blocks: block j starts as soon as the ranges ITS rows reference have
                           arrived (they are fetched first), so most of the cross part overlaps the rest of the exchange
      refined_needed_rows  the cross entries whose columns are the rank's own rows run with the local part (no remote data),
                           the others after the arrival (costs a second pass over the row metadata)"""

    def __init__(self, qb, M, nsites, nup, ndn, bonds, bounds, rank, world, real, gap=8):
        from math import comb
        self.qb, self.L = qb, qb.lib()
        self.args = (nsites, nup, ndn, bonds)
        self.bounds, self.rank, self.world, self.gap, self.real, self.M = bounds, rank, world, gap, real, M
        self.n, self.lo, self.hi = M.info.n, bounds[rank], bounds[rank + 1]
        self.dd = comb(nsites, ndn)
        self.tile = 64
        self.view = M.real_view() if real else M
        self.local, self.cross = self.view.species_parts()
        self._owned, self._views = [], []
        self._split = None
        self.ub = [x // self.dd for x in bounds]
        self.plans = {}
        self.installed = ([self.local], [self.cross])
        self.plan = []

    def _plan(self, cuts=None):
        key = tuple(cuts) if cuts else None
        if key not in self.plans:
            ns, nu, nd, bonds = self.args
            self.plans[key] = (species_needed_rows(ns, nu, nd, bonds, self.lo // self.dd, self.hi // self.dd, self.ub, gap=self.gap, row_cuts=cuts)
                               if self.world > 1 else ([], [0] * (len(cuts) - 1 if cuts else 1)))
        return self.plans[key]

    def _refined(self):
        if self._split is None:
            cuts = sorted({0, self.lo, self.hi, self.n})
            b = np.array(cuts, dtype=np.int64)
            hs = (C.c_void_p * (len(cuts) - 1))()
            rc = self.L.qbgpu_species_split_cross(self.M.handle, len(cuts) - 1, b.ctypes.data, hs)
            assert rc == 0, self.L.qbgpu_last_error()
            owned = [self.qb.csr_mat._adopt(C.c_void_p(hs[k]), True) for k in range(len(cuts) - 1)]
            self._owned += owned
            parts = [(cuts[k], cuts[k + 1], (p_.real_view() if self.real else p_)) for k, p_ in enumerate(owned)]
            self._views += [p_[2] for p_ in parts if self.real]
            early = [self.local] + [p_ for (a, b_, p_) in parts if a == self.lo and b_ == self.hi]
            late = [p_ for (a, b_, p_) in parts if not (a == self.lo and b_ == self.hi) and p_.info.nnz_stored > 0]
            self.own_cross_fraction = sum(p_.info.nnz_stored for p_ in early[1:]) / max(1, self.cross.info.nnz_stored)
            self._split = (early, late)
        return self._split

    def _row_blocks(self, k):
        """the cross part cut into k row blocks at multiples of lcm(32, D_dn) rows; returns (views, cuts in up configurations)"""
        from math import gcd
        step_u = 32 // gcd(32, self.dd)                     # up configurations per lcm(32, D_dn) rows
        u_lo, u_hi = self.lo // self.dd, self.hi // self.dd
        cuts = [u_lo]
        for j in range(1, k):
            c = u_lo + ((u_hi - u_lo) * j // k) // step_u * step_u
            if c > cuts[-1]:
                cuts.append(c)
        cuts.append(u_hi)
        views = []
        for a, b in zip(cuts[:-1], cuts[1:]):
            h = C.c_void_p()
            rc = self.L.qbgpu_row_view(self.cross.handle, (a - u_lo) * self.dd, (b - u_lo) * self.dd, self.dd, self.tile, C.byref(h))
            assert rc == 0, self.L.qbgpu_last_error()
            views.append(self.qb.csr_mat._adopt(h, not self.real))
        self._views += views
        return views, cuts

    def install(self, D, mode="plain_needed_rows", lanes=1):
        none = (None, None, None)
        cuts = None
        if mode == "plain_whole_slices" or mode == "plain_needed_rows":
            early, late = [self.local], [self.cross]
        elif mode == "refined_needed_rows":
            early, late = self._refined()
        elif mode.startswith("rows") and mode.endswith("_needed_rows"):
            views, cuts = self._row_blocks(int(mode[4:-12]))
            early, late = [self.local], views
        else:
            raise ValueError(mode)
        ne, nl = len(early), len(late)
        ea = (C.c_void_p * max(ne, 1))(*[p_.handle for p_ in early])
        la = (C.c_void_p * max(nl, 1))(*[p_.handle for p_ in late])
        D._chk(self.L.qbgpu_dist_set_parts(D.h, ne, ea, nl, la))
        self.installed = (early, late)
        if mode == "plain_whole_slices" or D.world == 1:
            D._chk(self.L.qbgpu_dist_set_pull_plan(D.h, 0, *none, lanes))
            self.plan = []
            return
        plan, wait_after = self._plan(cuts)
        self.plan = plan
        ow = np.array([t[0] for t in plan] or [0], dtype=np.int32)
        fi = np.array([t[1] for t in plan] or [0], dtype=np.int64)
        nr = np.array([t[2] for t in plan] or [0], dtype=np.int64)
        D._chk(self.L.qbgpu_dist_set_pull_plan(D.h, len(plan), ow.ctypes.data, fi.ctypes.data, nr.ctypes.data, lanes))
        if cuts is not None and nl > 1:
            wa = np.array(wait_after, dtype=np.int32)
            D._chk(self.L.qbgpu_dist_set_wait_points(D.h, nl, wa.ctypes.data))

    @property
    def pulled_rows(self):
        return sum(t[2] for t in self.plan) if self.plan else (self.n - (self.hi - self.lo) if self.world > 1 else 0)

    def destroy(self):
        for v_ in self._views + [self.local, self.cross]:
            v_.destroy()
        if self.real:
            self.view.destroy()
        for p_ in self._owned:
            p_.destroy()


def _timed(torch, dist, stream, fn, steps, warmup):
    """warmup + `steps` timed calls bracketed by barrier + synchronize; device time, max over ranks (ms per step)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize(); dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def bench_sharded_species(args, WORKLOADS, algorithmic_bytes, measured_peak, ClockSampler):
    """bench.py's N > 1 arm for the Hubbard workloads: stored species-order shards (whole up configurations, balanced by
    stored entries), the native drivers of csrc/dist.cu -- peer-memory pulls overlapped with the local part, the push-based
    all-reduce kernel -- and the Lanczos loop with the reference's stop rule, so that E0 and its time-to-solution are
    measured at every N.  Strong scaling: the total work is fixed."""
    import torch
    import torch.distributed as dist
    import quantum_basis_b200 as qb
    from quantum_basis_b200.bench_support import square_bonds
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = qb.lib()
    stream = torch.cuda.current_stream()
    fam, p = WORKLOADS[args.workload]
    ns = p["Lx"] * p["Ly"]
    bonds = square_bonds(p["Lx"], p["Ly"])
    n = L.qbgpu_dim_hubbard(ns, p["nup"], p["ndn"])
    bounds, d_dn = species_nnz_balanced_bounds(ns, p["nup"], p["ndn"], bonds, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    nloc = hi - lo
    t0 = time.time()
    M = qb.hubbard(ns, p["nup"], p["ndn"], bonds, p["t"], p["U"], flags=128, rows=(lo, hi))     # complex API handle, real values
    torch.cuda.synchronize()
    t_build = time.time() - t0
    inf = M.info

    def exchange(b):
        out = [None] * world
        dist.all_gather_object(out, b)
        return out

    peak, peak_src = measured_peak()
    res = {}
    ref_rows = torch.empty(max(nloc, 1), dtype=torch.int32, device="cuda")
    assert L.qbgpu_species_ref_rows(ns, p["nup"], p["ndn"], lo, hi, C.c_void_p(ref_rows.data_ptr())) == 0, L.qbgpu_last_error()
    nnz_all = torch.tensor([inf.nnz_stored], dtype=torch.int64, device="cuda")
    dist.all_reduce(nnz_all)
    Z = int(nnz_all.item())
    sampler = ClockSampler(local_rank)
    sampler.start()
    L.qbgpu_kernel_launches(1)
    launches = 0
    for tag, cplx in (("fp64", False), ("complex128", True)):
        shard = SpeciesShard(qb, M, ns, p["nup"], p["ndn"], bonds, bounds, rank, world, real=not cplx)
        loc, cross = shard.local, shard.cross
        D = NativeDist(qb, n, bounds, rank, world, cplx, exchange)
        lanes = int(os.environ.get("QB_DIST_LANES", "1"))
        D.randomize(0, 1, ref_rows.data_ptr())                       # the reference's start vector vec_randomize(seed 1), this rank's rows
        y = torch.zeros((2 if cplx else 1) * max(nloc, 1), dtype=torch.float64, device="cuda")
        # three ways to run the same shard; the fastest (max over ranks) is the headline and serves the Lanczos leg
        modes = (["plain_whole_slices", "plain_needed_rows", "rows2_needed_rows", "rows3_needed_rows", "rows4_needed_rows", "refined_needed_rows"]
                 if world > 1 else ["plain_whole_slices"])
        if os.environ.get("QB_DIST_MODES"):
            modes = os.environ["QB_DIST_MODES"].split(",")
        tv = {}
        for vname in modes:
            shard.install(D, vname, lanes=lanes)
            D.barrier()
            tv[vname] = _timed(torch, dist, stream, lambda: D.mv(loc, cross, 0, y.data_ptr(), barrier=True), max(5, args.steps // 2), 3)
        best = min(tv, key=tv.get)
        shard.install(D, best, lanes=lanes)
        ms = _timed(torch, dist, stream, lambda: D.mv(loc, cross, 0, y.data_ptr(), barrier=True), args.steps, args.warmup)
        launches += int(L.qbgpu_kernel_launches(1))
        # the parts alone (no exchange): where the time goes
        one_, zero_ = (C.c_double * 2)(1.0, 0.0), (C.c_double * 2)(0.0, 0.0)

        def run_parts(parts, first_opens):
            for k_, pt in enumerate(parts):
                beta = 0.0 if (first_opens and k_ == 0) else 1.0
                yp = y.data_ptr() + (pt.info.row_lo - lo) * (16 if cplx else 8)           # a row view addresses its own rows
                if cplx:
                    L.qbgpu_zmv(pt.handle, one_, C.c_void_p(D.full(0)), (C.c_double * 2)(beta, 0.0), C.c_void_p(yp), 1)
                else:
                    L.qbgpu_dmv(pt.handle, 1.0, C.c_void_p(D.full(0)), beta, C.c_void_p(yp), 1)
        early_, late_ = shard.installed
        ms_early = _timed(torch, dist, stream, lambda: run_parts(early_, True), max(3, args.steps // 2), 2)
        ms_late = _timed(torch, dist, stream, lambda: run_parts(late_, False), max(3, args.steps // 2), 2) if late_ else 0.0
        ms_local, ms_cross = ms_early, ms_late
        esz = 16 if cplx else 8
        res[tag] = {"ms_per_product": ms, "products_per_s": 1e3 / ms, "early_parts_ms": ms_early, "late_parts_ms": ms_late,
                    "exposed_exchange_ms": max(0.0, ms - ms_early - ms_late), "decomposition": best, "decompositions_ms": tv,
                    "remote_bytes_pulled_rank0": shard.pulled_rows * esz,
                    "remote_bytes_if_whole_slices_rank0": (n - nloc) * esz, "pull_segments_rank0": len(shard.plan),
                    "parts": "early (no remote data: local part + cross entries with own columns) | late (the other cross entries)"}
        if not cplx and not args.no_lanczos:
            # E0 by the reference's Lanczos with its stop rule, on the shards (fp64: H and the start vector are real)
            D.randomize(0, 1, ref_rows.data_ptr())
            D.lanczos(loc, cross, 6, 1000, "sr_val0")                # warm-up: every kernel of the loop has been loaded and launched once
            D.randomize(0, 1, ref_rows.data_ptr())
            torch.cuda.synchronize(); dist.barrier()
            tl = time.time()
            m, hess = D.lanczos(loc, cross, 999, 1000, "sr_val0")
            torch.cuda.synchronize(); dist.barrier()
            tl = time.time() - tl
            tmax = torch.tensor([tl], dtype=torch.float64, device="cuda")
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            ritz, _ = qb.hess_eigen(hess, 1000, m)
            res["lanczos"] = {"vectors": "fp64 (real mode)", "steps": m, "seconds": float(tmax.item()), "iters_per_s": m / float(tmax.item()),
                              "E0": float(ritz[0]), "stop_rule": "src/lanczos.cc:228-248 on the all-reduced (a, b), identical on every rank",
                              "timing": "start vector to converged E0, wall clock, max over ranks, after a 6-step warm-up run (kernels loaded)",
                              "a0": float(hess[1000]), "b1": float(hess[1])}
        if not cplx:
            # e2e: every rank uploads its slice of x (fp64: the complex API vector has no imaginary part) and downloads its slice of y
            xh = torch.empty(max(nloc, 1), dtype=torch.float64).pin_memory()
            yh = torch.empty(max(nloc, 1), dtype=torch.float64).pin_memory()
            xh[:nloc] = torch.from_numpy(D.download_own(0))

            def e2e_step():
                assert L.qbgpu_memcpy_h2d(C.c_void_p(D.own(0)), C.c_void_p(xh.data_ptr()), nloc * 8) == 0
                D.mv(loc, cross, 0, y.data_ptr(), barrier=3)       # closing barrier too: the next step rewrites the own slice of X[0]
                assert L.qbgpu_memcpy_d2h(C.c_void_p(yh.data_ptr()), C.c_void_p(y.data_ptr()), nloc * 8) == 0
            for _ in range(2):
                e2e_step()
            torch.cuda.synchronize(); dist.barrier()
            te = time.time()
            ne = max(3, min(args.steps, 10))
            for _ in range(ne):
                e2e_step()
            torch.cuda.synchronize(); dist.barrier()
            e2e_s = torch.tensor([(time.time() - te) / ne], dtype=torch.float64, device="cuda")
            dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
            res["e2e_s"] = float(e2e_s.item())
        D.destroy()
        shard.destroy()
    clocks = sampler.stop()
    if rank == 0:
        ms = res["fp64"]["ms_per_product"]
        B_local = algorithmic_bytes(inf.nnz_stored, nloc, n, 8, 8)
        kern_ms = res["fp64"]["early_parts_ms"] + res["fp64"]["late_parts_ms"]
        line = {"metric": "H*v/sec", "value": 1e3 / ms, "unit": "H*v/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": args.workload, "dim": n, "stored_entries": Z, "S_val": 8, "S_vec": 8,
                           "partition": "species-order row shards: whole up configurations, balanced by stored entries (nnz)",
                           "rows_per_rank": [bounds[q + 1] - bounds[q] for q in range(world)],
                           "exchange": "peer-memory pulls (CUDA IPC, copy engines, ring order) of the row ranges the late parts reference only, overlapped with the "
                                       "parts that need no remote data (local part + cross entries with own columns); the other cross entries after the arrival; "
                                       "device-side push all-reduce kernel as barrier (csrc/dist.cu: no NCCL in the loop)",
                           "vectors": "x = this rank's rows of vec_randomize(seed 1) in the internal order; fp64: the complex128 vectors of the reference's "
                                      "calling convention have imag == 0 (what the single-GPU MultMv detects); the complex128 product is reported beside it",
                           "n1_note": "the 1-GPU line includes the reference-order boundary (permutation in and out, 2.3 ms of its 16.9 ms); shards work in the internal order",
                           "l2": "inputs larger than L2"},
                "roofline": {"bound": "hbm", "achieved": B_local / (kern_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": B_local / (kern_ms * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "local_product_ms": kern_ms,
                             "note": "per GPU (rank 0's shard): both parts of the local rows' product without the exchange; the exchange is in `value`"},
                "e2e": {"value": 1.0 / res["e2e_s"], "unit": "H*v/s", "h2d_bytes_per_step": nloc * 8, "d2h_bytes_per_step": nloc * 8,
                        "ms_per_step": 1e3 * res["e2e_s"], "note": "per rank: its fp64 slice of x up, its slice of y down, pinned host memory"},
                "products": {k: v for k, v in res.items() if k in ("fp64", "complex128")},
                "gpu_launches": launches, "clocks": clocks, "host_phases": {"generate_shard_s": t_build}}
        if "lanczos" in res:
            line["lanczos"] = res["lanczos"]
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()


def bench_sharded(args, WORKLOADS, build_matrix, algorithmic_bytes, measured_peak, ClockSampler, workload_upper_nnz):
    """bench.py's N > 1 arm: H row-sharded over the ranks (strong scaling: the total work is fixed).  One product =
    exchange of x + the local rows' product, timed on the device, max over ranks.  Two exchange schemes are timed and the
    faster is the headline: (A) one all_gather then the whole shard, (B) one broadcast per owner overlapped with the
    per-owner column blocks."""
    if WORKLOADS[args.workload][0] == "hubbard" and not os.environ.get("QB_DIST_LEGACY"):
        return bench_sharded_species(args, WORKLOADS, algorithmic_bytes, measured_peak, ClockSampler)
    import torch
    import torch.distributed as dist
    import quantum_basis_b200 as qb
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    L = qb.lib()
    stream = torch.cuda.current_stream()          # bench.py installed a dedicated stream and handed it to the library
    fam, p = WORKLOADS[args.workload]
    if fam == "hubbard":
        n = L.qbgpu_dim_hubbard(p["Lx"] * p["Ly"], p["nup"], p["ndn"])
    else:
        n = L.qbgpu_dim_heisenberg(p["L"], p["L"] // 2)
    bounds, chunk = equal_row_bounds(n, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    t0 = time.time()
    M = build_matrix(qb, args.workload, row_range=(lo, hi))
    torch.cuda.synchronize()
    t_build = time.time() - t0
    inf = M.info
    comm = TorchComm()
    col_bounds = [min(n, q * chunk) for q in range(world)] + [n]
    t0 = time.time()
    parts = DeviceKernels.split(qb, M, col_bounds)
    torch.cuda.synchronize()
    t_split = time.time() - t0
    kern = DeviceKernels(qb, M, real=False, parts=parts)
    opA = ShardedOperator(kern, n, rank, world, comm)
    opB = PipelinedOperator(kern, n, rank, world, comm)
    x_loc = kern.alloc(chunk)
    y_loc = kern.alloc(chunk)
    y_ref = kern.alloc(chunk)
    full = qb.vec_randomize(n, 1)                  # generated on the device, sliced on the host
    x_loc[:2 * (hi - lo)] = torch.from_numpy(np.ascontiguousarray(full[lo:hi]).view(np.float64)).cuda()

    sampler = ClockSampler(local_rank)
    sampler.start()
    L.qbgpu_kernel_launches(1)
    msA = _timed(torch, dist, stream, lambda: opA.matvec(x_loc, y_ref), args.steps, args.warmup)
    launchesA = int(L.qbgpu_kernel_launches(1))
    msB = _timed(torch, dist, stream, lambda: opB.matvec(x_loc, y_loc), args.steps, args.warmup)
    launchesB = int(L.qbgpu_kernel_launches(1))
    agree = float((y_loc - y_ref).abs().max().item()) / max(1e-300, float(y_ref.abs().max().item()))
    # (C) peer-memory pulls over NVLink (copy engines, one stream per peer) overlapped with the column blocks
    msC, agreeC = None, None
    try:
        opC = PeerExchangeOperator(qb, kern, n, rank, world, comm, torch)
        opC.own(0).upload(np.ascontiguousarray(full[lo:hi]))
        comm.all_reduce(opC.token)
        y_c = kern.alloc(chunk)
        msC = _timed(torch, dist, stream, lambda: opC.matvec(0, y_c), args.steps, args.warmup)
        agreeC = float((y_c - y_ref).abs().max().item()) / max(1e-300, float(y_ref.abs().max().item()))
    except Exception as e:                                     # e.g. no peer access between the GPUs of this box
        msC, agreeC = None, f"unavailable: {e}"
    launchesC = int(L.qbgpu_kernel_launches(1))
    clocks = sampler.stop()
    # the local product alone (no exchange): the per-GPU roofline number
    opA.gather(x_loc)
    ms_kernel = _timed(torch, dist, stream, lambda: kern.multmv(opA.x_full, y_ref), max(3, args.steps // 2), 2)

    # e2e: host vectors -- every rank uploads its slice of x from pinned memory and downloads its slice of y
    xh = torch.empty(2 * chunk, dtype=torch.float64).pin_memory(); xh.copy_(x_loc.cpu())
    yh = torch.empty(2 * chunk, dtype=torch.float64).pin_memory()
    best = opB if msB < msA else opA
    use_peer = msC is not None and msC < min(msA, msB)
    nb_slice = (hi - lo) * 16

    def e2e_step():
        if use_peer:                       # host slice -> staging tensor -> this rank's exported buffer (all stream-ordered)
            x_loc.copy_(xh, non_blocking=True)
            assert L.qbgpu_memcpy_d2d(C.c_void_p(opC.own(0).ptr), C.c_void_p(x_loc.data_ptr()), nb_slice) == 0
            opC.matvec(0, y_c)
            yh.copy_(y_c, non_blocking=True)
        else:
            x_loc.copy_(xh, non_blocking=True)
            best.matvec(x_loc, y_loc)
            yh.copy_(y_loc, non_blocking=True)
    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize(); dist.barrier()
    te = time.time()
    ne = max(3, min(args.steps, 10))
    for _ in range(ne):
        e2e_step()
        torch.cuda.synchronize()
    dist.barrier()
    e2e_s = torch.tensor([(time.time() - te) / ne], dtype=torch.float64, device="cuda")
    dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_s.item())

    nnz_all = torch.tensor([inf.nnz_stored], dtype=torch.int64, device="cuda")
    dist.all_reduce(nnz_all)
    Z = int(nnz_all.item())
    s_val = 8 if inf.val_is_real else 16
    s_vec = 16
    ms_per_step = min(m for m in (msA, msB, msC) if m is not None)
    used = {msA: "allgather", msB: "pipelined_broadcast"}
    if msC is not None:
        used[msC] = "peer_pull"
    B_local = algorithmic_bytes(inf.nnz_stored, hi - lo, n, s_val, s_vec)
    peak, peak_src = measured_peak()

    # sharded Lanczos (real mode when the stored values are real: the start vector vec_randomize is real), fixed step
    # count: the rate is what is measured here; the stop rule lives in the single-GPU driver
    lan = None
    if not args.no_lanczos:
        real = bool(inf.val_is_real)
        kr = DeviceKernels(qb, M, real=real, parts=parts)
        oA = ShardedOperator(kr, n, rank, world, comm)
        oB = PipelinedOperator(kr, n, rank, world, comm)
        u0 = kr.alloc(chunk)
        if real:
            u0[: hi - lo] = torch.from_numpy(np.ascontiguousarray(full[lo:hi].real)).cuda()
        else:
            u0.copy_(x_loc)
        steps = 40
        out = {}
        try:
            oC = PeerExchangeOperator(qb, kr, n, rank, world, comm, torch)
        except Exception:
            oC = None
        schemes = [("allgather", sharded_lanczos, oA), ("pipelined", pipelined_lanczos, oB)]
        if oC is not None:
            schemes.append(("peer_pull", None, oC))
        for tag, fn, op in schemes:
            state = torch.zeros(8, dtype=torch.float64, device="cuda"); state[0] = 1.0
            a_dev = torch.zeros(256, dtype=torch.float64, device="cuda"); b_dev = torch.zeros(256, dtype=torch.float64, device="cuda")
            ua, ub = u0.clone(), kr.alloc(chunk)

            def run(nsteps):
                if tag == "peer_pull":
                    op.own(0).upload(u0[: kr.ncomp * (hi - lo)].cpu().numpy())
                    comm.all_reduce(op.token)
                    peer_lanczos(op, nsteps, state, a_dev, b_dev)
                else:
                    ua.copy_(u0)
                    fn(op, ua, ub, 256, nsteps, state, a_dev, b_dev)
            run(3)                                               # warm-up
            torch.cuda.synchronize(); dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            state[:] = 0.0; state[0] = 1.0
            if tag == "peer_pull":
                op.own(0).upload(u0[: kr.ncomp * (hi - lo)].cpu().numpy())
                comm.all_reduce(op.token)
            else:
                ua.copy_(u0)
            torch.cuda.synchronize(); dist.barrier()
            e0.record(stream)
            if tag == "peer_pull":
                peer_lanczos(op, steps, state, a_dev, b_dev)
            else:
                fn(op, ua, ub, 256, steps, state, a_dev, b_dev)
            e1.record(stream)
            torch.cuda.synchronize(); dist.barrier()
            t = torch.tensor([e0.elapsed_time(e1) * 1e-3], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            out[tag] = {"steps": steps, "seconds": float(t.item()), "iters_per_s": steps / float(t.item()),
                        "a0": float(a_dev[0].item()), "b1": float(b_dev[1].item()), "a_last": float(a_dev[steps - 1].item())}
        lan = {"vectors": "fp64 (real mode)" if real else "complex128", **out,
               "iters_per_s": max(v["iters_per_s"] for v in out.values())}
    del full

    if rank == 0:
        line = {"metric": "H*v/sec", "value": 1e3 / ms_per_step, "unit": "H*v/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": args.workload, "dim": n, "stored_entries": Z, "S_val": s_val, "S_vec": s_vec,
                           "partition": "contiguous equal-row blocks, full expanded rows per rank",
                           "exchange": {"allgather_ms": msA, "pipelined_broadcast_ms": msB, "peer_pull_ms": msC, "used": used[ms_per_step],
                                        "schemes_agree_rel": agree, "peer_pull_agree_rel": agreeC},
                           "l2": "inputs larger than L2"},
                "roofline": {"bound": "hbm", "achieved": B_local / (ms_kernel * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": B_local / (ms_kernel * 1e-3) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "local_product_ms": ms_kernel,
                             "note": "per GPU: the local rows' product alone (max over ranks); the exchange is in `value`, not here"},
                "e2e": {"value": 1.0 / e2e_s, "unit": "H*v/s", "h2d_bytes_per_step": (hi - lo) * s_vec, "d2h_bytes_per_step": (hi - lo) * s_vec,
                        "ms_per_step": 1e3 * e2e_s, "note": "per rank: its slice of x up, its slice of y down, pinned host memory"},
                "gpu_launches": launchesA + launchesB + launchesC, "clocks": clocks,
                "host_phases": {"generate_matrix_s": t_build, "split_columns_s": t_split}}
        if lan:
            line["lanczos"] = lan
        print(json.dumps(line))
    dist.barrier()
    dist.destroy_process_group()
