"""Multi-GPU commit: one process per GPU, sharded by polynomial column, exchanged column->row, hashed by leaf range.

SURVEY.md §8(e) / BASELINE.json north_star:
  1. rank g runs the iNTT + coset LDE of its column slice  (gl_dev_lde; columns are independent polynomials);
  2. one all-to-all turns column slices into row slices: rank q receives, from every rank, the rows of its contiguous
     leaf range  [q*R/G, (q+1)*R/G)  — whole cap subtrees, because 2^cap_height >= G;
  3. rank q hashes its leaves and builds its 2^cap_height/G subtrees (gl_dev_merkle); the local digest buffer is exactly
     this rank's slice of plonky2's `digests` vector;
  4. the subtree roots are all-gathered into the MerkleCap.

`ShardPlan` is pure host arithmetic (tested on CPU with gloo, world_size 2); `ShardedCommit` needs CUDA + NCCL.
torch.distributed is plumbing only: the exchange is `all_to_all_single` on device buffers the library filled.
"""
from __future__ import annotations

import ctypes
import time
from typing import List, Tuple

import numpy as np


def _round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


class ShardPlan:
    """Who owns which columns (LDE stage) and which leaf rows (Merkle stage), and the all-to-all split sizes."""

    def __init__(self, n_cols: int, log_n: int, rate_bits: int, cap_height: int, world: int):
        if world < 1 or world & (world - 1):
            raise ValueError("world size must be a power of two")
        if (1 << cap_height) < world:
            raise ValueError("cap_height too small: every rank must own at least one whole cap subtree")
        if n_cols < world:
            raise ValueError("fewer columns than ranks")
        self.n_cols, self.log_n, self.rate_bits, self.cap_height, self.world = n_cols, log_n, rate_bits, cap_height, world
        self.n_rows = 1 << (log_n + rate_bits)               # R
        self.rows_per_rank = self.n_rows // world
        self.local_cap_height = cap_height - (world.bit_length() - 1)
        # Columns are dealt in groups of 4 (32 bytes of a leaf row) so that every rank's column offset is sector aligned: the
        # fused exchange stores whole 32-byte sectors into the owners' leaf buffers (a rank starting at an odd multiple of
        # 16 bytes was measured 1.5x slower: two partial sectors per segment over NVLink).  The NTTs work on 4-column
        # groups anyway, so the padded work per rank is the same as for an even per-column split.
        n_groups = (n_cols + 3) // 4
        if n_groups >= world:
            base, rem = divmod(n_groups, world)
            groups = [base + (1 if g < rem else 0) for g in range(world)]
            self.col_counts = [4 * k for k in groups]
            self.col_counts[-1] -= 4 * n_groups - n_cols          # the last group may be partial
        else:                                                     # very narrow batches: plain even split
            base, rem = divmod(n_cols, world)
            self.col_counts = [base + (1 if g < rem else 0) for g in range(world)]
        self.col_offsets = [sum(self.col_counts[:g]) for g in range(world)]
        # device pitch of a rank's LDE output: multiple of 4 words (see gl_dev_lde), of 8 when that wastes < 4 columns
        self.pitches = [_round_up(c, 8) if _round_up(c, 8) - c < 4 else _round_up(c, 4) for c in self.col_counts]
        self.leaf_pitch = _round_up(n_cols, 8)

    def col_range(self, rank: int) -> Tuple[int, int]:
        return self.col_offsets[rank], self.col_offsets[rank] + self.col_counts[rank]

    def row_range(self, rank: int) -> Tuple[int, int]:
        return rank * self.rows_per_rank, (rank + 1) * self.rows_per_rank

    def send_splits(self, rank: int) -> List[int]:
        """words sent by `rank` to each peer: its rows_per_rank x pitch[rank] slab of that peer's leaf range"""
        return [self.rows_per_rank * self.pitches[rank]] * self.world

    def recv_splits(self, rank: int) -> List[int]:
        return [self.rows_per_rank * self.pitches[q] for q in range(self.world)]

    # ---- streamed coset plan (include/gl_commit.h · gl_commit_coset_stream): columns dealt cyclically in groups of gw, waves of G groups ----
    def stream_group_width(self) -> int:
        """8-column groups when that still leaves >= 4 waves to pipeline (the NTT's preferred tile), else 4"""
        return 8 if self.n_cols >= 4 * 8 * self.world or self.world == 1 else 4

    def stream_waves(self) -> int:
        gw = self.stream_group_width()
        n_groups = (self.n_cols + gw - 1) // gw
        return (n_groups + self.world - 1) // self.world

    def stream_columns(self, rank: int) -> List[int]:
        """global indices of the columns rank `rank` supplies to the streamed plan, in the order it supplies them (wave by wave)"""
        gw = self.stream_group_width()
        out = []
        for w in range(self.stream_waves()):
            g0 = gw * (w * self.world + rank)
            out.extend(range(g0, min(g0 + gw, self.n_cols)))
        return out

    def digests_per_rank(self) -> int:
        return 2 * (self.rows_per_rank - (1 << self.local_cap_height))

    def exchange_bytes_per_rank(self) -> int:
        """algorithmic bytes a rank sends to OTHER ranks (8*C_g*R*(G-1)/G)"""
        return 8 * self.rows_per_rank * (self.world - 1) * max(self.col_counts)


def coset_blocks_of_rank(plan: ShardPlan, rank: int) -> List[Tuple[int, int]]:
    """Coset-sharded plan: the (leaf block, LDE coset) pairs rank `rank` evaluates.  Leaf rows are stored in bit-reversed LDE order, so leaf
    block b (rows [b*N, (b+1)*N)) is exactly coset s = bitrev_r(b) — the points 7 * w_R^s * w_N^m — in the in-place-DIF order of m; a rank
    owns 2^r / G consecutive blocks (its contiguous leaf range = whole cap subtrees)."""
    n_cosets = 1 << plan.rate_bits
    if plan.world > n_cosets:
        raise ValueError("coset sharding needs world <= 2^rate_bits")
    per = n_cosets // plan.world
    rev = lambda b: int(format(b, "0%db" % plan.rate_bits)[::-1], 2) if plan.rate_bits else 0
    return [(b, rev(b)) for b in range(rank * per, (rank + 1) * per)]


def exchange_reference(plan: ShardPlan, shards: List[np.ndarray]) -> List[np.ndarray]:
    """Host model of step 2 for tests: shards[g] is rank g's [R][pitch_g] LDE output; returns each rank's [R/G][n_cols] leaves."""
    out = []
    for q in range(plan.world):
        r0, r1 = plan.row_range(q)
        out.append(np.concatenate([shards[g][r0:r1, :plan.col_counts[g]] for g in range(plan.world)], axis=1))
    return out


class ShardedCommit:
    """Device buffers + the four steps above for one rank.  Buffers are allocated once and reused by every commit.

    exchange="p2p" (default when the ranks can map each other's memory): steps 1 and 2 are one call — gl_dev_lde_scatter /
    gl_lde_scatter deliver every coset's rows into the owners' leaf buffers over NVLink (buffers exported/mapped with CUDA IPC)
    while the next coset's NTT runs (DESIGN.md §6: the rank's own cosets are stored by the NTT, the others shipped by the copy
    engines), so there is no all-to-all, no receive buffer and no repacking; the ranks only meet at a stream-ordered
    1-element all-reduce before hashing.  exchange="nccl": gl_dev_lde + all_to_all_single + gl_dev_repack (the baseline the
    fused path is measured against, and the collective fallback when peer mapping is unavailable).
    exchange="coset" (what "auto" picks for device-resident columns when world <= 2^rate_bits): the ranks exchange COEFFICIENT blocks and
    every rank evaluates only its own cosets (gl_dev_intt + gl_dev_lde_own_cosets).  exchange="stream" (what "auto" picks for HOST columns,
    commit_host only): the coset plan cut into waves and fused with the leaf sponge (gl_commit_coset_stream) — the columns are dealt
    cyclically, so ask host_columns() which ones this rank supplies."""

    def __init__(self, ctx, plan: ShardPlan, rank: int, dist, torch, exchange: str = "auto"):
        self.ctx, self.plan, self.rank, self.dist, self.torch = ctx, plan, rank, dist, torch
        dev = torch.device("cuda", ctx.device)
        p = plan
        i64 = torch.int64
        self._host_impl = None
        self._auto = exchange == "auto"
        if exchange == "auto":      # coset sharding whenever every rank can own whole cosets, else the column->row shipment
            exchange = "coset" if p.world <= (1 << p.rate_bits) else "p2p"
        self.exchange = exchange
        self.coeffs = torch.empty((1 << p.log_n) * p.pitches[rank], dtype=i64, device=dev)  # [N][pitch_g]
        self.digests = torch.empty(max(p.digests_per_rank() * 4, 1), dtype=i64, device=dev)
        self.cap_local = np.zeros(4 << p.local_cap_height, dtype=np.uint64)
        self.cap_dev = torch.empty(4 << p.local_cap_height, dtype=i64, device=dev)
        self.cap_all = torch.empty(4 << p.cap_height, dtype=i64, device=dev)
        self.exchange_ms = 0.0
        self.phase_ms = {}
        self._merkle_call_ms = 0.0
        self._peer_ptrs = None
        self._stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
        # leaf row i = LDE point bitrev(i): the rows of rank q are those of cosets bitrev_r(j), j in [q*2^r/G, (q+1)*2^r/G)
        # (G <= 2^r), so starting rank q at coset bitrev_r(q*2^r/G) makes every rank store into its OWN buffer first and into
        # a different owner than any other rank at every later step
        n_cosets = 1 << p.rate_bits
        j = (rank * n_cosets // p.world) % n_cosets
        self._first_coset = int(format(j, "0%db" % p.rate_bits)[::-1], 2) if p.rate_bits else 0
        self._flag = torch.zeros(1, dtype=torch.int32, device=dev)
        self._coeff_ptr = None
        self._epoch = 0
        if exchange == "stream":
            if p.world <= (1 << p.rate_bits) and p.n_cols > 4 and self._init_stream(dev):
                return
            self.exchange = exchange = "p2p"
        if exchange == "coset" and p.world <= (1 << p.rate_bits) and self._init_coset(dev):
            return
        if exchange == "coset":
            self.exchange = exchange = "p2p"
        if exchange == "p2p" and self._init_p2p(dev):
            return
        self.exchange = "nccl"      # requested, or the ranks cannot map each other's memory (all ranks agree on this)
        self.rows = torch.empty(p.n_rows * p.pitches[rank], dtype=i64, device=dev)          # [R][pitch_g]
        self.recv = torch.empty(sum(p.recv_splits(rank)), dtype=i64, device=dev)
        self.leaves = torch.zeros(p.rows_per_rank * p.leaf_pitch, dtype=i64, device=dev)    # [R/G][leaf_pitch]
        self.leaves_ptr = self.leaves.data_ptr()

    def _init_coset(self, dev) -> bool:
        """Coset-sharded plan (include/gl_commit.h · gl_dev_lde_own_cosets): export this rank's COEFFICIENT block, map every peer's, and
        allocate local staging for the peers' blocks and the own leaf range.  Collective; False on every rank if any rank failed."""
        p, torch = self.plan, self.torch
        n = 1 << p.log_n
        if not self._map_peers(dev, n * p.pitches[self.rank]):
            return False
        self._coeff_ptr, self._peer_coeffs = self.leaves_ptr, self._peer_ptrs     # the exported buffer holds coefficients in this mode
        self._peer_ptrs = None
        self._stage = [None if q == self.rank else torch.empty(n * p.pitches[q], dtype=torch.int64, device=dev) for q in range(p.world)]
        self._stage_ptrs = (ctypes.c_void_p * p.world)(*[0 if t is None else t.data_ptr() for t in self._stage])
        u32 = ctypes.c_uint32 * p.world
        self._pitches, self._counts, self._offsets = u32(*p.pitches), u32(*p.col_counts), u32(*p.col_offsets)
        self.leaves = torch.zeros(p.rows_per_rank * p.leaf_pitch, dtype=torch.int64, device=dev)
        self.leaves_ptr = self.leaves.data_ptr()
        return True

    def _init_stream(self, dev) -> bool:
        """Streamed coset plan (include/gl_commit.h · gl_commit_coset_stream): one exported buffer per rank (coefficient groups + ticket words),
        local staging for the pulled groups, the own leaf range.  Collective; False on every rank if any rank failed."""
        from ._lib import StreamPlan
        p, torch, lib = self.plan, self.torch, self.ctx.lib
        self._splan = StreamPlan(p.n_cols, p.log_n, p.rate_bits, p.local_cap_height, p.world, self.rank, p.stream_group_width(), p.leaf_pitch, 0)
        exported, stage, waves, n_own = ctypes.c_uint64(), ctypes.c_uint64(), ctypes.c_uint32(), ctypes.c_uint32()
        self._check(lib.gl_stream_plan_sizes(ctypes.byref(self._splan), ctypes.byref(exported), ctypes.byref(stage), ctypes.byref(waves),
                                             ctypes.byref(n_own)))
        assert waves.value == p.stream_waves() and n_own.value == len(p.stream_columns(self.rank))
        if not self._map_peers(dev, exported.value):
            return False
        self._coeff_ptr, self._peer_coeffs = self.leaves_ptr, self._peer_ptrs     # the exported buffer holds coefficient groups + tickets
        self._peer_ptrs = None
        self._stage_all = torch.empty(stage.value, dtype=torch.int64, device=dev)
        self.leaves = torch.zeros(p.rows_per_rank * p.leaf_pitch, dtype=torch.int64, device=dev)
        self.leaves_ptr = self.leaves.data_ptr()
        return True

    def _init_p2p(self, dev) -> bool:
        """Export this rank's leaf buffer and map every peer's (CUDA IPC).  Collective; returns False on EVERY rank if any
        rank failed (no IPC in this container, no peer access), after releasing whatever was mapped."""
        p = self.plan
        return self._map_peers(dev, p.rows_per_rank * p.leaf_pitch)

    def _map_peers(self, dev, words) -> bool:
        p, lib, h, torch, dist = self.plan, self.ctx.lib, self.ctx.handle, self.torch, self.dist
        own = ctypes.c_void_p()
        handle = (ctypes.c_uint8 * 64)()
        ok = lib.gl_dev_ipc_alloc(h, words, ctypes.byref(own), handle) == 0
        mine = torch.tensor(list(handle) + [1 if ok else 0], dtype=torch.uint8, device=dev)
        allh = torch.empty(65 * p.world, dtype=torch.uint8, device=dev)
        dist.all_gather_into_tensor(allh, mine)
        allh = allh.cpu().numpy().reshape(p.world, 65)
        ptrs, opened = [], []
        ok = bool(allh[:, 64].all())
        if ok:
            for q in range(p.world):
                if q == self.rank:
                    ptrs.append(own.value)
                    continue
                hq = (ctypes.c_uint8 * 64)(*allh[q, :64].tolist())
                pq = ctypes.c_void_p()
                if lib.gl_dev_ipc_open(h, hq, ctypes.byref(pq)) != 0:
                    ok = False
                    break
                ptrs.append(pq.value)
                opened.append(pq.value)
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            for ptr in opened:
                lib.gl_dev_ipc_close(h, ptr)
            dist.barrier()
            if own.value:
                lib.gl_dev_ipc_free(h, own.value)
            return False
        self.leaves_ptr = own.value
        self._peer_ptrs = (ctypes.c_void_p * p.world)(*ptrs)
        dist.barrier()
        return True

    def close(self):
        if self._host_impl is not None:
            self._host_impl.close()
            self._host_impl = None
        mapped = self._peer_ptrs if self._peer_ptrs is not None else getattr(self, "_peer_coeffs", None)
        if mapped is not None:
            lib, h = self.ctx.lib, self.ctx.handle
            own = self._coeff_ptr if self._coeff_ptr is not None else self.leaves_ptr
            self.dist.barrier()
            for q, ptr in enumerate(mapped):
                if q != self.rank:
                    lib.gl_dev_ipc_close(h, ptr)
            self.dist.barrier()
            lib.gl_dev_ipc_free(h, own)
            self._peer_ptrs = self._peer_coeffs = None

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(self.ctx.lib.gl_ctx_last_error(self.ctx.handle).decode())

    def commit(self, d_cols) -> np.ndarray:
        """d_cols: this rank's [n_cols_g][N] device tensor (column-major, int64 storage of u64 words).  Returns the full cap."""
        p, lib, h, torch = self.plan, self.ctx.lib, self.ctx.handle, self.torch
        n = 1 << p.log_n
        ncg = p.col_counts[self.rank]
        assert d_cols.shape == (ncg, n) and d_cols.is_contiguous()
        t0 = time.perf_counter()
        if self.exchange == "stream":
            raise ValueError("the streamed plan takes HOST columns (commit_host); device-resident columns use exchange='coset'")
        if self.exchange == "coset":
            # iNTT of the own column shard into the exported coefficient block; a stream-ordered 1-element all-reduce tells every rank
            # that all blocks are complete; then pull + evaluate the own cosets of every block (pulls overlap the NTTs).  Nobody rewrites
            # its block before all peers have pulled it: the next commit starts after the cap all-gather, which a rank enters only after
            # its own hashing, i.e. after its pulls.
            self._check(lib.gl_dev_intt(h, d_cols.data_ptr(), n, ncg, p.log_n, 0, self._coeff_ptr, p.pitches[self.rank]))
            return self._coset_tail()
        if self.exchange == "p2p":
            # Nobody may write into a leaf buffer its owner is still hashing: the previous commit ended with the cap
            # all-gather, which no rank enters before its own hashing is done, and every rank read its result — so all
            # leaf buffers are free here without a further barrier (the first commit follows _init_p2p's barrier).
            self._check(lib.gl_dev_lde_scatter(h, d_cols.data_ptr(), n, ncg, p.log_n, p.rate_bits, 0, self._peer_ptrs, p.world,
                                               p.leaf_pitch, p.col_offsets[self.rank], self.coeffs.data_ptr(), p.pitches[self.rank],
                                               self._first_coset))
            # device-side barrier on the library's stream: a 1-element all-reduce completes only after every rank's scatter
            # kernels (stream order), and the hashing kernels queue behind it — no host round trip
            t1 = time.perf_counter()
            with torch.cuda.stream(self._stream):
                self.dist.all_reduce(self._flag)
            t2 = time.perf_counter()
            out = self._hash()
            t3 = time.perf_counter()
            self.phase_ms = {"lde_scatter_call": (t1 - t0) * 1e3, "barrier_enqueue": (t2 - t1) * 1e3, "hash_and_cap_gather": (t3 - t2) * 1e3,
                             "merkle_call": self._merkle_call_ms}
            return out
        self._check(lib.gl_dev_lde(h, d_cols.data_ptr(), n, ncg, p.log_n, p.rate_bits, 0, self.rows.data_ptr(), p.pitches[self.rank],
                                   self.coeffs.data_ptr()))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        self.dist.all_to_all_single(self.recv, self.rows, p.recv_splits(self.rank), p.send_splits(self.rank))
        e1.record()
        torch.cuda.current_stream().synchronize()
        self.exchange_ms = e0.elapsed_time(e1)
        off = 0
        for q in range(p.world):
            self._check(lib.gl_dev_repack(h, self.recv.data_ptr() + 8 * off, p.pitches[q], p.col_counts[q], p.rows_per_rank,
                                          self.leaves_ptr, p.leaf_pitch, p.col_offsets[q]))
            off += p.rows_per_rank * p.pitches[q]
        return self._hash()

    def _coset_tail(self) -> np.ndarray:
        """coset plan after the own coefficient block is complete: barrier, pull + own cosets, hash, cap gather"""
        p, lib, h, torch = self.plan, self.ctx.lib, self.ctx.handle, self.torch
        with torch.cuda.stream(self._stream):
            self.dist.all_reduce(self._flag)
        self._check(lib.gl_dev_lde_own_cosets(h, self._peer_coeffs, self._stage_ptrs, self._pitches, self._counts, self._offsets, p.world,
                                              self.rank, p.log_n, p.rate_bits, self.leaves_ptr, p.leaf_pitch))
        return self._hash()

    def commit_host(self, h_cols) -> np.ndarray:
        """The same commit from HOST columns: h_cols = this rank's [n_cols_g][N] tensor in (ideally pinned) host memory.  In the
        fused mode the shard crosses PCIe in chunks behind the NTTs of the previous chunk (gl_lde_scatter)."""
        p, lib, h, torch = self.plan, self.ctx.lib, self.ctx.handle, self.torch
        n = 1 << p.log_n
        if self._auto:
            # HOST columns: in the coset plan nothing can start before every rank's whole shard has crossed PCIe and gone through the iNTT,
            # so with exchange="auto" host inputs take the STREAMED coset plan (gl_commit_coset_stream: copies, pulls and NTTs of wave w+1
            # run while wave w is hashed), or the column->row plan when there are more ranks than cosets / peer mapping fails.  The
            # buffers are created on first use and kept.
            impl = self._host()
            out = impl.commit_host(h_cols)
            self.digests = impl.digests
            return out
        ncg = len(self.host_columns())
        assert tuple(h_cols.shape) == (ncg, n) and h_cols.is_contiguous() and not h_cols.is_cuda
        if self.exchange == "stream":
            base = h_cols.data_ptr()
            ptrs = (ctypes.c_void_p * max(ncg, 1))(*[base + 8 * n * j for j in range(ncg)])
            self._splan.epoch = self._epoch
            self._epoch += 1
            self._check(lib.gl_commit_coset_stream(h, ctypes.byref(self._splan), ptrs, 0, self._peer_coeffs, self._stage_all.data_ptr(),
                                                   self.leaves_ptr, self.digests.data_ptr(), self.cap_local.ctypes.data))
            return self._gather_cap()
        if self.exchange == "coset":
            base = h_cols.data_ptr()
            ptrs = (ctypes.c_void_p * ncg)(*[base + 8 * n * j for j in range(ncg)])
            self._check(lib.gl_intt_host(h, ptrs, ncg, p.log_n, 0, self._coeff_ptr, p.pitches[self.rank]))   # chunked H2D behind the iNTTs
            return self._coset_tail()
        if self.exchange != "p2p":
            d = h_cols.to(torch.device("cuda", self.ctx.device), non_blocking=True)
            torch.cuda.current_stream().synchronize()
            return self.commit(d)
        base = h_cols.data_ptr()
        ptrs = (ctypes.c_void_p * ncg)(*[base + 8 * n * j for j in range(ncg)])
        self._check(lib.gl_lde_scatter(h, ptrs, ncg, p.log_n, p.rate_bits, 0, self._peer_ptrs, p.world, p.leaf_pitch,
                                       p.col_offsets[self.rank], self.coeffs.data_ptr(), p.pitches[self.rank], self._first_coset))
        with torch.cuda.stream(self._stream):
            self.dist.all_reduce(self._flag)
        return self._hash()

    def _host(self):
        """exchange="auto": the implementation behind commit_host (collective on first use)"""
        if self._host_impl is None:
            self._host_impl = ShardedCommit(self.ctx, self.plan, self.rank, self.dist, self.torch, exchange="stream")
        return self._host_impl

    def host_columns(self) -> List[int]:
        """Global indices of the columns this rank passes to commit_host, in order (collective on first use with exchange="auto": the
        streamed plan deals columns cyclically, the other plans use the contiguous ShardPlan.col_range)."""
        impl = self._host() if self._auto else self
        if impl.exchange == "stream":
            return self.plan.stream_columns(self.rank)
        return list(range(*self.plan.col_range(self.rank)))

    def _hash(self) -> np.ndarray:
        p, lib, h, torch = self.plan, self.ctx.lib, self.ctx.handle, self.torch
        t0 = time.perf_counter()
        self._check(lib.gl_dev_merkle(h, self.leaves_ptr, p.rows_per_rank, p.n_cols, p.leaf_pitch, p.local_cap_height,
                                      self.digests.data_ptr(), self.cap_local.ctypes.data))
        self._merkle_call_ms = (time.perf_counter() - t0) * 1e3
        return self._gather_cap()

    def _gather_cap(self) -> np.ndarray:
        torch = self.torch
        with torch.cuda.stream(self._stream):
            self.cap_dev.copy_(torch.from_numpy(self.cap_local.view(np.int64)))
            self.dist.all_gather_into_tensor(self.cap_all, self.cap_dev)
            return self.cap_all.cpu().numpy().view(np.uint64)
