"""Row-sharded catalogs across the GPUs of one box (one process per GPU, NCCL over NVLink).

Catalog rows are independent and top-k is decomposable (global top-k ⊆ union of shard
top-k), so the path shards with ONE exchange step: every rank scores the replicated query
batch against its contiguous row block with the fused kernel, the per-rank [Q, k]
(score, global id) candidates are all-gathered, and K4 (``icr_topk_merge``) selects the global
top-k on every rank. The reference has no multi-GPU path at all (SURVEY §2.1); this is the
extension BASELINE.json's north_star defines for catalogs larger than one GPU.
"""

from __future__ import annotations

from typing import Callable

import numpy as np
import torch
import torch.distributed as dist

from . import _lib, ops
from .index import DeviceCatalog


def shard_bounds(n_rows: int, world_size: int, rank: int) -> tuple[int, int]:
    """Contiguous block [lo, hi) of rank `rank`: blocks of ceil(N/G) rows, the last ones may be short or empty."""
    per = (n_rows + world_size - 1) // world_size
    lo = min(n_rows, rank * per)
    return lo, min(n_rows, lo + per)


def pack_candidates(vals: torch.Tensor, ids: torch.Tensor) -> torch.Tensor:
    """[Q,k] f32 + [Q,k] i64 -> one int64 [2,Q,k] buffer (score bits in plane 0) for a single collective."""
    return torch.stack([vals.contiguous().view(torch.int32).to(torch.int64), ids.to(torch.int64)])


def unpack_candidates(buf: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """[G,2,Q,k] int64 -> (scores f32 [G,Q,k], ids i64 [G,Q,k])."""
    scores = buf[:, 0].to(torch.int32).view(torch.float32)
    return scores.contiguous(), buf[:, 1].contiguous()


class PeerExchange:
    """All-gather of [Q, k] candidates through NVLink peer memory (``icr_peer_exchange``) instead of NCCL.

    PyTorch's symmetric memory is the plumbing: it allocates one buffer per rank and maps every rank's buffer into
    every process; the exchange itself is one kernel of ours per call (peer stores + system-scope flags). Collective:
    every rank of `group` constructs it and calls ``all_gather`` with the same shapes in the same order (lockstep: the
    kernel of call e waits for every peer's call e). A rank that waits longer than ``ICR_PEER_TIMEOUT_S`` seconds (default
    600) for a peer gives up without poisoning its CUDA context: it records the call's epoch in the buffer header and
    ``check()`` - called at any host synchronisation point - raises. The results of such a call are invalid.
    """

    STATUS_OFFSET = 768  # csrc/exchange.cu kPeerStatusOff

    def __init__(self, group: dist.ProcessGroup | None, device: torch.device, max_candidates: int):
        import torch.distributed._symmetric_memory as symm

        self.group = group if group is not None else dist.group.WORLD
        self.world_size = dist.get_world_size(self.group)
        self.rank = dist.get_rank(self.group)
        if self.world_size > 16:
            raise ValueError("peer exchange supports up to 16 ranks (one NVLink domain)")
        self.device = torch.device(device)
        self.n_max = int(max_candidates)
        lib = _lib.load()
        nbytes = lib.icr_peer_buffer_bytes(self.n_max, self.world_size)
        with torch.cuda.device(self.device):
            self.buf = symm.empty(nbytes, dtype=torch.uint8, device=self.device)
            self.buf.zero_()
            self.handle = symm.rendezvous(self.buf, self.group)
        import ctypes

        self._ptrs = (ctypes.c_uint64 * self.world_size)(*[int(p) for p in self.handle.buffer_ptrs])
        self.epoch = 0
        torch.cuda.synchronize(self.device)
        dist.barrier(self.group)  # every buffer is zeroed before anyone's first push can land in it

    def check(self) -> None:
        """Raise if an exchange on this buffer timed out waiting for a peer (synchronises the device)."""
        failed = int(self.buf[self.STATUS_OFFSET : self.STATUS_OFFSET + 4].view(torch.int32).item())
        if failed:
            raise RuntimeError(f"peer exchange call {failed} on rank {self.rank} timed out waiting for a peer (ICR_PEER_TIMEOUT_S): "
                               "a rank died or the ranks are not calling in lockstep; results since that call are invalid")

    def next_call(self) -> tuple[int, int, int, int, int]:
        """Counts one exchange call and returns its (rank, world, pointer-array address, epoch, n_max) for ``ops.cos_topk(peer=)`` /
        ``ops.peer_exchange_merge``. Every rank must then make that call."""
        import ctypes

        self.epoch += 1
        return (self.rank, self.world_size, ctypes.addressof(self._ptrs), self.epoch, self.n_max)

    def exchange_merge(self, vals: torch.Tensor, ids: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
        """vals f32 [Q,k], ids i64 [Q,k] of this rank -> the global top-k per query on every rank, one kernel."""
        if vals.numel() > self.n_max:
            raise ValueError(f"peer exchange sized for {self.n_max} candidates per rank, got {vals.numel()}")
        return ops.peer_exchange_merge(vals, ids, self.next_call())

    def all_gather(self, vals: torch.Tensor, ids: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
        """vals f32 [Q,k], ids i64 [Q,k] -> (scores [G,Q,k], ids [G,Q,k]): views of this rank's buffer, valid until the
        call after next."""
        import ctypes

        vals, ids = vals.contiguous(), ids.contiguous()
        n = vals.numel()
        if n > self.n_max or vals.dtype != torch.float32 or ids.dtype != torch.int64 or ids.numel() != n:
            raise ValueError(f"peer exchange sized for {self.n_max} f32/i64 candidates per rank, got {n}")
        self.epoch += 1
        so, io = ctypes.c_size_t(0), ctypes.c_size_t(0)
        lib = _lib.load()
        with ops._on(self.device):
            _lib.check(lib.icr_peer_exchange(vals.data_ptr(), ids.data_ptr(), n, self.rank, self.world_size, ctypes.addressof(self._ptrs),
                                             self.epoch, self.n_max, ctypes.addressof(so), ctypes.addressof(io), ops._stream(self.device)))
        G = self.world_size
        scores = self.buf[so.value : so.value + G * n * 4].view(torch.float32).view(G, *vals.shape)
        gids = self.buf[io.value : io.value + G * n * 8].view(torch.int64).view(G, *ids.shape)
        return scores, gids


MAX_GLOBAL_ROWS = 2**32 - 1  # icr_topk_merge carries global ids in the 32-bit half of its candidate keys


class ShardedCatalog:
    """This rank's block of a row-sharded catalog plus the exchange + merge step.

    ``exchange="nccl"`` (default) all-gathers the packed candidates with NCCL; ``exchange="peer"`` pushes them
    straight into the peers' buffers over NVLink with ``icr_peer_exchange`` (one kernel, no NCCL launch) — same result.
    """

    def __init__(
        self,
        local_rows,
        *,
        row_offset: int,
        total_rows: int,
        group: dist.ProcessGroup | None = None,
        dtype: torch.dtype = torch.float32,
        device: torch.device | None = None,
        exchange: str = "nccl",
        _local_topk: Callable | None = None,
        _merge: Callable | None = None,
    ):
        if exchange not in ("nccl", "peer"):
            raise ValueError("exchange must be 'nccl' or 'peer'")
        self.exchange = exchange
        self._peer: PeerExchange | None = None
        self.group = group
        self.world_size = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.total_rows = int(total_rows)
        self.row_offset = int(row_offset)
        if self.total_rows >= MAX_GLOBAL_ROWS:
            # the K4 merge keys candidates by (score, 32-bit id): larger catalogs would return truncated ids silently
            raise ValueError(f"a sharded catalog holds at most {MAX_GLOBAL_ROWS - 1} rows in total (got {self.total_rows})")
        # test seams: the gloo/CPU tests of the host logic plug the oracle in here; product code never does
        self._local_topk = _local_topk
        self._merge = _merge
        if _local_topk is None:
            # an already resident shard (DeviceCatalog.from_index) is taken as is
            self.local = local_rows if isinstance(local_rows, DeviceCatalog) else DeviceCatalog(local_rows, device=device, dtype=dtype, row_offset=row_offset)
            self.n_local = len(self.local)
            self.device = self.local.device
        else:
            self.local = local_rows
            self.n_local = len(local_rows)
            self.device = torch.device("cpu") if device is None else device

    @classmethod
    def from_full(cls, embeddings, *, group=None, **kw) -> "ShardedCatalog":
        """Every rank holds (or can address) the full host matrix and keeps only its block."""
        ws = dist.get_world_size(group) if dist.is_initialized() else 1
        rk = dist.get_rank(group) if dist.is_initialized() else 0
        lo, hi = shard_bounds(len(embeddings), ws, rk)
        return cls(embeddings[lo:hi], row_offset=lo, total_rows=len(embeddings), group=group, **kw)

    @classmethod
    def from_index(cls, index, product_ids: list[str], *, group=None, dtype: torch.dtype = torch.float32,
                   device: torch.device | None = None, exchange: str = "nccl", **load_kw) -> "ShardedCatalog | None":
        """Every rank streams only ITS row block of a validated on-disk index into HBM (``DeviceCatalog.from_index``)."""
        ws = dist.get_world_size(group) if dist.is_initialized() else 1
        rk = dist.get_rank(group) if dist.is_initialized() else 0
        lo, hi = shard_bounds(len(product_ids), ws, rk)
        local = DeviceCatalog.from_index(index, product_ids, dtype=dtype, device=device, rows=(lo, hi), **load_kw)
        if local is None:
            return None
        return cls(local, row_offset=lo, total_rows=len(product_ids), group=group, dtype=dtype, device=device, exchange=exchange)

    def with_exchange(self, exchange: str) -> "ShardedCatalog":
        """The same resident shard behind the other candidate exchange ("nccl" / "peer"): for A/B measurements."""
        import copy

        other = copy.copy(self)
        if exchange not in ("nccl", "peer"):
            raise ValueError("exchange must be 'nccl' or 'peer'")
        other.exchange, other._peer = exchange, None
        return other

    def local_topk(self, queries, k: int, include_rows=None):
        """[Q,k] candidates of this shard with GLOBAL ids; short shards pad with (-inf, -1). ``include_rows``: per-query
        candidate lists of GLOBAL ids (``topk``); the shard ranks the entries that fall in its block."""
        kk = min(k, self.n_local)
        local_lists = None if include_rows is None else self._local_lists(include_rows)
        if self._local_topk is not None:
            if local_lists is None:
                vals, ids = self._local_topk(queries, self.local, kk, self.row_offset)
            else:
                vals, ids = self._local_topk(queries, self.local, kk, self.row_offset, include_rows=local_lists)
        elif kk > 0:
            vals, ids = self.local.topk(queries, kk, include_rows=local_lists)
        else:
            Q = queries.shape[0] if hasattr(queries, "shape") and len(queries.shape) == 2 else 1
            vals = torch.empty(Q, 0, dtype=torch.float32, device=self.device)
            ids = torch.empty(Q, 0, dtype=torch.int64, device=self.device)
        if kk < k:
            Q = vals.shape[0]
            vals = torch.cat([vals, torch.full((Q, k - kk), float("-inf"), dtype=torch.float32, device=vals.device)], dim=1)
            ids = torch.cat([ids, torch.full((Q, k - kk), -1, dtype=torch.int64, device=ids.device)], dim=1)
        return vals, ids

    def _local_lists(self, include_rows):
        """Global candidate lists -> this shard's local lists (global id - row_offset, ids outside the block dropped): Q
        arrays for Q iterables, or a CSR pair for a CSR pair."""
        lo, hi = self.row_offset, self.row_offset + self.n_local
        if isinstance(include_rows, tuple) and len(include_rows) == 2 and all(isinstance(t, torch.Tensor) for t in include_rows):
            offsets, rows = (t.to(torch.int64) for t in include_rows)
            keep = (rows >= lo) & (rows < hi)
            seg = torch.repeat_interleave(torch.arange(offsets.numel() - 1, device=rows.device), offsets[1:] - offsets[:-1])
            counts = torch.zeros(offsets.numel() - 1, dtype=torch.int64, device=rows.device).index_add_(0, seg[keep], torch.ones_like(seg[keep]))
            new_off = torch.zeros_like(offsets)
            new_off[1:] = torch.cumsum(counts, 0)
            return new_off, rows[keep] - lo
        out = []
        for r in include_rows:
            g = np.unique(np.asarray(list(r) if not isinstance(r, np.ndarray) else r, dtype=np.int64).reshape(-1))
            out.append(g[(g >= lo) & (g < hi)] - lo)
        return out

    def topk(self, queries, k: int, *, include_rows=None):
        """Global (values [Q,k'], ids [Q,k']) on every rank, k' = min(k, total rows).

        ``include_rows``: one candidate list of GLOBAL ids per query (Q iterables, or an ``(offsets, rows)`` CSR pair with
        distinct ids per list); query q ranks only its list. Each rank runs the subset search over the ids in its block and
        the candidates go through the usual exchange. Collective: every rank passes the same lists."""
        k = min(int(k), self.total_rows)
        if include_rows is not None:
            if k > ops.MAX_K:
                raise ValueError(f"k={k} outside [1, {ops.MAX_K}]")
            vals, ids = self.local_topk(queries, k, include_rows)
            return self.exchange_merge(vals, ids, k)
        if self.exchange == "peer" and self.world_size > 1 and self._local_topk is None and 1 <= k <= self.n_local:
            # one library call: the shard's search with the exchange and the merge behind it - a single launch for request-sized
            # batches (icr_cos_topk_sharded). Ranks whose shard is shorter than k take the route below; the protocols mix.
            q = self.local._device_queries(queries)
            return self.local.topk(q, k, peer=self._peer_for(q.shape[0] * k).next_call())
        vals, ids = self.local_topk(queries, k)
        return self.exchange_merge(vals, ids, k)

    def update_rows(self, global_rows, embeddings) -> None:
        """Replace catalog rows by GLOBAL id in place (``DeviceCatalog.update_rows``). Every rank makes the same call and
        applies the rows that fall in its block; no collective is needed. Appending and removing rows would move the shard
        boundaries, and with them the global ids, so a sharded catalog does not offer them."""
        g = np.asarray(global_rows.detach().cpu() if isinstance(global_rows, torch.Tensor) else global_rows, dtype=np.int64).reshape(-1)
        if g.size and (g.min() < 0 or g.max() >= self.total_rows):
            raise ValueError(f"global row ids must lie in [0, {self.total_rows})")
        if np.unique(g).size != g.size:
            raise ValueError("duplicate row ids")
        if len(embeddings) != g.size:
            raise ValueError(f"{g.size} rows but {len(embeddings)} embeddings")
        pick = np.flatnonzero((g >= self.row_offset) & (g < self.row_offset + self.n_local))
        if isinstance(embeddings, torch.Tensor):
            mine = embeddings[torch.from_numpy(pick).to(embeddings.device)]
        else:
            mine = np.asarray(embeddings)[pick]
        self.local.update_rows(g[pick] - self.row_offset, mine)

    def _peer_for(self, n: int) -> "PeerExchange":
        if self._peer is None or self._peer.n_max < n:
            self._peer = PeerExchange(self.group, self.device, max(n, 1 << 16))
        return self._peer

    def exchange_merge(self, vals: torch.Tensor, ids: torch.Tensor, k: int):
        """The collective half of ``topk``: every rank's [Q,k] candidates -> the global top-k on every rank."""
        if self.world_size == 1:
            return vals, ids
        if self.exchange == "peer":
            return self._peer_for(vals.numel()).exchange_merge(vals, ids)
        mine = pack_candidates(vals, ids)
        # output concatenated along dim 0 (the layout every backend's all_gather_into_tensor accepts)
        gathered = torch.empty((self.world_size * mine.shape[0], *mine.shape[1:]), dtype=mine.dtype, device=mine.device)
        dist.all_gather_into_tensor(gathered, mine, group=self.group)
        scores, gids = unpack_candidates(gathered.view(self.world_size, *mine.shape))
        merge = self._merge if self._merge is not None else ops.topk_merge
        return merge(scores, gids, k)
