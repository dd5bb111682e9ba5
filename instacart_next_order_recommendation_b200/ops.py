"""Tensor-level wrappers over the C ABI: CUDA tensors in, CUDA tensors out.

PyTorch is plumbing here (device memory from the caching allocator, the current stream);
the arithmetic runs in libicr_b200.so. Non-CUDA tensors raise: there is no fallback.
"""

from __future__ import annotations

import contextlib

import torch

from . import _lib
from ._lib import ICR_BF16, ICR_F16, ICR_F32, MAX_K, PATH_AUTO, PATH_GEMM, PATH_GEMV, PATH_WS_RESIDENT  # noqa: F401

_DTYPES = {torch.float32: ICR_F32, torch.bfloat16: ICR_BF16, torch.float16: ICR_F16}


def _dtype_code(t: torch.Tensor) -> int:
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError(f"libicr_b200 supports float32, bfloat16 and float16 embeddings, got {t.dtype}") from None


def _require_cuda(name: str, t: torch.Tensor) -> None:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the retrieval path runs only as sm_100a kernels (no CPU fallback)")


def _rows(t: torch.Tensor) -> torch.Tensor:
    """2-D, contiguous in the embedding dimension (row stride may exceed dim)."""
    if t.dim() != 2:
        raise ValueError(f"expected a [rows, dim] matrix, got shape {tuple(t.shape)}")
    vec = 16 // t.element_size()
    if t.shape[1] % vec:
        # zero columns change neither dot products nor norms; they make rows 16-byte multiples
        t = torch.nn.functional.pad(t, (0, vec - t.shape[1] % vec))
    if t.shape[1] > 0 and (t.stride(1) != 1 or (t.shape[0] > 1 and (t.stride(0) < t.shape[1] or t.stride(0) % vec))):
        t = t.contiguous()
    if t.data_ptr() % 16:
        t = t.clone(memory_format=torch.contiguous_format)
    return t


_NULL_CTX = contextlib.nullcontext()


def _on(device: torch.device):
    """Device guard that costs nothing in the common case (the tensor's device is already current)."""
    if device.index is None or device.index == torch.cuda.current_device():
        return _NULL_CTX
    return torch.cuda.device(device)


def _ld(t: torch.Tensor) -> int:
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]


def _stream(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def _workspace(nbytes: int, device) -> torch.Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _ptr(t):
    return None if t is None else t.data_ptr()


def last_launch_count() -> int:
    return _lib.load().icr_last_launch_count()


def kernel_timing(step_fn, steps: int, flush: torch.Tensor | None = None) -> dict:
    """Run `step_fn` `steps` times with the library timing its dominant kernel (CUDA events on the launch stream)."""
    import ctypes

    lib = _lib.load()
    torch.cuda.synchronize()
    lib.icr_profile_enable(1)
    total, n_launch = 0.0, 0
    kid, terms = ctypes.c_int(0), ctypes.c_int(1)
    try:
        for _ in range(steps):
            if flush is not None:
                flush.zero_()
            step_fn()
            ms, n = ctypes.c_float(0), ctypes.c_int(0)
            _lib.check(lib.icr_profile_collect(ctypes.byref(ms), ctypes.byref(n), ctypes.byref(kid), ctypes.byref(terms)))
            total += ms.value
            n_launch += n.value
    finally:
        lib.icr_profile_enable(0)
    return {
        "kernel": {1: "gemv_topk", 2: "gemm_topk"}.get(kid.value, "none"),
        "ms_per_step": total / max(steps, 1),
        "ms_per_launch": total / max(n_launch, 1),
        "launches_per_step": n_launch / max(steps, 1),
        "mma_terms": terms.value,
    }


def row_inv_norms(x: torch.Tensor) -> torch.Tensor:
    """inv[r] = 1 / max(||x_r||, 1e-12) as f32 [rows]."""
    _require_cuda("x", x)
    x = _rows(x)
    lib = _lib.load()
    out = torch.empty(x.shape[0], dtype=torch.float32, device=x.device)
    with _on(x.device):
        _lib.check(lib.icr_row_inv_norms(x.data_ptr(), x.shape[0], x.shape[1], _ld(x), _dtype_code(x), out.data_ptr(), _stream(x.device)))
    return out


def split_f16_planes(x: torch.Tensor) -> torch.Tensor:
    """fp32 [rows, D] -> normalised fp16 (hi | lo) planes [rows, 2*round_up(D,64)] (tensor-path operand)."""
    _require_cuda("x", x)
    if x.dtype != torch.float32:
        raise TypeError("split_f16_planes expects float32 rows")
    x = _rows(x)
    lib = _lib.load()
    planes = torch.empty(x.shape[0], lib.icr_planes_row_elems(x.shape[1]), dtype=torch.float16, device=x.device)
    with _on(x.device):
        _lib.check(lib.icr_split_f16_planes(x.data_ptr(), x.shape[0], x.shape[1], _ld(x), planes.data_ptr(), _stream(x.device)))
    return planes


def screen_plane(x: torch.Tensor, *, with_inv_norms: bool = True):
    """fp32 [rows, D] -> (fp16 screening plane [rows, round_up(D,64)] of the normalised rows x 256, f32 inverse norms [rows] or None).

    The operand of the tensor-core top-k sweep over an fp32 catalog; the sweep's survivors are re-scored exactly from `x`."""
    _require_cuda("x", x)
    if x.dtype != torch.float32:
        raise TypeError("screen_plane expects float32 rows")
    x = _rows(x)
    lib = _lib.load()
    plane = torch.empty(x.shape[0], lib.icr_screen_plane_row_elems(x.shape[1]), dtype=torch.float16, device=x.device)
    inv = torch.empty(x.shape[0], dtype=torch.float32, device=x.device) if with_inv_norms else None
    with _on(x.device):
        _lib.check(lib.icr_screen_plane(x.data_ptr(), x.shape[0], x.shape[1], _ld(x), plane.data_ptr(), _ptr(inv), _stream(x.device)))
    return plane, inv


def convert_rows(x: torch.Tensor, out: torch.Tensor, *, normalize: bool = False) -> torch.Tensor:
    """fp32 device rows -> `out` (float32, bfloat16 or float16 device rows of the same shape), optionally L2-normalised
    first. The rounding is round-to-nearest-even, bit for bit torch's ``.to(out.dtype)``."""
    _require_cuda("x", x)
    _require_cuda("out", out)
    if x.dtype != torch.float32 or x.dim() != 2 or out.shape != x.shape or x.stride(1) != 1 or out.stride(1) != 1:
        raise ValueError("convert_rows expects float32 [rows, dim] input and an output of the same shape, both contiguous in dim")
    lib = _lib.load()
    with _on(x.device):
        _lib.check(lib.icr_convert_rows(x.data_ptr(), x.shape[0], x.shape[1], _ld(x), out.data_ptr(), _ld(out), _dtype_code(out), int(normalize),
                                        _stream(x.device)))
    return out


def normalized_f16(x: torch.Tensor) -> torch.Tensor:
    """Device rows -> float16 [rows, round_up(dim, 8)]: L2-normalised in fp32, then rounded (one ``icr_convert_rows``).

    The form queries take against a float16 catalog. Cosine does not depend on a row's scale, while a plain
    ``.to(float16)`` of un-normalised fp32 rows overflows to inf or flushes to zero. The padding columns are zero."""
    _require_cuda("x", x)
    if x.dim() != 2:
        raise ValueError(f"expected a [rows, dim] matrix, got shape {tuple(x.shape)}")
    x = x.float()
    if x.shape[1] % 8:
        x = torch.nn.functional.pad(x, (0, 8 - x.shape[1] % 8))
    x = _rows(x)
    return convert_rows(x, torch.empty(x.shape, dtype=torch.float16, device=x.device), normalize=True)


def _like_catalog(q: torch.Tensor, catalog_dtype: torch.dtype) -> torch.Tensor:
    """Queries in the catalog's dtype: float16 catalogs take normalised-then-rounded queries (``normalized_f16``)."""
    if q.dtype == catalog_dtype:
        return q
    return normalized_f16(q) if catalog_dtype == torch.float16 else q.to(catalog_dtype)


def exclusion_words(n_rows: int) -> int:
    """Words per query of a per-query exclusion bitmap over `n_rows` catalog rows: ceil(n_rows / 32)."""
    return (int(n_rows) + 31) // 32


def query_exclusion_bits(rows_per_query, n_rows: int, device=None) -> torch.Tensor:
    """Per-query exclusion bitmap uint32 [ceil(n_rows/32), Q] for ``cos_topk(..., exclude_bits=...)``.

    `rows_per_query` is a sequence of Q iterables of catalog rows (local rows, before any row offset), or a CSR pair
    ``(offsets [Q+1], rows)`` of int64 tensors. Any order, duplicates allowed; rows outside [0, n_rows) are ignored.
    Row r is excluded for query q when bit r % 32 of ``bits[r // 32, q]`` is set. Built on the device
    (``icr_query_exclusion_bits``); a bitmap can be reused by every call with the same queries' exclusions."""
    import numpy as np

    n_rows = int(n_rows)
    if n_rows < 0:
        raise ValueError("n_rows must be >= 0")
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    if dev.type != "cuda":
        raise RuntimeError("the exclusion bitmap is built on a CUDA device (no CPU fallback)")
    if isinstance(rows_per_query, tuple) and len(rows_per_query) == 2 and all(isinstance(t, torch.Tensor) for t in rows_per_query):
        offsets, rows = rows_per_query
        if offsets.dim() != 1 or offsets.numel() < 1 or rows.dim() != 1:
            raise ValueError("CSR exclusions must be 1-D offsets [Q+1] and rows tensors")
        offsets = offsets.to(device=dev, dtype=torch.int64).contiguous()
        rows = rows.to(device=dev, dtype=torch.int64).contiguous()
    else:
        lists = [np.asarray(list(r) if not isinstance(r, np.ndarray) else r, dtype=np.int64).reshape(-1) for r in rows_per_query]
        off = np.zeros(len(lists) + 1, dtype=np.int64)
        if lists:
            np.cumsum([len(r) for r in lists], out=off[1:])
        flat = np.concatenate(lists) if lists and off[-1] > 0 else np.zeros(1, np.int64)
        offsets = torch.from_numpy(off).to(dev)
        rows = torch.from_numpy(flat).to(dev)
    Q = offsets.numel() - 1
    bits = torch.empty(exclusion_words(n_rows), Q, dtype=torch.uint32, device=dev)
    lib = _lib.load()
    with _on(dev):
        _lib.check(lib.icr_query_exclusion_bits(offsets.data_ptr(), rows.data_ptr(), Q, n_rows, bits.data_ptr(), _stream(dev)))
    return bits


def cos_topk(
    queries: torch.Tensor,
    catalog: torch.Tensor,
    k: int,
    *,
    cat_planes: torch.Tensor | None = None,
    cat_inv_norms: torch.Tensor | None = None,
    exclude_mask: torch.Tensor | None = None,
    exclude_bits: torch.Tensor | None = None,
    row_offset: int = 0,
    path: int = PATH_AUTO,
    out: tuple[torch.Tensor, torch.Tensor] | None = None,
    workspace: torch.Tensor | None = None,
    peer: tuple[int, int, int, int, int] | None = None,
):
    """(values f32 [Q,k] descending, ids int64 [Q,k]) == torch.topk(cos_sim(q, c), k, dim=1).

    The catalog is float32, bfloat16 or float16; queries of another dtype are converted to the catalog's (for float16:
    ``normalized_f16``). ``exclude_mask`` (uint8/bool [N]) drops rows for every query; ``exclude_bits`` (``query_exclusion_bits``, uint32
    [ceil(N/32), Q]) drops rows per query. A row is dropped when either says so; queries with fewer than k eligible rows
    get a (-inf, -1) tail.

    ``peer`` = (rank, world, address of the uint64 buffer-pointer array, epoch, n_max) from ``PeerExchange.next_call()``:
    `catalog` is this rank's row shard and the call also exchanges and merges the candidates of all ranks
    (``icr_cos_topk_sharded``): the outputs are the GLOBAL top-k, identical on every rank. Collective: every rank calls."""
    _require_cuda("queries", queries)
    _require_cuda("catalog", catalog)
    queries, catalog = _rows(_like_catalog(queries, catalog.dtype)), _rows(catalog)
    if queries.shape[1] != catalog.shape[1]:
        raise ValueError(f"embedding dims differ: {queries.shape[1]} vs {catalog.shape[1]}")
    Q, D = queries.shape
    N = catalog.shape[0]
    dev = catalog.device
    lib = _lib.load()
    dt = _dtype_code(catalog)
    if exclude_mask is not None:
        _require_cuda("exclude_mask", exclude_mask)
        if exclude_mask.dtype not in (torch.uint8, torch.bool) or exclude_mask.numel() != N:
            raise ValueError("exclude_mask must be uint8/bool with one entry per catalog row")
        exclude_mask = exclude_mask.contiguous().view(torch.uint8)
    if exclude_bits is not None:
        _require_cuda("exclude_bits", exclude_bits)
        if exclude_bits.dtype not in (torch.uint32, torch.int32) or tuple(exclude_bits.shape) != (exclusion_words(N), Q):
            raise ValueError(f"exclude_bits must be uint32 [ceil(N/32), Q] = [{exclusion_words(N)}, {Q}] (query_exclusion_bits)")
        if exclude_bits.device != catalog.device:
            raise ValueError("exclude_bits must live on the catalog's device")
        if peer is not None:
            raise ValueError("per-query exclusions are not supported on the sharded call")
        exclude_bits = exclude_bits.contiguous()
    if cat_planes is not None:
        if cat_planes.dtype != torch.float16 or cat_planes.shape != (N, lib.icr_screen_plane_row_elems(D)) or not cat_planes.is_contiguous():
            raise ValueError("cat_planes must be the contiguous plane returned by screen_plane(catalog)")
    if cat_inv_norms is not None:
        if cat_inv_norms.dtype != torch.float32 or cat_inv_norms.shape != (N,) or not cat_inv_norms.is_contiguous():
            raise ValueError("cat_inv_norms must be the output of row_inv_norms(catalog)")
    if out is None:
        vals = torch.empty(Q, k, dtype=torch.float32, device=dev)
        ids = torch.empty(Q, k, dtype=torch.int64, device=dev)
    else:
        vals, ids = out
    with _on(dev):
        ws_bytes = lib.icr_cos_topk_workspace_bytes if peer is None else lib.icr_cos_topk_sharded_workspace_bytes
        need = ws_bytes(Q, N, D, dt, k, path, int(cat_planes is not None))
        if workspace is not None:
            # resident workspace (zero-filled once by its owner, reused call after call on one stream): no merge-counter memset
            if workspace.numel() < need or workspace.dtype != torch.uint8 or workspace.device != dev:
                raise ValueError(f"resident workspace must be a uint8 tensor of >= {need} bytes on {dev}")
            ws, path = workspace, path | PATH_WS_RESIDENT
        else:
            ws = _workspace(need, dev)
        if peer is not None:
            rank, world, ptrs, epoch, n_max = peer
            _lib.check(
                lib.icr_cos_topk_sharded(
                    queries.data_ptr(), Q, _ld(queries), catalog.data_ptr(), N, _ld(catalog), D, dt, _ptr(cat_planes), _ptr(cat_inv_norms),
                    _ptr(exclude_mask), k, row_offset, path, rank, world, ptrs, epoch, n_max, vals.data_ptr(), ids.data_ptr(),
                    ws.data_ptr(), ws.numel(), _stream(dev),
                )
            )
            return vals, ids
        if exclude_bits is not None:
            _lib.check(
                lib.icr_cos_topk_excl(
                    queries.data_ptr(), Q, _ld(queries), catalog.data_ptr(), N, _ld(catalog), D, dt, _ptr(cat_planes), _ptr(cat_inv_norms),
                    _ptr(exclude_mask), exclude_bits.data_ptr(), k, row_offset, path, vals.data_ptr(), ids.data_ptr(), ws.data_ptr(),
                    ws.numel(), _stream(dev),
                )
            )
            return vals, ids
        _lib.check(
            lib.icr_cos_topk(
                queries.data_ptr(), Q, _ld(queries), catalog.data_ptr(), N, _ld(catalog), D, dt, _ptr(cat_planes), _ptr(cat_inv_norms),
                _ptr(exclude_mask), k, row_offset, path, vals.data_ptr(), ids.data_ptr(), ws.data_ptr(), ws.numel(), _stream(dev),
            )
        )
    return vals, ids


def peer_exchange_merge(vals: torch.Tensor, ids: torch.Tensor, peer: tuple[int, int, int, int, int]):
    """This rank's [Q,k] candidates (f32 scores, i64 global ids) -> the global top-k of every query on every rank, in ONE kernel
    (``icr_peer_exchange_merge``: NVLink push, flags, wait, merge). ``peer`` as for ``cos_topk``. Collective."""
    _require_cuda("vals", vals)
    if vals.dtype != torch.float32 or ids.dtype != torch.int64 or vals.shape != ids.shape or vals.dim() != 2:
        raise ValueError("candidates must be f32 scores and i64 ids of one [Q, k] shape")
    vals, ids = vals.contiguous(), ids.contiguous()
    Q, k = vals.shape
    out_v, out_i = torch.empty_like(vals), torch.empty_like(ids)
    rank, world, ptrs, epoch, n_max = peer
    with _on(vals.device):
        _lib.check(lib_call("icr_peer_exchange_merge")(vals.data_ptr(), ids.data_ptr(), Q, k, rank, world, ptrs, epoch, n_max,
                                                       out_v.data_ptr(), out_i.data_ptr(), _stream(vals.device)))
    return out_v, out_i


def lib_call(name: str):
    return getattr(_lib.load(), name)


def cos_sim_dense(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """f32 [Qa, Nb] cosine similarity matrix. `a` is converted to b's dtype as ``cos_topk`` converts queries."""
    _require_cuda("a", a)
    _require_cuda("b", b)
    a, b = _rows(_like_catalog(a, b.dtype)), _rows(b)
    if a.shape[1] != b.shape[1]:
        raise ValueError(f"embedding dims differ: {a.shape[1]} vs {b.shape[1]}")
    lib = _lib.load()
    dev = b.device
    out = torch.empty(a.shape[0], b.shape[0], dtype=torch.float32, device=dev)
    with _on(dev):
        ws = _workspace(lib.icr_cos_sim_dense_workspace_bytes(a.shape[0], b.shape[0], a.shape[1], _dtype_code(b)), dev)
        _lib.check(
            lib.icr_cos_sim_dense(
                a.data_ptr(), a.shape[0], _ld(a), b.data_ptr(), b.shape[0], _ld(b), a.shape[1], _dtype_code(b), out.data_ptr(),
                max(out.shape[1], 1), ws.data_ptr(), ws.numel(), _stream(dev),
            )
        )
    return out


def topk_merge(cand_scores: torch.Tensor, cand_ids: torch.Tensor, k_out: int):
    """[G,Q,k_in] shard candidates -> global (values [Q,k_out], ids [Q,k_out])."""
    _require_cuda("cand_scores", cand_scores)
    _require_cuda("cand_ids", cand_ids)
    if cand_scores.dim() != 3 or cand_scores.shape != cand_ids.shape:
        raise ValueError("cand_scores / cand_ids must both be [G, Q, k_in]")
    cand_scores = cand_scores.contiguous().float()
    cand_ids = cand_ids.contiguous().long()
    G, Q, k_in = cand_scores.shape
    lib = _lib.load()
    dev = cand_scores.device
    vals = torch.empty(Q, k_out, dtype=torch.float32, device=dev)
    ids = torch.empty(Q, k_out, dtype=torch.int64, device=dev)
    with _on(dev):
        ws = _workspace(lib.icr_topk_merge_workspace_bytes(Q, G, k_in, k_out), dev)
        _lib.check(
            lib.icr_topk_merge(cand_scores.data_ptr(), cand_ids.data_ptr(), Q, G, k_in, k_out, vals.data_ptr(), ids.data_ptr(),
                               ws.data_ptr(), ws.numel(), _stream(dev))
        )
    return vals, ids


# metric kinds of include/icr_b200.h (icr_metric_kind)
METRIC_ACCURACY, METRIC_PRECISION, METRIC_RECALL, METRIC_MRR, METRIC_NDCG, METRIC_MAP, METRIC_NDCG_RETRIEVED, METRIC_MAP_RETRIEVED = range(8)
MAX_METRICS = 32


class RelevanceTable:
    """relevant_docs in the form the metric kernel reads: per query an ascending run of catalog rows (CSR) + |relevant|."""

    def __init__(self, relevant_rows, n_relevant=None, device=None):
        import numpy as np

        runs = [np.unique(np.asarray(r, dtype=np.int64)) for r in relevant_rows]
        offsets = np.zeros(len(runs) + 1, dtype=np.int64)
        if runs:
            np.cumsum([len(r) for r in runs], out=offsets[1:])
        flat = np.concatenate(runs) if runs else np.zeros(0, np.int64)
        nrel = np.asarray([len(r) for r in runs] if n_relevant is None else n_relevant, dtype=np.int32)
        if nrel.shape != (len(runs),):
            raise ValueError("n_relevant must have one entry per query")
        self.n_queries = len(runs)
        self.offsets = torch.from_numpy(offsets).to(device)
        self.rows = torch.from_numpy(flat if flat.size else np.zeros(1, np.int64)).to(device)
        self.n_relevant = torch.from_numpy(nrel if nrel.size else np.zeros(1, np.int32)).to(device)


def ir_metrics(ids: torch.Tensor, table: RelevanceTable, metrics: list[tuple[int, int]]):
    """(means f64 [M], per_query f64 [Q, M]) of the (kind, k) metrics over the retrieved-id matrix `ids` [Q, K]."""
    import ctypes

    _require_cuda("ids", ids)
    if ids.dim() != 2 or ids.dtype != torch.int64:
        raise ValueError("ids must be an int64 [Q, K] matrix (the second output of cos_topk)")
    if ids.stride(1) != 1:
        ids = ids.contiguous()
    Q, K = ids.shape
    if Q != table.n_queries:
        raise ValueError(f"{Q} id rows but the relevance table holds {table.n_queries} queries")
    if table.offsets.device != ids.device:
        raise ValueError("relevance table and ids live on different devices")
    M = len(metrics)
    kinds = (ctypes.c_int32 * max(M, 1))(*[int(m[0]) for m in metrics])
    ks = (ctypes.c_int32 * max(M, 1))(*[int(m[1]) for m in metrics])
    dev = ids.device
    per_query = torch.empty(Q, max(M, 1), dtype=torch.float64, device=dev)
    means = torch.empty(max(M, 1), dtype=torch.float64, device=dev)
    lib = _lib.load()
    with _on(dev):
        _lib.check(
            lib.icr_ir_metrics(ids.data_ptr(), Q, K, ids.stride(0) if Q > 1 else K, table.offsets.data_ptr(), table.rows.data_ptr(),
                               table.n_relevant.data_ptr(), ctypes.addressof(kinds), ctypes.addressof(ks), M, per_query.data_ptr(),
                               means.data_ptr(), _stream(dev))
        )
    return means, per_query


def _fast_rows(t: torch.Tensor) -> torch.Tensor:
    """_rows() without the checks' cost for the common case: contiguous, 16-byte aligned, D a multiple of 8."""
    if t.dim() == 2 and t.is_contiguous() and t.shape[1] % 8 == 0 and t.data_ptr() % 16 == 0:
        return t
    return _rows(t)


def mnrl_forward(anchors: torch.Tensor, positives: torch.Tensor, scale: float):
    """Returns (loss f32 scalar tensor, saved): saved = lse | inv_a | inv_p, B floats each."""
    _require_cuda("anchors", anchors)
    _require_cuda("positives", positives)
    if anchors.dtype != positives.dtype or anchors.shape != positives.shape:
        raise ValueError("anchors and positives must share dtype and shape [B, D]")
    a, p = _fast_rows(anchors), _fast_rows(positives)
    B, D = a.shape
    dev = a.device
    lib = _lib.load()
    loss = torch.empty((), dtype=torch.float32, device=dev)
    saved = torch.empty(3 * B, dtype=torch.float32, device=dev)  # lse | inv_a | inv_p
    base = saved.data_ptr()
    with _on(dev):
        ws = _workspace(lib.icr_mnrl_workspace_bytes(B, D), dev)
        _lib.check(
            lib.icr_mnrl_fwd(a.data_ptr(), _ld(a), p.data_ptr(), _ld(p), B, D, _dtype_code(a), float(scale), loss.data_ptr(),
                             base, base + 4 * B, base + 8 * B, ws.data_ptr(), ws.numel(), _stream(dev))
        )
    return loss, saved


def mnrl_forward_backward(anchors: torch.Tensor, positives: torch.Tensor, scale: float):
    """(loss, grad_anchors, grad_positives) with the gradients taken for dL/dloss = 1: one library call for a training step."""
    _require_cuda("anchors", anchors)
    _require_cuda("positives", positives)
    if anchors.dtype != positives.dtype or anchors.shape != positives.shape:
        raise ValueError("anchors and positives must share dtype and shape [B, D]")
    a, p = _fast_rows(anchors), _fast_rows(positives)
    B, D = a.shape
    dev = a.device
    lib = _lib.load()
    loss = torch.empty((), dtype=torch.float32, device=dev)
    saved = torch.empty(3 * B, dtype=torch.float32, device=dev)
    grads = torch.empty(2, B, D, dtype=a.dtype, device=dev)
    base = saved.data_ptr()
    gbytes = B * D * a.element_size()
    with _on(dev):
        ws = _workspace(lib.icr_mnrl_workspace_bytes(B, D), dev)
        _lib.check(
            lib.icr_mnrl_fwd_bwd(a.data_ptr(), _ld(a), p.data_ptr(), _ld(p), B, D, _dtype_code(a), float(scale), loss.data_ptr(),
                                 base, base + 4 * B, base + 8 * B, grads.data_ptr(), D, grads.data_ptr() + gbytes, D,
                                 ws.data_ptr(), ws.numel(), _stream(dev))
        )
    return loss, grads  # grads[0] = d loss / d anchors, grads[1] = d loss / d positives, [2, B, D (padded)]


def mnrl_scale_grads(grads: torch.Tensor, grad_out: torch.Tensor) -> torch.Tensor:
    """grads * grad_out for the [2, B, D] gradient pair of mnrl_forward_backward, one launch; `grads` is left untouched."""
    dev = grads.device
    go = grad_out
    if not (go.is_cuda and go.dtype == torch.float32 and go.is_contiguous()):
        go = go.detach().to(device=dev, dtype=torch.float32).contiguous()
    out = torch.empty_like(grads)
    half = grads.numel() // 2
    nbytes = half * grads.element_size()
    lib = _lib.load()
    with _on(dev):
        _lib.check(lib.icr_mnrl_scale_grads(grads.data_ptr(), grads.data_ptr() + nbytes, half, _dtype_code(grads), go.data_ptr(),
                                            out.data_ptr(), out.data_ptr() + nbytes, _stream(dev)))
    return out


def mnrl_backward(anchors: torch.Tensor, positives: torch.Tensor, scale: float, saved: torch.Tensor, grad_out: torch.Tensor):
    a, p = _fast_rows(anchors), _fast_rows(positives)
    B, D = a.shape
    dev = a.device
    lib = _lib.load()
    grads = torch.empty(2, B, D, dtype=a.dtype, device=dev)
    go = grad_out
    if not (go.is_cuda and go.dtype == torch.float32 and go.is_contiguous()):
        go = go.detach().to(device=dev, dtype=torch.float32).contiguous()
    base = saved.data_ptr()
    gbytes = B * D * a.element_size()
    with _on(dev):
        ws = _workspace(lib.icr_mnrl_workspace_bytes(B, D), dev)
        _lib.check(
            lib.icr_mnrl_bwd(a.data_ptr(), _ld(a), p.data_ptr(), _ld(p), B, D, _dtype_code(a), float(scale), base, base + 4 * B,
                             base + 8 * B, go.data_ptr(), grads.data_ptr(), D, grads.data_ptr() + gbytes, D,
                             ws.data_ptr(), ws.numel(), _stream(dev))
        )
    ga, gp = grads[0], grads[1]
    D0 = anchors.shape[1]
    return (ga[:, :D0], gp[:, :D0]) if D0 != D else (ga, gp)


def mnrl_forward_rect(anchors: torch.Tensor, candidates: torch.Tensor, scale: float, label_offset: int):
    """MNRL of B anchors against Bc >= B candidates, the positive of anchor i at candidate i + label_offset.
    Returns (loss f32 scalar tensor, saved = lse [B] | inv_a [B] | inv_c [Bc])."""
    _require_cuda("anchors", anchors)
    _require_cuda("candidates", candidates)
    if anchors.dtype != candidates.dtype or anchors.dim() != 2 or candidates.dim() != 2 or anchors.shape[1] != candidates.shape[1]:
        raise ValueError("anchors [B, D] and candidates [Bc, D] must share dtype and embedding dim")
    a, c = _fast_rows(anchors), _fast_rows(candidates)
    B, D = a.shape
    Bc = c.shape[0]
    dev = a.device
    lib = _lib.load()
    loss = torch.empty((), dtype=torch.float32, device=dev)
    saved = torch.empty(2 * B + Bc, dtype=torch.float32, device=dev)
    base = saved.data_ptr()
    with _on(dev):
        ws = _workspace(lib.icr_mnrl_rect_workspace_bytes(B, Bc, D), dev)
        _lib.check(
            lib.icr_mnrl_fwd_rect(a.data_ptr(), _ld(a), c.data_ptr(), _ld(c), B, Bc, int(label_offset), D, _dtype_code(a), float(scale),
                                  loss.data_ptr(), base, base + 4 * B, base + 8 * B, ws.data_ptr(), ws.numel(), _stream(dev))
        )
    return loss, saved


def mnrl_backward_rect(anchors: torch.Tensor, candidates: torch.Tensor, scale: float, label_offset: int, saved: torch.Tensor,
                       grad_out: torch.Tensor):
    """(grad_anchors [B, D], grad_candidates [Bc, D]) of mnrl_forward_rect's loss times grad_out."""
    a, c = _fast_rows(anchors), _fast_rows(candidates)
    B, D = a.shape
    Bc = c.shape[0]
    dev = a.device
    lib = _lib.load()
    ga = torch.empty(B, D, dtype=a.dtype, device=dev)
    gc = torch.empty(Bc, D, dtype=a.dtype, device=dev)
    go = grad_out
    if not (go.is_cuda and go.dtype == torch.float32 and go.is_contiguous()):
        go = go.detach().to(device=dev, dtype=torch.float32).contiguous()
    base = saved.data_ptr()
    with _on(dev):
        ws = _workspace(lib.icr_mnrl_rect_workspace_bytes(B, Bc, D), dev)
        _lib.check(
            lib.icr_mnrl_bwd_rect(a.data_ptr(), _ld(a), c.data_ptr(), _ld(c), B, Bc, int(label_offset), D, _dtype_code(a), float(scale),
                                  base, base + 4 * B, base + 8 * B, go.data_ptr(), ga.data_ptr(), D, gc.data_ptr(), D,
                                  ws.data_ptr(), ws.numel(), _stream(dev))
        )
    D0 = anchors.shape[1]
    return (ga[:, :D0], gc[:, :D0]) if D0 != D else (ga, gc)
