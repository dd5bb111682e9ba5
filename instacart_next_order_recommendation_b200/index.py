"""Embedding index: the reference's on-disk catalog cache plus its device-resident form.

``EmbeddingIndex`` keeps the reference's format byte for byte
(src/inference/serve_recommendations.py:66-130; file names from src/constants.py:88-92):

    <corpus dir>/.embedding_index/<sha256(model_dir|corpus_path)[:16]>/
        manifest.json   {"corpus_path", "model_dir", "corpus_mtime", "n_products"}
        embeddings.npy  float32 [N, D]
        product_ids.json

``EmbeddingIndex.open`` memory-maps the same file instead of reading it, ``save_bf16_sidecar`` /
``open_bf16_sidecar`` add an optional ``embeddings.bf16.bin`` next to it (half the bytes on disk and
over PCIe, valid only while the manifest-validated ``embeddings.npy`` it was made from is unchanged),
and ``DeviceCatalog.from_index`` streams either one into HBM chunk by chunk through pinned staging
buffers — for a whole catalog or for one rank's row block of a sharded one (SURVEY §8f row 3).

``DeviceCatalog`` is what the kernels read: the same rows resident in HBM (fp32, or bf16 or fp16
on request), plus the inverse row norms and — for fp32 — the fp16 screening plane of the
tensor-core path, built once at load instead of re-normalising the catalog on every request as
``sentence_transformers.util.cos_sim`` does (serve_recommendations.py:214).
"""

from __future__ import annotations

import hashlib
import json
import threading
import logging
from pathlib import Path

import numpy as np
import torch

from . import ops
from .similarity import default_device, to_device_matrix

# the current stream's handle without building a torch.cuda.Stream object (the request path asks for it on every call)
_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None) or (lambda idx: torch.cuda.current_stream(idx).cuda_stream)

logger = logging.getLogger(__name__)

INDEX_SUBDIR = ".embedding_index"
MANIFEST_FILENAME = "manifest.json"
EMBEDDINGS_FILENAME = "embeddings.npy"
PRODUCT_IDS_FILENAME = "product_ids.json"
BF16_SIDECAR_FILENAME = "embeddings.bf16.bin"  # raw bfloat16 [N, D], row-major, no header (shape comes from embeddings.npy)


class EmbeddingIndex:
    """Disk cache of product embeddings, keyed by corpus path + model dir + corpus mtime."""

    def __init__(self, corpus_path: Path, model_dir: Path | str):
        self.corpus_path = Path(corpus_path).resolve()
        self.model_dir = model_dir
        self._dir = self._index_dir()

    def _index_dir(self) -> Path:
        key = hashlib.sha256(f"{self.model_dir!s}|{self.corpus_path!s}".encode()).hexdigest()[:16]
        return self.corpus_path.parent / INDEX_SUBDIR / key

    @property
    def directory(self) -> Path:
        return self._dir

    def _corpus_mtime(self):
        try:
            return self.corpus_path.stat().st_mtime
        except OSError:
            return None

    def load(self, product_ids: list[str]) -> np.ndarray | None:
        """Embeddings if every validity check of the reference passes, else None."""
        try:
            meta = json.loads((self._dir / MANIFEST_FILENAME).read_text())
        except (OSError, json.JSONDecodeError):
            return None
        if meta.get("corpus_path") != str(self.corpus_path) or meta.get("model_dir") != str(self.model_dir):
            return None
        mtime = self._corpus_mtime()
        if mtime is None or meta.get("corpus_mtime") != mtime:
            return None
        try:
            embeddings = np.load(self._dir / EMBEDDINGS_FILENAME)
            cached_ids = json.loads((self._dir / PRODUCT_IDS_FILENAME).read_text())
        except (OSError, ValueError):
            return None
        if cached_ids != product_ids or len(embeddings) != len(product_ids):
            return None
        return embeddings

    def _valid_manifest(self) -> bool:
        try:
            meta = json.loads((self._dir / MANIFEST_FILENAME).read_text())
        except (OSError, json.JSONDecodeError):
            return False
        if meta.get("corpus_path") != str(self.corpus_path) or meta.get("model_dir") != str(self.model_dir):
            return False
        mtime = self._corpus_mtime()
        return mtime is not None and meta.get("corpus_mtime") == mtime

    def open(self, product_ids: list[str]) -> np.ndarray | None:
        """Like ``load`` (same validity rules) but memory-maps embeddings.npy read-only instead of reading it."""
        if not self._valid_manifest():
            return None
        try:
            embeddings = np.load(self._dir / EMBEDDINGS_FILENAME, mmap_mode="r")
            cached_ids = json.loads((self._dir / PRODUCT_IDS_FILENAME).read_text())
        except (OSError, ValueError):
            return None
        if cached_ids != product_ids or len(embeddings) != len(product_ids):
            return None
        return embeddings

    def save_bf16_sidecar(self, *, normalize: bool = False) -> Path:
        """Write embeddings.bf16.bin from the index's embeddings.npy (rows optionally L2-normalised, then rounded to
        nearest-even bfloat16). Host-side file conversion, chunked; the index itself is not touched."""
        emb = np.load(self._dir / EMBEDDINGS_FILENAME, mmap_mode="r")
        path = self._dir / BF16_SIDECAR_FILENAME
        tmp = path.with_suffix(".tmp")
        with open(tmp, "wb") as f:
            for s0 in range(0, emb.shape[0], 1 << 16):
                t = torch.from_numpy(np.array(emb[s0 : s0 + (1 << 16)], dtype=np.float32))
                if normalize:
                    t = torch.nn.functional.normalize(t, p=2, dim=1, eps=1e-12)
                f.write(t.to(torch.bfloat16).view(torch.int16).numpy().tobytes())
        tmp.replace(path)
        return path

    def open_bf16_sidecar(self, product_ids: list[str], _emb: np.ndarray | None = None) -> np.ndarray | None:
        """uint16 memmap [N, D] of the sidecar's bfloat16 bit patterns, or None unless the index itself is valid for
        `product_ids`, and the sidecar is as large as embeddings.npy says and not older than it."""
        emb = _emb if _emb is not None else self.open(product_ids)  # _emb: the caller has just validated the index
        if emb is None or emb.ndim != 2:
            return None
        side, base = self._dir / BF16_SIDECAR_FILENAME, self._dir / EMBEDDINGS_FILENAME
        try:
            st_side, st_base = side.stat(), base.stat()
        except OSError:
            return None
        if st_side.st_size != emb.shape[0] * emb.shape[1] * 2 or st_side.st_mtime < st_base.st_mtime:
            return None
        return np.memmap(side, dtype=np.uint16, mode="r", shape=emb.shape)

    def save(self, product_ids: list[str], embeddings: np.ndarray) -> None:
        self._dir.mkdir(parents=True, exist_ok=True)
        mtime = self._corpus_mtime()
        manifest = {
            "corpus_path": str(self.corpus_path),
            "model_dir": str(self.model_dir),
            "corpus_mtime": 0 if mtime is None else mtime,
            "n_products": len(product_ids),
        }
        (self._dir / MANIFEST_FILENAME).write_text(json.dumps(manifest, indent=2))
        np.save(self._dir / EMBEDDINGS_FILENAME, np.asarray(embeddings).astype(np.float32))
        (self._dir / PRODUCT_IDS_FILENAME).write_text(json.dumps(product_ids))
        logger.info("Saved embedding index to %s (%d products)", self._dir, len(product_ids))


def _is_f16(x) -> bool:
    return getattr(x, "dtype", None) in (torch.float16, np.float16)


def _f16_matrix(x, device: torch.device) -> torch.Tensor:
    """A float16 tensor or array as a [rows, dim] tensor on `device`, values untouched (no round trip through fp32)."""
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    if t.dim() == 1:
        t = t.unsqueeze(0)
    if t.dim() != 2:
        raise ValueError(f"expected a vector or a [rows, dim] matrix, got shape {tuple(t.shape)}")
    return t.to(device, non_blocking=True)


class DeviceCatalog:
    """Catalog rows resident in HBM, with whatever the kernels want precomputed.

    dtype float32 keeps the reference's numerics (scores within 1e-5 of the fp32 oracle);
    dtype bfloat16 halves the bytes a batch-1 request streams (scores within 2e-3);
    dtype float16 streams as many bytes as bfloat16 with 8x finer rounding: scores are fp32 arithmetic on the fp16
    values (within 1e-5 of fp64 on them), and queries are L2-normalised in fp32 before they are rounded to fp16.
    float16 rows must be finite: un-normalised rows beyond fp16's range raise (normalise them first).
    dtype int8 quarters the bytes of fp32: each row is stored as int8 codes with one fp32 factor (``ops.quantize_rows``,
    per-row scalar quantisation) and queries stay float32, quantised by the kernel the same way. Results are exact on the
    quantised values (ids and score bits are those of integer dot products scaled by the two factors), not within a
    tolerance of fp32: expect recall@10 around 0.98 against fp32 exact. Rows must be finite.

    ``update_rows``, ``append_rows`` and ``remove_rows`` change the catalog in place. The result equals a catalog freshly built
    from the updated fp32 matrix in the same row order through the same constructor path: rows, planes and inverse norms
    bit for bit, and so every top-k result. Updated rows are normalised when ``from_index(normalize=True)`` normalised the
    catalog (``normalized``). A bfloat16 catalog loaded from the sidecar converts updated fp32 rows with round-to-nearest-even,
    as ``from_index(use_sidecar=False)`` would. A catalog built from a float32 device tensor shares that tensor's memory until
    its first change, which copies it. Each change holds ``request_lock``, waits for the work already enqueued on the device
    and synchronises before it returns; ``topk`` batches that other threads run during a change must be ordered by the caller.
    """

    # the kernels keep row ids in 32 bits, with 2^32 - 1 reserved
    MAX_ROWS = 0xFFFFFFFF - 1
    # first growth of an appended catalog: rows, plane and inverse norms are reallocated together with this much headroom
    GROWTH = 1.5

    def __init__(self, embeddings, *, device: torch.device | None = None, dtype: torch.dtype = torch.float32,
                 row_offset: int = 0, build_planes: bool | None = None):
        if dtype not in (torch.float32, torch.bfloat16, torch.float16, torch.int8):
            raise TypeError("catalog dtype must be float32, bfloat16, float16 or int8")
        dev = device if device is not None else (embeddings.device if isinstance(embeddings, torch.Tensor) and embeddings.is_cuda else default_device())
        if dtype == torch.int8:
            if isinstance(embeddings, tuple):  # (codes, factors) of from_index, quantised while streaming
                codes, factors, input_dim = embeddings
            else:
                x = to_device_matrix(embeddings, device=dev).float()
                if x.numel() and not bool(torch.isfinite(x).all()):
                    raise ValueError("int8 catalog rows must be finite")
                input_dim = int(x.shape[1])
                codes, factors = ops.quantize_rows(x) if x.shape[0] > 0 else (
                    torch.empty(0, (input_dim + 15) // 16 * 16, dtype=torch.int8, device=dev), torch.empty(0, device=dev))
            self._init_i8(codes, factors, input_dim, row_offset)
            return
        if dtype == torch.float16 and _is_f16(embeddings):
            rows = _f16_matrix(embeddings, dev)  # taken bit for bit
        else:
            rows = to_device_matrix(embeddings, device=dev)  # uploaded in the dtype it has (float64 / float16 become float32)
        if rows.dtype != dtype:
            if rows.dtype == torch.float32 and rows.dim() == 2 and rows.shape[1] % 4 == 0 and rows.shape[0] > 0:
                rows = ops._rows(rows)
                rows = ops.convert_rows(rows, torch.empty(rows.shape, dtype=dtype, device=dev))  # fp32 -> bf16 / fp16 on the device (RNE)
            else:
                rows = rows.to(dtype)
        if dtype == torch.float16 and rows.numel() and not bool(torch.isfinite(rows).all()):
            raise ValueError("catalog rows exceed float16's range (inf or NaN after conversion): L2-normalise them first "
                             "(convert with normalize=True, e.g. DeviceCatalog.from_index(..., normalize=True))")
        self.input_dim = int(rows.shape[1]) if rows.dim() == 2 else 0  # before the 16-byte padding of _rows()
        self.rows = ops._rows(rows)
        self.row_offset = int(row_offset)
        self.request_lock = threading.RLock()  # guards the shared static tensors of topk_small(copy=False)
        self._plans: dict = {}  # prepared request calls, see _prepared_call
        self.planes: torch.Tensor | None = None
        if build_planes is None:
            build_planes = dtype == torch.float32
        self.normalized = False  # set by from_index(normalize=True): updated rows are normalised alike
        self._with_planes = bool(build_planes) and dtype == torch.float32
        # the rows may be the caller's tensor (an fp32 device matrix is taken as is): the first change copies them
        self._shared_rows = isinstance(embeddings, torch.Tensor) and embeddings.is_cuda and \
            embeddings.untyped_storage().data_ptr() == self.rows.untyped_storage().data_ptr()
        self._reserve: tuple | None = None  # (rows, planes, inv_norms) storage once the catalog has changed
        self.inv_norms: torch.Tensor | None = None
        if build_planes and dtype == torch.float32 and self.rows.shape[0] > 0:
            # fp32 catalogs: the fp32 rows serve the GEMV path and the exact re-scoring; the tensor-core sweep reads a
            # single fp16 screening plane (half the rows' bytes) - 1.5x the catalog resident, not 2x as with hi|lo planes
            self.planes, self.inv_norms = ops.screen_plane(self.rows)
        elif self.rows.shape[0] > 0:
            self.inv_norms = ops.row_inv_norms(self.rows)

    def _init_i8(self, codes: torch.Tensor, factors: torch.Tensor | None, input_dim: int, row_offset: int) -> None:
        self.input_dim = input_dim
        self.rows = codes
        self.row_offset = int(row_offset)
        self.request_lock = threading.RLock()
        self._plans: dict = {}
        self.planes = None
        self.normalized, self._with_planes, self._shared_rows, self._reserve = False, False, False, None
        # int8 catalogs: the per-row factors of ops.quantize_rows, passed where the ABI takes inverse norms (the factor
        # carries the row's 1 / |x|, times its quantisation step)
        self.inv_norms = factors

    @classmethod
    def from_index(cls, index: "EmbeddingIndex", product_ids: list[str], *, dtype: torch.dtype = torch.float32,
                   device: torch.device | None = None, rows: tuple[int, int] | None = None, normalize: bool = False,
                   use_sidecar: bool = True, chunk_rows: int = 1 << 15, row_offset: int | None = None) -> "DeviceCatalog | None":
        """Stream a validated on-disk index (or the row block `rows` = [lo, hi) of it) into HBM.

        None if the index is missing or stale (the caller re-encodes, as the reference does,
        serve_recommendations.py:183-204). With dtype bfloat16 a valid ``embeddings.bf16.bin`` sidecar is uploaded
        as is (half the bytes); otherwise (and always for float16) the fp32 rows go up chunk by chunk and
        ``icr_convert_rows`` writes the resident form. ``row_offset`` defaults to lo, so a row-sharded catalog returns global ids.
        dtype int8 streams the fp32 rows through ``icr_quantize_rows`` (never the sidecar); ``normalize=True`` is rejected,
        since the factors already normalise.
        """
        if dtype == torch.int8 and normalize:
            raise ValueError("normalize=True does not apply to an int8 catalog: its factors carry each row's inverse norm")
        emb = index.open(product_ids)
        if emb is None:
            return None
        dev = device if device is not None else default_device()
        lo, hi = (0, emb.shape[0]) if rows is None else (max(0, int(rows[0])), min(emb.shape[0], int(rows[1])))
        hi = max(lo, hi)
        if dtype == torch.int8:
            if emb.shape[1] % 4:  # icr_quantize_rows reads 16-byte vectors: such a catalog goes up as fp32 and is padded
                resident = upload_rows(emb, lo, hi, device=dev, dtype=torch.float32, chunk_rows=chunk_rows)
                return cls(resident, device=dev, dtype=dtype, row_offset=lo if row_offset is None else row_offset)
            codes, factors = upload_quantized(emb, lo, hi, device=dev, chunk_rows=chunk_rows)
            return cls((codes, factors, int(emb.shape[1])), device=dev, dtype=dtype, row_offset=lo if row_offset is None else row_offset)
        side = index.open_bf16_sidecar(product_ids, _emb=emb) if (use_sidecar and dtype == torch.bfloat16 and not normalize) else None
        # icr_convert_rows works on 16-byte vectors: an embedding dim that is not a multiple of 4 goes up as fp32 and is
        # converted (and padded) by the DeviceCatalog constructor instead
        odd = side is None and emb.shape[1] % 4 != 0 and (dtype != torch.float32 or normalize)
        if odd and normalize:
            raise ValueError("normalize=True needs an embedding dim that is a multiple of 4")
        resident = upload_rows(side if side is not None else emb, lo, hi, device=dev, dtype=torch.float32 if odd else dtype,
                               normalize=normalize, chunk_rows=chunk_rows, source_is_bf16_bits=side is not None)
        cat = cls(resident, device=dev, dtype=dtype, row_offset=lo if row_offset is None else row_offset)
        cat.normalized = bool(normalize)
        cat._shared_rows = False  # the loader's tensor: nobody else holds it
        return cat

    @property
    def device(self) -> torch.device:
        return self.rows.device

    @property
    def dtype(self) -> torch.dtype:
        return self.rows.dtype

    def __len__(self) -> int:
        return self.rows.shape[0]

    @property
    def dim(self) -> int:
        return self.rows.shape[1]

    @property
    def query_dtype(self) -> torch.dtype:
        """The dtype of the queries the kernels read: the catalog's, except float32 for an int8 catalog."""
        return torch.float32 if self.dtype == torch.int8 else self.dtype

    def _device_queries(self, queries) -> torch.Tensor:
        """Queries on the catalog's device in the form its kernels take: ``query_dtype``; for float16 catalogs float16
        queries as given and any other dtype through ``ops.normalized_f16``."""
        if self.dtype == torch.int8:
            return to_device_matrix(queries, device=self.device, dtype=torch.float32)
        if self.dtype != torch.float16:
            return to_device_matrix(queries, device=self.device, dtype=self.dtype)
        if _is_f16(queries):
            return _f16_matrix(queries, self.device)
        return ops.normalized_f16(to_device_matrix(queries, device=self.device))

    @property
    def nbytes(self) -> int:
        extra = sum(t.numel() * t.element_size() for t in (self.planes, self.inv_norms) if t is not None)
        return self.rows.numel() * self.rows.element_size() + extra

    # ---- in-place changes ----------------------------------------------------------------------------------
    def update_rows(self, rows, embeddings) -> None:
        """Replace the local rows `rows` (before ``row_offset``) with `embeddings` [len(rows), input_dim] of any float
        dtype (up-cast to float32; float16 rows land bit for bit in a float16 catalog), in place: one ``icr_update_rows``
        launch writes each row in the resident form with its inverse norm (int8: codes and factor) and, for float32, its
        screening-plane row. Pointers and length do not change, so cached CUDA graphs, prepared calls and resident
        workspaces stay valid and return the new rows' results. Raises ValueError, leaving the catalog unchanged, on
        duplicate or out-of-range rows, a dim mismatch, non-finite input or float16 overflow."""
        with self.request_lock:
            idx = self._row_index(rows, len(self))
            x = self._update_source(embeddings)
            if x.shape[0] != idx.size:
                raise ValueError(f"{idx.size} rows but {x.shape[0]} embeddings")
            if idx.size == 0:
                return
            torch.cuda.synchronize(self.device)  # work enqueued on any stream of the device reads the old rows first
            if self._shared_rows:
                self._reallocate(len(self), len(self))
            self._write(idx, x)
            torch.cuda.current_stream(self.device).synchronize()

    def append_rows(self, embeddings) -> range:
        """Append `embeddings` [M, input_dim] as new rows; returns their local row range. The first append reserves
        ``GROWTH`` times the rows (rows, plane and inverse norms reallocated together); later appends write into the reserve
        until it is full. ``rows`` stays a [len, ld] tensor (a view of the reserve). Prepared calls, CUDA graphs and resident
        workspaces are sized for the old length and are dropped. Validation as ``update_rows``; more than ``MAX_ROWS`` rows
        raise."""
        with self.request_lock:
            x = self._update_source(embeddings)
            n, m = len(self), x.shape[0]
            if m == 0:
                return range(n, n)
            if n + m > self.MAX_ROWS:
                raise ValueError(f"a catalog holds at most {self.MAX_ROWS} rows ({n} + {m} requested)")
            torch.cuda.synchronize(self.device)
            cap = self._reserve[0].shape[0] if self._reserve is not None and not self._shared_rows else 0
            if n + m > cap:
                self._reallocate(n, max(n + m, int(n * self.GROWTH)))
            self._set_length(n + m)
            self._write(np.arange(n, n + m, dtype=np.int64), x)
            torch.cuda.current_stream(self.device).synchronize()
            return range(n, n + m)

    # rows moved per step of remove_rows: its extra memory is one such chunk of rows, planes and norms
    REMOVE_CHUNK_ROWS = 1 << 16

    def remove_rows(self, rows) -> np.ndarray:
        """Remove the local rows `rows` and compact the rest in place, stably: the remaining rows keep their order (ties
        still go to the lower row, as in a fresh build). Returns the old indices of the kept rows, ascending. The memory
        freed stays reserved for appends; the extra memory of the call is one chunk of ``REMOVE_CHUNK_ROWS`` rows. Drops the
        cached request state as ``append_rows`` does. Duplicate or out-of-range rows raise ValueError and change nothing."""
        with self.request_lock:
            n = len(self)
            idx = self._row_index(rows, n)
            keep = np.ones(n, dtype=bool)
            keep[idx] = False
            kept = np.flatnonzero(keep)
            if idx.size == 0:
                return kept
            torch.cuda.synchronize(self.device)
            if self._shared_rows:
                self._reallocate(n, n)
            self._reserve = self._storage()
            bufs = [t for t in self._reserve if t is not None]
            first = int(idx.min())  # rows below the first removed one stay where they are
            for a in range(first, kept.size, self.REMOVE_CHUNK_ROWS):
                b = min(kept.size, a + self.REMOVE_CHUNK_ROWS)
                src = torch.from_numpy(kept[a:b]).to(self.device)
                for t in bufs:  # kept[j] >= j: a chunk reads only rows at or beyond the ones it writes
                    t[a:b] = t.index_select(0, src)
            self._set_length(kept.size)
            torch.cuda.current_stream(self.device).synchronize()
            return kept

    def _row_index(self, rows, n: int) -> np.ndarray:
        t = rows.detach().cpu().numpy() if isinstance(rows, torch.Tensor) else np.asarray(list(rows) if not isinstance(rows, np.ndarray) else rows)
        if t.size and not np.issubdtype(t.dtype, np.integer):
            raise ValueError(f"row indices must be integers, got {t.dtype}")
        idx = t.astype(np.int64).reshape(-1)
        if idx.size and (idx.min() < 0 or idx.max() >= n):
            raise ValueError(f"row indices must lie in [0, {n})")
        if np.unique(idx).size != idx.size:
            raise ValueError("duplicate row indices")
        return idx

    def _update_source(self, embeddings) -> torch.Tensor:
        """`embeddings` as validated float32 device rows [M, rows.shape[1]] (the padding columns zero)."""
        x = embeddings if isinstance(embeddings, torch.Tensor) else torch.as_tensor(np.asarray(embeddings))
        if x.dim() == 1:
            x = x.unsqueeze(0)
        if x.dim() != 2 or not x.is_floating_point():
            raise ValueError(f"expected floating-point [rows, dim] embeddings, got {x.dtype} {tuple(x.shape)}")
        if x.shape[1] != self.input_dim:
            raise ValueError(f"embedding dims differ: {x.shape[1]} vs catalog {self.input_dim}")
        x = x.to(device=self.device, dtype=torch.float32)
        if x.numel() and not bool(torch.isfinite(x).all()):
            raise ValueError("catalog rows must be finite")
        if self.dtype == torch.float16 and not self.normalized and x.numel() and not bool(torch.isfinite(x.half()).all()):
            raise ValueError("catalog rows exceed float16's range (inf after conversion): L2-normalise them first")
        if x.shape[1] != self.rows.shape[1]:
            x = torch.nn.functional.pad(x, (0, self.rows.shape[1] - x.shape[1]))
        return x.contiguous()

    def _write(self, idx: np.ndarray, x: torch.Tensor) -> None:
        ops.update_rows(x, torch.from_numpy(idx).to(self.device), self.rows, self.inv_norms, planes=self.planes, normalize=self.normalized)

    def _storage(self) -> tuple:
        return self._reserve if self._reserve is not None else (self.rows, self.planes, self.inv_norms)

    def _reallocate(self, n: int, cap: int) -> None:
        """New storage for `cap` rows holding the first `n` rows of the current one."""
        dev, width = self.device, self.rows.shape[1]
        rows = torch.empty(cap, width, dtype=self.rows.dtype, device=dev)
        rows[:n] = self.rows[:n]
        planes = None
        if self.planes is not None or (n == 0 and self._with_planes):
            planes = torch.empty(cap, ops._lib.load().icr_screen_plane_row_elems(width), dtype=torch.float16, device=dev)
            if n:
                planes[:n] = self.planes[:n]
        inv = torch.empty(cap, dtype=torch.float32, device=dev)
        if n:
            inv[:n] = self.inv_norms[:n]
        self._reserve, self._shared_rows = (rows, planes, inv), False
        self._set_length(n)

    def _set_length(self, n: int) -> None:
        """Views of the first n rows of the storage; the request state bound to the old length or pointers is dropped."""
        rows, planes, inv = self._storage()
        self.rows, self.planes, self.inv_norms = rows[:n], None if planes is None else planes[:n], inv[:n]
        self._plans = {}
        self.__dict__.pop("_graphs", None)
        self.__dict__.pop("_resident", None)

    # ---- request-sized calls: one CUDA graph per (Q, k) -------------------------------------------------
    def _graph_for(self, Q: int, k: int, path: int, convert: bool = False):
        """Capture prep + scoring + select of a fixed-shape request once; replays cost one graph launch.

        The serve path is launch-latency-bound (a batch-1 request streams 76 MB in ~12 µs of HBM time), so the
        Python/ctypes work and the gaps between the 2-3 kernels of a call matter more than the kernels.
        ``convert`` (float16 catalogs, queries of another dtype): the graph takes fp32 queries and its first kernel
        normalises and rounds them (``ops.normalized_f16``).
        """
        if not hasattr(self, "_graphs"):
            self._graphs = {}
        key = (Q, k, path, convert)
        entry = self._graphs.get(key)
        if entry is None:
            static_q = torch.zeros(Q, self.rows.shape[1], dtype=torch.float32 if convert else self.query_dtype, device=self.device)
            static_q16 = torch.empty(Q, self.rows.shape[1], dtype=torch.float16, device=self.device) if convert else None

            # the graph owns its workspace: zero-filled once here, then only this graph's kernels touch it, so the per-call
            # memset of the merge counter drops out of the captured sequence (ICR_PATH_WS_RESIDENT)
            lib = ops._lib.load()
            need = lib.icr_cos_topk_workspace_bytes(Q, self.rows.shape[0], self.rows.shape[1], ops._dtype_code(self.rows), k, path,
                                                    int(self.planes is not None))
            resident = torch.zeros(max(int(need), 256), dtype=torch.uint8, device=self.device)
            kw = dict(cat_planes=self.planes, cat_inv_norms=self.inv_norms, row_offset=self.row_offset, path=path, workspace=resident)

            def call():
                q = ops.convert_rows(static_q, static_q16, normalize=True) if convert else static_q
                return ops.cos_topk(q, self.rows, k, **kw)

            side = torch.cuda.Stream(self.device)
            side.wait_stream(torch.cuda.current_stream(self.device))
            with torch.cuda.stream(side):  # warm-up outside capture: one-time attribute setting, lazy module load
                call()
            torch.cuda.current_stream(self.device).wait_stream(side)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                vals, ids = call()
            entry = (graph, static_q, vals, ids, resident, static_q16)
            self._graphs[key] = entry
        return entry

    def topk_small(self, queries, k: int, *, path: int = ops.PATH_AUTO, copy: bool = True):
        """topk() for request-sized batches (Q <= 8) through a cached CUDA graph.

        `queries` may live on the host (numpy / CPU tensor, as SentenceTransformer.encode returns it) or on the
        device. With copy=False the returned tensors are the graph's static outputs, overwritten by the next call:
        callers that may run concurrently hold ``self.request_lock`` around the call AND their read of the results
        (Recommender._rank does); copy=True takes the lock itself and returns private tensors.
        """
        q = queries if isinstance(queries, torch.Tensor) else torch.as_tensor(queries)
        if q.dim() == 1:
            q = q.unsqueeze(0)
        rows = self.rows
        k = min(int(k), rows.shape[0])
        Q, D = q.shape
        if k < 1 or Q == 0:
            return self.topk(q, max(k, 1))
        if D != self.input_dim:
            raise ValueError(f"embedding dims differ: query {D} vs catalog {self.input_dim}")
        if Q <= 7 and q.is_cuda and q.dtype == self.query_dtype and q.device == rows.device and D == rows.shape[1] and q.is_contiguous() \
                and q.data_ptr() % 16 == 0:
            # a device-resident query in the catalog's own layout (what encode(convert_to_tensor=True) hands over): the kernel
            # reads it where it lies - no copy into a graph's input buffer, one kernel launch through a prepared argument list
            with self.request_lock:
                vals, ids = self._prepared_call(q, k, path)
                return (vals.clone(), ids.clone()) if copy else (vals, ids)
        with self.request_lock:
            convert = self.dtype == torch.float16 and q.dtype != torch.float16
            graph, static_q, vals, ids = self._graph_for(q.shape[0], k, path, convert)[:4]
            D = q.shape[1]  # columns beyond the catalog's own dim are the zero padding of _rows(); they stay zero
            static_q[:, :D].copy_(q, non_blocking=True)  # H2D (or D2D) + dtype conversion in one op
            graph.replay()
            return (vals.clone(), ids.clone()) if copy else (vals, ids)

    def topk_request(self, q: torch.Tensor, k: int, *, path: int = ops.PATH_AUTO):
        """One request, query on the device, result on the HOST: ``(scores, ids)`` as Python lists of Q lists of k.

        The kernel's last CTA stores the k results straight into pinned, device-mapped host memory (16 x 12 bytes over PCIe
        behind the merge), so the request is one kernel launch and one stream synchronisation - no device-to-host copies
        (two ``.tolist()`` reads of device tensors cost two synchronising copies, ~10 us each). Takes the same queries as the
        prepared-call path of ``topk_small`` (device tensor in the catalog's dtype and layout, Q <= 7); anything else falls
        back to ``topk_small`` + ``.tolist()``. Holds ``request_lock`` until the results are Python objects."""
        if q.dim() == 1:
            q = q.unsqueeze(0)
        rows = self.rows
        k = min(int(k), rows.shape[0])
        Q, D = q.shape
        with self.request_lock:
            if not (1 <= Q <= 7 and k >= 1 and q.is_cuda and q.dtype == self.query_dtype and q.device == rows.device and D == rows.shape[1]
                    and D == self.input_dim and q.is_contiguous() and q.data_ptr() % 16 == 0):
                vals, ids = self.topk_small(q, k, path=path, copy=False)
                return vals.tolist(), ids.tolist()
            vals, ids = self._prepared_call(q, k, path, host_out=True)
            torch.cuda.current_stream(self.device).synchronize()
            return vals.tolist(), ids.tolist()

    def _prepared_call(self, q: torch.Tensor, k: int, path: int, host_out: bool = False, fresh_out: bool = False):
        """icr_cos_topk for a request-sized device query with everything but the query pointer bound once per
        (Q, k, path, stream): static outputs, a resident zero-filled workspace, ready-made ctypes arguments. The Python
        side of a request is then ~5 us (ops.cos_topk: ~40 us of checks, allocations and argument conversion) and the
        device side is the one GEMV kernel."""
        Q = q.shape[0]
        dev_index = self.rows.device.index
        stream = _raw_stream(dev_index)
        key = (Q, k, path, stream, host_out)
        plans = self._plans
        plan = plans.get(key)
        if plan is None:
            import ctypes

            lib = ops._lib.load()
            N, D = self.rows.shape
            dt = ops._dtype_code(self.rows)
            need = lib.icr_cos_topk_workspace_bytes(Q, N, D, dt, k, path, int(self.planes is not None))
            ws = torch.zeros(max(int(need), 256), dtype=torch.uint8, device=self.device)
            if host_out:  # pinned host memory is mapped into the device's address space (UVA): the kernel writes it directly
                vals = torch.empty(Q, k, dtype=torch.float32).pin_memory()
                ids = torch.empty(Q, k, dtype=torch.int64).pin_memory()
            else:
                vals = torch.empty(Q, k, dtype=torch.float32, device=self.device)
                ids = torch.empty(Q, k, dtype=torch.int64, device=self.device)
            c64, cvp = ctypes.c_int64, ctypes.c_void_p
            args = [None, c64(Q), c64(D), cvp(self.rows.data_ptr()), c64(N), c64(ops._ld(self.rows)), c64(D), ctypes.c_int(dt),
                    cvp(ops._ptr(self.planes)), cvp(ops._ptr(self.inv_norms)), cvp(None), ctypes.c_int(k), c64(self.row_offset),
                    ctypes.c_int(path | ops.PATH_WS_RESIDENT), cvp(vals.data_ptr()), cvp(ids.data_ptr()), cvp(ws.data_ptr()),
                    ctypes.c_size_t(ws.numel()), cvp(stream)]
            if len(plans) >= 64:
                plans.clear()
            plan = plans[key] = (lib.icr_cos_topk, args, vals, ids, ws, vals.data_ptr(), ids.data_ptr())
        fn, args, vals, ids = plan[:4]
        args[0] = q.data_ptr()
        if fresh_out:  # the caller keeps the result: new tensors instead of the plan's static ones
            out_v = torch.empty(Q, k, dtype=torch.float32, device=self.device)
            out_i = torch.empty(Q, k, dtype=torch.int64, device=self.device)
            args[14], args[15] = out_v.data_ptr(), out_i.data_ptr()
        else:
            out_v, out_i = vals, ids
            args[14], args[15] = plan[5], plan[6]
        if dev_index != torch.cuda.current_device():
            with torch.cuda.device(self.device):
                rc = fn(*args)
        else:
            rc = fn(*args)
        if rc:
            ops._lib.check(rc)
        return out_v, out_i

    def topk_host(self, queries: torch.Tensor, k: int, *, out: tuple[torch.Tensor, torch.Tensor] | None = None,
                  n_chunks: int | None = None, path: int = ops.PATH_AUTO, splits: list[int] | None = None, join: bool = True):
        """Host-to-host top-k: CPU query matrix in, CPU (values [Q,k] f32, ids [Q,k] i64) out.

        The batch is cut into pieces that flow through three side streams - upload, rank, download - so the copies of
        one piece overlap the kernels of another (the B200 has a copy engine per direction). All uploads are enqueued
        first: they then run back to back from the first microsecond instead of waiting for the host to enqueue the
        kernels of the piece before. The kernels of the pieces run in order on ONE stream: side by side they only slow
        each other down (measured, benchmarks/e2e_timeline.py). What stays exposed is the first piece's upload and the
        last piece's download, while every piece costs ~0.1 ms of fixed kernel time on the 49,688-row catalog; the
        default cut for large batches is 15 % / 70 % / 15 % (C2: 1.00 ms against 1.04 ms for 30 % / 70 % and 1.21 ms
        unpipelined; the round-1 layout, one stream per piece, measured 1.16 ms). Pass pinned tensors
        (and pinned `out`) for truly asynchronous copies. Returns after enqueueing; the current stream waits on the
        side streams, so `torch.cuda.current_stream().synchronize()` makes the outputs valid.

        ``join=False`` (batches in flight): the current stream does NOT wait; the call returns ``(values, ids, done)`` with
        ``done`` a CUDA event recorded behind the last download. Successive calls then pipeline through the three side
        streams - the upload of batch s+1 runs under the kernels of batch s and the download of batch s-1 - which is how a
        bulk job keeps both copy engines and the SMs busy at once. Each batch in flight needs its own `out` buffers; wait on
        ``done`` (``done.synchronize()``) before reading or re-using them.
        """
        if queries.is_cuda:
            raise ValueError("topk_host takes host tensors; use topk() for device-resident queries")
        if queries.dim() == 1:
            queries = queries.unsqueeze(0)
        Q = queries.shape[0]
        k = min(int(k), len(self))
        if out is None:
            out = (torch.empty(Q, k, dtype=torch.float32).pin_memory(), torch.empty(Q, k, dtype=torch.int64).pin_memory())
        vals_h, ids_h = out
        if Q == 0 or k < 1:
            return vals_h, ids_h
        if not hasattr(self, "_side_streams"):
            self._side_streams = [torch.cuda.Stream(self.device) for _ in range(3)]
        up, rank, down = self._side_streams
        cur = torch.cuda.current_stream(self.device)
        if splits is None and n_chunks is None:
            if Q >= 2048:
                edge = 3 * Q // 20
                splits = [edge, Q - 2 * edge, edge]
            else:
                n_chunks = 1
        if splits is None:
            n_chunks = max(1, min(n_chunks, (Q + 255) // 256))
            per = -(-Q // n_chunks)
            bounds = [(c * per, min(Q, (c + 1) * per)) for c in range(n_chunks)]
        else:  # explicit piece sizes (a short first piece starts the kernels sooner, a short last one shortens the D2H tail)
            edges = [0]
            for n in splits:
                edges.append(min(Q, edges[-1] + int(n)))
            edges[-1] = Q
            bounds = list(zip(edges[:-1], edges[1:]))
        bounds = [(lo, hi) for lo, hi in bounds if lo < hi]
        start = torch.cuda.Event()
        start.record(cur)
        for st in (up, rank, down):
            st.wait_event(start)
        staged = []
        with torch.cuda.stream(up):
            for lo, hi in bounds:
                qd = queries[lo:hi].to(self.device, non_blocking=True)
                qd.record_stream(rank)  # allocated on `up`, read on `rank`
                ev = torch.cuda.Event()
                ev.record(up)
                staged.append((qd, ev))
        for (lo, hi), (qd, ev) in zip(bounds, staged):
            rank.wait_event(ev)
            with torch.cuda.stream(rank):
                qd = ops._like_catalog(qd, self.dtype)
                v, i = ops.cos_topk(qd, self.rows, k, cat_planes=self.planes, cat_inv_norms=self.inv_norms,
                                    row_offset=self.row_offset, path=path)
                v.record_stream(down)
                i.record_stream(down)
                done = torch.cuda.Event()
                done.record(rank)
            down.wait_event(done)
            with torch.cuda.stream(down):
                vals_h[lo:hi].copy_(v, non_blocking=True)
                ids_h[lo:hi].copy_(i, non_blocking=True)
        if not join:
            done_all = torch.cuda.Event()
            done_all.record(down)
            return vals_h, ids_h, done_all
        cur.wait_stream(down)  # `down` waited on every piece of `rank`, which waited on every upload
        return vals_h, ids_h

    # per-query exclusion bitmaps of one call stay below this; larger batches are split into query chunks
    EXCLUSION_BITS_MAX_BYTES = 256 << 20

    def topk(self, queries, k: int, *, exclude_mask: torch.Tensor | None = None, exclude_rows=None, path: int = ops.PATH_AUTO,
             peer=None, include_rows=None):
        """(values [Q,k], global ids [Q,k]) of the k most cosine-similar rows per query. With ``peer``
        (``PeerExchange.next_call()``; needs k <= len(self)) the rows are one rank's shard and the result is the global
        top-k over all ranks' shards (``ops.cos_topk``).

        ``exclude_mask`` (uint8/bool [len(self)]) drops rows for every query. ``exclude_rows`` gives one collection of
        local rows per query (before ``row_offset``; out-of-range rows are ignored) that this query never returns: the
        batch is searched in one fused call per chunk of queries whose exclusion bitmap (``ops.query_exclusion_bits``,
        ceil(len(self)/32) words per query) fits EXCLUSION_BITS_MAX_BYTES. A query with fewer than k eligible rows gets a
        (-inf, -1) tail.

        ``include_rows`` is the opposite: one candidate list of local rows per query (Q iterables, or an ``(offsets, rows)``
        CSR pair of int64 tensors with distinct rows per list), and query q ranks only its list (``ops.cos_topk_subset``):
        the call reads the listed rows, not the catalog. It cannot be combined with ``exclude_rows``, ``exclude_mask`` or
        ``peer``; out-of-range rows are ignored and a list with fewer than k valid rows gets a (-inf, -1) tail."""
        if include_rows is not None:
            if exclude_rows is not None or exclude_mask is not None or peer is not None:
                raise ValueError("include_rows cannot be combined with exclude_rows, exclude_mask or peer")
            return self._topk_including(queries, k, include_rows)
        if exclude_rows is not None:
            return self._topk_excluding(queries, k, exclude_rows, exclude_mask, path, peer)
        q = queries
        rows = self.rows
        if (exclude_mask is None and peer is None and isinstance(q, torch.Tensor) and q.dim() == 2 and 1 <= q.shape[0] <= 7 and q.is_cuda
                and q.dtype == self.query_dtype and q.device == rows.device and q.shape[1] == rows.shape[1] == self.input_dim and q.is_contiguous()
                and q.data_ptr() % 16 == 0 and 1 <= int(k) <= rows.shape[0]):
            # request-sized device query in the catalog's layout: the prepared argument list of the request path, fresh outputs
            with self.request_lock:
                return self._prepared_call(q, int(k), path, fresh_out=True)
        q = self._device_queries(queries)
        if peer is not None and int(k) > len(self):
            raise ValueError("a sharded call needs k <= the shard's rows (pad the shard's own lists and use peer_exchange_merge instead)")
        k = min(int(k), len(self))
        if k < 1:
            return (torch.empty(q.shape[0], 0, device=self.device), torch.empty(q.shape[0], 0, dtype=torch.int64, device=self.device))
        ws = self._resident_workspace(q.shape[0], k, path, peer is not None) if q.shape[0] <= 8 else None
        return ops.cos_topk(q, self.rows, k, cat_planes=self.planes, cat_inv_norms=self.inv_norms, exclude_mask=exclude_mask,
                            row_offset=self.row_offset, path=path, workspace=ws, peer=peer)

    def _topk_including(self, queries, k: int, include_rows):
        q = self._device_queries(queries)
        if q.dim() == 1:
            q = q.unsqueeze(0)
        Q = q.shape[0]
        if int(k) > ops.MAX_K:
            raise ValueError(f"k={k} outside [1, {ops.MAX_K}]")
        k = min(int(k), len(self))
        if k < 1:
            return (torch.empty(Q, 0, device=self.device), torch.empty(Q, 0, dtype=torch.int64, device=self.device))
        csr = include_rows if isinstance(include_rows, tuple) and len(include_rows) == 2 and all(
            isinstance(t, torch.Tensor) for t in include_rows) else list(include_rows)
        if not isinstance(csr, tuple) and len(csr) != Q:
            raise ValueError(f"include_rows has {len(csr)} entries for {Q} queries")
        return ops.cos_topk_subset(q, self.rows, k, csr, cat_inv_norms=self.inv_norms, row_offset=self.row_offset)

    def _topk_excluding(self, queries, k: int, exclude_rows, exclude_mask, path: int, peer):
        if peer is not None:
            raise ValueError("exclude_rows is not supported on a sharded call")
        q = self._device_queries(queries)
        if q.dim() == 1:
            q = q.unsqueeze(0)
        Q = q.shape[0]
        exclude_rows = list(exclude_rows)
        if len(exclude_rows) != Q:
            raise ValueError(f"exclude_rows has {len(exclude_rows)} entries for {Q} queries")
        k = min(int(k), len(self))
        if k < 1:
            return (torch.empty(Q, 0, device=self.device), torch.empty(Q, 0, dtype=torch.int64, device=self.device))
        per_query = 4 * ops.exclusion_words(len(self))
        chunk = max(1, self.EXCLUSION_BITS_MAX_BYTES // per_query)
        outs = []
        for lo in range(0, Q, chunk):
            hi = min(Q, lo + chunk)
            bits = ops.query_exclusion_bits(exclude_rows[lo:hi], len(self), self.device)
            outs.append(ops.cos_topk(q[lo:hi], self.rows, k, cat_planes=self.planes, cat_inv_norms=self.inv_norms,
                                     exclude_mask=exclude_mask, exclude_bits=bits, row_offset=self.row_offset, path=path))
        if len(outs) == 1:
            return outs[0]
        return torch.cat([v for v, _ in outs]), torch.cat([i for _, i in outs])

    def _resident_workspace(self, Q: int, k: int, path: int, sharded: bool = False) -> torch.Tensor:
        """Request-sized calls keep one zero-initialised workspace per (shape, stream): the library then skips the memset of
        its merge counter (ICR_PATH_WS_RESIDENT), 2-3 µs of a ~30 µs request. Keyed by stream: calls on one stream are ordered."""
        if not hasattr(self, "_resident"):
            self._resident = {}
        key = (Q, k, path, sharded, torch.cuda.current_stream(self.device).cuda_stream)
        ws = self._resident.get(key)
        if ws is None:
            lib = ops._lib.load()
            ws_bytes = lib.icr_cos_topk_sharded_workspace_bytes if sharded else lib.icr_cos_topk_workspace_bytes
            need = ws_bytes(Q, self.rows.shape[0], self.rows.shape[1], ops._dtype_code(self.rows), k, path, int(self.planes is not None))
            ws = torch.zeros(max(int(need), 256), dtype=torch.uint8, device=self.device)
            if len(self._resident) >= 64:  # many distinct request shapes: start over rather than grow without bound
                self._resident.clear()
            self._resident[key] = ws
        return ws


def chunk_spans(lo: int, hi: int, chunk_rows: int) -> list[tuple[int, int]]:
    """[lo, hi) cut into consecutive spans of at most chunk_rows rows."""
    chunk_rows = max(1, int(chunk_rows))
    return [(s, min(hi, s + chunk_rows)) for s in range(lo, hi, chunk_rows)]


_PINNED: dict = {}  # (slot, element size) -> pinned byte buffer, kept between loads (cudaHostAlloc costs tens of ms)
_COPY_THREADS = 4
_copy_pool = None


def _pinned_stage(slot: int, rows: int, cols: int, dtype: torch.dtype) -> torch.Tensor:
    need = rows * cols * torch.empty((), dtype=dtype).element_size()
    buf = _PINNED.get(slot)
    if buf is None or buf.numel() < need:
        buf = torch.empty(need, dtype=torch.uint8).pin_memory()
        _PINNED[slot] = buf
    return buf[:need].view(dtype).view(rows, cols)


def release_staging() -> None:
    """Free the pinned staging buffers and the copy threads kept between loads (they are re-created on demand)."""
    global _copy_pool
    _PINNED.clear()
    if _copy_pool is not None:
        _copy_pool.shutdown(wait=True)
        _copy_pool = None


def _host_copy(dst: np.ndarray, src: np.ndarray) -> None:
    """dst[:] = src with a few threads: numpy releases the GIL while copying, and one core moves only ~8 GB/s out of
    the page cache — less than the PCIe link the staging buffer feeds."""
    global _copy_pool
    n = dst.shape[0]
    if n < 4096:
        np.copyto(dst, src, casting="same_kind")
        return
    if _copy_pool is None:
        from concurrent.futures import ThreadPoolExecutor

        _copy_pool = ThreadPoolExecutor(_COPY_THREADS)
    step = -(-n // _COPY_THREADS)
    list(_copy_pool.map(lambda s: np.copyto(dst[s : s + step], src[s : s + step], casting="same_kind"), range(0, n, step)))


def upload_rows(src: np.ndarray, lo: int, hi: int, *, device: torch.device, dtype: torch.dtype, normalize: bool = False,
                chunk_rows: int = 1 << 15, source_is_bf16_bits: bool = False) -> torch.Tensor:
    """Rows [lo, hi) of a host (typically memory-mapped) matrix -> a device tensor [hi-lo, D] of `dtype`.

    Two pinned staging buffers alternate: while chunk i crosses PCIe (and is converted by ``icr_convert_rows`` on
    the same side stream), the host copies chunk i+1 out of the page cache into the other buffer. fp32 -> fp32
    without normalisation lands directly in the destination; bf16 bit patterns from the sidecar likewise.
    """
    n, D = hi - lo, int(src.shape[1])
    out = torch.empty(n, D, dtype=dtype, device=device)
    if n == 0:
        return out
    if source_is_bf16_bits and (dtype != torch.bfloat16 or normalize):
        raise ValueError("the bf16 sidecar can only be uploaded as an un-normalised bfloat16 catalog")
    direct = source_is_bf16_bits or (dtype == torch.float32 and not normalize)
    if not direct and D % 4:
        raise ValueError("icr_convert_rows needs an embedding dim that is a multiple of 4")
    stage_dtype = torch.int16 if source_is_bf16_bits else torch.float32
    np_dtype = np.uint16 if source_is_bf16_bits else np.float32
    chunk_rows = min(max(1, int(chunk_rows)), n)
    pinned = [_pinned_stage(b, chunk_rows, D, stage_dtype) for b in range(2)]
    staged = None if direct else [torch.empty(chunk_rows, D, dtype=torch.float32, device=device) for _ in range(2)]
    free = [torch.cuda.Event(), torch.cuda.Event()]  # recorded when the buffer pair's last consumer has run
    side = torch.cuda.Stream(device)
    side.wait_stream(torch.cuda.current_stream(device))
    dst_bits = out.view(torch.int16) if source_is_bf16_bits else None
    for i, (s0, s1) in enumerate(chunk_spans(lo, hi, chunk_rows)):
        b, m = i & 1, s1 - s0
        if i >= 2:
            free[b].synchronize()
        host = pinned[b][:m]
        _host_copy(host.numpy().view(np_dtype), src[s0:s1])
        with torch.cuda.stream(side):
            if direct:
                (dst_bits if source_is_bf16_bits else out)[s0 - lo : s1 - lo].copy_(host, non_blocking=True)
            else:
                staged[b][:m].copy_(host, non_blocking=True)
                ops.convert_rows(staged[b][:m], out[s0 - lo : s1 - lo], normalize=normalize)
            free[b].record(side)
    torch.cuda.current_stream(device).wait_stream(side)
    for t in staged or ():
        t.record_stream(side)  # allocated on the current stream, last used on the side stream
    side.synchronize()  # the staging buffers are reused by the next load
    return out


def upload_quantized(src: np.ndarray, lo: int, hi: int, *, device: torch.device,
                     chunk_rows: int = 1 << 15) -> tuple[torch.Tensor, torch.Tensor]:
    """Rows [lo, hi) of a host fp32 matrix (D % 4 == 0) -> (int8 codes [hi-lo, round_up(D, 16)], factors [hi-lo]) on the
    device, chunk by chunk through the pinned staging of ``upload_rows``: ``icr_quantize_rows`` writes each chunk's codes
    and factors where they belong. Raises ValueError if a row is not finite (checked on the device, one sync at the end)."""
    n, D = hi - lo, int(src.shape[1])
    codes = torch.empty(n, (D + 15) // 16 * 16, dtype=torch.int8, device=device)
    factors = torch.empty(n, dtype=torch.float32, device=device)
    if n == 0:
        return codes, factors
    lib = ops._lib.load()
    chunk_rows = min(max(1, int(chunk_rows)), n)
    pinned = [_pinned_stage(b, chunk_rows, D, torch.float32) for b in range(2)]
    staged = [torch.empty(chunk_rows, D, dtype=torch.float32, device=device) for _ in range(2)]
    bad = torch.zeros((), dtype=torch.int64, device=device)
    free = [torch.cuda.Event(), torch.cuda.Event()]
    side = torch.cuda.Stream(device)
    side.wait_stream(torch.cuda.current_stream(device))
    for i, (s0, s1) in enumerate(chunk_spans(lo, hi, chunk_rows)):
        b, m = i & 1, s1 - s0
        if i >= 2:
            free[b].synchronize()
        host = pinned[b][:m]
        _host_copy(host.numpy(), src[s0:s1])
        with torch.cuda.stream(side):
            x = staged[b][:m]
            x.copy_(host, non_blocking=True)
            bad += (~torch.isfinite(x)).sum()
            with ops._on(device):
                ops._lib.check(lib.icr_quantize_rows(x.data_ptr(), m, D, D, codes[s0 - lo].data_ptr(), codes.shape[1],
                                                     factors[s0 - lo :].data_ptr(), side.cuda_stream))
            free[b].record(side)
    torch.cuda.current_stream(device).wait_stream(side)
    for t in (*staged, bad):
        t.record_stream(side)
    side.synchronize()
    if int(bad):
        raise ValueError("int8 catalog rows must be finite")
    return codes, factors
