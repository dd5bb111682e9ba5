"""``Recommender`` / ``MonitoredRecommender`` drop-ins with the catalog resident on the B200.

Same constructor, attributes and ``recommend`` signatures as the reference
(src/inference/serve_recommendations.py:133-293); the encoder (SentenceTransformer) and the
on-disk index are unchanged. What changes is the tail: instead of
``cos_sim(query, catalog)[0]`` -> full ``argsort`` -> Python walk (:213-225, :250-262), one fused
kernel scores the HBM-resident catalog and selects the top ``top_k + |excluded ∩ catalog|`` rows,
and the walk runs over those few candidates — the observable result is identical. ``recommend_batch``
serves many requests in one encode and one fused top-k, each request with its own exclusion set.
"""

from __future__ import annotations

import contextlib
import json
import logging
import os
import threading
import time
from dataclasses import dataclass
from pathlib import Path
from typing import Optional

import numpy as np
import torch

from . import ops
from .index import DeviceCatalog, EmbeddingIndex

logger = logging.getLogger(__name__)


@dataclass
class RecommendationMetrics:
    """Per-request metrics, field for field the reference's dataclass (serve_recommendations.py:52-63)."""

    user_id: str
    query_embedding_time_ms: float
    similarity_compute_time_ms: float
    total_latency_ms: float
    num_recommendations: int
    top_score: float
    avg_score: float
    timestamp: float


class _ReadWriteLock:
    """Many readers or one writer; a waiting writer keeps new readers out until it is done."""

    def __init__(self):
        self._cond = threading.Condition()
        self._readers = 0
        self._writing = False
        self._writers_waiting = 0

    @contextlib.contextmanager
    def read(self):
        with self._cond:
            while self._writing or self._writers_waiting:
                self._cond.wait()
            self._readers += 1
        try:
            yield
        finally:
            with self._cond:
                self._readers -= 1
                if self._readers == 0:
                    self._cond.notify_all()

    @contextlib.contextmanager
    def write(self):
        with self._cond:
            self._writers_waiting += 1
            while self._writing or self._readers:
                self._cond.wait()
            self._writers_waiting -= 1
            self._writing = True
        try:
            yield
        finally:
            with self._cond:
                self._writing = False
                self._cond.notify_all()


class Recommender:
    """Two-tower recommender: encode the user context, return top-k products by cosine similarity.

    ``update_products``, ``remove_products`` and ``update_corpus`` change the catalog under a running server: the texts that
    are new or changed are encoded, and the resident catalog is changed in place (``DeviceCatalog.update_rows`` /
    ``append_rows`` / ``remove_rows``) instead of being rebuilt. Requests run concurrently with each other; a change waits
    for the running ones and holds new ones back until it is done, so a request sees the catalog wholly before or wholly
    after it."""

    def __init__(
        self,
        model_dir: Path | str,
        corpus_path: Path,
        batch_size: int = 64,
        use_index: bool = True,
        *,
        model=None,
        catalog_dtype: torch.dtype | None = None,
        device: torch.device | str | None = None,
    ):
        p = Path(model_dir)
        self.model_dir = p.resolve() if p.exists() else model_dir
        self._batch_size = batch_size
        self._rw = _ReadWriteLock()  # requests read, catalog changes write
        self._update_lock = threading.RLock()  # one change at a time, encoding included
        self.corpus_path = Path(corpus_path).resolve()
        self.product_ids, self.product_texts = self._load_corpus()
        self.pid_to_text = dict(zip(self.product_ids, self.product_texts))
        self._pid_to_row = {pid: i for i, pid in enumerate(self.product_ids)}
        self.model = model if model is not None else self._load_model()
        # host copy kept because callers read `.product_embeddings` (routes, tests/conftest.py:34-49)
        self.product_embeddings = self._load_or_build_embeddings(batch_size, use_index)
        if catalog_dtype is None:
            env = os.getenv("ICR_CATALOG_DTYPE", "fp32").lower()
            catalog_dtype = {"bf16": torch.bfloat16, "bfloat16": torch.bfloat16, "fp16": torch.float16, "float16": torch.float16,
                             "int8": torch.int8, "i8": torch.int8}.get(env, torch.float32)
        dev = torch.device(device) if device is not None else None
        self.catalog = DeviceCatalog(self.product_embeddings, device=dev, dtype=catalog_dtype)
        # SURVEY §8f row 1: ask the encoder for a device tensor so that the query never visits the host between the
        # encoder and the scoring kernel (the reference takes numpy, serve_recommendations.py:213); encoders that do
        # not know `convert_to_tensor` (test doubles) keep the reference call.
        self._query_on_device = os.getenv("ICR_QUERY_ON_DEVICE", "1") != "0"

    # ---- loading: same behaviour as the reference ------------------------------------------
    def _load_corpus(self) -> tuple[list[str], list[str]]:
        with open(self.corpus_path) as f:
            corpus = json.load(f)
        ids = list(corpus.keys())
        return ids, [corpus[pid] for pid in ids]

    def _inference_device(self) -> str:
        override = os.getenv("INFERENCE_DEVICE")
        if override:
            return override
        return "cuda" if torch.cuda.is_available() else "cpu"

    def _load_model(self):
        try:
            from sentence_transformers import SentenceTransformer
        except ImportError as e:  # the encoder is the reference's dependency, not part of this path
            raise ImportError("sentence-transformers is required to load an encoder; pass model=<object with .encode()> otherwise") from e
        device = self._inference_device()
        logger.info("Using inference device: %s", device)
        return SentenceTransformer(str(self.model_dir), device=device)

    def _load_or_build_embeddings(self, batch_size: int, use_index: bool) -> np.ndarray:
        index = EmbeddingIndex(self.corpus_path, self.model_dir)
        if use_index:
            cached = index.load(self.product_ids)
            if cached is not None:
                logger.info("Loaded model from %s, corpus %d products (embeddings from index)", self.model_dir, len(self.product_ids))
                return cached
        embeddings = self.model.encode(self.product_texts, batch_size=batch_size, show_progress_bar=True, normalize_embeddings=True)
        embeddings = np.asarray(embeddings)
        if use_index:
            index.save(self.product_ids, embeddings)
        logger.info("Loaded model from %s, corpus %d products", self.model_dir, len(self.product_ids))
        return embeddings

    # ---- the hot path ----------------------------------------------------------------------
    def _encode_query(self, query: str):
        if self._query_on_device:
            try:
                return self.model.encode([query], normalize_embeddings=True, convert_to_tensor=True)[0]
            except TypeError:
                self._query_on_device = False
        return self.model.encode([query], normalize_embeddings=True)[0]

    def _rank(self, query_emb, top_k: int, exclude_product_ids: set[str] | None) -> list[tuple[str, float]]:
        """Equals: sort all rows by score, drop excluded ids, keep the first top_k."""
        with self._rw.read():
            return self._rank_locked(query_emb, top_k, exclude_product_ids)

    def _rank_locked(self, query_emb, top_k: int, exclude_product_ids: set[str] | None) -> list[tuple[str, float]]:
        n = len(self.product_ids)
        if top_k <= 0 or n == 0:
            return []
        if top_k > ops.MAX_K:
            raise ValueError(f"top_k={top_k} exceeds the fused kernel limit {ops.MAX_K} (the reference API caps top_k at 100)")
        excluded_rows = [self._pid_to_row[p] for p in (exclude_product_ids or ()) if p in self._pid_to_row]
        want = min(top_k, n - len(excluded_rows))
        if want <= 0:
            return []
        if top_k + len(excluded_rows) <= ops.MAX_K:
            # exact: the best (top_k + #excluded) rows contain the best top_k non-excluded ones
            k_fetch = top_k + len(excluded_rows)
            # few distinct shapes -> few prepared calls / CUDA graphs; exact up to 16 (the one-trip merge: top-10 with no
            # exclusions is 2 us faster at k = 10 than at k = 16), then steps (profiles/r02_k1_request_by_k.txt)
            k_fetch = min(n, k_fetch if k_fetch <= 16 else next(b for b in (24, 32, 48, 64, 100, 128, 192, 256) if b >= k_fetch))
            # the graph's static query / output tensors are shared by every caller of this catalog: copy-in, replay and
            # host read happen under the catalog's lock so that concurrent requests (a sync route, run_in_executor, a batch
            # job) cannot read each other's results - the reference's recommend() is safe to call from several threads
            if isinstance(query_emb, torch.Tensor) and query_emb.is_cuda:
                # one kernel launch; its last CTA writes the k results into pinned host memory, one stream synchronisation
                vals, ids = self.catalog.topk_request(query_emb, k_fetch)
                vals, ids = vals[0], ids[0]
            else:
                with self.catalog.request_lock:
                    vals, ids = self.catalog.topk_small(query_emb, k_fetch, copy=False)
                    vals = vals[0].tolist()  # device->host reads; they synchronise the stream
                    ids = ids[0].tolist()
            mask_rows = set(excluded_rows)
        else:
            # unbounded exclusion lists: mask rows on the device instead of over-fetching
            mask = torch.zeros(n, dtype=torch.uint8, device=self.catalog.device)
            if excluded_rows:
                mask[torch.as_tensor(excluded_rows, device=self.catalog.device)] = 1
            k_fetch = min(want, ops.MAX_K)
            vals, ids = self.catalog.topk(query_emb, k_fetch, exclude_mask=mask)
            mask_rows = set()
            vals = vals[0].tolist()
            ids = ids[0].tolist()
        out: list[tuple[str, float]] = []
        for s, r in zip(vals, ids):
            if r < 0 or r in mask_rows:
                continue
            out.append((self.product_ids[r], float(s)))
            if len(out) >= top_k:
                break
        return out

    def _rank_candidates(self, query_emb, top_k: int, exclude_product_ids, candidate_product_ids) -> list[tuple[str, float]]:
        """Equals: sort all rows by score, keep the candidates that are not excluded, keep the first top_k. Only the
        candidates' rows are read (``DeviceCatalog.topk(..., include_rows=...)``)."""
        with self._rw.read():
            if top_k <= 0 or not self.product_ids:
                return []
            if top_k > ops.MAX_K:
                raise ValueError(f"top_k={top_k} exceeds the fused kernel limit {ops.MAX_K} (the reference API caps top_k at 100)")
            rows = self._candidate_rows(candidate_product_ids, exclude_product_ids)
            if not rows:
                return []
            vals, ids = self.catalog.topk(query_emb, min(top_k, len(rows)), include_rows=[rows])
            return [(self.product_ids[r], float(s)) for s, r in zip(vals[0].tolist(), ids[0].tolist()) if r >= 0]

    def _candidate_rows(self, candidate_product_ids, exclude_product_ids) -> list[int]:
        """Catalog rows of the known candidates minus the exclusions, each once."""
        excluded = set(exclude_product_ids or ())
        return [self._pid_to_row[p] for p in dict.fromkeys(candidate_product_ids) if p in self._pid_to_row and p not in excluded]

    def recommend(self, query: str, top_k: int = 10, exclude_product_ids: set[str] | None = None, *,
                  candidate_product_ids=None) -> list[tuple[str, float]]:
        """Return top-k (product_id, score) sorted by cosine similarity.

        ``candidate_product_ids`` restricts the ranking to those products (a user's previous purchases, the products in
        stock, one aisle, a candidate set from another stage): the result equals ranking every product and keeping the
        candidates that are not excluded. Unknown ids are ignored; an empty collection gives []."""
        if candidate_product_ids is None:
            return self._rank(self._encode_query(query), top_k, exclude_product_ids)
        return self._rank_candidates(self._encode_query(query), top_k, exclude_product_ids, candidate_product_ids)

    def _encode_queries(self, queries: list[str]):
        if self._query_on_device:
            try:
                return self.model.encode(queries, normalize_embeddings=True, convert_to_tensor=True)
            except TypeError:
                self._query_on_device = False
        return self.model.encode(queries, normalize_embeddings=True)

    def recommend_batch(self, queries: list[str], top_k: int = 10,
                        exclude_product_ids: list[set[str] | None] | None = None, *,
                        candidate_product_ids: list | None = None) -> list[list[tuple[str, float]]]:
        """``recommend`` for many requests at once: entry i equals ``recommend(queries[i], top_k, exclude_product_ids[i])``.

        The queries are encoded in one ``encode`` call and ranked in one fused top-k over the resident catalog, each with
        its own exclusion set applied on the device (``DeviceCatalog.topk(..., exclude_rows=...)``): no per-request
        launches, and no limit on the size of an exclusion set. Unknown product ids are ignored; a request with fewer
        eligible products than top_k gets a shorter list.

        ``candidate_product_ids``: one entry per query, as ``recommend``'s keyword; ``None`` entries rank the whole catalog.
        The restricted queries run in one candidate-list call, the others in the fused call above."""
        queries = list(queries)
        if exclude_product_ids is not None and len(exclude_product_ids) != len(queries):
            raise ValueError(f"exclude_product_ids has {len(exclude_product_ids)} entries for {len(queries)} queries")
        if candidate_product_ids is not None:
            return self._recommend_batch_candidates(queries, top_k, exclude_product_ids, list(candidate_product_ids))
        if not queries:
            return []
        if top_k <= 0 or not self.product_ids:
            return [[] for _ in queries]
        if top_k > ops.MAX_K:
            raise ValueError(f"top_k={top_k} exceeds the fused kernel limit {ops.MAX_K} (the reference API caps top_k at 100)")
        embs = self._encode_queries(queries)
        with self._rw.read():
            n = len(self.product_ids)  # the catalog may have changed while the queries were encoded
            if n == 0:
                return [[] for _ in queries]
            excluded = [[self._pid_to_row[p] for p in (ex or ()) if p in self._pid_to_row]
                        for ex in (exclude_product_ids or [None] * len(queries))]
            k = min(top_k, n)
            vals, ids = self.catalog.topk(embs, k, exclude_rows=excluded if any(excluded) else None)
            return [[(self.product_ids[r], float(s)) for s, r in zip(vr, ir) if r >= 0] for vr, ir in zip(vals.tolist(), ids.tolist())]

    def _recommend_batch_candidates(self, queries, top_k, exclude_product_ids, candidates) -> list[list[tuple[str, float]]]:
        if len(candidates) != len(queries):
            raise ValueError(f"candidate_product_ids has {len(candidates)} entries for {len(queries)} queries")
        if not queries:
            return []
        if top_k <= 0 or not self.product_ids:
            return [[] for _ in queries]
        if top_k > ops.MAX_K:
            raise ValueError(f"top_k={top_k} exceeds the fused kernel limit {ops.MAX_K} (the reference API caps top_k at 100)")
        embs = self._encode_queries(queries)
        exclude = exclude_product_ids or [None] * len(queries)
        out: list[list[tuple[str, float]]] = [[] for _ in queries]
        with self._rw.read():
            n = len(self.product_ids)
            if n == 0:
                return out
            k = min(top_k, n)
            restricted = [i for i, c in enumerate(candidates) if c is not None]
            free = [i for i, c in enumerate(candidates) if c is None]
            if restricted:
                lists = [self._candidate_rows(candidates[i], exclude[i]) for i in restricted]
                vals, ids = self.catalog.topk(_pick(embs, restricted), k, include_rows=lists)
                for i, vr, ir in zip(restricted, vals.tolist(), ids.tolist()):
                    out[i] = [(self.product_ids[r], float(s)) for s, r in zip(vr, ir) if r >= 0]
            if free:
                excluded = [[self._pid_to_row[p] for p in (exclude[i] or ()) if p in self._pid_to_row] for i in free]
                vals, ids = self.catalog.topk(_pick(embs, free), k, exclude_rows=excluded if any(excluded) else None)
                for i, vr, ir in zip(free, vals.tolist(), ids.tolist()):
                    out[i] = [(self.product_ids[r], float(s)) for s, r in zip(vr, ir) if r >= 0]
        return out

    # ---- catalog changes ---------------------------------------------------------------------------------
    def update_products(self, products: dict[str, str]) -> None:
        """Add or change products ({product id: text}). Only texts that are new or differ from the current ones are encoded,
        in one ``encode`` call; changed products are replaced in place and new ones appended, in the dict's order.
        ``product_ids``, ``product_texts``, ``pid_to_text`` and ``product_embeddings`` follow."""
        self._change({}, products)

    def remove_products(self, ids) -> None:
        """Remove products by id; unknown ids are ignored. The remaining products keep their order."""
        with self._update_lock:
            gone = [pid for pid in dict.fromkeys(ids) if pid in self._pid_to_row]
            with self._rw.write():
                self._remove_locked(gone)

    def update_corpus(self, corpus: dict[str, str]) -> None:
        """The corpus becomes `corpus`: products not in it are removed, changed ones replaced and new ones appended.
        Afterwards ``product_ids`` holds the surviving ids in their old order, then the new ids in corpus order, and
        ``recommend`` / ``recommend_batch`` answer as a fresh ``Recommender`` over ``{pid: corpus[pid] for pid in
        product_ids}`` with the same encoder. Writing the corpus file or the ``EmbeddingIndex`` is left to the caller
        (``EmbeddingIndex.save(product_ids, product_embeddings)``)."""
        with self._update_lock:
            self._change(corpus, corpus, remove_missing=True)

    def _plan_change(self, corpus: dict[str, str], products: dict[str, str], remove_missing: bool):
        """(removed ids, changed ids, new ids) of a change; reads the current state only."""
        gone = [pid for pid in self.product_ids if pid not in corpus] if remove_missing else []
        changed = [pid for pid, text in products.items() if pid in self._pid_to_row and self.pid_to_text[pid] != text]
        new = [pid for pid in products if pid not in self._pid_to_row]
        return gone, changed, new

    def _change(self, corpus: dict[str, str], products: dict[str, str], remove_missing: bool = False) -> None:
        with self._update_lock:
            products = {str(pid): text for pid, text in products.items()}
            gone, changed, new = self._plan_change(corpus, products, remove_missing)
            emb = None
            if changed or new:  # encoded before requests are held back
                emb = np.asarray(self.model.encode([products[p] for p in changed + new], batch_size=self._batch_size,
                                                   show_progress_bar=False, normalize_embeddings=True), dtype=np.float32)
                if emb.ndim != 2 or emb.shape[0] != len(changed) + len(new) or emb.shape[1] != self.catalog.input_dim:
                    raise ValueError(f"the encoder returned {emb.shape} for {len(changed) + len(new)} texts of dim {self.catalog.input_dim}")
                if not np.isfinite(emb).all():
                    raise ValueError("the encoder returned non-finite embeddings")
            if not (gone or changed or new):
                return
            with self._rw.write():
                self._remove_locked(gone)
                nc = len(changed)
                if changed:
                    rows = [self._pid_to_row[p] for p in changed]
                    self.catalog.update_rows(rows, emb[:nc])
                    if not self.product_embeddings.flags.writeable:
                        self.product_embeddings = np.array(self.product_embeddings)
                    self.product_embeddings[rows] = emb[:nc]
                    for p, r in zip(changed, rows):
                        self.product_texts[r] = products[p]
                        self.pid_to_text[p] = products[p]
                if new:
                    first = self.catalog.append_rows(emb[nc:]).start
                    self.product_embeddings = np.concatenate([np.asarray(self.product_embeddings), emb[nc:].astype(self.product_embeddings.dtype)])
                    for j, p in enumerate(new):
                        self.product_ids.append(p)
                        self.product_texts.append(products[p])
                        self.pid_to_text[p] = products[p]
                        self._pid_to_row[p] = first + j

    def _remove_locked(self, gone: list[str]) -> None:
        if not gone:
            return
        kept = self.catalog.remove_rows([self._pid_to_row[p] for p in gone])
        for p in gone:
            del self.pid_to_text[p]
        self.product_ids = [self.product_ids[i] for i in kept]
        self.product_texts = [self.product_texts[i] for i in kept]
        self.product_embeddings = np.asarray(self.product_embeddings)[kept]
        self._pid_to_row = {pid: i for i, pid in enumerate(self.product_ids)}


def _pick(embs, idx: list[int]):
    """Rows `idx` of a batch of query embeddings (an array or tensor, or a list of vectors)."""
    return embs[idx] if hasattr(embs, "shape") else [embs[i] for i in idx]


class MonitoredRecommender(Recommender):
    """Recommender with timing; sets ``last_metrics`` after each ``recommend``."""

    def __init__(self, *args, metrics_logger: Optional[logging.Logger] = None, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self.metrics_logger = metrics_logger or logging.getLogger("recommender.metrics")
        self.last_metrics: Optional[RecommendationMetrics] = None

    def recommend(self, query: str, top_k: int = 10, user_id: Optional[str] = None,
                  exclude_product_ids: set[str] | None = None, *, candidate_product_ids=None) -> list[tuple[str, float]]:
        start = time.time()
        query_emb = self._encode_query(query)
        encode_ms = (time.time() - start) * 1000
        sim_start = time.time()
        if candidate_product_ids is None:
            results = self._rank(query_emb, top_k, exclude_product_ids)  # includes the host read, so it is complete
        else:
            results = self._rank_candidates(query_emb, top_k, exclude_product_ids, candidate_product_ids)
        sim_ms = (time.time() - sim_start) * 1000
        total_ms = (time.time() - start) * 1000
        self.last_metrics = RecommendationMetrics(
            user_id=user_id or "anonymous",
            query_embedding_time_ms=encode_ms,
            similarity_compute_time_ms=sim_ms,
            total_latency_ms=total_ms,
            num_recommendations=len(results),
            top_score=results[0][1] if results else 0.0,
            avg_score=sum(s for _, s in results) / len(results) if results else 0.0,
            timestamp=time.time(),
        )
        m = self.last_metrics
        self.metrics_logger.info(
            "recommendation_served",
            extra={
                "user_id": m.user_id,
                "latency_ms": m.total_latency_ms,
                "encode_time_ms": m.query_embedding_time_ms,
                "similarity_time_ms": m.similarity_compute_time_ms,
                "num_results": m.num_recommendations,
                "top_score": m.top_score,
                "avg_score": m.avg_score,
            },
        )
        return results
