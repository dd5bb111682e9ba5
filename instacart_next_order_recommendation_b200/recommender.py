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

import json
import logging
import os
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


class Recommender:
    """Two-tower recommender: encode the user context, return top-k products by cosine similarity."""

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
        self.corpus_path = Path(corpus_path).resolve()
        self.product_ids, self.product_texts = self._load_corpus()
        self.pid_to_text = dict(zip(self.product_ids, self.product_texts))
        self._pid_to_row = {pid: i for i, pid in enumerate(self.product_ids)}
        self.model = model if model is not None else self._load_model()
        # host copy kept because callers read `.product_embeddings` (routes, tests/conftest.py:34-49)
        self.product_embeddings = self._load_or_build_embeddings(batch_size, use_index)
        if catalog_dtype is None:
            env = os.getenv("ICR_CATALOG_DTYPE", "fp32").lower()
            catalog_dtype = {"bf16": torch.bfloat16, "bfloat16": torch.bfloat16, "fp16": torch.float16, "float16": torch.float16}.get(env, torch.float32)
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

    def recommend(self, query: str, top_k: int = 10, exclude_product_ids: set[str] | None = None) -> list[tuple[str, float]]:
        """Return top-k (product_id, score) sorted by cosine similarity."""
        return self._rank(self._encode_query(query), top_k, exclude_product_ids)

    def _encode_queries(self, queries: list[str]):
        if self._query_on_device:
            try:
                return self.model.encode(queries, normalize_embeddings=True, convert_to_tensor=True)
            except TypeError:
                self._query_on_device = False
        return self.model.encode(queries, normalize_embeddings=True)

    def recommend_batch(self, queries: list[str], top_k: int = 10,
                        exclude_product_ids: list[set[str] | None] | None = None) -> list[list[tuple[str, float]]]:
        """``recommend`` for many requests at once: entry i equals ``recommend(queries[i], top_k, exclude_product_ids[i])``.

        The queries are encoded in one ``encode`` call and ranked in one fused top-k over the resident catalog, each with
        its own exclusion set applied on the device (``DeviceCatalog.topk(..., exclude_rows=...)``): no per-request
        launches, and no limit on the size of an exclusion set. Unknown product ids are ignored; a request with fewer
        eligible products than top_k gets a shorter list."""
        queries = list(queries)
        if exclude_product_ids is not None and len(exclude_product_ids) != len(queries):
            raise ValueError(f"exclude_product_ids has {len(exclude_product_ids)} entries for {len(queries)} queries")
        if not queries:
            return []
        n = len(self.product_ids)
        if top_k <= 0 or n == 0:
            return [[] for _ in queries]
        if top_k > ops.MAX_K:
            raise ValueError(f"top_k={top_k} exceeds the fused kernel limit {ops.MAX_K} (the reference API caps top_k at 100)")
        excluded = [[self._pid_to_row[p] for p in (ex or ()) if p in self._pid_to_row] for ex in (exclude_product_ids or [None] * len(queries))]
        embs = self._encode_queries(queries)
        k = min(top_k, n)
        vals, ids = self.catalog.topk(embs, k, exclude_rows=excluded if any(excluded) else None)
        return [[(self.product_ids[r], float(s)) for s, r in zip(vr, ir) if r >= 0] for vr, ir in zip(vals.tolist(), ids.tolist())]


class MonitoredRecommender(Recommender):
    """Recommender with timing; sets ``last_metrics`` after each ``recommend``."""

    def __init__(self, *args, metrics_logger: Optional[logging.Logger] = None, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        self.metrics_logger = metrics_logger or logging.getLogger("recommender.metrics")
        self.last_metrics: Optional[RecommendationMetrics] = None

    def recommend(self, query: str, top_k: int = 10, user_id: Optional[str] = None,
                  exclude_product_ids: set[str] | None = None) -> list[tuple[str, float]]:
        start = time.time()
        query_emb = self._encode_query(query)
        encode_ms = (time.time() - start) * 1000
        sim_start = time.time()
        results = self._rank(query_emb, top_k, exclude_product_ids)  # includes the host read, so it is complete
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
