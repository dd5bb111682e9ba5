"""Parity of the CUDA path (through the C ABI) with the oracle, on a B200.

Tolerances are BASELINE.json's: top-k scores within 1e-5 relative for fp32 and 2e-3 for bf16
(oracle = fp32 math on the bf16-rounded inputs), ids identical except across ties closer than the
tolerance, MNRL loss and gradients within 1e-4.
"""

import json
import math

import numpy as np
import pytest
import torch

import instacart_next_order_recommendation_b200 as icr
from instacart_next_order_recommendation_b200 import ops
from oracle import oracle

pytestmark = pytest.mark.gpu

F32_RTOL = 1e-5
BF16_RTOL = 2e-3
MNRL_ATOL = 1e-4


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert torch.cuda.is_available(), "run with -m gpu on a GPU box"
    torch.cuda.set_device(0)
    from instacart_next_order_recommendation_b200 import _lib

    assert _lib.load().icr_device_supported() == 1
    yield
    torch.cuda.synchronize()


def _check_topk(v, i, rv, ri, rtol):
    assert v.shape == rv.shape and i.shape == ri.shape
    v, i = v.cpu(), i.cpu()
    assert (v[:, :-1] >= v[:, 1:]).all(), "scores must be non-increasing"
    err, mism = oracle.compare_topk(v, i, rv, ri, rtol=rtol)
    assert err <= rtol, f"max relative score error {err}"
    assert mism == 0, f"{mism} id mismatches outside ties"
    for r in range(i.shape[0]):  # no duplicates
        assert len(set(i[r].tolist())) == i.shape[1]
    # rank-k membership: the last returned score may not fall below the oracle's k-th score by more than the tolerance
    # (compare_topk never treats the last rank as decisive for ids, so the boundary is asserted on the scores)
    rk = np.asarray(rv, dtype=np.float64)[:, -1]
    assert (v.double().numpy()[:, -1] >= rk - rtol * np.maximum(np.abs(rk), 0.05)).all(), "k-th returned score below the oracle's k-th"


PATHS = [ops.PATH_GEMV, ops.PATH_GEMM]


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("Q,N,D,k", [(1, 49688, 384, 10), (1, 49688, 384, 100), (3, 5000, 384, 10), (7, 20000, 768, 100),
                                      (9, 3000, 128, 32), (16, 7777, 384, 100), (1, 300, 64, 256)])
def test_f32_topk_vs_oracle(path, Q, N, D, k):
    if path == ops.PATH_GEMM and not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    items, _ = oracle.synth_clustered(N, D, seed=1234)
    queries, _ = oracle.synth_queries_from_items(items, Q, seed=4321)
    v, i = icr.cos_topk(queries.cuda(), items.cuda(), k, path=path)
    rv, ri = oracle.cos_topk(queries, items, k)
    _check_topk(v, i, rv, ri, F32_RTOL)


def _gemm_ok():
    try:
        q = torch.randn(128, 64, device="cuda")
        c = torch.randn(1024, 64, device="cuda")
        ops.cos_topk(q, c, 10, path=ops.PATH_GEMM)
        torch.cuda.synchronize()
        return True
    except ValueError:
        return False


@pytest.mark.parametrize("path", PATHS)
def test_isotropic_and_unnormalised_inputs(path):
    if path == ops.PATH_GEMM and not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    items = oracle.synth_isotropic(30000, 384, seed=1234)
    queries = oracle.synth_isotropic(5, 384, seed=4321)
    v, i = icr.cos_topk(queries.cuda(), items.cuda(), 100, path=path)
    _check_topk(v, i, *oracle.cos_topk(queries, items, 100), F32_RTOL)
    un_c = oracle.synth_unnormalised(9000, 384, seed=7)
    un_q = oracle.synth_unnormalised(4, 384, seed=8)
    v, i = icr.cos_topk(un_q.cuda(), un_c.cuda(), 50, path=path)
    _check_topk(v, i, *oracle.cos_topk(un_q, un_c, 50), F32_RTOL)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
@pytest.mark.parametrize("D", [384, 128, 768, 192, 64, 200, 1024])
@pytest.mark.parametrize("use_norms", [False, True])
def test_single_query_ring_kernel_row_shapes(dtype, D, use_norms):
    """K1 for one query across row lengths: full iterations only, a half-filled last iteration (the two half-warps
    split the tail's rows: 16-byte vector count % 32 == 16), other tails; with the row norms accumulated in the kernel
    or precomputed (icr_row_inv_norms, as DeviceCatalog passes them for bf16 catalogs). Un-normalised rows."""
    N = 30011
    items = oracle.synth_unnormalised(N, D, seed=77).to(dtype)
    query = oracle.synth_unnormalised(1, D, seed=78).to(dtype)
    it, qt = items.cuda(), query.cuda()
    inv = ops.row_inv_norms(it) if use_norms else None
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[::17] = 1
    rv_all = oracle.cos_sim(query.float(), items.float())[0]
    rtol = F32_RTOL if dtype == torch.float32 else 5e-5
    for k, m in ((100, None), (10, mask)):
        v, i = ops.cos_topk(qt, it, k, cat_inv_norms=inv, exclude_mask=m, path=ops.PATH_GEMV, row_offset=5)
        s = rv_all.clone()
        if m is not None:
            s[m.cpu().bool()] = float("-inf")
        rv, ri = torch.topk(s, k)
        _check_topk(v, i - 5, rv[None], ri[None], rtol)


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("Q,N,D,k", [(1, 40000, 768, 100), (3, 10000, 384, 10), (6, 25000, 768, 100)])
def test_bf16_topk_vs_fp32_math_on_rounded_inputs(path, Q, N, D, k):
    if path == ops.PATH_GEMM and not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    items, _ = oracle.synth_clustered(N, D, seed=1234)
    queries, _ = oracle.synth_queries_from_items(items, Q, seed=4321)
    ib, qb = items.bfloat16(), queries.bfloat16()
    v, i = icr.cos_topk(qb.cuda(), ib.cuda(), k, path=path)
    rv, ri = oracle.cos_topk(qb.float(), ib.float(), k)
    _check_topk(v, i, rv, ri, BF16_RTOL)
    # the kernel accumulates in fp32: it is in fact much closer than the bf16 tolerance
    err, _ = oracle.compare_topk(v.cpu(), i.cpu(), rv, ri, rtol=BF16_RTOL)
    assert err < 5e-5


def test_known_answers_on_device():
    d = 384
    e = torch.eye(d, device="cuda")
    s = icr.cos_sim(e[3] * 7.5, e[:8])
    assert s.shape == (1, 8) and s[0, 3].item() == pytest.approx(1.0, abs=1e-6) and s[0, 4].item() == 0.0
    assert icr.cos_sim(-2 * e[3], e[3]).item() == pytest.approx(-1.0, abs=1e-6)
    z = icr.cos_sim(torch.zeros(d, device="cuda"), e[:5])
    assert torch.isfinite(z).all() and (z == 0).all()
    q = torch.zeros(d)
    q[:6] = torch.tensor([0.1, -0.9, 0.5, 0.3, 0.0, 0.7])
    v, i = icr.cos_topk(q.cuda(), e, 3)
    assert i.tolist() == [[5, 2, 3]]
    # ties: equal scores come back in ascending row order
    c = torch.ones(1000, 64, device="cuda")
    v, i = icr.cos_topk(torch.ones(64, device="cuda"), c, 17)
    assert i.tolist() == [list(range(17))]
    # k clamps to the catalog size; numpy / list inputs are uploaded
    v, i = icr.cos_topk(np.ones(8, dtype=np.float32), [[1.0] * 8, [-1.0] * 8], 10)
    assert v.shape == (1, 2) and i.tolist() == [[0, 1]]


def test_dense_cos_sim_vs_oracle():
    a = oracle.synth_unnormalised(130, 384, seed=3)
    b = oracle.synth_unnormalised(777, 384, seed=4)
    got = icr.cos_sim(a.cuda(), b.cuda()).cpu()
    ref = oracle.cos_sim(a, b)
    # all-scores check: absolute, because cosines near 0 have unbounded relative error (SURVEY §8c)
    assert (got - ref).abs().max() <= 1e-5 * max(1.0, ref.abs().max().item())
    got = icr.cos_sim(a.bfloat16().cuda(), b.bfloat16().cuda()).cpu()
    ref = oracle.cos_sim(a.bfloat16().float(), b.bfloat16().float())
    assert (got - ref).abs().max() <= 1e-5
    # odd embedding dim (padded internally), 1-D operand
    a = torch.randn(50), torch.randn(9, 50)
    assert (icr.cos_sim(a[0], a[1]).cpu() - oracle.cos_sim(a[0], a[1])).abs().max() < 1e-6


@pytest.mark.parametrize("Qa,Nb,D", [(300, 5000, 384), (257, 5001, 384), (1000, 3000, 768), (64, 1024, 100), (300, 3000, 2048), (256, 2000, 4096)])
def test_dense_cos_sim_tensor_core_path(Qa, Nb, D):
    """Large enough for the tcgen05 dense epilogue (K2'): fp32 keeps 1e-5 through the fp16 hi/lo planes."""
    a = oracle.synth_unnormalised(Qa, D, seed=13)
    b = oracle.synth_unnormalised(Nb, D, seed=14)
    got = icr.cos_sim(a.cuda(), b.cuda()).cpu()
    ref = oracle.cos_sim(a, b)
    assert got.shape == ref.shape
    assert (got - ref).abs().max() <= 1e-5
    got = icr.cos_sim(a.bfloat16().cuda(), b.bfloat16().cuda()).cpu()
    ref = oracle.cos_sim(a.bfloat16().float(), b.bfloat16().float())
    assert (got - ref).abs().max() <= 1e-5


@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_edge_shapes(path, dtype):
    """Tiny / ragged problems through the C ABI: k > N pads with (-inf, -1), single rows, zero vectors, odd D,
    query counts that straddle the internal chunking, empty query batches."""
    tol = F32_RTOL if dtype == torch.float32 else BF16_RTOL
    g = torch.Generator().manual_seed(77)
    # k larger than the catalog: the ABI pads, the drop-in clamps
    c = torch.randn(5, 64, generator=g).to(dtype)
    q = torch.randn(3, 64, generator=g).to(dtype)
    v, i = ops.cos_topk(q.cuda(), c.cuda(), 9, path=path)
    rv, ri = oracle.cos_topk(q.float(), c.float(), 5)
    assert (i[:, 5:] == -1).all() and torch.isinf(v[:, 5:]).all() and (v[:, 5:] < 0).all()
    _check_topk(v[:, :5], i[:, :5], rv, ri, tol)
    v, i = icr.cos_topk(q.cuda(), c.cuda(), 9, path=path)
    assert v.shape == (3, 5)
    # one row, one query
    v, i = ops.cos_topk(q[:1].cuda(), c[:1].cuda(), 1, path=path)
    assert i.tolist() == [[0]] and abs(v.item() - oracle.cos_sim(q[:1].float(), c[:1].float()).item()) < 1e-3
    # zero rows in the catalog and a zero query score 0, never NaN
    c2 = torch.randn(300, 72, generator=g)
    c2[::7] = 0
    q2 = torch.randn(4, 72, generator=g)
    q2[1] = 0
    v, i = ops.cos_topk(q2.to(dtype).cuda(), c2.to(dtype).cuda(), 20, path=path)
    assert torch.isfinite(v).all() and (v[1] == 0).all()
    rv, ri = oracle.cos_topk(q2.to(dtype).float(), c2.to(dtype).float(), 20)
    err, _ = oracle.compare_topk(v.cpu(), i.cpu(), rv, ri, rtol=tol)
    assert err <= tol
    # embedding dim that is not a multiple of 64 (K tail of the tensor path), query count across chunk boundaries
    items, _ = oracle.synth_clustered(4100, 200, seed=78, n_centres=9)
    nq = 259 if path == ops.PATH_GEMV else 513
    queries, _ = oracle.synth_queries_from_items(items, nq, seed=79)
    v, i = ops.cos_topk(queries.to(dtype).cuda(), items.to(dtype).cuda(), 12, path=path)
    rv, ri = oracle.cos_topk(queries.to(dtype).float(), items.to(dtype).float(), 12)
    _check_topk(v, i, rv, ri, tol)
    # empty query batch
    v, i = ops.cos_topk(queries[:0].to(dtype).cuda(), items.to(dtype).cuda(), 12, path=path)
    assert v.shape == (0, 12) and i.shape == (0, 12)


def test_gemm_path_honours_exclusion_mask():
    items, _ = oracle.synth_clustered(6000, 128, seed=80)
    queries, _ = oracle.synth_queries_from_items(items, 140, seed=81)
    rv, ri = oracle.cos_topk(queries, items, 30)
    mask = torch.zeros(6000, dtype=torch.bool)
    mask[ri[:, :10].reshape(-1)] = True  # ban every query's ten best rows
    v, i = ops.cos_topk(queries.cuda(), items.cuda(), 15, exclude_mask=mask.cuda(), path=ops.PATH_GEMM)
    assert not mask[i.cpu()].any()
    sims = oracle.cos_sim(queries, items)
    sims[:, mask] = float("-inf")
    wv, wi = torch.topk(sims, 15, dim=1)
    _check_topk(v, i, wv, wi, F32_RTOL)


def test_exclusion_mask_and_row_offset():
    items, _ = oracle.synth_clustered(8000, 384, seed=5)
    queries, _ = oracle.synth_queries_from_items(items, 2, seed=6)
    rv, ri = oracle.cos_topk(queries, items, 40)
    mask = torch.zeros(8000, dtype=torch.uint8)
    banned = ri[0, :20:2]
    mask[banned] = 1
    v, i = ops.cos_topk(queries[:1].cuda(), items.cuda(), 10, exclude_mask=mask.cuda(), row_offset=1_000_000, path=ops.PATH_GEMV)
    want = [int(x) for x in ri[0].tolist() if x not in set(banned.tolist())][:10]
    assert (i[0].cpu() - 1_000_000).tolist() == want


def test_merge_of_fake_shards_equals_global_topk():
    items, _ = oracle.synth_clustered(20000, 384, seed=9)
    queries, _ = oracle.synth_queries_from_items(items, 33, seed=10)
    k, G = 100, 8
    rv, ri = oracle.cos_topk(queries, items, k)
    cs, ci = [], []
    from instacart_next_order_recommendation_b200.sharded import shard_bounds

    for r in range(G):
        lo, hi = shard_bounds(20000, G, r)
        v, i = ops.cos_topk(queries.cuda(), items[lo:hi].cuda(), k, row_offset=lo)
        cs.append(v)
        ci.append(i)
    v, i = ops.topk_merge(torch.stack(cs), torch.stack(ci), k)
    _check_topk(v, i, rv, ri, F32_RTOL)
    # empty slots (-inf, -1) from short shards are ignored
    cs[3][:, 50:] = float("-inf")
    ci[3][:, 50:] = -1
    v2, i2 = ops.topk_merge(torch.stack(cs), torch.stack(ci), k)
    assert (i2 >= 0).all()


def test_recommender_dropin_matches_reference_golden(golden_dir, tmp_path):
    z = np.load(golden_dir / "embeddings_small.npz")
    gold = json.loads((golden_dir / "recommend_golden.json").read_text())
    pids = [str(p) for p in z["product_ids"]]

    class Enc:
        def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True, **kw):
            tab = {"c": z["items"], "q": z["queries"]}
            return np.stack([tab[t.split(":")[0]][int(t.split(":")[1])] for t in texts]).astype(np.float32)

    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text(json.dumps({pid: f"c:{i}" for i, pid in enumerate(pids)}))
    for dtype, tol in ((torch.float32, 1e-5),):
        rec = icr.MonitoredRecommender("fake-model", corpus, model=Enc(), catalog_dtype=dtype)
        assert (corpus.parent / ".embedding_index").exists()
        for case in gold["cases"]:
            got = rec.recommend(f"q:{case['q']}", top_k=case["top_k"], exclude_product_ids=set(case["exclude"]))
            assert [p for p, _ in got] == [p for p, _ in case["result"]], case
            np.testing.assert_allclose([s for _, s in got], [s for _, s in case["result"]], rtol=tol)
        m = rec.last_metrics
        assert m.num_recommendations == len(got) and m.user_id == "anonymous" and m.similarity_compute_time_ms > 0
        # very long exclusion list -> device-side mask path, same semantics as the reference walk
        excl = set(pids[::2])
        got = rec.recommend("q:1", top_k=10, exclude_product_ids=excl)
        want = oracle.recommend_tail(z["queries"][1], z["items"], pids, 10, excl)
        assert [p for p, _ in got] == [p for p, _ in want]
    # second construction hits the on-disk index written by the first
    rec2 = icr.Recommender("fake-model", corpus, model=Enc())
    np.testing.assert_array_equal(rec2.product_embeddings, z["items"])

    # an encoder that honours convert_to_tensor hands the query over on the device (SURVEY §8f row 1): same answers
    class DeviceEnc(Enc):
        calls = 0

        def encode(self, texts, convert_to_tensor=False, **kw):
            out = Enc.encode(self, texts, **kw)
            if convert_to_tensor:
                DeviceEnc.calls += 1
                return torch.from_numpy(out).cuda()
            return out

    class StrictEnc:  # the reference's exact call only: any other keyword is a TypeError
        def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True):
            return Enc().encode(texts)

    rec3 = icr.Recommender("fake-model", corpus, model=DeviceEnc())
    rec4 = icr.Recommender("fake-model", corpus, model=StrictEnc())
    for case in gold["cases"][:20]:
        args = dict(top_k=case["top_k"], exclude_product_ids=set(case["exclude"]))
        want = rec2.recommend(f"q:{case['q']}", **args)
        assert rec3.recommend(f"q:{case['q']}", **args) == want
        assert rec4.recommend(f"q:{case['q']}", **args) == want
    assert DeviceEnc.calls >= 20 and rec4._query_on_device is False


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_resident_workspace_skips_the_counter_reset_safely(dtype):
    """ICR_PATH_WS_RESIDENT: a workspace zero-filled once and reused call after call gives the same answers as a fresh
    workspace per call (the merging CTA of K1 leaves its counter at zero), for changing queries and batch sizes 1-7."""
    items = oracle.synth_unnormalised(30000, 384, seed=1).to(dtype).cuda()
    lib = ops._lib.load()
    for Q in (1, 3, 7):
        need = lib.icr_cos_topk_workspace_bytes(Q, 30000, 384, ops._dtype_code(items), 10, ops.PATH_GEMV, 0)
        ws = torch.zeros(need, dtype=torch.uint8, device="cuda")
        for rep in range(4):
            q = oracle.synth_unnormalised(Q, 384, seed=50 + rep).to(dtype).cuda()
            v0, i0 = ops.cos_topk(q, items, 10, path=ops.PATH_GEMV)
            v1, i1 = ops.cos_topk(q, items, 10, path=ops.PATH_GEMV, workspace=ws)
            assert torch.equal(v0, v1) and torch.equal(i0, i1)
    with pytest.raises(ValueError):
        ops.cos_topk(q, items, 10, path=ops.PATH_GEMV, workspace=torch.zeros(16, dtype=torch.uint8, device="cuda"))


def test_import_swap_with_cached_host_catalog(monkeypatch):
    """INTEGRATION.md §1: cos_sim(query_emb, product_embeddings) with the reference's numpy catalog; with
    ICR_CACHE_HOST_OPERANDS=1 the device copy is reused between requests and refreshed when the array changes."""
    from instacart_next_order_recommendation_b200 import similarity

    monkeypatch.setenv("ICR_CACHE_HOST_OPERANDS", "1")
    similarity._HOST_CACHE.clear()
    items = oracle.synth_clustered(4000, 384, seed=5)[0].numpy()  # 6 MB: above the caching threshold
    q = oracle.synth_isotropic(1, 384, seed=6).numpy()[0]
    s1 = icr.cos_sim(q, items)
    assert len(similarity._HOST_CACHE) == 1
    dev_copy = next(iter(similarity._HOST_CACHE.values()))[1]
    s2 = icr.cos_sim(q, items)
    assert next(iter(similarity._HOST_CACHE.values()))[1] is dev_copy and torch.equal(s1, s2)
    ref = oracle.cos_sim(q, items)
    assert (s1.cpu() - ref).abs().max() < 1e-6
    order = s1[0].argsort(descending=True)  # the reference's next line (serve_recommendations.py:215)
    assert int(order[0]) == int(ref[0].argmax())
    items[:] = np.roll(items, 1, axis=0)  # rewritten in place: the sample check notices and uploads again
    s3 = icr.cos_sim(q, items)
    assert (s3.cpu() - oracle.cos_sim(q, items)).abs().max() < 1e-6
    similarity._HOST_CACHE.clear()


def test_ir_evaluator_and_rank_all_against_oracle(golden_dir):
    z = np.load(golden_dir / "embeddings_small.npz")
    gold = json.loads((golden_dir / "metrics_golden.json").read_text())
    pids = [str(p) for p in z["product_ids"]]
    qids = list(gold["rank_all_top100"].keys())
    got = icr.rank_all(z["queries"], z["items"], qids, pids, limit=100)
    assert got == gold["rank_all_top100"]  # the reference's own ContentBasedBaseline.rank_all output
    rel = {k: set(v) for k, v in gold["relevant"].items()}
    m = icr.compute_ir_metrics(got, rel)
    for key, val in gold["metrics"].items():
        assert m[key] == pytest.approx(val, abs=1e-12)

    class Enc:
        def encode(self, texts, **kw):
            tab = {"c": z["items"], "q": z["queries"]}
            return np.stack([tab[t.split(":")[0]][int(t.split(":")[1])] for t in texts]).astype(np.float32)

    queries = {qid: f"q:{i}" for i, qid in enumerate(qids)}
    corpus = {pid: f"c:{i}" for i, pid in enumerate(pids)}
    ev = icr.InformationRetrievalEvaluator(queries, corpus, rel, name="order-recommendation")
    out = ev(Enc())
    assert ev.primary_metric in out and 0.0 <= out[ev.primary_metric] <= 1.0
    # same numbers from the oracle's chunked-topk + heap restatement of the upstream evaluator core
    keep = [i for i, q in enumerate(qids) if rel.get(q)]
    lists = oracle.ir_eval_topk(z["queries"][keep], z["items"], max_k=100)
    ids = np.array([[ci for _, ci in l] for l in lists])
    want = ev.compute_metrics_from_ids(ids)
    for k, val in want.items():
        assert out[f"order-recommendation_cosine_{k}"] == pytest.approx(val, abs=1e-12)


def _index_on_disk(tmp_path, n, d, seed=3):
    from instacart_next_order_recommendation_b200.index import EmbeddingIndex

    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text("{}")
    ids = [str(i) for i in range(n)]
    emb = oracle.synth_unnormalised(n, d, seed=seed).numpy()
    idx = EmbeddingIndex(corpus, "fake-model")
    idx.save(ids, emb)
    return idx, ids, emb


@pytest.mark.parametrize("chunk_rows", [1 << 17, 1000, 37])
def test_catalog_streamed_from_index_equals_catalog_from_memory(tmp_path, chunk_rows):
    """DeviceCatalog.from_index (memmap -> pinned staging -> HBM, icr_convert_rows) holds bit-identical rows."""
    idx, ids, emb = _index_on_disk(tmp_path, 5003, 384)
    t = torch.from_numpy(emb)
    cat = icr.DeviceCatalog.from_index(idx, ids, chunk_rows=chunk_rows)
    assert torch.equal(cat.rows.cpu(), t) and cat.row_offset == 0
    bf = icr.DeviceCatalog.from_index(idx, ids, dtype=torch.bfloat16, chunk_rows=chunk_rows)
    assert torch.equal(bf.rows.cpu(), t.to(torch.bfloat16))
    # a row block of a sharded catalog: global ids through row_offset
    part = icr.DeviceCatalog.from_index(idx, ids, rows=(1200, 3100), chunk_rows=chunk_rows)
    assert torch.equal(part.rows.cpu(), t[1200:3100]) and part.row_offset == 1200
    # pre-normalised upload: rows are x / max(|x|, eps) (one rounding apart from torch's at most)
    nrm = icr.DeviceCatalog.from_index(idx, ids, normalize=True, chunk_rows=chunk_rows)
    ref = torch.nn.functional.normalize(t, dim=1)
    assert (nrm.rows.cpu() - ref).abs().max() <= 2e-7
    # the bf16 sidecar is uploaded as is and gives the same resident bytes as converting on the device
    idx.save_bf16_sidecar()
    side = icr.DeviceCatalog.from_index(idx, ids, dtype=torch.bfloat16, chunk_rows=chunk_rows)
    assert torch.equal(side.rows.cpu(), t.to(torch.bfloat16))
    # stale index -> None, like EmbeddingIndex.load
    assert icr.DeviceCatalog.from_index(idx, ids[:-1]) is None
    # and the streamed catalog answers like the in-memory one
    queries = oracle.synth_unnormalised(9, 384, seed=11)
    v, i = cat.topk(queries.cuda(), 100)
    rv, ri = oracle.cos_topk(queries, t, 100)
    _check_topk(v, i, rv, ri, F32_RTOL)
    # an embedding dim that is not a multiple of 4 (no 16-byte vectors): still loads, fp32 and bf16
    (tmp_path / "odd").mkdir()
    idx2, ids2, emb2 = _index_on_disk(tmp_path / "odd", 777, 50)
    for dt in (torch.float32, torch.bfloat16):
        c2 = icr.DeviceCatalog.from_index(idx2, ids2, dtype=dt, chunk_rows=chunk_rows)
        q2 = oracle.synth_unnormalised(3, 50, seed=12)
        v, i = c2.topk(q2.cuda().to(dt), 20)
        rv, ri = oracle.cos_topk(q2.to(dt).float(), torch.from_numpy(emb2).to(dt).float(), 20)
        _check_topk(v, i, rv, ri, F32_RTOL if dt == torch.float32 else BF16_RTOL)
    sh = icr.ShardedCatalog.from_index(idx, ids, dtype=torch.bfloat16)
    v, i = sh.topk(queries.cuda().to(torch.bfloat16), 50)
    rv, ri = oracle.cos_topk(queries.to(torch.bfloat16).float(), t.to(torch.bfloat16).float(), 50)
    _check_topk(v, i, rv, ri, BF16_RTOL)


def _random_rankings(rng, Q, K, n_corpus, short_rows=True):
    ids = np.stack([rng.permutation(n_corpus)[:K] for _ in range(Q)]).astype(np.int64)
    relevant = [set(int(x) for x in rng.choice(n_corpus, size=rng.integers(1, 15), replace=False)) for _ in range(Q)]
    for q in range(0, Q, 3):  # plant hits near the top so that every metric is exercised
        ids[q, rng.integers(0, min(10, K))] = next(iter(relevant[q]))
    if short_rows:
        for q in range(1, Q, 7):  # rows with fewer than K results end in -1
            ids[q, rng.integers(0, K):] = -1
    # |relevant| may count documents that are not in the catalog
    n_rel = [len(r) + (int(rng.integers(0, 3)) if q % 5 == 0 else 0) for q, r in enumerate(relevant)]
    return ids, relevant, n_rel


@pytest.mark.parametrize("Q,K,n_corpus", [(257, 100, 500), (40, 37, 300), (1, 10, 50), (1000, 256, 5000), (9, 1, 20)])
def test_ir_metric_kernel_vs_oracle_loops(Q, K, n_corpus):
    """icr_ir_metrics == the evaluator's per-query loops (oracle.st_ir_metrics), per query and in the mean."""
    rng = np.random.default_rng(Q * 1000 + K)
    ids, relevant, n_rel = _random_rankings(rng, Q, K, n_corpus)
    specs = ([(ops.METRIC_ACCURACY, k) for k in (1, 3, 5, 10)] + [(ops.METRIC_PRECISION, k) for k in (1, 3, 5, 10)]
             + [(ops.METRIC_RECALL, k) for k in (1, 3, 5, 10)] + [(ops.METRIC_MRR, 10), (ops.METRIC_NDCG, 10), (ops.METRIC_MAP, 100)])
    table = ops.RelevanceTable([sorted(r) for r in relevant], n_rel, device="cuda")
    means, per_query = ops.ir_metrics(torch.from_numpy(ids).cuda(), table, specs)
    want_means, want_pq = oracle.st_ir_metrics([list(r) for r in ids], relevant, n_rel, per_query=True)
    np.testing.assert_allclose(per_query.cpu().numpy(), want_pq, rtol=0, atol=1e-12)
    np.testing.assert_allclose(means.cpu().numpy(), np.array(list(want_means.values())), rtol=0, atol=1e-12)


def test_ir_metric_kernel_baseline_flavour_vs_reference_metrics(golden_dir):
    """The *_RETRIEVED kinds equal src/baselines/metrics.py (pinned by the reference's own outputs in metrics_golden.json)."""
    from instacart_next_order_recommendation_b200 import evaluation

    gold = json.loads((golden_dir / "metrics_golden.json").read_text())
    cases = [(gold["rank_all_top100"], gold["relevant"], gold["metrics"])] + [(c["rankings"], c["relevant"], c["metrics"]) for c in gold["extra"]]
    specs = [(kind, k) for _, kind, k in evaluation.BASELINE_METRICS]
    for rankings, relevant, want in cases:
        qids = [q for q in rankings if relevant.get(q)]
        if not qids:
            continue
        pids = sorted({p for q in qids for p in rankings[q]} | {p for q in qids for p in relevant[q]})
        row_of = {p: i for i, p in enumerate(pids)}
        K = max(1, min(100, max(len(rankings[q]) for q in qids)))
        ids = np.full((len(qids), K), -1, dtype=np.int64)
        for r, q in enumerate(qids):
            top = rankings[q][:K]
            ids[r, : len(top)] = [row_of[p] for p in top]
        table = ops.RelevanceTable([[row_of[p] for p in relevant[q]] for q in qids], [len(set(relevant[q])) for q in qids], device="cuda")
        means, _ = ops.ir_metrics(torch.from_numpy(ids).cuda(), table, specs)
        for (name, _, _), v in zip(evaluation.BASELINE_METRICS, means.tolist()):
            assert v == pytest.approx(want[name], abs=1e-12), name
    # and the fused consumer: embeddings in, the reference's metric dict out
    z = np.load(golden_dir / "embeddings_small.npz")
    pids = [str(p) for p in z["product_ids"]]
    qids = list(gold["rank_all_top100"].keys())
    m = evaluation.evaluate_rankings(z["queries"], z["items"], qids, pids, {k: set(v) for k, v in gold["relevant"].items()})
    for key, val in gold["metrics"].items():
        assert m[key] == pytest.approx(val, abs=1e-12), key


def test_ir_metric_kernel_argument_errors():
    table = ops.RelevanceTable([[1, 2]], device="cuda")
    ids = torch.zeros(1, 10, dtype=torch.int64, device="cuda")
    with pytest.raises(ValueError):
        ops.ir_metrics(ids, table, [(99, 10)])
    with pytest.raises(ValueError):
        ops.ir_metrics(ids, table, [(ops.METRIC_MRR, 0)])
    with pytest.raises(ValueError):
        ops.ir_metrics(torch.zeros(2, 10, dtype=torch.int64, device="cuda"), table, [(ops.METRIC_MRR, 10)])
    with pytest.raises(RuntimeError):
        ops.ir_metrics(ids.cpu(), table, [(ops.METRIC_MRR, 10)])


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,D,scale", [(256, 384, 20.0), (64, 384, 30.0), (37, 768, 20.0), (8, 64, 20.0), (1024, 384, 20.0),
                                       (130, 384, 20.0), (288, 384, 20.0), (384, 384, 20.0), (512, 384, 30.0), (1000, 128, 30.0), (300, 768, 20.0), (2048, 384, 20.0), (4096, 64, 20.0)])
def test_mnrl_forward_backward_vs_autograd(dtype, B, D, scale):
    g = torch.Generator().manual_seed(2024)
    items, _ = oracle.synth_clustered(B, D, seed=2024, n_centres=12)
    a = torch.nn.functional.normalize(items + 0.3 * torch.randn(B, D, generator=g), dim=1)
    p = items * (1.0 + 0.5 * torch.rand(B, 1, generator=g))  # un-normalised positives exercise the Jacobian
    a, p = a.to(dtype), p.to(dtype)
    ad = a.cuda().requires_grad_(True)
    pd = p.cuda().requires_grad_(True)
    loss = icr.mnrl_loss(ad, pd, scale)
    (loss * 1.7).backward()
    rl, rga, rgp = oracle.mnrl_loss_and_grads(a.float(), p.float(), scale)
    assert loss.dtype == torch.float32
    assert abs(loss.item() - rl.item()) <= MNRL_ATOL
    # bf16 gradients are rounded when the step's one library call writes them (for dL/dloss = 1) and again after the scaling by the incoming gradient
    tol = MNRL_ATOL if dtype == torch.float32 else MNRL_ATOL + 2 ** -7 * rga.abs().max().item() * 1.7
    assert (ad.grad.float().cpu() - 1.7 * rga).abs().max() <= tol
    assert (pd.grad.float().cpu() - 1.7 * rgp).abs().max() <= tol
    # gradients shrink like 1/B, so the absolute bound alone says little for large batches: also bound the error
    # relative to the largest gradient entry (fp16 operands of the gradient products: 2^-11 per element)
    rel = 2e-3 if dtype == torch.float32 else 2e-3 + 2 ** -7
    assert (ad.grad.float().cpu() - 1.7 * rga).abs().max() <= rel * 1.7 * rga.abs().max()
    assert (pd.grad.float().cpu() - 1.7 * rgp).abs().max() <= rel * 1.7 * rgp.abs().max()


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16])
@pytest.mark.parametrize("B,D", [(256, 384), (64, 768), (512, 384)])
def test_mnrl_step_graph_equals_the_autograd_path(dtype, B, D):
    """MnrlStepGraph replays loss + both gradients of a fixed-shape step as one CUDA graph: same numbers as mnrl_loss().backward(),
    on fresh inputs at every replay, and usable inside an autograd graph through backward_into()."""
    g = torch.Generator().manual_seed(5)
    step = icr.mnrl_step_graph(B, D, dtype, 20.0)
    for it in range(3):
        a = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1).to(dtype).cuda()
        p = (a.float().cpu() + 0.4 * torch.randn(B, D, generator=g)).to(dtype).cuda()
        loss, ga, gp = step(a, p)
        ar, pr = a.clone().requires_grad_(True), p.clone().requires_grad_(True)
        ref = icr.mnrl_loss(ar, pr, 20.0)
        ref.backward()
        assert abs(loss.item() - ref.item()) <= 1e-6
        assert torch.equal(ga, ar.grad) and torch.equal(gp, pr.grad)
    w = torch.nn.Parameter(torch.eye(D, device="cuda"))
    a32, p32 = a.float(), p.float()
    loss = step.backward_into((a32 @ w).to(dtype), (p32 @ w).to(dtype))
    assert torch.isfinite(loss) and w.grad is not None and torch.isfinite(w.grad).all() and w.grad.abs().max() > 0
    with pytest.raises(ValueError):
        step(a[:-1], p[:-1])


def test_shard_merge_tolerates_duplicated_candidates():
    """Replicated shards hand the merge identical (score, id) pairs: the selection must terminate and return k entries in
    (score desc, id asc) order (round-1 advice: >128 identical keys in the boundary bin never terminated)."""
    g = torch.Generator().manual_seed(9)
    Q, k = 37, 100
    base_v = torch.sort(torch.rand(Q, k, generator=g), dim=1, descending=True).values
    base_i = torch.stack([torch.randperm(5000, generator=g)[:k] for _ in range(Q)])
    G = 4
    vals = base_v[None].repeat(G, 1, 1).cuda()
    ids = base_i[None].repeat(G, 1, 1).cuda()
    v, i = ops.topk_merge(vals, ids, k)
    torch.cuda.synchronize()
    assert (v[:, :-1] >= v[:, 1:]).all()
    # the k best of G copies of a k-list: its best ceil(k / G) entries, each G times
    top = base_v[:, : (k + G - 1) // G]
    assert torch.allclose(v.cpu()[:, ::G][:, : top.shape[1]], top)
    same = torch.full((1, 1, 300), 0.5).repeat(1, 3, 1).cuda()
    same_ids = torch.full((1, 3, 300), 7, dtype=torch.int64).cuda()
    v2, i2 = ops.topk_merge(same, same_ids, 100)
    torch.cuda.synchronize()
    assert (v2 == 0.5).all() and (i2 == 7).all()


@pytest.mark.parametrize("B,D,scale", [(256, 384, 20.0), (64, 384, 30.0), (37, 768, 20.0), (512, 384, 30.0), (300, 768, 20.0), (2048, 384, 20.0)])
def test_mnrl_fp16_inputs_are_read_natively(B, D, scale, monkeypatch):
    """The reference trains with fp16=use_fp16 on CUDA (src/training/train_sbert.py:210,232): under autocast the embeddings
    reach the loss as float16. Both kernel families take them as they are (no eager .float() round trip) and return float16
    gradients; the oracle is fp32 math on the fp16-rounded inputs."""
    g = torch.Generator().manual_seed(77)
    items, _ = oracle.synth_clustered(B, D, seed=77, n_centres=12)
    a = torch.nn.functional.normalize(items + 0.3 * torch.randn(B, D, generator=g), dim=1).half()
    p = (items * (1.0 + 0.5 * torch.rand(B, 1, generator=g))).half()
    ad = a.cuda().requires_grad_(True)
    pd = p.cuda().requires_grad_(True)
    called = []
    real = torch.Tensor.float
    monkeypatch.setattr(torch.Tensor, "float", lambda self, *a_, **k_: (called.append(self.dtype), real(self, *a_, **k_))[1])
    loss = icr.mnrl_loss(ad, pd, scale)
    loss.backward()
    monkeypatch.undo()
    assert torch.float16 not in called, "fp16 embeddings were up-cast eagerly"
    assert ad.grad.dtype == torch.float16 and pd.grad.dtype == torch.float16 and loss.dtype == torch.float32
    rl, rga, rgp = oracle.mnrl_loss_and_grads(a.float(), p.float(), scale)
    assert abs(loss.item() - rl.item()) <= MNRL_ATOL
    tol = MNRL_ATOL + 2 ** -10 * rga.abs().max().item()  # fp16 rounding of the stored gradients
    assert (ad.grad.float().cpu() - rga).abs().max() <= tol
    assert (pd.grad.float().cpu() - rgp).abs().max() <= MNRL_ATOL + 2 ** -10 * rgp.abs().max().item()
    # the module form under autocast, as the trainer calls it
    class Enc(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.w = torch.nn.Linear(D, D, bias=False)

        def forward(self, f):
            return {"sentence_embedding": self.w(f["x"])}

    enc = Enc().cuda()
    mod = icr.MultipleNegativesRankingLoss(enc, scale=scale)
    with torch.autocast("cuda", dtype=torch.float16):
        la = mod([{"x": a.cuda().float()}, {"x": p.cuda().float()}])
    la.backward()
    assert torch.isfinite(la) and enc.w.weight.grad is not None and torch.isfinite(enc.w.weight.grad).all()
    with torch.autocast("cuda", dtype=torch.float16):
        ea, ep = enc.w(a.cuda().float()), enc.w(p.cuda().float())
    assert ea.dtype == torch.float16
    rl2, _, _ = oracle.mnrl_loss_and_grads(ea.detach().float().cpu(), ep.detach().float().cpu(), scale)
    assert abs(la.item() - rl2.item()) <= MNRL_ATOL


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,Bc,off,D,scale", [(64, 512, 128, 384, 20.0), (256, 2048, 1792, 384, 20.0), (48, 96, 48, 128, 30.0),
                                              (100, 800, 300, 768, 20.0), (8, 16, 0, 64, 20.0), (300, 300, 0, 384, 20.0)])
def test_mnrl_rectangular_gathered_candidates_vs_autograd(dtype, B, Bc, off, D, scale):
    """Cross-device negatives: B anchors against Bc gathered candidates, label i + off (icr_mnrl_fwd_rect / bwd_rect)."""
    g = torch.Generator().manual_seed(B + Bc)
    cand, _ = oracle.synth_clustered(Bc, D, seed=2025, n_centres=16)
    cand = cand * (1.0 + 0.5 * torch.rand(Bc, 1, generator=g))
    a = torch.nn.functional.normalize(cand[off : off + B] + 0.3 * torch.randn(B, D, generator=g), dim=1)
    a, cand = a.to(dtype), cand.to(dtype)
    ad, cd = a.cuda(), cand.cuda()
    loss, saved = ops.mnrl_forward_rect(ad, cd, scale, off)
    go = torch.tensor(1.3, device="cuda")
    ga, gc = ops.mnrl_backward_rect(ad, cd, scale, off, saved, go)
    rl, rga, rgc = oracle.mnrl_rect_loss_and_grads(a.float(), cand.float(), scale, off)
    assert abs(loss.item() - rl.item()) <= MNRL_ATOL
    out_round = 0.0 if dtype == torch.float32 else 2 ** -8
    for got, want in ((ga, rga), (gc, rgc)):
        err = (got.float().cpu() - 1.3 * want).abs().max().item()
        # the gradient products run on fp16 operands (softmax - I and x^, 2^-11 relative each): absolute error
        # <= ~2^-10 * scale * grad_out * max|x^| / B, i.e. below 1e-4 from B ~ 32 up; a tiny rectangular batch
        # (the square form takes the fp32 CUDA-core kernels there) is held to that bound instead
        atol = MNRL_ATOL if B >= 32 else max(MNRL_ATOL, 2 ** -10 * scale * 1.3 * 0.5 / B)
        assert err <= atol + out_round * 1.3 * want.abs().max().item()
        assert err <= ((2e-3 if Bc >= 64 else 8e-3) + out_round) * 1.3 * want.abs().max().item()  # fp16 operands, few terms to average over
    with pytest.raises(ValueError):
        ops.mnrl_forward_rect(ad, cd, scale, Bc - B + 1)  # the positives would fall off the end of the candidates


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B", [48, 256, 640])
def test_mnrl_one_call_step_equals_separate_forward_and_backward(dtype, B):
    """icr_mnrl_fwd_bwd (what a training step uses) == icr_mnrl_fwd followed by icr_mnrl_bwd with the same dL/dloss,
    on both kernel families; a loss computed without gradients takes the forward-only entry point."""
    g = torch.Generator().manual_seed(B)
    a = torch.randn(B, 384, generator=g).to(dtype).cuda()
    p = (torch.randn(B, 384, generator=g) * 2).to(dtype).cuda()
    loss1, grads1 = ops.mnrl_forward_backward(a, p, 20.0)
    ga1, gp1 = grads1[0], grads1[1]
    assert torch.equal(ops.mnrl_scale_grads(grads1, torch.tensor(0.5, device="cuda")).float(), (grads1.float() * 0.5).to(dtype).float())
    loss0, saved = ops.mnrl_forward(a, p, 20.0)
    go = torch.tensor(1.0, device="cuda")
    ga0, gp0 = ops.mnrl_backward(a, p, 20.0, saved, go)
    assert abs(loss1.item() - loss0.item()) <= 1e-6
    tol = 1e-7 if dtype == torch.float32 else 2 ** -8 * ga0.float().abs().max().item()
    assert (ga1.float() - ga0.float()).abs().max().item() <= tol and (gp1.float() - gp0.float()).abs().max().item() <= tol
    with torch.no_grad():
        assert abs(icr.mnrl_loss(a, p, 20.0).item() - loss0.item()) <= 1e-6
    ar = a.clone().requires_grad_(True)
    (icr.mnrl_loss(ar, p, 20.0) * 0.25).backward()  # only one side needs a gradient, scaled dL/dloss
    assert (ar.grad.float() - 0.25 * ga0.float()).abs().max().item() <= tol + 1e-7


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_mnrl_tensor_path_equals_cuda_core_path(dtype, monkeypatch):
    """The two MNRL kernel families (mnrl.cu / mnrl_tc.cu) agree on the same batch (subprocess: the switch is read once)."""
    import subprocess
    import sys

    code = (
        "import sys, torch; sys.path.insert(0, '.');"
        "import instacart_next_order_recommendation_b200 as icr;"
        f"dt = torch.{str(dtype).split('.')[-1]};"
        "g = torch.Generator().manual_seed(7);"
        "a = torch.randn(192, 384, generator=g).to(dt).cuda().requires_grad_(True);"
        "p = (torch.randn(192, 384, generator=g) * 3).to(dt).cuda().requires_grad_(True);"
        "l = icr.mnrl_loss(a, p, 20.0); l.backward();"
        "torch.save((l.detach().cpu(), a.grad.float().cpu(), p.grad.float().cpu()), sys.argv[1])"
    )
    import os
    import tempfile

    outs = {}
    for path in ("tc", "simt"):
        with tempfile.NamedTemporaryFile(suffix=".pt") as f:
            env = dict(os.environ, ICR_MNRL_PATH=path)
            subprocess.run([sys.executable, "-c", code, f.name], check=True, env=env, cwd=str(__import__("pathlib").Path(__file__).resolve().parents[1]))
            outs[path] = torch.load(f.name)
    (l1, ga1, gp1), (l2, ga2, gp2) = outs["tc"], outs["simt"]
    assert abs(l1.item() - l2.item()) <= 2e-5
    tol = 2e-3 if dtype == torch.float32 else 2e-3 + 2 ** -7
    assert (ga1 - ga2).abs().max() <= tol * ga2.abs().max()
    assert (gp1 - gp2).abs().max() <= tol * gp2.abs().max()


def test_mnrl_known_answers_and_module_interface():
    B, d, scale = 16, 64, 20.0
    q, _ = torch.linalg.qr(torch.randn(d, d, generator=torch.Generator().manual_seed(0)))
    a = q[:B].contiguous().cuda()
    assert icr.mnrl_loss(a, a.clone(), scale).item() == pytest.approx(math.log(1 + (B - 1) * math.exp(-scale)), abs=1e-6)
    same = torch.ones(B, d, device="cuda")
    assert icr.mnrl_loss(same, same, scale).item() == pytest.approx(math.log(B), abs=1e-5)

    class Tower(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = torch.nn.Linear(32, 64)

        def forward(self, feats):
            return {"sentence_embedding": self.lin(feats["x"])}

    tower = Tower().cuda()
    loss_mod = icr.MultipleNegativesRankingLoss(tower, scale=30.0)
    xa, xp = torch.randn(24, 32, device="cuda"), torch.randn(24, 32, device="cuda")
    loss = loss_mod([{"x": xa}, {"x": xp}], labels=None)
    loss.backward()
    ref = oracle.mnrl_loss(tower.lin(xa).detach().cpu(), tower.lin(xp).detach().cpu(), 30.0)
    assert abs(loss.item() - ref.item()) < 1e-4 and tower.lin.weight.grad is not None


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("Q,k", [(1, 10), (1, 100), (2, 32), (5, 200), (7, 10)])
def test_gemv_row_strided_catalog_and_in_kernel_merge(dtype, Q, k):
    """Row-strided catalogs take the direct-load GEMV kernel, contiguous ones the bulk-copy ring kernel; both end
    with the in-kernel merge (rank counting for <=1024 candidates, streaming fallback beyond)."""
    N, D = 30011, 384
    items, _ = oracle.synth_clustered(N, D, seed=41)
    queries, _ = oracle.synth_queries_from_items(items, Q, seed=42)
    wide = torch.zeros(N, D + 16, dtype=dtype, device="cuda")
    wide[:, :D] = items.to(dtype).cuda()
    strided = wide[:, :D]
    assert strided.stride(0) == D + 16
    rv, ri = oracle.cos_topk(queries.to(dtype).float(), items.to(dtype).float(), k)
    tol = F32_RTOL if dtype == torch.float32 else BF16_RTOL
    for cat in (strided, strided.contiguous()):
        v, i = ops.cos_topk(queries.to(dtype).cuda(), cat, k, path=ops.PATH_GEMV)
        _check_topk(v, i, rv, ri, tol)
    # many equal scores (k > 32 with heavy ties): exercises the merge's overflow fallback
    dup = items[torch.arange(N) % 50].to(dtype).cuda()
    v, i = ops.cos_topk(queries[:1].to(dtype).cuda(), dup, 256, path=ops.PATH_GEMV)
    rv, ri = oracle.cos_topk(queries[:1].to(dtype).float(), dup.float().cpu(), 256)
    err, _ = oracle.compare_topk(v.cpu(), i.cpu(), rv, ri, rtol=tol)
    assert err <= tol and len(set(i[0].tolist())) == 256


def test_topk_small_cuda_graph_equals_plain_call():
    items, _ = oracle.synth_clustered(20000, 384, seed=31)
    queries, _ = oracle.synth_queries_from_items(items, 6, seed=32)
    for dtype in (torch.float32, torch.bfloat16):
        cat = icr.DeviceCatalog(items, dtype=dtype)
        for qn in (1, 3):
            for rep in range(3):  # replays of the same captured graph with different queries
                q = queries[rep : rep + qn]
                v, i = cat.topk(q.cuda(), 16)
                vs, is_ = cat.topk_small(q.numpy(), 16)  # host numpy in, like SentenceTransformer.encode
                assert torch.equal(vs, v) and torch.equal(is_, i)
        assert len(cat._graphs) == 2
    # a captured call that contains a select launch: 8 queries against 300,000 rows leave too many survivors for the in-kernel
    # select, so prep + GEMM + select are all in the graph
    big, _ = oracle.synth_clustered(300_000, 128, seed=33)
    q8, _ = oracle.synth_queries_from_items(big, 8, seed=34)
    cat = icr.DeviceCatalog(big, dtype=torch.bfloat16)
    for rep in range(3):
        q = torch.roll(q8, rep, 0)
        v, i = cat.topk(q.cuda(), 100)
        vs, is_ = cat.topk_small(q.numpy(), 100)
        assert torch.equal(vs, v) and torch.equal(is_, i)
    rv, ri = oracle.cos_topk(q.to(torch.bfloat16).float(), cat.rows.float().cpu(), 100)
    _check_topk(vs, is_, rv, ri, 5e-5)


def test_topk_small_device_query_takes_the_prepared_call_and_matches_the_oracle():
    """A device-resident query in the catalog's layout is scored where it lies (no graph, no copy): one launch through the
    prepared argument list; repeated requests re-use the resident workspace (ticket and slab counters left at zero)."""
    items, _ = oracle.synth_clustered(49_688, 384, seed=41)
    queries, _ = oracle.synth_queries_from_items(items, 12, seed=42)
    for dtype, tol in ((torch.float32, F32_RTOL), (torch.bfloat16, BF16_RTOL)):
        cat = icr.DeviceCatalog(items, dtype=dtype)
        ref_items = cat.rows.float().cpu()
        for qn, k in ((1, 10), (1, 16), (1, 100), (2, 10), (7, 16), (1, 32), (1, 24), (1, 14), (1, 33)):  # k <= 16: the one-trip merge; above: heads + walk
            for rep in range(3):
                q = queries[rep : rep + qn].to(dtype).cuda()
                v, i = cat.topk_small(q, k)
                if dtype == torch.float32 or qn <= 3:  # GEMV path: the whole request is one kernel
                    assert ops.last_launch_count() == 1
                rv, ri = oracle.cos_topk(q.float().cpu(), ref_items, k)
                _check_topk(v, i, rv, ri, tol)
        assert len(cat._plans) == 9 and not getattr(cat, "_graphs", {})
        # a query in another dtype or on the host still goes through the graph path
        v, i = cat.topk_small(queries[:1].numpy(), 10)
        rv, ri = oracle.cos_topk(queries[:1].to(dtype).float(), ref_items, 10)
        _check_topk(v, i, rv, ri, tol)
        assert len(cat._graphs) == 1


def test_topk_request_writes_pinned_host_results():
    """Query on the device, result on the host: the kernel's last CTA stores into pinned host memory (no device-to-host copy)."""
    items, _ = oracle.synth_clustered(49_688, 384, seed=51)
    queries, _ = oracle.synth_queries_from_items(items, 8, seed=52)
    for dtype, tol in ((torch.float32, F32_RTOL), (torch.bfloat16, BF16_RTOL)):
        cat = icr.DeviceCatalog(items, dtype=dtype)
        for qn, k in ((1, 16), (1, 10), (1, 128), (3, 32), (7, 16)):
            for rep in range(2):
                q = queries[rep : rep + qn].to(dtype).cuda()
                vals, ids = cat.topk_request(q, k)
                assert isinstance(vals, list) and len(vals) == qn and len(vals[0]) == k
                dv, di = cat.topk(q, k)
                assert torch.equal(torch.tensor(vals), dv.cpu()) and torch.equal(torch.tensor(ids), di.cpu())
        rv, ri = oracle.cos_topk(q.float().cpu(), cat.rows.float().cpu(), k)
        _check_topk(torch.tensor(vals), torch.tensor(ids), rv, ri, tol)
        # host queries and 1-D queries fall back to the graph path, same results
        vals, ids = cat.topk_request(queries[0].to(dtype).cuda(), 10)
        dv, di = cat.topk(queries[:1].to(dtype).cuda(), 10)
        assert torch.equal(torch.tensor(vals), dv.cpu()) and torch.equal(torch.tensor(ids), di.cpu())


def test_topk_host_pipeline_equals_device_path():
    items, _ = oracle.synth_clustered(30000, 384, seed=21)
    queries, _ = oracle.synth_queries_from_items(items, 3001, seed=22)
    cat = icr.DeviceCatalog(items)
    v, i = cat.topk(queries.cuda(), 100)
    vh, ih = cat.topk_host(queries.pin_memory(), 100)
    torch.cuda.current_stream().synchronize()
    assert torch.equal(vh, v.cpu()) and torch.equal(ih, i.cpu())
    rv, ri = oracle.cos_topk(queries[:200], items, 100)
    _check_topk(vh[:200], ih[:200], rv, ri, F32_RTOL)
    # batches in flight: join=False returns at once with an event; four different batches through two rotating output buffers
    qp = queries.pin_memory()
    outs = [(torch.empty(1000, 100).pin_memory(), torch.empty(1000, 100, dtype=torch.int64).pin_memory()) for _ in range(2)]
    done, got = [], []
    for b in range(4):
        if b >= 2:
            done[b - 2].synchronize()
            got.append((outs[b % 2][0].clone(), outs[b % 2][1].clone()))
        done.append(cat.topk_host(qp[b * 600 : b * 600 + 1000], 100, out=outs[b % 2], join=False, n_chunks=1)[2])
    for b in (2, 3):
        done[b].synchronize()
        got.append((outs[b % 2][0].clone(), outs[b % 2][1].clone()))
    for b, (gv, gi) in enumerate(got):
        assert torch.equal(gv, v[b * 600 : b * 600 + 1000].cpu()) and torch.equal(gi, i[b * 600 : b * 600 + 1000].cpu())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_gemm_path_ties_duplicates_and_adversarial_order(dtype):
    """Exactness of the threshold filter + histogram select under ties and a catalog sorted by similarity."""
    if not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    g = torch.Generator().manual_seed(3)
    base = torch.nn.functional.normalize(torch.randn(64, 128, generator=g), dim=1)
    # 9,000 rows drawn from only 64 distinct vectors: every score has ~140 exact duplicates
    rows = base[torch.randint(0, 64, (9000,), generator=g)].to(dtype)
    q = torch.nn.functional.normalize(torch.randn(300, 128, generator=g), dim=1).to(dtype)
    v, i = ops.cos_topk(q.cuda(), rows.cuda(), 100, path=ops.PATH_GEMM)
    rv, ri = oracle.cos_topk(q.float(), rows.float(), 100)
    tol = F32_RTOL if dtype == torch.float32 else BF16_RTOL
    err, _ = oracle.compare_topk(v.cpu(), i.cpu(), rv, ri, rtol=tol)
    assert err <= tol
    i = i.cpu()
    for r in range(0, 300, 17):
        assert len(set(i[r].tolist())) == 100
        # within a run of equal scores the lower rows must win (deterministic tie-break)
        vr = v[r].cpu()
        for a, b in zip(range(99), range(1, 100)):
            if vr[a] == vr[b]:
                assert i[r, a] < i[r, b]
    # catalog sorted so that every later row beats all earlier ones for query 0: the running threshold never helps,
    # segments overflow and the in-kernel compaction has to keep the result exact
    c = oracle.synth_isotropic(40000, 128, seed=5)
    q0 = oracle.synth_isotropic(130, 128, seed=6)
    order = torch.argsort(oracle.cos_sim(q0[:1], c)[0])
    c_sorted = c[order].to(dtype)
    v, i = ops.cos_topk(q0.to(dtype).cuda(), c_sorted.cuda(), 100, path=ops.PATH_GEMM)
    rv, ri = oracle.cos_topk(q0.to(dtype).float(), c_sorted.float(), 100)
    _check_topk(v, i, rv, ri, tol)


@pytest.mark.parametrize("Q", [300, 700])  # block-per-query select / warp-per-query select
def test_screened_fp32_band_overflow_is_ranked_exactly(Q):
    """The fp32 tensor path screens with ONE fp16 MMA term and carries every row within a band of the k-th screened score
    (k + k slots). 1,500 near-duplicates around the k-th rank overflow that band: those queries must fall back to the exact
    ranking of the whole catalog; the others (random directions) take the normal re-scoring. Also run with an exclusion mask."""
    if not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    g = torch.Generator().manual_seed(5)
    N, D, k = 20000, 384, 100
    items = oracle.synth_isotropic(N, D, seed=11)
    base = torch.nn.functional.normalize(torch.randn(1, D, generator=g), dim=1)
    dup_rows = torch.randperm(N, generator=g)[:1500]
    items[dup_rows] = torch.nn.functional.normalize(base + 2e-4 * torch.randn(1500, D, generator=g) / math.sqrt(D), dim=1)
    near = torch.nn.functional.normalize(base + 0.3 * torch.randn(Q // 2, D, generator=g) / math.sqrt(D), dim=1)
    queries = torch.cat([near, oracle.synth_isotropic(Q - Q // 2, D, seed=12)])[torch.randperm(Q, generator=g)]
    full = oracle.cos_sim(queries, items)
    cat = icr.DeviceCatalog(items)
    for mask in (None, (torch.arange(N) % 7 == 3)):
        v, i = cat.topk(queries.cuda(), k, exclude_mask=None if mask is None else mask.cuda(), path=ops.PATH_GEMM)
        s = full.clone()
        if mask is not None:
            s[:, mask] = float("-inf")
        rv, ri = torch.topk(s, k, dim=1)
        _check_topk(v, i, rv, ri, F32_RTOL)
        # every returned id carries its own exact score (a wrong row with a plausible score would pass the rank-wise check)
        got = torch.gather(s, 1, i.cpu())
        assert (got - v.cpu()).abs().max() < 2e-6


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("Q,N,D,k", [(8, 49688, 384, 10), (16, 49688, 384, 100), (64, 30000, 384, 10), (128, 49688, 384, 100), (9, 20000, 768, 256),
                                      (200, 49688, 384, 10), (256, 49688, 384, 32), (160, 40000, 384, 100),  # more queries than CTAs: rounds in the select tail / the select launch
                                      (33, 19200, 128, 1), (5, 100000, 384, 37), (2, 262144, 64, 5)])
def test_single_launch_swapped_path_vs_oracle(dtype, Q, N, D, k):
    """Request-sized batches on the tensor path: ONE GEMM launch whose thresholds are bootstrapped in the kernel (k-th largest
    of the per-warp group maxima of every CTA's first tile, grid barrier, then the filtered sweep) + one select. Covers ties
    at the bootstrap threshold (exact duplicates of the best rows), exclusion masks and k = 1 / 256."""
    if not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    items, _ = oracle.synth_clustered(N, D, seed=99)
    queries, src = oracle.synth_queries_from_items(items, Q, seed=98)
    items[::997] = items[src[0]]  # exact duplicates of one query's best row: equal scores at the threshold
    it, qt = items.to(dtype), queries.to(dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    rtol = F32_RTOL if dtype == torch.float32 else 5e-5
    full = oracle.cos_sim(qt.float(), it.float())
    for mask in (None, (torch.arange(N) % 5 == 1)):
        v, i = cat.topk(qt.cuda(), k, exclude_mask=None if mask is None else mask.cuda(), path=ops.PATH_GEMM)
        if Q <= 128 and D <= 384:
            assert ops.last_launch_count() <= 3, "expected the single-launch path (prep + GEMM + select)"
        sc = full.clone()
        if mask is not None:
            sc[:, mask] = float("-inf")
        rv, ri = torch.topk(sc, k, dim=1)
        _check_topk(v, i, rv, ri, rtol)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("Q,k", [(16, 100), (8, 10), (64, 37)])
def test_select_in_the_gemm_tail_on_a_catalog_sorted_by_similarity(dtype, Q, k):
    """Single-launch swapped path with the select in the kernel's tail (prep + ONE GEMM launch, no select launch). A catalog
    sorted by similarity to the queries is the worst case for its bootstrap threshold: the best rows all sit in the first
    chunks, the k-th largest group maximum comes from far down the order, thousands of rows pass the filter, the GEMM cuts
    its segments back and the tail's buffer overflows into the segment-by-segment loop. Results stay exact."""
    if not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    N, D = 49_688, 384
    g = torch.Generator().manual_seed(77)
    direction = torch.nn.functional.normalize(torch.randn(D, generator=g), dim=0)
    items = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1)
    order = torch.argsort(items @ direction, descending=True)
    items = items[order].contiguous()
    queries = torch.nn.functional.normalize(direction[None, :] + 0.05 * torch.randn(Q, D, generator=g), dim=1)
    it, qt = items.to(dtype), queries.to(dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    v, i = cat.topk(qt.cuda(), k, path=ops.PATH_GEMM)
    assert ops.last_launch_count() == 2, "expected prep + one GEMM launch with the select in its tail"
    rv, ri = oracle.cos_topk(qt.float(), it.float(), k)
    _check_topk(v, i, rv, ri, F32_RTOL if dtype == torch.float32 else 5e-5)
    # the ordinary case on the same catalog object: random queries, few survivors, the sparse gather
    q2 = torch.nn.functional.normalize(torch.randn(Q, D, generator=g), dim=1).to(dtype)
    v, i = cat.topk(q2.cuda(), k, path=ops.PATH_GEMM)
    assert ops.last_launch_count() == 2
    rv, ri = oracle.cos_topk(q2.float(), it.float(), k)
    _check_topk(v, i, rv, ri, F32_RTOL if dtype == torch.float32 else 5e-5)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_single_launch_k2_with_coarse_bootstrap_maxima(dtype):
    """One query block (Q = 200) on a catalog that streams from HBM (600,000 x 384): the queries-on-M kernel runs as ONE launch
    whose thresholds come from one maximum per bootstrap tile and column group (the 32-score block maxima would be more than the
    in-kernel ranking holds) - prep + GEMM + select, instead of four phases with a select each."""
    if not _gemm_ok():
        pytest.skip("GEMM path not built yet")
    N, D, Q, k = 600_000, 384, 200, 100
    g = torch.Generator(device="cuda").manual_seed(5)
    items = torch.nn.functional.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
    items[::1009] = items[7]  # exact duplicates: equal scores at and around the thresholds
    queries = torch.nn.functional.normalize(items[torch.arange(Q, device="cuda") * 2999] + 0.3 * torch.randn(Q, D, device="cuda", generator=g), dim=1)
    cat = icr.DeviceCatalog(items, dtype=dtype)
    qd = queries.to(dtype)
    v, i = cat.topk(qd, k)
    assert ops.last_launch_count() == 3, "expected prep + one GEMM launch + one select"
    ref = torch.nn.functional.normalize(qd.float(), dim=1) @ torch.nn.functional.normalize(cat.rows.float(), dim=1).T  # fp32 witness on the stored rows
    rv, ri = torch.topk(ref, k, dim=1)
    _check_topk(v, i, rv.cpu(), ri.cpu(), 2e-5 if dtype == torch.float32 else 5e-5)
    sample = torch.arange(0, Q, 25)
    ov, oi = oracle.cos_topk(qd[sample.cuda()].float().cpu(), cat.rows.float().cpu(), k)
    _check_topk(v[sample.cuda()], i[sample.cuda()], ov, oi, F32_RTOL if dtype == torch.float32 else 5e-5)


def test_full_size_properties_c2_shape():
    """BASELINE config 2 at full size through size-independent properties (the oracle is too slow for all of it):
    a row-permuted catalog returns the permuted ids with identical scores, every returned score is reproduced by
    a direct dot product, and a sample of queries matches the oracle exactly."""
    N, D, Q, k = 49688, 384, 10000, 100
    g = torch.Generator(device="cuda").manual_seed(1234)
    items = torch.nn.functional.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
    queries = torch.nn.functional.normalize(torch.randn(Q, D, device="cuda", generator=g), dim=1)
    v, i = icr.cos_topk(queries, items, k)
    assert (v[:, :-1] >= v[:, 1:]).all() and (i >= 0).all() and (i < N).all()
    direct = (queries[:, None, :] * items[i[:, :5]]).sum(-1)
    assert (direct - v[:, :5]).abs().max() < 2e-6
    perm = torch.randperm(N, device="cuda", generator=g)
    v2, i2 = icr.cos_topk(queries[:512], items[perm], k)
    assert torch.allclose(v2, v[:512], rtol=1e-6, atol=1e-7)
    same = perm[i2] == i[:512]
    assert same.float().mean() > 0.999  # differences only across exact-score ties
    sample = torch.arange(0, Q, 97, device="cuda")
    rv, ri = oracle.cos_topk(queries[sample].cpu(), items.cpu(), k)
    _check_topk(v[sample], i[sample], rv, ri, F32_RTOL)


def test_c2_planted_relevance_recall_and_ndcg_full_size():
    """BASELINE config 2 end to end at full size: recall@10 / NDCG@10 (and the rest of the evaluator's metrics) from
    planted relevance, computed by the device pipeline (fused top-100 -> metric kernel) and by the oracle
    (cos_sim + topk on the CPU -> per-query loops) — identical up to tie swaps, i.e. to ~1e-4 in the mean."""
    N, D, Q, k = 49688, 384, 10000, 100
    items, centre_of = oracle.synth_clustered(N, D, seed=1234)
    queries, src = oracle.synth_queries_from_items(items, Q, seed=4321)
    src = src.tolist()
    rng = np.random.default_rng(99)
    by_centre: dict[int, list[int]] = {}
    for r, c in enumerate(centre_of.tolist()):
        by_centre.setdefault(c, []).append(r)
    relevant = []
    for q in range(Q):  # the item the query was generated from plus a few of its cluster
        mates = by_centre[int(centre_of[src[q]])]
        relevant.append({src[q], *(int(x) for x in rng.choice(mates, size=min(4, len(mates)), replace=False))})
    v, i = icr.cos_topk(queries.cuda(), items.cuda(), k)
    table = ops.RelevanceTable([sorted(r) for r in relevant], device="cuda")
    specs = [(ops.METRIC_RECALL, 10), (ops.METRIC_NDCG, 10), (ops.METRIC_MRR, 10), (ops.METRIC_ACCURACY, 1), (ops.METRIC_MAP, 100)]
    means, per_query = ops.ir_metrics(i, table, specs)
    rv, ri = oracle.cos_topk(queries, items, k)
    want, want_pq = oracle.st_ir_metrics(ri.tolist(), relevant, accuracy_at_k=(1,), precision_recall_at_k=(10,), mrr_at_k=(10,),
                                         ndcg_at_k=(10,), map_at_k=(100,), per_query=True)
    got = dict(zip(["recall@10", "ndcg@10", "mrr@10", "accuracy@1", "map@100"], means.tolist()))
    assert got["recall@10"] > 0.2  # the planted item is found: the numbers are not trivially zero
    for name, val in got.items():
        assert val == pytest.approx(want[name], abs=2e-4), name
    # per query: identical wherever the id lists are identical (they differ only across score ties)
    same_rows = (i.cpu() == ri).all(dim=1).numpy()
    assert same_rows.mean() > 0.95  # rows with a swap across a score tie (adjacent top-100 gaps below 1e-5 relative occur in ~1 % of positions)
    cols = {"accuracy@1": 0, "precision@10": 1, "recall@10": 2, "mrr@10": 3, "ndcg@10": 4, "map@100": 5}
    pq = per_query.cpu().numpy()
    for j, name in enumerate(["recall@10", "ndcg@10", "mrr@10", "accuracy@1", "map@100"]):
        np.testing.assert_allclose(pq[same_rows, j], want_pq[same_rows, cols[name]], rtol=0, atol=1e-12)


def test_peer_memory_exchange_equals_nccl_all_gather():
    """icr_peer_exchange (NVLink peer stores + flags) gathers the same candidates as the NCCL all-gather: 2 ranks."""
    import os
    import subprocess
    import sys
    from pathlib import Path

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one machine")
    root = Path(__file__).resolve().parents[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29517",
           str(root / "benchmarks" / "peer_exchange_case.py"), "100000"]
    out = subprocess.run(cmd, cwd=str(root), capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert out.returncode == 0, out.stderr[-2000:]
    assert "PEER_EXCHANGE_OK" in out.stdout, out.stdout[-2000:]


def test_mnrl_gathered_negatives_two_ranks_nccl():
    """MultipleNegativesRankingLoss(gather_across_devices=True) on 2 GPUs == the oracle's single-process restatement."""
    import os
    import subprocess
    import sys
    from pathlib import Path

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one machine")
    root = Path(__file__).resolve().parents[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29519",
           str(root / "benchmarks" / "mnrl_gathered_case.py")]
    out = subprocess.run(cmd, cwd=str(root), capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert out.returncode == 0, out.stderr[-2000:]
    assert "MNRL_GATHERED_OK" in out.stdout, out.stdout[-2000:]
