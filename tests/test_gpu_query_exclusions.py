"""Per-query exclusions in the fused cosine top-k (icr_query_exclusion_bits / icr_cos_topk_excl) and
Recommender.recommend_batch, on every plan branch, against an fp32 torch witness (B200 only)."""

import json
import os

import numpy as np
import pytest
import torch

import instacart_next_order_recommendation_b200 as icr
from instacart_next_order_recommendation_b200 import ops
from oracle import oracle

pytestmark = pytest.mark.gpu

F32_RTOL, BF16_RTOL = 1e-5, 2e-3


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert torch.cuda.is_available(), "run with -m gpu on a GPU box"
    torch.cuda.set_device(0)
    assert icr._lib.load().icr_device_supported() == 1
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
    rk = np.asarray(rv, dtype=np.float64)[:, -1]
    assert (v.double().numpy()[:, -1] >= rk - rtol * np.maximum(np.abs(rk), 0.05)).all(), "k-th returned score below the oracle's k-th"


def _excluded_matrix(lists, Q, N):
    """bool [Q, N] on the device: True where query q excludes row r (rows outside [0, N) ignored)."""
    arrs = [np.asarray(r, dtype=np.int64).reshape(-1) for r in lists]
    qi = np.repeat(np.arange(Q, dtype=np.int64), [a.size for a in arrs])
    ri = np.concatenate(arrs) if arrs else np.zeros(0, np.int64)
    keep = (ri >= 0) & (ri < N)
    m = torch.zeros(Q, N, dtype=torch.bool, device="cuda")
    m[torch.from_numpy(qi[keep]).cuda(), torch.from_numpy(ri[keep]).cuda()] = True
    return m


def _witness_check(v, i, qt, it, k, lists, rtol, mask=None):
    """fp32 cos_sim on the (rounded) inputs with the excluded entries at -inf, then torch.topk."""
    Q, N = qt.shape[0], it.shape[0]
    s = torch.nn.functional.normalize(qt.float().cuda(), dim=1) @ torch.nn.functional.normalize(it.float().cuda(), dim=1).T
    ex = _excluded_matrix(lists, Q, N)
    if mask is not None:
        ex |= mask.bool().cuda()[None, :]
    s[ex] = float("-inf")
    rv, ri = torch.topk(s, k, dim=1)
    rv, ri = rv.cpu(), ri.cpu()
    ri = torch.where(torch.isinf(rv), torch.full_like(ri, -1), ri)
    v, i = v.cpu(), i.cpu()
    live = ~torch.isinf(rv)
    assert torch.equal(torch.isinf(v), ~live), "eligible-row count differs"
    assert (i[~live] == -1).all()
    got_ex = ex.cpu().gather(1, i.clamp(min=0))
    assert not (got_ex & live).any(), "an excluded row was returned"
    full = live.all(dim=1)
    if full.any():
        _check_topk(v[full], i[full], rv[full], ri[full], rtol)
    for q in torch.nonzero(~full).flatten().tolist():  # short lists: exactly the eligible rows, best first
        n = int(live[q].sum())
        if n:
            _check_topk(v[q : q + 1, :n], i[q : q + 1, :n], rv[q : q + 1, :n], ri[q : q + 1, :n], rtol)


def _data(N, D, Q, seed, dtype):
    items, _ = oracle.synth_clustered(N, D, seed=seed)
    queries, _ = oracle.synth_queries_from_items(items, Q, seed=seed + 1)
    return items.to(dtype), queries.to(dtype)


def _random_lists(Q, N, per_query, seed):
    rng = np.random.default_rng(seed)
    return [rng.choice(N, size=min(per_query, N), replace=False).tolist() for _ in range(Q)]


def _own_best(qt, it, n):
    s = torch.nn.functional.normalize(qt.float().cuda(), dim=1) @ torch.nn.functional.normalize(it.float().cuda(), dim=1).T
    return torch.topk(s, n, dim=1).indices.cpu().tolist()


def _run(cat, qt, k, lists, path=ops.PATH_AUTO, mask=None):
    return cat.topk(qt.cuda(), k, exclude_rows=lists, exclude_mask=None if mask is None else mask.cuda(), path=path)


DTYPES = [(torch.float32, F32_RTOL), (torch.bfloat16, BF16_RTOL)]


def test_bitmap_layout_and_csr_form():
    N, lists = 100, [[0, 31, 32, 99, 99, -1, 100, 5000], [], [64]]
    bits = ops.query_exclusion_bits(lists, N, "cuda")
    assert bits.dtype == torch.uint32 and tuple(bits.shape) == (4, 3)
    b = bits.view(torch.int32).cpu().numpy().view(np.uint32)
    assert b[0, 0] == (1 | (1 << 31)) and b[1, 0] == 1 and b[3, 0] == (1 << 3) and b[2, 0] == 0
    assert (b[:, 1] == 0).all() and b[2, 2] == 1
    off = torch.tensor([0, 8, 8, 9], dtype=torch.int64)
    rows = torch.tensor([r for l in lists for r in l], dtype=torch.int64)
    assert torch.equal(ops.query_exclusion_bits((off, rows), N, "cuda").view(torch.int32), bits.view(torch.int32))
    with pytest.raises(ValueError):
        ops.cos_topk(torch.randn(2, 64, device="cuda"), torch.randn(N, 64, device="cuda"), 5, exclude_bits=bits)  # Q mismatch


@pytest.mark.parametrize("dtype,rtol", DTYPES)
@pytest.mark.parametrize("Q", [1, 3, 7])
def test_gemv_path(dtype, rtol, Q):
    it, qt = _data(49_688, 384, Q, 11, dtype)
    for norms in (True, False):  # the single-query ring kernel with precomputed norms, and without
        cat = icr.DeviceCatalog(it.cuda(), dtype=dtype, build_planes=False)
        if not norms:
            cat.inv_norms = None
        lists = _own_best(qt, it, 100)
        lists[0] = lists[0][:10] + [-5, 10**9, lists[0][0]]  # out-of-range and duplicate ids
        v, i = _run(cat, qt, 10, lists, path=ops.PATH_GEMV)
        assert ops.last_launch_count() == 1
        _witness_check(v, i, qt, it, 10, lists, rtol)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
@pytest.mark.parametrize("Q", [8, 32, 64])
def test_swapped_single_launch_select_in_tail(dtype, rtol, Q):
    it, qt = _data(49_688, 384, Q, 12, dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    lists = _own_best(qt, it, 1000)
    lists = [l[: (10, 100, 1000)[q % 3]] for q, l in enumerate(lists)]  # every bootstrap maximum moves
    v, i = _run(cat, qt, 10, lists, path=ops.PATH_GEMM)
    assert ops.last_launch_count() == 2, "expected prep + one GEMM launch with the select in its tail"
    _witness_check(v, i, qt, it, 10, lists, rtol)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
def test_swapped_single_launch_with_select_launch(dtype, rtol):
    it, qt = _data(49_688, 384, 256, 13, dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    lists = [l + r for l, r in zip(_own_best(qt, it, 100), _random_lists(256, 49_688, 16, 3))]
    v, i = _run(cat, qt, 100, lists, path=ops.PATH_GEMM)
    assert ops.last_launch_count() == 3, "expected prep + one GEMM launch + one select"
    _witness_check(v, i, qt, it, 100, lists, rtol)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
def test_k2_single_launch(dtype, rtol):
    Q = 1000
    it, qt = _data(49_688, 384, Q, 14, dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    lists = _own_best(qt, it, 100)
    lists = [l[: (10, 100, 0)[q % 3]] + r for q, (l, r) in enumerate(zip(lists, _random_lists(Q, 49_688, 16, 4)))]
    lists[5] = []
    v, i = _run(cat, qt, 100, lists)
    # prep + GEMM + select (+ the exact re-scoring of screened fp32 candidates)
    assert ops.last_launch_count() == (4 if dtype == torch.float32 else 3)
    _witness_check(v, i, qt, it, 100, lists, rtol)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
def test_k2_coarse_bootstrap(dtype, rtol):
    N, D, Q, k = 600_000, 384, 200, 100
    g = torch.Generator(device="cuda").manual_seed(5)
    items = torch.nn.functional.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
    items[::1009] = items[7]
    queries = torch.nn.functional.normalize(items[torch.arange(Q, device="cuda") * 2999] + 0.3 * torch.randn(Q, D, device="cuda", generator=g), dim=1)
    cat = icr.DeviceCatalog(items, dtype=dtype)
    qd = queries.to(dtype)
    it = cat.rows[:, :D]
    lists = _own_best(qd, it, 300)
    v, i = _run(cat, qd, k, lists)
    assert ops.last_launch_count() == 3, "expected prep + one GEMM launch + one select"
    _witness_check(v, i, qd, it, k, lists, 2e-5 if dtype == torch.float32 else rtol)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
@pytest.mark.parametrize("Q", [300, 600])  # block-per-query select, warp-per-query select over the dense first phase
def test_phased_path_with_dense_first_phase(dtype, rtol, Q):
    N, k = 5000, 100
    it, qt = _data(N, 384, Q, 15, dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    lists = _own_best(qt, it, 200)
    lists = [l[: (10, 200, 0)[q % 3]] + r for q, (l, r) in enumerate(zip(lists, _random_lists(Q, N, 16, 5)))]
    lists[1] = list(range(0, 1024, 2))  # half of the densely scored rows
    v, i = _run(cat, qt, k, lists, path=ops.PATH_GEMM)
    assert ops.last_launch_count() >= 5, "expected prep, the dense first phase and its select, then sparse phases"
    _witness_check(v, i, qt, it, k, lists, rtol)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
@pytest.mark.parametrize("Q,k", [(16, 100), (8, 10), (300, 50)])
def test_catalog_sorted_by_similarity(dtype, rtol, Q, k):
    """The best rows sit in the first chunks: segments are cut back in the kernel; the exclusions hit exactly those rows."""
    N, D = 49_688, 384
    g = torch.Generator().manual_seed(77)
    direction = torch.nn.functional.normalize(torch.randn(D, generator=g), dim=0)
    items = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1)
    items = items[torch.argsort(items @ direction, descending=True)].contiguous()
    queries = torch.nn.functional.normalize(direction[None, :] + 0.05 * torch.randn(Q, D, generator=g), dim=1)
    it, qt = items.to(dtype), queries.to(dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    lists = [list(range(q % 7, 3000, 3)) for q in range(Q)]
    v, i = _run(cat, qt, k, lists, path=ops.PATH_GEMM)
    _witness_check(v, i, qt, it, k, lists, rtol)


@pytest.mark.parametrize("Q", [8, 1000])
def test_near_duplicates_overflow_the_screening_band(Q):
    """1,500 near-copies of one row: more near-ties than the fp32 screening band carries, so the whole catalog is ranked
    exactly for these queries - with each query's own exclusions."""
    N, D = 49_688, 384
    g = torch.Generator().manual_seed(3)
    items = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1)
    dup = torch.arange(1500) * 31
    items[dup] = torch.nn.functional.normalize(items[0][None, :] + 1e-4 * torch.randn(1500, D, generator=g), dim=1)
    queries = torch.nn.functional.normalize(items[0][None, :] + 1e-3 * torch.randn(Q, D, generator=g), dim=1)
    cat = icr.DeviceCatalog(items.cuda(), dtype=torch.float32)
    rng = np.random.default_rng(9)
    lists = [dup[rng.random(1500) < 0.4].tolist() for _ in range(Q)]
    v, i = _run(cat, queries, 100, lists)
    _witness_check(v, i, queries, items, 100, lists, F32_RTOL)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
@pytest.mark.parametrize("Q", [2, 16, 1000])
def test_every_row_and_all_but_k_minus_3(dtype, rtol, Q):
    N, k = 20_000, 50
    it, qt = _data(N, 384, Q, 16, dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    rng = np.random.default_rng(17)
    lists = [[] for _ in range(Q)]
    lists[0] = list(range(N))  # nothing eligible: an all (-inf, -1) row
    lists[1] = rng.permutation(N)[: N - k + 3].tolist()  # k - 3 eligible rows
    for q in range(2, Q):
        lists[q] = rng.choice(N, size=int(rng.integers(0, 64)), replace=True).tolist() + [-1, N, N + 40]
    mask = torch.zeros(N, dtype=torch.uint8)
    mask[::97] = 1  # combined with the shared mask
    v, i = _run(cat, qt, k, lists, mask=mask)
    assert (i[0] == -1).all() and torch.isinf(v[0]).all()
    assert int((i[1] >= 0).sum()) <= k - 3
    _witness_check(v, i, qt, it, k, lists, rtol, mask=mask)


@pytest.mark.parametrize("dtype,rtol", DTYPES)
@pytest.mark.parametrize("Q,N,k,path", [(1, 49_688, 10, ops.PATH_GEMV), (5, 30_000, 100, ops.PATH_GEMV), (32, 49_688, 10, ops.PATH_GEMM),
                                         (256, 49_688, 100, ops.PATH_GEMM), (1000, 49_688, 100, ops.PATH_AUTO), (400, 5000, 100, ops.PATH_GEMM)])
def test_same_list_for_every_query_equals_the_shared_mask(dtype, rtol, Q, N, k, path):
    it, qt = _data(N, 384, Q, 18, dtype)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype)
    rows = np.random.default_rng(19).choice(N, size=N // 10, replace=False)
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[torch.as_tensor(rows, device="cuda")] = 1
    v0, i0 = cat.topk(qt.cuda(), k, exclude_mask=mask, path=path)
    v1, i1 = cat.topk(qt.cuda(), k, exclude_rows=[rows.tolist()] * Q, path=path)
    assert torch.equal(i0, i1) and torch.equal(v0, v1)


def test_bitmap_chunks_for_large_batches(monkeypatch):
    it, qt = _data(20_000, 128, 300, 20, torch.float32)
    cat = icr.DeviceCatalog(it.cuda())
    lists = _random_lists(300, 20_000, 40, 21)
    v0, i0 = cat.topk(qt.cuda(), 20, exclude_rows=lists)
    monkeypatch.setattr(icr.DeviceCatalog, "EXCLUSION_BITS_MAX_BYTES", 64 * 4 * ops.exclusion_words(20_000))
    v1, i1 = cat.topk(qt.cuda(), 20, exclude_rows=lists)  # five chunks of <= 64 queries
    assert torch.equal(i0, i1) and torch.equal(v0, v1)
    _witness_check(v1, i1, qt, it, 20, lists, F32_RTOL)


# ---- Recommender.recommend_batch ---------------------------------------------------------------------------------------------
def _recommender(golden_dir, tmp_path, encoder_cls):
    z = np.load(golden_dir / "embeddings_small.npz")
    pids = [str(p) for p in z["product_ids"]]
    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text(json.dumps({pid: f"c:{i}" for i, pid in enumerate(pids)}))
    return icr.Recommender("fake-model", corpus, model=encoder_cls(z)), pids


class _HostEnc:
    """The reference's encode call only: any other keyword (convert_to_tensor) is a TypeError."""

    def __init__(self, z):
        self.z = z

    def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True):
        tab = {"c": self.z["items"], "q": self.z["queries"]}
        return np.stack([tab[t.split(":")[0]][int(t.split(":")[1])] for t in texts]).astype(np.float32)


class _DeviceEnc(_HostEnc):
    calls = 0

    def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True, convert_to_tensor=False):
        out = _HostEnc.encode(self, texts)
        if convert_to_tensor:
            _DeviceEnc.calls += 1
            return torch.from_numpy(out).cuda()
        return out


@pytest.mark.parametrize("enc", [_DeviceEnc, _HostEnc])
def test_recommend_batch_matches_golden(golden_dir, tmp_path, enc):
    gold = json.loads((golden_dir / "recommend_golden.json").read_text())
    rec, _ = _recommender(golden_dir, tmp_path, enc)
    by_k = {}
    for case in gold["cases"]:
        by_k.setdefault(case["top_k"], []).append(case)
    for top_k, cases in by_k.items():
        got = rec.recommend_batch([f"q:{c['q']}" for c in cases], top_k=top_k, exclude_product_ids=[set(c["exclude"]) for c in cases])
        for g, c in zip(got, cases):
            assert [p for p, _ in g] == [p for p, _ in c["result"]], c
            np.testing.assert_allclose([s for _, s in g], [s for _, s in c["result"]], rtol=1e-5)
    assert rec._query_on_device is (enc is _DeviceEnc)


def test_recommend_batch_equals_a_recommend_loop(golden_dir, tmp_path):
    rec, pids = _recommender(golden_dir, tmp_path, _DeviceEnc)
    rng = np.random.default_rng(23)
    queries = [f"q:{q % 10}" for q in range(24)]
    excl = [set(rng.choice(pids, size=int(rng.choice([0, 5, 300, 700])), replace=False).tolist()) | {"no-such-id"} for _ in queries]
    excl[3] = None
    excl[4] = set(pids)  # nothing eligible
    excl[5] = set(pids[: len(pids) - 4])  # fewer eligible products than top_k
    def same(got, want):  # same products in the same order; scores of the batched and the request kernels agree to 1e-6
        assert [[p for p, _ in r] for r in got] == [[p for p, _ in r] for r in want]
        for g, w in zip(got, want):
            np.testing.assert_allclose([s for _, s in g], [s for _, s in w], rtol=1e-6)

    for top_k in (1, 10, 100):
        got = rec.recommend_batch(queries, top_k=top_k, exclude_product_ids=excl)
        same(got, [rec.recommend(q, top_k=top_k, exclude_product_ids=e) for q, e in zip(queries, excl)])
        assert got[4] == [] and len(got[5]) == min(top_k, 4)
    same(rec.recommend_batch(queries[:3], top_k=5), [rec.recommend(q, top_k=5) for q in queries[:3]])
    assert rec.recommend_batch([], top_k=10) == []
    assert rec.recommend_batch(queries[:2], top_k=0) == [[], []]
    with pytest.raises(ValueError):
        rec.recommend_batch(queries[:2], top_k=ops.MAX_K + 1)
    with pytest.raises(ValueError):
        rec.recommend_batch(queries[:2], exclude_product_ids=[None])


# ---- seeded fuzz against the witness ---------------------------------------------------------------------------------------
_N_CASES = int(os.environ.get("ICR_XFUZZ_CASES", "48"))
_SEED = int(os.environ.get("ICR_XFUZZ_SEED", "20261021"))


def _fuzz_cases(n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for c in range(n):
        Q = int(rng.choice([1, 2, 3, 5, 7, 8, 33, 130, 256, 300, 700, 1100]))
        N = int(rng.choice([7, 100, 1000, 4097, 20_000, 49_688, 70_001]))
        D = int(rng.choice([64, 128, 384, 768]))
        k = int(rng.choice([1, 5, 10, 37, 100, 256]))
        dtype = torch.float32 if rng.random() < 0.5 else torch.bfloat16
        path = int(rng.choice([ops.PATH_AUTO, ops.PATH_GEMV, ops.PATH_GEMM]))
        density = float(rng.choice([0.0, 1e-3, 0.01, 0.2, 0.9]))
        out.append((c, Q, N, D, k, dtype, path, density))
    return out


@pytest.mark.parametrize("case", _fuzz_cases(_N_CASES, _SEED), ids=lambda c: f"{c[0]}-Q{c[1]}-N{c[2]}-D{c[3]}-k{c[4]}-{str(c[5]).split('.')[-1]}-p{c[6]}-x{c[7]}")
def test_fuzz_against_witness(case):
    c, Q, N, D, k, dtype, path, density = case
    if path == ops.PATH_GEMV and Q > 64:
        path = ops.PATH_AUTO  # keeps the case fast; small batches cover the GEMV kernels
    it = oracle.synth_unnormalised(N, D, seed=3000 + c).to(dtype)
    qt = oracle.synth_unnormalised(Q, D, seed=4000 + c).to(dtype)
    rng = np.random.default_rng(5000 + c)
    lists = [np.nonzero(rng.random(N) < density)[0] for _ in range(Q)]
    if Q > 1:
        lists[-1] = np.zeros(0, np.int64)
    kk = min(k, N)
    cat = icr.DeviceCatalog(it.cuda(), dtype=dtype, row_offset=3)
    v, i = cat.topk(qt.cuda(), kk, exclude_rows=lists, path=path)
    i = torch.where(i >= 0, i - 3, i)
    _witness_check(v, i, qt, it, kk, lists, F32_RTOL if dtype == torch.float32 else BF16_RTOL)
