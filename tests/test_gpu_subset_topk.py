"""Top-k over per-query candidate lists (icr_cos_topk_subset): ops.cos_topk_subset, DeviceCatalog.topk(include_rows=...),
ShardedCatalog.topk(include_rows=...) and Recommender's candidate_product_ids.

fp32 and int8 catalogs must return, bit for bit, what the fused top-k returns on the same DeviceCatalog with the complement
of each list excluded (fp32: the tensor-core path, whose exact re-scoring arithmetic the subset kernel shares). bf16 / fp16
catalogs are checked against fp64 on the values the kernel consumed. The CPU-only cases at the top check the ABI surface and
the argument errors that need no device."""

import ctypes
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import instacart_next_order_recommendation_b200 as icr
from instacart_next_order_recommendation_b200 import _lib, ops
from oracle import oracle


# ---- CPU-only: ABI surface and argument errors ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def lib():
    try:
        return _lib.load()
    except _lib.NativeLibraryMissing:
        pytest.skip("library not built")


def test_subset_entry_is_declared_and_exported(lib):
    header = (_lib.Path(__file__).resolve().parents[1] / "include" / "icr_b200.h").read_text()
    for name in ("icr_cos_topk_subset", "icr_cos_topk_subset_workspace_bytes"):
        assert name in header and name in _lib.SIGNATURES
        assert getattr(lib, name) is not None


def _subset_call(lib, *, dtype=_lib.ICR_F32, D=384, k=10, offsets=1, rows=1, nnz=4, inv=16, Q=2):
    fake = ctypes.c_void_p(1 << 20)  # 16-byte aligned non-null stand-ins: every check below fails before any access
    ptr = lambda v: None if v is None else ctypes.c_void_p(v << 20) if v else None  # noqa: E731
    return lib.icr_cos_topk_subset(fake, Q, D, fake, 100, D, D, dtype, ptr(inv), ptr(offsets), ptr(rows), nnz, k, 0, fake, fake,
                                   fake, 1 << 20, None)


def test_argument_errors_without_a_device(lib):
    assert _subset_call(lib, rows=None) == -1  # null CSR rows with nnz > 0
    assert _subset_call(lib, offsets=None) == -1  # null offsets
    assert _subset_call(lib, k=0) == -4
    assert _subset_call(lib, k=257) == -4
    assert _subset_call(lib, dtype=_lib.ICR_I8, D=40) == -3  # int8 rows need D % 16 == 0
    assert _subset_call(lib, inv=None) == -1  # the inverse norms (int8: factors) are required
    assert _subset_call(lib, dtype=_lib.ICR_I8, D=384, inv=None) == -1
    assert b"cos_topk_subset" in lib.icr_last_error_string()


def test_workspace_is_not_nnz_sized(lib):
    small = lib.icr_cos_topk_subset_workspace_bytes(1, 5_000, 384, _lib.ICR_F32, 10)
    big = lib.icr_cos_topk_subset_workspace_bytes(1, 10_000_000, 384, _lib.ICR_F32, 10)
    assert small < 64 * 1024
    assert big < 10_000_000 * 8 // 4  # 2 * ceil(nnz / chunk) * k keys, chunk >= 4k
    assert lib.icr_cos_topk_subset_workspace_bytes(1, 10_000_000, 384, _lib.ICR_F32, 256) < 10_000_000 * 8 // 2


# ---- GPU -----------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@pytest.fixture(scope="module")
def cuda0():
    assert torch.cuda.is_available(), "run with -m gpu on a GPU box"
    torch.cuda.set_device(0)
    assert _lib.load().icr_device_supported() == 1
    yield
    torch.cuda.synchronize()


def _data(N, D, Q, seed, normalize=True):
    items, _ = oracle.synth_clustered(N, D, seed=seed)
    queries, _ = oracle.synth_queries_from_items(items, Q, seed=seed + 1)
    if not normalize:
        g = torch.Generator().manual_seed(seed + 2)
        items = items * (0.5 + 3 * torch.rand(N, 1, generator=g))
        queries = queries * (0.5 + 3 * torch.rand(Q, 1, generator=g))
    return items.float(), queries.float()


def _lists(Q, N, seed, lo=0, hi=None):
    rng = np.random.default_rng(seed)
    hi = N if hi is None else hi
    return [rng.choice(N, size=int(rng.integers(lo, hi + 1)), replace=False).tolist() for _ in range(Q)]


def _complement(lists, N):
    out = []
    for r in lists:
        keep = np.ones(N, bool)
        r = np.asarray(r, np.int64)
        keep[r[(r >= 0) & (r < N)]] = False
        out.append(np.flatnonzero(keep).tolist())
    return out


def _same(a, b):
    (v0, i0), (v1, i1) = a, b
    assert v0.shape == v1.shape and i0.shape == i1.shape
    assert torch.equal(i0.cpu(), i1.cpu()), "ids differ"
    assert torch.equal(v0.cpu().view(torch.int32), v1.cpu().view(torch.int32)), "score bits differ"


EXACT_CASES = []
for _dt in ("f32", "i8"):
    for _j, _Q in enumerate([1, 3, 7, 8, 64, 256, 10_000]):
        for _k in ([1, 10, 100, 256] if _Q <= 256 else [10, 100]):
            EXACT_CASES.append((_dt, _Q, _k, [384, 768, 100 if _dt == "f32" else 112][(_j + _k) % 3], (_j + _k) % 2 == 0))


@gpu
@pytest.mark.parametrize("dt,Q,k,D,normalize", EXACT_CASES)
def test_bit_identity_with_the_complement_call(cuda0, dt, Q, k, D, normalize):
    N = 3_000 if Q < 10_000 else 1_000
    items, queries = _data(N, D, Q, seed=Q + k + D, normalize=normalize)
    cat = icr.DeviceCatalog(items, dtype=torch.float32 if dt == "f32" else torch.int8)
    lists = _lists(Q, N, seed=k, lo=0, hi=min(N, 600))
    got = cat.topk(queries.cuda(), k, include_rows=lists)
    # fp32: the tensor-core path (its re-scoring arithmetic is the subset kernel's); int8: the planned path
    path = ops.PATH_GEMM if dt == "f32" else ops.PATH_AUTO
    _same(got, cat.topk(queries.cuda(), k, exclude_rows=_complement(lists, N), path=path))


@gpu
@pytest.mark.parametrize("Q", [1, 3, 7])
def test_fp32_gemv_plan_agrees_up_to_rounding(cuda0, Q):
    """The fused fp32 GEMV path normalises the query before the dot product and sums in another order than the
    tensor-core path's exact re-scoring, so the two fused paths differ in the last bits. The subset call follows the
    tensor-core path bit for bit; against the GEMV plan it agrees to fp32 rounding, ids equal outside ties."""
    N, D, k = 3_000, 384, 10
    items, queries = _data(N, D, Q, seed=Q)
    cat = icr.DeviceCatalog(items)
    lists = _lists(Q, N, seed=Q, lo=50, hi=800)
    v, i = cat.topk(queries.cuda(), k, include_rows=lists)
    rv, ri = cat.topk(queries.cuda(), k, exclude_rows=_complement(lists, N), path=ops.PATH_GEMV)
    err, mism = oracle.compare_topk(v.cpu(), i.cpu(), rv.cpu(), ri.cpu(), rtol=1e-6)
    assert err <= 1e-6 and mism == 0, (err, mism)


def _tol(s, D):
    t = 1e-5 * s.abs().clamp(min=0.05)
    return t + (2e-6 + (D / 16) * 2.0**-23 * s.abs()) if D >= 2048 else t


def _check_16(v, i, q16, c16, k, lists, offset=0):
    """fp64 on the 16-bit values consumed, only the listed rows eligible; tie-tolerant ids, rank-k membership."""
    Q, N, D = q16.shape[0], c16.shape[0], q16.shape[1]
    s = F.normalize(q16.cuda().double(), dim=1) @ F.normalize(c16.cuda().double(), dim=1).T
    allowed = torch.zeros(Q, N, dtype=torch.bool, device="cuda")
    for q, r in enumerate(lists):
        r = np.asarray(r, np.int64)
        r = r[(r >= 0) & (r < N)]
        allowed[q, torch.from_numpy(r).cuda()] = True
    s[~allowed] = float("-inf")
    if N < k:
        s = torch.cat([s, torch.full((Q, k - N), float("-inf"), dtype=s.dtype, device=s.device)], dim=1)
    rv = torch.topk(s, k, dim=1).values
    v, i = v.cuda().double(), i.cuda()
    i = torch.where(i >= 0, i - offset, i)
    live = torch.isfinite(rv)
    assert (v[:, :-1] >= v[:, 1:]).all()
    assert torch.equal(torch.isfinite(v), live), "eligible-row count differs"
    assert (i[~live] == -1).all()
    sv = s.gather(1, i.clamp(min=0))
    assert torch.isfinite(sv[live]).all(), "a row outside the list was returned"
    assert ((v - sv).abs() <= _tol(sv, D))[live].all(), "score outside the contract"
    tol_r = _tol(rv.masked_fill(~live, 0.0), D)
    assert ((sv - rv).abs() <= 2 * tol_r + 1e-12)[live].all(), "an id differs from the reference outside near-ties"
    assert (v[:, -1] >= rv[:, -1] - tol_r[:, -1])[live[:, -1]].all()
    for q in range(Q):
        got = [x for x in i[q].tolist() if x >= 0]
        assert len(set(got)) == len(got)


@gpu
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("Q,k,D", [(1, 10, 384), (3, 100, 768), (64, 256, 128), (1000, 10, 2048)])
def test_16bit_against_fp64(cuda0, dtype, Q, k, D):
    N = 4_000
    items, queries = _data(N, D, Q, seed=D + k)
    cat = icr.DeviceCatalog(items, dtype=dtype)
    lists = _lists(Q, N, seed=Q, lo=0, hi=900)
    q16 = cat._device_queries(queries)
    v, i = cat.topk(q16, k, include_rows=lists)
    _check_16(v, i, q16, cat.rows, k, lists)


# ---- list shapes (exact witness: fp32 vs the tensor-core complement call, int8 vs the planned one) ----------------------
def _exact_pair(dt, N=2_000, D=384, Q=5, seed=0):
    items, queries = _data(N, D, Q, seed=seed)
    cat = icr.DeviceCatalog(items, dtype=torch.float32 if dt == "f32" else torch.int8)
    return cat, queries.cuda(), (ops.PATH_GEMM if dt == "f32" else ops.PATH_AUTO)


@gpu
@pytest.mark.parametrize("dt", ["f32", "i8"])
def test_list_shapes(cuda0, dt):
    cat, q, path = _exact_pair(dt)
    N = len(cat)
    rng = np.random.default_rng(3)
    shapes = [
        [],  # empty
        rng.choice(N, 4, replace=False).tolist(),  # shorter than k
        [17],  # a single row
        list(range(N))[::-1],  # the whole catalog, unsorted
        rng.permutation(N)[:700].tolist() + [-5, N, N + 100, 1 << 40],  # unsorted, with out-of-range rows
    ]
    k = 10
    got = cat.topk(q, k, include_rows=shapes)
    _same(got, cat.topk(q, k, exclude_rows=_complement(shapes, N), path=path))
    v, i = got
    assert torch.isinf(v[0]).all() and (i[0] == -1).all()
    assert (i[1, 4:] == -1).all() and torch.isinf(v[1, 4:]).all()
    assert i[2, 0].item() == 17 and (i[2, 1:] == -1).all()
    # the whole catalog equals the plain fused call
    whole = cat.topk(q[3:4], k, include_rows=[list(range(N))])
    _same(whole, cat.topk(q[3:4], k, path=path))


@gpu
def test_fewer_rows_than_k_and_row_offset(cuda0):
    items, queries = _data(6, 64, 2, seed=4)
    v, i = ops.cos_topk_subset(queries.cuda(), items.cuda(), 10, [[0, 1, 2, 3, 4, 5], [5, 2]], row_offset=1000)
    rv, ri = oracle.cos_topk(queries, items, 6)
    assert torch.equal(i[0, :6].cpu(), ri[0] + 1000) and (i[0, 6:] == -1).all()
    assert set(i[1, :2].tolist()) == {1002, 1005} and (i[1, 2:] == -1).all()
    np.testing.assert_allclose(v[0, :6].cpu().numpy(), rv[0].numpy(), rtol=1e-6)
    cat = icr.DeviceCatalog(items, row_offset=1000)
    v2, i2 = cat.topk(queries.cuda(), 10, include_rows=[[0, 1, 2, 3, 4, 5], [5, 2]])
    assert v2.shape == (2, 6)  # k is capped at the catalog's rows, as for every DeviceCatalog call
    assert torch.equal(i2, i[:, :6])


@gpu
@pytest.mark.parametrize("dt", ["f32", "i8"])
def test_skewed_batch_and_long_single_list(cuda0, dt):
    N = 60_000
    cat, _, path = _exact_pair(dt, N=N, D=128, Q=1, seed=9)
    queries = _data(N, 128, 1024, seed=10)[1].cuda()
    rng = np.random.default_rng(5)
    lists = [rng.permutation(N)[:50_000].tolist()] + [rng.choice(N, 10, replace=False).tolist() for _ in range(1023)]
    for k in (10, 256):
        _same(cat.topk(queries, k, include_rows=lists), cat.topk(queries, k, exclude_rows=_complement(lists, N), path=path))
        # Q = 1 with a list far longer than one chunk
        _same(cat.topk(queries[:1], k, include_rows=lists[:1]), cat.topk(queries[:1], k, exclude_rows=_complement(lists[:1], N), path=path))


@gpu
@pytest.mark.parametrize("dt", ["f32", "i8"])
def test_ties_go_to_the_lower_row(cuda0, dt):
    items, queries = _data(1_000, 384, 4, seed=12)
    items[700] = items[30]
    items[900] = items[30]
    items[500] = items[30]
    cat = icr.DeviceCatalog(items, dtype=torch.float32 if dt == "f32" else torch.int8)
    q = items[30:31].repeat(4, 1).cuda()
    lists = [[900, 700, 30, 500, 1, 2], [700, 900], [500, 900, 700], [900]]
    v, i = cat.topk(q, 3, include_rows=lists)
    assert i[0].tolist() == [30, 500, 700] and i[1].tolist()[:2] == [700, 900] and i[2].tolist() == [500, 700, 900]
    path = ops.PATH_GEMM if dt == "f32" else ops.PATH_AUTO
    _same((v, i), cat.topk(q, 3, exclude_rows=_complement(lists, 1_000), path=path))


@gpu
def test_csr_form_and_validation(cuda0):
    items, queries = _data(500, 64, 3, seed=13)
    lists = [[4, 9, 1], [], [499, 0]]
    off = torch.tensor([0, 3, 3, 5], dtype=torch.int64)
    rows = torch.tensor([4, 9, 1, 499, 0], dtype=torch.int64)
    a = ops.cos_topk_subset(queries.cuda(), items.cuda(), 4, lists)
    b = ops.cos_topk_subset(queries.cuda(), items.cuda(), 4, (off.cuda(), rows.cuda()))
    _same(a, b)
    c = ops.cos_topk_subset(queries.cuda(), items.cuda(), 4, [[4, 9, 1, 9, 4], [], [0, 499, 0]])  # Python lists are deduplicated
    _same(a, c)
    with pytest.raises(ValueError, match="distinct"):
        ops.cos_topk_subset(queries.cuda(), items.cuda(), 4, (off.cuda(), torch.tensor([4, 4, 1, 499, 0]).cuda()))
    with pytest.raises(ValueError):
        ops.cos_topk_subset(queries.cuda(), items.cuda(), 4, (torch.tensor([0, 3, 2, 5]).cuda(), rows.cuda()))
    with pytest.raises(ValueError):
        ops.cos_topk_subset(queries.cuda(), items.cuda(), 4, (torch.tensor([1, 3, 3, 5]).cuda(), rows.cuda()))
    with pytest.raises(ValueError):
        ops.cos_topk_subset(queries.cuda(), items.cuda(), 0, lists)
    with pytest.raises(ValueError):
        ops.cos_topk_subset(queries.cuda(), items.cuda(), 257, lists)
    codes, factors = ops.quantize_rows(items.cuda())
    with pytest.raises(ValueError, match="factors"):
        ops.cos_topk_subset(queries.cuda(), codes, 4, lists)


@gpu
def test_request_is_two_launches(cuda0):
    items, queries = _data(3_000, 384, 1, seed=14)
    cat = icr.DeviceCatalog(items)
    cat.topk(queries.cuda(), 10, include_rows=[list(range(0, 3_000, 3))])
    assert ops.last_launch_count() == 2


# ---- DeviceCatalog ---------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16, torch.float16, torch.int8])
def test_device_catalog_after_changes(cuda0, dtype):
    N, D = 2_000, 384
    items, queries = _data(N, D, 6, seed=15)
    cat = icr.DeviceCatalog(items, dtype=dtype)
    exact = dtype in (torch.float32, torch.int8)
    path = ops.PATH_GEMM if dtype == torch.float32 else ops.PATH_AUTO
    q = queries.cuda()

    def check():
        n = len(cat)
        lists = _lists(6, n, seed=n, lo=0, hi=300)
        got = cat.topk(q, 10, include_rows=lists)
        if exact:
            _same(got, cat.topk(q, 10, exclude_rows=_complement(lists, n), path=path))
        else:
            q16 = cat._device_queries(q)
            _check_16(got[0], got[1], q16, cat.rows, 10, lists)

    check()
    new = _data(40, D, 1, seed=16)[0]
    cat.update_rows(list(range(0, 40)), new)
    check()
    cat.append_rows(_data(300, D, 1, seed=17)[0])
    check()
    cat.remove_rows(list(range(100, 400)))
    check()


@gpu
def test_device_catalog_rejects_combinations(cuda0):
    items, queries = _data(300, 64, 2, seed=18)
    cat = icr.DeviceCatalog(items)
    q = queries.cuda()
    with pytest.raises(ValueError):
        cat.topk(q, 5, include_rows=[[1], [2]], exclude_rows=[[3], [4]])
    with pytest.raises(ValueError):
        cat.topk(q, 5, include_rows=[[1], [2]], exclude_mask=torch.zeros(300, dtype=torch.uint8, device="cuda"))
    with pytest.raises(ValueError):
        cat.topk(q, 5, include_rows=[[1], [2]], peer=(0, 1, 0, 0, 0))
    with pytest.raises(ValueError):
        cat.topk(q, 5, include_rows=[[1]])
    with pytest.raises(ValueError):
        cat.topk(q, 257, include_rows=[[1], [2]])


# ---- sharding ----------------------------------------------------------------------------------------------------------------
@gpu
def test_sharded_world_size_one(cuda0):
    items, queries = _data(3_000, 128, 4, seed=19)
    sc = icr.ShardedCatalog.from_full(items)
    lists = _lists(4, 3_000, seed=19, lo=0, hi=500)
    _same(sc.topk(queries, 20, include_rows=lists), icr.DeviceCatalog(items).topk(queries.cuda(), 20, include_rows=lists))


# ---- Recommender -----------------------------------------------------------------------------------------------------------
class _Enc:
    def __init__(self, z):
        self.z = z

    def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True, convert_to_tensor=False):
        tab = {"c": self.z["items"], "q": self.z["queries"]}
        out = np.stack([tab[t.split(":")[0]][int(t.split(":")[1])] for t in texts]).astype(np.float32)
        return torch.from_numpy(out).cuda() if convert_to_tensor else out


def _recommender(golden_dir, tmp_path, dtype, cls=icr.Recommender):
    z = np.load(golden_dir / "embeddings_small.npz")
    pids = [str(p) for p in z["product_ids"]]
    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text(json.dumps({pid: f"c:{i}" for i, pid in enumerate(pids)}))
    return cls("fake-model", corpus, model=_Enc(z), catalog_dtype=dtype), pids, z


def _reference_tail(z, pids, qi, top_k, cands, excl):
    """The reference tail on the oracle's fp32 scores: sort all products, keep the candidates not excluded, take top_k."""
    s = oracle.cos_sim(torch.from_numpy(z["queries"][qi : qi + 1]).float(), torch.from_numpy(z["items"]).float())[0].numpy()
    order = np.lexsort((np.arange(len(pids)), -s.astype(np.float64)))
    keep = set(cands) - set(excl or ())
    return [pids[r] for r in order if pids[r] in keep][:top_k]


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.int8])
def test_recommend_with_candidates(cuda0, golden_dir, tmp_path, dtype):
    rec, pids, z = _recommender(golden_dir, tmp_path, dtype)
    rng = np.random.default_rng(21)
    for qi in range(6):
        cands = rng.choice(pids, size=int(rng.choice([1, 8, 60, 400])), replace=False).tolist()
        excl = set(rng.choice(cands, size=len(cands) // 4, replace=False).tolist())
        got = rec.recommend(f"q:{qi}", top_k=10, exclude_product_ids=excl, candidate_product_ids=cands + ["no-such-id"])
        want = _reference_tail(z, pids, qi, 10, cands, excl)
        if dtype == torch.float32:
            assert [p for p, _ in got] == want
        else:  # 16-bit / int8 rounding may swap near-ties: the same products, scores within the catalog's precision
            assert len(got) == len(want)
            assert len(set(p for p, _ in got) & set(want)) >= len(want) - 2
    assert rec.recommend("q:0", candidate_product_ids=[]) == []
    assert rec.recommend("q:0", candidate_product_ids=["no-such-id"]) == []
    assert rec.recommend("q:0", top_k=7, candidate_product_ids=None) == rec.recommend("q:0", top_k=7)
    with pytest.raises(ValueError):
        rec.recommend("q:0", top_k=257, candidate_product_ids=pids[:3])


@gpu
def test_recommend_batch_mixed_equals_a_loop(cuda0, golden_dir, tmp_path):
    rec, pids, _ = _recommender(golden_dir, tmp_path, torch.float32)
    rng = np.random.default_rng(22)
    queries = [f"q:{q % 10}" for q in range(12)]
    cands = [None if q % 3 == 0 else rng.choice(pids, size=int(rng.choice([0, 5, 200])), replace=False).tolist() for q in range(12)]
    excl = [set(rng.choice(pids, size=20, replace=False).tolist()) if q % 2 else None for q in range(12)]
    got = rec.recommend_batch(queries, top_k=10, exclude_product_ids=excl, candidate_product_ids=cands)
    for q in range(12):
        want = rec.recommend(queries[q], top_k=10, exclude_product_ids=excl[q], candidate_product_ids=cands[q])
        assert [p for p, _ in got[q]] == [p for p, _ in want]
        np.testing.assert_allclose([s for _, s in got[q]], [s for _, s in want], rtol=1e-6)


@gpu
def test_monitored_recommender_sets_metrics(cuda0, golden_dir, tmp_path):
    rec, pids, _ = _recommender(golden_dir, tmp_path, torch.float32, cls=icr.MonitoredRecommender)
    out = rec.recommend("q:1", top_k=5, candidate_product_ids=pids[:50])
    assert rec.last_metrics is not None and rec.last_metrics.num_recommendations == len(out) == 5
    assert {p for p, _ in out} <= set(pids[:50])


# ---- fuzz ----------------------------------------------------------------------------------------------------------------------
def _fuzz_cases(n, seed):
    rng = np.random.default_rng(seed)
    cases = []
    for c in range(n):
        dt = ["f32", "i8", "bf16", "f16"][c % 4]
        cases.append(dict(dt=dt, Q=int(rng.choice([1, 2, 5, 9, 40, 300])), N=int(rng.choice([7, 300, 2_500, 9_000])),
                          D=int(rng.choice([64, 128, 384] if dt == "i8" else [32, 100, 384, 768])) if dt != "f16" and dt != "bf16"
                          else int(rng.choice([64, 384, 776])), k=int(rng.choice([1, 5, 10, 64, 256])),
                          dist=str(rng.choice(["short", "long", "mixed"])), seed=int(rng.integers(1 << 30))))
    return cases


@gpu
@pytest.mark.parametrize("case", _fuzz_cases(int(os.environ.get("ICR_SUBSET_FUZZ_CASES", "24")), 2026))
def test_fuzz_against_the_witness(cuda0, case):
    dt, Q, N, D, k = case["dt"], case["Q"], case["N"], case["D"], case["k"]
    rng = np.random.default_rng(case["seed"])
    items, queries = _data(N, D, Q, seed=case["seed"] % 1000, normalize=bool(case["seed"] & 1))
    dtype = {"f32": torch.float32, "i8": torch.int8, "bf16": torch.bfloat16, "f16": torch.float16}[dt]
    cat = icr.DeviceCatalog(items, dtype=dtype)
    hi = {"short": min(N, 20), "long": N, "mixed": N}[case["dist"]]
    lists = [rng.choice(N + 5, size=int(rng.integers(0, min(N + 5, hi) + 1)), replace=False).tolist() for _ in range(Q)]
    if case["dist"] == "mixed":
        lists = [r[:3] if q % 2 else r for q, r in enumerate(lists)]
    kk = min(k, N)
    got = cat.topk(queries.cuda(), k, include_rows=lists)
    if dt in ("f32", "i8"):
        _same(got, cat.topk(queries.cuda(), k, exclude_rows=_complement(lists, N), path=ops.PATH_GEMM if dt == "f32" else ops.PATH_AUTO))
    else:
        q16 = cat._device_queries(queries)
        _check_16(got[0], got[1], q16, cat.rows, kk, lists)


# ---- rank routing of ShardedCatalog.topk(include_rows=...) with gloo (host stand-ins for the shards) -----------------------
def _free_port() -> int:
    import socket

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _seam_local_topk(queries, rows, k, row_offset, include_rows=None):
    """The shard's subset search on the host: the oracle's scores, only the listed LOCAL rows eligible."""
    s = oracle.cos_sim(queries, rows).double()
    allowed = torch.zeros_like(s, dtype=torch.bool)
    for q, r in enumerate(include_rows):
        r = np.asarray(r, np.int64)
        assert ((r >= 0) & (r < rows.shape[0])).all(), "a rank received an id outside its block"
        allowed[q, torch.from_numpy(r)] = True
    s[~allowed] = float("-inf")
    v, i = torch.topk(s, k, dim=1)
    i = torch.where(torch.isinf(v), torch.full_like(i, -1), i + row_offset)
    return v.float(), i


def _seam_merge(scores, ids, k):
    G, Q, kin = scores.shape
    s = scores.permute(1, 0, 2).reshape(Q, G * kin).double()
    g = ids.permute(1, 0, 2).reshape(Q, G * kin)
    s = torch.where(g < 0, torch.full_like(s, float("-inf")), s)
    out_v, out_i = [], []
    for q in range(Q):
        order = sorted(range(G * kin), key=lambda j: (-s[q, j].item(), g[q, j].item() if g[q, j] >= 0 else 1 << 62))[:k]
        out_v.append(s[q, order].float())
        out_i.append(g[q, order])
    return torch.stack(out_v), torch.stack(out_i)


def _routing_worker(rank: int, world: int, port: int, out_dir: str):
    import sys

    import torch.distributed as dist

    sys.path.insert(0, str(_lib.Path(__file__).resolve().parents[1]))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from instacart_next_order_recommendation_b200.sharded import ShardedCatalog

        n_rows = 301
        full = oracle.synth_clustered(n_rows, 32, seed=31, n_centres=8)[0]
        queries = oracle.synth_isotropic(4, 32, seed=32)
        cat = ShardedCatalog.from_full(full, _local_topk=_seam_local_topk, _merge=_seam_merge)
        lists = [[0, 300, 150, 151, 149, 7], [], [299, 298, -3, 5_000], list(range(140, 170))]
        v, i = cat.topk(queries, 5, include_rows=lists)
        local = cat._local_lists(lists)
        lo, hi = cat.row_offset, cat.row_offset + cat.n_local
        for g, l in zip(lists, local):
            want = sorted(x - lo for x in set(g) if lo <= x < hi)
            assert sorted(np.asarray(l).tolist()) == want
        off, rows = cat._local_lists((torch.tensor([0, 6, 6, 10, 40]), torch.tensor([x for r in lists for x in r])))
        for q in range(4):
            assert sorted(rows[off[q] : off[q + 1]].tolist()) == sorted(np.asarray(local[q]).tolist())
        torch.save({"v": v, "i": i}, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_sharded_rank_routing_with_gloo(tmp_path):
    import torch.multiprocessing as mp

    mp.spawn(_routing_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    a, b = torch.load(tmp_path / "r0.pt"), torch.load(tmp_path / "r1.pt")
    assert torch.equal(a["i"], b["i"]) and torch.equal(a["v"], b["v"])
    full = oracle.synth_clustered(301, 32, seed=31, n_centres=8)[0]
    queries = oracle.synth_isotropic(4, 32, seed=32)
    lists = [[0, 300, 150, 151, 149, 7], [], [299, 298], list(range(140, 170))]
    want, ref_i = _seam_local_topk(queries, full, 5, 0, include_rows=lists)
    got_i = a["i"]
    assert (got_i[1] == -1).all()
    assert (got_i[2, 2:] == -1).all() and set(got_i[2, :2].tolist()) == {298, 299}
    assert torch.equal(got_i, ref_i)
    torch.testing.assert_close(a["v"], want)
