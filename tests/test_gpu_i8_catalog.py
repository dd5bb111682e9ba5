"""int8 catalogs in the fused top-k, from the quantiser to DeviceCatalog and Recommender.

Contract: rows and queries are quantised per row (I8Rows in csrc/common.cuh): m = max|x|, codes
clamp(rint(127 * (x / m)), -127, 127) in fp32 with round-to-nearest, factor (m / 127) / max(|x|, 1e-12). Row r is ranked
for query q by key = fp32(S) * f_r, S the exact integer dot product of the codes, ties to the lower row; the returned score
is key * f_q. That is deterministic, so the kernels must equal the restatement below BIT FOR BIT (ids and score bits), fed
with the device's own codes and factors. The restatement's codes are numpy float32 arithmetic; its dot products are exact
(fp64 sums of integer products below 2^53).

Tests without the gpu mark check the C ABI's int8 surface and the restatement itself on the host.
"""

import json
import re
import zlib
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from instacart_next_order_recommendation_b200 import _lib
from oracle import oracle

gpu = pytest.mark.gpu


# ---- the restatement ----------------------------------------------------------------------------------------------------------
def quantize_ref(x):
    """numpy float32 restatement of icr_quantize_rows: (codes int8 [rows, D], factors float64 [rows]). The codes are bit
    exact; the factor is computed in float64 (the device's fp32 one is within a few ulp of it)."""
    x = np.asarray(x, dtype=np.float32)
    m = np.abs(x).max(axis=1)
    safe = np.where(m > 0, m, np.float32(1)).astype(np.float32)
    with np.errstate(invalid="ignore", divide="ignore"):
        c = np.clip(np.rint(np.float32(127) * (x / safe[:, None])), -127, 127).astype(np.int8)
    c[m == 0] = 0
    n = np.sqrt((x.astype(np.float64) ** 2).sum(axis=1))
    f = np.where(m > 0, (m.astype(np.float64) / 127.0) / np.maximum(n, 1e-12), 0.0)
    return c, f


def topk_ref(qc, qf, cc, cf, k, excl=None):
    """(scores f32 [Q, k], ids [Q, k]) of the int8 contract for query codes / factors qc, qf and catalog codes / factors
    cc, cf (device tensors; codes int8, factors float32). excl: bool [Q, N] or None. Keys fp32(S) * f_r, ranked by key
    then lower row; score = key * f_q; (-inf, -1) tail when fewer than k rows are eligible."""
    Q, N = qc.shape[0], cc.shape[0]
    cd = cc.double()
    vals, ids = [], []
    for q0 in range(0, Q, 128):
        S = qc[q0 : q0 + 128].double() @ cd.T  # exact: |S| <= 4096 * 127^2 < 2^53
        key = S.float() * cf[None, :]  # fp64 -> fp32 of an integer rounds as __int2float_rn does
        if excl is not None:
            key[excl[q0 : q0 + 128]] = float("-inf")
        if N < k:
            key = torch.cat([key, torch.full((key.shape[0], k - N), float("-inf"), device=key.device)], dim=1)
        order = torch.sort(key, dim=1, descending=True, stable=True).indices[:, :k]  # stable: lower row first among ties
        kv = key.gather(1, order)
        live = torch.isfinite(kv)
        vals.append(torch.where(live, kv * qf[q0 : q0 + 128, None], kv))
        ids.append(torch.where(live, order, torch.full_like(order, -1)))
    return torch.cat(vals), torch.cat(ids)


def _assert_exact(v, i, rv, ri, offset=0):
    i = torch.where(i >= 0, i - offset, i)
    assert torch.equal(i, ri), f"ids differ at {int((i != ri).sum())} positions"
    assert torch.equal(v.view(torch.int32), rv.view(torch.int32)), "score bits differ"


# ---- host-only checks -----------------------------------------------------------------------------------------------------------
def test_header_value_and_symbol_are_mirrored():
    header = (Path(__file__).resolve().parents[1] / "include" / "icr_b200.h").read_text()
    assert re.search(r"\bICR_I8\s*=\s*3\b", header) and _lib.ICR_I8 == 3
    assert "icr_quantize_rows" in _lib.SIGNATURES and re.search(r"\bint icr_quantize_rows\(", header)
    lib = _lib.load()
    assert hasattr(lib, "icr_quantize_rows")


def test_int8_is_rejected_by_the_dense_and_mnrl_entries_before_any_cuda_call():
    lib = _lib.load()
    p = 1 << 20  # never dereferenced: the dtype check comes first
    assert lib.icr_cos_sim_dense(p, 4, 64, p, 4, 64, 64, 3, p, 4, p, 1 << 16, None) == -2
    assert lib.icr_row_inv_norms(p, 4, 64, 64, 3, p, None) == -2
    assert lib.icr_mnrl_fwd(p, 64, p, 64, 4, 64, 3, 20.0, p, p, p, p, p, 1 << 20, None) == -2
    assert lib.icr_mnrl_fwd_bwd(p, 64, p, 64, 4, 64, 3, 20.0, p, p, p, p, p, 64, p, 64, p, 1 << 20, None) == -2
    assert lib.icr_convert_rows(p, 4, 64, 64, p, 64, 3, 0, None) == -2
    # an int8 top-k call without its factors is an argument error, also before any CUDA call
    assert lib.icr_cos_topk(p, 1, 64, p, 10, 64, 64, 3, None, None, None, 5, 0, 0, p, p, p, 1 << 20, None) == -1
    assert b"factors" in lib.icr_last_error_string()


def test_restatement_known_answers():
    x = np.array([[1.0, -0.5, 0.25, 0.0], [0.0, 0.0, 0.0, 0.0], [0.0, 3.0, 0.0, 0.0], [2.0, 2.0, 2.0, 2.0]], dtype=np.float32)
    c, f = quantize_ref(x)
    # 127 * 0.25 = 31.75 -> 32; 127 * -0.5 = -63.5 -> -64 (half to even)
    assert c.tolist() == [[127, -64, 32, 0], [0, 0, 0, 0], [0, 127, 0, 0], [127, 127, 127, 127]]
    assert f[1] == 0.0 and abs(f[2] - 3.0 / 127 / 3.0) < 1e-15 and abs(f[3] - 2.0 / 127 / 4.0) < 1e-15
    assert abs(f[0] - (1.0 / 127) / np.sqrt(1 + 0.25 + 0.0625)) < 1e-15
    # keys and ties on the host (the restatement runs on whichever device its inputs are on)
    qc = torch.tensor([[127, 0, 0, 0]], dtype=torch.int8)
    cc = torch.tensor([[127, 0, 0, 0], [0, 127, 0, 0], [127, 0, 0, 0], [-127, 0, 0, 0]], dtype=torch.int8)
    cf = torch.tensor([0.5, 1.0, 0.5, 0.25])
    v, i = topk_ref(qc, torch.tensor([2.0]), cc, cf, 3)
    assert i.tolist() == [[0, 2, 1]]  # key 8064.5 twice (lower row first), then 0
    assert v.tolist() == [[16129.0, 16129.0, 0.0]]
    v, i = topk_ref(qc, torch.tensor([2.0]), cc, cf, 6, excl=torch.tensor([[True, False, False, False]]))
    assert i.tolist() == [[2, 1, 3, -1, -1, -1]] and v[0, 3:].isinf().all()


# ---- GPU ----------------------------------------------------------------------------------------------------------------------------
def _icr():
    import instacart_next_order_recommendation_b200 as icr

    return icr


@pytest.fixture(scope="module")
def cuda0():
    assert torch.cuda.is_available(), "run with -m gpu on a GPU box"
    torch.cuda.set_device(0)
    assert _lib.load().icr_device_supported() == 1
    yield
    torch.cuda.synchronize()


def _ref_for(cat, queries, k, excl=None):
    from instacart_next_order_recommendation_b200 import ops

    qc, qf = ops.quantize_rows(queries.cuda().float())
    return topk_ref(qc[:, : cat.rows.shape[1]], qf, cat.rows, cat.inv_norms, k, excl)


def _excl_matrix(lists, Q, N, mask=None):
    ex = torch.zeros(Q, N, dtype=torch.bool, device="cuda")
    for q, l in enumerate(lists or []):
        l = [r for r in l if 0 <= r < N]
        if l:
            ex[q, torch.as_tensor(l, device="cuda")] = True
    if mask is not None:
        ex |= mask.bool().cuda()[None, :]
    return ex


def _data(N, D, Q, seed):
    items, _ = oracle.synth_clustered(N, D, seed=seed)
    queries, _ = oracle.synth_queries_from_items(items, Q, seed=seed + 1)
    return items.cuda(), queries.cuda()


@gpu
@pytest.mark.parametrize("D", [16, 48, 384, 768, 1000, 4096])
def test_quantizer_matches_the_restatement(cuda0, D):
    from instacart_next_order_recommendation_b200 import ops

    rng = np.random.default_rng(D)
    x = rng.standard_normal((300, D)).astype(np.float32)
    x *= (10.0 ** rng.uniform(-3, 3, size=(300, 1))).astype(np.float32)  # scales 1e-3 .. 1e3
    x[::37] = 0.0  # exact-zero rows
    x[5::41] = 0.0
    x[5::41, D // 3] = -2.5  # a single non-zero element
    x[7, :] = 0.5  # every element at the maximum
    codes, factors = ops.quantize_rows(torch.from_numpy(x).cuda())
    rc, rf = quantize_ref(x)
    Dp = (D + 15) // 16 * 16
    assert codes.shape == (300, Dp) and codes.dtype == torch.int8
    assert np.array_equal(codes[:, :D].cpu().numpy(), rc)
    assert (codes[:, D:] == 0).all()  # padding columns
    f = factors.cpu().numpy().astype(np.float64)
    assert (f[rf == 0] == 0).all()
    ulp = np.spacing(np.abs(rf).astype(np.float32)).astype(np.float64)
    assert (np.abs(f - rf) <= 4 * ulp).all(), float(np.max(np.abs(f - rf) / np.maximum(ulp, 1e-45)))


# name -> (N, Q, D, k, path, launches): the plan branches of tests/test_gpu_f16_catalog.py. An int8 call is planned as an
# fp16 call of the same shape and takes as many launches; the tensor-core branches run MODE 5 (kind::i8).
BRANCHES = {
    "gemv_q1_k10": (49_688, 1, 384, 10, 0, 1),
    "gemv_q1_k100": (49_688, 1, 384, 100, 1, 1),
    "gemv_q2_k16": (49_688, 2, 384, 16, 1, 1),
    "gemv_q3_k100": (49_688, 3, 384, 100, 1, 1),
    "gemv_q7_k10": (49_688, 7, 384, 10, 1, 1),
    "gemv_q7_k100": (49_688, 7, 384, 100, 1, 1),
    "swap_tail_q8_k10": (49_688, 8, 384, 10, 2, 2),
    "swap_tail_q16_k100": (49_688, 16, 384, 100, 2, 2),
    "swap_tail_q64_k100": (49_688, 64, 384, 100, 2, 2),
    "swap_select_q256": (49_688, 256, 384, 100, 2, 3),
    "swap_phased": (3_000, 16, 384, 256, 2, 5),
    "k2_single": (49_688, 1000, 384, 100, 0, 3),
    "k2_coarse": (600_000, 200, 384, 100, 0, 3),
    "k2_phased_q300": (5_000, 300, 384, 100, 2, 5),
    "k2_phased_q600": (5_000, 600, 384, 100, 2, 5),
    "swap_short_rows_d128": (2_600_000, 1, 128, 10, 0, 3),
}


def _branch_data(name, N, Q, D):
    seed = zlib.crc32(name.encode()) % 1000
    if N >= 500_000:
        g = torch.Generator(device="cuda").manual_seed(seed)
        items = F.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
        items[::1009] = items[7]
        queries = F.normalize(items[torch.arange(Q, device="cuda") * (N // Q - 1)] + 0.3 * torch.randn(Q, D, device="cuda", generator=g), dim=1)
        return items, queries
    return _data(N, D, Q, seed)


@gpu
@pytest.mark.parametrize("variant", ["plain", "excl", "excl_mask"])
@pytest.mark.parametrize("name", list(BRANCHES))
def test_every_plan_branch(cuda0, name, variant):
    from instacart_next_order_recommendation_b200 import ops

    icr = _icr()
    N, Q, D, k, path, launches = BRANCHES[name]
    items, queries = _branch_data(name, N, Q, D)
    cat = icr.DeviceCatalog(items, dtype=torch.int8)
    lists, mask = None, None
    if variant != "plain":
        rng = np.random.default_rng(zlib.crc32(name.encode()) % 997)
        _, best = _ref_for(cat, queries, min(N, 2 * k))
        best = best.cpu().tolist()
        lists = [best[q][: (0, k // 2, 2 * k)[q % 3]] + rng.choice(N, 16, replace=False).tolist() for q in range(Q)]
    if variant == "excl_mask":
        mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
        mask[torch.as_tensor(np.random.default_rng(3).choice(N, N // 50, replace=False), device="cuda")] = 1
    v, i = cat.topk(queries, k, exclude_rows=lists, exclude_mask=mask, path=path)
    n8 = ops.last_launch_count()
    cat16 = icr.DeviceCatalog(items, dtype=torch.float16)
    cat16.topk(queries, k, exclude_rows=lists, exclude_mask=mask, path=path)
    assert n8 == ops.last_launch_count() == launches, f"{name}: {n8} launches on int8, expected {launches} as on fp16"
    ex = _excl_matrix(lists, Q, N, mask) if (lists is not None or mask is not None) else None
    rv, ri = _ref_for(cat, queries, k, ex)
    _assert_exact(v, i, rv, ri)


@gpu
def test_ring_and_direct_kernels_agree_bitwise(cuda0):
    """The bulk-copy ring kernel (contiguous codes) and the direct-load kernel (row-strided codes) return the same bits."""
    from instacart_next_order_recommendation_b200 import ops

    N, D = 30_011, 384
    items, queries = _data(N, D, 7, 41)
    codes, factors = ops.quantize_rows(items)
    wide = torch.zeros(N, D + 64, dtype=torch.int8, device="cuda")
    wide[:, :D] = codes
    strided = wide[:, :D]
    for Q, k in ((1, 10), (3, 100), (7, 40), (1, 256)):
        v1, i1 = ops.cos_topk(queries[:Q], codes, k, cat_inv_norms=factors, path=ops.PATH_GEMV)
        assert ops.last_launch_count() == 1
        v2, i2 = ops.cos_topk(queries[:Q], strided, k, cat_inv_norms=factors, path=ops.PATH_GEMV)
        assert ops.last_launch_count() == 1
        assert torch.equal(i1, i2) and torch.equal(v1.view(torch.int32), v2.view(torch.int32))
        qc, qf = ops.quantize_rows(queries[:Q])
        _assert_exact(v1, i1, *topk_ref(qc, qf, codes, factors, k))
    with pytest.raises(ValueError, match="factors"):
        ops.cos_topk(queries[:1], codes, 10)


@gpu
@pytest.mark.parametrize("Q", [1, 3, 7])
@pytest.mark.parametrize("k", [10, 100])
def test_gemv_and_tensor_core_paths_agree_bitwise(cuda0, Q, k):
    from instacart_next_order_recommendation_b200 import ops

    items, queries = _data(49_688, 384, Q, 300 + Q)
    codes, factors = ops.quantize_rows(items)
    v1, i1 = ops.cos_topk(queries, codes, k, cat_inv_norms=factors, path=ops.PATH_GEMV)
    v2, i2 = ops.cos_topk(queries, codes, k, cat_inv_norms=factors, path=ops.PATH_GEMM)
    assert torch.equal(i1, i2) and torch.equal(v1.view(torch.int32), v2.view(torch.int32))
    qc, qf = ops.quantize_rows(queries)
    _assert_exact(v1, i1, *topk_ref(qc, qf, codes, factors, k))


@gpu
@pytest.mark.parametrize("Q", [64, 256])
@pytest.mark.parametrize("D", [384, 768, 1024])
def test_swapped_and_queries_on_m_kernels_agree_bitwise(cuda0, Q, D):
    """K2s (Q <= 256, queries resident) and K2 (the same queries as the first rows of a 300-query batch) give the same bits.
    D = 1024 takes the A-streaming K2 variant (more than 6 K blocks of 128 codes)."""
    from instacart_next_order_recommendation_b200 import ops

    items, queries = _data(20_011, D, 300, 500 + Q)
    codes, factors = ops.quantize_rows(items)
    vs, is_ = ops.cos_topk(queries[:Q], codes, 100, cat_inv_norms=factors, path=ops.PATH_GEMM)
    vk, ik = ops.cos_topk(queries, codes, 100, cat_inv_norms=factors, path=ops.PATH_GEMM)
    assert torch.equal(is_, ik[:Q]) and torch.equal(vs.view(torch.int32), vk[:Q].view(torch.int32))
    qc, qf = ops.quantize_rows(queries)
    _assert_exact(vk, ik, *topk_ref(qc, qf, codes, factors, 100))


@gpu
@pytest.mark.parametrize("D", [16, 1040, 2048, 4096])
def test_dims_including_rounded_dot_products(cuda0, D):
    """D >= 2048 lets |S| pass 2^24, where fp32(S) rounds - the same way on every path."""
    icr = _icr()
    N = 5_003
    items = torch.ones(N, D, device="cuda") + 0.01 * torch.randn(N, D, device="cuda")  # near-maximal codes: |S| up to D * 127^2
    items[1::2] = torch.randn(N // 2, D, device="cuda")
    queries = torch.ones(5, D, device="cuda")
    queries[1:] = torch.randn(4, D, device="cuda")
    cat = icr.DeviceCatalog(items, dtype=torch.int8)
    from instacart_next_order_recommendation_b200 import ops

    for Q in (1, 3, 5):
        for path in (ops.PATH_GEMV, ops.PATH_GEMM):
            v, i = cat.topk(queries[:Q], 50, path=path)
            _assert_exact(v, i, *_ref_for(cat, queries[:Q], 50))


@gpu
def test_edges(cuda0):
    icr = _icr()
    from instacart_next_order_recommendation_b200 import ops

    # fewer rows than k, and ragged N
    for N in (7, 100, 777, 20_001):
        items, queries = _data(N, 72 if N == 777 else 64, 3, N)
        cat = icr.DeviceCatalog(items, dtype=torch.int8)
        for Q, k in ((1, 10), (3, 256)):
            for path in (ops.PATH_GEMV, ops.PATH_GEMM):
                v, i = cat.topk(queries[:Q], k, path=path)
                _assert_exact(v, i, *_ref_for(cat, queries[:Q], min(k, N)))
    # every row excluded for some queries
    items, queries = _data(500, 384, 5, 9)
    cat = icr.DeviceCatalog(items, dtype=torch.int8)
    lists = [list(range(500)) if q % 2 == 0 else [1, 2, 3] for q in range(5)]
    for path in (ops.PATH_GEMV, ops.PATH_GEMM):
        v, i = cat.topk(queries, 20, exclude_rows=lists, path=path)
        _assert_exact(v, i, *_ref_for(cat, queries, 20, _excl_matrix(lists, 5, 500)))
        assert (i[0] == -1).all() and torch.isinf(v[0]).all()
    # duplicate rows: ties go to the lower row
    items, queries = _data(3_000, 384, 3, 11)
    items[100:200] = items[5]
    items[2_999] = items[5]
    cat = icr.DeviceCatalog(items, dtype=torch.int8)
    q = items[5:6].repeat(8, 1)
    for path in (ops.PATH_GEMV, ops.PATH_GEMM):
        v, i = cat.topk(q, 50, path=path)
        _assert_exact(v, i, *_ref_for(cat, q, 50))
        assert i[:, :3].tolist() == [[5, 100, 101]] * 8
        # a zero query scores 0 everywhere: ids 0 .. k-1
        v, i = cat.topk(torch.zeros(8, 384, device="cuda"), 10, path=path)
        assert i.tolist() == [list(range(10))] * 8 and (v == 0).all()
    # non-finite rows are refused
    bad = items[:10].clone()
    bad[3, 7] = float("nan")
    with pytest.raises(ValueError, match="finite"):
        icr.DeviceCatalog(bad, dtype=torch.int8)
    assert ops.quantize_rows(torch.zeros(0, 384, device="cuda"))[0].shape == (0, 384)


_N_FUZZ = 60


def _fuzz_cases(n, seed=20261022):
    rng = np.random.default_rng(seed)
    return [(c, int(rng.choice([1, 2, 3, 5, 7, 8, 33, 130, 300])), int(rng.choice([7, 100, 1000, 4097, 20_000, 49_688])),
             int(rng.choice([16, 64, 128, 208, 384, 768])), int(rng.choice([1, 5, 10, 37, 100, 256])),
             float(rng.choice([0.0, 0.0, 1e-3, 0.01, 0.2, 0.9])), int(rng.choice([0, 1, 2]))) for c in range(n)]


@gpu
@pytest.mark.parametrize("case", _fuzz_cases(_N_FUZZ), ids=lambda c: f"{c[0]}-Q{c[1]}-N{c[2]}-D{c[3]}-k{c[4]}-x{c[5]}-p{c[6]}")
def test_fuzz(cuda0, case):
    icr = _icr()
    c, Q, N, D, k, density, path = case
    if path == 1 and Q > 64:
        path = 0
    it = oracle.synth_unnormalised(N, D, seed=3000 + c).cuda()
    qt = oracle.synth_unnormalised(Q, D, seed=4000 + c).cuda()
    rng = np.random.default_rng(5000 + c)
    lists = [np.nonzero(rng.random(N) < density)[0].tolist() for _ in range(Q)] if density > 0 else None
    kk = min(k, N)
    cat = icr.DeviceCatalog(it, dtype=torch.int8, row_offset=3)
    v, i = cat.topk(qt if c % 2 else qt.half(), kk, exclude_rows=lists, path=path)
    _assert_exact(v, i, *_ref_for(cat, qt if c % 2 else qt.half().float(), kk, _excl_matrix(lists, Q, N) if lists else None), offset=3)


@gpu
def test_device_catalog_from_index_and_request_paths(cuda0, tmp_path):
    from instacart_next_order_recommendation_b200.index import EmbeddingIndex

    icr = _icr()
    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text("{}")
    n, d = 5_003, 384
    ids = [str(i) for i in range(n)]
    emb = oracle.synth_unnormalised(n, d, seed=3).numpy()
    idx = EmbeddingIndex(corpus, "fake-model")
    idx.save(ids, emb)
    cat = icr.DeviceCatalog(torch.from_numpy(emb), dtype=torch.int8)
    assert cat.dtype == torch.int8 and cat.planes is None and cat.query_dtype == torch.float32
    assert cat.nbytes == n * d + 4 * n
    idx.save_bf16_sidecar()  # never read for int8
    for chunk_rows in (1 << 17, 1000, 37):
        fc = icr.DeviceCatalog.from_index(idx, ids, dtype=torch.int8, chunk_rows=chunk_rows)
        assert torch.equal(fc.rows, cat.rows) and torch.equal(fc.inv_norms.view(torch.int32), cat.inv_norms.view(torch.int32))
    part = icr.DeviceCatalog.from_index(idx, ids, dtype=torch.int8, rows=(1200, 3100))
    assert torch.equal(part.rows, cat.rows[1200:3100]) and part.row_offset == 1200
    with pytest.raises(ValueError, match="normalize"):
        icr.DeviceCatalog.from_index(idx, ids, dtype=torch.int8, normalize=True)
    bad = emb.copy()
    bad[17, 3] = np.inf
    idx.save(ids, bad)
    with pytest.raises(ValueError, match="finite"):
        icr.DeviceCatalog.from_index(idx, ids, dtype=torch.int8)
    # the request paths agree with topk: graph (host / device fp32 queries), prepared call, pinned-output request
    from instacart_next_order_recommendation_b200 import ops

    q32 = F.normalize(oracle.synth_unnormalised(7, d, seed=11).cuda(), dim=1)
    cat16 = icr.DeviceCatalog(torch.from_numpy(emb), dtype=torch.float16)
    for Q in (1, 3, 7):
        for k in (10, 100):
            v, i = cat.topk(q32[:Q], k)
            _assert_exact(v, i, *_ref_for(cat, q32[:Q], k))
            for src in (q32[:Q].cpu(), q32[:Q].cpu().numpy(), q32[:Q]):
                vs, is_ = cat.topk_small(src, k)
                assert torch.equal(vs, v) and torch.equal(is_, i)
            vs, is_ = cat.topk_small(q32[:Q].half().cpu(), k)  # other dtypes are up-cast
            _assert_exact(vs.cuda(), is_.cuda(), *_ref_for(cat, q32[:Q].half().float(), k))
            cat.topk_small(q32[:Q], k)  # the prepared call: as many launches as fp16's on the same call
            n8 = ops.last_launch_count()
            cat16.topk_small(q32[:Q].half(), k)
            assert n8 == ops.last_launch_count()
            sv, si = cat.topk_request(q32[:Q], k)
            assert ops.last_launch_count() == n8
            assert si == i.tolist() and np.array_equal(np.asarray(sv, dtype=np.float32), v.cpu().numpy())
            vh, ih = cat.topk_host(q32[:Q].cpu(), k)
            torch.cuda.synchronize()
            assert torch.equal(vh, v.cpu()) and torch.equal(ih, i.cpu())


class _DeviceEnc:
    def __init__(self, z):
        self.z = z

    def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True, convert_to_tensor=False):
        tab = {"c": self.z["items"], "q": self.z["queries"]}
        out = np.stack([tab[t.split(":")[0]][int(t.split(":")[1])] for t in texts]).astype(np.float32)
        return torch.from_numpy(out).cuda() if convert_to_tensor else out


class _HostEnc(_DeviceEnc):
    def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True):
        return _DeviceEnc.encode(self, texts)


@gpu
@pytest.mark.parametrize("env", ["int8", "i8"])
@pytest.mark.parametrize("enc", [_DeviceEnc, _HostEnc])
def test_recommender_int8(cuda0, golden_dir, tmp_path, monkeypatch, enc, env):
    icr = _icr()
    z = np.load(golden_dir / "embeddings_small.npz")
    pids = [str(p) for p in z["product_ids"]]
    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text(json.dumps({pid: f"c:{i}" for i, pid in enumerate(pids)}))
    monkeypatch.setenv("ICR_CATALOG_DTYPE", env)
    rec = icr.Recommender("fake-model", corpus, model=enc(z), use_index=False)
    assert rec.catalog.dtype == torch.int8
    gold = json.loads((golden_dir / "recommend_golden.json").read_text())
    rng = np.random.default_rng(4)
    cases = [(c["q"], c["top_k"], set(c["exclude"])) for c in gold["cases"]]
    cases += [(q % len(z["queries"]), 10, set(rng.choice(pids, 300, replace=False).tolist())) for q in range(3)]
    n = len(pids)

    def want(q, top_k, excl):
        # the restated tail: every row ranked by the int8 key, excluded ones dropped, the first top_k kept
        v, i = _ref_for(rec.catalog, torch.from_numpy(z["queries"][q : q + 1]), n)
        out = [(pids[r], float(s)) for s, r in zip(v[0].tolist(), i[0].tolist()) if pids[r] not in excl]
        return out[:top_k]

    for q, top_k, excl in cases:
        w = want(q, top_k, excl)
        got = rec.recommend(f"q:{q}", top_k=top_k, exclude_product_ids=excl)
        assert got == w
        assert rec.recommend_batch([f"q:{q}"], top_k=top_k, exclude_product_ids=[excl])[0] == w
    batch = rec.recommend_batch([f"q:{q}" for q, _, _ in cases], top_k=10, exclude_product_ids=[e for _, _, e in cases])
    for b, (q, _, e) in zip(batch, cases):
        assert b == want(q, 10, e)
    mon = icr.MonitoredRecommender("fake-model", corpus, model=enc(z), use_index=False, catalog_dtype=torch.int8)
    q, top_k, excl = cases[0]
    assert mon.recommend(f"q:{q}", top_k=top_k, exclude_product_ids=excl) == want(q, top_k, excl)


@gpu
def test_recall_against_fp32_exact(cuda0):
    """SQ8's usual trade, known before the run from the restatement: mean recall@10 >= 0.95 on both synthetic sets."""
    icr = _icr()
    N, D, Q = 49_688, 384, 256
    sets = {"clustered": _data(N, D, Q, 1234),
            "isotropic": (oracle.synth_isotropic(N, D, seed=7).cuda(), oracle.synth_isotropic(Q, D, seed=8).cuda())}
    for name, (items, queries) in sets.items():
        exact = torch.topk(F.normalize(queries.double(), dim=1) @ F.normalize(items.double(), dim=1).T, 10, dim=1).indices
        _, i = icr.DeviceCatalog(items, dtype=torch.int8).topk(queries, 10)
        rec = float(np.mean([len(set(a) & set(b)) / 10 for a, b in zip(i.cpu().tolist(), exact.cpu().tolist())]))
        print(f"\nint8 recall@10 against fp32 exact, {name}: {rec:.4f}")
        assert rec >= 0.95, (name, rec)


@gpu
def test_sharded_catalog_int8_world_size_1(cuda0):
    icr = _icr()
    items, queries = _data(30_011, 384, 9, 71)
    sh = icr.ShardedCatalog(items, row_offset=0, total_rows=30_011, dtype=torch.int8)
    assert sh.local.dtype == torch.int8
    for Q, k in ((1, 10), (9, 100)):
        v, i = sh.topk(queries[:Q], k)
        _assert_exact(v, i, *_ref_for(sh.local, queries[:Q], k))


@gpu
def test_sharded_catalog_int8_two_gpus(cuda0):
    import os
    import subprocess
    import sys

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one machine")
    root = Path(__file__).resolve().parents[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29524",
           str(root / "benchmarks" / "i8_sharded_case.py")]
    out = subprocess.run(cmd, cwd=str(root), capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert out.returncode == 0, out.stderr[-2000:]
    assert "I8_SHARDED_OK" in out.stdout, out.stdout[-2000:]
