"""fp16 catalogs in the fused top-k and the dense cos_sim, from the kernels to DeviceCatalog and Recommender (B200 only).

Precision contract: s_ref is fp64 arithmetic on the fp16 values the kernels consumed (the catalog rows and the converted
queries). fp16 x fp16 products are exact in fp32, so every returned score is within 1e-5 * max(|s_ref|, 0.05) of s_ref;
ids equal the reference's except where neighbouring reference scores are closer than that, and the k-th score is not
below the reference's k-th by more than it. Any bf16 rounding on the way would cost up to 6.8e-4 and fail these bounds.

For D >= 2048 the tensor cores' fp32 accumulation over K = D terms adds to that: 2e-6 absolute, plus (D / 16) * 2^-23
relative to |s_ref| - one fp32 ulp per K = 16 MMA step, which is what a score near 1 drifts by when every product has the
same sign (measured on a B200: 2.2e-5 relative at D = 4096 for scores of 0.98, 1.1e-5 at D = 2048).
"""

import json
import os
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import instacart_next_order_recommendation_b200 as icr
from instacart_next_order_recommendation_b200 import ops
from oracle import oracle

pytestmark = pytest.mark.gpu

RTOL = 1e-5
MAX_ERR: dict = {}  # path -> largest |s - s_ref| / max(|s_ref|, 0.05) seen, printed at the end of the module


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert torch.cuda.is_available(), "run with -m gpu on a GPU box"
    torch.cuda.set_device(0)
    assert icr._lib.load().icr_device_supported() == 1
    yield
    torch.cuda.synchronize()
    print("\nlargest fp16-catalog score error per path (|s - s_ref| / max(|s_ref|, 0.05)):")
    for name, e in sorted(MAX_ERR.items()):
        print(f"  {name:28s} {e:.3e}")


def _tol(s, D):
    """The contract's allowance for scores s (a tensor of reference scores) at embedding dim D."""
    t = RTOL * s.abs().clamp(min=0.05)
    return t + (2e-6 + (D / 16) * 2.0**-23 * s.abs()) if D >= 2048 else t


def _record(name, err):
    MAX_ERR[name] = max(MAX_ERR.get(name, 0.0), float(err))


def _s_ref(q16, c16):
    """fp64 cosine of the fp16 values [Q, N] on the device (F.normalize's eps: zero rows score 0)."""
    return F.normalize(q16.cuda().double(), dim=1) @ F.normalize(c16.cuda().double(), dim=1).T


def _check_topk(v, i, q16, c16, k, excl=None, name="topk", offset=0):
    """The contract for one call: v, i [Q, k] against fp64 on the fp16 inputs, with the excluded (q, row) pairs out.
    excl: bool [Q, N] (device) or None."""
    Q, N = q16.shape[0], c16.shape[0]
    D = q16.shape[1]
    v, i = v.cuda().double(), i.cuda()
    i = torch.where(i >= 0, i - offset, i)
    assert v.shape == (Q, k) and i.shape == (Q, k)
    assert not torch.isnan(v).any(), "NaN score"
    assert (v[:, :-1] >= v[:, 1:]).all(), "scores must be non-increasing"
    for q0 in range(0, Q, 256):
        s = _s_ref(q16[q0 : q0 + 256], c16)
        if excl is not None:
            s[excl[q0 : q0 + 256]] = float("-inf")
        if N < k:
            s = torch.cat([s, torch.full((s.shape[0], k - N), float("-inf"), dtype=s.dtype, device=s.device)], dim=1)
        rv = torch.topk(s, k, dim=1).values
        vb, ib = v[q0 : q0 + 256], i[q0 : q0 + 256]
        live = torch.isfinite(rv)
        assert torch.equal(torch.isfinite(vb), live), "eligible-row count differs from the reference"
        assert (ib[~live] == -1).all(), "the tail of a short list must be (-inf, -1)"
        sv = s.gather(1, ib.clamp(min=0))
        assert torch.isfinite(sv[live]).all(), "an excluded row was returned"
        tol_v = _tol(sv, D)
        err = ((vb - sv).abs() / sv.abs().clamp(min=0.05))[live]
        assert ((vb - sv).abs() <= tol_v)[live].all(), f"max score error {float(err.max()):.3e}"
        # position by position the returned row's reference score equals the reference's: ids differ only where two
        # reference scores are closer than the tolerance (each side may be off by one tolerance)
        tol_r = _tol(rv.masked_fill(~live, 0.0), D)
        assert ((sv - rv).abs() <= 2 * tol_r + 1e-12)[live].all(), "an id differs from the reference outside near-ties"
        assert (vb[:, -1] >= rv[:, -1] - tol_r[:, -1])[live[:, -1]].all(), "k-th returned score below the reference's k-th"
        for r in range(ib.shape[0]):
            got = ib[r][live[r]].tolist()
            assert len(set(got)) == len(got), "duplicate ids"
        if err.numel():
            _record(name, err.max())


def _excl_matrix(lists, Q, N, mask=None):
    ex = torch.zeros(Q, N, dtype=torch.bool, device="cuda")
    if lists is not None:
        for q, l in enumerate(lists):
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


def _own_best(q16, c16, n):
    return torch.topk(_s_ref(q16, c16), n, dim=1).indices.cpu().tolist()


# ---- every plan branch ------------------------------------------------------------------------------------------------------
# name -> (N, Q, D, k, path, launches of the call on a 16-bit catalog). The tensor-core shapes are those of
# tests/test_gpu_screening_band.py; on a 16-bit catalog they take the same branches (the plan looks at the row bytes only
# through D and the catalog size), with one launch fewer wherever fp32 re-scores its screened candidates.
BRANCHES = {
    "gemv_q1_ring_norms_k10": (49_688, 1, 384, 10, ops.PATH_AUTO, 1),
    "gemv_q1_k100": (49_688, 1, 384, 100, ops.PATH_GEMV, 1),
    "gemv_q2_k16": (49_688, 2, 384, 16, ops.PATH_GEMV, 1),
    "gemv_q3_k100": (49_688, 3, 384, 100, ops.PATH_GEMV, 1),
    "gemv_q7_k10": (49_688, 7, 384, 10, ops.PATH_GEMV, 1),
    "gemv_q7_k100": (49_688, 7, 384, 100, ops.PATH_GEMV, 1),
    "swap_tail_q8_k10": (49_688, 8, 384, 10, ops.PATH_GEMM, 2),
    "swap_tail_q16_k100": (49_688, 16, 384, 100, ops.PATH_GEMM, 2),
    "swap_tail_q64_k100": (49_688, 64, 384, 100, ops.PATH_GEMM, 2),
    "swap_select_q256": (49_688, 256, 384, 100, ops.PATH_GEMM, 3),
    "swap_phased": (3_000, 16, 384, 256, ops.PATH_GEMM, 5),
    "k2_single": (49_688, 1000, 384, 100, ops.PATH_AUTO, 3),
    "k2_coarse": (600_000, 200, 384, 100, ops.PATH_AUTO, 3),
    "k2_phased_q300": (5_000, 300, 384, 100, ops.PATH_GEMM, 5),
    "k2_phased_q600": (5_000, 600, 384, 100, ops.PATH_GEMM, 5),
    # rows shorter than 512 bytes on a catalog of >= 640 MB: even one query takes the swapped tensor-core kernel
    "swap_short_rows_d128": (2_600_000, 1, 128, 10, ops.PATH_AUTO, 3),
}


def _branch_data(name, N, Q, D):
    seed = zlib.crc32(name.encode()) % 1000
    if N >= 500_000:  # generated on the device
        g = torch.Generator(device="cuda").manual_seed(seed)
        items = F.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
        items[::1009] = items[7]
        queries = F.normalize(items[torch.arange(Q, device="cuda") * (N // Q - 1)] + 0.3 * torch.randn(Q, D, device="cuda", generator=g), dim=1)
        return items, queries
    return _data(N, D, Q, seed)


def _branch_lists(name, q16, c16, k, Q, N):
    rng = np.random.default_rng(zlib.crc32(name.encode()) % 997)
    best = _own_best(q16, c16, min(N, 2 * k))
    # each query drops some of its own best rows (every bootstrap maximum and threshold moves) and random ones
    return [best[q][: (0, k // 2, 2 * k)[q % 3]] + rng.choice(N, 16, replace=False).tolist() for q in range(Q)]


@pytest.mark.parametrize("variant", ["plain", "excl", "excl_mask"])
@pytest.mark.parametrize("name", list(BRANCHES))
def test_every_plan_branch(name, variant):
    N, Q, D, k, path, want = BRANCHES[name]
    items, queries = _branch_data(name, N, Q, D)
    cat16 = icr.DeviceCatalog(items, dtype=torch.float16)
    cat_bf = icr.DeviceCatalog(items, dtype=torch.bfloat16)
    if "norms" not in name and name.startswith("gemv"):
        cat16.inv_norms = None  # the ring kernel that accumulates the rows' norms itself
    del items
    q16, qbf = queries.half(), queries.bfloat16()
    c16 = cat16.rows[:, :D]
    lists = _branch_lists(name, q16, c16, k, Q, N) if variant != "plain" else None
    mask = None
    if variant == "excl_mask":
        mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
        mask[torch.as_tensor(np.random.default_rng(3).choice(N, N // 50, replace=False), device="cuda")] = 1
    v, i = cat16.topk(q16, k, exclude_rows=lists, exclude_mask=mask, path=path)
    n16 = ops.last_launch_count()
    cat_bf.topk(qbf, k, exclude_rows=lists, exclude_mask=mask, path=path)
    nbf = ops.last_launch_count()
    assert n16 == nbf == want, f"{name}: {n16} launches on fp16, {nbf} on bf16, expected {want}"
    ex = _excl_matrix(lists, Q, N, mask) if (lists is not None or mask is not None) else None
    _check_topk(v, i, q16, c16, k, ex, name=name.split("_q")[0].split("_d")[0])


def test_gemv_direct_kernel_on_row_strided_catalog():
    """A catalog whose row stride exceeds its dim streams through the direct-load GEMV kernel (not the bulk-copy ring)."""
    N, D = 30_011, 384
    items, queries = _data(N, D, 7, 41)
    wide = torch.zeros(N, D + 64, dtype=torch.float16, device="cuda")
    wide[:, :D] = items.half()
    c16 = wide[:, :D]
    assert c16.stride(0) == D + 64
    for Q, k in ((1, 10), (3, 100), (7, 40)):
        q16 = queries[:Q].half()
        inv = ops.row_inv_norms(c16)
        v, i = ops.cos_topk(q16, c16, k, cat_inv_norms=inv, path=ops.PATH_GEMV)
        assert ops.last_launch_count() == 1
        _check_topk(v, i, q16, c16, k, name="gemv_direct")
        bits = ops.query_exclusion_bits(_own_best(q16, c16, 2 * k), N, "cuda")
        v, i = ops.cos_topk(q16, c16, k, exclude_bits=bits, path=ops.PATH_GEMV)
        _check_topk(v, i, q16, c16, k, _excl_matrix(_own_best(q16, c16, 2 * k), Q, N), name="gemv_direct")


# D = 768 ... 4096: the fp32 accumulation over K = D terms; D > 384 takes the A-streaming K2 variant. The swapped kernel keeps
# its queries resident: 16 queries of 4096 elements (128 KB) do not fit beside its ring, so D = 4096 runs on K2 only.
LARGE_D = [("swap_tail_q16_k100", 768), ("swap_tail_q16_k100", 1024), ("swap_tail_q16_k100", 2048),
           ("k2_single", 768), ("k2_single", 1024), ("k2_single", 2048), ("k2_single", 4096)]


@pytest.mark.parametrize("name,D", LARGE_D, ids=[f"{b}-D{d}" for b, d in LARGE_D])
def test_large_d(name, D):
    N, Q, _, k, path, want = BRANCHES[name]
    items, queries = _data(N, D, Q, D + 3)
    cat16 = icr.DeviceCatalog(items, dtype=torch.float16)
    v, i = cat16.topk(queries.half(), k, path=path)
    assert ops.last_launch_count() == want
    _check_topk(v, i, queries.half(), cat16.rows[:, :D], k, name=f"large_d_{D}")
    lists = _branch_lists(name, queries.half(), cat16.rows[:, :D], k, Q, N)
    v, i = cat16.topk(queries.half(), k, exclude_rows=lists, path=path)
    _check_topk(v, i, queries.half(), cat16.rows[:, :D], k, _excl_matrix(lists, Q, N), name=f"large_d_{D}")


# ---- inputs -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [8, 72, 200, 384])
@pytest.mark.parametrize("N", [777, 5_003, 20_001])
@pytest.mark.parametrize("path", [ops.PATH_GEMV, ops.PATH_GEMM])
def test_dims_and_ragged_catalogs(D, N, path):
    items, queries = _data(N, D, 9, D * 7 + N)
    cat = icr.DeviceCatalog(items, dtype=torch.float16)
    for k in (10, 100):
        v, i = cat.topk(queries, k, path=path)  # fp32 queries: normalised, then rounded
        _check_topk(v, i, ops.normalized_f16(queries), cat.rows, k, name="gemv" if path == ops.PATH_GEMV else "gemm")


@pytest.mark.parametrize("path", [ops.PATH_GEMV, ops.PATH_GEMM])
def test_fewer_rows_than_k(path):
    items, queries = _data(50, 384, 4, 5)
    cat = icr.DeviceCatalog(items, dtype=torch.float16)
    v, i = ops.cos_topk(queries.half(), cat.rows, 100, cat_inv_norms=cat.inv_norms, path=path)
    assert (i[:, 50:] == -1).all() and torch.isinf(v[:, 50:]).all()
    _check_topk(v, i, queries.half(), cat.rows, 100, name="gemv" if path == ops.PATH_GEMV else "gemm")


def _special_catalog(D=384, N=3_000, seed=8):
    """Zero rows, rows of fp16 subnormals, rows with elements up to 3e4 and exact duplicates; queries that rank each kind
    first."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    items = F.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
    q = F.normalize(torch.randn(6, D, device="cuda", generator=g), dim=1)
    items[100:140] = 0.0
    # subnormal rows: a query's direction in multiples of 2^-24 (at most 1023 of them: every element subnormal)
    sub = torch.round(q[0] / q[0].abs().max() * 1000.0)
    items[500] = sub * 2.0**-24
    items[501] = torch.round(q[1] / q[1].abs().max() * 700.0) * 2.0**-24
    # large-magnitude rows: a query's direction scaled to a largest element of 3e4
    items[900] = q[2] / q[2].abs().max() * 3.0e4
    items[901] = (q[3] + 0.1 * items[5]) / (q[3] + 0.1 * items[5]).abs().max() * 2.5e4
    # exact duplicates of a row close to query 4: the lower row ranks first
    items[1200] = F.normalize(q[4] + 0.01 * items[7], dim=0)
    items[2200] = items[1200]
    items[2900] = items[1200]
    return items, q


@pytest.mark.parametrize("path", [ops.PATH_GEMV, ops.PATH_GEMM])
def test_zero_subnormal_large_and_duplicate_rows(path):
    items, q = _special_catalog()
    cat = icr.DeviceCatalog(items, dtype=torch.float16)
    r = cat.rows
    assert (r[500] != 0).any() and (r[500].abs() < 2.0**-14).all(), "row 500 must be all fp16 subnormals"
    assert float(r[900].abs().max()) == 3.0e4
    q16 = q.half()
    v, i = ops.cos_topk(q16, r, 256, cat_inv_norms=cat.inv_norms, path=path)
    name = "gemv" if path == ops.PATH_GEMV else "gemm"
    _check_topk(v, i, q16, r, 256, name=name)
    assert int(i[0, 0]) == 500 and int(i[1, 0]) == 501, "subnormal rows must score as s_ref says (not flushed to 0)"
    assert int(i[2, 0]) == 900 and int(i[3, 0]) == 901
    assert i[4, :3].tolist() == [1200, 2200, 2900] and v[4, 0] == v[4, 1] == v[4, 2]
    # zero rows score exactly 0, not NaN: against an all-positive query every other row of -|r| scores below 0, so the
    # 40 zero rows lead the list (in row order)
    neg = -r.abs()
    qp = q16[5:6].abs()
    v, i = ops.cos_topk(qp, neg, 256, path=path)
    assert i[0, :40].tolist() == list(range(100, 140)) and (v[0, :40] == 0).all() and not torch.isnan(v).any()
    _check_topk(v, i, qp, neg, 256, name=name)


@pytest.mark.parametrize("Q,k", [(8, 10), (16, 100), (300, 50)])
def test_catalog_sorted_by_similarity(Q, k):
    """The best rows come first: segments are cut back in the kernels and the tail buffer overflows."""
    N, D = 49_688, 384
    g = torch.Generator().manual_seed(77)
    direction = F.normalize(torch.randn(D, generator=g), dim=0)
    items = F.normalize(torch.randn(N, D, generator=g), dim=1)
    items = items[torch.argsort(items @ direction, descending=True)].contiguous().cuda()
    queries = F.normalize(direction[None, :] + 0.05 * torch.randn(Q, D, generator=g), dim=1).cuda()
    cat = icr.DeviceCatalog(items, dtype=torch.float16)
    q16 = queries.half()
    v, i = cat.topk(q16, k, path=ops.PATH_GEMM)
    _check_topk(v, i, q16, cat.rows, k, name="gemm_sorted")
    lists = [list(range(q % 7, 3000, 3)) for q in range(Q)]
    v, i = cat.topk(q16, k, exclude_rows=lists, path=ops.PATH_GEMM)
    _check_topk(v, i, q16, cat.rows, k, _excl_matrix(lists, Q, N), name="gemm_sorted")


@pytest.mark.parametrize("Q,path", [(2, ops.PATH_GEMV), (16, ops.PATH_GEMM), (1000, ops.PATH_AUTO)])
def test_every_row_excluded_for_some_queries(Q, path):
    N, k = 20_000, 50
    items, queries = _data(N, 384, Q, 16)
    cat = icr.DeviceCatalog(items, dtype=torch.float16)
    rng = np.random.default_rng(17)
    lists = [rng.choice(N, size=int(rng.integers(0, 64))).tolist() for _ in range(Q)]
    lists[0] = list(range(N))
    lists[1] = rng.permutation(N)[: N - k + 3].tolist()
    v, i = cat.topk(queries.half(), k, exclude_rows=lists, path=path)
    assert (i[0] == -1).all() and torch.isinf(v[0]).all()
    assert int((i[1] >= 0).sum()) == k - 3
    _check_topk(v, i, queries.half(), cat.rows, k, _excl_matrix(lists, Q, N), name="excl_all")


@pytest.mark.parametrize("path", [ops.PATH_GEMV, ops.PATH_GEMM])
def test_fp32_queries_of_any_scale_are_normalised_before_rounding(path):
    items, queries = _data(20_000, 384, 5, 31)
    cat = icr.DeviceCatalog(items, dtype=torch.float16)
    ref16 = F.normalize(queries, dim=1).half()
    v0, i0 = cat.topk(ref16, 20, path=path)
    for scale in (1e-6, 1e6):
        qs = queries * scale
        q16 = ops.normalized_f16(qs)
        assert torch.isfinite(q16.float()).all() and (q16 != 0).any(dim=1).all()
        ulp = 2.0 ** (torch.floor(torch.log2(ref16.double().abs().clamp(min=2.0**-14))) - 10)
        assert ((q16.double() - ref16.double()).abs() <= ulp).all(), "normalised fp16 queries differ by more than one ulp"
        v, i = cat.topk(qs, 20, path=path)
        _check_topk(v, i, q16, cat.rows, 20, name="gemv" if path == ops.PATH_GEMV else "gemm")
        assert (v - v0).abs().max() <= 1e-3 and (i == i0).float().mean() >= 0.9


# ---- dense cos_sim ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("Qa,Nb,D", [(5, 300, 72), (63, 4000, 384), (64, 1000, 384), (64, 1024, 384), (300, 5000, 384), (128, 2048, 1024),
                                     (96, 1500, 4096)])
def test_dense_cos_sim(Qa, Nb, D):
    g = torch.Generator(device="cuda").manual_seed(Qa * 7 + D)
    a = (torch.randn(Qa, D, device="cuda", generator=g) * 3).half()
    b = (torch.randn(Nb, D, device="cuda", generator=g) * 0.2).half()
    b[3] = 0.0
    out = ops.cos_sim_dense(a, b)
    ref = _s_ref(a, b)
    err = (out.double() - ref).abs()
    assert not torch.isnan(out).any() and (out[:, 3] == 0).all()
    assert (err <= _tol(ref, D)).all(), f"max error {float(err.max()):.3e}"
    _record("dense_tc" if Qa >= 64 and Nb >= 1024 else "dense_cuda_core", (err / ref.abs().clamp(min=0.05)).max())


# ---- conversion and norms -----------------------------------------------------------------------------------------------------
def _conversion_rows(D):
    rng = np.random.default_rng(D)
    x = rng.standard_normal((64, D)) * 10.0 ** rng.uniform(-9, 5, (64, D))  # overflow, subnormals and underflow to zero
    x[3] = 0.0
    x[4, :4] = [65519.0, 65520.0, -1e6, 2.0**-25]  # the largest value that rounds down, the first that overflows, ...
    wide = torch.zeros(64, D + 8, dtype=torch.float32)
    wide[:, 8:] = torch.from_numpy(x).float()
    return wide.cuda()[:, 8:]


@pytest.mark.parametrize("D", [8, 72, 384, 4096])
def test_convert_rows_to_f16(D):
    x = _conversion_rows(D)
    out = ops.convert_rows(x, torch.empty(x.shape, dtype=torch.float16, device="cuda"))
    want = x.to(torch.float16)
    assert torch.isinf(want).any() and ((want != 0) & (want.abs() < 2.0**-14)).any()
    assert torch.equal(out.view(torch.int16), want.view(torch.int16)), "fp16 must be torch's RNE, overflow and subnormals included"
    n = ops.convert_rows(x, torch.empty(x.shape, dtype=torch.float16, device="cuda"), normalize=True).double()
    ref = F.normalize(x.double(), dim=1).half().double()
    ulp = 2.0 ** (torch.floor(torch.log2(ref.abs().clamp(min=2.0**-14))) - 10)
    assert ((n - ref).abs() <= ulp).all()
    assert (n[3] == 0).all()


@pytest.mark.parametrize("D", [8, 200, 4096])
def test_row_inv_norms_f16(D):
    x = (_conversion_rows(D) * 1e-3).clamp(-6e4, 6e4).half()
    inv = ops.row_inv_norms(x).double()
    ref = 1.0 / x.double().norm(dim=1).clamp(min=1e-12)
    assert ((inv - ref).abs() <= 1e-6 * ref).all()


# ---- DeviceCatalog --------------------------------------------------------------------------------------------------------
def _index_on_disk(tmp_path, n, d, seed=3):
    from instacart_next_order_recommendation_b200.index import EmbeddingIndex

    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text("{}")
    ids = [str(i) for i in range(n)]
    emb = oracle.synth_unnormalised(n, d, seed=seed).numpy()
    idx = EmbeddingIndex(corpus, "fake-model")
    idx.save(ids, emb)
    return idx, ids, emb


def test_device_catalog_f16(tmp_path):
    idx, ids, emb = _index_on_disk(tmp_path, 5_003, 384)
    t = torch.from_numpy(emb)
    cat = icr.DeviceCatalog(t, dtype=torch.float16)
    assert torch.equal(cat.rows.cpu().view(torch.int16), t.half().view(torch.int16))
    assert cat.planes is None and cat.inv_norms is not None and cat.dtype == torch.float16
    assert cat.nbytes == 5_003 * 384 * 2 + 4 * 5_003
    idx.save_bf16_sidecar()  # never used for fp16
    for chunk_rows in (1 << 17, 1000, 37):
        fc = icr.DeviceCatalog.from_index(idx, ids, dtype=torch.float16, chunk_rows=chunk_rows)
        assert torch.equal(fc.rows.cpu().view(torch.int16), t.half().view(torch.int16))
        assert fc.planes is None and fc.nbytes == 5_003 * 384 * 2 + 4 * 5_003
    nrm = icr.DeviceCatalog.from_index(idx, ids, dtype=torch.float16, normalize=True, chunk_rows=1000)
    ref = F.normalize(t.double(), dim=1).half().double()
    ulp = 2.0 ** (torch.floor(torch.log2(ref.abs().clamp(min=2.0**-14))) - 10)
    assert ((nrm.rows.cpu().double() - ref).abs() <= ulp).all()
    part = icr.DeviceCatalog.from_index(idx, ids, dtype=torch.float16, rows=(1200, 3100))
    assert torch.equal(part.rows.cpu(), t[1200:3100].half()) and part.row_offset == 1200
    # an fp16 tensor is taken bit for bit: -0.0, subnormals and inf-free extremes unchanged
    h = t[:100].half().clone()
    h[0, 0] = -0.0
    h[1, :3] = torch.tensor([2.0**-24, -(2.0**-20), 65504.0])
    for src in (h, h.cuda(), h.numpy()):
        c = icr.DeviceCatalog(src, dtype=torch.float16)
        assert torch.equal(c.rows.cpu().view(torch.int16), h.view(torch.int16))
    # rows beyond fp16's range raise, and name the way out
    with pytest.raises(ValueError, match="normalize=True"):
        icr.DeviceCatalog(t * 1e5, dtype=torch.float16)
    with pytest.raises(ValueError, match="float16's range"):
        icr.DeviceCatalog(torch.full((4, 16), 7e4), dtype=torch.float16)
    # the same through from_index; normalize=True loads
    (tmp_path / "big").mkdir()
    idx2, ids2, emb2 = _index_on_disk(tmp_path / "big", 300, 384)
    idx2.save(ids2, emb2 * 1e5)
    with pytest.raises(ValueError, match="float16's range"):
        icr.DeviceCatalog.from_index(idx2, ids2, dtype=torch.float16)
    big = icr.DeviceCatalog.from_index(idx2, ids2, dtype=torch.float16, normalize=True)
    assert torch.isfinite(big.rows).all()
    # queries through every entry of the catalog answer alike: fp16 as given, other dtypes normalised then rounded
    q = oracle.synth_unnormalised(9, 384, seed=11)
    v, i = cat.topk(q.cuda(), 50)
    _check_topk(v, i, ops.normalized_f16(q.cuda()), cat.rows, 50, name="gemm")
    v2, i2 = cat.topk(q.numpy(), 50)
    assert torch.equal(v, v2) and torch.equal(i, i2)
    v3, i3 = cat.topk_host(q, 50)
    torch.cuda.synchronize()
    assert torch.equal(v.cpu(), v3) and torch.equal(i.cpu(), i3)


def test_request_paths_agree_with_topk():
    items, queries = _data(49_688, 384, 7, 61)
    cat = icr.DeviceCatalog(items, dtype=torch.float16)
    cat_bf = icr.DeviceCatalog(items, dtype=torch.bfloat16)
    for Q in (1, 3, 7):
        q32 = queries[:Q]
        q16 = ops.normalized_f16(q32)
        for k in (10, 100):
            v, i = cat.topk(q32, k)
            _check_topk(v, i, q16, cat.rows, k, name="gemv")
            # the CUDA graph with the query conversion captured (host and device fp32 queries)
            for src in (q32.cpu(), q32.cpu().numpy(), q32):
                vs, is_ = cat.topk_small(src, k)
                assert torch.equal(vs, v) and torch.equal(is_, i)
            # a device fp16 query in the catalog's layout: the prepared call, as many launches as for bf16
            vs, is_ = cat.topk_small(q16, k)
            n16 = ops.last_launch_count()
            assert torch.equal(vs, v) and torch.equal(is_, i)
            cat_bf.topk_small(q32.bfloat16(), k)
            assert ops.last_launch_count() == n16 == (1 if Q <= 3 else 2)
            sv, si = cat.topk_request(q16, k)
            assert ops.last_launch_count() == n16
            assert si == i.tolist() and np.array_equal(np.asarray(sv, dtype=np.float32), v.cpu().numpy())
            sv, si = cat.topk_request(q32, k)  # fp32 device query: through the graph
            assert si == i.tolist()


# ---- Recommender --------------------------------------------------------------------------------------------------------------
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


def _tie_safe_equal(got, want, tol):
    """Same products where the neighbouring reference scores are more than `tol` apart, scores within `tol`."""
    assert len(got) == len(want)
    ws = [s for _, s in want]
    for j, ((gp, gs), (wp, w)) in enumerate(zip(got, want)):
        assert abs(gs - w) <= tol, (j, gs, w)
        gap = min(abs(w - ws[j - 1]) if j > 0 else 1.0, abs(w - ws[j + 1]) if j + 1 < len(ws) else 0.0)
        if gap > tol:  # the last position competes with the unseen next one: never decisive
            assert gp == wp, (j, gp, wp)


def _same(got, want):
    """The batched and the request kernels: same products in the same order, scores equal to 1e-6."""
    assert [p for p, _ in got] == [p for p, _ in want]
    np.testing.assert_allclose([s for _, s in got], [s for _, s in want], rtol=1e-6)


@pytest.mark.parametrize("enc", [_DeviceEnc, _HostEnc])
def test_recommender_f16(golden_dir, tmp_path, monkeypatch, enc):
    z = np.load(golden_dir / "embeddings_small.npz")
    pids = [str(p) for p in z["product_ids"]]
    corpus = tmp_path / "eval_corpus.json"
    corpus.write_text(json.dumps({pid: f"c:{i}" for i, pid in enumerate(pids)}))
    monkeypatch.setenv("ICR_CATALOG_DTYPE", "fp16")
    rec = icr.Recommender("fake-model", corpus, model=enc(z), use_index=False)
    assert rec.catalog.dtype == torch.float16
    items16 = torch.from_numpy(z["items"]).half().float()
    gold = json.loads((golden_dir / "recommend_golden.json").read_text())
    rng = np.random.default_rng(4)
    cases = [(c["q"], c["top_k"], set(c["exclude"])) for c in gold["cases"]]
    cases += [(q % len(z["queries"]), 10, set(rng.choice(pids, 300, replace=False).tolist())) for q in range(3)]  # the long-list mask path
    for q, top_k, excl in cases:
        q16 = ops.normalized_f16(torch.from_numpy(z["queries"][q : q + 1]).cuda()).float().cpu()
        want = oracle.recommend_tail(q16[0], items16, pids, top_k, excl)
        got = rec.recommend(f"q:{q}", top_k=top_k, exclude_product_ids=excl)
        tol = RTOL * max(max((abs(s) for _, s in want), default=0.0), 0.05)
        _tie_safe_equal(got, want, 2 * tol)
        _same(rec.recommend_batch([f"q:{q}"], top_k=top_k, exclude_product_ids=[excl])[0], got)
    batch = rec.recommend_batch([f"q:{q}" for q, _, _ in cases], top_k=10, exclude_product_ids=[e for _, _, e in cases])
    for b, (q, _, e) in zip(batch, cases):
        _same(b, rec.recommend(f"q:{q}", top_k=10, exclude_product_ids=e))
    # against the fp32 golden results: fp16 rounding of the embeddings moves scores by < 2e-4
    for c in gold["cases"]:
        got = rec.recommend(f"q:{c['q']}", top_k=c["top_k"], exclude_product_ids=set(c["exclude"]))
        _tie_safe_equal(got, [tuple(r) for r in c["result"]], 2e-4)


# ---- ranking quality on the clustered generator -----------------------------------------------------------------------------
def test_top10_id_sets_match_fp64_for_99_percent_of_queries():
    N, D, Q, k = 49_688, 384, 1000, 10
    items, _ = oracle.synth_clustered(N, D, seed=1234)
    queries, _ = oracle.synth_queries_from_items(items, Q, seed=1235)
    exact = torch.topk(F.normalize(queries.double(), dim=1) @ F.normalize(items.double(), dim=1).T, k, dim=1).indices
    share = {}
    for dt in (torch.float16, torch.bfloat16):
        cat = icr.DeviceCatalog(items.cuda(), dtype=dt)
        _, i = cat.topk(queries.cuda(), k)
        share[dt] = float(np.mean([set(a) == set(b) for a, b in zip(i.cpu().tolist(), exact.tolist())]))
    print(f"\ntop-10 id set equal to fp64: fp16 catalog {share[torch.float16]:.1%}, bf16 catalog {share[torch.bfloat16]:.1%}")
    assert share[torch.float16] >= 0.99


# ---- seeded fuzz ------------------------------------------------------------------------------------------------------------
_N_CASES = int(os.environ.get("ICR_F16_FUZZ_CASES", "200"))
_SEED = int(os.environ.get("ICR_F16_FUZZ_SEED", "20261021"))


def _fuzz_cases(n, seed):
    rng = np.random.default_rng(seed)
    out = []
    for c in range(n):
        Q = int(rng.choice([1, 2, 3, 5, 7, 8, 33, 130, 256, 300, 700]))
        N = int(rng.choice([7, 100, 1000, 4097, 20_000, 49_688, 70_001]))
        D = int(rng.choice([8, 64, 128, 200, 384, 768]))
        k = int(rng.choice([1, 5, 10, 37, 100, 256]))
        path = int(rng.choice([ops.PATH_AUTO, ops.PATH_GEMV, ops.PATH_GEMM]))
        density = float(rng.choice([0.0, 0.0, 1e-3, 0.01, 0.2, 0.9]))
        out.append((c, Q, N, D, k, path, density))
    return out


@pytest.mark.parametrize("case", _fuzz_cases(_N_CASES, _SEED), ids=lambda c: f"{c[0]}-Q{c[1]}-N{c[2]}-D{c[3]}-k{c[4]}-p{c[5]}-x{c[6]}")
def test_fuzz(case):
    c, Q, N, D, k, path, density = case
    if path == ops.PATH_GEMV and Q > 64:
        path = ops.PATH_AUTO
    it = oracle.synth_unnormalised(N, D, seed=3000 + c).cuda()
    qt = oracle.synth_unnormalised(Q, D, seed=4000 + c).cuda()
    rng = np.random.default_rng(5000 + c)
    lists = [np.nonzero(rng.random(N) < density)[0].tolist() for _ in range(Q)] if density > 0 else None
    kk = min(k, N)
    cat = icr.DeviceCatalog(it, dtype=torch.float16, row_offset=3)
    q16 = qt.half() if c % 2 else qt  # fp16 queries as given, or fp32 ones normalised and rounded
    v, i = cat.topk(q16, kk, exclude_rows=lists, path=path)
    qref = q16 if c % 2 else ops.normalized_f16(qt)
    _check_topk(v, i, qref, cat.rows, kk, _excl_matrix(lists, Q, N) if lists else None, name="fuzz", offset=3)


# ---- sharded --------------------------------------------------------------------------------------------------------------------
def test_sharded_catalog_f16_world_size_1():
    items, queries = _data(30_011, 384, 9, 71)
    sh = icr.ShardedCatalog(items, row_offset=0, total_rows=30_011, dtype=torch.float16)
    assert sh.local.dtype == torch.float16
    for Q, k in ((1, 10), (9, 100)):
        v, i = sh.topk(queries[:Q], k)
        _check_topk(v, i, ops.normalized_f16(queries[:Q]), sh.local.rows, k, name="sharded")


def test_sharded_catalog_f16_two_gpus():
    import subprocess
    import sys
    from pathlib import Path

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs on one machine")
    root = Path(__file__).resolve().parents[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nproc-per-node", "2", "--master-addr", "127.0.0.1", "--master-port", "29523",
           str(root / "benchmarks" / "f16_sharded_case.py")]
    out = subprocess.run(cmd, cwd=str(root), capture_output=True, text=True, timeout=600, env=dict(os.environ))
    assert out.returncode == 0, out.stderr[-2000:]
    assert "F16_SHARDED_OK" in out.stdout, out.stdout[-2000:]
