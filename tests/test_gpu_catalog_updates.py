"""In-place catalog updates: DeviceCatalog.update_rows / append_rows / remove_rows, ShardedCatalog.update_rows and the
Recommender's update_products / remove_products / update_corpus.

Contract: a catalog changed in place equals a catalog freshly built from the updated fp32 matrix, in the same row order,
through the same constructor path: rows, planes and inverse norms bit for bit (compared as integer views), and therefore
every top-k result (ids and score bits) on every plan branch.

Tests without the gpu mark check the C ABI surface, the Recommender's corpus diff with a host stand-in for the catalog, and
the rank routing of ShardedCatalog.update_rows with gloo.
"""

import json
import os
import re
import socket
import sys
import threading
import time
import zlib
from pathlib import Path

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from instacart_next_order_recommendation_b200 import _lib
from oracle import oracle

gpu = pytest.mark.gpu
ROOT = Path(__file__).resolve().parents[1]


# ---- host-only checks -----------------------------------------------------------------------------------------------------------
def test_symbol_is_declared_mirrored_and_exported():
    header = (ROOT / "include" / "icr_b200.h").read_text()
    assert re.search(r"\bint icr_update_rows\(", header)
    assert "icr_update_rows" in _lib.SIGNATURES and len(_lib.SIGNATURES["icr_update_rows"][1]) == 13
    assert hasattr(_lib.load(), "icr_update_rows")


def test_bad_arguments_return_their_codes_before_any_cuda_call():
    lib = _lib.load()
    p = 1 << 20  # never dereferenced: every check below comes before the device is touched
    ok = dict(x=p, M=4, dim=64, ldx=64, dst=p, N=10, dtype=0, rows=p, ld=64, plane=None, inv=p, norm=0)

    def call(**kw):
        a = {**ok, **kw}
        return lib.icr_update_rows(a["x"], a["M"], a["dim"], a["ldx"], a["dst"], a["N"], a["dtype"], a["rows"], a["ld"], a["plane"],
                                   a["inv"], a["norm"], None)

    assert call(dtype=3, norm=1) == -1 and b"normalize" in lib.icr_last_error_string()  # int8 with normalize
    assert call(dtype=5) == -2
    assert call(dtype=1, plane=p) == -1  # only fp32 catalogs have a plane
    assert call(dst=None) == -1 and call(inv=None) == -1 and call(rows=None) == -1
    assert call(M=-1) == -1 and call(N=-1) == -1
    assert call(dim=62, ldx=62, ld=62) == -3  # fp32 rows need dim % 4 == 0
    assert call(dtype=1, dim=100, ldx=100, ld=104) == -3  # bf16 rows need dim % 8 == 0
    assert call(dtype=3, dim=100, ldx=100, ld=100) == -3  # int8 codes need a row stride >= round_up(dim, 16)
    assert call(ld=32) == -1  # row stride below dim
    assert call(plane=p + 64) == -3  # the plane is 128-byte aligned


class _HostCatalog:
    """The DeviceCatalog surface the Recommender changes, on the host."""

    def __init__(self, emb):
        self.rows = np.array(emb, dtype=np.float32)
        self.input_dim = self.rows.shape[1]
        self.calls = []

    def update_rows(self, rows, x):
        self.calls.append(("update", list(rows)))
        self.rows[list(rows)] = x

    def append_rows(self, x):
        n = len(self.rows)
        self.calls.append(("append", len(x)))
        self.rows = np.concatenate([self.rows, x])
        return range(n, n + len(x))

    def remove_rows(self, rows):
        self.calls.append(("remove", sorted(rows)))
        kept = np.setdiff1d(np.arange(len(self.rows)), rows)
        self.rows = self.rows[kept]
        return kept


class _StubEncoder:
    """Deterministic text -> unit vector; counts the texts it encodes."""

    def __init__(self, dim=64, device=False):
        self.dim, self.device, self.encoded = dim, device, []

    def vec(self, text):
        v = np.random.default_rng(zlib.crc32(text.encode())).standard_normal(self.dim).astype(np.float32)
        return v / np.linalg.norm(v)

    def encode(self, texts, batch_size=64, show_progress_bar=False, normalize_embeddings=True, convert_to_tensor=False):
        self.encoded.extend(texts)
        out = np.stack([self.vec(t) for t in texts])
        return torch.from_numpy(out).cuda() if (convert_to_tensor and self.device) else out


def _host_recommender(corpus, enc):
    from instacart_next_order_recommendation_b200.recommender import Recommender, _ReadWriteLock

    rec = object.__new__(Recommender)  # the host half of the constructor: no device catalog
    rec.product_ids, rec.product_texts = list(corpus), list(corpus.values())
    rec.pid_to_text = dict(corpus)
    rec._pid_to_row = {p: i for i, p in enumerate(rec.product_ids)}
    rec.model, rec._batch_size = enc, 64
    rec._rw, rec._update_lock = _ReadWriteLock(), threading.RLock()
    rec.product_embeddings = np.stack([enc.vec(t) for t in rec.product_texts])
    rec.catalog = _HostCatalog(rec.product_embeddings)
    return rec


def test_corpus_diff_encodes_only_new_and_changed_texts():
    enc = _StubEncoder()
    old = {f"p{i}": f"text {i}" for i in range(8)}
    rec = _host_recommender(old, enc)
    new = {"p1": "text 1", "p9": "text 9", "p3": "text 3 changed", "p0": "text 0", "p10": "text 10", "p6": "text 6"}
    rec.update_corpus(new)
    assert enc.encoded == ["text 3 changed", "text 9", "text 10"]
    # removed first (p2, p4, p5, p7), then the changed row in place (p3, now row 2), then the new ids in corpus order
    assert rec.catalog.calls == [("remove", [2, 4, 5, 7]), ("update", [2]), ("append", 2)]
    assert rec.product_ids == ["p0", "p1", "p3", "p6", "p9", "p10"]
    assert rec.product_texts == [new[p] for p in rec.product_ids] and rec.pid_to_text == {p: new[p] for p in rec.product_ids}
    assert rec._pid_to_row == {p: i for i, p in enumerate(rec.product_ids)}
    want = np.stack([enc.vec(new[p]) for p in rec.product_ids])
    assert np.array_equal(rec.product_embeddings, want) and np.array_equal(rec.catalog.rows, want)
    # nothing new or changed: no encode call, no catalog call
    enc.encoded.clear()
    rec.catalog.calls.clear()
    rec.update_products({"p0": "text 0", "p9": "text 9"})
    rec.remove_products(["unknown"])
    assert enc.encoded == [] and rec.catalog.calls == []
    rec.remove_products(["p3", "unknown", "p3"])
    assert rec.catalog.calls == [("remove", [2])] and rec.product_ids == ["p0", "p1", "p6", "p9", "p10"]


# ---- rank routing of ShardedCatalog.update_rows (gloo, host stand-ins for the shards) ------------------------------------------
class _HostShard:
    def __init__(self, rows):
        self.rows = rows.clone()

    def __len__(self):
        return self.rows.shape[0]

    def update_rows(self, rows, x):
        rows = np.asarray(rows)
        if len(rows):
            self.rows[torch.from_numpy(rows)] = torch.as_tensor(x, dtype=torch.float32)


def _oracle_local_topk(queries, shard, k, row_offset):
    v, i = oracle.cos_topk(queries, shard.rows, k)
    return v, i + row_offset


def _oracle_merge(scores, ids, k):
    G, Q, kin = scores.shape
    s = scores.permute(1, 0, 2).reshape(Q, G * kin).double()
    i = ids.permute(1, 0, 2).reshape(Q, G * kin)
    s = torch.where(i < 0, torch.full_like(s, float("-inf")), s)
    order = torch.from_numpy(np.lexsort((i.numpy(), -s.numpy()), axis=1)[:, :k])
    return s.gather(1, order).float(), i.gather(1, order)


def _routing_worker(rank, world, port, out_dir):
    import torch.distributed as dist

    sys.path.insert(0, str(ROOT))
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from instacart_next_order_recommendation_b200.sharded import ShardedCatalog, shard_bounds

        full = oracle.synth_clustered(301, 32, seed=21, n_centres=8)[0]
        lo, hi = shard_bounds(301, world, rank)
        cat = ShardedCatalog(_HostShard(full[lo:hi]), row_offset=lo, total_rows=301, _local_topk=_oracle_local_topk, _merge=_oracle_merge)
        g = [0, 150, 151, 300, 77, 200]  # both blocks (151 + 150 rows), both edges of each
        x = oracle.synth_isotropic(len(g), 32, seed=22)
        cat.update_rows(g, x)
        want = full.clone()
        want[g] = x
        assert torch.equal(cat.local.rows, want[lo:hi])
        for bad in ([301], [-1], [5, 5]):  # every rank rejects alike, before it writes
            try:
                cat.update_rows(bad, x[: len(bad)])
                raise AssertionError(f"accepted {bad}")
            except ValueError:
                pass
        assert torch.equal(cat.local.rows, want[lo:hi])
        q = oracle.synth_isotropic(5, 32, seed=23)
        v, i = cat.topk(q, 10)
        rv, ri = oracle.cos_topk(q, want, 10)
        err, mism = oracle.compare_topk(v, i, rv, ri, rtol=1e-6)
        assert err < 1e-6 and mism == 0, (err, mism)
        torch.save({"i": i}, os.path.join(out_dir, f"r{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_sharded_update_routes_rows_to_their_rank(tmp_path):
    import torch.multiprocessing as mp

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_routing_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert torch.equal(torch.load(tmp_path / "r0.pt")["i"], torch.load(tmp_path / "r1.pt")["i"])


# ---- GPU ------------------------------------------------------------------------------------------------------------------------
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


# kind -> (dtype, normalize, build_planes). Catalogs with normalize come from from_index(normalize=True), the only way to build
# one; the others from the constructor.
KINDS = {
    "f32": (torch.float32, False, True),
    "f32_norm": (torch.float32, True, True),
    "f32_noplanes": (torch.float32, False, False),
    "bf16": (torch.bfloat16, False, None),
    "bf16_norm": (torch.bfloat16, True, None),
    "f16": (torch.float16, False, None),
    "f16_norm": (torch.float16, True, None),
    "i8": (torch.int8, False, None),
}


def _build(kind, X, tmp_path=None):
    """A catalog over the fp32 matrix X (host) through the constructor path of `kind`."""
    icr = _icr()
    dtype, normalize, planes = KINDS[kind]
    if not normalize:  # a host matrix: the catalog owns its rows (a device fp32 matrix would be shared until the first change)
        return icr.DeviceCatalog(X, dtype=dtype, build_planes=planes)
    d = tmp_path / f"idx{zlib.crc32(X.numpy().tobytes())}"
    d.mkdir(exist_ok=True)
    (d / "corpus.json").write_text("{}")
    idx = icr.EmbeddingIndex(d / "corpus.json", "fake-model")
    ids = [str(i) for i in range(X.shape[0])]
    idx.save(ids, X.numpy())
    cat = icr.DeviceCatalog.from_index(idx, ids, dtype=dtype, normalize=True)
    assert cat.normalized
    return cat


def _bits(t):
    if t is None:
        return None
    return t.view({4: torch.int32, 2: torch.int16, 1: torch.int8}[t.element_size()])


def _assert_same_catalog(cat, fresh, what):
    assert cat.rows.shape == fresh.rows.shape, what
    assert torch.equal(_bits(cat.rows), _bits(fresh.rows)), f"{what}: rows differ"
    assert (cat.planes is None) == (fresh.planes is None), what
    if fresh.planes is not None:
        assert torch.equal(_bits(cat.planes), _bits(fresh.planes)), f"{what}: planes differ"
    assert torch.equal(_bits(cat.inv_norms), _bits(fresh.inv_norms)), f"{what}: inverse norms differ"


def _assert_same_results(a, b):
    assert torch.equal(a[1], b[1]), f"ids differ at {int((a[1] != b[1]).sum())} positions"
    assert torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)), "score bits differ"


@gpu
@pytest.mark.parametrize("D", [100, 384, 768, 4096])
@pytest.mark.parametrize("kind", list(KINDS))
def test_bit_identity_after_update_append_remove(cuda0, tmp_path, kind, D):
    N = 2000
    g = torch.Generator().manual_seed(D * 31 + len(kind))
    X = torch.randn(N, D, generator=g) * torch.exp(torch.randn(N, 1, generator=g))  # un-normalised rows
    cat = _build(kind, X, tmp_path)
    nbytes = cat.nbytes
    # update in place: scattered rows, the first and the last, with fresh values
    rows = torch.randperm(N, generator=g)[:300].tolist() + [0, N - 1]
    rows = list(dict.fromkeys(rows))
    Y = torch.randn(len(rows), D, generator=g) * 3.0
    ptr = cat.rows.data_ptr()
    cat.update_rows(rows, Y)
    X[rows] = Y
    assert cat.rows.data_ptr() == ptr and cat.nbytes == nbytes
    _assert_same_catalog(cat, _build(kind, X, tmp_path), "update_rows")
    # the first append reallocates with headroom; the second lands inside the reserve
    A = torch.randn(50, D, generator=g)
    assert cat.append_rows(A) == range(N, N + 50)
    X = torch.cat([X, A])
    _assert_same_catalog(cat, _build(kind, X, tmp_path), "append_rows (reallocation)")
    ptr = cat.rows.data_ptr()
    B = torch.randn(20, D, generator=g)
    assert cat.append_rows(B.numpy()) == range(N + 50, N + 70)
    X = torch.cat([X, B])
    assert cat.rows.data_ptr() == ptr
    _assert_same_catalog(cat, _build(kind, X, tmp_path), "append_rows (reserve)")
    # stable removal of scattered rows, including the first and the last
    gone = sorted(set(torch.randperm(N + 70, generator=g)[:150].tolist()) | {0, N + 69})
    kept = cat.remove_rows(gone)
    assert np.array_equal(kept, np.setdiff1d(np.arange(N + 70), gone))
    X = X[torch.from_numpy(kept)]
    _assert_same_catalog(cat, _build(kind, X, tmp_path), "remove_rows")
    # and appending after a removal reuses the freed rows
    ptr = cat.rows.data_ptr()
    C = torch.randn(30, D, generator=g)
    cat.append_rows(C)
    X = torch.cat([X, C])
    assert cat.rows.data_ptr() == ptr
    _assert_same_catalog(cat, _build(kind, X, tmp_path), "append_rows after remove_rows")


@gpu
def test_f16_inputs_land_bit_for_bit_and_shared_rows_are_copied(cuda0):
    icr = _icr()
    X = oracle.synth_unnormalised(500, 64, seed=5)
    cat = icr.DeviceCatalog(X.half(), dtype=torch.float16)
    h = (torch.randn(3, 64) * 0.1).half()
    h[0, 0], h[1, 1], h[2, 2] = -0.0, 2.0**-24, 65504.0
    cat.update_rows([7, 8, 9], h)
    assert torch.equal(cat.rows[7:10].cpu().view(torch.int16), h.view(torch.int16))
    # an fp32 device matrix is taken as is: the catalog's first change copies it instead of writing into the caller's tensor
    dev = X.cuda()
    before = dev.clone()
    c32 = icr.DeviceCatalog(dev)
    assert c32.rows.data_ptr() == dev.data_ptr()
    c32.update_rows([3], torch.ones(1, 64))
    assert torch.equal(dev, before) and c32.rows.data_ptr() != dev.data_ptr()
    assert torch.equal(c32.rows[3].cpu(), torch.ones(64))


# ---- results on every plan branch -----------------------------------------------------------------------------------------------
# name -> (N, Q, D, k, path, launches on a 16-bit or int8 catalog): the branches tests/test_gpu_f16_catalog.py and
# tests/test_gpu_i8_catalog.py pin with ops.last_launch_count()
BRANCHES = {
    "gemv_q1_ring_k10": (49_688, 1, 384, 10, 0, 1),
    "gemv_q3_k100": (49_688, 3, 384, 100, 1, 1),
    "gemv_q7_k100": (49_688, 7, 384, 100, 1, 1),
    "swap_tail_q8_k10": (49_688, 8, 384, 10, 2, 2),
    "swap_tail_q64_k100": (49_688, 64, 384, 100, 2, 2),
    "swap_select_q256": (49_688, 256, 384, 100, 2, 3),
    "swap_phased": (3_000, 16, 384, 256, 2, 5),
    "k2_single": (49_688, 1000, 384, 100, 0, 3),
    "k2_coarse": (600_000, 200, 384, 100, 0, 3),
    "k2_phased_q300": (5_000, 300, 384, 100, 2, 5),
    "swap_short_rows_d128": (2_600_000, 1, 128, 10, 0, 3),
}


def _branch_data(name, N, Q, D):
    g = torch.Generator(device="cuda").manual_seed(zlib.crc32(name.encode()) % 1000)
    X = F.normalize(torch.randn(N, D, device="cuda", generator=g), dim=1)
    X[::1009] = X[7]  # exact ties
    q = F.normalize(X[torch.arange(Q, device="cuda") * (N // Q - 1)] + 0.3 * torch.randn(Q, D, device="cuda", generator=g), dim=1)
    return X, q, g


@gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.int8, torch.float32], ids=["f16", "i8", "f32"])
@pytest.mark.parametrize("name", list(BRANCHES))
def test_results_equal_a_fresh_catalog_on_every_plan_branch(cuda0, name, dtype):
    from instacart_next_order_recommendation_b200 import ops

    icr = _icr()
    if dtype == torch.float32 and BRANCHES[name][0] > 100_000:
        pytest.skip("the large branches are pinned for the 16-bit and int8 layouts")
    N, Q, D, k, path, want = BRANCHES[name]
    X, q, g = _branch_data(name, N, Q, D)
    rows = torch.randperm(N, device="cuda", generator=g)[: max(N // 100, 16)]
    old = X.clone()
    old[rows] = F.normalize(torch.randn(rows.numel(), D, device="cuda", generator=g), dim=1)
    cat = icr.DeviceCatalog(old, dtype=dtype)
    del old
    # the rows a query would have returned are among those replaced: the results move
    best = cat.topk(q[:1], k)[1][0]
    rows = torch.unique(torch.cat([rows, best[best >= 0]]))
    cat.update_rows(rows, X[rows])
    fresh = icr.DeviceCatalog(X, dtype=dtype)
    del X
    rng = np.random.default_rng(zlib.crc32(name.encode()))
    lists = [rng.choice(N, 40, replace=False).tolist() for _ in range(Q)]
    mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
    mask[torch.as_tensor(rng.choice(N, N // 50, replace=False), device="cuda")] = 1
    for excl, m in ((None, None), (lists, None), (lists, mask), (None, mask)):
        a = cat.topk(q, k, exclude_rows=excl, exclude_mask=m, path=path)
        n_a = ops.last_launch_count()
        b = fresh.topk(q, k, exclude_rows=excl, exclude_mask=m, path=path)
        if dtype != torch.float32 and (excl is not None or m is None):
            assert n_a == ops.last_launch_count() == want, f"{name}: {n_a} launches, expected {want}"
        _assert_same_results(a, b)


@gpu
@pytest.mark.parametrize("dtype", [torch.float16, torch.int8, torch.float32], ids=["f16", "i8", "f32"])
def test_gemv_direct_kernel_on_an_updated_catalog(cuda0, dtype):
    """A row stride above the dim streams through the direct-load GEMV kernel: a catalog whose last 64 columns are zero,
    searched over its first D columns."""
    from instacart_next_order_recommendation_b200 import ops

    icr = _icr()
    N, D = 30_011, 384
    X, q, g = _branch_data("direct", N, 7, D)
    wide = F.pad(X, (0, 64))
    old = wide.clone()
    old[: N // 10] = F.pad(F.normalize(torch.randn(N // 10, D, device="cuda", generator=g), dim=1), (0, 64))
    cat = icr.DeviceCatalog(old, dtype=dtype)
    cat.update_rows(range(N // 10), wide[: N // 10])
    fresh = icr.DeviceCatalog(wide, dtype=dtype)
    for Q, k in ((1, 10), (3, 100), (7, 40)):
        qq = cat._device_queries(q[:Q])[:, :D].contiguous()
        a = ops.cos_topk(qq, cat.rows[:, :D], k, cat_inv_norms=cat.inv_norms, path=ops.PATH_GEMV)
        assert ops.last_launch_count() == 1
        b = ops.cos_topk(qq, fresh.rows[:, :D], k, cat_inv_norms=fresh.inv_norms, path=ops.PATH_GEMV)
        _assert_same_results(a, b)


# ---- request paths ------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.int8], ids=["f32", "f16", "i8"])
def test_request_paths_return_the_new_rows(cuda0, dtype):
    icr = _icr()
    N, D = 49_688, 384
    X, q, g = _branch_data("requests", N, 3, D)
    old = X.clone()
    old[:5000] = F.normalize(torch.randn(5000, D, device="cuda", generator=g), dim=1)
    cat = icr.DeviceCatalog(old.cpu(), dtype=dtype)  # owned rows: the update stays in place
    qd = cat._device_queries(q[:1])  # the catalog's own layout: the prepared call
    qh = q[:1].cpu()  # a host query: the CUDA graph

    def all_paths(c):
        r = [c.topk_small(qh, 10), c.topk_small(qd, 10), c.topk(qd, 10)]
        sv, si = c.topk_request(qd, 10)
        r.append((torch.tensor(sv, dtype=torch.float32, device="cuda"), torch.tensor(si, device="cuda")))
        return r

    before = all_paths(cat)  # builds the graph, the prepared calls and the resident workspaces
    graphs, plans = dict(cat._graphs), dict(cat._plans)
    cat.update_rows(range(5000), X[:5000])
    fresh = icr.DeviceCatalog(X, dtype=dtype)
    want = fresh.topk(qd, 10)
    assert not torch.equal(before[0][1], want[1])  # the update moves this query's results
    for got in all_paths(cat):
        _assert_same_results(got, want)
    assert cat._graphs.keys() == graphs.keys() and cat._plans.keys() == plans.keys()  # in place: nothing was rebuilt
    # a change of length: the request state is rebuilt over the new rows
    A = F.normalize(torch.randn(100, D, device="cuda", generator=g), dim=1)
    A[0] = q[0]  # the query's own direction: the new best row
    cat.append_rows(A)
    X = torch.cat([X, A])
    want = icr.DeviceCatalog(X, dtype=dtype).topk(q[:1].cuda(), 10)
    assert int(want[1][0, 0]) == N
    for got in all_paths(cat):
        _assert_same_results(got, want)
    kept = cat.remove_rows(list(range(0, N, 7)))
    X = X[torch.from_numpy(kept).cuda()]
    want = icr.DeviceCatalog(X, dtype=dtype).topk(q[:1].cuda(), 10)
    for got in all_paths(cat):
        _assert_same_results(got, want)


# ---- rejected input -------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("kind", ["f32", "f16", "i8", "bf16_norm"])
def test_rejected_input_leaves_the_catalog_unchanged(cuda0, tmp_path, kind):
    X = oracle.synth_unnormalised(400, 96, seed=9) * 10.0
    cat = _build(kind, X, tmp_path)
    snap = [None if t is None else t.clone() for t in (cat.rows, cat.planes, cat.inv_norms)]
    good = torch.randn(2, 96)
    nan = good.clone()
    nan[1, 5] = float("nan")
    inf = good.clone()
    inf[0, 0] = float("inf")
    cases = [
        ("update", ([1, 1], good)),  # duplicate
        ("update", ([1, 400], good)),  # out of range
        ("update", ([-1, 2], good)),
        ("update", ([1, 2], nan)),  # non-finite
        ("update", ([1, 2], inf)),
        ("update", ([1, 2], torch.randn(2, 95))),  # dim mismatch
        ("update", ([1, 2, 3], good)),  # count mismatch
        ("update", ([1.0, 2.0], good)),  # not integers
        ("append", (nan,)),
        ("append", (torch.randn(2, 97),)),
        ("remove", ([3, 3],)),
        ("remove", ([400],)),
    ]
    if kind == "f16":
        cases += [("update", ([1, 2], good * 1e5)), ("append", (good * 1e5,))]  # fp16 overflow after conversion
    for op, args in cases:
        with pytest.raises(ValueError):
            getattr(cat, f"{op}_rows")(*args)
        for a, b in zip((cat.rows, cat.planes, cat.inv_norms), snap):
            assert (a is None) == (b is None) and (a is None or torch.equal(_bits(a), _bits(b))), (op, args)
    if kind == "bf16_norm":  # normalised catalogs take rows of any magnitude
        cat.update_rows([1, 2], good * 1e30)


# ---- sharded, world size 1 ------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.int8], ids=["f32", "f16", "i8"])
def test_sharded_update_world_size_1_equals_a_fresh_shard(cuda0, dtype):
    icr = _icr()
    X = oracle.synth_clustered(20_011, 384, seed=31)[0]
    Y = oracle.synth_clustered(500, 384, seed=32)[0]
    sh = icr.ShardedCatalog(X, row_offset=0, total_rows=20_011, dtype=dtype)
    rows = np.random.default_rng(4).choice(20_011, 500, replace=False)
    sh.update_rows(rows, Y)
    X[torch.from_numpy(rows)] = Y
    fresh = icr.ShardedCatalog(X, row_offset=0, total_rows=20_011, dtype=dtype)
    _assert_same_catalog(sh.local, fresh.local, "sharded")
    q = oracle.synth_queries_from_items(X, 9, seed=33)[0].cuda()
    _assert_same_results(sh.topk(q, 50), fresh.topk(q, 50))


# ---- Recommender ----------------------------------------------------------------------------------------------------------------
def _results_equal(a, b):
    assert [p for p, _ in a] == [p for p, _ in b]
    assert np.array_equal(np.asarray([s for _, s in a], dtype=np.float32), np.asarray([s for _, s in b], dtype=np.float32))


def _corpus_file(tmp_path, name, corpus):
    p = tmp_path / name
    p.write_text(json.dumps(corpus))
    return p


def _check_against_fresh(rec, enc, tmp_path, dtype, queries):
    icr = _icr()
    corpus = {pid: rec.pid_to_text[pid] for pid in rec.product_ids}
    fresh = icr.Recommender("fake-model", _corpus_file(tmp_path, f"fresh{len(corpus)}.json", corpus), model=enc, use_index=False,
                            catalog_dtype=dtype)
    assert fresh.product_ids == rec.product_ids
    assert np.array_equal(np.asarray(rec.product_embeddings), np.asarray(fresh.product_embeddings))
    pids = rec.product_ids
    excl = [set(), set(pids[:3]), set(pids[::7][:40]) | {"unknown"}]
    for q in queries:
        for top_k in (1, 10, 100):
            for ex in excl:
                _results_equal(rec.recommend(q, top_k=top_k, exclude_product_ids=ex), fresh.recommend(q, top_k=top_k, exclude_product_ids=ex))
    for got, want in zip(rec.recommend_batch(queries, top_k=20, exclude_product_ids=[excl[i % 3] for i in range(len(queries))]),
                         fresh.recommend_batch(queries, top_k=20, exclude_product_ids=[excl[i % 3] for i in range(len(queries))])):
        _results_equal(got, want)


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.int8], ids=["f32", "f16", "i8"])
def test_recommender_changes_equal_a_fresh_recommender(cuda0, tmp_path, dtype):
    icr = _icr()
    enc = _StubEncoder(dim=384, device=True)
    corpus = {f"p{i}": f"product {i}" for i in range(3000)}
    rec = icr.Recommender("fake-model", _corpus_file(tmp_path, "corpus.json", corpus), model=enc, use_index=False, catalog_dtype=dtype)
    queries = [f"user {i}" for i in range(5)] + ["product 17", "product 2999 new"]
    _check_against_fresh(rec, enc, tmp_path, dtype, queries)
    # change and add
    enc.encoded.clear()
    rec.update_products({"p17": "product 17 new", "p5": "product 5", "n1": "product new 1", "n2": "product 2999 new"})
    assert sorted(enc.encoded) == ["product 17 new", "product 2999 new", "product new 1"]
    assert rec.product_ids[-2:] == ["n1", "n2"] and rec.pid_to_text["p17"] == "product 17 new"
    _check_against_fresh(rec, enc, tmp_path, dtype, queries)
    # remove (unknown ids ignored)
    rec.remove_products(["p0", "p17", "nope", "n1"])
    assert "p17" not in rec.pid_to_text and rec.product_ids[-1] == "n2"
    _check_against_fresh(rec, enc, tmp_path, dtype, queries)
    # the incremental /admin/corpus: removals, a change, and new ids in corpus order
    new_corpus = {pid: rec.pid_to_text[pid] for pid in rec.product_ids[::2]}
    new_corpus["p2"] = "product 2 renamed"
    new_corpus = {"z9": "product z9", **new_corpus, "z1": "product z1"}
    survivors = [pid for pid in rec.product_ids if pid in new_corpus]
    enc.encoded.clear()
    rec.update_corpus(new_corpus)
    assert sorted(enc.encoded) == ["product 2 renamed", "product z1", "product z9"]
    assert rec.product_ids == survivors + ["z9", "z1"]
    _check_against_fresh(rec, enc, tmp_path, dtype, queries + ["product z9"])


@gpu
def test_requests_beside_an_update_see_the_before_or_the_after_state(cuda0, tmp_path):
    icr = _icr()
    enc = _StubEncoder(dim=384, device=True)
    corpus = {f"p{i}": f"product {i}" for i in range(20_000)}
    rec = icr.Recommender("fake-model", _corpus_file(tmp_path, "corpus.json", corpus), model=enc, use_index=False)
    queries = [f"product {i}" for i in range(0, 20_000, 2500)] + ["product new 3"]
    new_corpus = {pid: t for i, (pid, t) in enumerate(corpus.items()) if i % 3}
    new_corpus.update({f"n{i}": f"product new {i}" for i in range(50)})
    new_corpus["p1"] = "product 0"
    before = [rec.recommend(q, top_k=10) for q in queries], rec.recommend_batch(queries, top_k=10)
    shadow = icr.Recommender("fake-model", _corpus_file(tmp_path, "c2.json", corpus), model=enc, use_index=False)
    shadow.update_corpus(new_corpus)
    after = [shadow.recommend(q, top_k=10) for q in queries], shadow.recommend_batch(queries, top_k=10)
    seen, stop, errors = [], threading.Event(), []

    def requests():
        try:
            while not stop.is_set():
                j = len(seen) % len(queries)
                seen.append((j, rec.recommend(queries[j], top_k=10), rec.recommend_batch(queries, top_k=10)))
        except Exception as e:  # pragma: no cover - reported below
            errors.append(e)

    t = threading.Thread(target=requests)
    t.start()
    while len(seen) < 3:
        time.sleep(0.001)
    rec.update_corpus(new_corpus)
    n_during = len(seen)
    while len(seen) < n_during + 3:
        time.sleep(0.001)
    stop.set()
    t.join()
    assert not errors, errors
    states = set()
    for j, one, batch in seen:  # the update may fall between the two calls: each result is one state or the other
        for got, b, a in ((one, before[0][j], after[0][j]), (batch, before[1], after[1])):
            assert got in (b, a), f"query {j}: a result of neither state"
            states.add("before" if got == b else "after")
    assert states == {"before", "after"}
