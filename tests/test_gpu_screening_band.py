"""The fp32 screening band at its worst case, on every tensor-core plan branch (B200 only).

fp32 catalogs are searched on ONE fp16 plane per operand, fp16(256 * x / |x|); every selection keeps the keys within
kScreenBandRaw (select_args.cuh) below the k-th best screened score, and only those are re-scored exactly. With random
inputs the 384 rounding errors cancel and screening errors stay near 1e-5, far inside the band. Here the rounding is
chosen instead: every coordinate that carries score sits 0.47 fp16 ulp above a power of two (rounds down, on support A)
or 0.53 ulp above it (rounds up, on support B). One true top-k row `r` lives on A, the other k - 1 top rows and a few
decoys (exact scores >= 1e-4 below r) on B, so the screened order inverts r and the decoys by more than one eps
(69 raw units, checked in `_self_check` from the planes `ops.screen_plane` returns). A band without its factor 2, or
missing at any one place that applies it, loses r and returns a decoy.

The operand kernels themselves (screen plane, hi|lo planes, row conversion) are checked element by element at the end.
"""

import math
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import instacart_next_order_recommendation_b200 as icr
from instacart_next_order_recommendation_b200 import ops
from oracle import oracle

pytestmark = pytest.mark.gpu

F32_RTOL = 1e-5
U = 2.0**-10  # fp16 ulp relative to a power of two
F_DOWN, F_UP = 0.47, 0.53  # placement above a power of two, in ulps: rounds down / up with a 0.03 ulp margin
N_DECOYS = 3
DECOY_GAP = 1e-4  # exact score of the best decoy <= s_r - 1e-4
MIN_INVERSION = 1.05e-3  # 69 raw units (65536 * cosine): more than one eps = 2^-10


@pytest.fixture(scope="module", autouse=True)
def _device():
    assert torch.cuda.is_available(), "run with -m gpu on a GPU box"
    torch.cuda.set_device(0)
    assert icr._lib.load().icr_device_supported() == 1
    yield
    torch.cuda.synchronize()


# ---- the host plan, restated (gemm_topk.cu: swap_applies, boot_pairs_for, k2_boot_plan) -------------------------------------
# Only used to put rows into the tiles the in-kernel bootstraps read; ops.last_launch_count() pins the branch of every call.
NUM_SMS, BN, BM, BK = 148, 256, 128, 64


def _swap_applies(Q, N, D):
    if Q > 256:
        return False
    qpad = (Q + 31) // 32 * 32
    kb = (D + BK - 1) // BK
    res = kb * (qpad // 2) * 128
    return res <= (100 * 1024 if N * kb * BK * 2 <= (96 << 20) else 64 * 1024)


def _balanced_chunks(qblocks, c0, T):
    npairs = NUM_SMS // 2
    best, best_load = c0, -1
    c = c0
    while c <= T and c < c0 + 24:
        load = ((qblocks * c + npairs - 1) // npairs) * ((T + c - 1) // c)
        if best_load < 0 or load < best_load:
            best, best_load = c, load
        c += 1
    return best


def _boot_plan(Q, N, D, k):
    """(chunks, boot tiles per chunk, rows per bootstrap group) of the single-launch modes, or None (phased path)."""
    T = (N + BN - 1) // BN
    if _swap_applies(Q, N, D):
        pairs = min(T, NUM_SMS // 2)
        if 8 * pairs < 2 * k or 8 * pairs > 640:
            return None
        tiles = max(1, (N // 4000 * k + BN * pairs - 1) // (BN * pairs))
        if tiles > 1 and tiles * 4 > T // pairs:
            return None
        return pairs, tiles, 32
    qblocks = (Q + 2 * BM - 1) // (2 * BM)
    c0 = min(max((2 * (NUM_SMS // 2) + qblocks - 1) // qblocks, (550 + 71) // 72), T)
    best = _balanced_chunks(qblocks, c0, T)
    tiles = max(1, (N * k // 550 + BN * best - 1) // (BN * best))
    while best * tiles * 8 < 2 * k:
        tiles += 1
    if best * tiles * 8 > 640:
        ct = min(640 // (best * 2), tiles)
        if qblocks != 1 or T < 2048 or ct < 1 or best * ct * 2 < 2 * k or N * k / (BN * best * ct) > 2500.0 or ct * 4 > T // best:
            return None
        return best, ct, 128
    l2_sized = N * ((D + 63) // 64 * 64) * 2 <= (96 << 20)
    if tiles * (2 if l2_sized else 4) > T // best:
        return None
    return best, tiles, 32


def _chunk_tiles(c, chunks, T):
    return c * T // chunks, (c + 1) * T // chunks


# ---- adversarial construction -----------------------------------------------------------------------------------------------
def _geometry(D, k):
    """Coordinates (scaled units, |x| = 256): supports A and B of n coordinates each at magnitude m (and 2m), then the
    tuning coordinate, the query's slack and the rows' slack."""
    for e in (2, 3, 4):  # as many coordinates as fit: the accumulation runs over all of them
        n = 31744 // 4**e
        if 2 * n + 3 <= D:
            m = 2.0**e
            break
    x_max = 0.125 * (k + 16)
    budget = 65536.0 - (x_max + 2) ** 2 - 64.0
    n2 = int((budget / m**2 - n) // 3)  # coordinates of a row at 2m (the rest at m): |row_A| as close to 256 as fits
    return n, m, n2


class Adversarial:
    """Rows and queries of `n_adv` adversarial queries, written into an ordinary catalog and batch at the given rows."""

    def __init__(self, D, k, n_adv, seed):
        self.D, self.k, self.n_adv = D, k, n_adv
        n, m, n2 = self.n, self.m, self.n2 = _geometry(D, k)
        A, B = np.arange(n), np.arange(n, 2 * n)
        self.t, qs, rs = 2 * n, 2 * n + 1, 2 * n + 2
        rng = np.random.default_rng(seed)
        self.signs = rng.choice([-1.0, 1.0], size=(n_adv, D))
        down, up = 1 + F_DOWN * U, 1 + F_UP * U
        mag_r = np.where(np.arange(n) < n2, 2 * m, m)  # row pattern on its support
        # exact parts of the scores (raw units) before tuning: sum over the support of q_i * row_i
        p_r = float(np.sum(m * down * mag_r * down))
        p_o = float(np.sum(m * up * mag_r * up))
        x_d0 = math.floor((p_r - p_o - DECOY_GAP * 65536) / 32 / 0.125) * 0.125
        x_o0 = math.ceil((p_r - p_o + DECOY_GAP * 65536) / 32 / 0.125) * 0.125
        tune = {"r": 0.0}
        q = np.zeros((n_adv, D))
        rows = {}  # (a, kind, j) -> vector
        for a in range(n_adv):
            s = self.signs[a]
            qa = np.zeros(D)
            qa[A], qa[B], qa[self.t] = m * down, m * up, 32.0
            qa[qs] = math.sqrt(65536.0 - float(np.sum(qa**2)))
            q[a] = qa * s

            def row(support, f, x):
                v = np.zeros(D)
                v[support] = mag_r * f
                v[self.t] = x
                v[rs] = math.sqrt(65536.0 - float(np.sum(v**2)))
                return v * s

            rows[(a, "r", 0)] = row(A, down, tune["r"])
            for j in range(k - 1):
                rows[(a, "o", j)] = row(B, up, x_o0 + 0.125 * j)
            for j in range(N_DECOYS):
                rows[(a, "d", j)] = row(B, up, x_d0 - 0.25 * j)
        self.q = q
        self.rows = rows
        self.crowd_rng = rng

    def crowd_row(self, a):
        """A row that scores ~0.25 for query a: far below its top-k (>= 5e-3), far above random rows."""
        v = np.zeros(self.D)
        B = np.arange(self.n, 2 * self.n)
        v[B] = self.m * (self.crowd_rng.random(self.n) < 0.5)
        v[2 * self.n + 2] = math.sqrt(65536.0 - float(np.sum(v**2)))
        return v * self.signs[a]


def _ordinary(N, Q, D, seed):
    g = torch.Generator().manual_seed(seed)
    return F.normalize(torch.randn(N, D, generator=g), dim=1), F.normalize(torch.randn(Q, D, generator=g), dim=1)


def _placements(kind, adv, N, Q, D, k):
    """{(a, kind, j): catalog row} for every adversarial row, plus crowd rows {row: a}."""
    T = (N + BN - 1) // BN
    plan = _boot_plan(Q, N, D, k)
    per_q = k - 1 + N_DECOYS
    where, crowd = {}, {}
    if kind == "head":
        # the top rows and decoys each open their own bootstrap group (single launch) or sit in the first tiles (phased);
        # r comes last in the catalog
        if plan is not None:
            chunks, tiles, group = plan
            slots = [(lo + bt) * BN + o for c in range(chunks) for bt in range(tiles)
                     for lo in [_chunk_tiles(c, chunks, T)[0]] for o in range(0, BN, group)]
            slots = [s for s in slots if s < N - BN]
        else:
            slots = list(range(0, N - BN))
        assert len(slots) >= adv.n_adv * per_q, "not enough bootstrap groups for these adversarial queries"
        it = iter(slots)
        for a in range(adv.n_adv):
            for key in [(a, "o", j) for j in range(k - 1)] + [(a, "d", j) for j in range(N_DECOYS)]:
                where[key] = next(it)
            where[(a, "r", 0)] = N - 1 - 37 * a
    elif kind == "spread":
        # one row per stride through the whole catalog (a tile or more apart where N allows), r last
        total = adv.n_adv * per_q
        stride = max(1, (N - BN) // total)
        pos = iter(range(stride // 2, N - BN, stride))
        for j in range(per_q):
            for a in range(adv.n_adv):
                key = (a, "o", j) if j < k - 1 else (a, "d", j - (k - 1))
                where[key] = next(pos)
        for a in range(adv.n_adv):
            where[(a, "r", 0)] = N - 1 - 37 * a
    elif kind == "packed":
        # the top rows, decoys and a crowd fill one column half of one work item: its segment overflows and is cut back
        # in the kernel while r, in the same half of the work item's last tile, is still to come
        chunks, _, _ = plan
        need = 4 if not _swap_applies(Q, N, D) else 3
        cands = [c for c in range(1, chunks) if _chunk_tiles(c, chunks, T)[1] - _chunk_tiles(c, chunks, T)[0] >= need]
        assert len(cands) >= adv.n_adv
        for a in range(adv.n_adv):
            lo, hi = _chunk_tiles(cands[a], chunks, T)
            rows = [t * BN + i for t in range(lo, hi - 1) for i in range(BN // 2)]
            keys = [(a, "o", j) for j in range(k - 1)] + [(a, "d", j) for j in range(N_DECOYS)]
            for key, r in zip(keys, rows):
                where[key] = r
            for r in rows[len(keys):]:
                crowd[r] = a
            where[(a, "r", 0)] = (hi - 1) * BN + 5
    else:
        raise ValueError(kind)
    assert len(set(where.values())) == len(where) and not set(where.values()) & set(crowd)
    return where, crowd


def _build(N, Q, D, k, n_adv, kind, seed):
    adv = Adversarial(D, k, n_adv, seed)
    items, queries = _ordinary(N, Q, D, seed + 1)
    items, queries = items.double(), queries.double()
    where, crowd = _placements(kind, adv, N, Q, D, k)
    for key, r in where.items():
        items[r] = torch.from_numpy(adv.rows[key] / 256.0)
    for r, a in crowd.items():
        items[r] = torch.from_numpy(adv.crowd_row(a) / 256.0)
    qrows = np.linspace(0, Q - 1, n_adv).round().astype(int)
    for a, qr in enumerate(qrows):
        queries[qr] = torch.from_numpy(adv.q[a] / 256.0)
    r_rows = [where[(a, "r", 0)] for a in range(n_adv)]
    decoys = [[where[(a, "d", j)] for j in range(N_DECOYS)] for a in range(n_adv)]
    return items.float(), queries.float(), qrows.tolist(), r_rows, decoys


def _self_check(it_d, qt_d, qrows, r_rows, decoys, k):
    """From the planes the library builds: r is a true top-k row whose screened score is >= 69 raw units below the k-th
    best screened score; the decoys are decisively below r in exact score."""
    cp, _ = ops.screen_plane(it_d)
    qp, _ = ops.screen_plane(qt_d[qrows])
    scr = (qp.double() @ cp.double().T) / 65536.0
    ex = F.normalize(qt_d[qrows].double(), dim=1) @ F.normalize(it_d.double(), dim=1).T
    for a, r in enumerate(r_rows):
        kth_exact = torch.topk(ex[a], k).values[-1]
        assert ex[a, r] == kth_exact, "r must be the k-th true top row"
        assert float(ex[a, r] - ex[a, decoys[a]].max()) >= DECOY_GAP * 0.99
        kth_scr = torch.topk(scr[a], k).values[-1]
        inv = float(kth_scr - scr[a, r])
        assert inv >= MIN_INVERSION, f"screened inversion {inv:.3e} < {MIN_INVERSION:.3e}"
        # every row outside the top k + decoys scores >= 5e-3 below r
        rest = ex[a].clone()
        rest[torch.topk(ex[a], k).indices] = -2
        rest[decoys[a]] = -2
        assert float(ex[a, r] - rest.max()) >= 5e-3


def _check_topk(v, i, rv, ri, rtol):
    v, i = v.cpu(), i.cpu()
    assert v.shape == rv.shape and i.shape == ri.shape
    assert (v[:, :-1] >= v[:, 1:]).all(), "scores must be non-increasing"
    err, mism = oracle.compare_topk(v, i, rv, ri, rtol=rtol)
    assert err <= rtol, f"max relative score error {err}"
    assert mism == 0, f"{mism} id mismatches outside ties"
    for r in range(i.shape[0]):
        assert len(set(i[r].tolist())) == i.shape[1]


def _excluded(lists, Q, N, mask):
    ex = torch.zeros(Q, N, dtype=torch.bool, device="cuda")
    if lists is not None:
        for q, l in enumerate(lists):
            if len(l):
                ex[q, torch.as_tensor(l, device="cuda")] = True
    if mask is not None:
        ex |= mask.bool()[None, :]
    return ex


def _verify(v, i, it_d, qt_d, k, qrows, r_rows, decoys, lists, mask):
    Q, N = qt_d.shape[0], it_d.shape[0]
    ex = _excluded(lists, Q, N, mask)
    # fp64 ranking, with the excluded pairs out
    rv, ri = [], []
    cn = F.normalize(it_d.double(), dim=1)
    for q0 in range(0, Q, 256):
        s = F.normalize(qt_d[q0 : q0 + 256].double(), dim=1) @ cn.T
        s[ex[q0 : q0 + 256]] = float("-inf")
        t = torch.topk(s, k, dim=1)
        rv.append(t.values.cpu())
        ri.append(t.indices.cpu())
    rv, ri = torch.cat(rv), torch.cat(ri)
    _check_topk(v, i, rv, ri, F32_RTOL)
    # fp32 witness at the returned rows
    w = (F.normalize(qt_d, dim=1)[:, None, :] * F.normalize(it_d, dim=1)[i.clamp(min=0)]).sum(-1)
    assert torch.allclose(v, w, rtol=F32_RTOL, atol=0), f"max |v - witness| {float((v - w).abs().max()):.3e}"
    assert not ex.gather(1, i.clamp(min=0)).any(), "an excluded row was returned"
    ic = i.cpu()
    for a, qr in enumerate(qrows):
        got = set(ic[qr].tolist())
        assert r_rows[a] in got, f"adversarial query {a}: the true top-k row {r_rows[a]} was screened out"
        assert not got & set(decoys[a]), f"adversarial query {a}: a decoy was returned"


# branch -> (N, Q, k, path, launches: exact int or (">", n) / (">=", n))
BRANCHES = {
    "swap_tail_q8_k10": (49_688, 8, 10, ops.PATH_GEMM, 2),
    "swap_tail_q16_k100": (49_688, 16, 100, ops.PATH_GEMM, 2),
    "swap_tail_q64_k100": (49_688, 64, 100, ops.PATH_GEMM, 2),
    "swap_select_q256": (49_688, 256, 100, ops.PATH_GEMM, 3),
    "swap_phased": (3_000, 16, 256, ops.PATH_GEMM, (">", 3)),
    "k2_single": (49_688, 1000, 100, ops.PATH_AUTO, 4),
    "k2_coarse": (600_000, 200, 100, ops.PATH_AUTO, 3),
    "k2_phased_q300": (5_000, 300, 100, ops.PATH_GEMM, (">=", 5)),
    "k2_phased_q600": (5_000, 600, 100, ops.PATH_GEMM, (">=", 5)),
}
SINGLE_LAUNCH = {"swap_tail_q8_k10", "swap_tail_q16_k100", "swap_tail_q64_k100", "swap_select_q256", "k2_single", "k2_coarse"}


def _launches_ok(n, want):
    if isinstance(want, int):
        return n == want
    op, m = want
    return n > m if op == ">" else n >= m


def _n_adv(branch, kind, N, Q, D, k):
    if kind == "head":
        plan = _boot_plan(Q, N, D, k)
        slots = N - BN if plan is None else plan[0] * plan[1] * (BN // plan[2])
        return max(1, min(4, Q // 2, slots // (k + N_DECOYS + 2)))
    return max(1, min(4, Q // 2, (N - BN) // (BN * (k + N_DECOYS)) if kind == "spread" else 4))


def _run_case(branch, kind, D, excl, mask_rows=False, seed=0):
    N, Q, k, path, want = BRANCHES[branch]
    n_adv = _n_adv(branch, kind, N, Q, D, k)
    it, qt, qrows, r_rows, decoys = _build(N, Q, D, k, n_adv, kind, seed)
    it_d, qt_d = it.cuda(), qt.cuda()
    _self_check(it_d, qt_d, qrows, r_rows, decoys, k)
    cat = icr.DeviceCatalog(it_d, dtype=torch.float32)
    protected = set(r_rows) | {d for ds in decoys for d in ds}
    rng = np.random.default_rng(seed + 7)
    lists = None
    if excl:
        # each query drops 16 rows that take no part in the construction (the XB kernels run; the inversion stays)
        lists = [[int(x) for x in rng.choice(N, 24, replace=False) if int(x) not in protected][:16] for _ in range(Q)]
    mask = None
    if mask_rows:
        mask = torch.zeros(N, dtype=torch.uint8, device="cuda")
        ex = F.normalize(qt_d[qrows], dim=1) @ F.normalize(it_d, dim=1).T
        top = set(torch.topk(ex, k, dim=1).indices.flatten().tolist())
        cand = [int(x) for x in rng.choice(N, N // 50, replace=False) if int(x) not in top and int(x) not in protected]
        mask[torch.as_tensor(cand, device="cuda")] = 1
    if lists is not None:
        # an adversarial query must keep its k - 1 other top rows: drop any of its own top rows from its list
        ex = F.normalize(qt_d[qrows], dim=1) @ F.normalize(it_d, dim=1).T
        for a, qr in enumerate(qrows):
            top = set(torch.topk(ex[a], k + N_DECOYS).indices.tolist())
            lists[qr] = [x for x in lists[qr] if x not in top]
    v, i = cat.topk(qt_d, k, exclude_rows=lists, exclude_mask=mask, path=path)
    n = ops.last_launch_count()
    assert _launches_ok(n, want), f"{branch}: {n} launches, expected {want}: the shape no longer takes this branch"
    _verify(v, i, it_d, qt_d, k, qrows, r_rows, decoys, lists, mask)
    # second witness: the GEMV path (fp32, no screening) returns the same ids for the adversarial queries
    sub = [lists[q] for q in qrows] if lists is not None else None
    v1, i1 = cat.topk(qt_d[qrows], k, exclude_rows=sub, exclude_mask=mask, path=ops.PATH_GEMV)
    for a, qr in enumerate(qrows):
        assert set(i1[a].tolist()) == set(i[qr].tolist())


CASES = [(b, kind) for b in BRANCHES for kind in ("head", "spread")] + [(b, "packed") for b in ("swap_tail_q16_k100", "k2_single", "k2_coarse")]


@pytest.mark.parametrize("excl", [False, True], ids=["plain", "excl"])
@pytest.mark.parametrize("branch,kind", CASES, ids=[f"{b}-{k}" for b, k in CASES])
def test_screening_band_holds_the_inverted_row(branch, kind, excl):
    _run_case(branch, kind, 384, excl, seed=zlib.crc32(f"{branch}-{kind}".encode()) % 1000)


def test_screening_band_with_shared_mask_and_exclusions():
    _run_case("k2_single", "spread", 384, True, mask_rows=True, seed=5)
    _run_case("swap_tail_q16_k100", "head", 384, False, mask_rows=True, seed=6)


# Large D: the fp32 accumulation of the tensor cores over K = D terms; D > 384 also takes the A-streaming K2 variant.
LARGE_D = [("swap_tail_q16_k100", 1024), ("swap_tail_q16_k100", 2048), ("k2_single", 1024), ("k2_single", 2048), ("k2_single", 4096)]


@pytest.mark.parametrize("kind", ["head", "spread"])
@pytest.mark.parametrize("branch,D", LARGE_D, ids=[f"{b}-D{d}" for b, d in LARGE_D])
def test_screening_band_large_d(branch, D, kind):
    _run_case(branch, kind, D, False, seed=D + 11)


# ---- operand kernels ----------------------------------------------------------------------------------------------------------
def _f16_ulp(v):
    a = np.abs(v)
    e = np.floor(np.log2(np.maximum(a, 2.0**-14)))
    return 2.0 ** (e - 10)


def _operand_rows(D, seed):
    """Ordinary rows of mixed scale, zero rows, and rows with a large dynamic range (fp16 subnormals after scaling),
    returned as a row-strided view."""
    rng = np.random.default_rng(seed)
    R = 96
    x = rng.standard_normal((R, D)) * 10.0 ** rng.uniform(-3, 3, (R, 1))
    x[5] = 0.0
    x[R - 1] = 0.0
    for r in range(10, 30):
        x[r] = rng.choice([-1.0, 1.0], D) * 10.0 ** rng.uniform(-9, 0, D)
        x[r, rng.integers(D)] = 1.0
    wide = torch.zeros(R, D + 12, dtype=torch.float32)
    wide[:, 3 * 4 : 3 * 4 + D] = torch.from_numpy(x).float()
    return wide.cuda()[:, 12:]


@pytest.mark.parametrize("D", [8, 72, 200, 384, 4096])
def test_screen_plane_is_the_rounded_scaled_row(D):
    xd = _operand_rows(D, D)
    assert xd.stride(0) == D + 12
    plane, inv = ops.screen_plane(xd)
    dp = (D + 63) // 64 * 64
    assert plane.shape == (xd.shape[0], dp)
    x64 = xd.cpu().double().numpy()
    nrm = np.linalg.norm(x64, axis=1)
    inv_ref = 1.0 / np.maximum(nrm, 1e-12)
    inv = inv.cpu().double().numpy()
    assert np.all(np.abs(inv - inv_ref) <= 1e-6 * inv_ref)
    p = plane.cpu().double().numpy()
    assert (p[:, D:] == 0).all(), "padding must be zero"
    v = 256.0 * x64 * inv_ref[:, None]
    err = np.abs(p[:, :D] - v)
    # round to nearest: half an ulp (1e-5 of it for the bound) plus the fp32 normalisation (< 1e-6 relative)
    assert np.all(err <= 0.5 * _f16_ulp(v) * (1 + 1e-5) + 1e-6 * np.abs(v)), f"max error {np.max(err / _f16_ulp(v)):.4f} ulp"
    # and bit for bit what one fp32 multiply by the returned scale, then fp16 RN, gives
    sc = (np.float32(256.0) * inv.astype(np.float32)).astype(np.float32)
    v32 = xd.cpu().numpy() * sc[:, None]
    assert np.array_equal(p[:, :D].astype(np.float16).view(np.uint16), v32.astype(np.float16).view(np.uint16))
    assert (p[5] == 0).all() and (p[-1] == 0).all(), "a zero row gives a zero plane"
    assert (p[10:30, :D] != 0).any() and (np.abs(p[10:30, :D]) < 2.0**-14).any() and (np.abs(p[10:30, :D]) > 0).any()


@pytest.mark.parametrize("D", [72, 384, 4096])
def test_split_f16_planes_carry_22_bits(D):
    xd = _operand_rows(D, D + 1)
    planes = ops.split_f16_planes(xd)
    dp = (D + 63) // 64 * 64
    assert planes.shape == (xd.shape[0], 2 * dp)
    hi, lo = planes[:, :dp].cpu().double().numpy(), planes[:, dp:].cpu().double().numpy()
    assert (hi[:, D:] == 0).all() and (lo[:, D:] == 0).all(), "padding must be zero"
    x64 = xd.cpu().double().numpy()
    v = 256.0 * x64 / np.maximum(np.linalg.norm(x64, axis=1), 1e-12)[:, None]
    # the row's fp32 scale, recovered from hi + lo (least squares): within 1e-6 of the exact one
    num, den = np.sum((hi + lo)[:, :D] * v, axis=1), np.sum(v * v, axis=1)
    c = np.where(den > 0, num / np.where(den > 0, den, 1), 1.0)
    assert np.all(np.abs(c - 1) <= 1e-6)
    vc = v * c[:, None]
    hi, lo = hi[:, :D], lo[:, :D]
    assert np.all(np.abs(hi - vc) <= 0.5 * _f16_ulp(vc) * (1 + 1e-5) + 2.0**-23 * np.abs(vc)), "hi = RN(v)"
    # lo = RN(v - hi): |hi + lo - v| <= 2^-22 |v| + 2^-24 (+ the fp32 multiply's rounding of v and the fit of c)
    assert np.all(np.abs(hi + lo - vc) <= (2.0**-22 + 2.0**-23) * np.abs(vc) + 2.0**-24)
    assert np.all(np.abs(lo) <= 0.5 * _f16_ulp(vc) * (1 + 1e-5) + 2.0**-23 * np.abs(vc))
    assert (hi[5] == 0).all() and (lo[5] == 0).all()


@pytest.mark.parametrize("D", [8, 384, 4096])
def test_convert_rows(D):
    xd = _operand_rows(D, D + 2)
    out = ops.convert_rows(xd, torch.empty(xd.shape, dtype=torch.bfloat16, device="cuda"))
    assert torch.equal(out.view(torch.int16), xd.to(torch.bfloat16).view(torch.int16)), "bf16 must be torch's RNE"
    out32 = ops.convert_rows(xd, torch.empty(xd.shape, dtype=torch.float32, device="cuda"))
    assert torch.equal(out32, xd)
    ref = F.normalize(xd.double(), dim=1)
    n32 = ops.convert_rows(xd, torch.empty(xd.shape, dtype=torch.float32, device="cuda"), normalize=True).double()
    assert ((n32 - ref).abs() <= 1e-6 * ref.abs() + 1e-30).all()
    nb = ops.convert_rows(xd, torch.empty(xd.shape, dtype=torch.bfloat16, device="cuda"), normalize=True).double()
    # one bf16 rounding of the (fp32-normalised) value: within one bf16 ulp, 2^-7 relative
    assert ((nb - ref).abs() <= 2.0**-8 * ref.abs() * (1 + 1e-5) + 2.0**-133).all()
    assert (nb[5] == 0).all() and (n32[5] == 0).all()
