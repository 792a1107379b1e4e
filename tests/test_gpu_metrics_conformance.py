"""GPU: the metric kernels — lhn_pck_accumulate (its all-f32 FAST instantiation and the general one),
lhn_mpii_pckh_accumulate, lhn_evaluate_pck and lhn_metrics_finalize (in test_gpu_round2.py) — against the oracle at
their edges, and the fused decode counters against lhn_pck_accumulate where its grid is capped.

Every comparison is bit for bit: the counters are integers and the oracle restates their rules (hits `d < f32(thr)`
after rounding the distance to f32, the fixed-point EPE term of O.epe_fix_counts, MPII's `<=` in f64), and
evaluate_pck's per-image values and mean are exact for the reason given in its test.

lhn_pck_accumulate launches at most 8 * SMs blocks of 256 threads, lhn_mpii_pckh_accumulate 4 * SMs.  N is computed
from the device's cap, so the cases past it stay past it on any SM count, and every case that is meant to sit in
the gap between the cap and the next multiple of K (the elements a stride rounded UP to a multiple of K skipped)
asserts that it does: cap % K != 0 and N * K > cap.  On 148 SMs the cap is 2^13 * 37 threads, so K = 1 and 16 never
have a gap and K = 17, 21 and 62 do.

Reachable paths the tables leave out, and why:
  - pck FAST path refused because gt or the normaliser alone is misaligned or strided: the same `al8` / stride rule as
    pred, which the offset view and the stride-3 pred cover;
  - pck general path with an f32 normaliser at stride != 2: ops.pck_accumulate makes the normaliser contiguous and the
    C ABI has no normaliser stride;
  - evaluate_pck weights other than 0, 1/2 and 1: the per-image f32 weight sum would then depend on the order of the
    additions (the warp's lanes against NumPy's pairwise sum), so it could not be compared bit for bit; the reference
    only counts hits where the weight is exactly 1, which these values cover;
  - evaluate_pck's decode (argmax) itself: covered by the decode tests; here heatmaps are whatever argmax finds.
"""
import ctypes
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from litehandnet_b200 import _lib as L
from litehandnet_b200 import metrics as M
from litehandnet_b200 import ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
F32, F64 = np.float32, np.float64
AUC20 = [1.0 * i / 20 for i in range(20)]
PCK4 = [0.05, 0.1, 0.2, 0.5]


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def pck_cap():
    return 8 * sms() * 256


def mpii_cap():
    return 4 * sms() * 256


def n_for(kind, K, cap):
    """Sample counts at the edges of the capped grid: S = cap // K samples fill one pass of the fixed stride S * K."""
    S = cap // K
    return dict(zero=0, one=S, gap=S + 1, four=4 * S + 3, five=5 * S - 1, two=2 * S + 5)[kind]


def assert_gap(K, N, cap):
    assert cap % K != 0 and N * K > cap, (K, N, cap)


def cu(a, dtype=None):
    t = torch.as_tensor(np.ascontiguousarray(a)).to(DEV)
    return t if dtype is None else t.to(dtype)


def offset_view(t, off):
    """t's values in a buffer whose data pointer is `off` elements past an aligned allocation."""
    buf = torch.empty(t.numel() + off, dtype=t.dtype, device=t.device)
    v = buf[off:].view(t.shape)
    v.copy_(t)
    return v


def route(pdt, gdt, ndt, pred_stride=2, aligned=True):
    """The instantiation lhn_pck_accumulate's host rules pick (lhn_metrics.cu, `all_f32` and `fast`)."""
    all_f32 = pdt == "f32" and gdt == "f32" and ndt == "f32"
    if all_f32 and pred_stride == 2 and aligned:
        return "fast"
    return "gen32" if all_f32 else "gen64"


# ---- lhn_pck_accumulate: seeded data with every edge planted ---------------------------------------------------------
def pck_data(N, K, thr, seed, norm_const=None):
    """pred, gt [N,K,2] and the normaliser [N,2] as f64 arrays (cast per case: the oracle sees the same casts), mask
    [N,K].  Distances spread over [0, 0.6] of the normaliser; a fifth of them lie within a few ulps of a threshold,
    so f32 and f64 evaluation disagree about some hits.  Planted, each in a row of its own:
      - normaliser rows: 0 on x, 0 on y, -0, negative on x (-> 1e6), negative on both, NaN on y;
      - predictions NaN, +inf and -inf;
      - on rows with normaliser 1 (or norm_const): distances 2^43 - 2^19 (the largest f32 that the EPE term holds)
        and 2^43 (too large); for each of up to 8 thresholds t a distance of exactly f32(t), and an f64 distance
        f32(t) less an eighth of its ulp (rounds up to f32(t), so no hit) through pred and through gt."""
    rng = np.random.default_rng(seed)
    gt = rng.uniform(0, 256, (N, K, 2)).astype(F32).astype(F64)
    if norm_const is None:
        z = np.repeat(rng.uniform(60, 200, (N, 1)), 2, 1).astype(F32).astype(F64)
    else:
        z = np.full((N, 2), float(norm_const))
    r = rng.uniform(0, 0.6, (N, K))
    if thr:
        t32 = np.asarray(thr, F32).astype(F64)
        near = rng.uniform(0, 1, (N, K)) < 0.2
        r = np.where(near, t32[rng.integers(0, len(thr), (N, K))] * (1 + rng.integers(-6, 7, (N, K)) * 2.0 ** -23), r)
    ang = rng.uniform(0, 2 * np.pi, (N, K))
    pred = gt + np.stack([r * np.cos(ang), r * np.sin(ang)], -1) * z[:, None, :]
    mask = rng.uniform(0, 1, (N, K)) < 0.9
    if N >= 64:
        rows = iter(rng.permutation(N))
        if norm_const is None:
            for v in ((0.0, 150.0), (150.0, 0.0), (-0.0, -0.0), (-5.0, 150.0), (-1.0, -2.0), (150.0, np.nan)):
                z[next(rows)] = v
        for v in ((np.nan, 3.0), (4.0, np.inf), (-np.inf, 1.0)):
            n, k = next(rows), rng.integers(K)
            pred[n, k] = v; mask[n, k] = True
        zc = 1.0 if norm_const is None else float(norm_const)
        unit = [((2.0 ** 43 - 2.0 ** 19) * zc, 0.0, 0.0), (0.0, 2.0 ** 43 * zc, 0.0)]
        for t in sorted(set(np.asarray(thr, F32).tolist()))[:8]:
            t = float(t)
            below = t - np.spacing(F32(t)).item() / 8
            unit += [(t * zc, 0.0, 0.0), (below * zc, 0.0, 0.0), (0.0, 0.0, -below * zc)]
        for px, py, gx in unit:
            n, k = next(rows), rng.integers(K)
            if norm_const is None:
                z[n] = 1.0
            pred[n, k] = (px, py); gt[n, k] = (gx, 0.0); mask[n, k] = True
    return pred, gt, z, mask


def cast(a, dt):
    return a.astype(F32 if dt == "f32" else F64)


def pck_oracle(P, G, mask, thr, Z):
    """(hits[T,K], valid[K], epe_fix[K]) from O.pck_counters and O.epe_fix_counts on the arrays the kernel reads."""
    with np.errstate(all="ignore"):
        if thr:
            hits, valid = O.pck_counters(P, G, mask, thr, Z)
        else:
            hits, valid = np.zeros((0, P.shape[1]), np.int64), None
        d = O.calc_distances(P, G, mask, Z)
    fix = O.epe_fix_counts(d)
    if valid is None:
        valid = (d != -1).sum(axis=1).astype(np.int64)
    return np.concatenate([hits, valid[None], fix[None]]).astype(np.int64)


def categories(P, G, mask, thr, Z):
    """How many counted elements sit exactly on f32(t), how many f64 distances lie below f32(t) and round up to it, and
    how many hits the f32 and the f64 evaluation of the same values disagree about."""
    if not thr:
        return 0, 0, 0
    with np.errstate(all="ignore"):
        d = O.calc_distances(P, G, mask, Z)
        d32 = O.calc_distances(P.astype(F32), G.astype(F32), mask, Z.astype(F32))
        d64 = O.calc_distances(P.astype(F64), G.astype(F64), mask, Z.astype(F64))
        zz = np.asarray(Z, F64).copy()
        zz[zz <= 0] = 1e6
        q = (P.astype(F64) - G.astype(F64)) / zz[:, None, :]
        exact = np.sqrt((q * q).sum(-1)).T                          # the f64 distance before its rounding to f32
    valid = d != -1
    ties = roundup = disagree = 0
    for t in thr:
        t32 = F32(t)
        ties += int((valid & (d == t32)).sum())
        roundup += int((valid & (exact < float(t32)) & (exact.astype(F32) == t32)).sum())
        disagree += int((valid & ((d32 < t32) != (d64 < t32))).sum())
    return ties, roundup, disagree


def run_pck(P, G, mask, thr, Z, norm_const, how):
    """Counters of one lhn_pck_accumulate call on the cast arrays; `how` picks the layout (contiguous, pred through a
    4-byte-offset view, or pred with a third column)."""
    p = cu(P)
    if how == "offset":
        p = offset_view(p, 1)
        assert p.numel() == 0 or p.data_ptr() % 8 == 4                  # an empty view has no data pointer
    elif how == "stride3":
        p = cu(np.concatenate([P, np.full(P.shape[:2] + (1,), 7.0, P.dtype)], -1))
    z = None if Z is None else cu(Z)
    K = P.shape[1]
    out = ops.pck_accumulate(p, cu(G), cu(mask), thr, z, 1.0 if norm_const is None else norm_const)
    return out.cpu().numpy().reshape(len(thr) + 2, K)


def assert_counters(got, want, what):
    if not np.array_equal(got, want):
        bad = np.argwhere(got != want)[:6].tolist()
        raise AssertionError(f"{what}: counters differ at [row, joint] {bad}: got {got[tuple(np.array(bad).T)]} "
                             f"want {want[tuple(np.array(bad).T)]}")


def check_categories(P, G, mask, thr, Z, pdt, gdt, ndt, norm_const):
    """The planted edges are really in the data: a `<=` for `<`, a comparison before the rounding to f32 or the other
    promotion would change a counter."""
    ties, roundup, disagree = categories(P, G, mask, thr, Z)
    if not thr:
        return
    if max(thr) > 0:                                                      # nothing is below a threshold of 0
        assert disagree > 0, "no element where f32 and f64 promotion disagree about a hit"
    if norm_const is None or pdt == "f64":
        assert ties > 0, "no distance exactly on a threshold"
    if "f64" in (pdt, gdt) and max(thr) > 0:
        assert roundup > 0, "no f64 distance below a threshold that rounds up to it"


SHAPE_K = (1, 16, 17, 21, 62)
SHAPE_N = ("one", "gap", "four", "five", "zero")


@pytest.mark.parametrize("nkind", SHAPE_N)
@pytest.mark.parametrize("K", SHAPE_K)
def test_pck_accumulate_shapes_and_paths(K, nkind):
    """Every path at the edges of the capped grid: FAST (all f32, strides 2, aligned), the general instantiation on the
    same f32 data (pred through a 4-byte offset, and pred at stride 3) and the general f64 one.  All three counter
    rows equal the oracle's, and FAST equals the general all-f32 instantiation."""
    cap = pck_cap()
    N = n_for(nkind, K, cap)
    if nkind in ("gap", "four", "five") and K in (17, 21, 62):
        assert_gap(K, N, cap)
    thr = PCK4
    pred, gt, z, mask = pck_data(N, K, thr, seed=1000 + 10 * K + SHAPE_N.index(nkind))
    P, G, Z = cast(pred, "f32"), cast(gt, "f32"), cast(z, "f32")
    want = pck_oracle(P, G, mask, thr, Z)
    fast = run_pck(P, G, mask, thr, Z, None, "plain")
    assert route("f32", "f32", "f32") == "fast"
    assert_counters(fast, want, "fast")
    for how in ("offset", "stride3"):
        assert route("f32", "f32", "f32", 3 if how == "stride3" else 2, how != "offset") == "gen32"
        assert_counters(run_pck(P, G, mask, thr, Z, None, how), fast, f"general all-f32 ({how}) against fast")
    P64 = cast(pred, "f64")
    assert route("f64", "f32", "f32") == "gen64"
    assert_counters(run_pck(P64, G, mask, thr, Z, None, "plain"), pck_oracle(P64, G, mask, thr, Z), "general f64")
    if N:
        check_categories(P, G, mask, thr, Z, "f32", "f32", "f32", None)
        check_categories(P64, G, mask, thr, Z, "f64", "f32", "f32", None)
    else:
        assert not fast.any()


DT_CASES = [(p, g, n) for p in ("f32", "f64") for g in ("f32", "f64") for n in ("f32", "f64")] + \
           [("f32", "f32", None), ("f64", "f32", None)]


@pytest.mark.parametrize("pdt,gdt,ndt", DT_CASES, ids=lambda v: str(v))
def test_pck_accumulate_dtypes(pdt, gdt, ndt):
    """All eight f32/f64 combinations of pred, gt and normaliser, and no normaliser with norm_const = 30 (the AUC
    caller, promoted to f64 like NumPy's python float), at K = 21 one sample past the gap."""
    K = 21
    cap = pck_cap()
    N = n_for("gap", K, cap)
    assert_gap(K, N, cap)
    norm_const = 30.0 if ndt is None else None
    thr = AUC20 if ndt is None else [0.2]
    pred, gt, z, mask = pck_data(N, K, thr, seed=2000 + DT_CASES.index((pdt, gdt, ndt)), norm_const=norm_const)
    P, G = cast(pred, pdt), cast(gt, gdt)
    Z = cast(z, ndt) if ndt else None
    Zo = Z if ndt else np.full((N, 2), norm_const)
    want = pck_oracle(P, G, mask, thr, Zo)
    got = run_pck(P, G, mask, thr, Z, norm_const, "plain")
    assert_counters(got, want, f"{route(pdt, gdt, ndt or 'f64')}")
    check_categories(P, G, mask, thr, Zo, pdt, gdt, ndt or "f64", norm_const)


_rs = np.random.default_rng(5)
THR_CASES = dict(
    t0=[],
    t1=[0.2],
    t1_zero=[0.0],
    t1_one=[1.0],
    auc20=AUC20,
    duplicated=[0.1, 0.1, 0.2, 0.2, 0.2, 0.5],
    descending=[0.5, 0.2, 0.1, 0.05],
    shuffled=[AUC20[i] for i in _rs.permutation(20)],
    t64=[float(t) for t in np.linspace(0.0, 1.0, 64)],
)


@pytest.mark.parametrize("name", list(THR_CASES))
def test_pck_accumulate_thresholds(name):
    """T = 0 (EPE only), one threshold (a register count) at 0, 0.2 and 1, the 20 AUC steps (the histogram), duplicated
    thresholds, descending and shuffled ones (one shared add per threshold passed) and T = 64 at K = 62, the most
    joints whose shared memory fits — on the FAST and the general f64 path, past the gap."""
    thr = THR_CASES[name]
    K = 62 if len(thr) == 64 else 21
    cap = pck_cap()
    N = n_for("gap", K, cap)
    assert_gap(K, N, cap)
    pred, gt, z, mask = pck_data(N, K, thr, seed=3000 + list(THR_CASES).index(name))
    G, Z = cast(gt, "f32"), cast(z, "f32")
    for pdt in ("f32", "f64"):
        P = cast(pred, pdt)
        assert_counters(run_pck(P, G, mask, thr, Z, None, "plain"), pck_oracle(P, G, mask, thr, Z),
                        f"{route(pdt, 'f32', 'f32')} T={len(thr)}")
        check_categories(P, G, mask, thr, Z, pdt, "f32", "f32", None)


@pytest.mark.parametrize("what", ["norm_const_zero", "mask_all_false"])
def test_pck_accumulate_masks_everything(what):
    """norm_const = 0 masks every row (`normalize == 0`), as a mask of all False does: no hit, no valid count, no EPE."""
    K = 21
    N = n_for("gap", K, pck_cap())
    pred, gt, z, mask = pck_data(N, K, AUC20, seed=4000)
    P, G = cast(pred, "f32"), cast(gt, "f64")
    if what == "mask_all_false":
        mask[:] = False
        got = run_pck(P, G, mask, AUC20, cast(z, "f32"), None, "plain")
        want = pck_oracle(P, G, mask, AUC20, cast(z, "f32"))
    else:
        got = run_pck(P, G, mask, AUC20, None, 0.0, "plain")
        want = pck_oracle(P, G, mask, AUC20, np.zeros((N, 2)))
    assert not want.any()
    assert_counters(got, want, what)


def test_pck_accumulate_refuses():
    """T = 65, shared memory over 48 KB (K = 63 at T = 64; K = 62 fits) and a null threshold list with T > 0 are
    refused, and the counters are left untouched."""
    N, K = 100, 63
    p = torch.zeros((N, K, 2), dtype=torch.float32, device=DEV)
    m = torch.ones((N, K), dtype=torch.bool, device=DEV)
    ones = torch.ones((N, 2), dtype=torch.float32, device=DEV)
    cnt = torch.full((66 * K,), 7, dtype=torch.int64, device=DEV)
    with pytest.raises(L.LhnError):
        ops.pck_accumulate(p[:, :1], p[:, :1], m[:, :1], [0.1] * 65, ones, counters=cnt[:67])
    with pytest.raises(L.LhnError):
        ops.pck_accumulate(p, p, m, [0.1] * 64, ones, counters=cnt)
    mu8 = m.to(torch.uint8)
    rc = L.lib().lhn_pck_accumulate(L.ptr(p), L.F32, 2, L.ptr(p), L.F32, 2, L.ptr(mu8), L.ptr(ones), L.F32, 1.0, N, K,
                                    None, 1, L.ptr(cnt), L.stream())
    assert rc == -1
    torch.cuda.synchronize()
    assert bool((cnt == 7).all())
    ok = ops.pck_accumulate(p[:, :62], p[:, :62], m[:, :62], [0.1] * 64, ones)
    assert ok.view(66, 62)[64].sum().item() == N * 62


def test_pck_accumulate_sharded_equals_monolithic():
    """Uneven shards, one of them past the cap itself, added into one counter block equal the monolithic block and the
    oracle (FAST path, K = 21)."""
    K = 21
    cap = pck_cap()
    S = cap // K
    N = n_for("two", K, cap)
    assert_gap(K, N, cap)
    assert_gap(K, S + 3, cap)
    pred, gt, z, mask = pck_data(N, K, AUC20, seed=5000)
    P, G, Z = cast(pred, "f32"), cast(gt, "f32"), cast(z, "f32")
    mono = run_pck(P, G, mask, AUC20, Z, None, "plain")
    assert_counters(mono, pck_oracle(P, G, mask, AUC20, Z), "monolithic")
    acc = torch.zeros((len(AUC20) + 2) * K, dtype=torch.int64, device=DEV)
    for a, b in ((0, 7), (7, S + 10), (S + 10, N - 1), (N - 1, N)):
        ops.pck_accumulate(cu(P[a:b]), cu(G[a:b]), cu(mask[a:b]), AUC20, cu(Z[a:b]), counters=acc)
    assert_counters(acc.cpu().numpy().reshape(-1, K), mono, "sharded")


# ---- lhn_mpii_pckh_accumulate ---------------------------------------------------------------------------------------
def mpii_data(N, K, seed):
    """preds [N,K,2] f32 (0-based) and the mpii_gt_val arrays (1-based ground truth, head boxes, jnt_missing), with
    planted: exact `<=` boundaries (head box 6 x 8 -> norm 10, offsets (1.5, 2), (0.75, 1), (0.375, 0.5) give ratios
    0.5, 0.25 and 0.125 at sc_bias 0.5), zero-size head boxes (ratio inf, or NaN for a perfect prediction), invisible
    joints."""
    rng = np.random.default_rng(seed)
    gt = np.round(rng.uniform(20, 200, (N, K, 2)))                        # integers: pred + 1 - gt is exact below
    off = rng.normal(0, 4, (N, K, 2))
    pred = (gt - 1 + off).astype(F32)
    x1 = np.round(rng.uniform(0, 100, N)); y1 = np.round(rng.uniform(0, 100, N))
    head = np.stack([x1, y1, x1 + np.round(rng.uniform(8, 40, N)), y1 + np.round(rng.uniform(8, 40, N))], 1)
    missing = (rng.uniform(0, 1, (N, K)) < 0.1).astype(F64)
    rows = rng.permutation(N)
    for i, (dx, dy) in enumerate(((1.5, 2.0), (0.75, 1.0), (0.375, 0.5), (1.5, 2.0))):
        n = rows[i]
        head[n] = (x1[n], y1[n], x1[n] + 6, y1[n] + 8)
        pred[n] = (gt[n] - 1 + np.array([dx, dy])).astype(F32)
        missing[n] = 0
    for n in rows[4:7]:
        head[n] = (x1[n], y1[n], x1[n], y1[n])
        missing[n] = 0
    n = rows[7]
    head[n] = (x1[n], y1[n], x1[n], y1[n])
    pred[n] = (gt[n] - 1).astype(F32)
    missing[n] = 0
    gtd = dict(jnt_missing=missing.T, pos_gt_src=np.transpose(gt, (1, 2, 0)),
               headboxes_src=np.stack([head[:, :2].T, head[:, 2:].T]))
    return pred, gtd


MPII_EXTRA = [0.25, 0.125, float(np.nextafter(0.5, 0)), float(np.nextafter(0.25, 0))]
MpiiCase = namedtuple("MpiiCase", "K stride sc_bias thr")
MPII_CASES = dict(
    k16_s2=MpiiCase(16, 2, 0.5, M.MPII_THRESHOLDS + MPII_EXTRA),
    k16_s3=MpiiCase(16, 3, 0.6, M.MPII_THRESHOLDS),
    k21_s2=MpiiCase(21, 2, 0.6, M.MPII_THRESHOLDS),
    k21_s3=MpiiCase(21, 3, 0.5, M.MPII_THRESHOLDS + MPII_EXTRA),
    k21_t64=MpiiCase(21, 2, 0.5, [float(t) for t in np.linspace(0.0, 0.63, 64)]),
)


@pytest.mark.parametrize("name", list(MPII_CASES))
def test_mpii_pckh_accumulate(name):
    """hits[T][K] and count[K] equal O.mpii_pckh_counters (tied to O.mpii_pckh on the golden file by a CPU test) at
    N past the capped grid, pred strides 2 and 3, the real threshold list, exact `<=` boundaries, zero-size heads and
    invisible joints; T = 64 is accepted."""
    c = MPII_CASES[name]
    cap = mpii_cap()
    N = n_for("two", c.K, cap)
    assert N * c.K > cap
    pred, gtd = mpii_data(N, c.K, seed=6000 + list(MPII_CASES).index(name))
    hits, count = O.mpii_pckh_counters(pred, gtd, c.thr, c.sc_bias)
    p = pred if c.stride == 2 else np.concatenate([pred, np.full((N, c.K, 1), 0.5, F32)], -1)
    got = M.mpii_pckh_counters(cu(p), gtd, c.thr, sc_bias=c.sc_bias).cpu().numpy().reshape(len(c.thr) + 1, c.K)
    assert_counters(got, np.concatenate([hits, count[None]]), name)
    assert count.sum() < N * c.K                                           # invisible joints are left out
    if c.sc_bias == 0.5 and MPII_EXTRA[2] in c.thr:
        i5, ib = c.thr.index(0.5), c.thr.index(float(np.nextafter(0.5, 0)))
        assert (hits[i5] - hits[ib]).sum() >= c.K * 2                       # the planted ratios of exactly 0.5 (`<=`)


def test_mpii_pckh_accumulate_refuses():
    N, K = 40, 16
    pred, gtd = mpii_data(N, K, seed=7)
    for thr, sc in (([0.1] * 65, 0.6), ([0.5], 0.0), ([0.5], -1.0)):
        with pytest.raises(L.LhnError):
            M.mpii_pckh_counters(cu(pred), gtd, thr, sc_bias=sc)
    M.mpii_pckh_counters(cu(pred), gtd, [0.1] * 64)


# ---- lhn_evaluate_pck ----------------------------------------------------------------------------------------------
EvalCase = namedtuple("EvalCase", "K B H dtype weights")
EVAL_CASES = dict(
    k16_b7_f32=EvalCase(16, 7, 64, "f32", None),
    k21_b13_bf16=EvalCase(21, 13, 64, "bf16", "half"),
    k42_b5_f16=EvalCase(42, 5, 32, "f16", "zero_image"),
    k42_b9_f32=EvalCase(42, 9, 64, "f32", "half"),
    k16_b1_f16=EvalCase(16, 1, 32, "f16", None),
    k21_b6001_f32=EvalCase(21, 6001, 16, "f32", "zero_image"),
    k21_b4099_bf16=EvalCase(21, 4099, 16, "bf16", None),
)
TDT = dict(f32=torch.float32, bf16=torch.bfloat16, f16=torch.float16)


@pytest.mark.parametrize("name", list(EVAL_CASES))
def test_evaluate_pck(name):
    """Per-image values and the mean bit-equal to the oracle.  Each per-image value is hits / sum(w), an f32 in [0, 2]
    whose smallest nonzero value is at least 1/(2K), so it is a multiple of 2^-31 and B of them (< 2^20) sum exactly
    in f64 in any order; `/ B` then rounds once, as np.mean does.  With weights in {0, 1/2, 1} the f32 weight sums
    are exact too.  K = 42 makes the per-image warp loop over the joints twice."""
    c = EVAL_CASES[name]
    seed = 8000 + list(EVAL_CASES).index(name)
    hm, cen = synth.blob_heatmaps(c.B, c.K, c.H, c.H, seed=seed, device=DEV, margin=1.0)
    g = torch.Generator(device=DEV).manual_seed(seed)
    gcen = (cen + torch.randn(cen.shape, generator=g, device=DEV) * 1.5).cpu()
    ghm, _ = synth.blob_heatmaps(c.B, c.K, c.H, c.H, seed=seed + 1, device=DEV, centers=gcen)
    hm, ghm = hm.to(TDT[c.dtype]), ghm.to(TDT[c.dtype])
    rng = np.random.default_rng(seed)
    wh = rng.uniform(40, 200, (c.B, 2)).astype(F32)
    if c.B > 1:
        assert (wh[:, 0] > wh[:, 1]).any() and (wh[:, 0] < wh[:, 1]).any()
    bbox = np.zeros((c.B, 1, 4), F32); bbox[:, 0, 2:] = wh
    w = None
    if c.weights:
        w = rng.choice(np.array([0.0, 0.5, 1.0], F32), (c.B, c.K), p=[0.15, 0.15, 0.7])
        if c.weights == "zero_image":
            w[c.B // 2] = 0.0
    with np.errstate(all="ignore"):
        want_mean, want = O.evaluate_pck(hm.float().cpu().numpy(), ghm.float().cpu().numpy(), bbox, 256, w, 0.2,
                                         per_image=True)
    pck, mean = ops.evaluate_pck(hm, ghm, cu(wh), None if w is None else cu(w), (256, 256), 0.2)
    got = pck.cpu().numpy()
    same = (got.view(np.int32) == want.view(np.int32)) | (np.isnan(got) & np.isnan(want))
    assert same.all(), (np.argwhere(~same)[:5].tolist(), got[~same][:5], want[~same][:5])
    m = mean.cpu().numpy()[0]
    assert m == want_mean or (np.isnan(m) and np.isnan(want_mean)), (m, want_mean)
    if c.weights == "zero_image":
        assert np.isnan(got[c.B // 2]) and np.isnan(m)
    if c.B > 1:
        assert np.nanmax(got) > 0 and np.nanmin(got) < np.nanmax(got)     # a mix of hits and misses


# ---- the fused counters against three lhn_pck_accumulate calls, at the gap ---------------------------------------
def test_fused_counters_equal_pck_accumulate_at_the_gap(monkeypatch):
    """MetricAccumulator.update_from_heatmaps (the team kernel, and the CTA-per-plane kernel) against update_from_preds
    (three lhn_pck_accumulate calls on the kernel's own keypoints) and against the oracle on those keypoints, at K = 21
    one sample past the gap, with negative and zero boxes and one sample with an inf centre (EPE rule)."""
    K, H = 21, 16
    cap = pck_cap()
    N = n_for("gap", K, cap)
    assert_gap(K, N, cap)
    hm, cen = synth.blob_heatmaps(N, K, H, H, seed=91, device=DEV, margin=2.0)
    center, scale = synth.bbox_center_scale(N, fixed=True, device=DEV)
    gt, mask, wh = synth.pck_inputs(cen, stride=256 / H, seed=92, device=DEV)
    wh[5:9] = -wh[5:9]
    wh[11] = 0.0
    center[N - 3, 0] = float("inf")
    want = None
    for env, path in (({}, 1), ({"LHN_FORCE_CTA_KERNEL": "1"}, 2)):
        monkeypatch.delenv("LHN_FORCE_CTA_KERNEL", raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        fused = M.MetricAccumulator(K, device=DEV)
        r = fused.update_from_heatmaps(hm, center, scale, gt, mask, wh)
        info = L.K1LaunchInfo()
        L.check(L.lib().lhn_k1_last_launch(ctypes.byref(info)), "lhn_k1_last_launch")
        assert info.path == path
        kp = r["kpts"][..., :2]
        assert torch.isinf(kp[N - 3, :, 0]).all()
        from_preds = M.MetricAccumulator(K, device=DEV)
        from_preds.update_from_preds(r["kpts"], gt, mask, wh)
        got_f = fused.counters.cpu().numpy().reshape(-1, K)
        got_p = from_preds.counters.cpu().numpy().reshape(-1, K)
        kp64 = kp.double().cpu().numpy()
        g, m = gt.cpu().numpy(), mask.cpu().numpy()
        t = wh.max(1).values.double().cpu().numpy()
        pck = pck_oracle(kp64, g, m, [0.2], np.stack([t, t], 1))
        auc = pck_oracle(kp64, g, m, AUC20, np.full((N, 2), 30.0))
        epe = pck_oracle(kp64, g, m, [], np.ones((N, 2), F32))
        exp = np.concatenate([pck[:2], auc[:21], epe])
        assert_counters(got_p, exp, f"update_from_preds (path {path})")
        assert_counters(got_f, exp, f"update_from_heatmaps (path {path})")
        if want is not None:
            assert np.array_equal(got_f, want)
        want = got_f
    assert want[-1].min() >= 0
