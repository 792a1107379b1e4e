"""GPU: every SimDR kernel path — target render, decode, loss, backward and the fused heads — against the f64 oracle.

The host code picks a kernel per call from the shape, the alignment and environment switches (LHN_SIMDR_RING,
LHN_SIMDR_WARPS, LHN_SIMDR_STAGES, LHN_SIMDR_LOSS_PATH, LHN_HEADS_BN; all read on every call).  Each case below names
its inputs AND the launch record (`lhn_simdr_last_launch`) they must produce, so a policy change fails here instead of
silently moving what the suite covers.  Every comparison is either bit for bit against the oracle's own arithmetic or
within a bound derived (in a comment next to it) from the operations the kernel performs, and each bound comes with an
assertion that it is tight enough to see a plausible bug (a dropped k-block, a neighbouring joint's coefficient).

Reachable paths the tables leave out, and why:
  - decode, ring kernel with NMS or `ranges`: the ring is never taken with NMS (the NMS rows run the grid-stride kernel);
  - decode, ring kernel at 2 to 32 warps other than 1/8/16/24: same code, the warp count only changes the grid;
  - loss, the joint kernel's workspace guard (warps * 24 bytes > workspace): the workspace of B*K*16 bytes always holds
    the at most B*K/4.9 entries the grid sizing produces, so the guard cannot fail for a correctly sized workspace;
  - render, the non-vector path reached by a misaligned output: ops.render_simdr allocates the outputs; the plain path
    is reached through the window width (sigma 9.7) and through Lx % 4 != 0 instead.
"""
import ctypes
import math
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from litehandnet_b200 import _lib as L
from litehandnet_b200 import ops

pytestmark = pytest.mark.gpu
DEV = "cuda"
F32, F64 = np.float32, np.float64
DT = dict(f32=torch.float32, bf16=torch.bfloat16, f16=torch.float16)
DCODE = dict(f32=L.F32, bf16=L.BF16, f16=L.F16)
U = 2.0 ** -24                                   # f32 unit roundoff
U_T = dict(f32=2.0 ** -24, bf16=2.0 ** -8, f16=2.0 ** -11)        # unit roundoff of the stored type
SUB_T = dict(f32=2.0 ** -150, bf16=2.0 ** -134, f16=2.0 ** -25)   # half the smallest subnormal of the stored type
ENV = ("LHN_SIMDR_RING", "LHN_SIMDR_WARPS", "LHN_SIMDR_STAGES", "LHN_SIMDR_LOSS_PATH", "LHN_HEADS_BN")
FAMILY = dict(render=1, decode=2, loss=3, backward=4, heads=5)


def report(what, ratio):
    """The largest error seen as a fraction of its bound (shown with pytest -s)."""
    print(f"bound-ratio {what}: {ratio:.4g}")


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def record():
    r = L.SimdrLaunchInfo()
    L.check(L.lib().lhn_simdr_last_launch(ctypes.byref(r)), "lhn_simdr_last_launch")
    return {n: getattr(r, n) for n, _ in L.SimdrLaunchInfo._fields_}


def set_env(monkeypatch, env):
    for n in ENV:
        monkeypatch.delenv(n, raising=False)
    for n, v in env.items():
        monkeypatch.setenv(n, str(v))


def assert_bits(got, want, what):
    """Bit-for-bit f32 equality (the sign of zero included); any NaN matches any NaN."""
    g = np.ascontiguousarray(got, dtype=F32)
    w = np.ascontiguousarray(want, dtype=F32)
    assert g.shape == w.shape, (what, g.shape, w.shape)
    bad = (g.view(np.int32) != w.view(np.int32)) & ~(np.isnan(g) & np.isnan(w))
    if bad.any():
        at = np.argwhere(bad)[:5]
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} differ, first at {at.tolist()}: "
                             f"got {g[bad][:5]} want {w[bad][:5]}")


def offset_view(t, off):
    """t's values in a fresh buffer whose data pointer is `off` elements past an aligned allocation."""
    if not off:
        return t.contiguous()
    buf = torch.empty(t.numel() + off, dtype=t.dtype, device=t.device)
    v = buf[off:].view(t.shape)
    v.copy_(t)
    return v


def to_dt(a, dt):
    """(device tensor of dtype dt, the f32 values it holds as NumPy)."""
    t = torch.from_numpy(np.ascontiguousarray(a, F32)).to(DEV).to(DT[dt])
    return t, t.float().cpu().numpy()


# ================================================ decode ============================================================
# Values planted in row r of every case, pattern r % len(PATTERNS), on both the x- and the y-vector.  Positions are
# fractions of L so that the same patterns apply to L = 1 .. 768 (at small L they may coincide; the oracle decides).
def _plant(v, p):
    n = v.shape[0]
    at = lambda f: min(n - 1, int(f * n))           # noqa: E731
    nan, inf = np.nan, np.inf
    if p == 1:                                       # NaN first seen in a later quad than a larger finite value
        v[at(0.05)] = 100.0; v[at(0.9)] = nan
    elif p == 2:                                     # NaNs in several lanes: the first one wins
        v[at(0.6)] = nan; v[at(0.3)] = nan; v[at(0.8)] = nan
    elif p == 3:                                     # NaN at L - 1
        v[n - 1] = nan
    elif p == 4:                                     # all -inf: index 0, score -inf
        v[:] = -inf
    elif p == 5:                                     # +inf ties
        v[at(0.2)] = inf; v[at(0.7)] = inf
    elif p == 6:                                     # -0 then +0 as the maxima: index of the -0, score -0
        v[:] = -np.abs(v) - 1; v[at(0.1)] = -0.0; v[at(0.5)] = 0.0
    elif p == 7:                                     # +0 then -0
        v[:] = -np.abs(v) - 1; v[at(0.1)] = 0.0; v[at(0.5)] = -0.0
    elif p == 8:                                     # equal maxima in lane 31 of quad q and lane 0 of quad q + 1
        i = 127 if n > 128 else max(0, n // 2 - 1)
        v[i] = 50.0; v[min(n - 1, i + 1)] = 50.0
    elif p == 9:                                     # the same across the scalar scan's lanes 31 | 0
        i = 31 if n > 32 else max(0, n // 2 - 1)
        v[i] = 40.0; v[min(n - 1, i + 1)] = 40.0
    elif p == 10:                                    # maximum at 0
        v[0] = 60.0
    elif p == 11:                                    # maximum at L - 1
        v[n - 1] = 60.0


N_PATTERNS = 12


def simdr_vectors(B, K, Lx, Ly, seed):
    g = np.random.default_rng(seed)
    xv = g.standard_normal((B, K, Lx)).astype(F32)
    yv = g.standard_normal((B, K, Ly)).astype(F32)
    for r in range(B * K):
        b, j = divmod(r, K)
        _plant(xv[b, j], r % N_PATTERNS)
        _plant(yv[b, j], r % N_PATTERNS)
    return xv, yv


def ranges_for(B, Lx, Ly):
    """x1 = x2 (an empty window), x2 > L (clipped by the kernel and by numpy's slice) and the whole vector, in turn."""
    r = np.zeros((B, 4), np.int32)
    for b in range(B):
        m = b % 3
        if m == 0:
            r[b] = (Lx // 3, Lx // 3, Ly // 2, Ly // 2)
        elif m == 1:
            r[b] = (Lx // 3, Lx + 7, Ly // 4, Ly + 100)
        else:
            r[b] = (0, Lx, 0, Ly)
    return r


def decode_oracle(xv, yv, k, center, scale, nms, ranges):
    """(out [B,K,3] f32, idx [B,K,2]) from the oracle's own arithmetic."""
    with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
        if nms:
            nx, ny = O.vector_nms(xv), O.vector_nms(yv)
            B, K, Lx = xv.shape
            Ly = yv.shape[2]
            rg = ranges if ranges is not None else np.tile(np.array([0, Lx, 0, Ly], np.int32), (B, 1))
            mx = np.zeros((B, 1, Lx), bool); my = np.zeros((B, 1, Ly), bool)
            for b in range(B):
                mx[b, 0, rg[b, 0]:rg[b, 1]] = True; my[b, 0, rg[b, 2]:rg[b, 3]] = True
            idx = np.stack([np.argmax(nx * mx, 2), np.argmax(ny * my, 2)], 2)
            return O.coordinates_from_vectors(xv, yv, rg, k), idx
        idx = np.stack([np.argmax(xv, 2), np.argmax(yv, 2)], 2)
        if center is not None:
            return O.keypoints_from_simdr(xv, yv, center, scale, k), idx
        # keypoints_from_simdr without transform_preds (k >= 2^24 or L < k leave no output size to transform to)
        xm = np.take_along_axis(xv, idx[..., :1], 2); ym = np.take_along_axis(yv, idx[..., 1:], 2)
        preds = (idx / k).astype(F32)
        return np.concatenate([preds, ((xm + ym) / 2).astype(F32)], 2), idx


# name, dtype, B, K, Lx, Ly, split ratio k, environment, base offset (elements), nms, ranges, transform_preds,
# expected record (path, warps, stages).  ctas and the dtype follow from the inputs and are checked as well.
D_ = namedtuple("D_", "name dt B K Lx Ly k env off nms ranges xform rec")
RING1 = {"LHN_SIMDR_WARPS": 1}            # the ring needs only 148 * 1 * 4 = 592 pairs at one warp per CTA
DCASES = [
    # ---- the TMA ring kernel: warps x stages, dtypes, Lx != Ly, split ratios -----------------------------------
    D_("ring-w1-s2", "f32", 29, 21, 512, 512, 2, dict(RING1, LHN_SIMDR_STAGES=2), 0, False, None, True, (1, 1, 2)),
    D_("ring-w1-s3", "f32", 29, 21, 512, 512, 2, dict(RING1, LHN_SIMDR_STAGES=3), 0, False, None, True, (1, 1, 3)),
    D_("ring-w1-s4", "f32", 29, 21, 512, 512, 2, RING1, 0, False, None, True, (1, 1, 4)),
    D_("ring-w8", "f32", 226, 21, 512, 512, 2, {"LHN_SIMDR_WARPS": 8}, 0, False, None, True, (1, 8, 4)),
    D_("ring-w8-s2", "f32", 226, 21, 512, 512, 2, {"LHN_SIMDR_WARPS": 8, "LHN_SIMDR_STAGES": 2}, 0, False, None, True,
       (1, 8, 2)),
    D_("ring-w16-default", "f32", 452, 21, 512, 512, 2, {}, 0, False, None, True, (1, 16, 3)),
    D_("ring-w16-s2", "f32", 452, 21, 512, 512, 2, {"LHN_SIMDR_STAGES": 2}, 0, False, None, True, (1, 16, 2)),
    D_("ring-w24", "f32", 677, 21, 512, 512, 2, {"LHN_SIMDR_WARPS": 24}, 0, False, None, True, (1, 24, 2)),
    # a 6 KB pair leaves the default 16-warp ring exactly two stages
    D_("ring-768-two-stages", "f32", 452, 21, 768, 768, 2, {}, 0, False, None, True, (1, 16, 2)),
    D_("ring-bf16", "bf16", 29, 21, 512, 512, 2, RING1, 0, False, None, True, (1, 1, 4)),
    D_("ring-f16", "f16", 29, 21, 512, 512, 2, RING1, 0, False, None, True, (1, 1, 4)),
    D_("ring-lx>ly-k3", "f32", 29, 21, 512, 256, 3, RING1, 0, False, None, True, (1, 1, 4)),
    D_("ring-lx<ly-k1", "bf16", 29, 21, 256, 512, 1, RING1, 0, False, None, True, (1, 1, 4)),
    D_("ring-k4-not-pow2-out", "f16", 29, 21, 384, 640, 4, RING1, 0, False, None, True, (1, 1, 4)),
    D_("ring-k-2^24+3", "f32", 29, 21, 512, 512, 2 ** 24 + 3, RING1, 0, False, None, False, (1, 1, 4)),
    D_("ring-k-2^25", "f32", 29, 21, 512, 512, 2 ** 25, RING1, 0, False, None, False, (1, 1, 4)),
    # ---- the grid-stride pair scan: small batches, the ring switched off, vectors TMA cannot copy -----------------
    D_("pair-f32", "f32", 2, 21, 512, 512, 2, {}, 0, False, None, True, (2, 8, 0)),
    D_("pair-bf16-k3", "bf16", 2, 21, 384, 256, 3, {}, 0, False, None, True, (2, 8, 0)),
    D_("pair-f16", "f16", 2, 21, 256, 384, 2, {}, 0, False, None, True, (2, 8, 0)),
    D_("pair-L4-L8", "f32", 3, 21, 4, 8, 1, {}, 0, False, None, True, (2, 8, 0)),
    D_("pair-ring-off", "f32", 29, 21, 512, 512, 2, dict(RING1, LHN_SIMDR_RING=0), 0, False, None, True, (2, 8, 0)),
    D_("pair-bf16-520-byte-rows", "bf16", 29, 21, 260, 512, 2, RING1, 0, False, None, True, (2, 8, 0)),
    D_("pair-k-2^24", "f32", 2, 21, 512, 512, 2 ** 24, {}, 0, False, None, False, (2, 8, 0)),
    # ---- the scalar scan: L % 4 != 0, or a base one element off alignment ---------------------------------------
    D_("scalar-L1-L2", "f32", 3, 21, 1, 2, 1, {}, 0, False, None, True, (3, 8, 0)),
    D_("scalar-L3", "bf16", 3, 21, 3, 3, 1, {}, 0, False, None, True, (3, 8, 0)),
    D_("scalar-L5-L7", "f16", 3, 21, 5, 7, 2, {}, 0, False, None, True, (3, 8, 0)),
    D_("scalar-offset-f32-ring-size", "f32", 29, 21, 512, 512, 2, RING1, 1, False, None, True, (3, 8, 0)),
    D_("scalar-offset-bf16", "bf16", 2, 21, 512, 256, 2, {}, 1, False, None, True, (3, 8, 0)),
    D_("scalar-k-2^24+1", "f16", 2, 21, 6, 8, 2 ** 24 + 1, {}, 0, False, None, False, (3, 8, 0)),
    # ---- vector_nms, with and without the bbox ranges ----------------------------------------------------------
    D_("nms-f32", "f32", 6, 21, 512, 512, 2, {}, 0, True, None, False, (4, 8, 0)),
    D_("nms-ranges-f32", "f32", 6, 21, 512, 384, 2, {}, 0, True, "mixed", False, (4, 8, 0)),
    D_("nms-ranges-bf16-odd", "bf16", 6, 21, 255, 130, 3, {}, 0, True, "mixed", False, (4, 8, 0)),
    D_("nms-ranges-f16-L1", "f16", 6, 21, 1, 4, 1, {}, 0, True, "mixed", False, (4, 8, 0)),
    D_("nms-ring-size", "f32", 29, 21, 512, 512, 2, RING1, 0, True, "mixed", False, (4, 8, 0)),
]


@pytest.mark.parametrize("c", DCASES, ids=[c.name for c in DCASES])
def test_decode_case(c, monkeypatch):
    """Bit for bit against keypoints_from_simdr / coordinates_from_vectors: coordinates and score as int32 bit
    patterns (the sign of zero included: the score carries the sign of the element at the first maximal index, on
    every path; any NaN matches any NaN), the indices exactly."""
    set_env(monkeypatch, c.env)
    xv, yv = simdr_vectors(c.B, c.K, c.Lx, c.Ly, seed=zlib.crc32(c.name.encode()))
    xt, xv = to_dt(xv, c.dt)
    yt, yv = to_dt(yv, c.dt)
    xt, yt = offset_view(xt, c.off), offset_view(yt, c.off)
    g = np.random.default_rng(7)
    center = (g.uniform(50, 200, (c.B, 2)).astype(F32) if c.xform else None)
    scale = (g.uniform(0.5, 2.0, (c.B, 2)).astype(F32) if c.xform else None)
    rg = ranges_for(c.B, c.Lx, c.Ly) if c.ranges else None
    out, idx = ops.decode_simdr(xt, yt, c.k, None if center is None else torch.from_numpy(center).to(DEV),
                                None if scale is None else torch.from_numpy(scale).to(DEV), nms=c.nms,
                                ranges=None if rg is None else torch.from_numpy(rg).to(DEV), want_idx=True)
    rec = record()
    torch.cuda.synchronize()
    n = c.B * c.K
    ctas = sms() if c.rec[0] == 1 else min((n * 32 + 255) // 256, sms() * 6)
    assert (rec["family"], rec["path"], rec["warps"], rec["stages"], rec["dtype"], rec["ctas"]) == \
        (FAMILY["decode"], *c.rec, DCODE[c.dt], ctas), rec
    want, widx = decode_oracle(xv, yv, c.k, center, scale, c.nms, rg)
    np.testing.assert_array_equal(idx.cpu().numpy(), widx, err_msg=f"{c.name}: indices")
    assert_bits(out.cpu().numpy(), want, f"{c.name}: out")


def test_decode_patterns_hit_every_rule():
    """The planted patterns are what the cases rely on: -0 maxima on both vectors (a -0 score), first NaN after a
    larger finite value, ties across the lane 31 | lane 0 boundary."""
    xv, yv = simdr_vectors(2, 21, 512, 512, seed=1)
    out, idx = decode_oracle(xv, yv, 2, None, None, False, None)
    s = out[..., 2].ravel()
    assert (np.signbit(s) & (s == 0)).any() and ((~np.signbit(s)) & (s == 0)).any()
    assert idx.reshape(-1, 2)[1, 0] == int(0.9 * 512)           # pattern 1: the NaN, not the 100 before it
    assert idx.reshape(-1, 2)[8, 0] == 127 and idx.reshape(-1, 2)[9, 0] == 31


def test_decode_overlap_over_rotating_outputs(monkeypatch):
    """LHN_FLAG_OVERLAP_PREVIOUS on the ring kernel over two rotating input / output sets: every launch's output is
    still bit-identical to the oracle's."""
    set_env(monkeypatch, RING1)
    sets = []
    for s in range(2):
        xv, yv = simdr_vectors(29, 21, 512, 512, seed=100 + s)
        sets.append((torch.from_numpy(xv).to(DEV), torch.from_numpy(yv).to(DEV), xv, yv,
                     torch.empty((29, 21, 3), dtype=torch.float32, device=DEV)))
    for i in range(6):
        xt, yt, _, _, out = sets[i % 2]
        ops.decode_simdr(xt, yt, 2, overlap_previous=True, out=out)
        assert record()["path"] == 1
    torch.cuda.synchronize()
    for xt, yt, xv, yv, out in sets:
        want, _ = decode_oracle(xv, yv, 2, None, None, False, None)
        assert_bits(out.cpu().numpy(), want, "overlap")


# ================================================ render ============================================================
def render_f32_steps(joints, vis, isz, k, den):
    """The reference expression step by step in f32 (the subtraction, the square and the division are IEEE f32 in numpy
    too) with exp correctly rounded from the f32 argument — the kernel's arithmetic, given the denominator."""
    j = np.asarray(joints, F32)
    nx, ny = int(isz[0] * k), int(isz[1] * k)
    out = []
    for ax, n in ((0, nx), (1, ny)):
        mu = j[..., ax:ax + 1] * F32(k)
        d = np.arange(n, dtype=F32) - mu
        with np.errstate(invalid="ignore", over="ignore"):
            a = -(d * d) / F32(den)
            v = np.exp(a.astype(F64)).astype(F32)
        out.append(np.where(np.asarray(vis, F32)[..., :1] > 0, v, F32(0)))
    return out


def render_joints(B, K, isz, seed):
    g = np.random.default_rng(seed)
    j = np.zeros((B, K, 3), F32)
    j[..., 0] = g.uniform(-20, isz[0] + 20, (B, K)); j[..., 1] = g.uniform(-20, isz[1] + 20, (B, K))
    j[0, 0, :2] = (0.0, isz[1] - 0.25)                              # on the first / near the last bin
    j[0, 1, :2] = (np.nan, 10.0)                                    # NaN: every x bin NaN
    j[0, 2, :2] = (np.inf, -1e12)                                   # infinite / far away: all zero
    v = (g.uniform(0, 1, (B, K, 1)) > 0.2).astype(F32)
    v[0, :3] = 1
    return j, v


# sigma, image size, k, expected path (1 windowed, 2 plain)
RCASES = [(1.3, (128, 96), 2, 1), (2.0, (128, 128), 2, 1), (2.1, (96, 128), 3, 1), (2.7, (64, 64), 2, 1),
          (3.3, (128, 128), 2, 1), (9.7, (128, 128), 2, 2), (2.1, (127.5, 128), 2, 2)]


@pytest.mark.parametrize("sigma,isz,k,path", RCASES, ids=[f"s{c[0]}-{c[1][0]}x{c[1][1]}-k{c[2]}" for c in RCASES])
def test_render_case(sigma, isz, k, path):
    """Bit for bit against the reference expression evaluated in its own f32 steps with the reference's denominator
    f32(2 * sigma ** 2), and within a derived bound of an f64 evaluation of the same expression.

    Bound: the kernel rounds d = pos - mu, d * d and -d^2 / den once each (relative u = 2^-24 each, so the argument a
    carries |theta| <= 4u(1 + 4u)), then exp(a (1 + theta)) = exp(a) exp(a theta) adds |a| |theta| (1 + |a theta|)
    relative (|a| <= 104 at the cut, so |a theta| < 2.5e-5), and the f64 exp rounded to f32 adds u relative, or 2^-150
    absolute where the result is subnormal:
        |got - e| <= e (4.001 |a| + 1.001) u + 2^-150,   e = exp(-(pos - mu)^2 / f32(2 sigma^2)) in f64."""
    B, K = 16, 21
    j, v = render_joints(B, K, isz, seed=int(sigma * 10))
    sx, sy = ops.render_simdr(torch.from_numpy(j).to(DEV), torch.from_numpy(v).to(DEV), isz, k, sigma)
    rec = record()
    Lx, Ly = int(isz[0] * k), int(isz[1] * k)
    assert (rec["family"], rec["path"], rec["warps"], rec["ctas"]) == \
        (FAMILY["render"], path, 8, min((B * K + 7) // 8, sms() * 8) if path == 1 else B * K), rec
    den = F32(2 * sigma ** 2)
    want = render_f32_steps(j, v, isz, k, den)
    got = (sx.cpu().numpy(), sy.cpu().numpy())
    for ax in range(2):
        assert_bits(got[ax], want[ax], f"sigma {sigma} axis {ax}")
        n = (Lx, Ly)[ax]
        # mu as the reference forms it, joints * k in f32 (rounded for k = 3): an input of the expression
        mu = (j[..., ax:ax + 1] * F32(k)).astype(F64)
        with np.errstate(invalid="ignore", over="ignore"):
            a = -((np.arange(n, dtype=F64) - mu) ** 2) / F64(den)
            e = np.where(v[..., :1] > 0, np.exp(a), 0.0)
        fin = np.isfinite(e) & np.isfinite(a)
        bnd = e * (4.001 * np.abs(np.where(fin, a, 0)) + 1.001) * U + 2.0 ** -150
        err = np.abs(got[ax].astype(F64) - e)
        report(f"render sigma {sigma} axis {ax}", float((err[fin] / bnd[fin]).max()))
        assert (err[fin] <= bnd[fin]).all(), (sigma, ax, float((err[fin] / bnd[fin]).max()))
        assert np.isnan(got[ax][~fin & np.isnan(e)]).all()


def test_render_denominator_is_the_references():
    """The f32-steps reproduction above is sensitive to the one-ulp denominator difference: with 2.f * s * s from an f32
    sigma (lhn_render_simdr's denominator) the bits differ for these sigma.  Host-only arithmetic."""
    isz = (128, 128)
    j, v = render_joints(4, 21, isz, seed=3)
    for sigma in (1.3, 2.1, 2.7, 3.3):
        good = F32(2 * sigma ** 2)
        bad = F32(2) * F32(sigma) * F32(sigma)
        assert good != bad
        a, b = render_f32_steps(j, v, isz, 2, good)[0], render_f32_steps(j, v, isz, 2, bad)[0]
        assert (a.view(np.int32) != b.view(np.int32)).any(), sigma


@pytest.mark.parametrize("sigma", [1.3, 2.0, 9.7])
def test_render_f32_sigma_entry_keeps_its_denominator(sigma):
    """lhn_render_simdr (f32 sigma, for C callers) is the same kernel with 2.f * s * s as the denominator: bit for bit
    the f32-steps reproduction with that denominator, on the windowed and (sigma 9.7) the plain path."""
    isz, k, B, K = (128, 128), 2, 8, 21
    j, v = render_joints(B, K, isz, seed=17)
    jt, vt = torch.from_numpy(j).to(DEV), torch.from_numpy(v).to(DEV)
    sx = torch.empty((B, K, 256), dtype=torch.float32, device=DEV)
    sy = torch.empty((B, K, 256), dtype=torch.float32, device=DEV)
    L.check(L.lib().lhn_render_simdr(L.ptr(jt), 3, L.ptr(vt), 1, B, K, 256, 256, float(k), sigma, L.ptr(sx), L.ptr(sy),
                                     L.stream()), "lhn_render_simdr")
    assert record()["path"] == (2 if sigma > 9 else 1)
    want = render_f32_steps(j, v, isz, k, F32(2) * F32(sigma) * F32(sigma))
    assert_bits(sx.cpu().numpy(), want[0], "x")
    assert_bits(sy.cpu().numpy(), want[1], "y")


def test_render_windowed_and_plain_paths_agree():
    """The same joints through the windowed (Lx % 4 == 0) and the plain (Lx % 4 != 0) kernel: identical bits."""
    j, v = render_joints(8, 21, (128, 128), seed=5)
    jt, vt = torch.from_numpy(j).to(DEV), torch.from_numpy(v).to(DEV)
    ax, ay = ops.render_simdr(jt, vt, (128, 128), 2, 2.7)
    assert record()["path"] == 1
    bx, by = ops.render_simdr(jt, vt, (128.5, 128), 2, 2.7)
    assert record()["path"] == 2
    assert_bits(bx[..., :256].cpu().numpy(), ax.cpu().numpy(), "x")
    assert_bits(by.cpu().numpy(), ay.cpu().numpy(), "y")


# ================================================= loss =============================================================
def ulp_neighbours(dt):
    one = torch.tensor(1.0, dtype=DT[dt])
    up = torch.nextafter(one.float(), torch.tensor(2.0)).to(DT[dt]) if dt == "f32" else \
        (one.float() + 2 * U_T[dt]).to(DT[dt])
    dn = torch.nextafter(one.float(), torch.tensor(0.0)).to(DT[dt]) if dt == "f32" else \
        (one.float() - U_T[dt]).to(DT[dt])
    return float(up.float()), float(dn.float())


def loss_inputs(dt, B, K, Lx, Ly, seed, nan=False, zero_w=False):
    """Targets in [0, 1), outputs target + N(0, 0.7); per row some |d| exactly 1, one ulp of the type above and below,
    and d = 0; weights in [0, 2) with zeros, joint 0 all zero (K > 1); NaN at one output when `nan`."""
    g = np.random.default_rng(seed)
    up, dn = ulp_neighbours(dt)
    arrs = []
    for n in (Lx, Ly):
        t = g.uniform(0, 1, (B, K, n)).astype(F32)
        o = (t + g.normal(0, 0.7, (B, K, n))).astype(F32)
        for c, dv in enumerate((1.0, -1.0, up, -up, dn, -dn)):
            if c < n:
                t[..., c] = 0.0; o[..., c] = dv
        if n > 6:
            o[..., 6] = t[..., 6]
        arrs += [o, t]
    w = (g.uniform(0, 2, (B, K)) * (g.uniform(0, 1, (B, K)) > 0.15)).astype(F32)
    if K > 1:
        w[:, 0] = 0.0
    if zero_w:
        w[:] = 0.0
    ox, tx, oy, ty = arrs
    if nan:
        ox[B // 2, K // 2, Lx // 2] = np.nan
    out = []
    for a in (ox, oy, tx, ty):
        t_, a_ = to_dt(a, dt)
        out += [t_, a_]
    return out, w


def kl_loss_f64(ox, oy, tx, ty, w):
    """KLDiscretLoss in f64, not rounded: (1/K) sum_j (mean SL1(x_j) + mean SL1(y_j)) * mean_b w[:, j]."""
    sl = lambda d: np.where(np.abs(d) < 1.0, 0.5 * d * d, np.abs(d) - 0.5)   # noqa: E731
    lx = sl(ox.astype(F64) - tx.astype(F64)).mean(axis=(0, 2))
    ly = sl(oy.astype(F64) - ty.astype(F64)).mean(axis=(0, 2))
    return float(((lx + ly) * w.astype(F64).mean(axis=0)).sum() / ox.shape[1])


# name, dtype, B, K, Lx, Ly, LHN_SIMDR_LOSS_PATH, base offset, expected path
# (1 joint + cluster, 2 rows + cluster, 3 rows + one block, 4 loop), expected vector flag
S_ = namedtuple("S_", "name dt B K Lx Ly mode off path vec")
SCASES = [
    # joint kernel: more than 148 * 8 CTAs of rows (> 9472 rows), vector rows, K <= 128
    S_("joint-f32-K21", "f32", 456, 21, 64, 64, None, 0, 1, 1),
    S_("joint-bf16-K1", "bf16", 9600, 1, 64, 32, None, 0, 1, 1),
    S_("joint-f16-K128", "f16", 75, 128, 32, 64, None, 0, 1, 1),
    # rows + cluster: 8192 .. 9472 vector rows, non-vector rows at any size >= 8192, or the joint kernel switched off
    S_("rows-cluster-vec-f32", "f32", 400, 21, 64, 64, None, 0, 2, 1),
    S_("rows-cluster-nonvec-bf16", "bf16", 456, 21, 63, 64, None, 0, 2, 0),
    S_("rows-cluster-forced-f16", "f16", 456, 21, 64, 64, 2, 0, 2, 1),
    S_("rows-cluster-K128-offset-f32", "f32", 72, 128, 64, 64, None, 1, 2, 0),
    # rows + one block: fewer than 8192 rows, K in 129 .. 1024, or forced
    S_("rows-block-small-f32", "f32", 4, 21, 512, 512, None, 0, 3, 1),
    S_("rows-block-K129-f32", "f32", 80, 129, 64, 64, None, 0, 3, 1),
    S_("rows-block-K129-bf16", "bf16", 4, 129, 36, 92, None, 0, 3, 1),
    S_("rows-block-K1-f16", "f16", 3, 1, 4, 8, None, 0, 3, 1),
    S_("rows-block-forced-f32", "f32", 456, 21, 64, 64, 1, 0, 3, 1),
    S_("rows-block-offset-f16", "f16", 4, 21, 64, 64, None, 1, 3, 0),
    # the single-thread loop of the one-block finalise: K > 1024
    S_("loop-K1025-f32", "f32", 2, 1025, 8, 12, None, 0, 4, 1),
    S_("loop-K1025-bf16", "bf16", 2, 1025, 7, 4, None, 0, 4, 0),
]


def loss_rel_bound(Lx, Ly):
    """Relative bound of the kernel's loss on the f64 value (all terms non-negative).

    Each SmoothL1 term is formed from d = fl(o - t) with at most three roundings (the difference, the square or
    |d| - 0.5, the product with 0.5 is exact): relative gamma_3.  A lane adds its terms to an f32 accumulator in order —
    n_acc = max(ceil(L / 32) (scalar scan: one accumulator), 2 ceil(L / 128) (vector scan: two per vector)) terms —
    which for non-negative terms adds gamma_(n_acc - 1) relative; the per-lane sums then meet in f64 (relative
    < 1e-12 here, counted as one u), and the loss is rounded to f32 once (u).  With non-negative weights the same
    relative bound holds for the weighted mean over joints:  (n_acc + 4) u."""
    n_acc = max(max(math.ceil(n / 32), 2 * math.ceil(n / 128)) for n in (Lx, Ly))
    return (n_acc + 4) * U


@pytest.mark.parametrize("c", SCASES, ids=[c.name for c in SCASES])
def test_loss_case(c, monkeypatch):
    set_env(monkeypatch, {} if c.mode is None else {"LHN_SIMDR_LOSS_PATH": c.mode})
    (ox, oxn, oy, oyn, tx, txn, ty, tyn), w = loss_inputs(c.dt, c.B, c.K, c.Lx, c.Ly, seed=len(c.name) * 31 + c.K)
    ox, oy, tx, ty = (offset_view(t, c.off) for t in (ox, oy, tx, ty))
    wt = torch.from_numpy(w).to(DEV)
    got = ops.simdr_smoothl1(ox, oy, tx, ty, wt)
    rec = record()
    assert (rec["family"], rec["path"], rec["vec_x"], rec["dtype"], rec["warps"]) == \
        (FAMILY["loss"], c.path, c.vec, DCODE[c.dt], 8), rec
    again = ops.simdr_smoothl1(ox, oy, tx, ty, wt)
    got, again = float(got.item()), float(again.item())
    assert np.float32(got).view(np.int32) == np.float32(again).view(np.int32), "not bitwise reproducible"
    want = kl_loss_f64(oxn, oyn, txn, tyn, w)
    rel = loss_rel_bound(c.Lx, c.Ly)
    report(f"loss {c.name}", abs(got - want) / (rel * want))
    assert want > 0 and abs(got - want) <= rel * want, (got, want, abs(got - want) / want / U, rel / U)
    # sensitivity: leaving out one row of x terms (of the joint with the largest mean weight) moves the loss by more
    # than the bound
    j = int(np.argmax(w.mean(axis=0)))
    ox2 = oxn.copy(); ox2[0, j] = txn[0, j]
    assert abs(kl_loss_f64(ox2, oyn, txn, tyn, w) - want) > rel * want


@pytest.mark.parametrize("name", ["rows-block-small-f32", "joint-f32-K21", "rows-cluster-nonvec-bf16"])
def test_loss_nan_and_zero_weights(name):
    """A NaN output makes the loss NaN on every route; all-zero weights make it exactly 0."""
    c = next(s for s in SCASES if s.name == name)
    (ox, _, oy, _, tx, _, ty, _), w = loss_inputs(c.dt, c.B, c.K, c.Lx, c.Ly, seed=9, nan=True)
    assert math.isnan(float(ops.simdr_smoothl1(ox, oy, tx, ty, torch.from_numpy(w).to(DEV)).item()))
    assert record()["path"] == c.path
    (ox, _, oy, _, tx, _, ty, _), w = loss_inputs(c.dt, c.B, c.K, c.Lx, c.Ly, seed=9, zero_w=True)
    z = float(ops.simdr_smoothl1(ox, oy, tx, ty, torch.from_numpy(w).to(DEV)).item())
    assert z == 0.0 and not math.copysign(1.0, z) < 0


# =============================================== backward ===========================================================
def kl_grad_f64(o, t, w, scale, grad_out):
    """d KLDiscretLoss / d output in f64, not rounded: g SmoothL1'(d) mean_b(w)[j] / (K B L)."""
    B, K, n = o.shape
    d = o.astype(F64) - t.astype(F64)
    sl = np.where(np.abs(d) < 1.0, d, np.sign(d))
    return sl * w.astype(F64).mean(axis=0).reshape(1, K, 1) / (K * B * n) * scale * grad_out


# name, dtype, B, K, Lx, Ly, base offset, grad_out (None = the default 1), expected (vec_x, vec_y)
G_ = namedtuple("G_", "name dt B K Lx Ly off grad_out vec")
GCASES = [
    G_("vec-f32", "f32", 4, 21, 64, 64, 0, 2.5, (1, 1)),
    G_("vec-f32-none", "f32", 3, 21, 512, 256, 0, None, (1, 1)),
    G_("mixed-bf16", "bf16", 4, 21, 64, 63, 0, 2.5, (1, 0)),
    G_("mixed-f16-none", "f16", 4, 21, 37, 92, 0, None, (0, 1)),
    G_("scalar-offset-f16", "f16", 4, 21, 64, 64, 1, 2.5, (0, 0)),
    G_("scalar-offset-bf16-none", "bf16", 4, 21, 64, 64, 1, None, (0, 0)),
    G_("scalar-f32-L1-L3", "f32", 3, 5, 1, 3, 0, 2.5, (0, 0)),
    G_("vec-bf16-K129", "bf16", 2, 129, 64, 64, 0, 2.5, (1, 1)),
]


@pytest.mark.parametrize("c", GCASES, ids=[c.name for c in GCASES])
def test_backward_case(c):
    """Elementwise against the f64 gradient, within
        |got - r| <= |r| (6.01 u + 1.0001 u_T) + sub_T,
    derived from the kernel's arithmetic: the joint coefficient c = f32(f64(1 / (K B L)) * f32(mean_b w)) * g with
    g = f32(scale * grad_out) carries four f32 roundings; SmoothL1'(d) is exactly +-1 or d = fl(o - t) (one rounding,
    none for bf16 / f16 inputs; at |d| = 1 both branches agree to that rounding); the product one more: gamma_6 in f32;
    then the store rounds to the tensor's type once (u_T relative, or half its smallest subnormal absolute)."""
    scale = 3.0
    (ox, oxn, oy, oyn, tx, txn, ty, tyn), _ = loss_inputs(c.dt, c.B, c.K, c.Lx, c.Ly, seed=c.K + c.Lx, nan=True)
    g = np.random.default_rng(c.Lx)
    # joint means at least 4 % apart, so a neighbour's coefficient is visible above the bound (bf16: 2^-8)
    w = (0.5 + 0.05 * np.arange(c.K)[None, :] + g.uniform(0, 0.002, (c.B, c.K))).astype(F32)
    ox, oy, tx, ty = (offset_view(t, c.off) for t in (ox, oy, tx, ty))
    go = None if c.grad_out is None else torch.tensor([c.grad_out], dtype=torch.float32, device=DEV)
    gx, gy = ops.simdr_smoothl1_backward(ox, oy, tx, ty, torch.from_numpy(w).to(DEV), scale, go)
    rec = record()
    assert (rec["family"], rec["vec_x"], rec["vec_y"], rec["dtype"]) == (FAMILY["backward"], *c.vec, DCODE[c.dt]), rec
    gov = 1.0 if c.grad_out is None else c.grad_out
    for got, o, t in ((gx, oxn, txn), (gy, oyn, tyn)):
        got = got.float().cpu().numpy().astype(F64)
        r = kl_grad_f64(o, t, w, scale, gov)
        nan = np.isnan(r)
        np.testing.assert_array_equal(np.isnan(got), nan)
        bnd = np.abs(r) * (6.01 * U + 1.0001 * U_T[c.dt]) + SUB_T[c.dt]
        err = np.abs(got - r)
        report(f"backward {c.name}", float((err[~nan] / bnd[~nan]).max()))
        assert (err[~nan] <= bnd[~nan]).all(), float((err[~nan] / bnd[~nan]).max())
        # sensitivity: joint j with joint j + 1's coefficient leaves the bound wherever SmoothL1' is not tiny
        if c.K > 1:
            rs = kl_grad_f64(o, t, np.roll(w, -1, axis=1), scale, gov)
            big = ~nan & (np.abs(r) > 1000 * SUB_T[c.dt])
            assert (np.abs(rs - r)[big] > bnd[big]).all()


# ================================================= heads ============================================================
HEADS_STAGES = {64: 4, 80: 4, 128: 3}


def default_bn(M, N):
    """lhn_simdr_heads.cu pick_bn: 64-column tiles when 128-column tiles leave more than half of the SMs idle and the
    64-column grid still fits in one wave, else 128."""
    mt = (M + 127) // 128
    c128, c64 = mt * ((N + 127) // 128), mt * ((N + 63) // 64)
    return 64 if (c128 * 2 <= sms() and c64 <= sms()) else 128


def heads_inputs(B, K, H, W, Lx, Ly, seed):
    g = np.random.default_rng(seed)
    hm = np.abs(g.normal(0, 0.3, (B, K, H, W))).astype(F32)             # heatmaps are non-negative
    w = (g.normal(0, 1.0, (Lx + Ly, H * W)) / math.sqrt(H * W) * 3).astype(F32)
    bias = g.normal(0, 0.2, Lx + Ly).astype(F32)
    tx = g.uniform(0, 1, (B, K, Lx)).astype(F32); ty = g.uniform(0, 1, (B, K, Ly)).astype(F32)
    wt = g.uniform(0.2, 1.5, (B, K)).astype(F32)
    return hm, w, bias, tx, ty, wt


def gemm_bound(Kd, S, ref):
    """|pred - ref| per element for the bf16 x 3 product (x = hi + lo from lhn_split_bf16), S = sum_k |a_k| |w_k| + |b|.

    Split: hi = bf16(x) is within 2^-8 |x|, lo = bf16(x - hi) within 2^-8 |x - hi|, so e = x - hi - lo is within
    2^-16 |x| and |lo| <= 2^-8 (1 + 2^-8) |x|.  Each product a w then misses lo_a lo_w + e_a w + (hi_a + lo_a) e_w,
    less than 3.1 * 2^-16 |a| |w|.  The bf16 x bf16 products are exact in f32; the 3 Kd / 16 MMA instructions each add
    their 16 products into the f32 accumulator with at most two roundings, each at most one ulp (2u) of a magnitude
    below S: (3 Kd / 4) u S.  The bias add rounds once: u |pred|."""
    return 3.1 * 2.0 ** -16 * S + (0.75 * Kd + 1) * U * S + U * np.abs(ref) * 1.0001


# name, B, K, H, W, Lx, Ly, LHN_HEADS_BN (None = the default choice)
H_ = namedtuple("H_", "name B K H W Lx Ly bn")
HCASES = [
    H_("m1-kb1-36x92", 1, 1, 8, 8, 36, 92, None),
    H_("m127-kb2-4x60-bn64", 127, 1, 8, 16, 4, 60, 64),
    H_("m128-kb3-60x4-bn80", 128, 1, 8, 24, 60, 4, 80),
    H_("m129-kb4-36x92-bn128", 129, 1, 16, 16, 36, 92, 128),
    H_("m256-kb5-448-default", 64, 4, 16, 20, 448, 448, None),
    H_("m256-kb5-448-bn80", 64, 4, 16, 20, 448, 448, 80),
    H_("m129-kb64-512-bn64", 129, 1, 64, 64, 512, 512, 64),
    H_("m5377-kb64-512-default", 283, 19, 64, 64, 512, 512, None),
    H_("m5377-kb5-36x92-bn80", 283, 19, 16, 20, 36, 92, 80),
    H_("m128-kb1-4x60-bn128", 8, 16, 8, 8, 4, 60, 128),
]


def heads_direct(hm_t, w_hi, w_lo, bias, tx, ty, wt, B, K, Kd, Lx, Ly):
    """split + lhn_simdr_heads_loss, without the one-call wrapper."""
    a_hi, a_lo = ops.split_bf16(hm_t.reshape(B * K, Kd))
    nbytes = int(L.lib().lhn_simdr_heads_workspace_bytes(B, K, Lx, Ly))
    ws = torch.empty(nbytes, dtype=torch.uint8, device=DEV)
    loss = torch.empty(1, dtype=torch.float32, device=DEV)
    dpred = torch.empty((B * K, Lx + Ly), dtype=torch.float32, device=DEV)
    pred = torch.empty((B * K, Lx + Ly), dtype=torch.float32, device=DEV)
    L.check(L.lib().lhn_simdr_heads_loss(L.ptr(a_hi), L.ptr(a_lo), L.ptr(w_hi), L.ptr(w_lo), L.ptr(bias), L.ptr(tx),
                                         L.ptr(ty), L.ptr(wt), B, K, Kd, Lx, Ly, L.ptr(ws), nbytes, L.ptr(loss),
                                         L.ptr(dpred), L.ptr(pred), L.stream()), "lhn_simdr_heads_loss")
    return loss, dpred, pred


@pytest.mark.parametrize("c", HCASES, ids=[c.name for c in HCASES])
def test_heads_case(c, monkeypatch):
    set_env(monkeypatch, {} if c.bn is None else {"LHN_HEADS_BN": c.bn})
    B, K, Kd, N = c.B, c.K, c.H * c.W, c.Lx + c.Ly
    M = B * K
    hm, w, bias, tx, ty, wt = heads_inputs(B, K, c.H, c.W, c.Lx, c.Ly, seed=M + Kd)
    ts = [torch.from_numpy(a).to(DEV) for a in (hm, w, bias, tx, ty, wt)]
    hm_t, w_t, b_t, tx_t, ty_t, wt_t = ts
    w_split = ops.split_bf16(w_t)
    loss, dpred, pred = ops.simdr_heads_loss(hm_t, w_split, b_t, tx_t, ty_t, wt_t, want_dpred=True, want_pred=True)
    rec = record()
    bn = c.bn or default_bn(M, N)
    assert (rec["family"], rec["bn"], rec["stages"], rec["warps"], rec["ctas"]) == \
        (FAMILY["heads"], bn, HEADS_STAGES[bn], 8, ((N + bn - 1) // bn) * ((M + 127) // 128)), rec
    # the one-call f32 entry is split + lhn_simdr_heads_loss, bit for bit
    l2, d2, p2 = heads_direct(hm_t, *w_split, b_t, tx_t, ty_t, wt_t, B, K, Kd, c.Lx, c.Ly)
    assert torch.equal(loss.view(torch.int32), l2.view(torch.int32))
    assert torch.equal(pred.view(torch.int32), p2.view(torch.int32)) and torch.equal(dpred.view(torch.int32),
                                                                                      d2.view(torch.int32))
    p = pred.cpu().numpy()
    # the oracle GEMMs in f64 (on the device: 5377 x 4096 x 1024 twice is slow on the host; f64 rounding is ~1e-16)
    a64, w64 = hm_t.reshape(M, Kd).double(), w_t.double()
    ref = (a64 @ w64.T + b_t.double()).cpu().numpy()
    S = (a64.abs() @ w64.abs().T + b_t.double().abs()).cpu().numpy()
    bnd = gemm_bound(Kd, S, ref)
    err = np.abs(p.astype(F64) - ref)
    report(f"heads gemm {c.name}", float((err / bnd).max()))
    assert (err <= bnd).all(), float((err / bnd).max())
    # sensitivity: leaving out the last k-block moves some prediction by more than the bound
    drop = (a64[:, -64:] @ w64[:, -64:].T).abs().cpu().numpy()
    assert (drop > bnd).any()
    # dpred = clamp(pred - t, -1, 1) from the kernel's own pred, bit for bit (both branches occur)
    t_all = np.concatenate([tx.reshape(M, c.Lx), ty.reshape(M, c.Ly)], 1)
    dref = torch.clamp(pred.cpu() - torch.from_numpy(t_all), -1, 1).numpy()
    assert_bits(dpred.cpu().numpy(), dref, "dpred")
    assert (np.abs(p - t_all) > 1).any() and (np.abs(p - t_all) < 1).any()
    # the loss: tight against f64 from the kernel's own pred, and within the GEMM bound of the f64 GEMM's
    px, py = p[:, :c.Lx].reshape(B, K, c.Lx), p[:, c.Lx:].reshape(B, K, c.Ly)
    own = kl_loss_f64(px, py, tx, ty, wt)
    got = float(loss.item())
    # per term: d = fl(pred - t), SL1 (gamma_3 as in the loss bound above); groups of four summed pairwise (2 more);
    # a row's <= BN / 4 group sums per N tile added in order in f32; the tiles and rows in f64; the loss rounded once
    tight = (bn // 4 + 8) * U * own
    report(f"heads loss-vs-own-pred {c.name}", abs(got - own) / tight)
    assert abs(got - own) <= tight, (got, own, abs(got - own) / own / U)
    rx, ry = ref[:, :c.Lx].reshape(B, K, c.Lx), ref[:, c.Lx:].reshape(B, K, c.Ly)
    full = kl_loss_f64(rx, ry, tx, ty, wt)
    # SmoothL1 is 1-Lipschitz: |loss(pred) - loss(ref)| <= sum_e coef_e |pred_e - ref_e|, coef = mean_b w_j / (K B L)
    wm = wt.astype(F64).mean(0)[None, :, None]
    coef = np.concatenate([np.broadcast_to(wm / (K * B * n), (B, K, n)).reshape(M, n) for n in (c.Lx, c.Ly)], 1)
    report(f"heads loss-vs-f64-gemm {c.name}", abs(got - full) / (tight + float((coef * bnd).sum())))
    assert abs(got - full) <= tight + float((coef * bnd).sum())


def test_heads_nan_stays_in_its_row():
    """A NaN in heatmap row r makes exactly prediction row r NaN (and its dpred, and the loss)."""
    B, K, H, W, Lx, Ly = 3, 43, 8, 16, 36, 92
    hm, w, bias, tx, ty, wt = heads_inputs(B, K, H, W, Lx, Ly, seed=11)
    hm[1, 5, 0, 3] = np.nan
    ts = [torch.from_numpy(a).to(DEV) for a in (hm, w, bias, tx, ty, wt)]
    loss, dpred, pred = ops.simdr_heads_loss(ts[0], ops.split_bf16(ts[1]), *ts[2:], want_dpred=True, want_pred=True)
    rows = torch.isnan(pred).any(1).nonzero().flatten().tolist()
    assert rows == [1 * K + 5] and bool(torch.isnan(pred[1 * K + 5]).all())
    assert torch.isnan(dpred).any(1).nonzero().flatten().tolist() == rows and bool(torch.isnan(dpred[rows[0]]).all())
    assert math.isnan(float(loss.item()))


def test_split_bf16_special_values():
    """hi = bf16(x) and lo = bf16(x - hi), round to nearest even, exactly — subnormals, +-0, +-inf, NaN, the largest
    f32 (hi overflows to inf, lo = -inf) included; any NaN matches any NaN."""
    g = np.random.default_rng(2)
    sp = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e-45, -1e-45, 1.1754942e-38, 3e-39, -7.1e-40, 1e-40,
                   3.4028235e38, -3.4028235e38, 1.0, 1.00390625, 1.005859375, 65504.0, 2.0 ** -126], F32)
    x = np.concatenate([sp, g.standard_normal(1000).astype(F32) * 10.0 ** g.integers(-40, 38, 1000)]).astype(F32)
    x = np.concatenate([x, np.zeros((-len(x)) % 4, F32)])
    hi, lo = ops.split_bf16(torch.from_numpy(x).to(DEV))
    xt = torch.from_numpy(x)
    rhi = xt.to(torch.bfloat16)
    with np.errstate(invalid="ignore", over="ignore"):
        rlo = (xt - rhi.float()).to(torch.bfloat16)
    for got, want, what in ((hi.cpu(), rhi, "hi"), (lo.cpu(), rlo, "lo")):
        gb, wb = got.view(torch.int16).numpy(), want.view(torch.int16).numpy()
        nan = torch.isnan(got.float()).numpy() & torch.isnan(want.float()).numpy()
        bad = (gb != wb) & ~nan
        assert not bad.any(), (what, x[bad][:5], got.float().numpy()[bad][:5], want.float().numpy()[bad][:5])
