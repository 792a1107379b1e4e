"""The heatmap training target every kernel renders, pixel by pixel, against the f64 oracle at the geometry edges.

Five kernels draw the same Gaussian target from the joints.  Only lhn_render_targets writes it out; the others are read
out exactly:
- lhn_render_loss_backward: hm = 0, LHN_LOSS_DISTANCE, sums = (0, 0, 0, 2).  The coefficient is then 1 and each
  element is w * fmaf(-gx, gy, 0), i.e. grad == -(w * T) bit for bit;
- lhn_render_loss_backward_cond, forced to recompute (the assumed upstream value differs): the same bits;
- lhn_render_loss_grad: hm = 0, LHN_LOSS_DISTANCE, loss_scale = numel / 2: coefficient 1 again;
- K1 (the persistent team kernel and the CTA-per-plane kernel) writes no target: its per-plane partials (S_pos,
  S_neg, N_pos) and weights are probed, with positive thresholds taken from the target itself.

Error bound against the f64 oracle.  A table entry is exp_f32_from_f64(a) = fmaf(expf(ah), al, expf(ah)): expf is
within 2 ulp, the fma adds half an ulp, so a factor is within 2.5 ulp of itself, i.e. 2.5 * 2^-23 relative at worst
(at the bottom of its binade).  The target is the f32 product of two factors: relative error <= 5 * 2^-23 + 2^-24 =
11 * 2^-24.  That is 5.5 ulp of a result at the bottom of its binade and up to 11 ulp at the top, so the test
asserts the relative form.  Below 2^-126 the factors and the product round to the denormal grid: each adds at most
its rounding in absolute terms, 3 * 2^-149 in all.  The largest error in ulp of the oracle is printed per kernel.
"""
import ctypes
import math
import time
import zlib

import numpy as np
import pytest
import torch

from oracle import np_oracle as O
from litehandnet_b200 import _lib as L
from litehandnet_b200 import ops

DEV = "cuda"
F32 = np.float32
REL_BOUND = 11.0 * 2.0 ** -24
ABS_BOUND = 3.0 * 2.0 ** -149
TINY = 2.0 ** -126
SWITCHES = ("LHN_NO_FAST", "LHN_TEAM_POLICY", "LHN_TEAM_STAGES", "LHN_STAGGER_NS", "LHN_CTAS_PER_SM", "LHN_FORCE_CTA_KERNEL")
MAX_ULP = {}                  # kernel -> largest error seen against the f64 oracle, in ulp of the oracle
NEXT_HALF = float(np.nextafter(F32(0.5), F32(1)))


# ---------------------------------------------------------------------------------------------------------------------
# the case table (plain NumPy)
# ---------------------------------------------------------------------------------------------------------------------
class Case:
    def __init__(self, name, mode, sigma, img, hw, K, dtype="f32", flip=False, js=3, vs=3, cta=False):
        self.name, self.mode, self.sigma, self.img, self.hw, self.K = name, mode, sigma, img, hw, K
        self.dtype, self.flip, self.js, self.vs = dtype, flip, js, vs
        self.cta = cta or hw[0] % 4 != 0             # the CTA-per-plane kernel is what the default policy picks
        self.sigmas = list(sigma) if isinstance(sigma, (list, tuple)) else [sigma]

    def feat(self):
        (wi, hi), (W, H) = self.img, self.hw
        if self.mode == 2:
            return ((wi - 1.0) / (W - 1.0), (hi - 1.0) / (H - 1.0))
        return (wi / W, hi / H)


SIZES = [  # name, image (W, H), plane (W, H)
    ("256-64", (256, 256), (64, 64)),
    ("224-56", (224, 224), (56, 56)),
    ("256x192-64x48", (256, 192), (64, 48)),        # anisotropic plane, H != W
    ("192x256-64x48", (192, 256), (64, 48)),        # x stride 3, y stride 16/3: neither a power of two
    ("255x250-64", (255, 250), (64, 64)),           # strides 255/64, 250/64
    ("120x88-30x22", (120, 88), (30, 22)),          # W not a multiple of 4
]
SIGMAS = (1.5, 2.0, 2.5, 3.0)
DTYPES = ("f32", "bf16", "f16")


def _build_cases():
    cases, i = [], 0
    for sname, img, hw in SIZES:
        for mode in (0, 1, 2):
            sig = SIGMAS[i % 4]
            cases.append(Case(f"{sname}-m{mode}-s{sig}", mode, sig, img, hw, 21, dtype=DTYPES[i % 3],
                              js=(2, 3, 4)[i % 3], vs=(1, 3)[i % 2]))
            i += 1
    for mode in (0, 1, 2):                           # every sigma at the headline size
        for sig in SIGMAS:
            if not any(c.mode == mode and c.sigma == sig and c.hw == (64, 64) and c.img == (256, 256) for c in cases):
                cases.append(Case(f"256-64-m{mode}-s{sig}", mode, sig, (256, 256), (64, 64), 21, dtype=DTYPES[i % 3],
                                  js=(2, 3, 4)[i % 3], vs=(1, 3)[i % 2]))
                i += 1
    for mode in (0, 1, 2):                           # the CTA-per-plane kernel's natural shape: 128^2 f32 with flip
        cases.append(Case(f"512-128-flip-m{mode}", mode, SIGMAS[(i + mode) % 4] * 2, (512, 512), (128, 128), 6,
                          flip=True, js=3, vs=3, cta=True))
    stacks = [(2, 21, [2.0, 3.0]), (8, 21, [1.5, 2.0, 2.5, 3.0, 1.5, 2.0, 2.5, 3.0]), (2, 5, [3.0, 1.5]),
              (8, 5, [2.5, 1.5, 3.0, 2.0, 2.0, 3.0, 1.5, 2.5])]
    for n, (S, K, sl) in enumerate(stacks):
        for mode in (0, 1, 2):
            cases.append(Case(f"stack{S}-k{K}-m{mode}", mode, sl, (256, 256), (64, 64), K, dtype=DTYPES[(n + mode) % 3],
                              js=(4, 2, 3)[mode], vs=(3, 1)[n % 2]))
    return cases


CASES = _build_cases()


def _up(j):
    return F32(np.nextafter(F32(j), F32(np.inf)))


def _down(j):
    return F32(np.nextafter(F32(j), F32(-np.inf)))


def axis_geom(j, feat, tmp, mode):
    """(mu, ul, br) along one axis in f64, exactly as the reference (and every kernel) computes them; int() is
    np.trunc, which also carries NaN and inf through the way the kernels' f64 trunc does."""
    mu = float(F32(j)) / feat
    if mode == 1:
        return mu, mu - tmp, mu + tmp + 1
    mi = float(np.trunc(mu + 0.5))
    return mu, float(np.trunc(mi - tmp)), float(np.trunc(mi + tmp + 1))


def _key(f):
    """Monotone integer key of an f32 (ordered like the floats)."""
    i = int(np.asarray(f, F32).view(np.int32))
    return i if i >= 0 else -(i & 0x7fffffff)


def _unkey(k):
    return F32(np.asarray(k if k >= 0 else -k - 2 ** 31, np.int32).view(F32))


def _boundary(pred, lo, hi):
    """Smallest f32 j in (lo, hi] with pred(j) true, by bisection (pred is false at lo, true at hi, monotone)."""
    a, b = _key(F32(lo)), _key(F32(hi))
    assert not pred(_unkey(a)) and pred(_unkey(b)), (lo, hi)
    while b - a > 1:
        m = (a + b) // 2
        a, b = (a, m) if pred(_unkey(m)) else (m, b)
    return _unkey(b)


def _exact(pred, guess, span=64):
    """An f32 j within `span` ulps of guess with pred(j) true, or None."""
    lo = hi = F32(guess)
    for _ in range(span):
        if pred(lo):
            return lo
        if pred(hi):
            return hi
        lo, hi = _down(lo), _up(hi)
    return None


AXIS_KINDS = ("interior", "half", "neg07", "neg03", "ulshift", "ulW-", "ulW", "ulW+", "br0-", "br0", "br0+",
              "farpos", "farneg", "posinf", "neginf")


def place(kind, n, feat, tmp, mode, rng):
    """An f32 coordinate along an axis of n pixels that meets `kind` (None when the geometry cannot)."""
    geo = lambda j: axis_geom(j, feat, tmp, mode)   # noqa: E731
    if kind == "interior":
        return F32(rng.uniform(0.3 * n, 0.7 * n) * feat)
    if kind == "half":
        k = n // 2
        return _exact(lambda j: geo(j)[0] == k + 0.5, (k + 0.5) * feat)
    if kind in ("neg07", "neg03"):
        return F32(-(0.7 if kind == "neg07" else 0.3) * feat)
    if kind == "ulshift":                            # integer centre mi = floor(tmp): mi - tmp in (-1, 0)
        if mode == 1 or tmp == math.floor(tmp):
            return None
        mi = math.floor(tmp)
        return _exact(lambda j: math.trunc(geo(j)[0] + 0.5) == mi, mi * feat)
    if kind.startswith("ulW"):
        j = _exact(lambda j: geo(j)[1] == n, (n + tmp) * feat) if mode == 1 else None
        if j is None or mode != 1:                   # the first f32 with ul >= n (ul == n exactly in modes 0, 2)
            j = _boundary(lambda j: geo(j)[1] >= n, (n - 5) * feat, (n + tmp + 5) * feat)
        return {"ulW-": _down(j), "ulW": j, "ulW+": _up(j)}[kind]
    if kind.startswith("br0"):
        j = _exact(lambda j: geo(j)[2] == 0, (-tmp - 1) * feat) if mode == 1 else None
        if j is None or mode != 1:                   # the first f32 with br >= 0 (br == 0 exactly in modes 0, 2)
            j = _boundary(lambda j: geo(j)[2] >= 0, (-tmp - 5) * feat, 5 * feat)
        return {"br0-": _down(j), "br0": j, "br0+": _up(j)}[kind]
    if kind == "farpos":
        return F32((n + 100) * feat)
    if kind == "farneg":
        return F32((-100 - 2 * tmp) * feat)
    if kind == "posinf":
        return F32(np.inf)
    if kind == "neginf":
        return F32(-np.inf)
    if kind == "nan":
        return F32(np.nan)
    raise KeyError(kind)


def kind_holds(kind, j, n, feat, tmp, mode):
    """Does coordinate j meet the condition `kind` promises (in f64, as the kernels evaluate it)?"""
    mu, ul, br = axis_geom(j, feat, tmp, mode)
    if kind == "interior":
        return 0.0 <= mu <= n - 1
    if kind == "half":
        return mu == math.floor(mu) + 0.5
    if kind == "neg07":                              # int() and floor() round the centre differently here
        return -1.0 < mu < -0.5 and (mode == 1 or (math.trunc(mu + 0.5) == 0 and math.floor(mu + 0.5) == -1))
    if kind == "neg03":
        return -0.5 < mu < 0.0
    if kind == "ulshift":                            # ul = int(mi - tmp) = 0 where floor would give -1
        mi = math.trunc(mu + 0.5)
        return -1.0 < mi - tmp < 0.0 and ul == 0.0 and math.floor(mi - tmp) == -1
    prev, nxt = axis_geom(_down(j), feat, tmp, mode), axis_geom(_up(j), feat, tmp, mode)
    if kind == "ulW":                                # the first f32 with ul >= n; ul == n exactly where reachable
        return ul >= n and prev[1] < n and (mode == 1 or ul == n)
    if kind == "ulW-":
        return ul < n and nxt[1] >= n
    if kind == "ulW+":
        return ul >= n and prev[1] >= n and axis_geom(_down(_down(j)), feat, tmp, mode)[1] < n
    if kind == "br0":
        return br >= 0 and prev[2] < 0 and (mode == 1 or br == 0)
    if kind == "br0-":
        return br < 0 and nxt[2] >= 0
    if kind == "br0+":
        return br >= 0 and prev[2] >= 0 and axis_geom(_down(_down(j)), feat, tmp, mode)[2] < 0
    if kind == "farpos":
        return ul >= n
    if kind == "farneg":
        return br < 0
    if kind == "posinf":
        return mu == np.inf
    if kind == "neginf":
        return mu == -np.inf
    if kind == "nan":
        return math.isnan(mu)
    raise KeyError(kind)


def slots(case):
    """(kind_x, kind_y, visibility, stack the tmp-dependent kinds are built for), one per joint slot."""
    out, s = [], 0
    for axis in (0, 1):
        for k in AXIS_KINDS[(1 if axis else 0):]:
            out.append((k, "interior", 1.0, s) if axis == 0 else ("interior", k, 1.0, s))
            s = (s + 1) % len(case.sigmas)
    out += [("nan", "interior", 1.0, 0), ("interior", "nan", 1.0, 0), ("nan", "nan", 1.0, 0)]
    out += [("interior", "interior", v, 0) for v in (0.0, 0.3, 0.5, NEXT_HALF, 2.0)]
    out += [("ulW-", "interior", 2.0, 0), ("interior", "br0", 2.0, 0), ("neg07", "neg03", 1.0, 0)]
    return out


def build_inputs(case):
    """joints [B,K,js] and vis [B,K,vs] (f32) holding every slot of the case, plus the slot of each joint."""
    sl = slots(case)
    K = case.K
    B = -(-len(sl) // K) + 1                          # one more sample of plain interior joints
    rng = np.random.default_rng(zlib.crc32(case.name.encode()))
    W, H = case.hw
    fx, fy = case.feat()
    joints = np.zeros((B, K, case.js), F32)
    joints[..., 2:] = 1.0                             # joints_3d's third column; must not be read
    vis = np.full((B, K, case.vs), 7.0, F32)          # only column 0 is the visibility
    table = {}
    for b in range(B):
        for k in range(K):
            i = b * K + k
            kx, ky, v, s = sl[i] if i < len(sl) else ("interior", "interior", 1.0, 0)
            tmp = case.sigmas[s] * 3
            jx = place(kx, W, fx, tmp, case.mode, rng)
            jy = place(ky, H, fy, tmp, case.mode, rng)
            if jx is None or jy is None:              # the geometry cannot meet this kind: an interior joint instead
                kx, ky = ("interior" if jx is None else kx), ("interior" if jy is None else ky)
                jx = place(kx, W, fx, tmp, case.mode, rng) if jx is None else jx
                jy = place(ky, H, fy, tmp, case.mode, rng) if jy is None else jy
            joints[b, k, 0], joints[b, k, 1], vis[b, k, 0] = jx, jy, v
            table[(b, k)] = (kx, ky, v, s)
    return joints, vis, table


def f64_reference(case, joints, vis):
    """Target [B,S,K,H,W] in f64 and weights [B,S,K] in f32, by the reference's geometry (generateTarget.py) with the
    Gaussian evaluated in f64.  Non-finite joints in modes 0 and 2, where the reference's int() raises, follow the
    kernels' rule: the bound comparisons with NaN are false (weight kept, nothing drawn), ±inf puts the patch outside
    (weight 0)."""
    W, H = case.hw
    fx, fy = case.feat()
    B, K = joints.shape[:2]
    S = len(case.sigmas)
    T = np.zeros((B, S, K, H, W))
    Wt = np.zeros((B, S, K), F32)
    xs, ys = np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64)
    for s, sig in enumerate(case.sigmas):
        tmp = sig * 3
        for b in range(B):
            for k in range(K):
                mx, ulx, brx = axis_geom(joints[b, k, 0], fx, tmp, case.mode)
                my, uly, bry = axis_geom(joints[b, k, 1], fy, tmp, case.mode)
                w = F32(vis[b, k, 0])
                if ulx >= W or uly >= H or brx < 0 or bry < 0:
                    w = F32(0)
                Wt[b, s, k] = w
                if not w > 0.5:
                    continue
                if case.mode == 1:
                    with np.errstate(invalid="ignore"):
                        T[b, s, k] = np.exp(-((xs[None, :] - mx) ** 2 + (ys[:, None] - my) ** 2) / (2 * sig ** 2))
                    continue
                if not (math.isfinite(mx) and math.isfinite(my)):
                    continue
                half = math.floor((2 * tmp + 1) / 2)
                x0 = half + (mx - math.trunc(mx + 0.5) if case.mode == 2 else 0.0)
                y0 = half + (my - math.trunc(my + 0.5) if case.mode == 2 else 0.0)
                inx = (xs >= ulx) & (xs < brx)
                iny = (ys >= uly) & (ys < bry)
                g = np.exp(-(((xs - ulx) - x0)[None, :] ** 2 + ((ys - uly) - y0)[:, None] ** 2) / (2 * sig ** 2))
                T[b, s, k] = np.where(iny[:, None] & inx[None, :], g, 0.0)
    return T, Wt


def oracle_targets(case, joints, vis):
    """oracle/np_oracle.py render_targets on the case, [B,S,K,H,W] f32 and [B,S,K] f32.  In modes 0 and 2 the joints the
    reference cannot take (int() of NaN or inf raises) are swapped for a far-outside one first; the caller does not
    compare those planes with it."""
    j3 = joints[..., :3].copy() if joints.shape[2] >= 3 else np.concatenate([joints, np.ones_like(joints[..., :1])], -1)
    v3 = np.repeat(vis[..., :1], 3, -1)
    bad = ~np.isfinite(j3[..., :2]).all(-1)
    if case.mode != 1:
        j3[bad, :2] = -1e4
    with np.errstate(all="ignore"):
        t, w = O.render_targets(j3, v3, case.img, case.hw, case.sigma, unbiased=case.mode)
    B, K = joints.shape[:2]
    S = len(case.sigmas)
    return t.reshape(B, S, K, *t.shape[-2:]), w.reshape(B, S, K), bad


def ulp_of(x):
    x = np.abs(np.asarray(x, np.float64))
    e = np.floor(np.log2(np.maximum(x, TINY)))
    return np.maximum(2.0 ** (e - 23), 2.0 ** -149)


def test_case_table_conditions():
    """CPU: every joint of every case meets the geometric condition it was built for, exactly, in f64; the table
    reaches every kind somewhere; and the f64 reference agrees with oracle/np_oracle.py."""
    seen = set()
    for case in CASES:
        joints, vis, table = build_inputs(case)
        W, H = case.hw
        fx, fy = case.feat()
        for (b, k), (kx, ky, v, s) in table.items():
            tmp = case.sigmas[s] * 3
            assert kind_holds(kx, joints[b, k, 0], W, fx, tmp, case.mode), (case.name, b, k, kx)
            assert kind_holds(ky, joints[b, k, 1], H, fy, tmp, case.mode), (case.name, b, k, ky)
            assert F32(vis[b, k, 0]) == F32(v)
            seen.update((kx, ky))
        ref, rw = f64_reference(case, joints, vis)
        ot, ow, bad = oracle_targets(case, joints, vis)
        keep = np.ones(rw.shape, bool) if case.mode == 1 else ~np.broadcast_to(bad[:, None, :], rw.shape)
        assert np.array_equal(rw[keep], ow[keep]), case.name
        r32 = ref.astype(F32)[keep]
        o32 = ot[keep]
        assert np.array_equal(np.isnan(r32), np.isnan(o32)), case.name
        assert np.array_equal(r32 == 0, o32 == 0), case.name
        if case.mode == 0:
            # the reference evaluates the integer-centre patch in f32 (exp of an f32 argument); the f64 restatement
            # is the better value, within the rounding of that argument (|arg| <= 18 * 2^-24 relative) and f32 exp
            fin = np.isfinite(r32)
            assert np.all(np.abs(r32[fin].astype(np.float64) - o32[fin]) <= 24 * 2.0 ** -24 * o32[fin] + 2.0 ** -149)
        else:
            assert np.array_equal(r32, o32, equal_nan=True), case.name
    assert seen >= set(AXIS_KINDS) | {"nan"}, set(AXIS_KINDS) - seen


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
def last_path():
    r = L.K1LaunchInfo()
    L.check(L.lib().lhn_k1_last_launch(ctypes.byref(r)), "lhn_k1_last_launch")
    return r.path                                    # 1 = team kernel, 2 = CTA-per-plane kernel


def _set_env(monkeypatch, force_cta):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    if force_cta:
        monkeypatch.setenv("LHN_FORCE_CTA_KERNEL", "1")


def _render(case, loss_mode, value=0.5):
    return dict(loss_mode=loss_mode, image_size=case.img, sigma=case.sigma, unbiased=case.mode, pos_value=value)


def _shape(case, B):
    W, H = case.hw
    S = len(case.sigmas)
    return (B, S, case.K, H, W) if isinstance(case.sigma, list) else (B, case.K, H, W)


def _np5(t, case, B):
    W, H = case.hw
    return t.detach().cpu().numpy().reshape(B, len(case.sigmas), case.K, H, W)


def read_targets(case, jd, vd, B):
    """The target as lhn_render_targets, lhn_render_loss_backward, its _cond recompute and lhn_render_loss_grad
    draw it, [B,S,K,H,W] f32 each (the readouts are grad = -(w * T); T is recovered where w is 1 or 2, elsewhere the
    caller compares -(w * T) itself), and the weights each returns."""
    t, tw = ops.render_targets(jd, vd, case.img, case.hw, case.sigma, unbiased=case.mode)
    hm0 = torch.zeros(_shape(case, B), dtype=torch.float32, device=DEV)
    dist = _render(case, L.LOSS_DISTANCE)
    sums = torch.tensor([0.0, 0.0, 0.0, 2.0], dtype=torch.float64, device=DEV)
    g_bwd = ops.render_loss_backward(hm0, jd, vd, dist, sums)
    g_cond = torch.full_like(hm0, 7.0)
    rec = torch.zeros(1, dtype=torch.int32, device=DEV)
    ops.render_loss_backward_cond(hm0, jd, vd, dist, sums, g_cond, torch.tensor([0.5], device=DEV), recomputed=rec)
    one = ops.render_loss_grad(hm0, jd, vd, dist, "mean", loss_scale=hm0.numel() / 2)
    torch.cuda.synchronize()
    assert int(rec.item()) == 1, "the conditional backward did not recompute"
    return dict(rt=_np5(t, case, B), bwd=-_np5(g_bwd, case, B), cond=-_np5(g_cond, case, B),
                one=-_np5(one["grad"], case, B)), \
        dict(rt=tw.cpu().numpy().reshape(B, -1), one=one["weight"].cpu().numpy())


def run_k1(case, hm, hf, jd, vd, value, monkeypatch, force_cta):
    _set_env(monkeypatch, force_cta)
    r = ops.decode_heatmap(hm, L.MASK_NEG1, L.REFINE_NONE, hm_flip=hf, render=_render(case, L.LOSS_DISTANCE_BALANCE, value),
                           joints=jd, vis=vd)
    path = last_path()
    torch.cuda.synchronize()
    _set_env(monkeypatch, False)
    return r["partials"].cpu().numpy(), r["weight"].cpu().numpy(), path


def _dtype(name):
    return {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}[name]


def check_against_oracle(what, T, ref):
    """T (f32) within the derived bound of the f64 oracle; zero exactly where the oracle is zero (and the reverse,
    except where the oracle is below 2^-126); NaN exactly where the oracle is NaN.  Returns the largest ulp error."""
    assert np.array_equal(np.isnan(T), np.isnan(ref)), f"{what}: NaN pattern differs from the oracle"
    fin = ~np.isnan(ref)
    t64, r = T[fin].astype(np.float64), ref[fin]
    err = np.abs(t64 - r)
    bad = err > REL_BOUND * r + ABS_BOUND
    assert not bad.any(), f"{what}: {bad.sum()} elements off the oracle, worst {err.max()} at ref {r[np.argmax(err)]}"
    sure = (r == 0) | (r >= TINY)
    zt, zr = t64[sure] == 0, r[sure] == 0
    assert np.array_equal(zt, zr), f"{what}: zero pattern differs from the oracle ({(zt != zr).sum()} elements)"
    ulp = float((err / ulp_of(r)).max()) if err.size else 0.0
    MAX_ULP[what] = max(MAX_ULP.get(what, 0.0), ulp)
    return ulp


@pytest.fixture(scope="module", autouse=True)
def _report():
    t0 = time.time()
    yield
    if MAX_ULP:
        print("\nlargest error against the f64 oracle, ulp: " +
              ", ".join(f"{k} {v:.2f}" for k, v in sorted(MAX_ULP.items())) + f"; {time.time() - t0:.1f} s")


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_render_conformance(case, monkeypatch):
    joints, vis, table = build_inputs(case)
    B, K = joints.shape[:2]
    S = len(case.sigmas)
    W, H = case.hw
    ref, rw = f64_reference(case, joints, vis)
    jd, vd = torch.from_numpy(joints).to(DEV), torch.from_numpy(vis).to(DEV)
    if case.vs == 1:
        vd = vd[..., 0]                              # [B, K]: the wrappers pass vis stride 1

    # ---- 1. the same target from every kernel that writes one; 2. close to the oracle; 3. weights ---------------
    Ts, ws = read_targets(case, jd, vd, B)
    T = Ts["rt"]
    wgt = rw.reshape(B, S * K)
    wb = wgt.reshape(B, S, K)[..., None, None]
    exact = (wb == 1.0) | (wb == 2.0)                # there -T * w / w is T bit for bit
    for k in ("bwd", "cond", "one"):
        want = (wb * T).astype(F32)                  # the readouts are w * T rounded once, as the kernels multiply
        assert np.array_equal(Ts[k], want, equal_nan=True), f"{case.name}: {k} differs from lhn_render_targets"
        Tk = np.where(np.broadcast_to(exact, T.shape), Ts[k] / np.broadcast_to(wb, T.shape), T)
        assert np.array_equal(Tk, T, equal_nan=True)
    for k, w in ws.items():
        assert np.array_equal(w, wgt), f"{case.name}: {k} weights differ from the oracle"
    ulp = check_against_oracle("render_targets", T, ref)
    for k in ("bwd", "cond", "one"):
        MAX_ULP[k] = max(MAX_ULP.get(k, 0.0), ulp)

    # ---- K1, both kernels: weights, N_pos at thresholds taken from the target, per-plane sums --------------------
    g = torch.Generator(device="cpu").manual_seed(len(case.name))
    hm = (-0.2 - 0.1 * torch.rand(_shape(case, B), generator=g)).to(_dtype(case.dtype)).to(DEV)
    hf = (-0.2 - 0.1 * torch.rand(_shape(case, B), generator=g)).to(_dtype(case.dtype)).to(DEV) if case.flip else None
    hm0 = torch.zeros(_shape(case, B), dtype=torch.float32, device=DEV)
    hf0 = torch.zeros_like(hm0) if case.flip else None
    on = np.array([table[(b, k)][:2] == ("interior", "interior") and table[(b, k)][2] == 1.0
                   for b in range(B) for k in range(K)]).reshape(B, K)
    b0, k0 = np.argwhere(on)[0]
    plane = T[b0, 0, k0]
    cy, cx = np.unravel_index(np.argmax(plane), plane.shape)
    pv = plane[min(cy + 1, H - 1), min(cx + 2, W - 1)]
    probes = [0.5, pv, _up(pv), _down(pv), plane[plane > 0].min(), 0.0, -0.25, 1.0, 0.9999]
    for v in probes:
        v = float(F32(v))
        pos = T > v                                  # NaN is not a positive
        want_planes = pos.sum((-2, -1)).reshape(-1).astype(np.float64)
        with np.errstate(invalid="ignore"):
            near = np.abs(ref - v) <= REL_BOUND * np.abs(ref) + ABS_BOUND
            n_ref = int((ref > v).sum())
        assert abs(int(pos.sum()) - n_ref) <= int(near.sum()), f"{case.name} v={v}: N_pos {pos.sum()} vs oracle {n_ref}"
        for force in (False, True):
            part, wk, path = run_k1(case, hm0, hf0, jd, vd, v, monkeypatch, force)
            kname = "CTA" if force or case.cta else "team"
            assert path == (2 if force or case.cta else 1), f"{case.name}: K1 path {path}"
            assert np.array_equal(part[:, 2], want_planes), \
                f"{case.name} {kname} v={v}: per-plane N_pos differs in planes {np.nonzero(part[:, 2] != want_planes)[0][:8]}"
            assert np.array_equal(wk, wgt), f"{case.name} {kname}: weights"
        one = ops.render_loss_grad(hm0, jd, vd, _render(case, L.LOSS_DISTANCE_BALANCE, v))
        s1 = one["sums"].cpu().numpy()
        assert s1[2] == pos.sum(), f"{case.name} one-pass v={v}: N_pos {s1[2]} vs {pos.sum()}"

    # ---- 5. per-plane S_pos / S_neg at 0.5 against an f64 recomputation from (hm, T, w) ------------------------
    h64 = _np5(hm.float(), case, B).astype(np.float64)
    with np.errstate(invalid="ignore"):
        ell = (h64 - T.astype(np.float64)) ** 2 * wgt.reshape(B, S, K)[..., None, None]
    pos = T > 0.5
    sp = np.where(pos, ell, 0).sum((-2, -1)).reshape(-1)
    sn = np.where(pos, 0, ell).sum((-2, -1)).reshape(-1)
    sall = sp + sn
    # The check must resolve one border pixel: on every drawn plane, the smallest target >= 0.01 (the patch edge at
    # 3 sigma is exp(-4.5) ~ 0.011) moved to 0 must change the plane's sum by more than twice the tolerance.
    rtol = 1e-6
    T64 = T.astype(np.float64)
    with np.errstate(invalid="ignore"):
        edge = np.where(T64 >= 0.01, T64, np.inf).reshape(B * S * K, -1)
    e = np.argmin(edge, 1)
    drawn = np.isfinite(edge[np.arange(B * S * K), e])
    he, te = h64.reshape(B * S * K, -1)[np.arange(B * S * K), e], T64.reshape(B * S * K, -1)[np.arange(B * S * K), e]
    moved = np.abs((he - te) ** 2 - he ** 2) * wgt.reshape(-1)
    assert drawn.sum() > 0 and (rtol * sall[drawn] < 0.5 * moved[drawn]).all(), "the sums check would miss a border pixel"
    for force in (False, True):
        part, _, _ = run_k1(case, hm, hf, jd, vd, 0.5, monkeypatch, force)
        for i, want in ((0, sp), (1, sn)):
            got = part[:, i]
            assert np.array_equal(np.isnan(got), np.isnan(want)), f"{case.name} force_cta={force}: NaN pattern of sum {i}"
            f = ~np.isnan(want)
            d = np.abs(got[f] - want[f])
            tol = rtol * np.where(np.isnan(sall[f]), 0.0, sall[f]) + 1e-300    # a NaN plane's S_pos is exactly 0
            assert (d <= tol).all(), \
                f"{case.name} force_cta={force}: sum {i} off by {d.max()} (rel {(d / np.maximum(sall[f], 1e-300)).max()})"
        assert np.array_equal(part[:, 2], pos.sum((-2, -1)).reshape(-1).astype(np.float64))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", (0, 1, 2))
def test_nan_joint_planes(mode, monkeypatch):
    """A NaN joint: mode 1 follows the reference (target NaN on that plane, weight kept, N_pos not counted, S_neg, loss
    and gradient NaN); modes 0 and 2, where the reference raises, keep the weight and draw nothing.  Every other plane
    is bit-identical to a run with a finite joint in its place."""
    case = Case(f"nan-m{mode}", mode, 2.0, (256, 256), (64, 64), 21)
    B, K, W, H = 2, 21, 64, 64
    rng = np.random.default_rng(5)
    joints = np.concatenate([rng.uniform(60, 200, (B, K, 2)), np.ones((B, K, 1))], -1).astype(F32)
    vis = np.ones((B, K, 3), F32)
    nanj = joints.copy()
    nanj[0, 3, 0] = np.nan
    nanj[1, 5, 1] = np.nan
    nanj[1, 8, :2] = np.nan
    bad = np.zeros((B, K), bool)
    bad[0, 3] = bad[1, 5] = bad[1, 8] = True
    g = torch.Generator(device="cpu").manual_seed(11)
    hm = (torch.rand((B, K, H, W), generator=g) * 0.5).to(DEV)
    runs = {}
    for name, j in (("nan", nanj), ("fin", joints)):
        jd, vd = torch.from_numpy(j).to(DEV), torch.from_numpy(vis).to(DEV)
        Ts, ws = read_targets(case, jd, vd, B)
        r = dict(T=Ts, w=ws)
        for force in (False, True):
            r[f"k1{int(force)}"] = run_k1(case, hm, None, jd, vd, 0.5, monkeypatch, force)
        bal = _render(case, L.LOSS_DISTANCE_BALANCE)
        one = ops.render_loss_grad(hm, jd, vd, bal)
        r["one"] = {k: v.cpu().numpy() for k, v in one.items()}
        runs[name] = r
    n, f = runs["nan"], runs["fin"]
    keep = ~bad
    for k in ("rt", "bwd", "cond", "one"):
        assert np.array_equal(n["T"][k][:, 0][keep], f["T"][k][:, 0][keep]), k
        if mode == 1:
            assert np.isnan(n["T"][k][:, 0][bad]).all(), f"{k}: the NaN joint's target is not NaN"
        else:
            assert np.array_equal(n["T"][k][:, 0][bad], np.zeros((3, H, W), F32)), k
    for k in ("rt", "one"):
        assert np.array_equal(n["w"][k], vis[..., 0]), f"{k}: the weight of a NaN joint is its visibility"
    for force in (0, 1):
        pn, wn, _ = n[f"k1{force}"]
        pf, wf, _ = f[f"k1{force}"]
        assert np.array_equal(wn, vis[..., 0])
        assert np.array_equal(pn.reshape(B, K, 4)[keep], pf.reshape(B, K, 4)[keep]), f"force_cta={force}: other planes"
        nb = pn.reshape(B, K, 4)[bad]
        if mode == 1:
            assert (nb[:, 2] == 0).all() and (nb[:, 0] == 0).all() and np.isnan(nb[:, 1]).all(), nb
        else:
            assert np.isfinite(nb).all() and (nb[:, 2] == 0).all(), nb
    on, of = n["one"], f["one"]
    assert np.array_equal(on["weight"], vis[..., 0])
    assert on["sums"][2] == n["k1" + "0"][0][:, 2].sum(), "one-pass N_pos differs from K1's"
    gn, gf = on["grad"], of["grad"]
    if mode == 1:
        assert np.isnan(on["loss"]).all() and np.isnan(on["sums"][1])
        assert np.isnan(gn[bad]).all()
    else:
        assert np.isfinite(on["loss"]).all()
    # the finite joints' positives are counted in the finite run only, so the balanced coefficients differ; the
    # gradient of the other planes is compared under the plain distance loss, which has no N_pos
    dist = _render(case, L.LOSS_DISTANCE)
    gd = {name: ops.render_loss_grad(hm, torch.from_numpy(j).to(DEV), torch.from_numpy(vis).to(DEV), dist)["grad"].cpu().numpy()
          for name, j in (("nan", nanj), ("fin", joints))}
    assert np.array_equal(gd["nan"][keep], gd["fin"][keep])
