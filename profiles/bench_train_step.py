#!/usr/bin/env python
"""Training-step cost of the fused heatmap loss: the two-pass route against the one-pass route, side by side in one
process on the same inputs.

  two-pass  lhn_fused_render_loss_decode (as _FusedHeatmapLossFn calls it: loss only, no idx), then
            lhn_render_loss_backward                                        2 reads + 1 write of the heatmaps
  one-pass  lhn_render_loss_grad, then the no-op lhn_render_loss_backward_cond  1 read + 1 write

Device time: CUDA events around >= 50 steps after 10 warm-up steps, input sets rotated so that their heatmaps and
gradients together exceed 4x L2; every measurement is repeated (the routes alternate) and the median and the
min-max spread are reported.  Also: CUDA-graph replay of the same steps (back-to-back kernels, no host), each
main kernel on its own, and the eager autograd step `loss, _ = crit(out, meta); loss.backward()` with the default
criterion and with one_pass_grad.  Bytes are algorithmic (heatmap reads + gradient writes); the fraction is of the
measured 6540.5 GB/s copy peak.

python profiles/bench_train_step.py [--steps 50] [--repeats 5] [--out FILE]"""
import argparse
import ctypes as C
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from litehandnet_b200 import _lib as L, ops, synth  # noqa: E402
from litehandnet_b200 import loss as LS  # noqa: E402

DEV = torch.device("cuda", 0)
PEAK_GBS = 6540.5
IMG = (256, 256)

# name, heatmap shape, dtype, sigma
SHAPES = [
    ("1024x21x64x64 f32", (1024, 21, 64, 64), torch.float32, 2.0),
    ("1024x21x64x64 bf16", (1024, 21, 64, 64), torch.bfloat16, 2.0),
    ("64x21x64x64 f32 (reference training batch)", (64, 21, 64, 64), torch.float32, 2.0),
    ("1024x21x56x56 f32", (1024, 21, 56, 56), torch.float32, 2.0),
    ("256x2x21x64x64 f32, sigma [2, 3]", (256, 2, 21, 64, 64), torch.float32, [2.0, 3.0]),
]


def gpu_info():
    name = torch.cuda.get_device_name(DEV)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                                    # read-only query; report what is missing
        q = f"nvidia-smi unavailable ({type(e).__name__})"
    return name, q


class Case:
    """Rotating input sets of one shape with every pointer and argument of the four library calls prepared."""

    def __init__(self, shape, dtype, sigma):
        self.shape, self.dtype = shape, dtype
        B, K, H, W = shape[0], shape[-3], shape[-2], shape[-1]
        S = shape[1] if len(shape) == 5 else 1
        self.B, self.K, self.S, self.H, self.W = B, K, S, H, W
        esz = torch.finfo(dtype).bits // 8
        self.hm_bytes = B * S * K * H * W * esz
        l2 = torch.cuda.get_device_properties(DEV).L2_cache_size
        self.nsets = max(2, math.ceil(4 * l2 / (2 * self.hm_bytes)))   # heatmaps + gradients of all sets > 4x L2
        self.render = dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=IMG, sigma=sigma, unbiased=True, pos_value=0.5)
        self.rp = ops._render_params(L.LOSS_DISTANCE_BALANCE, IMG, sigma, True, 0.5)
        self.dp = ops._decode_params(L.MASK_NEG1, L.REFINE_NONE, L.XFORM_NONE)
        self.sets = []
        for r in range(self.nsets):
            j, v = synth.hand_joints(B, K, IMG, seed=r, device=DEV)
            g = torch.Generator(device=DEV).manual_seed(r)
            hm = (torch.rand(shape, generator=g, device=DEV) * 0.9).to(dtype)
            vis = v[..., :1].contiguous()
            self.sets.append(dict(hm=hm, j=j.contiguous(), v=vis, grad=torch.empty_like(hm),
                                  weight=torch.empty(B, S * K, device=DEV), hmk=torch.empty(B, S * K, 3, device=DEV),
                                  kp=torch.empty(B, S * K, 3, device=DEV)))
        self.sums = torch.zeros(4, dtype=torch.float64, device=DEV)
        self.loss = torch.zeros(1, device=DEV)
        self.one = torch.ones(1, device=DEV)
        self.used = torch.zeros(1, device=DEV)
        self.fws = ops.fused_workspace(DEV, B, K, S)
        self.gws = ops.render_loss_grad_workspace(DEV, B, K, S)
        self.lib = L.lib()
        self.code = L.dtype_code(self.sets[0]["hm"])
        self.sb = S * K * H * W
        self.sc = H * W

    def _p(self, i):
        return self.sets[i % self.nsets]

    def fwd(self, i):
        s = self._p(i)
        rc = self.lib.lhn_fused_render_loss_decode(
            L.ptr(s["hm"]), None, None, self.code, self.B, self.K, self.H, self.W, self.sb, self.sc, 0, 0, None, None,
            C.byref(self.dp), L.ptr(s["hmk"]), L.ptr(s["kp"]), None, C.byref(self.rp), L.ptr(s["j"]), 3, L.ptr(s["v"]), 1,
            L.ptr(s["weight"]), None, L.ptr(self.fws), self.fws.numel(), L.ptr(self.sums), 0, 1.0, L.ptr(self.loss),
            L.stream())
        L.check(rc, "lhn_fused_render_loss_decode")

    def bwd(self, i):
        s = self._p(i)
        rc = self.lib.lhn_render_loss_backward(L.ptr(s["hm"]), self.code, self.B, self.K, self.H, self.W, self.sb, self.sc,
                                               C.byref(self.rp), L.ptr(s["j"]), 3, L.ptr(s["v"]), 1, L.ptr(self.sums), 0,
                                               1.0, L.ptr(self.one), L.ptr(s["grad"]), L.stream())
        L.check(rc, "lhn_render_loss_backward")

    def grad(self, i):
        s = self._p(i)
        rc = self.lib.lhn_render_loss_grad(L.ptr(s["hm"]), self.code, self.B, self.K, self.H, self.W, self.sb, self.sc,
                                           C.byref(self.rp), L.ptr(s["j"]), 3, L.ptr(s["v"]), 1, L.ptr(s["weight"]),
                                           L.ptr(self.gws), self.gws.numel(), L.ptr(self.sums), 0, 1.0, L.ptr(self.loss),
                                           L.ptr(self.one), L.ptr(self.used), L.ptr(s["grad"]), L.stream())
        L.check(rc, "lhn_render_loss_grad")

    def cond(self, i):
        s = self._p(i)
        rc = self.lib.lhn_render_loss_backward_cond(L.ptr(s["hm"]), self.code, self.B, self.K, self.H, self.W, self.sb,
                                                    self.sc, C.byref(self.rp), L.ptr(s["j"]), 3, L.ptr(s["v"]), 1,
                                                    L.ptr(self.sums), 0, 1.0, L.ptr(self.one), L.ptr(self.used), None,
                                                    L.ptr(s["grad"]), L.stream())
        L.check(rc, "lhn_render_loss_backward_cond")


def time_eager(step, steps, warm=10):
    for i in range(warm):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1e3 / steps


def time_graph(step, steps, warm=10):
    for i in range(warm):
        step(i)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            for i in range(steps):
                step(i)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    g.replay()
    e1.record()
    torch.cuda.synchronize()
    del g
    return e0.elapsed_time(e1) * 1e3 / steps


def stats(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2], xs[0], xs[-1]


def fmt(name, us, nbytes):
    med, lo, hi = us
    gbs = nbytes / (med * 1e-6) / 1e9
    return f"  {name:<44s} {med:9.2f} us  [{lo:8.2f} .. {hi:8.2f}]  {nbytes / 1e6:8.1f} MB  {gbs:7.1f} GB/s  {gbs / PEAK_GBS:6.1%}"


def autograd_rows(c, steps, repeats, out):
    """Eager autograd step through TopdownHeatmapLoss, default criterion vs one_pass_grad (4-D shapes only)."""
    from oracle.ref_loader import _AttrDict
    cfg = lambda op: _AttrDict(  # noqa: E731
        DATASET=dict(image_size=list(IMG), heatmap_size=[c.W, c.H], num_joints=c.K),
        PIPELINE=dict(unbiased_encoding=True, kernel=(11, 11), use_udp=False, simdr_split_ratio=0, sigma=2),
        MODEL=dict(name="litehandnet"),
        LOSS=dict(type="TopdownHeatmapLoss", loss_weight=[1.0, 1.0], auto_weight=False, one_pass_grad=op))
    crits = {"default": LS.get_loss(cfg(False)), "one_pass_grad": LS.get_loss(cfg(True))}
    leaves = [s["hm"].detach().clone().requires_grad_(True) for s in c.sets]
    metas = [dict(joints_3d=s["j"], joints_3d_visible=s["v"]) for s in c.sets]

    def step_of(crit):
        def step(i):
            x = leaves[i % len(leaves)]
            x.grad = None
            loss, _ = crit(x, metas[i % len(metas)])
            loss.backward()
        return step
    res = {k: [] for k in crits}
    for _ in range(repeats):
        for k, crit in crits.items():
            res[k].append(time_eager(step_of(crit), steps))
    for k in crits:
        med, lo, hi = stats(res[k])
        out(f"  autograd step, {k:<30s} {med:9.2f} us  [{lo:8.2f} .. {hi:8.2f}]  (host-bound: includes .item())")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_train_step.py needs a CUDA device")
    lines = []

    def out(s=""):
        print(s, flush=True)
        lines.append(s)
    name, q = gpu_info()
    out(f"# GPU: {name}; nvidia-smi name, power.limit, clocks.max.sm: {q}")
    out(f"# steps {args.steps} after 10 warm-ups, {args.repeats} repeats (routes alternate); "
        f"median [min .. max]; fraction of {PEAK_GBS} GB/s")
    for label, shape, dtype, sigma in SHAPES:
        c = Case(shape, dtype, sigma)
        two = 3 * c.hm_bytes
        one = 2 * c.hm_bytes
        out(f"\n== {label}: {c.nsets} rotating input sets ({c.nsets * 2 * c.hm_bytes / 1e6:.0f} MB of heatmaps + gradients)")
        # correctness of what is timed: same gradient bits, same N_pos, on set 0
        c.fwd(0); c.bwd(0)
        g2, s2 = c.sets[0]["grad"].clone(), c.sums.clone()
        c.grad(0); c.cond(0)
        torch.cuda.synchronize()
        same = torch.equal(c.sets[0]["grad"], g2) and float(c.sums[2]) == float(s2[2]) and float(c.sums[3]) == float(s2[3])
        out(f"  gradient bit-identical to the two-pass route, same N_pos and numel: {same}")
        routes = {
            "two-pass step (fused fwd + backward)": (lambda i: (c.fwd(i), c.bwd(i)), two),
            "one-pass step (loss_grad + no-op cond)": (lambda i: (c.grad(i), c.cond(i)), one),
            "  fused forward alone (1R)": (c.fwd, c.hm_bytes),
            "  lhn_render_loss_backward alone (1R+1W)": (c.bwd, one),
            "  lhn_render_loss_grad alone (1R+1W)": (c.grad, one),
            "  lhn_render_loss_backward_cond no-op alone": (c.cond, 0),
        }
        for mode, timer in (("eager, CUDA events", time_eager), ("CUDA-graph replay", time_graph)):
            res = {k: [] for k in routes}
            for _ in range(args.repeats):
                for k, (fn, _) in routes.items():
                    res[k].append(timer(fn, args.steps))
            out(f" {mode}:")
            for k, (fn, nb) in routes.items():
                out(fmt(k, stats(res[k]), nb))
            t2, t1 = stats(res["two-pass step (fused fwd + backward)"])[0], stats(res["one-pass step (loss_grad + no-op cond)"])[0]
            out(f"  one-pass / two-pass: {t1 / t2:.3f}  ({t2 / t1:.2f}x faster)")
        if len(shape) == 4:
            autograd_rows(c, args.steps, args.repeats, out)
        del c
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
