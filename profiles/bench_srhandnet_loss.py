"""SRHandNetLoss forward + backward for one training step, four routes, on one GPU:
  (a) today's route with the targets rendered on the GPU (render_srhandnet_targets, pred_bbox=False: one
      lhn_render_targets per scale), then lhn_loss_mse_multi and one lhn_loss_backward per scale;
  (b) today's route with the targets already resident (the dataloader case): lhn_loss_mse_multi + 4 backward launches;
  (c) the fused route: lhn_render_loss_multi + lhn_render_loss_backward_multi;
  (d) the fused route in one pass (cfg.LOSS.one_pass_grad): lhn_render_loss_grad_multi (count + stream launch) +
      lhn_render_loss_backward_multi_cond (a no-op for loss.backward()).
Reports CUDA-graph replay and eager medians per step, the fused kernels' times and their share of the copy peak
(bytes from shapes: the forward reads the outputs, the backward and the one-pass call read them and write the
gradients), launches per step, and parity checks of (a) against (c) and of (d) against (c) (loss relative difference,
gradients bit for bit).  Inputs rotate over more than the 126 MB L2 (the line says how many sets).

    python profiles/bench_srhandnet_loss.py [--out profiles/r05_srhandnet_one_pass.txt]
"""
import argparse
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from litehandnet_b200 import _lib as L  # noqa: E402
from litehandnet_b200 import loss as LS, ops, synth  # noqa: E402
from litehandnet_b200.render import render_srhandnet_targets  # noqa: E402

COPY_PEAK = 6540.5e9          # B/s: device-to-device copy rate measured on this B200 (profiles/r01_bw_probe.txt)
IMG = (256, 256)
LW = [0.3, 0.3, 0.5, 1.0]
SIGMAS = [2, 2, 2, 2]
ROTATE_BYTES = 256 << 20
DT = {"f32": torch.float32, "bf16": torch.bfloat16}


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        return f"{torch.cuda.get_device_name()} (power limit not read: {e})"


def make_sets(B, K, sizes, dtype):
    one = sum(B * K * s * s for s in sizes) * torch.finfo(DT[dtype]).bits // 8
    n = max(1, min(16, math.ceil(ROTATE_BYTES / one)))
    sets = []
    for i in range(n):
        g = torch.Generator(device="cpu").manual_seed(i)
        outs = [(torch.rand((B, K, s, s), generator=g) * 0.9).to(DT[dtype]).to("cuda").requires_grad_(True)
                for s in sizes]
        j, v = synth.hand_joints(B, K, IMG, seed=100 + i)
        j, v = j.cuda(), v.cuda()
        tg, tw = render_srhandnet_targets(j, v, None, IMG, [[s, s] for s in sizes], SIGMAS, pred_bbox=False,
                                          unbiased_encoding=False)
        sets.append(dict(outs=outs, j=j, v=v, tg=tg, tw=tw))
    return sets, one, n


def render_dict():
    return dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=IMG, sigma=SIGMAS, unbiased=False, pos_value=0.5)


def step_fn(route, sizes):
    n = len(sizes)

    def explicit(outs, tg, tw):
        return LS._MultiHeatmapLossFn.apply(L.LOSS_DISTANCE_BALANCE, 0.5, "mean", LW, n, *outs, *tg, *tw)

    def run(s):
        for o in s["outs"]:
            o.grad = None
        if route == "a":
            tg, tw = render_srhandnet_targets(s["j"], s["v"], None, IMG, [[x, x] for x in sizes], SIGMAS,
                                              pred_bbox=False, unbiased_encoding=False)
            loss = explicit(s["outs"], tg, tw)
        elif route == "b":
            loss = explicit(s["outs"], s["tg"], s["tw"])
        elif route == "d":
            loss = LS._FusedMultiHeatmapLossOnePassFn.apply(render_dict(), "mean", LW, 1.0, s["j"], s["v"], *s["outs"])
        else:
            loss = LS._FusedMultiHeatmapLossFn.apply(render_dict(), "mean", LW, s["j"], s["v"], *s["outs"])
        loss.backward()
        return loss
    return run


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def time_eager(fn, sets, reps):
    for s in sets:
        fn(s)
    torch.cuda.synchronize()
    ts = []
    for r in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn(sets[r % len(sets)])
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return median(ts)


def time_graph(fn, sets, reps):
    graphs = []
    st = torch.cuda.Stream()
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        for s in sets:
            for _ in range(2):
                fn(s)
    torch.cuda.current_stream().wait_stream(st)
    torch.cuda.synchronize()
    for s in sets:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn(s)
        graphs.append(g)
    for g in graphs:
        g.replay()
    torch.cuda.synchronize()
    ts = []
    for r in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        graphs[r % len(graphs)].replay()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return median(ts)


def time_kernels(sets, reps):
    """Each new kernel alone: events around `reps` back-to-back launches over the rotating sets."""
    rd = render_dict()
    fw = [ops.render_loss_multi([o.detach() for o in s["outs"]], s["j"], s["v"], rd, LW, "mean", want_weights=False)
          for s in sets]
    torch.cuda.synchronize()

    def loop(f):
        f(0)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for r in range(reps):
            f(r % len(sets))
        e1.record()
        e1.synchronize()
        return e0.elapsed_time(e1) * 1e3 / reps

    tf = loop(lambda i: ops.render_loss_multi([o.detach() for o in sets[i]["outs"]], sets[i]["j"], sets[i]["v"], rd, LW,
                                              "mean", want_weights=False))
    tb = loop(lambda i: ops.render_loss_backward_multi([o.detach() for o in sets[i]["outs"]], sets[i]["j"],
                                                       sets[i]["v"], rd, fw[i][1], LW, "mean"))
    tg = loop(lambda i: ops.render_loss_grad_multi([o.detach() for o in sets[i]["outs"]], sets[i]["j"], sets[i]["v"],
                                                   rd, LW, "mean", want_weights=False))
    op = [ops.render_loss_grad_multi([o.detach() for o in s["outs"]], s["j"], s["v"], rd, LW, "mean", want_weights=False)
          for s in sets]
    one = torch.ones(1, device="cuda")
    tcnd = loop(lambda i: ops.render_loss_backward_multi_cond([o.detach() for o in sets[i]["outs"]], sets[i]["j"],
                                                              sets[i]["v"], rd, op[i][1], op[i][3], op[i][4], LW,
                                                              "mean", one))
    return tf, tb, tg, tcnd


def launches(fn, s):
    from torch.profiler import ProfilerActivity, profile
    fn(s)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn(s)
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and
               "memcpy" not in e.name.lower() and "memset" not in e.name.lower())


def one_pass_kernels(sizes, sets, reps=20):
    """Device time of each kernel of route (d), from torch.profiler over `reps` steps in a run of their own: the count,
    the stream and the conditional backward (mean per step, us)."""
    from torch.profiler import ProfilerActivity, profile
    fn = step_fn("d", sizes)
    fn(sets[0])
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for r in range(reps):
            fn(sets[r % len(sets)])
        torch.cuda.synchronize()
    t = {"count": 0.0, "stream": 0.0, "cond": 0.0}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        key = ("count" if "render_count_multi_kernel" in e.name else "stream" if "render_loss_grad_multi_kernel" in e.name
               else "cond" if "render_loss_backward_multi_kernel" in e.name else None)
        if key:
            t[key] += e.time_range.elapsed_us()
    return {k: v / reps for k, v in t.items()}


def parity(sizes, s):
    fa, fc, fd = step_fn("a", sizes), step_fn("c", sizes), step_fn("d", sizes)
    la = fa(s).item()
    ga = [o.grad.clone() for o in s["outs"]]
    lc = fc(s).item()
    gc = [o.grad.clone() for o in s["outs"]]
    ld = fd(s).item()
    gd = [o.grad.clone() for o in s["outs"]]
    dg = max(((x.float() - y.float()).abs().max() / y.float().abs().max().clamp_min(1e-30)).item() for x, y in zip(gc, ga))
    same = sum(int(torch.equal(x.view(torch.int16 if x.element_size() == 2 else torch.int32),
                               y.view(torch.int16 if y.element_size() == 2 else torch.int32))) for x, y in zip(gd, gc))
    return abs(lc - la) / abs(la), dg, abs(ld - lc) / abs(lc), same


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.abspath(__file__)), "r04_srhandnet_loss.txt"))
    ap.add_argument("--reps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a GPU")
    lines = [f"# SRHandNetLoss forward + backward per step, K = 21, DistanceLoss balance, mean; {gpu_info()}",
             "# eager / graph: median per step (us) of CUDA-event-timed steps over rotating input sets; kernel: mean "
             "per launch of back-to-back launches; share = shape bytes / time / 6540.5 GB/s copy peak"]
    for sizes in ([16, 16, 32, 64], [14, 14, 28, 56]):
        for B in (64, 1024):
            for dtype in ("f32", "bf16"):
                sets, nbytes, nsets = make_sets(B, 21, sizes, dtype)
                row = f"sizes={sizes} B={B} {dtype}: outputs {nbytes / 1e6:.1f} MB x {nsets} sets " \
                      f"({nbytes * nsets / 2**20:.0f} MiB rotated)"
                lines.append(row)
                for route, label in (("a", "(a) render + explicit"), ("b", "(b) resident targets"), ("c", "(c) fused"),
                                     ("d", "(d) fused, one pass")):
                    fn = step_fn(route, sizes)
                    te = time_eager(fn, sets, args.reps)
                    tgph = time_graph(fn, sets, args.reps)
                    nl = launches(fn, sets[0])
                    lines.append(f"  {label:24s} eager {te:9.1f} us  graph {tgph:9.1f} us  launches/step {nl}")
                tf, tb, tg, tcnd = time_kernels(sets, args.reps)
                lines.append(f"  lhn_render_loss_multi          {tf:9.1f} us  {nbytes / tf / 1e3:7.1f} GB/s  "
                             f"{100 * nbytes / (tf * 1e-6) / COPY_PEAK:5.1f} % of copy peak")
                lines.append(f"  lhn_render_loss_backward_multi {tb:9.1f} us  {2 * nbytes / tb / 1e3:7.1f} GB/s  "
                             f"{100 * 2 * nbytes / (tb * 1e-6) / COPY_PEAK:5.1f} % of copy peak")
                lines.append(f"  lhn_render_loss_grad_multi     {tg:9.1f} us  {2 * nbytes / tg / 1e3:7.1f} GB/s  "
                             f"{100 * 2 * nbytes / (tg * 1e-6) / COPY_PEAK:5.1f} % of copy peak  (count + stream launch)")
                lines.append(f"  lhn_render_loss_backward_multi_cond, upstream as assumed {tcnd:9.1f} us (host-bound loop)")
                kt = one_pass_kernels(sizes, sets)
                lines.append(f"  (d) kernels, profiler: count {kt['count']:6.1f} us, stream {kt['stream']:6.1f} us "
                             f"({100 * 2 * nbytes / (kt['stream'] * 1e-6) / COPY_PEAK:5.1f} % of copy peak), "
                             f"conditional backward {kt['cond']:5.1f} us")
                dl, dg, dd, same = parity(sizes, sets[0])
                lines.append(f"  parity (a) vs (c): loss rel {dl:.2e}, gradient max |diff| / max |grad| {dg:.2e}")
                lines.append(f"  parity (d) vs (c): loss rel {dd:.2e}, gradients bit-equal {same} / {len(sizes)}")
                print("\n".join(lines[-12:]), flush=True)
                del sets
                torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
