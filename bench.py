#!/usr/bin/env python
"""bench.py — benchmark of the B200-native heatmap hot path (BASELINE.json configs 1-5).

  python bench.py [--config C] --gpus N --steps K --warmup W     (torchrun launches N ranks for N > 1)
  python bench.py --impl reference [--config C] ...              the reference's own CPU path on the host cores
  python bench.py ... --dump-outputs DIR                         also write the last timed step's outputs as .npy

--config (default 2 = the headline, BASELINE.json configs[1]; the other four are the parity-test shapes, measured
to the same contract):
  1  decode: argmax + quarter-offset ('default') + transform_preds, 21x64x64, batch 64       (lhn_decode_heatmap)
  2  fused Gaussian render + balanced target-weight MSE + flip average + DARK k=11 + transform_preds,
     21x64x64, batch 1024 per GPU                                                  (lhn_fused_render_loss_decode)
  3  SimDR decode k=2, 2 x [4096,21,512]                                                   (lhn_decode_simdr_flags)
  4  MPII 16x64x64 decode + PCK@0.2/AUC/EPE counters, batch 1024 per GPU; at N > 1 the int64 counter block is
     all-reduced EVERY eval step (NCCL) and must equal a monolithic run bit for bit         (lhn_decode_heatmap_pck)
  5  21x128x128 fused render + loss + DARK (no flip plane), GLOBAL batch 8192 sharded over the N GPUs (strong)

One JSON line on stdout (rank 0).  `value` = device-resident throughput (CUDA events, max over ranks);
`e2e` = the same step through the public host-buffer API (pinned host inputs, H2D + kernels + D2H inside the timed
region); `roofline` = the dominant kernel's algorithmic bytes / its event-timed duration vs the measured HBM peak;
`cpu_baseline` = the reference's own functions (oracle/_ref, `kind: "reference"`) or the numpy port timed on this
box's host cores on a bounded sample; `parity` = the outputs of the MEASURED path against the oracle (the run
exits non-zero when it is out of tolerance).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

UNIT = "samples/s"
FALLBACK_HBM_GBS = 6650.0            # /opt/skills/guides/B200_PROFILING.md fallback
PCIE_GEN5_X16_GBS = 63.0             # theoretical PCIe 5.0 x16 payload rate per direction (the e2e ceiling)

METRICS = {
    1: "heatmap decode (argmax + quarter offset) samples/s @21x64x64",
    2: "heatmap render+loss+decode samples/s @21x64x64",
    3: "SimDR 1D-logit decode samples/s @2x21x512",
    4: "heatmap decode + PCK/AUC/EPE samples/s @16x64x64",
    5: "heatmap render+loss+decode samples/s @21x128x128",
}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs: copy, read+write bytes, burst)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(cfg_id, batch):
    """dram bytes per launch of the dominant kernel from a committed ncu --set full capture of this workload
    (profiles/traffic.json; RECORDED in an earlier profiled run, not measured by this run)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f)
        ent = t.get("configs", {}).get(str(cfg_id)) or (t if cfg_id == 2 else None)
        if ent and int(ent.get("batch", -1)) == int(batch):
            return float(ent["dram_bytes_per_launch"])
    except Exception:
        pass
    return None


def _clock_proc(index, interval_s, active, stop, out):
    """Sampler PROCESS (no GIL shared with the launch loop, which starves a sampler thread down to one sample per
    timed region): SM clock + throttle reasons through NVML while `active` is set, until `stop`."""
    try:
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(index)
        max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        names = {"hw_slowdown": nv.nvmlClocksThrottleReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksThrottleReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksThrottleReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksThrottleReasonSwPowerCap}
        samples, reasons = [], set()
        out.put("ready")
        while not stop.is_set():
            if active.is_set():
                samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for n, bit in names.items():
                    if r & bit:
                        reasons.add(n)
            time.sleep(interval_s)
        out.put((samples, sorted(reasons), max_mhz))
    except Exception as e:                                   # no NVML: report nothing rather than die
        out.put("ready")
        out.put(([], [f"sampler error: {type(e).__name__}"], None))


class ClockSampler:
    """SM clock + throttle reasons sampled by a separate process while the timed region runs."""

    def __init__(self, index, interval_s=0.0005):
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        self.active, self._stop, self.q = ctx.Event(), ctx.Event(), ctx.Queue()
        self.p = ctx.Process(target=_clock_proc, args=(index, interval_s, self.active, self._stop, self.q), daemon=True)
        self.ok = True

    def start(self):
        """Start the process and wait until NVML is initialised in it (before the barrier: nvmlInit takes
        milliseconds); sampling itself begins with begin()."""
        try:
            self.p.start()
            self.q.get(timeout=20)
        except Exception:
            self.ok = False

    def begin(self):
        self.active.set()

    def stop(self):
        self.active.clear()
        self._stop.set()
        samples, reasons, max_mhz = [], [], None
        if self.ok:
            try:
                samples, reasons, max_mhz = self.q.get(timeout=10)
                self.p.join(timeout=5)
            except Exception:
                pass
        s = sorted(samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": max_mhz, "reasons": reasons, "samples": len(s),
                "how": "NVML from a sampler process during the timed region"}


def physical_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


def coord_check(got, ref, mag):
    """Element-wise |a-b| <= 2e-5 + 1e-5 max(|b|, mag) (tests/conftest.py::assert_coords_close): mag is the size of
    the terms of transform_preds, |c| + |100 s| — image coordinates near 0 are differences of terms that large.
    Returns (ok, max relative deviation against max(|b|, mag, 1))."""
    import numpy as np
    got = np.asarray(got, np.float64); ref = np.asarray(ref, np.float64)
    if mag is None:
        m = np.abs(ref)
    else:
        m = np.maximum(np.abs(ref), np.broadcast_to(mag, ref.shape))
    d = np.abs(got - ref)
    nan_ok = np.array_equal(np.isnan(got), np.isnan(ref))
    ok = bool(nan_ok and (np.nan_to_num(d) <= 2e-5 + 1e-5 * np.nan_to_num(m)).all())
    rel = float(np.nanmax(d / np.maximum(m, 1.0))) if d.size else 0.0
    return ok, rel


def xform_mag(center, scale):
    import numpy as np
    return (np.abs(np.asarray(center, np.float64)) + 100.0 * np.abs(np.asarray(scale, np.float64)))[:, None, :]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outputs, batch, directory, limit=DUMP_LIMIT_BYTES):
    """Write every output as DIR/<name>.npy so that two builds can be compared array for array.  Floating-point
    arrays keep f32/f64; integer ones are written as f64 (exact below 2^53).  When the arrays exceed `limit` bytes
    in all, every per-sample array ([batch, ...]) keeps the same seeded sample of rows, whose row numbers go to
    sample_rows.npy; the aggregates (loss, sums, counters) are written whole."""
    import numpy as np
    arrays = {}
    for name, t in outputs.items():
        a = t.detach().cpu().numpy()
        arrays[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    per_sample = [n for n, a in arrays.items() if a.ndim >= 2 and a.shape[0] == batch]
    header = 128                                     # bytes of an .npy header
    total = sum(a.nbytes + header for a in arrays.values())
    if total > limit:
        row_bytes = sum(arrays[n].nbytes for n in per_sample) // batch
        keep = min(batch, (limit - header - (total - row_bytes * batch)) // (row_bytes + 8))
        if not per_sample or keep < 1:
            raise ValueError(f"the outputs take {total} bytes and the arrays that are not per sample alone exceed "
                             f"the {limit}-byte dump limit: nothing can be sampled")
        rows = np.sort(np.random.default_rng(0).choice(batch, keep, replace=False))
        for n in per_sample:
            arrays[n] = arrays[n][rows]
        arrays["sample_rows"] = rows.astype(np.float64)
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a)


# =========================================================================================================
# Workloads
# =========================================================================================================
class Workload:
    """One BASELINE config: device-resident inputs, the bound launchers of the timed loop, the dominant kernel for
    the roofline, the host-buffer (e2e) path, the parity check of the measured outputs and the CPU inputs."""
    cfg_id = 0
    scaling = "weak"
    K = 21
    H = W = 64
    image_size = (256, 256)

    def __init__(self, args, rank, world, dev):
        self.args, self.rank, self.world, self.dev = args, rank, world, dev
        self.collective = "none"
        self.nccl_bytes_per_step = 0
        self.nvlink_bytes_per_step = 0

    # -- hooks -------------------------------------------------------------------------------------------
    def step(self, i):
        self.bound[i % self.R].launch()

    def kernel_step(self, i):
        b = self.bound[i % self.R]
        b.launch_kernel(b.stream())

    def end_of_epoch(self):
        pass

    def begin_epoch(self):
        pass

    def outputs(self, steps):
        """name -> device tensor: what a caller of the timed path holds after the last of `steps` timed steps."""
        raise NotImplementedError

    launches_per_step = 1


def make_set_2d(B, K, H, W, seed, dev, image_size, sigma=2.0, flip=True, margin=4.0, chunk=1024):
    """(hm, hf or None, joints, vis, center, scale) for the fused workloads, generated in chunks so that the
    generator's temporaries stay small next to an 11 GB batch."""
    import torch
    from litehandnet_b200 import synth
    hms, hfs = [], []
    for c0 in range(0, B, chunk):
        n = min(chunk, B - c0)
        hm, cen = synth.blob_heatmaps(n, K, H, W, seed=seed + 7919 * (c0 // chunk), device=dev, sigma=sigma, margin=margin)
        hms.append(hm)
        if flip:
            hfs.append(synth.flipped_blob_heatmaps(cen, H, W, seed=seed + 1 + 7919 * (c0 // chunk), device=dev, sigma=sigma))
    hm = hms[0] if len(hms) == 1 else torch.cat(hms)
    hf = None if not flip else (hfs[0] if len(hfs) == 1 else torch.cat(hfs))
    del hms, hfs
    joints, vis = synth.hand_joints(B, K, image_size, seed=seed + 2, device=dev)
    center, scale = synth.bbox_center_scale(B, seed=seed + 3, device=dev)
    return hm, hf, joints, vis, center, scale


class FusedWorkload(Workload):
    """Configs 2 and 5: render + balanced masked MSE + [flip average] + argmax + DARK + transform_preds, one launch."""

    def __init__(self, args, rank, world, dev, cfg_id):
        super().__init__(args, rank, world, dev)
        import torch
        from litehandnet_b200 import fused
        self.cfg_id = cfg_id
        if cfg_id == 2:
            self.B = args.batch or 1024
            self.flip, self.sigma = True, 2
            self.R_in = self.R = args.rotate
        else:
            self.H = self.W = 128
            self.image_size = (512, 512)
            self.global_batch = args.batch or 8192
            self.B = self.global_batch // world
            self.flip, self.sigma = False, 4
            self.scaling = "strong"
            self.R_in, self.R = 1, 2                  # one 11 GB / N input set (>> L2), two rotating OUTPUT sets
        B, K, H, W = self.B, self.K, self.H, self.W
        self.step_cfg = fused.FusedHeatmapStep(self.image_size, sigma=self.sigma, unbiased_encoding=True, balance=True,
                                               post_process="unbiased", kernel=11)
        self.sets = [make_set_2d(B, K, H, W, 1000 * rank + 10 * r + (0 if cfg_id == 2 else 50000), dev, self.image_size,
                                 sigma=float(self.sigma), flip=self.flip) for r in range(self.R_in)]
        self.global_loss = world > 1 and args.global_loss
        self.xch = None
        if self.global_loss and args.collective == "nvlink":
            from litehandnet_b200.dist import PeerExchange
            self.xch = PeerExchange(dev)
        self.epoch_loss = torch.zeros(1, dtype=torch.float32, device=dev) if (world > 1 and not self.global_loss) else None
        overlap = self.R >= 2 and not args.no_overlap
        self.overlap = overlap
        self.bound = []
        for r in range(self.R):
            s = self.sets[r % self.R_in]
            nccl_global = self.global_loss and self.xch is None
            self.bound.append(fused.BoundFusedStep(self.step_cfg, s[0], s[2], s[3], s[4], s[5], hm_flip=s[1],
                                                   finalize=not nccl_global, overlap_previous=overlap,
                                                   spare_sms=(args.spare_sms if nccl_global else 0),
                                                   accumulate_into=self.epoch_loss, exchange=self.xch))
        self.pending = []
        if world > 1:
            if self.xch is not None:
                self.collective = ("batch-global loss: the 4 f64 loss sums are all-gathered EVERY step INSIDE the kernel through "
                                   f"peer-mapped mailboxes over NVLink ({self.xch.how}) and added in rank order; no NCCL call, one launch per step")
                self.nvlink_bytes_per_step = self.xch.bytes_per_step(32)
            elif self.global_loss:
                self.collective = "ncclAllReduce of the 4 f64 loss sums EVERY step (batch-global N_pos), lhn_loss_finalize after it"
                self.nccl_bytes_per_step = 32
                self.launches_per_step = 2
            else:
                self.collective = ("per-rank loss (the reference's DDP semantics: loss/heatmapLoss.py:253-258 sees the rank's "
                                   "batch), ONE ncclAllReduce of the epoch loss sum per timed region (distributed_utils.py:65-76)")
        esz = 4
        planes = K * H * W * esz * (2 if self.flip else 1)
        self.bytes_per_launch = (planes + K * 3 * 4 + 16 + K * (12 + 12 + 4 + 4 + 32)) * B
        tw = 4 if self.flip else (2 if H == 64 else 8)
        self.kernel_name = f"heatmap_team_kernel<f32,{H}x{W},TW={tw},{'FLIP,' if self.flip else ''}LOSS,KS=11>"

    def workload(self):
        return workload_label(self.cfg_id, self.args.batch, self.world)

    def flush(self):
        while self.pending:
            work, b = self.pending.pop(0)
            work.wait()
            b.launch_finalize(b.stream())

    def step(self, i):
        import torch.distributed as dist
        b = self.bound[i % self.R]
        b.launch()
        if self.global_loss and self.xch is None:
            self.flush()
            self.pending.append((dist.all_reduce(b.sums, async_op=True), b))

    def end_of_epoch(self):
        import torch.distributed as dist
        self.flush()
        if self.epoch_loss is not None:
            self.local_epoch = self.epoch_loss.clone()     # this rank's own sum (parity), before the collective
            dist.all_reduce(self.epoch_loss)

    def begin_epoch(self):
        if self.epoch_loss is not None:
            self.epoch_loss.zero_()

    def config_extra(self):
        B, K, H, W = self.B, self.K, self.H, self.W
        return {"batch_per_gpu": B, "global_batch": B * self.world, "joints": K, "heatmap": f"{H}x{W}",
                "flip_test": self.flip, "loss": "DistanceLoss L2 balance=True",
                "decode": "argmax + DARK k=11 + transform_preds",
                "l2_policy": (f"inputs {(2 if self.flip else 1) * B * K * H * W * 4 / 1e6:.0f} MB/step > 126 MB L2, "
                              f"{self.R_in} input set(s), {self.R} rotating output sets, L2 evict_first loads")}

    def parity(self, steps):
        import numpy as np
        import torch
        from oracle import cpu_path
        from litehandnet_b200 import fused
        n_par = self.B if self.cfg_id == 2 else min(self.B, self.args.parity_samples or 512)
        idx_equal, coord_ok, max_rel, loss_rel, n = True, True, 0.0, 0.0, 0
        ref_losses = []
        for r in range(self.R_in):
            s = self.sets[r]
            runner = cpu_path.FusedCpuRunner(*[None if t is None else t[:n_par].cpu().numpy() for t in s],
                                             image_size=self.image_size, sigma=self.sigma, kernel=11)
            try:
                with np.errstate(all="ignore"):
                    preds, loss, _ = runner.run()
                ridx = runner.last_idx
            finally:
                runner.close()
            ref_losses.append(float(loss))
            for b in self.bound[r::self.R_in]:            # every output set fed by this input set
                got = b.preds[:n_par].cpu().numpy()
                idx_equal &= bool(np.array_equal(b.idx[:n_par].cpu().numpy(), ridx))
                ok, rel = coord_check(got[..., :2], preds[..., :2], xform_mag(s[4][:n_par].cpu().numpy(), s[5][:n_par].cpu().numpy()))
                coord_ok &= ok and bool(np.array_equal(got[..., 2], preds[..., 2], equal_nan=True))
                max_rel = max(max_rel, rel)
                n += n_par
        note = "loss of the timed loop's last step per set"
        if n_par < self.B:
            # the loss is a whole-batch quantity: one extra launch of the same bound step on the parity subset
            s = self.sets[0]
            b = fused.BoundFusedStep(self.step_cfg, s[0][:n_par], s[2][:n_par], s[3][:n_par], s[4][:n_par], s[5][:n_par],
                                     hm_flip=None if s[1] is None else s[1][:n_par])
            b.launch()
            torch.cuda.synchronize()
            loss_rel = abs(float(b.loss.item()) - ref_losses[0]) / abs(ref_losses[0])
            note = f"loss from one extra launch on the {n_par}-sample parity subset (the loss is a whole-batch quantity)"
        elif self.epoch_loss is not None:
            want = sum(ref_losses[(i % self.R) % self.R_in] for i in range(steps))
            loss_rel = abs(float(self.local_epoch.item()) - want) / abs(want)
            note = "epoch loss sum of this rank over the timed steps vs the sum of the per-step reference losses"
        elif self.global_loss:
            note = ("loss not compared here (the global-N_pos loss spans all ranks' inputs); tests/test_gpu_exchange.py checks it "
                    "against the oracle on the concatenated batch")
            if self.xch is not None and int(self.xch.status.item()) != 0:
                idx_equal = False
                note = "EXCHANGE TIMEOUT: a peer's block did not arrive"
        else:
            for r in range(self.R):
                lr = abs(float(self.bound[r].loss.item()) - ref_losses[r % self.R_in]) / abs(ref_losses[r % self.R_in])
                loss_rel = max(loss_rel, lr)
        tol = 5e-5 if self.epoch_loss is not None and n_par == self.B else 1e-5
        ok = idx_equal and coord_ok and loss_rel <= tol
        return {"ok": bool(ok), "idx_equal": idx_equal, "coord_within_1e-5": coord_ok, "coord_max_rel": max_rel,
                "loss_rel": loss_rel, "samples": n, "loss_note": note,
                "against": "oracle.cpu_path.FusedCpuRunner (the reference CPU pipeline restated, pinned to the executed "
                           "reference by tests/) on rank 0's inputs; outputs as the timed loop left them"}

    def e2e(self, steps, warmup):
        import torch
        from litehandnet_b200 import fused
        Be = self.B if self.cfg_id == 2 else min(self.B, 1024)
        s0 = [None if t is None else t[:Be] for t in self.sets[0]]
        host = [None if t is None else torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in s0]
        pipe = fused.HostPipeline(self.step_cfg, Be, self.K, self.H, self.W, flip=self.flip, chunks=self.args.chunks, device=self.dev)
        for _ in range(max(1, min(warmup, 3))):
            pipe(*host)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        launches = 0
        for _ in range(steps):
            pipe(*host)
            launches += pipe.launches
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return dict(seconds=dt, samples_per_step=Be, h2d=pipe.h2d_bytes, d2h=pipe.d2h_bytes, launches=launches,
                    api="litehandnet_b200.fused.HostPipeline (pinned host buffers, chunked H2D overlapped with the fused kernel)",
                    note=None if Be == self.B else f"e2e step = {Be} samples (a 1.4 GB pinned batch), not the {self.B}-sample device step")

    def cpu_inputs(self, n):
        return [None if t is None else t[:n].cpu().numpy() for t in self.sets[0]]

    def loss_check(self, steps):
        if self.epoch_loss is not None:
            return float(self.epoch_loss.item()) / (self.world * steps)
        return float(self.bound[(steps - 1) % self.R].loss.item())

    def outputs(self, steps):
        b = self.bound[(steps - 1) % self.R]
        # at N > 1 without --global-loss, b.loss is the shared accumulator: the epoch's loss sum over all ranks
        return {"preds": b.preds, "hm_preds": b.hm_preds, "idx": b.idx, "target_weight": b.weight,
                "loss_sums": b.sums, "loss" if self.epoch_loss is None else "epoch_loss_sum": b.loss}


class DecodeWorkload(Workload):
    """Configs 1 and 4: decode-only ('default' = sign quarter offset) [+ fused PCK/AUC/EPE counters]."""

    def __init__(self, args, rank, world, dev, cfg_id):
        super().__init__(args, rank, world, dev)
        import torch
        from litehandnet_b200 import _lib as L
        from litehandnet_b200 import fused, synth
        self.cfg_id = cfg_id
        self.metrics = cfg_id == 4
        if cfg_id == 1:
            self.K, self.B = 21, args.batch or 64
            # 22 MB per batch fits L2: rotate enough distinct batches to exceed 4 x L2 (SURVEY §8d)
            self.R = args.rotate if args.rotate > 2 else max(2, -(-4 * 126_000_000 // (self.B * 21 * 64 * 64 * 4)))
        else:
            self.K, self.B = 16, args.batch or 1024
            self.R = max(2, args.rotate)
        B, K, H, W = self.B, self.K, self.H, self.W
        self.sets = []
        for r in range(self.R):
            seed = 1000 * rank + 10 * r + 20000 * cfg_id
            self.sets.append(self.make_inputs(B, seed, dev))
        overlap = not args.no_overlap
        self.overlap = overlap
        self.bound = []
        self.T = 20
        self.xch = None
        if self.metrics and world > 1 and args.collective == "nvlink":
            from litehandnet_b200.dist import PeerExchange
            self.xch = PeerExchange(dev)
        if self.metrics:
            self.total = torch.zeros((self.T + 5) * K, dtype=torch.int64, device=dev)          # running global counters
            # per-step counter blocks (one per rotating set), all-reduced every step at N > 1
            self.step_cnt = [torch.zeros((self.T + 5) * K, dtype=torch.int64, device=dev) for _ in range(self.R)]
        for r, s in enumerate(self.sets):
            m = None
            if self.metrics:
                m = dict(gt=s[3], mask=s[4], bbox_wh=s[5], counters=self.step_cnt[r] if world > 1 else self.total,
                         pck_thr=0.2, auc_nor=30.0, auc_steps=self.T)
                if self.xch is not None:
                    m = dict(gt=s[3], mask=s[4], bbox_wh=s[5], pck_thr=0.2, auc_nor=30.0, auc_steps=self.T,
                             exchange=self.xch, totals=self.total)
            self.bound.append(fused.BoundDecodeStep(s[0], s[1], s[2], L.MASK_NEG1, L.REFINE_SIGN, L.XFORM_CENTER_SCALE,
                                                    overlap_previous=overlap, metrics=m))
        if self.xch is not None:
            self.collective = ("the per-step PCK/AUC/EPE counter block is all-gathered EVERY eval step INSIDE the kernel (one "
                               "launch behind: the next launch's courier CTA — an extra CTA on one SM without planes — sends it) through peer-mapped mailboxes over "
                               f"NVLink ({self.xch.how}) and added in rank order into the running totals; no NCCL call, one launch "
                               "per step + one flush per epoch (datasets/base_dataset.py:193-261, spawn_dist.py:68-80)")
            self.nvlink_bytes_per_step = self.xch.bytes_per_step((self.T + 5) * K * 8)
        elif self.metrics and world > 1:
            self.aux = torch.cuda.Stream(device=dev)
            self.done = [torch.cuda.Event() for _ in range(self.R)]
            self.freed = [torch.cuda.Event() for _ in range(self.R)]
            self.used = [False] * self.R
            self.collective = ("ncclAllReduce(int64, SUM) of the per-step PCK/AUC/EPE counter block EVERY eval step on a side "
                               "stream, then added into the running totals (datasets/base_dataset.py:193-261, spawn_dist.py:68-80)")
            self.nccl_bytes_per_step = (self.T + 5) * K * 8
            # (plus torch's add_ / zero_ of the 3 KB block on the side stream: not counted, they are not this library's)
        self.bytes_per_launch = (K * H * W * 4 + 16 + K * (12 + 12 + 4) + (K * (8 + 1) + 8 if self.metrics else 0)) * B
        self.kernel_name = f"heatmap_team_kernel<f32,64x64,TW=2,no-flip,no-loss,KS=0>{' + fused counters' if self.metrics else ''}"

    def make_inputs(self, B, seed, dev):
        from litehandnet_b200 import synth
        hm, cen = synth.blob_heatmaps(B, self.K, self.H, self.W, seed=seed, device=dev, zero_frac=0.02, tie_frac=0.01)
        if self.metrics:
            center, scale = synth.bbox_center_scale(B, seed=seed + 3, device=dev)
            gt, mask, wh = synth.pck_inputs(cen, seed=seed + 5, device=dev, stride=1.0, gt_noise=0.0)
            # ground truth in the IMAGE frame the decoder maps to (transform_preds), + N(0, 6 px) annotation noise
            import torch
            g = torch.Generator(device=dev)
            g.manual_seed(seed + 6)
            s200 = scale * 200.0
            gt = gt * (s200 / float(self.W))[:, None, :] + center[:, None, :] - 0.5 * s200[:, None, :]
            gt = (gt + torch.randn(gt.shape, generator=g, device=dev) * 6.0).float().contiguous()
            return hm, center, scale, gt, mask, wh
        center, scale = synth.bbox_center_scale(B, seed=seed + 3, device=dev, fixed=True)
        return hm, center, scale

    def workload(self):
        return workload_label(self.cfg_id, self.args.batch, self.world)

    def step(self, i):
        import torch
        import torch.distributed as dist
        r = i % self.R
        b = self.bound[r]
        if self.metrics and self.world > 1 and self.xch is None:
            comp = torch.cuda.current_stream(self.dev)
            if self.used[r]:
                comp.wait_event(self.freed[r])            # the block was folded into the totals and zeroed
            b.launch()
            self.done[r].record(comp)
            with torch.cuda.stream(self.aux):
                self.aux.wait_event(self.done[r])
                dist.all_reduce(self.step_cnt[r])        # on the side stream: the compute stream never waits for NCCL
                self.total.add_(self.step_cnt[r])
                self.step_cnt[r].zero_()
                self.freed[r].record(self.aux)
            self.used[r] = True
        else:
            b.launch()

    def end_of_epoch(self):
        import torch
        if self.metrics and self.world > 1 and self.xch is None:
            torch.cuda.current_stream(self.dev).wait_stream(self.aux)
        if self.xch is not None:
            self.xch.flush()                    # the in-kernel exchange runs one launch behind: complete the last step

    def begin_epoch(self):
        if self.metrics:
            self.total.zero_()

    def config_extra(self):
        d = {"batch_per_gpu": self.B, "global_batch": self.B * self.world, "joints": self.K, "heatmap": "64x64",
             "decode": "argmax (A2, -1 mask) + sign quarter offset (D3) + transform_preds (T1)",
             "l2_policy": f"{self.R} rotating input sets of {self.B * self.K * 64 * 64 * 4 / 1e6:.0f} MB "
                          f"(> 4 x 126 MB L2 in total), L2 evict_first loads"}
        if self.metrics:
            d["metrics"] = "PCK@0.2 / max(bbox w,h), AUC (20 thresholds, 30 px), EPE — fused int64 counters"
        return d

    def parity(self, steps):
        import numpy as np
        import torch
        from oracle import np_oracle as O
        idx_equal, coord_ok, max_rel, n = True, True, 0.0, 0
        sets = self.sets if self.cfg_id == 1 else self.sets[:2]
        cnt_equal = None
        for r, s in enumerate(sets):
            hm, c, sc = s[0].cpu().numpy(), s[1].cpu().numpy(), s[2].cpu().numpy()
            with np.errstate(all="ignore"):
                hp, preds, mv = O.keypoints_from_heatmaps(hm, c, sc, "default", 11)
            ridx = hm.reshape(hm.shape[0], hm.shape[1], -1).argmax(-1).astype(np.int32)
            b = self.bound[r]
            got = b.preds.cpu().numpy()
            idx_equal &= bool(np.array_equal(b.idx.cpu().numpy(), ridx))
            ok, rel = coord_check(got[..., :2], preds, xform_mag(c, sc))
            coord_ok &= ok and bool(np.array_equal(got[..., 2:], mv, equal_nan=True))
            max_rel = max(max_rel, rel)
            n += hm.shape[0]
            if self.metrics and r == 0:
                # the counters this shard contributes per step == the oracle's hit counts on the oracle's decoded points
                from litehandnet_b200 import metrics as M
                acc = M.MetricAccumulator(self.K, device=self.dev)
                acc.update_from_heatmaps(s[0], s[1], s[2], s[3], s[4], s[5], post_process="default")
                cnt = acc.counters.cpu().numpy().reshape(self.T + 5, self.K)
                p64 = preds.astype(np.float64)
                gt, mask, wh = s[3].cpu().numpy(), s[4].cpu().numpy(), s[5].cpu().numpy()
                t = wh.max(1).astype(np.float64)
                h1, v1 = O.pck_counters(p64, gt, mask, [0.2], np.stack([t, t], 1))
                nor = np.full((p64.shape[0], 2), 30.0)
                h2, v2 = O.pck_counters(p64, gt, mask, [1.0 * i / self.T for i in range(self.T)], nor)
                cnt_equal = bool(np.array_equal(cnt[0], h1[0]) and np.array_equal(cnt[1], v1) and
                                 np.array_equal(cnt[2:2 + self.T], h2) and np.array_equal(cnt[2 + self.T], v2))
        out = {"idx_equal": idx_equal, "coord_within_1e-5": coord_ok, "coord_max_rel": max_rel, "loss_rel": None, "samples": n,
               "against": "oracle.np_oracle.keypoints_from_heatmaps('default') (+ pck_counters) on rank 0's inputs; outputs as "
                          "the timed loop left them"}
        ok = idx_equal and coord_ok
        if self.metrics:
            out["pck_hit_counts_equal"] = cnt_equal
            ok = ok and bool(cnt_equal)
            mono = self.monolithic_counters(steps)
            out["counters_equal_monolithic"] = bool(torch.equal(mono, self.total))
            if self.xch is not None:
                out["exchange_timeouts"] = int(self.xch.status.item())
            ok = ok and out["counters_equal_monolithic"]
            from litehandnet_b200 import ops
            v = ops.metrics_finalize(self.total, self.K, self.T)[:3].cpu().numpy()
            out["metrics"] = {"PCK": float(v[0]), "AUC": float(v[1]), "EPE": float(v[2])}
        out["ok"] = bool(ok)
        return out

    def monolithic_counters(self, steps):
        """The running totals a SINGLE process would hold after the timed steps: every rank's shard of every step,
        accumulated on this GPU into one block (rank 0 regenerates the other ranks' seeded inputs)."""
        import torch
        from litehandnet_b200 import metrics as M
        per_set = []
        for r in range(self.R):
            acc = M.MetricAccumulator(self.K, device=self.dev)
            for rk in range(self.world):
                s = self.sets[r] if rk == self.rank else self.make_inputs(self.B, 1000 * rk + 10 * r + 20000 * self.cfg_id, self.dev)
                acc.update_from_heatmaps(s[0], s[1], s[2], s[3], s[4], s[5], post_process="default")
            per_set.append(acc.counters)
        mono = torch.zeros_like(self.total)
        for i in range(steps):
            mono += per_set[i % self.R]
        return mono

    def e2e(self, steps, warmup):
        import torch
        from litehandnet_b200 import fused
        s0 = self.sets[0]
        host = [torch.empty(t.shape, dtype=(torch.uint8 if t.dtype == torch.bool else t.dtype), pin_memory=True).copy_(
            t.view(torch.uint8) if t.dtype == torch.bool else t) for t in s0]
        cfg = fused.FusedHeatmapStep(self.image_size, post_process="default", kernel=11, loss_type=None)
        pipe = fused.HostPipeline(cfg, self.B, self.K, self.H, self.W, flip=False, chunks=min(self.args.chunks, max(1, self.B // 32)),
                                  device=self.dev, metrics=dict(pck_thr=0.2, auc_nor=30.0, auc_steps=self.T) if self.metrics else None)

        def call():
            if self.metrics:
                pipe(host[0], None, None, None, host[1], host[2], gt=host[3], mask=host[4], bbox_wh=host[5])
            else:
                pipe(host[0], None, None, None, host[1], host[2])

        for _ in range(max(1, min(warmup, 3))):
            call()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        launches = 0
        for _ in range(steps):
            call()
            launches += pipe.launches
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return dict(seconds=dt, samples_per_step=self.B, h2d=pipe.h2d_bytes, d2h=pipe.d2h_bytes, launches=launches,
                    api="litehandnet_b200.fused.HostPipeline (decode-only" + (" + fused counters + lhn_metrics_finalize" if self.metrics else "") +
                        "; pinned host buffers, chunked H2D overlapped with the kernel)", note=None)

    def cpu_inputs(self, n):
        s = self.sets[0]
        return [t[:n].cpu().numpy() for t in s]

    def loss_check(self, steps):
        return None

    def outputs(self, steps):
        b = self.bound[(steps - 1) % self.R]
        out = {"preds": b.preds, "hm_preds": b.hm_preds, "idx": b.idx}
        if self.metrics:
            out["counters"] = self.total            # running PCK/AUC/EPE counters over the timed steps
        return out


class SimdrWorkload(Workload):
    """Config 3: keypoints_from_simdr on 2 x [4096, 21, 512] f32."""
    cfg_id = 3

    def __init__(self, args, rank, world, dev):
        super().__init__(args, rank, world, dev)
        from litehandnet_b200 import fused, synth
        self.B, self.K, self.L, self.k = args.batch or 4096, 21, 512, 2
        self.R = max(2, args.rotate)
        self.sets = []
        for r in range(self.R):
            seed = 1000 * rank + 10 * r + 60000
            xv, yv = synth.simdr_vectors(self.B, self.K, self.L, seed=seed, device=dev, k=self.k)
            center, scale = synth.bbox_center_scale(self.B, seed=seed + 3, device=dev, fixed=True)
            self.sets.append((xv, yv, center, scale))
        self.overlap = not args.no_overlap
        self.bound = [fused.BoundSimdrStep(s[0], s[1], self.k, s[2], s[3], overlap_previous=self.overlap) for s in self.sets]
        self.bytes_per_launch = (2 * self.K * self.L * 4 + 16 + self.K * 12) * self.B
        self.kernel_name = "decode_simdr_ring_kernel<f32> (16 warps x 3-stage TMA ring per SM)"

    def workload(self):
        return workload_label(self.cfg_id, self.args.batch, self.world)

    def config_extra(self):
        return {"batch_per_gpu": self.B, "global_batch": self.B * self.world, "joints": self.K, "bins": self.L, "split_ratio": self.k,
                "decode": "argmax / k, score mean, transform_preds",
                "l2_policy": f"{self.R} rotating input sets of {2 * self.B * self.K * self.L * 4 / 1e6:.0f} MB > 126 MB L2, L2 evict_first loads"}

    def parity(self, steps):
        import numpy as np
        from oracle import np_oracle as O
        idx_equal, coord_ok, max_rel, n = True, True, 0.0, 0
        for r, s in enumerate(self.sets):
            xv, yv, c, sc = [t.cpu().numpy() for t in s]
            ref = O.keypoints_from_simdr(xv, yv, c, sc, self.k)
            b = self.bound[r]
            got = b.out.cpu().numpy()
            gi = b.idx.cpu().numpy()
            idx_equal &= bool(np.array_equal(gi[..., 0], xv.argmax(2)) and np.array_equal(gi[..., 1], yv.argmax(2)))
            ok, rel = coord_check(got[..., :2], ref[..., :2], xform_mag(c, sc))
            coord_ok &= ok and bool(np.array_equal(got[..., 2], ref[..., 2]))
            max_rel = max(max_rel, rel)
            n += xv.shape[0]
        return {"ok": bool(idx_equal and coord_ok), "idx_equal": idx_equal, "coord_within_1e-5": coord_ok, "coord_max_rel": max_rel,
                "loss_rel": None, "samples": n,
                "against": "oracle.np_oracle.keypoints_from_simdr on rank 0's inputs; outputs as the timed loop left them"}

    def e2e(self, steps, warmup):
        import torch
        from litehandnet_b200 import fused
        host = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in self.sets[0]]
        pipe = fused.SimdrHostPipeline(self.B, self.K, self.L, self.L, self.k, chunks=self.args.chunks, device=self.dev)
        for _ in range(max(1, min(warmup, 3))):
            pipe(*host)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        launches = 0
        for _ in range(steps):
            pipe(*host)
            launches += pipe.launches
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return dict(seconds=dt, samples_per_step=self.B, h2d=pipe.h2d_bytes, d2h=pipe.d2h_bytes, launches=launches,
                    api="litehandnet_b200.fused.SimdrHostPipeline (pinned host buffers, chunked H2D overlapped with the decode kernel)",
                    note=None)

    def cpu_inputs(self, n):
        return [t[:n].cpu().numpy() for t in self.sets[0]]

    def loss_check(self, steps):
        return None

    def outputs(self, steps):
        b = self.bound[(steps - 1) % self.R]
        return {"preds": b.out, "idx": b.idx}


def make_workload(args, rank, world, dev):
    c = args.config
    if c in (2, 5):
        return FusedWorkload(args, rank, world, dev, c)
    if c in (1, 4):
        return DecodeWorkload(args, rank, world, dev, c)
    return SimdrWorkload(args, rank, world, dev)


# =========================================================================================================
# CPU arm
# =========================================================================================================
class CpuArm:
    """The reference's CPU path for one config: the executed reference (oracle/_ref or /root/reference,
    kind 'reference') when it can be loaded, else the numpy port (kind 'port')."""

    def __init__(self, cfg_id, inputs, image_size, sigma):
        self.cfg_id = cfg_id
        self.kind = "port"
        self.runner = None
        err = None
        if not os.environ.get("LHN_CPU_PORT"):
            try:
                from oracle import ref_path
                if ref_path.available():
                    self.runner = ref_path.RefRunner(cfg_id, inputs, image_size=image_size, sigma=sigma, kernel=11)
                    self.kind = "reference"
            except Exception as e:                      # a broken staging must not take the bench down
                err = f"{type(e).__name__}: {e}"
                self.runner = None
        self.load_error = err
        if self.runner is None:
            self.runner = PortRunner(cfg_id, inputs, image_size, sigma)
        self.workers = self.runner.workers
        self.B = self.runner.B

    def run(self, n):
        """-> seconds for one pass over the first n samples"""
        return self.runner.run(n)[-1]

    def close(self):
        self.runner.close()

    def describe(self, sample):
        what = {1: "keypoints_from_heatmaps(post_process='default')",
                2: "TopDownGenerateTarget per sample -> DistanceLoss(L2, balance=True) -> flip_back + average -> "
                   "keypoints_from_heatmaps('unbiased', kernel=11)",
                3: "keypoints_from_simdr(k=2)",
                4: "keypoints_from_heatmaps('default') on 16 joints -> keypoint_pck_accuracy(0.2) / keypoint_auc(30) / keypoint_epe",
                5: "TopDownGenerateTarget per sample -> DistanceLoss(L2, balance=True) -> keypoints_from_heatmaps('unbiased', "
                   "kernel=11) at 128x128"}[self.cfg_id]
        how = ("the reference's own functions (oracle/_ref staged copy), per-sample Python loops sharded over "
               f"{self.workers} forked workers, torch parts on all cores" if self.kind == "reference" else
               f"numpy port of the reference pipeline (oracle/) in {self.workers} forked workers")
        return f"{sample} samples per pass; {what}; {how}"


class PortRunner:
    """numpy-port fallback with the RefRunner interface."""

    def __init__(self, cfg_id, inputs, image_size, sigma):
        from oracle import cpu_path
        self.cfg_id = cfg_id
        if cfg_id in (2, 5):
            self.r = cpu_path.FusedCpuRunner(*inputs, image_size=image_size, sigma=sigma, kernel=11)
            self.workers, self.B = self.r.workers, self.r.B
        else:
            self.r = None
            self.inputs = inputs
            self.workers, self.B = 1, inputs[0].shape[0]

    def run(self, n):
        import numpy as np
        from oracle import np_oracle as O
        if self.r is not None:
            return self.r.run(n)
        t0 = time.perf_counter()
        i = self.inputs
        with np.errstate(all="ignore"):
            if self.cfg_id == 3:
                out = O.keypoints_from_simdr(i[0][:n], i[1][:n], i[2][:n], i[3][:n], 2)
            else:
                _, preds, _ = O.keypoints_from_heatmaps(i[0][:n], i[1][:n], i[2][:n], "default", 11)
                out = preds
                if self.cfg_id == 4:
                    p64 = preds.astype(np.float64)
                    t = i[5][:n].max(1).astype(np.float64)
                    O.keypoint_pck_accuracy(p64, i[3][:n], i[4][:n], 0.2, np.stack([t, t], 1))
                    O.keypoint_auc(p64, i[3][:n], i[4][:n], 30)
                    O.keypoint_epe(p64, i[3][:n], i[4][:n])
        return out, time.perf_counter() - t0

    def close(self):
        if self.r is not None:
            self.r.close()


def cpu_sample_size(arm, requested, budget_s):
    """Bounded sample: a short probe gives the CPU rate; the sample is sized to ~budget_s per pass."""
    if requested:
        return min(int(requested), arm.B)
    probe = min(arm.B, max(16, 2 * arm.workers))
    arm.run(probe)                                        # warm the workers
    dt = arm.run(probe)
    rate = probe / max(dt, 1e-6)
    return int(max(min(16, arm.B), min(arm.B, rate * budget_s)))


CPU_SHAPES = {1: dict(K=21, H=64, B=64), 2: dict(K=21, H=64, B=1024), 3: dict(B=4096), 4: dict(K=16, H=64, B=1024),
              5: dict(K=21, H=128, B=1024)}


def cpu_only_inputs(cfg_id, batch):
    """Host inputs of one config generated on the CPU (the --impl reference arm never touches a GPU)."""
    from litehandnet_b200 import synth
    sh = CPU_SHAPES[cfg_id]
    B = min(batch or sh["B"], sh["B"])
    if cfg_id in (2, 5):
        img = (256, 256) if cfg_id == 2 else (512, 512)
        sig = 2.0 if cfg_id == 2 else 4.0
        hm, cen = synth.blob_heatmaps(B, sh["K"], sh["H"], sh["H"], seed=0, sigma=sig)
        hf = synth.flipped_blob_heatmaps(cen, sh["H"], sh["H"], seed=1, sigma=sig) if cfg_id == 2 else None
        joints, vis = synth.hand_joints(B, sh["K"], img, seed=2)
        center, scale = synth.bbox_center_scale(B, seed=3)
        return [None if t is None else t.numpy() for t in (hm, hf, joints, vis, center, scale)], img, int(sig)
    if cfg_id == 3:
        xv, yv = synth.simdr_vectors(B, 21, 512, seed=0)
        center, scale = synth.bbox_center_scale(B, seed=3, fixed=True)
        return [t.numpy() for t in (xv, yv, center, scale)], (256, 256), 2
    hm, cen = synth.blob_heatmaps(B, sh["K"], 64, 64, seed=0, zero_frac=0.02, tie_frac=0.01)
    if cfg_id == 4:
        import torch
        center, scale = synth.bbox_center_scale(B, seed=3)
        gt, mask, wh = synth.pck_inputs(cen, seed=5, stride=1.0, gt_noise=0.0)
        s200 = scale * 200.0
        gt = gt * (s200 / 64.0)[:, None, :] + center[:, None, :] - 0.5 * s200[:, None, :]
        gt = (gt + torch.randn(gt.shape, generator=torch.Generator().manual_seed(6)) * 6.0).float().contiguous()
        return [t.numpy() for t in (hm, center, scale, gt, mask, wh)], (256, 256), 2
    center, scale = synth.bbox_center_scale(B, seed=3, fixed=True)
    return [t.numpy() for t in (hm, center, scale)], (256, 256), 2


def workload_label(cfg_id, batch, world):
    names = {1: "litehandnet FreiHAND top-down 256x256 input, 21 joints, 64x64 heatmaps: argmax + quarter-offset decode, batch {b} (BASELINE configs[0])",
             2: "FreiHAND 21x64x64 fused Gaussian target render + target-weight MSE loss + DARK decode with flip-test, batch {b} per GPU (BASELINE configs[1])",
             3: "SimDR 1D-logit decode (x/y split-ratio 2, 21 joints, 512 bins) from centernet_simdr_loss, batch {b} per GPU (BASELINE configs[2])",
             4: "MPII-style 16-joint 64x64 decode + PCK@0.2/EPE/AUC counters, batch {b} per GPU, batch-sharded over {w} GPU(s) (BASELINE configs[3])",
             5: "high-res 21x128x128 fused Gaussian target render + target-weight MSE loss + DARK decode, global batch {g} sharded over {w} GPU(s) = {b} per GPU (BASELINE configs[4])"}
    default = {1: 64, 2: 1024, 3: 4096, 4: 1024, 5: 8192}[cfg_id]
    b = batch or default
    if cfg_id == 5:
        return names[5].format(g=b, w=world, b=b // world)
    return names[cfg_id].format(b=b, w=world)


def run_reference_arm(args, rank, world):
    """The reference's CPU path on the host cores, same metric and config; rank 0 only."""
    if rank != 0:
        return
    inputs, img, sig = cpu_only_inputs(args.config, args.batch)
    arm = CpuArm(args.config, inputs, img, sig)
    # keep the whole run within ~2.5 minutes: (steps + warmup) passes of `sample` samples each
    budget = max(0.05, min(2.0, 150.0 / max(1, args.steps + args.warmup)))
    sample = cpu_sample_size(arm, args.cpu_sample, budget)
    for _ in range(args.warmup):
        arm.run(sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        arm.run(sample)
    dt = time.perf_counter() - t0
    arm.close()
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRICS[args.config], "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong" if args.config == 5 else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_label(args.config, args.batch, world), "sample_per_step": sample,
                   "note": "each step is a bounded sample of the workload on the host CPU"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.workers, "kind": arm.kind, "sample": arm.describe(sample)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if arm.load_error:
        line["cpu_baseline"]["reference_load_error"] = arm.load_error
    print(json.dumps(line), flush=True)


# =========================================================================================================
# GPU arm
# =========================================================================================================
def run_gpu_arm(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    wl = make_workload(args, rank, world, dev)

    def fence():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # ---- warm-up, then the timed region ------------------------------------------------------------
    for i in range(args.warmup):
        wl.step(i)
    wl.end_of_epoch()
    # NVML is initialised and the sampler thread started BEFORE the barrier: nvmlInit from N processes at once takes
    # milliseconds and would otherwise skew the ranks' entry into the timed region.
    sampler = ClockSampler(physical_gpu_index(local_rank), args.clock_interval_ms * 1e-3 if args.clock_interval_ms > 0
                           else (0.0005 if world == 1 else 0.002))
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    wl.begin_epoch()
    fence()
    sampler.begin()
    e0.record()
    for i in range(args.steps):
        wl.step(i)
    wl.end_of_epoch()
    e1.record()
    fence()
    clocks = sampler.stop()
    ms_total = e0.elapsed_time(e1)
    loss_val = wl.loss_check(args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(wl.outputs(args.steps), wl.B, args.dump_outputs)

    # ---- parity of the measured outputs (rank 0; before anything else touches the output buffers) -----------
    parity = None
    if rank == 0 and not args.no_parity:
        parity = wl.parity(args.steps)
    fence()

    # ---- the dominant kernel alone: K back-to-back launches (no collective) between two events on the launching
    #      stream; a second pass WITHOUT the launch overlap gives the isolated-launch figure ------------------------
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for i in range(min(3, args.steps)):
        wl.kernel_step(i)
    k0.record()
    for i in range(args.steps):
        wl.kernel_step(i)
    k1.record()
    fence()
    kernel_ms = k0.elapsed_time(k1) / args.steps
    iso = []
    for i in range(min(args.steps, 20)):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        wl.kernel_step(i)
        b.record()
        torch.cuda.synchronize()
        iso.append(a.elapsed_time(b))
    iso.sort()
    kernel_ms_isolated = iso[len(iso) // 2]

    # ---- end to end through the host-buffer API ---------------------------------------------------------
    e2e = None
    if not args.no_e2e:
        fence()
        e2e = wl.e2e(args.steps, args.warmup)

    # ---- max over ranks ------------------------------------------------------------------------------------
    stats = torch.tensor([ms_total, kernel_ms, e2e["seconds"] if e2e else 0.0, kernel_ms_isolated], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
    ms_total, kernel_ms, e2e_s, kernel_ms_isolated = [float(v) for v in stats.tolist()]

    rc = 0
    if rank == 0:
        value = world * wl.B * args.steps / (ms_total * 1e-3)
        peak, peak_src = measured_peak()
        achieved = wl.bytes_per_launch / (kernel_ms * 1e-3) / 1e9
        cfg = {"workload": wl.workload(), "baseline_config": args.config}
        cfg.update(wl.config_extra())
        cfg["parallelism"] = f"batch-shard x{world}; {wl.collective}" if world > 1 else "single GPU"
        if world > 1:
            cfg["nccl_bytes_per_step"] = wl.nccl_bytes_per_step
            cfg["nvlink_bytes_per_step_per_rank"] = wl.nvlink_bytes_per_step
        cfg["launch"] = "eager C-ABI launches, one kernel per step" + (
            "; LHN_FLAG_OVERLAP_PREVIOUS (programmatic dependent launch over rotating buffer sets)" if wl.overlap else "")
        if loss_val is not None:
            cfg["loss_check"] = loss_val
        line = {
            "metric": METRICS[args.config], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": wl.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": recorded_traffic(args.config, wl.B),
                         "traffic_source": "recorded: ncu --set full capture committed under profiles/ (not measured in this run)",
                         "kernel": wl.kernel_name, "kernel_ms": kernel_ms,
                         "kernel_ms_note": "average over back-to-back launches" + (" overlapped by programmatic dependent launch "
                                           "(throughput of the stream, not the latency of one launch)" if wl.overlap else ""),
                         "kernel_ms_isolated": kernel_ms_isolated,
                         "frac_isolated": wl.bytes_per_launch / (kernel_ms_isolated * 1e-3) / 1e9 / peak,
                         "algorithmic_bytes_per_launch": wl.bytes_per_launch, "peak_source": peak_src,
                         "peak_note": "the peak is a COPY (read+write); a read-only TMA stream reaches 7.0-7.18 TB/s on this "
                                      "part (profiles/r01_bw_probe.txt), so frac slightly above 1 is a read-only kernel at the HBM limit"},
            "gpu_launches": args.steps * wl.launches_per_step,
        }
        if parity is not None:
            line["parity"] = parity
            if not parity["ok"]:
                rc = 3
        if e2e:
            ev = world * e2e["samples_per_step"] * args.steps / e2e_s
            h2d_gbs = e2e["h2d"] * args.steps / e2e_s / 1e9
            line["e2e"] = {"value": ev, "unit": UNIT, "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                           "api": e2e["api"], "gpu_launches": e2e["launches"],
                           "h2d_gbs_per_gpu": h2d_gbs, "pcie_peak_gbs": PCIE_GEN5_X16_GBS, "frac_of_pcie": h2d_gbs / PCIE_GEN5_X16_GBS,
                           "bound": "host->device copy (PCIe 5.0 x16: 63 GB/s theoretical, ~55 GB/s achievable with pinned memory)"}
            if e2e.get("note"):
                line["e2e"]["note"] = e2e["note"]
        if world == 1 and not args.no_cpu_baseline:
            n_cpu = min(wl.B, 1024)
            arm = CpuArm(args.config, wl.cpu_inputs(n_cpu), wl.image_size, getattr(wl, "sigma", 2))
            sample = cpu_sample_size(arm, args.cpu_sample, 6.0)
            dts = [arm.run(sample) for _ in range(2)]
            arm.close()
            line["cpu_baseline"] = {"value": sample / min(dts), "unit": UNIT, "cores": arm.workers, "kind": arm.kind,
                                    "sample": "best of 2 passes; " + arm.describe(sample)}
            if arm.load_error:
                line["cpu_baseline"]["reference_load_error"] = arm.load_error
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[1, 2, 3, 4, 5], help="BASELINE.json config (1-based); 2 = headline")
    ap.add_argument("--batch", type=int, default=0, help="samples per GPU per step (config 5: GLOBAL batch); 0 = the config's own")
    ap.add_argument("--rotate", type=int, default=2, help="distinct device-resident input sets (config 1: 0 = enough to exceed 4 x L2)")
    ap.add_argument("--chunks", type=int, default=8, help="H2D/compute pipeline chunks of the e2e path")
    ap.add_argument("--cpu-sample", type=int, default=0)
    ap.add_argument("--parity-samples", type=int, default=0, help="config 5: samples of rank 0's shard checked against the oracle (default 512)")
    ap.add_argument("--global-loss", action="store_true",
                    help="N > 1, configs 2/5: balanced loss with batch-global N_pos (an all-reduce of the f64 sums every step) "
                         "instead of the reference's per-rank loss")
    ap.add_argument("--collective", default="nvlink", choices=["nvlink", "nccl"],
                    help="N > 1: how a PER-STEP exchange (config 4 counters, --global-loss sums) is done: inside the kernel over "
                         "peer-mapped NVLink mailboxes (default) or as an NCCL all-reduce beside the kernel")
    ap.add_argument("--spare-sms", type=int, default=4,
                    help="N > 1 with --global-loss: SMs the persistent kernel leaves free for the NCCL all-reduce")
    ap.add_argument("--clock-interval-ms", type=float, default=0.0, help="NVML sampling period (0 = automatic)")
    ap.add_argument("--no-overlap", action="store_true", help="do not let a launch overlap the previous one's tail")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write rank 0's outputs of the last step as DIR/<name>.npy (f32/f64, "
                         "at most 64 MB in all); configs 2/5 at N > 1 without --global-loss write the epoch's loss sum "
                         "over all ranks as epoch_loss_sum instead of the step's loss")
    # accepted for old command lines (all are the default behaviour now)
    ap.add_argument("--no-graph", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-graph-all", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.config == 1 and args.rotate == 2:
        args.rotate = 0
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return
    if world != args.gpus and world == 1 and args.gpus > 1:
        # launched without torchrun: re-exec under torch.distributed.run
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29531", os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_gpu_arm(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
