"""GPU: the code path bench.py measures, under oracle parity at the full headline size.

bench.py's `value`, every N > 1 line and `e2e` come from fused.BoundFusedStep (rotating buffer sets,
LHN_FLAG_OVERLAP_PREVIOUS = programmatic dependent launch, LHN_FLAG_ACCUMULATE_LOSS, spare SMs,
finalize=False + launch_finalize) and fused.HostPipeline (chunked H2D pipeline).  These tests drive them
exactly as bench.py does and compare every step with the reference's CPU pipeline
(oracle.cpu_path.FusedCpuRunner = TopDownGenerateTarget -> DistanceLoss(balance) -> flip average ->
keypoints_from_heatmaps('unbiased'); top_down_eval.py:375-463, loss/heatmapLoss.py:242-265) on ALL 1024
samples: argmax indices bit-exact, coordinates 1e-5 element-wise, loss 1e-5 relative.
"""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import assert_coords_close, xform_magnitude
from oracle import cpu_path
from oracle import np_oracle as O
from litehandnet_b200 import _lib as L
from litehandnet_b200 import fused, synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
K, H, W = 21, 64, 64
IMAGE = (256, 256)


def make_set(B, seed, device=DEV, zero_frac=0.0, tie_frac=0.0):
    hm, cen = synth.blob_heatmaps(B, K, H, W, seed=seed, device=device, zero_frac=zero_frac, tie_frac=tie_frac)
    hf = synth.flipped_blob_heatmaps(cen, H, W, seed=seed + 1, device=device)
    joints, vis = synth.hand_joints(B, K, IMAGE, seed=seed + 2, device=device)
    center, scale = synth.bbox_center_scale(B, seed=seed + 3, device=device)
    return hm, hf, joints, vis, center, scale


_ORACLE_CACHE = {}


def oracle_of(s, key):
    """(preds [B,K,3], idx [B,K], loss, sums[4]) of the reference CPU pipeline on one input set (cached per key)."""
    if key not in _ORACLE_CACHE:
        r = cpu_path.FusedCpuRunner(*[t.cpu().numpy() for t in s], image_size=IMAGE, sigma=2, kernel=11)
        try:
            with np.errstate(all="ignore"):
                preds, loss, _ = r.run()
            mag = xform_magnitude(s[4].cpu().numpy(), s[5].cpu().numpy())
            _ORACLE_CACHE[key] = (preds, r.last_idx.copy(), float(loss), r.last_sums.copy(), mag)
        finally:
            r.close()
    return _ORACLE_CACHE[key]


def check_step(bound, ref, what, loss=True):
    preds, idx, rloss, _, mag = ref
    B = preds.shape[0]
    assert np.array_equal(bound.idx[:B].cpu().numpy(), idx), f"{what}: argmax indices differ"
    got = bound.preds[:B].cpu().numpy()
    assert_coords_close(got[..., :2], preds[..., :2], what=f"{what}: coordinates", mag=mag)
    assert np.array_equal(got[..., 2], preds[..., 2], equal_nan=True), f"{what}: maxvals differ"
    if loss:
        np.testing.assert_allclose(float(bound.loss.item()), rloss, rtol=1e-5, err_msg=f"{what}: loss")


@pytest.fixture(scope="module")
def sets():
    return [make_set(1024, 1000 + 10 * r) for r in range(2)]


def step_cfg():
    return fused.FusedHeatmapStep(IMAGE, sigma=2, unbiased_encoding=True, balance=True, post_process="unbiased", kernel=11)


def poison(b):
    b.preds.fill_(float("nan")); b.idx.fill_(-7); b.loss.fill_(float("nan")); b.sums.fill_(float("nan"))


@pytest.mark.parametrize("overlap", [False, True])
def test_bound_step_rotating_sets_full_batch(sets, overlap):
    """bench.py's timed loop at N = 1: two rotating sets, >= 8 back-to-back eager launches, one launch per step."""
    bound = [fused.BoundFusedStep(step_cfg(), s[0], s[2], s[3], s[4], s[5], hm_flip=s[1], overlap_previous=overlap)
             for s in sets]
    refs = [oracle_of(s, ("set", r)) for r, s in enumerate(sets)]
    for b in bound:
        poison(b)
    for i in range(9):                       # ends on set 0; set 1 was last written by step 7
        bound[i % 2].launch()
    torch.cuda.synchronize()
    for r in range(2):
        check_step(bound[r], refs[r], f"overlap={overlap} set {r}")
    # every step separately (a sync in between): each result is complete and correct on its own
    for i in range(4):
        poison(bound[i % 2])
        bound[i % 2].launch()
        torch.cuda.synchronize()
        check_step(bound[i % 2], refs[i % 2], f"overlap={overlap} step {i}")


def test_bound_step_accumulate_into_epoch_sum(sets):
    """N > 1 default of bench.py: LHN_FLAG_ACCUMULATE_LOSS adds every step's loss into one device scalar
    (train_one_epoch's loss_dict['sum'] += v, train/topdown_trainer.py:82-84) while launches overlap."""
    epoch = torch.zeros(1, dtype=torch.float32, device=DEV)
    bound = [fused.BoundFusedStep(step_cfg(), s[0], s[2], s[3], s[4], s[5], hm_flip=s[1], overlap_previous=True,
                                  accumulate_into=epoch) for s in sets]
    refs = [oracle_of(s, ("set", r)) for r, s in enumerate(sets)]
    n = 10
    for i in range(n):
        bound[i % 2].launch()
    torch.cuda.synchronize()
    want = 0.0
    for i in range(n):
        want = float(np.float32(want) + np.float32(refs[i % 2][2]))       # f32 running sum, like the kernel's
    np.testing.assert_allclose(float(epoch.item()), want, rtol=2e-5)
    for r in range(2):
        check_step(bound[r], refs[r], f"accumulate set {r}", loss=False)


@pytest.mark.parametrize("spare", [0, 4])
def test_bound_step_global_loss_mode(sets, spare):
    """bench.py --global-loss: the kernel leaves the f64 sums (finalize=False, spare SMs for NCCL); the sums of the
    ranks' shards are added (here: the two sets stand in for two ranks) and lhn_loss_finalize runs afterwards —
    equal to DistanceLoss(balance=True) on the concatenated batch (global N_pos)."""
    bound = [fused.BoundFusedStep(step_cfg(), s[0], s[2], s[3], s[4], s[5], hm_flip=s[1], finalize=False,
                                  overlap_previous=True, spare_sms=spare) for s in sets]
    refs = [oracle_of(s, ("set", r)) for r, s in enumerate(sets)]
    for b in bound:
        poison(b)
    for i in range(8):
        bound[i % 2].launch()
    torch.cuda.synchronize()
    for r in range(2):
        check_step(bound[r], refs[r], f"global-loss set {r}", loss=False)
        # (S_pos, S_neg) are f32 per-plane sums added in f64: 1e-6; (N_pos, numel) are counts: exact
        np.testing.assert_allclose(bound[r].sums.cpu().numpy()[:2], refs[r][3][:2], rtol=1e-6)
        assert np.array_equal(bound[r].sums.cpu().numpy()[2:], refs[r][3][2:])
    total = bound[0].sums + bound[1].sums                                  # what the all-reduce leaves on every rank
    bound[0].sums.copy_(total)
    bound[0].launch_finalize(bound[0].stream())
    torch.cuda.synchronize()
    want = O.distance_loss_from_sums(refs[0][3] + refs[1][3], True)
    np.testing.assert_allclose(float(bound[0].loss.item()), float(want), rtol=1e-5)


def test_bound_step_three_launch_form_matches(sets):
    """launch_kernel_partials + launch_reduce + launch_finalize (the per-plane-partials form) == the one-launch step."""
    s = sets[0]
    b = fused.BoundFusedStep(step_cfg(), s[0], s[2], s[3], s[4], s[5], hm_flip=s[1])
    b.launch()
    torch.cuda.synchronize()
    one = (b.preds.clone(), b.idx.clone(), float(b.loss.item()))
    poison(b)
    st = b.stream()
    b.launch_kernel_partials(st); b.launch_reduce(st); b.launch_finalize(st)
    torch.cuda.synchronize()
    assert torch.equal(b.preds, one[0]) and torch.equal(b.idx, one[1])
    np.testing.assert_allclose(float(b.loss.item()), one[2], rtol=1e-6)


def test_overlap_orders_a_launch_after_the_one_two_back():
    """The write-after-write case the overlap flag must exclude (two rotating OUTPUT sets X, Y):
        A (long, leaves spare SMs) -> X,  B (tiny) -> Y,  C (tiny) -> X[:1],  D (tiny) -> Y[:1]
    B, C and D fit into the SMs A leaves free, so with a trigger-at-entry scheme C would run beside A and A's
    later stores would overwrite C's results in X.  With the ordering rule (a launch lets its successor in only
    after its own predecessor completed) X[:1] must hold C's results and Y[:1] D's."""
    big = make_set(768, 300)
    tiny = [make_set(1, 310 + 10 * i, zero_frac=0.0) for i in range(3)]
    cfg = step_cfg()
    X = dict(preds=torch.empty((768, K, 3), device=DEV), idx=torch.empty((768, K), dtype=torch.int32, device=DEV),
             loss=torch.empty(1, device=DEV))
    Y = dict(preds=torch.empty((768, K, 3), device=DEV), idx=torch.empty((768, K), dtype=torch.int32, device=DEV),
             loss=torch.empty(1, device=DEV))

    def bind(s, out, spare):
        return fused.BoundFusedStep(cfg, s[0], s[2], s[3], s[4], s[5], hm_flip=s[1], overlap_previous=True,
                                    spare_sms=spare, outputs=out)

    a = bind(big, X, 48)
    b, c, d = bind(tiny[0], Y, 0), bind(tiny[1], X, 0), bind(tiny[2], Y, 0)
    ref_c, ref_d = oracle_of(tiny[1], ("tiny", 1)), oracle_of(tiny[2], ("tiny", 2))
    for trial in range(20):
        X["preds"].fill_(float("nan")); Y["preds"].fill_(float("nan"))
        a.launch(); b.launch(); c.launch(); d.launch()
        torch.cuda.synchronize()
        check_step(c, ref_c, f"trial {trial}: X after A,B,C,D")
        check_step(d, ref_d, f"trial {trial}: Y after A,B,C,D")


def test_small_batch_overlap_accumulate():
    """n_planes < SM count (grids can be co-resident): 3 rotating sets, many overlapped launches with the loss
    accumulated into one scalar — no update may be lost and every set must hold its own results."""
    sets3 = [make_set(3, 400 + 10 * i, zero_frac=0.05, tie_frac=0.05) for i in range(3)]
    refs = [oracle_of(s, ("small", i)) for i, s in enumerate(sets3)]
    epoch = torch.zeros(1, dtype=torch.float32, device=DEV)
    bound = [fused.BoundFusedStep(step_cfg(), s[0], s[2], s[3], s[4], s[5], hm_flip=s[1], overlap_previous=True,
                                  accumulate_into=epoch) for s in sets3]
    n = 60
    for i in range(n):
        bound[i % 3].launch()
    torch.cuda.synchronize()
    want = 0.0
    for i in range(n):
        want = float(np.float32(want) + np.float32(refs[i % 3][2]))
    np.testing.assert_allclose(float(epoch.item()), want, rtol=5e-5)
    for r in range(3):
        check_step(bound[r], refs[r], f"small set {r}", loss=False)


# ---- HostPipeline (bench.py's e2e number) --------------------------------------------------------------
@pytest.mark.parametrize("B,chunks", [(1024, 8), (1024, 3), (1024, 1), (1000, 7), (37, 8), (5, 8)])
def test_host_pipeline_vs_oracle(B, chunks):
    s = make_set(B, 500 + B + chunks, device="cpu", zero_frac=0.01, tie_frac=0.01)
    ref = oracle_of(s, ("host", B, chunks))
    pipe = fused.HostPipeline(step_cfg(), B, K, H, W, flip=True, chunks=chunks, device=DEV, want_idx=True)
    pinned = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t) for t in s]
    for rep in range(2):                                         # the second call reuses the staging buffers
        preds, loss = pipe(*pinned)
        assert np.array_equal(pipe.h_idx.numpy(), ref[1]), "argmax indices differ"
        assert_coords_close(preds.numpy()[..., :2], ref[0][..., :2], what=f"host pipeline B={B} chunks={chunks}", mag=ref[4])
        assert np.array_equal(preds.numpy()[..., 2], ref[0][..., 2], equal_nan=True)
        np.testing.assert_allclose(float(loss.item()), ref[2], rtol=1e-5)
    assert pipe.h2d_bytes == sum(t.numel() * t.element_size() for t in s)
    assert pipe.launches == len(pipe.bounds) + 2


def test_host_pipeline_accepts_numpy_and_pageable_inputs():
    """What a reference caller holds: pageable NumPy arrays (test.py:114-126 hands the decoder .cpu().numpy())."""
    B = 64
    s = make_set(B, 700, device="cpu")
    ref = oracle_of(s, ("host-np", B))
    pipe = fused.HostPipeline(step_cfg(), B, K, H, W, flip=True, chunks=4, device=DEV)
    preds, loss = pipe(*[t.numpy() for t in s])
    assert_coords_close(preds.numpy()[..., :2], ref[0][..., :2], what="numpy inputs", mag=ref[4])
    np.testing.assert_allclose(float(loss.item()), ref[2], rtol=1e-5)
    preds, loss = pipe(*s)                                                    # pageable torch tensors
    assert_coords_close(preds.numpy()[..., :2], ref[0][..., :2], what="pageable inputs", mag=ref[4])


def test_host_pipeline_decode_only():
    """loss_type=None: no render inputs, no loss buffers touched (ADVICE r1: it used to reduce uninitialised partials)."""
    B = 48
    s = make_set(B, 800, device="cpu")
    cfg = fused.FusedHeatmapStep(IMAGE, post_process="unbiased", kernel=11, loss_type=None)
    pipe = fused.HostPipeline(cfg, B, K, H, W, flip=True, chunks=3, device=DEV, want_idx=True)
    preds, loss = pipe(s[0], s[1], None, None, s[4], s[5])
    assert loss is None and pipe.launches == len(pipe.bounds)
    ref = oracle_of(s, ("host-dec", B))
    assert np.array_equal(pipe.h_idx.numpy(), ref[1])
    assert_coords_close(preds.numpy()[..., :2], ref[0][..., :2], what="decode-only host pipeline", mag=ref[4])


def test_ops_follow_the_tensors_device():
    """ADVICE r1: tensors on cuda:1 while cuda:0 is current must launch on cuda:1 (and mixed devices must raise)."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from litehandnet_b200 import ops
    s = make_set(4, 900, device="cuda:1")
    assert torch.cuda.current_device() == 0
    out = fused.fused_render_loss_decode(s[0], s[2], s[3], s[4], s[5], hm_flip=s[1])
    torch.cuda.synchronize("cuda:1")
    assert out["preds"].device == s[0].device
    ref = oracle_of(tuple(t.cpu() for t in s), ("dev1", 4))
    assert np.array_equal(out["idx"].cpu().numpy(), ref[1])
    with pytest.raises(L.LhnError):
        ops.decode_heatmap(s[0], L.MASK_NEG1, L.REFINE_NONE, L.XFORM_CENTER_SCALE, s[4].to("cuda:0"), s[5])


def test_bench_dump_outputs_are_the_last_timed_step(tmp_path):
    """bench.py --dump-outputs: the same arguments give the same arrays, and --steps decides which rotating input set
    the last timed step decoded (config 1 with three sets: steps 1 and 4 end on set 0, steps 5 on set 1).  The run
    exits non-zero when its outputs fail the oracle parity check."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

    def run(steps):
        d = tmp_path / f"steps{steps}"
        r = subprocess.run([sys.executable, "bench.py", "--config", "1", "--rotate", "3", "--steps", str(steps), "--warmup", "3",
                            "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           cwd=root, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
        return {f[:-4]: np.load(d / f) for f in os.listdir(d)}

    one, four, five = run(1), run(4), run(5)
    assert sorted(one) == ["hm_preds", "idx", "preds"]
    assert one["preds"].shape == (64, 21, 3) and one["preds"].dtype == np.float32 and one["idx"].dtype == np.float64
    assert all(np.array_equal(one[n], four[n], equal_nan=True) for n in one)
    assert not np.array_equal(four["idx"], five["idx"])


@pytest.mark.parametrize("config,names", [
    (2, {"preds": (64, 21, 3), "hm_preds": (64, 21, 3), "idx": (64, 21), "target_weight": (64, 21), "loss_sums": (4,),
         "loss": (1,)}),
    (3, {"preds": (64, 21, 3), "idx": (64, 21, 2)}),
    (4, {"preds": (64, 16, 3), "hm_preds": (64, 16, 3), "idx": (64, 16), "counters": (25 * 16,)})])
def test_bench_dump_outputs_of_every_workload(tmp_path, config, names):
    """bench.py --dump-outputs writes each workload's outputs under their names, in f32 or f64."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "bench.py", "--config", str(config), "--batch", "64", "--steps", "3", "--warmup", "3",
                        "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       cwd=root, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    got = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert {n: a.shape for n, a in got.items()} == names
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
