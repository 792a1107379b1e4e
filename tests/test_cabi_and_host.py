"""CPU (-m "not gpu"): the C-ABI library loads and exports every symbol include/lhn.h declares, the
host helpers behave, the product path refuses to run without a GPU (no silent fallback), and the
N>1 host logic works over gloo with world_size 2."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib_path():
    from litehandnet_b200 import build
    return build.build()


def test_library_exports_every_declared_symbol(lib_path):
    hdr = open(os.path.join(ROOT, "include", "lhn.h")).read()
    declared = set(re.findall(r"LHN_API\s+[\w\s\*]+?\b(lhn_\w+)\s*\(", hdr))
    assert len(declared) >= 17
    handle = ctypes.CDLL(lib_path)
    missing = [s for s in declared if not hasattr(handle, s)]
    assert not missing, missing
    from litehandnet_b200 import _lib
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    assert handle.lhn_version() == 100


def test_torch_extension_shim_loads():
    """The shim is built in-tree next to liblhn.so and exposes its two entry points (no compute without a GPU)."""
    from litehandnet_b200 import _lib
    e = _lib.ext()
    assert e is not None and hasattr(e, "decode_heatmap") and hasattr(e, "decode_simdr")
    assert os.path.dirname(e.__file__) == os.path.join(ROOT, "litehandnet_b200", "lib")


def test_struct_layouts_match_header():
    from litehandnet_b200 import _lib
    # lhn_decode_params: 6 int32 + 2 float + 31 double ; lhn_render_params: 4 int32 + 3 float + 8 float
    assert ctypes.sizeof(_lib.DecodeParams) == 6 * 4 + 2 * 4 + 31 * 8
    assert ctypes.sizeof(_lib.RenderParams) == 4 * 4 + 3 * 4 + 8 * 4
    assert _lib.DecodeParams.taps.offset == 32 and _lib.RenderParams.sigma.offset == 28
    # lhn_exchange: 8 pointers, world, rank, seq, timeout_ms, status*, prev_block*, prev_seq, prev2_seq, prev2_block*
    assert ctypes.sizeof(_lib.Exchange) == 8 * 8 + 4 * 4 + 8 + 8 + 2 * 4 + 8
    assert _lib.Exchange.status.offset == 80 and _lib.Exchange.prev_block.offset == 88 and _lib.Exchange.prev_seq.offset == 96
    assert _lib.Exchange.prev2_block.offset == 104
    assert _lib.XCH_MAILBOX_BYTES == 4 * 8 * 8192 + 4096


def test_exchange_argument_validation_without_gpu(lib_path):
    from litehandnet_b200 import _lib
    lib = _lib.lib()
    x = _lib.Exchange()
    x.world, x.rank, x.seq = 2, 0, 1
    x.mailbox[0] = 4096                                 # mailbox[1] missing
    x.prev_block, x.prev_seq = 4096, 1
    assert lib.lhn_exchange_flush(ctypes.byref(x), 400, ctypes.c_void_p(4096), None) == -1
    x.mailbox[1] = 8192
    x.prev_seq = 0                                      # step numbers start at 1
    assert lib.lhn_exchange_flush(ctypes.byref(x), 400, ctypes.c_void_p(4096), None) == -1
    x.prev_seq = 1
    assert lib.lhn_exchange_flush(ctypes.byref(x), 2000, ctypes.c_void_p(4096), None) == -1   # > payload
    x.prev_block, x.prev_seq = None, 0                  # nothing pending: a no-op
    assert lib.lhn_exchange_flush(ctypes.byref(x), 400, ctypes.c_void_p(4096), None) == 0
    assert lib.lhn_simdr_heads_workspace_bytes(64, 21, 512, 512) == 16 * 64 * 21 * 16
    assert lib.lhn_split_bf16(ctypes.c_void_p(16), 6, ctypes.c_void_p(16), ctypes.c_void_p(16), None) == -1       # n % 4


def test_gaussian_taps_match_opencv(lib_path):
    from litehandnet_b200 import _lib
    from oracle import np_oracle as O
    for k in (11, 19, 9, 31):
        taps = np.array(_lib.gaussian_taps(k))
        assert np.abs(taps - O.gaussian_kernel_1d(k, np.float64)).max() < 1e-16
    cv2 = pytest.importorskip("cv2")
    for k in (3, 5, 7, 11, 19):
        assert np.abs(np.array(_lib.gaussian_taps(k)) - cv2.getGaussianKernel(k, 0, cv2.CV_64F).ravel()).max() < 1e-16
    arr = (ctypes.c_double * 31)()
    assert _lib.lib().lhn_gaussian_taps(4, arr) == -1 and _lib.lib().lhn_gaussian_taps(33, arr) == -1


def test_host_argument_validation_without_gpu(lib_path):
    """Rejected calls return an error code before anything touches the device."""
    from litehandnet_b200 import _lib
    lib = _lib.lib()
    dp = _lib.DecodeParams()
    dp.mask_mode = 7
    rc = lib.lhn_decode_heatmap(ctypes.c_void_p(16), None, None, 0, 1, 21, 64, 64, 21 * 4096, 4096, 0, 0, None, None,
                                ctypes.byref(dp), None, None, None, None, None, 0, None, 0, None, None, None)
    assert rc == -1
    assert lib.lhn_decode_heatmap(None, None, None, 0, 1, 0, 64, 64, 0, 0, 0, 0, None, None, ctypes.byref(dp),
                                  None, None, None, None, None, 0, None, 0, None, None, None) == -1
    assert lib.lhn_loss_partials(None, None, None, 0, 1, 4096, 2, 0.5, None, None) == -1
    assert lib.lhn_simdr_loss_workspace_bytes(4096, 21) == 4096 * 21 * 16
    assert lib.lhn_evaluate_pck_workspace_bytes(64, 21) == 2 * 64 * 21 * 12


def test_k1_launch_record_without_gpu(lib_path):
    """lhn_k1_last_launch: a null pointer is refused; the record is per host thread, so a fresh thread reads
    path == 0 whatever ran before, and a call rejected before the launch (misaligned plane pointer) leaves it so."""
    import threading
    from litehandnet_b200 import _lib
    lib = _lib.lib()
    assert hasattr(lib, "lhn_k1_last_launch")
    assert ctypes.sizeof(_lib.K1LaunchInfo) == 15 * 4
    assert lib.lhn_k1_last_launch(None) == -1
    seen = []

    def probe():
        r = _lib.K1LaunchInfo()
        r.path, r.ctas = 7, 7
        seen.append((lib.lhn_k1_last_launch(ctypes.byref(r)), r.path, r.ctas))
        dp = _lib.DecodeParams()
        rc = lib.lhn_decode_heatmap(ctypes.c_void_p(18), None, None, _lib.F32, 1, 21, 64, 64, 21 * 4096, 4096, 0, 0,
                                    None, None, ctypes.byref(dp), None, None, None, None, None, 0, None, 0, None, None,
                                    None)
        r.path = 7
        seen.append((rc, lib.lhn_k1_last_launch(ctypes.byref(r)), r.path))

    t = threading.Thread(target=probe)
    t.start()
    t.join()
    assert seen == [(0, 0, 0), (-3, 0, 0)], seen


def test_simdr_launch_record_without_gpu(lib_path):
    """lhn_simdr_last_launch: a null pointer is refused; a fresh thread reads family == 0, and every SimDR entry point
    clears the record on entry, so a call rejected before its launch leaves it cleared."""
    import threading
    from litehandnet_b200 import _lib
    lib = _lib.lib()
    assert ctypes.sizeof(_lib.SimdrLaunchInfo) == 9 * 4
    assert lib.lhn_simdr_last_launch(None) == -1
    p = ctypes.c_void_p(16)
    rejected = {    # each call fails its argument checks before any device work
        "render": lambda: lib.lhn_render_simdr(p, 3, p, 1, 1, 21, 512, 512, 2.0, 0.0, p, p, None),
        "render_f64sigma": lambda: lib.lhn_render_simdr_f64sigma(p, 3, p, 1, 1, 21, 512, 512, 2.0, -1.0, p, p, None),
        "decode": lambda: lib.lhn_decode_simdr_flags(p, p, _lib.F32, 1, 0, 512, 512, 2, None, None, 0, None, p, None, 0,
                                                     None),
        "loss": lambda: lib.lhn_simdr_smoothl1(p, p, p, p, p, _lib.F32, 1, 21, 512, 512, p, 8, p, None),
        "backward": lambda: lib.lhn_simdr_smoothl1_backward(p, p, p, p, p, _lib.F32, 1, 21, 512, 512, 1.0, None, p, 4,
                                                           p, p, None),
        "heads": lambda: lib.lhn_simdr_heads_loss(p, p, p, p, p, p, p, p, 1, 21, 100, 512, 512, p, 1 << 20, p, None,
                                                  None, None),
        "heads_f32": lambda: lib.lhn_simdr_heads_loss_f32(p, p, p, p, p, p, p, 1, 21, 4096, 512, 512, p, 0, p, None,
                                                          None, None),
    }
    seen = []

    def probe():
        r = _lib.SimdrLaunchInfo()
        r.family, r.ctas = 7, 7
        seen.append(("fresh", lib.lhn_simdr_last_launch(ctypes.byref(r)), r.family, r.ctas))
        for name, call in rejected.items():
            rc = call()
            r.family = 7
            seen.append((name, rc < 0, lib.lhn_simdr_last_launch(ctypes.byref(r)), r.family))

    t = threading.Thread(target=probe)
    t.start()
    t.join()
    assert seen == [("fresh", 0, 0, 0)] + [(n, True, 0, 0) for n in rejected], seen


def test_no_cpu_fallback():
    """CPU tensors are refused loudly; nothing under litehandnet_b200/ imports the oracle."""
    from litehandnet_b200 import _lib, ops
    with pytest.raises(_lib.LhnError):
        ops.decode_heatmap(torch.zeros(1, 1, 64, 64), _lib.MASK_NONE, _lib.REFINE_NONE)
    with pytest.raises(_lib.LhnError):
        ops.loss_partials(torch.zeros(1, 1, 8, 8), torch.zeros(1, 1, 8, 8), torch.ones(1, 1), _lib.LOSS_DISTANCE)
    pkg = os.path.join(ROOT, "litehandnet_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f"{f} imports the oracle"
    if not torch.cuda.is_available():
        from litehandnet_b200 import decode
        with pytest.raises(_lib.LhnError):
            decode.keypoints_from_heatmaps(np.zeros((1, 1, 64, 64), np.float32), np.zeros((1, 2), np.float32),
                                           np.ones((1, 2), np.float32))


def test_missing_library_fails_loudly(tmp_path):
    code = ("import os; os.environ['LHN_LIB']=%r; from litehandnet_b200 import _lib; _lib.lib()" % str(tmp_path / "nope.so"))
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode != 0 and "no CPU or PyTorch fallback" in r.stderr


def test_shard_bounds_cover_batch():
    from litehandnet_b200 import dist as D
    for n, w in ((1024, 8), (1000, 3), (5, 8)):
        cuts = [D.shard_bounds(n, r, w) for r in range(w)]
        assert cuts[0][0] == 0 and cuts[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(cuts[:-1], cuts[1:]))


_GLOO_WORKER = r'''
import os, sys
sys.path.insert(0, %(root)r)
import numpy as np, torch, torch.distributed as dist
from litehandnet_b200 import dist as D
from oracle import np_oracle as O
rank = int(os.environ["RANK"]); world = int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo")
g = dict(np.load(os.path.join(%(root)r, "tests", "golden", "metrics_16.npz")))
p64 = g["preds"].astype(np.float64)
t = g["bbox_wh"].max(1).astype(np.float64); nor = np.stack([t, t], 1)
lo, hi = D.shard_bounds(len(p64), rank, world)
# metric counters of this rank's shard (oracle arithmetic stands in for the kernel on CPU)
hits, valid = O.pck_counters(p64[lo:hi], g["gt"][lo:hi], g["mask"][lo:hi], [0.2], nor[lo:hi])
cnt = torch.from_numpy(np.concatenate([hits.reshape(-1), valid]).astype(np.int64))
D.all_reduce_counters(cnt)
K = p64.shape[1]
acc, avg, n = O.pck_from_counters(cnt[:K].numpy(), cnt[K:].numpy())
assert np.array_equal(acc, g["ref_pck_acc"]) and avg == g["ref_pck_avg"], "sharded PCK != monolithic"
# loss sums: all-reduced shard sums == monolithic loss
rl = dict(np.load(os.path.join(%(root)r, "tests", "golden", "render_loss_64.npz")))
hm = np.nan_to_num(dict(np.load(os.path.join(%(root)r, "tests", "golden", "decode_64.npz")))["hm"], nan=0.25, posinf=1.0, neginf=-1.0)
tg, tw = rl["ref_target_unbiased"], rl["ref_weight_unbiased"]
lo, hi = D.shard_bounds(hm.shape[0], rank, world)
sums = torch.from_numpy(O.distance_loss_l2_sums(hm[lo:hi], tg[lo:hi], tw[lo:hi]))
D.all_reduce_loss_sums(sums)
loss = O.distance_loss_from_sums(sums.numpy(), True)
assert abs(float(loss) - float(rl["ref_distance_loss_unbiased_bal"])) <= 1e-6 * abs(float(loss)), (loss, rl["ref_distance_loss_unbiased_bal"])
# reference helper semantics
v = D.reduce_value(torch.tensor([float(rank + 1)]), average=True)
assert abs(v.item() - (world + 1) / 2) < 1e-6
s = D.all_reduce([1.0, float(rank)], device="cpu")
assert s.tolist() == [float(world), float(sum(range(world)))]
dist.destroy_process_group()
sys.stdout.write("rank " + str(rank) + " ok\n")      # ONE write: the two ranks share the pipe and print() writes piecewise
sys.stdout.flush()
'''


def test_sharded_counters_and_loss_sums_over_gloo(tmp_path):
    import socket
    script = tmp_path / "gloo_worker.py"
    script.write_text(_GLOO_WORKER % {"root": ROOT})
    for attempt in range(2):                          # the port can be taken between the probe and the rendezvous
        with socket.socket() as sk:                   # a free rendezvous port (a fixed one can be in TIME_WAIT)
            sk.bind(("127.0.0.1", 0))
            port = sk.getsockname()[1]
        r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
                            "--master-addr", "127.0.0.1", "--master-port", str(port), str(script)],
                           cwd=ROOT, capture_output=True, text=True, timeout=240)
        if r.returncode == 0:
            break
    assert r.returncode == 0, r.stdout + r.stderr
    assert "rank 0 ok" in r.stdout and "rank 1 ok" in r.stdout


@pytest.mark.parametrize("cfg", [1, 3, 4])
def test_bench_reference_arm_other_configs(cfg):
    import json
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--config", str(cfg), "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "16"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and f"configs[{cfg - 1}]" in line["config"]["workload"]


def test_bench_reference_arm_port_fallback():
    """LHN_CPU_PORT=1 forces the numpy port (what runs when no reference tree can be found)."""
    import json
    env = dict(os.environ, LHN_CPU_PORT="1")
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-sample", "16"],
                       cwd=ROOT, capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["cpu_baseline"]["kind"] == "port" and line["value"] > 0


def test_bench_reference_arm_prints_contract_line():
    import json
    r = subprocess.run([sys.executable, "bench.py", "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample", "16"], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    line = json.loads(r.stdout.strip().splitlines()[-1])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in line, key
    # kind: "reference" when the staged copy (oracle/_ref) or /root/reference is there, else the numpy port
    assert line["impl"] == "reference" and line["value"] > 0 and line["cpu_baseline"]["kind"] in ("reference", "port")


def test_bench_dump_outputs_types_and_sampling(tmp_path):
    """bench.dump_outputs: floats keep their precision, integers become exact f64; over the size limit every
    per-sample array keeps the same seeded rows (listed in sample_rows.npy) and the aggregates stay whole."""
    import bench
    B = 1000
    out = {"preds": torch.arange(B * 6, dtype=torch.float32).reshape(B, 2, 3),
           "idx": torch.arange(B * 2, dtype=torch.int32).reshape(B, 2),
           "loss_sums": torch.tensor([1.0, 2.0, 3.0, 4.0], dtype=torch.float64),
           "counters": torch.arange(B, dtype=torch.int64)}

    def load(d):
        return {f[:-4]: np.load(d / f) for f in os.listdir(d)}

    bench.dump_outputs(out, B, str(tmp_path / "whole"))
    whole = load(tmp_path / "whole")
    assert sorted(whole) == sorted(out)
    assert whole["preds"].dtype == np.float32 and whole["idx"].dtype == np.float64 and whole["counters"].dtype == np.float64
    for n, t in out.items():
        assert np.array_equal(whole[n], t.numpy()), n
    limit = 24000
    bench.dump_outputs(out, B, str(tmp_path / "a"), limit=limit)
    bench.dump_outputs(out, B, str(tmp_path / "b"), limit=limit)
    a, b = load(tmp_path / "a"), load(tmp_path / "b")
    assert sorted(a) == sorted(sorted(out) + ["sample_rows"]) and sorted(b) == sorted(a)
    assert all(np.array_equal(a[n], b[n]) for n in a), "the sample must not change from run to run"
    assert sum(os.path.getsize(tmp_path / "a" / f"{n}.npy") for n in a) <= limit
    rows = a["sample_rows"].astype(np.int64)
    assert 0 < len(rows) < B and np.all(np.diff(rows) > 0)
    assert np.array_equal(a["preds"], whole["preds"][rows]) and np.array_equal(a["idx"], whole["idx"][rows])
    assert np.array_equal(a["counters"], whole["counters"]) and np.array_equal(a["loss_sums"], whole["loss_sums"])
    with pytest.raises(ValueError):                  # aggregates alone over the limit: nothing to sample
        bench.dump_outputs({"counters": out["counters"]}, B, str(tmp_path / "c"), limit=4000)


def test_decode_params_cache_is_keyed_on_every_field(lib_path):
    """ops._decode_params shares one read-only struct between calls with equal arguments (host time per launch);
    any differing field — flags included — must give a different struct."""
    from litehandnet_b200 import _lib as L, ops
    a = ops._decode_params(L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, blur_ksize=11)
    b = ops._decode_params(L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, blur_ksize=11)
    assert a is b and a.blur_ksize == 11 and abs(sum(a.taps[i] for i in range(11)) - 1.0) < 1e-12
    c = ops._decode_params(L.MASK_NEG1, L.REFINE_DARK, L.XFORM_CENTER_SCALE, blur_ksize=11, flags=L.FLAG_OVERLAP_PREVIOUS)
    assert c is not a and c.flags == L.FLAG_OVERLAP_PREVIOUS and a.flags == 0
    d = ops._decode_params(L.MASK_NEG1, L.REFINE_DARK, L.XFORM_SCALE, scale_xy=(4.0, 2.0), blur_ksize=11)
    assert d is not a and (d.scale_x, d.scale_y, d.transform) == (4.0, 2.0, L.XFORM_SCALE)
    e = ops._decode_params(L.MASK_ZERO, L.REFINE_SIGN, L.XFORM_NONE, use_udp=True)
    assert e.use_udp == 1 and e.mask_mode == L.MASK_ZERO and e.blur_ksize == 0


def test_exchange_step_bookkeeping_on_cpu():
    """dist.PeerExchange.begin_step is the host half of the pipelined counter exchange (include/lhn.h
    lhn_decode_heatmap_pck_xch): launch s accumulates into block s % LHN_XCH_SLOTS, publishes the block of launch s-1 and
    adds the block of launch s-2 into the totals.  Checked here without a GPU on a CPU-resident instance."""
    import torch
    from litehandnet_b200 import _lib as L
    from litehandnet_b200.dist import PeerExchange
    x = PeerExchange.local_group(1, "cpu")[0]
    n = 25 * 16                                     # odd word counts are padded to an even row
    blocks = x.step_blocks(n + 1)
    assert blocks.shape == (L.XCH_SLOTS, n + 2) and blocks.dtype == torch.int64
    blocks = x.step_blocks(n)
    ptrs = [blocks[i].data_ptr() for i in range(L.XCH_SLOTS)]
    totals = torch.zeros(n, dtype=torch.int64)
    s = x.struct()
    assert s.world == 1 and s.rank == 0 and s.mailbox[0] == x.mailbox.data_ptr() and s.status == x.status.data_ptr()
    seen = []
    for step in range(1, 8):
        cur = x.begin_step(n, totals, s)
        assert s.seq == step and cur == ptrs[step % L.XCH_SLOTS]
        prev = (s.prev_seq, s.prev_block)
        prev2 = (s.prev2_seq, s.prev2_block)
        assert prev == ((step - 1, ptrs[(step - 1) % L.XCH_SLOTS]) if step > 1 else (0, None))
        assert prev2 == ((step - 2, ptrs[(step - 2) % L.XCH_SLOTS]) if step > 2 else (0, None))
        # a block is only reused after it was consumed (zeroed): LHN_XCH_SLOTS steps later, two after its consumption
        assert cur not in (s.prev_block, s.prev2_block)
        seen.append(cur)
    assert len(set(seen[:L.XCH_SLOTS])) == L.XCH_SLOTS
    assert [p[0] for p in x._pending] == [6, 7]     # what flush() completes: publish 7, consume 6 and 7
    with pytest.raises(L.LhnError):
        x.step_blocks(n + 8)                        # steps in flight: the block size cannot change before flush()
    assert x.bytes_per_step(n * 8) == 0             # one rank: nothing crosses NVLink
    y = PeerExchange.local_group(8, "cpu")[3]
    assert y.bytes_per_step(n * 8) == 7 * (n * 8 + 4)
