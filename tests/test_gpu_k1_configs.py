"""GPU: every launch configuration of the fused heatmap kernel (K1) against the NumPy oracle.

The host code picks one of many code paths per call: the persistent team kernel with one of the compile-time
instantiations of `dispatch_variant` or the run-time-size one, 2-, 4- or 8-warp teams with 1, 2 or 4 stages, render
tables built by the sweepers (`sweeper_tables`) or the epilogue warp, TMA bulk copies or element copies, teams dropped
to make room for the metric counters, or the CTA-per-plane kernel (plus the three-launch loss of the one-launch step).
Each case below names its inputs AND the launch record (`lhn_k1_last_launch`) the policy must produce for them, so a
policy change fails here instead of silently moving what the suite covers.  Then every entry point runs on the same
seeded inputs and is compared with the oracle, with a second run, and with the default configuration.
"""
import ctypes
import math
from collections import namedtuple

import numpy as np
import pytest
import torch

from conftest import assert_coords_close, xform_magnitude
from oracle import np_oracle as O
from litehandnet_b200 import _lib as L
from litehandnet_b200 import fused, ops, synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
DT = dict(f32=torch.float32, bf16=torch.bfloat16, f16=torch.float16)
DCODE = dict(f32=L.F32, bf16=L.BF16, f16=L.F16)
REF = dict(NONE=L.REFINE_NONE, OFFSET_HALF=L.REFINE_OFFSET_HALF, OFFSET=L.REFINE_OFFSET, SIGN=L.REFINE_SIGN,
           SIGN_ROUND=L.REFINE_SIGN_ROUND, DARK=L.REFINE_DARK, DARK_LEGACY=L.REFINE_DARK_LEGACY, DARK_UDP=L.REFINE_DARK_UDP)
LOSS = dict(bal=L.LOSS_DISTANCE_BALANCE, dist=L.LOSS_DISTANCE, mse=L.LOSS_JOINTS_MSE)
SWITCHES = ("LHN_NO_FAST", "LHN_TEAM_POLICY", "LHN_TEAM_STAGES", "LHN_STAGGER_NS", "LHN_CTAS_PER_SM", "LHN_FORCE_CTA_KERNEL")
# switches that leave the plane -> team assignment of the default configuration as it is: the loss sums are then
# added in the same order and must be bit-equal (element copies instead of TMA, the offset base, is another)
SAME_ORDER = {"LHN_NO_FAST", "LHN_TEAM_STAGES", "LHN_STAGGER_NS"}
ACC0 = 2.0 ** -20                       # loss already accumulated before a BoundFusedStep(accumulate_into=...) launch
RECORD = ("path", "wc", "twc", "ks", "team_warps", "nteams", "stages", "sweeper_tables")

# name, dtype, B, K, H, W, flip, loss (None = decode only), refinement, auc_steps of the fused counters (None = off),
# environment switches, base pointer 4 bytes off 16-byte alignment, overlap_previous,
# expected record: (path, wc, twc, ks, team_warps, nteams, stages, sweeper_tables).  ctas, use_tma and stagger_ns follow
# from the inputs and are checked as well.
C_ = namedtuple("C_", "name dt B K H W flip loss refine auc env off overlap rec")


def C(*a):
    return C_(*a)


CASES = [
    # ---- 1. every compile-time instantiation of dispatch_variant, loss off / on, KS = 11 (DARK, k = 11) / KS = 0 ----
    # Not reachable, so not listed:
    #  - f32 128x128 with flip: two 64 KB planes per team leave room for one team, the team kernel needs two; the
    #    CTA-per-plane kernel takes it ('f32-128-flip-bal-dark' in section 5).
    #  - f32 32x32 / 16x16 with flip: only instantiated without flip; with flip they take the run-time-size path.
    #  - bf16 / f16 128/4 with KS = 11: the DARK tiles make a team's auxiliary region too large for six 4-warp teams,
    #    so 128x128 without flip and with DARK runs 8-warp teams on the run-time-size instantiation (rows below).
    C('f32-128-decode-dark', 'f32', 32, 21, 128, 128, False, None, 'DARK', None, {}, False, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('f32-128-decode-sign', 'f32', 32, 21, 128, 128, False, None, 'SIGN', None, {}, False, False, (1, 128, 8, 0, 8, 3, 1, 0)),
    C('f32-128-dist-dark', 'f32', 32, 21, 128, 128, False, 'dist', 'DARK', None, {}, False, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('f32-128-mse-dark_udp', 'f32', 32, 21, 128, 128, False, 'mse', 'DARK_UDP', None, {}, False, False, (1, 128, 8, 0, 8, 3, 1, 0)),
    C('f32-32-decode-dark', 'f32', 127, 21, 32, 32, False, None, 'DARK', None, {}, False, False, (1, 32, 2, 11, 2, 12, 2, 0)),
    C('f32-32-decode-sign', 'f32', 127, 21, 32, 32, False, None, 'SIGN', None, {}, False, False, (1, 32, 2, 0, 2, 12, 4, 0)),
    C('f32-32-bal-dark', 'f32', 127, 21, 32, 32, False, 'bal', 'DARK', None, {}, False, False, (1, 32, 2, 11, 2, 12, 2, 0)),
    C('f32-32-dist-dark_udp', 'f32', 127, 21, 32, 32, False, 'dist', 'DARK_UDP', None, {}, False, False, (1, 32, 2, 0, 2, 12, 2, 0)),
    C('f32-16-decode-dark', 'f32', 127, 21, 16, 16, False, None, 'DARK', None, {}, False, False, (1, 16, 2, 11, 2, 12, 4, 0)),
    C('f32-16-decode-sign', 'f32', 127, 21, 16, 16, False, None, 'SIGN', None, {}, False, False, (1, 16, 2, 0, 2, 12, 4, 0)),
    C('f32-16-mse-dark', 'f32', 127, 21, 16, 16, False, 'mse', 'DARK', None, {}, False, False, (1, 16, 2, 11, 2, 12, 4, 0)),
    C('f32-16-bal-dark_udp', 'f32', 127, 21, 16, 16, False, 'bal', 'DARK_UDP', None, {}, False, False, (1, 16, 2, 0, 2, 12, 4, 0)),
    C('f32-64-decode-dark', 'f32', 106, 21, 64, 64, False, None, 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('f32-64-decode-sign', 'f32', 127, 21, 64, 64, False, None, 'SIGN', None, {}, False, False, (1, 64, 2, 0, 2, 12, 1, 0)),
    C('f32-64-dist-dark', 'f32', 106, 21, 64, 64, False, 'dist', 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('f32-64-mse-dark_udp', 'f32', 106, 21, 64, 64, False, 'mse', 'DARK_UDP', None, {}, False, False, (1, 64, 2, 0, 2, 10, 1, 0)),
    C('f32-64-flip-decode-dark', 'f32', 64, 21, 64, 64, True, None, 'DARK', None, {}, False, False, (1, 64, 4, 11, 4, 6, 1, 0)),
    C('f32-64-flip-decode-sign', 'f32', 64, 21, 64, 64, True, None, 'SIGN', None, {}, False, False, (1, 64, 4, 0, 4, 6, 1, 0)),
    C('f32-64-flip-bal-dark', 'f32', 64, 21, 64, 64, True, 'bal', 'DARK', None, {}, False, False, (1, 64, 4, 11, 4, 6, 1, 0)),
    C('f32-64-flip-dist-sign_round', 'f32', 64, 21, 64, 64, True, 'dist', 'SIGN_ROUND', None, {}, False, False, (1, 64, 4, 0, 4, 6, 1, 0)),
    C('f32-56-decode-dark', 'f32', 127, 21, 56, 56, False, None, 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 1, 0)),
    C('f32-56-decode-sign', 'f32', 127, 21, 56, 56, False, None, 'SIGN', None, {}, False, False, (1, 56, 2, 0, 2, 12, 1, 0)),
    C('f32-56-mse-dark', 'f32', 127, 21, 56, 56, False, 'mse', 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 1, 0)),
    C('f32-56-bal-dark_udp', 'f32', 127, 21, 56, 56, False, 'bal', 'DARK_UDP', None, {}, False, False, (1, 56, 2, 0, 2, 12, 1, 0)),
    C('f32-56-flip-decode-dark', 'f32', 64, 21, 56, 56, True, None, 'DARK', None, {}, False, False, (1, 56, 4, 11, 4, 6, 1, 0)),
    C('f32-56-flip-decode-sign', 'f32', 64, 21, 56, 56, True, None, 'SIGN', None, {}, False, False, (1, 56, 4, 0, 4, 6, 1, 0)),
    C('f32-56-flip-dist-dark', 'f32', 64, 21, 56, 56, True, 'dist', 'DARK', None, {}, False, False, (1, 56, 4, 11, 4, 6, 1, 0)),
    C('f32-56-flip-mse-dark_udp', 'f32', 64, 21, 56, 56, True, 'mse', 'DARK_UDP', None, {}, False, False, (1, 56, 4, 0, 4, 6, 1, 0)),
    C('bf16-128-decode-dark', 'bf16', 32, 21, 128, 128, False, None, 'DARK', None, {}, False, False, (1, 0, 0, 11, 8, 3, 2, 1)),
    C('bf16-128-decode-sign', 'bf16', 64, 21, 128, 128, False, None, 'SIGN', None, {}, False, False, (1, 128, 4, 0, 4, 6, 1, 0)),
    C('bf16-128-bal-dark', 'bf16', 32, 21, 128, 128, False, 'bal', 'DARK', None, {}, False, False, (1, 0, 0, 11, 8, 3, 2, 1)),
    C('bf16-128-dist-offset_half', 'bf16', 64, 21, 128, 128, False, 'dist', 'OFFSET_HALF', None, {}, False, False, (1, 128, 4, 0, 4, 6, 1, 0)),
    C('bf16-128-flip-decode-dark', 'bf16', 32, 21, 128, 128, True, None, 'DARK', None, {}, False, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('bf16-128-flip-decode-sign', 'bf16', 32, 21, 128, 128, True, None, 'SIGN', None, {}, False, False, (1, 128, 8, 0, 8, 3, 1, 0)),
    C('bf16-128-flip-mse-dark', 'bf16', 32, 21, 128, 128, True, 'mse', 'DARK', None, {}, False, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('bf16-128-flip-bal-dark_udp', 'bf16', 32, 21, 128, 128, True, 'bal', 'DARK_UDP', None, {}, False, False, (1, 128, 8, 0, 8, 3, 1, 0)),
    C('bf16-64-decode-dark', 'bf16', 127, 21, 64, 64, False, None, 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 12, 1, 0)),
    C('bf16-64-decode-sign', 'bf16', 127, 21, 64, 64, False, None, 'SIGN', None, {}, False, False, (1, 64, 2, 0, 2, 12, 2, 0)),
    C('bf16-64-dist-dark', 'bf16', 127, 21, 64, 64, False, 'dist', 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 12, 1, 0)),
    C('bf16-64-mse-dark_udp', 'bf16', 127, 21, 64, 64, False, 'mse', 'DARK_UDP', None, {}, False, False, (1, 64, 2, 0, 2, 12, 1, 0)),
    C('bf16-64-flip-decode-dark', 'bf16', 106, 21, 64, 64, True, None, 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('bf16-64-flip-decode-sign', 'bf16', 127, 21, 64, 64, True, None, 'SIGN', None, {}, False, False, (1, 64, 2, 0, 2, 12, 1, 0)),
    C('bf16-64-flip-bal-dark', 'bf16', 106, 21, 64, 64, True, 'bal', 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('bf16-64-flip-dist-dark_udp', 'bf16', 106, 21, 64, 64, True, 'dist', 'DARK_UDP', None, {}, False, False, (1, 64, 2, 0, 2, 10, 1, 0)),
    C('bf16-56-decode-dark', 'bf16', 127, 21, 56, 56, False, None, 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 2, 0)),
    C('bf16-56-decode-sign', 'bf16', 127, 21, 56, 56, False, None, 'SIGN', None, {}, False, False, (1, 56, 2, 0, 2, 12, 2, 0)),
    C('bf16-56-mse-dark', 'bf16', 127, 21, 56, 56, False, 'mse', 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 2, 0)),
    C('bf16-56-bal-dark_udp', 'bf16', 127, 21, 56, 56, False, 'bal', 'DARK_UDP', None, {}, False, False, (1, 56, 2, 0, 2, 12, 2, 0)),
    C('bf16-56-flip-decode-dark', 'bf16', 127, 21, 56, 56, True, None, 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 1, 0)),
    C('bf16-56-flip-decode-sign', 'bf16', 127, 21, 56, 56, True, None, 'SIGN', None, {}, False, False, (1, 56, 2, 0, 2, 12, 1, 0)),
    C('bf16-56-flip-dist-dark', 'bf16', 127, 21, 56, 56, True, 'dist', 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 1, 0)),
    C('bf16-56-flip-mse-dark_udp', 'bf16', 127, 21, 56, 56, True, 'mse', 'DARK_UDP', None, {}, False, False, (1, 56, 2, 0, 2, 12, 1, 0)),
    C('f16-128-decode-dark', 'f16', 32, 21, 128, 128, False, None, 'DARK', None, {}, False, False, (1, 0, 0, 11, 8, 3, 2, 1)),
    C('f16-128-decode-sign', 'f16', 64, 21, 128, 128, False, None, 'SIGN', None, {}, False, False, (1, 128, 4, 0, 4, 6, 1, 0)),
    C('f16-128-bal-dark', 'f16', 32, 21, 128, 128, False, 'bal', 'DARK', None, {}, False, False, (1, 0, 0, 11, 8, 3, 2, 1)),
    C('f16-128-dist-offset_half', 'f16', 64, 21, 128, 128, False, 'dist', 'OFFSET_HALF', None, {}, False, False, (1, 128, 4, 0, 4, 6, 1, 0)),
    C('f16-128-flip-decode-dark', 'f16', 32, 21, 128, 128, True, None, 'DARK', None, {}, False, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('f16-128-flip-decode-sign', 'f16', 32, 21, 128, 128, True, None, 'SIGN', None, {}, False, False, (1, 128, 8, 0, 8, 3, 1, 0)),
    C('f16-128-flip-mse-dark', 'f16', 32, 21, 128, 128, True, 'mse', 'DARK', None, {}, False, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('f16-128-flip-bal-dark_udp', 'f16', 32, 21, 128, 128, True, 'bal', 'DARK_UDP', None, {}, False, False, (1, 128, 8, 0, 8, 3, 1, 0)),
    C('f16-64-decode-dark', 'f16', 127, 21, 64, 64, False, None, 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 12, 1, 0)),
    C('f16-64-decode-sign', 'f16', 127, 21, 64, 64, False, None, 'SIGN', None, {}, False, False, (1, 64, 2, 0, 2, 12, 2, 0)),
    C('f16-64-dist-dark', 'f16', 127, 21, 64, 64, False, 'dist', 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 12, 1, 0)),
    C('f16-64-mse-dark_udp', 'f16', 127, 21, 64, 64, False, 'mse', 'DARK_UDP', None, {}, False, False, (1, 64, 2, 0, 2, 12, 1, 0)),
    C('f16-64-flip-decode-dark', 'f16', 106, 21, 64, 64, True, None, 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('f16-64-flip-decode-sign', 'f16', 127, 21, 64, 64, True, None, 'SIGN', None, {}, False, False, (1, 64, 2, 0, 2, 12, 1, 0)),
    C('f16-64-flip-bal-dark', 'f16', 106, 21, 64, 64, True, 'bal', 'DARK', None, {}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('f16-64-flip-dist-dark_udp', 'f16', 106, 21, 64, 64, True, 'dist', 'DARK_UDP', None, {}, False, False, (1, 64, 2, 0, 2, 10, 1, 0)),
    C('f16-56-decode-dark', 'f16', 127, 21, 56, 56, False, None, 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 2, 0)),
    C('f16-56-decode-sign', 'f16', 127, 21, 56, 56, False, None, 'SIGN', None, {}, False, False, (1, 56, 2, 0, 2, 12, 2, 0)),
    C('f16-56-mse-dark', 'f16', 127, 21, 56, 56, False, 'mse', 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 2, 0)),
    C('f16-56-bal-dark_udp', 'f16', 127, 21, 56, 56, False, 'bal', 'DARK_UDP', None, {}, False, False, (1, 56, 2, 0, 2, 12, 2, 0)),
    C('f16-56-flip-decode-dark', 'f16', 127, 21, 56, 56, True, None, 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 1, 0)),
    C('f16-56-flip-decode-sign', 'f16', 127, 21, 56, 56, True, None, 'SIGN', None, {}, False, False, (1, 56, 2, 0, 2, 12, 1, 0)),
    C('f16-56-flip-dist-dark', 'f16', 127, 21, 56, 56, True, 'dist', 'DARK', None, {}, False, False, (1, 56, 2, 11, 2, 12, 1, 0)),
    C('f16-56-flip-mse-dark_udp', 'f16', 127, 21, 56, 56, True, 'mse', 'DARK_UDP', None, {}, False, False, (1, 56, 2, 0, 2, 12, 1, 0)),
    # ---- 2. the run-time-size instantiation: LHN_NO_FAST=1 on the fast shapes, and H != W ----
    C('nofast-f32-128-decode-dark', 'f32', 32, 21, 128, 128, False, None, 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 8, 3, 1, 0)),
    C('nofast-f32-32-bal-dark', 'f32', 127, 21, 32, 32, False, 'bal', 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 2, 12, 2, 0)),
    C('nofast-f32-16-decode-sign', 'f32', 127, 21, 16, 16, False, None, 'SIGN', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 0, 2, 12, 4, 0)),
    C('nofast-f32-64-bal-dark', 'f32', 106, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 2, 10, 1, 0)),
    C('nofast-f32-64-flip-dist-dark', 'f32', 64, 21, 64, 64, True, 'dist', 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 4, 6, 1, 0)),
    C('nofast-f32-56-decode-dark', 'f32', 127, 21, 56, 56, False, None, 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 2, 12, 1, 0)),
    C('nofast-f32-56-flip-mse-dark', 'f32', 64, 21, 56, 56, True, 'mse', 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 4, 6, 1, 0)),
    C('nofast-bf16-128-decode-sign', 'bf16', 64, 21, 128, 128, False, None, 'SIGN', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 0, 4, 6, 1, 0)),
    C('nofast-bf16-128-flip-bal-dark', 'bf16', 32, 21, 128, 128, True, 'bal', 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 8, 3, 1, 0)),
    C('nofast-bf16-64-bal-dark', 'bf16', 127, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 2, 12, 1, 0)),
    C('nofast-f16-56-flip-dist-dark', 'f16', 127, 21, 56, 56, True, 'dist', 'DARK', None, {'LHN_NO_FAST': '1'}, False, False, (1, 0, 0, 11, 2, 12, 1, 0)),
    C('f32-64x48-bal-dark', 'f32', 127, 21, 64, 48, False, 'bal', 'DARK', None, {}, False, False, (1, 0, 0, 11, 2, 12, 1, 0)),
    C('f32-40x72-flip-decode-sign', 'f32', 64, 21, 40, 72, True, None, 'SIGN', None, {}, False, False, (1, 0, 0, 0, 4, 6, 1, 0)),
    C('f32-40x72-mse-dark', 'f32', 127, 21, 40, 72, False, 'mse', 'DARK', None, {}, False, False, (1, 0, 0, 11, 2, 12, 1, 0)),
    C('bf16-64x48-flip-bal-dark', 'bf16', 127, 21, 64, 48, True, 'bal', 'DARK', None, {}, False, False, (1, 0, 0, 11, 2, 12, 1, 0)),
    # ---- 3. team geometries: 4-warp teams with 2 and 4 stages and sweeper tables, 8-warp teams, stage counts lowered.
    # Every reachable (team_warps, stages, sweeper_tables) triple is here: (2, 1|2|4, 0), (4, 1, 0), (4, 2|4, 1),
    # (8, 1, 0), (8, 2, 1).  Sweeper tables come with every multi-stage team of 4 or more warps, and 2-warp teams never
    # have them.  (8, 4, 1) needs 6 teams that do not fit with two that hold four stages: a stage above 16 KB whose
    # team region is still small enough for 2 x 4 stages, so the auxiliary region (4 bytes per joint) has to carry K in
    # the thousands, with or without LHN_TEAM_POLICY=0.  It is left out for that reason. ----
    C('policy0-f32-64-bal-dark', 'f32', 127, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_TEAM_POLICY': '0'}, False, False, (1, 0, 0, 11, 4, 6, 2, 1)),
    C('policy0-f32-64-decode-sign', 'f32', 127, 21, 64, 64, False, None, 'SIGN', None, {'LHN_TEAM_POLICY': '0'}, False, False, (1, 0, 0, 0, 4, 6, 2, 1)),
    C('policy0-f32-32-bal-dark', 'f32', 254, 21, 32, 32, False, 'bal', 'DARK', None, {'LHN_TEAM_POLICY': '0'}, False, False, (1, 0, 0, 11, 4, 6, 4, 1)),
    C('policy0-f32-32-decode-sign', 'f32', 254, 21, 32, 32, False, None, 'SIGN', None, {'LHN_TEAM_POLICY': '0'}, False, False, (1, 0, 0, 0, 4, 6, 4, 1)),
    C('policy0-stages2-f32-32-bal-dark', 'f32', 254, 21, 32, 32, False, 'bal', 'DARK', None, {'LHN_TEAM_POLICY': '0', 'LHN_TEAM_STAGES': '2'}, False, False, (1, 0, 0, 11, 4, 6, 2, 1)),
    C('notma-policy0-f32-32-bal-dark', 'f32', 254, 21, 32, 32, False, 'bal', 'DARK', None, {'LHN_TEAM_POLICY': '0'}, True, False, (1, 0, 0, 11, 4, 6, 4, 1)),
    C('policy0-stages1-f32-64-bal-dark', 'f32', 127, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_TEAM_POLICY': '0', 'LHN_TEAM_STAGES': '1'}, False, False, (1, 0, 0, 11, 4, 6, 1, 0)),
    C('f32-96-bal-dark', 'f32', 64, 21, 96, 96, False, 'bal', 'DARK', None, {}, False, False, (1, 0, 0, 11, 8, 3, 1, 0)),
    C('f32-96-bal-sign', 'f32', 64, 21, 96, 96, False, 'bal', 'SIGN', None, {}, False, False, (1, 0, 0, 0, 8, 3, 2, 1)),
    C('f32-68x64-flip-dist-dark', 'f32', 64, 21, 68, 64, True, 'dist', 'DARK', None, {}, False, False, (1, 0, 0, 11, 8, 3, 2, 1)),
    C('f32-64x68-bal-dark', 'f32', 127, 21, 64, 68, False, 'bal', 'DARK', None, {}, False, False, (1, 0, 0, 11, 4, 6, 1, 0)),
    C('f32-48x44-flip-bal-sign', 'f32', 127, 21, 48, 44, True, 'bal', 'SIGN', None, {}, False, False, (1, 0, 0, 0, 4, 6, 2, 1)),
    C('f32-64-flip-bal-dark_legacy', 'f32', 22, 21, 64, 64, True, 'bal', 'DARK_LEGACY', None, {}, False, False, (1, 0, 0, 0, 8, 3, 2, 1)),
    C('f32-16-bal-dark-x4', 'f32', 508, 21, 16, 16, False, 'bal', 'DARK', None, {}, False, False, (1, 16, 2, 11, 2, 12, 4, 0)),
    C('stages2-f32-16-bal-dark', 'f32', 508, 21, 16, 16, False, 'bal', 'DARK', None, {'LHN_TEAM_STAGES': '2'}, False, False, (1, 16, 2, 11, 2, 12, 2, 0)),
    C('stages1-f32-16-bal-dark', 'f32', 508, 21, 16, 16, False, 'bal', 'DARK', None, {'LHN_TEAM_STAGES': '1'}, False, False, (1, 16, 2, 11, 2, 12, 1, 0)),
    C('stages1-f32-32-decode-sign', 'f32', 508, 21, 32, 32, False, None, 'SIGN', None, {'LHN_TEAM_STAGES': '1'}, False, False, (1, 32, 2, 0, 2, 12, 1, 0)),
    C('f32-32-bal-dark-x2', 'f32', 339, 21, 32, 32, False, 'bal', 'DARK', None, {}, False, False, (1, 32, 2, 11, 2, 12, 2, 0)),
    # ---- 4. element copies instead of TMA (base address = 4 mod 16) under 2-, 4- and 8-warp teams ----
    C('notma-f32-64-bal-dark', 'f32', 106, 21, 64, 64, False, 'bal', 'DARK', None, {}, True, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('notma-f32-64-flip-bal-dark', 'f32', 64, 21, 64, 64, True, 'bal', 'DARK', None, {}, True, False, (1, 64, 4, 11, 4, 6, 1, 0)),
    C('notma-f32-128-dist-dark', 'f32', 32, 21, 128, 128, False, 'dist', 'DARK', None, {}, True, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('notma-f32-128-decode-sign', 'f32', 32, 21, 128, 128, False, None, 'SIGN', None, {}, True, False, (1, 128, 8, 0, 8, 3, 1, 0)),
    C('notma-bf16-64-flip-mse-dark', 'bf16', 106, 21, 64, 64, True, 'mse', 'DARK', None, {}, True, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('notma-bf16-128-flip-bal-dark', 'bf16', 32, 21, 128, 128, True, 'bal', 'DARK', None, {}, True, False, (1, 128, 8, 11, 8, 3, 1, 0)),
    C('notma-policy0-f32-64-bal-dark', 'f32', 127, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_TEAM_POLICY': '0'}, True, False, (1, 0, 0, 11, 4, 6, 2, 1)),
    C('notma-f32-16-bal-dark', 'f32', 508, 21, 16, 16, False, 'bal', 'DARK', None, {}, True, False, (1, 16, 2, 11, 2, 12, 4, 0)),
    # ---- 5. the CTA-per-plane kernel: forced (64x64 run-time width, 128x128 its WT = 128 instantiation) and where
    #      the team kernel refuses the shape (W % 4 != 0; f32 128x128 with flip) ----
    C('cta-f32-64-decode-dark', 'f32', 12, 21, 64, 64, False, None, 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('cta-f32-64-bal-dark', 'f32', 12, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('cta-f32-64-flip-decode-dark', 'f32', 12, 21, 64, 64, True, None, 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('cta-f32-64-flip-bal-dark', 'f32', 12, 21, 64, 64, True, 'bal', 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('cta-f32-128-decode-dark', 'f32', 4, 21, 128, 128, False, None, 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    C('cta-f32-128-dist-dark', 'f32', 4, 21, 128, 128, False, 'dist', 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    C('cta-f32-128-flip-decode-dark', 'f32', 4, 21, 128, 128, True, None, 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    C('cta-f32-128-flip-dist-dark', 'f32', 4, 21, 128, 128, True, 'dist', 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    C('cta-f16-64-bal-dark', 'f16', 12, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('cta-bf16-128-decode-dark', 'bf16', 4, 21, 128, 128, False, None, 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    C('cta-bf16-128-flip-bal-dark', 'bf16', 4, 21, 128, 128, True, 'bal', 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    C('cta-f16-128-flip-mse-sign', 'f16', 4, 21, 128, 128, True, 'mse', 'SIGN', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    C('cta-bf16-64-flip-mse-sign', 'bf16', 12, 21, 64, 64, True, 'mse', 'SIGN', None, {'LHN_FORCE_CTA_KERNEL': '1'}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('cta-notma-f32-64-bal-dark', 'f32', 12, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_FORCE_CTA_KERNEL': '1'}, True, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('f32-14-bal-sign', 'f32', 40, 21, 14, 14, False, 'bal', 'SIGN', None, {}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('f32-14-flip-decode-dark', 'f32', 40, 21, 14, 14, True, None, 'DARK', None, {}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('f32-128-flip-bal-dark', 'f32', 6, 21, 128, 128, True, 'bal', 'DARK', None, {}, False, False, (2, 128, 0, 0, 0, 0, 0, 0)),
    # ---- 6. overlapped launches in half of the shared memory, and the stagger between teams ----
    C('ctas2-f32-64-decode-dark', 'f32', 53, 21, 64, 64, False, None, 'DARK', None, {'LHN_CTAS_PER_SM': '2'}, False, True, (1, 64, 2, 11, 2, 5, 1, 0)),
    C('ctas2-f32-64-flip-bal-dark', 'f32', 32, 21, 64, 64, True, 'bal', 'DARK', None, {'LHN_CTAS_PER_SM': '2'}, False, True, (1, 0, 0, 11, 8, 3, 1, 0)),
    C('stagger600-f32-64-bal-dark', 'f32', 8, 21, 64, 64, False, 'bal', 'DARK', None, {'LHN_STAGGER_NS': '600'}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
    C('f32-64-decode-sign-large', 'f32', 680, 21, 64, 64, False, None, 'SIGN', None, {}, False, False, (1, 64, 2, 0, 2, 12, 1, 0)),
    C('stagger0-f32-64-decode-sign-large', 'f32', 680, 21, 64, 64, False, None, 'SIGN', None, {'LHN_STAGGER_NS': '0'}, False, False, (1, 64, 2, 0, 2, 12, 1, 0)),
    # ---- 7. fused counters: teams dropped to make room (12 -> 10), and no room at all (CTA-per-plane kernel) ----
    C('cnt-f32-64-k64-auc64', 'f32', 40, 64, 64, 64, False, None, 'SIGN', 64, {}, False, False, (1, 64, 2, 0, 2, 10, 1, 0)),
    C('cnt-f32-64-k400-auc64', 'f32', 2, 400, 64, 64, False, None, 'SIGN', 64, {}, False, False, (2, 0, 0, 0, 0, 0, 0, 0)),
    C('cnt-f32-64-k21-auc20', 'f32', 100, 21, 64, 64, False, None, 'DARK', 20, {}, False, False, (1, 64, 2, 11, 2, 10, 1, 0)),
]


def last_launch():
    r = L.K1LaunchInfo()
    L.check(L.lib().lhn_k1_last_launch(ctypes.byref(r)), "lhn_k1_last_launch")
    return {f: getattr(r, f) for f, _ in L.K1LaunchInfo._fields_}


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


def set_env(monkeypatch, env):
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


# ---- seeded inputs and their oracle, shared by every configuration of the same shape ----------------------------------
_INPUTS, _ORACLE = {}, {}


def _sigma(W):
    return 2.0 * W / 64 if W >= 32 else 1.0


def inputs(case):
    key = (case.dt, case.B, case.K, case.H, case.W, case.flip, case.refine)
    if key in _INPUTS:
        return _INPUTS[key]
    B, K, H, W = case.B, case.K, case.H, case.W
    seed = (B * 131 + K * 17 + H * 7 + W) % 100003
    # exact ties only where the refinement is well conditioned on them: a tie puts DARK's peak on an isolated noise
    # spike where its 2x2 solve amplifies 1-ulp blur differences (test_gpu_round2.py)
    ties = 0.0 if case.refine.startswith("DARK") else 0.05
    hm, cen = synth.blob_heatmaps(B, K, H, W, seed=seed, sigma=max(1.0, 2.0 * min(H, W) / 64), margin=min(4.0, min(H, W) / 8),
                                  zero_frac=0.02, tie_frac=ties)
    hm = hm.to(DT[case.dt])
    hf = synth.flipped_blob_heatmaps(cen, H, W, seed=seed + 1, sigma=max(1.0, 2.0 * min(H, W) / 64)).to(DT[case.dt]) \
        if case.flip else None
    c, s = synth.bbox_center_scale(B, seed=seed + 2)
    s = s * torch.tensor([1.0, 0.8])                                      # anisotropic boxes
    img = (4 * W, 4 * H)
    j, v = synth.hand_joints(B, K, img, seed=seed + 3, vis_prob=0.9, outside_frac=0.05)
    gt, mask, wh = synth.pck_inputs(cen, seed=seed + 4)
    mask[0, 0] = False
    if B > 2:
        wh[1] = 0.0                                                       # PCK masks the sample, AUC / EPE do not
    d = dict(hm=hm, hf=hf, c=c, s=s, j=j, v=v, gt=gt, mask=mask, wh=wh, img=img, sigma=_sigma(W))
    d["dev"] = {k: (t.to(DEV) if isinstance(t, torch.Tensor) else t) for k, t in d.items()}
    _INPUTS.clear()
    _INPUTS[key] = d
    return d


def oracle(case, d):
    key = (case.dt, case.B, case.K, case.H, case.W, case.flip, case.refine, case.loss)
    if key in _ORACLE:
        return _ORACLE[key]
    hm32 = d["hm"].float().numpy()
    avg = hm32 if d["hf"] is None else O.flip_average(hm32, d["hf"].float().numpy(), ())
    r = dict(idx=O.argmax_planes(avg)[0])
    p0, mv, _ = O.max_preds(avg, "neg1")
    rf = case.refine
    with np.errstate(all="ignore"):
        want = {"NONE": lambda: p0, "OFFSET_HALF": lambda: O.refine_offset_clamped(p0, avg, True),
                "OFFSET": lambda: O.refine_offset_clamped(p0, avg, False), "SIGN": lambda: O.refine_sign_guarded(p0, avg),
                "SIGN_ROUND": lambda: O.refine_sign_guarded(p0, avg, round_half=True),
                "DARK": lambda: O.refine_dark(p0, avg, 11, False), "DARK_LEGACY": lambda: O.refine_dark(p0, avg, 19, True),
                "DARK_UDP": lambda: O.post_dark_udp(p0, avg.copy(), 11)}[rf]()
    c, s = d["c"].numpy(), d["s"].numpy()
    r["hm"], r["maxval"] = want, mv
    r["img"] = np.stack([O.transform_preds(want[i], c[i], s[i], [case.W, case.H], use_udp=(rf == "DARK_UDP"))[:, :2]
                         for i in range(case.B)])
    if case.loss is not None:
        tg, tw = O.render_targets(d["j"].numpy(), d["v"].numpy(), d["img"], (case.W, case.H), d["sigma"], True)
        r["weight"] = tw.reshape(case.B, case.K)
        o64, t64 = hm32.astype(np.float64), tg.astype(np.float64)
        w64 = tw.astype(np.float64)[..., None]
        if case.loss == "bal":
            r["sums"] = O.distance_loss_l2_sums(hm32, tg, tw)
            r["loss"] = O.distance_loss_l2(hm32, tg, tw, balance=True)
        else:
            w = w64 * w64 if case.loss == "mse" else w64
            r["sums"] = np.array([0.0, float((((o64 - t64) ** 2) * w).sum()), 0.0, float(o64.size)])
            r["loss"] = O.joints_distance_loss_mse(hm32, tg, tw) if case.loss == "mse" else \
                O.distance_loss_l2(hm32, tg, tw, balance=False)
    _ORACLE.clear()
    _ORACLE[key] = r
    return r


def oracle_counters(case, d, kpts, auc_steps, pck_thr=0.2, auc_nor=30.0):
    """Counters as lhn_decode_heatmap_pck lays them out, from the kernel's own image coordinates."""
    K = case.K
    pred = kpts[..., :2].astype(np.float64)
    gt, mask = d["gt"].numpy(), d["mask"].numpy()
    nb = np.maximum(d["wh"].numpy()[:, 0], d["wh"].numpy()[:, 1]).astype(np.float64)
    hits, valid = O.pck_counters(pred, gt, mask, [pck_thr], np.stack([nb, nb], 1))
    ahits, avalid = O.pck_counters(pred, gt, mask, [t / auc_steps for t in range(auc_steps)], np.full((case.B, 2), auc_nor))
    dd = pred - gt.astype(np.float64)
    epe = np.sqrt(dd[..., 0] * dd[..., 0] + dd[..., 1] * dd[..., 1]).astype(np.float32)
    fix = np.where(mask, np.rint(epe.astype(np.float64) * 1048576.0), 0).sum(0)
    return np.concatenate([hits[0], valid, ahits.reshape(-1), avalid, mask.sum(0), fix]).astype(np.int64)


def check_decode(case, orc, d, r, what):
    """idx bit-exact, coordinates at the suite's tolerances, maxvals exact."""
    assert np.array_equal(r["idx"].cpu().numpy(), orc["idx"]), f"{case.name} {what}: argmax"
    hk = r["hm_kpts"].cpu().numpy()
    assert_coords_close(hk[..., :2], orc["hm"], what=f"{case.name} {what}: heatmap coordinates")
    assert np.array_equal(hk[..., 2], orc["maxval"].reshape(hk.shape[:2]), equal_nan=True), f"{case.name} {what}: maxvals"
    kp = r["kpts"].cpu().numpy()
    assert_coords_close(kp[..., :2], orc["img"], what=f"{case.name} {what}: image coordinates",
                        mag=xform_magnitude(d["c"].numpy(), d["s"].numpy()))
    assert np.array_equal(kp[..., 2], hk[..., 2], equal_nan=True)


def check_sums(case, orc, sums, what):
    sums = np.asarray(sums, np.float64)
    want = orc["sums"]
    for i in (0, 1):
        assert abs(sums[i] - want[i]) <= 1e-5 * abs(want[i]) + 1e-300, f"{case.name} {what}: sum {i} {sums[i]} vs {want[i]}"
    assert sums[2] == want[2] and sums[3] == want[3], f"{case.name} {what}: N_pos / numel {sums[2:]} vs {want[2:]}"


def check_loss(case, orc, got, what, scale=1.0, reduction="mean"):
    want = float(orc["loss"]) * (orc["sums"][3] if reduction == "sum" else 1.0) * scale
    assert abs(float(got) - want) <= 1e-5 * abs(want), f"{case.name} {what}: loss {got} vs {want}"


def run_case(case, d, monkeypatch, env=None, off=None):
    """Every entry point of K1 on the case's inputs under `env` (default: the case's own switches).  Returns the
    outputs and the launch records."""
    env = case.env if env is None else env
    off = case.off if off is None else off
    set_env(monkeypatch, env)
    dv = d["dev"]
    hm = dv["hm"]
    if off:                                              # base address = 4 mod 16: element copies instead of TMA
        e = 4 // hm.element_size()
        buf = torch.empty(hm.numel() + 16, dtype=hm.dtype, device=DEV)
        hm = buf[e:e + hm.numel()].view(hm.shape)
        hm.copy_(dv["hm"])
        assert hm.data_ptr() % 16 == 4
    ref = REF[case.refine]
    udp = case.refine == "DARK_UDP"
    out, recs = {}, {}
    if case.loss is None:
        r = ops.decode_heatmap(hm, L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, dv["c"], dv["s"], hm_flip=dv["hf"], use_udp=udp,
                               overlap_previous=case.overlap)
        recs["decode"] = last_launch()
        out["decode"] = {k: v.clone() for k, v in r.items()}
        if case.auc is not None or not case.flip:
            steps = case.auc if case.auc is not None else 20
            cnt = torch.zeros((steps + 5) * case.K, dtype=torch.int64, device=DEV)
            r = ops.decode_heatmap_pck(hm, L.MASK_NEG1, ref, dv["c"], dv["s"], dv["gt"], dv["mask"], dv["wh"], cnt,
                                       auc_steps=steps, overlap_previous=case.overlap)
            recs["pck"] = last_launch()
            out["pck"] = dict(r, counters=cnt.clone(), steps=steps)
        return out, recs
    render = dict(loss_mode=LOSS[case.loss], image_size=d["img"], sigma=d["sigma"], unbiased=True)
    r = ops.decode_heatmap(hm, L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, dv["c"], dv["s"], hm_flip=dv["hf"], use_udp=udp,
                           render=render, joints=dv["j"], vis=dv["v"], overlap_previous=case.overlap)
    recs["partials"] = last_launch()
    out["partials"] = {k: v.clone() for k, v in r.items()}
    for red, scale in (("mean", 1.0), ("sum", 0.37)):
        r = ops.fused_render_loss_decode(hm, L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, dv["c"], dv["s"], render, dv["j"], dv["v"],
                                         hm_flip=dv["hf"], use_udp=udp, want_partials=True, reduction=red, loss_scale=scale,
                                         overlap_previous=case.overlap)
        recs["fused_" + red] = last_launch()
        out["fused_" + red] = {k: v.clone() for k, v in r.items()}
    if case.refine in ("DARK", "SIGN") and not case.overlap:
        step = fused.FusedHeatmapStep(image_size=d["img"], sigma=d["sigma"], balance=case.loss == "bal",
                                      post_process="unbiased" if case.refine == "DARK" else "default",
                                      loss_type="joints_mse" if case.loss == "mse" else "distance", loss_weight=1.0)
        acc = torch.full((1,), ACC0, dtype=torch.float32, device=DEV)
        bs = fused.BoundFusedStep(step, hm, dv["j"], dv["v"], dv["c"], dv["s"], hm_flip=dv["hf"], spare_sms=5,
                                  accumulate_into=acc)
        bs.launch()
        recs["bound"] = last_launch()
        out["bound"] = dict(hm_kpts=bs.hm_preds.clone(), kpts=bs.preds.clone(), idx=bs.idx.clone(), weight=bs.weight.clone(),
                            sums=bs.sums.clone(), acc=acc.clone())
    torch.cuda.synchronize()
    return out, recs


def _np(t):
    return t.cpu().numpy()


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_k1_configuration(case, monkeypatch):
    d = inputs(case)
    n = case.B * case.K
    if case.refine == "DARK_UDP" and case.rec[0] == 2:
        pytest.fail("the CTA-per-plane kernel has no UDP decode: such a case belongs in test_cta_kernel_refuses_udp")
    out, recs = run_case(case, d, monkeypatch)
    # ---- a. the launch record of every entry point -------------------------------------------------------------------
    for what, got in recs.items():
        spare = 5 if what == "bound" else 0
        rec = tuple(got[k] for k in RECORD)
        want = case.rec
        if what == "decode" and case.auc is not None:
            # the expected record is that of the counters launch; the same decode without counters keeps every team
            p = recs["pck"]
            assert got["path"] == 1 and (p["path"] == 2 or got["nteams"] >= p["nteams"]), (case.name, got, p)
            if case.K == 64:                          # the squeeze case: counters cost teams
                assert got["nteams"] > p["nteams"], (case.name, got, p)
        elif what == "pck" and case.auc is None:
            # 20 AUC steps of counters: the policy may drop teams, the rest of the geometry stays
            assert rec[:5] + rec[6:] == want[:5] + want[6:] and rec[5] <= want[5], (case.name, what, got)
        else:
            assert rec == want, f"{case.name} {what}: launch record {dict(zip(RECORD, rec))}, expected {dict(zip(RECORD, want))}"
        assert got["dtype"] == DCODE[case.dt] and got["flip"] == int(case.flip), (case.name, what, got)
        assert got["loss"] == int(case.loss is not None) and got["counters"] == int(what == "pck"), (case.name, what, got)
        assert got["use_tma"] == int(not case.off), (case.name, what, got)
        if got["path"] == 2:
            assert got["ctas"] == n and got["stagger_ns"] == 0, (case.name, what, got)
        else:
            assert got["ctas"] == min(n, sm_count() - spare), (case.name, what, got)
            stagger = int(case.env["LHN_STAGGER_NS"]) if "LHN_STAGGER_NS" in case.env else \
                (600 if n >= 8 * got["nteams"] * sm_count() else 0)
            assert got["stagger_ns"] == stagger, (case.name, what, got)
    first = next(iter(recs.values()))
    print(f"\nK1 case {case.name:40s} -> " + " ".join(f"{k}={first[k]}" for k in
                                                         ("path", "dtype", "flip", "loss", "counters", "wc", "twc", "ks",
                                                          "team_warps", "nteams", "stages", "sweeper_tables", "use_tma",
                                                          "ctas", "stagger_ns")) +
          (f"  [pck: nteams={recs['pck']['nteams']} path={recs['pck']['path']}]" if "pck" in recs else ""))
    # ---- c. against the oracle ---------------------------------------------------------------------------------------
    orc = oracle(case, d)
    for what, r in out.items():
        check_decode(case, orc, d, r, what)
        if case.loss is not None:
            assert np.array_equal(_np(r["weight"]), orc["weight"]), f"{case.name} {what}: target_weight"
    if "pck" in out:
        want = oracle_counters(case, d, _np(out["pck"]["kpts"]), out["pck"]["steps"])
        assert np.array_equal(_np(out["pck"]["counters"]), want), f"{case.name}: PCK / AUC / EPE counters"
        for k in ("idx", "hm_kpts", "kpts"):
            assert torch.equal(out["pck"][k], out["decode"][k]), f"{case.name}: decode_heatmap_pck {k} != decode_heatmap"
    if case.loss is not None:
        part = _np(out["partials"]["partials"])
        check_sums(case, orc, part.sum(0), "partials")
        for red, scale in (("mean", 1.0), ("sum", 0.37)):
            f = out["fused_" + red]
            check_sums(case, orc, _np(f["sums"]), "fused " + red)
            check_loss(case, orc, f["loss"].item(), "fused " + red, scale, red)
            assert torch.equal(f["partials"], out["partials"]["partials"]), f"{case.name} {red}: per-plane partials"
        for k in ("idx", "hm_kpts", "kpts", "weight"):
            assert torch.equal(out["fused_mean"][k], out["partials"][k]), f"{case.name}: fused {k} != decode_heatmap {k}"
            assert torch.equal(out["fused_sum"][k], out["partials"][k])
        assert torch.equal(out["fused_sum"]["sums"], out["fused_mean"]["sums"])
        if "bound" in out:
            b = out["bound"]
            check_sums(case, orc, _np(b["sums"]), "BoundFusedStep")
            lv = np.float32(np.float64(b["acc"].item()) - ACC0)
            check_loss(case, orc, lv, "BoundFusedStep accumulate_into")
            for k in ("idx", "hm_kpts", "kpts", "weight"):
                assert torch.equal(b[k], out["partials"][k]), f"{case.name}: BoundFusedStep {k}"
            if case.rec[0] == 1 and n <= sm_count() - 5:
                # fewer SMs, same teams per plane (one CTA per plane either way): the same sums, bit for bit
                assert torch.equal(b["sums"], out["fused_mean"]["sums"])
                assert b["acc"].item() == np.float32(ACC0) + np.float32(out["fused_mean"]["loss"].item())
    # ---- d. a second run is bit-identical -----------------------------------------------------------------------------
    out2, _ = run_case(case, d, monkeypatch)
    for what in out:
        for k, v in out[what].items():
            if isinstance(v, torch.Tensor):
                assert torch.equal(v, out2[what][k]), f"{case.name} {what}: {k} differs between two runs"
    # ---- d. against the default configuration on the same inputs ------------------------------------------------------
    if case.env or case.off:
        base, brecs = run_case(case, d, monkeypatch, env={}, off=False)
        same_order = set(case.env) <= SAME_ORDER
        if "LHN_NO_FAST" in case.env and case.W == 56:
            # Not the same order at 56x56: the compile-time sweep gives each of the first (32 * sweepers) // 14 * 14
            # threads one fixed column quad (14 quads per row), the run-time sweep strides all 32 * sweepers threads over
            # the plane.  Threads then hold other quads and a plane's squared errors are added in another order; the
            # argmax and coordinates stay bit-equal (checked above), the sums are checked against the oracle.
            same_order = False
        for what in out:
            for k in ("idx", "hm_kpts", "kpts", "weight"):
                if k in out[what]:
                    assert torch.equal(out[what][k], base[what][k]), f"{case.name} {what}: {k} != default configuration"
            if "counters" in out[what]:
                assert torch.equal(out[what]["counters"], base[what]["counters"]), f"{case.name}: counters != default"
            if case.loss is None:
                continue
            for k in ("sums", "partials", "loss", "acc"):
                if k not in out[what]:
                    continue
                if same_order or (k == "partials" and recs[what]["path"] == brecs[what]["path"] and
                                  recs[what]["team_warps"] == brecs[what]["team_warps"] and
                                  not ("LHN_NO_FAST" in case.env and case.W == 56)):
                    # a plane's partials are summed by the sweeper warps of one team: the same kernel with the same team
                    # width adds them in the same order, whatever the number of teams
                    assert torch.equal(out[what][k], base[what][k]), f"{case.name} {what}: {k} != default configuration"
                else:
                    diff = float((out[what][k].double() - base[what][k].double()).abs().max())
                    print(f"  {case.name} {what}: {k} vs default (other team order / kernel): max |diff| {diff:.3e}")


@pytest.mark.parametrize("H", [64, 128])
def test_cta_kernel_refuses_udp(H, monkeypatch):
    """REFINE_DARK_UDP exists on the team kernel only: forced onto the CTA-per-plane kernel the call is refused (and
    records nothing), it is not decoded some other way."""
    set_env(monkeypatch, {"LHN_FORCE_CTA_KERNEL": "1"})
    hm, _ = synth.blob_heatmaps(2, 3, H, H, seed=5, device=DEV)
    c, s = synth.bbox_center_scale(2, seed=6, device=DEV)
    with pytest.raises(L.LhnError):
        ops.decode_heatmap(hm, L.MASK_NEG1, L.REFINE_DARK_UDP, L.XFORM_CENTER_SCALE, c, s, use_udp=True)
    assert last_launch()["path"] == 0
    j, v = synth.hand_joints(2, 3, (4 * H, 4 * H), seed=7, device=DEV)
    render = dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=(4 * H, 4 * H), sigma=2.0, unbiased=True)
    with pytest.raises(L.LhnError):
        ops.fused_render_loss_decode(hm, L.MASK_NEG1, L.REFINE_DARK_UDP, L.XFORM_CENTER_SCALE, c, s, render, j, v, use_udp=True)
    assert last_launch()["path"] == 0


# ---- e. plane counts at the edges of the grid ----------------------------------------------------------------------------
# (name, H, W, refinement, switches, expected (team_warps, stages, sweeper_tables) of the loss launch)
GEOMETRIES = [("2warp-4stage-f32-16-dark", 16, 16, "DARK", {}, (2, 4, 0)),
              ("4warp-sweeper-f32-64-sign", 64, 64, "SIGN", {"LHN_TEAM_POLICY": "0"}, (4, 2, 1)),
              ("4warp-4stage-sweeper-f32-32-sign", 32, 32, "SIGN", {"LHN_TEAM_POLICY": "0"}, (4, 4, 1)),
              ("8warp-sweeper-f32-96-sign", 96, 96, "SIGN", {}, (8, 2, 1))]


@pytest.mark.parametrize("geo", GEOMETRIES, ids=[g[0] for g in GEOMETRIES])
@pytest.mark.parametrize("K", [1, 7])
def test_k1_plane_counts_at_grid_edges(geo, K, monkeypatch):
    """Teams without a plane leave at once, and the last team of a CTA (one-launch loss, counters) counts the active
    teams itself: n_planes around 1, nteams, ctas, ctas * nteams and ctas * nteams * stages, taken from the geometry of
    the loss launch and from that of the counters launch (which may drop teams).  With K = 1 every count is hit exactly;
    with K = 7 each count is rounded up to the next whole sample (a multiple of 7 planes), which puts the last sample
    across the edge.  Each result against the oracle and against the same rows of one large batch; overlapped launches
    into rotating outputs as well."""
    name, H, W, refine, env, geom = geo
    set_env(monkeypatch, env)
    sms = sm_count()
    ref = REF[refine]
    # the geometry, from a first call that fills the grid
    probe, pcen = synth.blob_heatmaps(sms * 12 * 4 // K + 1, K, H, W, seed=1, device=DEV)
    pj, pv = synth.hand_joints(probe.shape[0], K, (4 * W, 4 * H), seed=2, device=DEV)
    pc, ps = synth.bbox_center_scale(probe.shape[0], seed=3, device=DEV)
    render = dict(loss_mode=L.LOSS_DISTANCE_BALANCE, image_size=(4 * W, 4 * H), sigma=_sigma(W), unbiased=True)
    ops.fused_render_loss_decode(probe, L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, pc, ps, render, pj, pv)
    g = last_launch()
    assert (g["path"], g["team_warps"], g["stages"], g["sweeper_tables"]) == (1,) + geom, g
    nt, st, ctas = g["nteams"], g["stages"], g["ctas"]
    assert ctas == sms
    pgt, pmask, pwh = synth.pck_inputs(pcen, seed=4, device=DEV)
    ops.decode_heatmap_pck(probe, L.MASK_NEG1, ref, pc, ps, pgt, pmask, pwh, torch.zeros(25 * K, dtype=torch.int64, device=DEV))
    gc = last_launch()
    assert gc["path"] == 1 and gc["counters"] == 1 and gc["ctas"] == sms, gc

    def edges(nt, st):
        return {1, 2, nt - 1, ctas - 1, ctas, ctas + 1, ctas * nt - 1, ctas * nt, ctas * nt + 1, ctas * nt * st + 1}

    counts = sorted(edges(nt, st) | edges(gc["nteams"], gc["stages"]))
    Bs = sorted({max(1, math.ceil(n / K)) for n in counts})
    Bmax = Bs[-1]
    hm, cen = synth.blob_heatmaps(Bmax, K, H, W, seed=11 + K, sigma=max(1.0, 2.0 * W / 64), margin=min(4.0, W / 8), zero_frac=0.02)
    j, v = synth.hand_joints(Bmax, K, (4 * W, 4 * H), seed=12, vis_prob=0.9, outside_frac=0.05)
    c, s = synth.bbox_center_scale(Bmax, seed=13)
    gt, mask, wh = synth.pck_inputs(cen, seed=14)
    dv = dict(hm=hm.to(DEV), j=j.to(DEV), v=v.to(DEV), c=c.to(DEV), s=s.to(DEV), gt=gt.to(DEV), mask=mask.to(DEV), wh=wh.to(DEV))
    # oracle, per plane, of the whole batch
    hm32 = hm.numpy()
    idx_ref = O.argmax_planes(hm32)[0]
    p0, mv, _ = O.max_preds(hm32, "neg1")
    with np.errstate(all="ignore"):
        want = O.refine_dark(p0, hm32, 11, False) if refine == "DARK" else O.refine_sign_guarded(p0, hm32)
    img = np.stack([O.transform_preds(want[i], c.numpy()[i], s.numpy()[i], [W, H])[:, :2] for i in range(Bmax)])
    tg, tw = O.render_targets(j.numpy(), v.numpy(), (4 * W, 4 * H), (W, H), _sigma(W), True)
    ell = (hm32.astype(np.float64) - tg.astype(np.float64)) ** 2 * tw.astype(np.float64)[..., None]
    pos = tg > 0.5
    per_plane = np.stack([(ell * pos).sum((2, 3)), (ell * ~pos).sum((2, 3)), pos.sum((2, 3)).astype(np.float64),
                          np.full((Bmax, K), float(H * W))], -1)
    # the same rows of one large batch
    big = ops.fused_render_loss_decode(dv["hm"], L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, dv["c"], dv["s"], render, dv["j"], dv["v"])
    big_dec = ops.decode_heatmap(dv["hm"], L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, dv["c"], dv["s"])
    for B in Bs:
        n = B * K
        what = f"{name} K={K} B={B} n_planes={n}"
        sl = {k: t[:B] for k, t in dv.items()}
        # one-launch loss
        r = ops.fused_render_loss_decode(sl["hm"], L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, sl["c"], sl["s"], render, sl["j"], sl["v"])
        rec = last_launch()
        assert (rec["path"], rec["team_warps"], rec["nteams"], rec["stages"], rec["sweeper_tables"]) == (1,) + geom[:1] + (nt,) + geom[1:], (what, rec)
        assert rec["ctas"] == min(n, sms), (what, rec)
        assert np.array_equal(_np(r["idx"]), idx_ref[:B]), what
        assert_coords_close(_np(r["hm_kpts"])[..., :2], want[:B], what=what)
        assert_coords_close(_np(r["kpts"])[..., :2], img[:B], what=what, mag=xform_magnitude(c.numpy()[:B], s.numpy()[:B]))
        assert np.array_equal(_np(r["hm_kpts"])[..., 2], mv[:B, :, 0]), what
        assert np.array_equal(_np(r["weight"]), tw[:B].reshape(B, K)), what
        for k in ("idx", "hm_kpts", "kpts", "weight"):
            assert torch.equal(r[k], big[k][:B]), f"{what}: {k} != the same rows of the large batch"
        ws = per_plane[:B].reshape(-1, 4).sum(0)
        sums = _np(r["sums"])
        assert np.all(np.abs(sums[:2] - ws[:2]) <= 1e-5 * np.abs(ws[:2]) + 1e-300) and np.array_equal(sums[2:], ws[2:]), (what, sums, ws)
        lw = float(O.distance_loss_from_sums(ws))
        assert abs(r["loss"].item() - lw) <= 1e-5 * abs(lw), (what, r["loss"].item(), lw)
        r2 = ops.fused_render_loss_decode(sl["hm"], L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, sl["c"], sl["s"], render, sl["j"], sl["v"])
        assert torch.equal(r2["sums"], r["sums"]) and torch.equal(r2["loss"], r["loss"]), f"{what}: one-launch loss not reproducible"
        # counters (their own geometry: the policy may drop teams for them)
        cnt = torch.zeros(25 * K, dtype=torch.int64, device=DEV)
        rp = ops.decode_heatmap_pck(sl["hm"], L.MASK_NEG1, ref, sl["c"], sl["s"], sl["gt"], sl["mask"], sl["wh"], cnt)
        prec = last_launch()
        assert prec["path"] == 1 and prec["counters"] == 1 and prec["ctas"] == min(n, sms), (what, prec)
        for k in ("idx", "hm_kpts", "kpts"):
            assert torch.equal(rp[k], big_dec[k][:B]), f"{what}: pck {k} != the same rows of the large batch"
        case = C_(name, "f32", B, K, H, W, False, None, refine, 20, env, False, False, None)
        want_cnt = oracle_counters(case, dict(gt=gt[:B], mask=mask[:B], wh=wh[:B]), _np(rp["kpts"]), 20)
        assert np.array_equal(_np(cnt), want_cnt), f"{what}: counters"
        # two back-to-back overlapped launches into rotating outputs: the first rows and the last rows of the batch
        outs = [dict(hm_kpts=torch.full((B, K, 3), -7.0, device=DEV), kpts=torch.full((B, K, 3), -7.0, device=DEV),
                     idx=torch.full((B, K), -7, dtype=torch.int32, device=DEV),
                     partials=torch.full((n, 4), -7.0, dtype=torch.float64, device=DEV),
                     weight=torch.full((B, K), -7.0, device=DEV)) for _ in range(2)]
        rows = [slice(0, B), slice(Bmax - B, Bmax)]
        for o, rw in zip(outs, rows):
            ops.decode_heatmap(dv["hm"][rw], L.MASK_NEG1, ref, L.XFORM_CENTER_SCALE, dv["c"][rw], dv["s"][rw], render=render,
                               joints=dv["j"][rw], vis=dv["v"][rw], out=o, overlap_previous=True)
        torch.cuda.synchronize()
        for o, rw in zip(outs, rows):
            for k in ("idx", "hm_kpts", "kpts", "weight"):
                assert torch.equal(o[k], big[k][rw]), f"{what}: overlapped launch, {k} != the same rows of the large batch"
            ps = _np(o["partials"]).reshape(B, K, 4)
            assert np.array_equal(ps[..., 2:], per_plane[rw][..., 2:]), f"{what}: overlapped launch, N_pos / numel"
            assert np.all(np.abs(ps[..., :2] - per_plane[rw][..., :2]) <= 1e-5 * np.abs(per_plane[rw][..., :2]) + 1e-300), what
