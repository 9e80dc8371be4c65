"""The tcgen05 convolution of csrc/tq_gemm.cu (`conv_igemm_kernel<BLOCK_N, MODE, RELU, KIND, CG>`) at every instance the
host can pick, on real data, against the exact integer conv and the fp32 epilogue one IEEE step at a time.

Which instance runs is decided by plan_conv / pick_variant / pick_box / pick_box_halo; `conv_plan` below restates that
rule.  The default instances are CV_64_M0, CV_64_M1 (resident weights), CV_64_M3 (resident weights, halo load),
CV_128_M0, CV_128_M4 (streamed weights, halo load) and CV_128_M4_PAIR (the same on CTA pairs), CV_I8_64 and CV_I8_128
(kind::i8 planes), each with RELU true and false: 16 kernels.  The packed halo (several small images per tile) is a
runtime sub-mode of the two M4 kernels.  CV_256_M0 (TQ_CONV_N256=1) and CV_64_M3_PAIR (TQ_CONV_PAIR3=1) are only
reached through their switches, which are read once per process, so they run in child processes; so does CV_128_M4
under TQ_CONV_PAIR=0, the only way it runs several tiles per CTA.  A halo tiling whose buffers do not fit shared memory
beside a two-stage ring falls back to the plan it would replace; cases on both sides of that edge are included.

The cases cross every instance with its edges: output maps around the tile box, 1-pixel maps, packed tiles with a
ragged last image group, odd M-tile counts on CTA pairs, maps on which every persistent CTA runs three or more tiles;
C in {8, 16, 24, 72, 136, 200} (multiples of 16 on the plane engine), Cout with partial 32-column chunks and partial
N tiles (Cout % 8 == 4 goes with the fp32-only output); 1x1 to 7x7 filters, stride 1 and 2, padding 0 to k/2 + 1;
kind::f16 with 1, 2 and 4 accumulator groups and kind::i8 with every plane count.  The epilogue rotates through
bias / BN / both / neither, residual, no activation / ReLU / ReLU6, the three term encodings, consumer bits 1..10 and
term budgets 0, 1, bits and bits + 2; every case runs fp32 + codes, codes only and fp32 only where codes are legal.

Data: unsigned activation codes in [0, 2^b] for b up to 10, or signed codes in [-1024, 1024], half zeros.  The weights
of a kind::f16 case are scaled so that conv_codes.plan_weight proves exactly the intended number of K chunks with the
largest amplitude that still proves it, and one output position holds an adversarial patch: for every chunk, the
channels of that chunk are set so that one output channel's partial sum equals the chunk's proven bound.  The plane
engine has a case per instance whose accumulator passes 2^30.

Reference: oracle.fused_emul.conv_exact (fp64 conv of integers, exact), then fl32(acc) * scale, + bias, fmaf BN
(tq_oracle.fma_channels), + residual, activation (fused_emul._act), and oracle.tr for the codes in the consumer's
encoding.  Everything is compared bit for bit.
"""
import collections
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import bits_equal
from test_encodings_host import emul_encode

pytestmark = pytest.mark.gpu

B200_SMS = 148
EXACT = 1 << 24
ENCS = ("hese", "binary", "booth")
EPILOGUES = ("plain", "bias", "bn", "bias+bn")
ACT_SEQ = (False, True, False, "relu6")                 # half the cases of a variant without activation
BITS = (9, 4, 10, 1, 7, 3, 8, 2, 6, 5)
ABITS = (10, 9, 4, 10, 1, 7, 9, 2, 6, 3, 8, 5)         # unsigned activation codes in [0, 2^b]


def _cdiv(a, b):
    return -(-a // b)


# ---- the host rule, restated ------------------------------------------------------------------------------------

ConvCase = collections.namedtuple(
    "ConvCase", "N H W C Cout k stride pad kind groups planes signed act_max epi res act enc bits terms big seed")

VARIANTS = {(64, 0, 0, 1): "CV_64_M0", (64, 1, 0, 1): "CV_64_M1", (64, 3, 0, 1): "CV_64_M3",
            (64, 3, 0, 2): "CV_64_M3_PAIR", (128, 0, 0, 1): "CV_128_M0", (128, 4, 0, 1): "CV_128_M4",
            (128, 4, 0, 2): "CV_128_M4_PAIR", (256, 0, 0, 1): "CV_256_M0", (64, 0, 1, 1): "CV_I8_64",
            (128, 0, 1, 1): "CV_I8_128"}
DEFAULT_VARIANTS = ("CV_64_M0", "CV_64_M1", "CV_64_M3", "CV_128_M0", "CV_128_M4", "CV_128_M4_PAIR", "CV_I8_64",
                    "CV_I8_128")
ENV_VARIANTS = ("CV_256_M0", "CV_64_M3_PAIR")


def _out_hw(case):
    return ((case.H + 2 * case.pad - case.k) // case.stride + 1, (case.W + 2 * case.pad - case.k) // case.stride + 1)


def _pick_box(N, Ho, Wo, stride):
    """pick_box: the pixel box (wbox, hbox, nbox), product <= 128, with the fewest M tiles (then the widest)."""
    best, box = -1, None
    for wb in range(1, min(Wo, 128) + 1):
        if wb * stride > 256:
            break
        hb = 1
        while hb <= Ho and wb * hb <= 128:
            if hb * stride > 256:
                break
            nb = max(1, min(128 // (wb * hb), N)) if (wb == Wo and hb == Ho) else 1
            tiles = _cdiv(Wo, wb) * _cdiv(Ho, hb) * _cdiv(N, nb)
            if best < 0 or tiles < best or (tiles == best and wb > box[0]):
                best, box = tiles, (wb, hb, nb)
            hb += 1
    return box, best


def _pick_box_halo(N, Ho, Wo, R, S):
    """pick_box_halo: one image per tile, rows laid out wbox + S - 1 pixels apart inside 128 accumulator rows; fewest
    tiles, then the smallest halo."""
    best, best_halo, box = -1, 0, None
    for wb in range(1, Wo + 1):
        hw = wb + S - 1
        if hw > 128:
            break
        hb = min(128 // hw, Ho)
        if hb < 1 or hb + R - 1 > 256:
            continue
        tiles = _cdiv(Wo, wb) * _cdiv(Ho, hb) * N
        halo = hw * (hb + R - 1)
        if best < 0 or tiles < best or (tiles == best and halo < best_halo):
            best, best_halo, box = tiles, halo, (wb, hb, 1)
    return box, best


SMEM_BUDGET, MAX_STAGES, A_BYTES, EPI_F32, EPI_CODES = 227 * 1024, 8, 128 * 128, 16384, 8192
CODE_TABLE = ((2 << 10) * 2 + 15) & ~15                 # the 10-bit code table every conv plan reserves


def _smem_fits(block_n, prog_taps, a_tx, packed_tail, pair, f32, codes):
    """plan_smem: whether the ring keeps two stages beside the resident weights / halo buffers and the epilogue
    staging (f32: an fp32 tile is written or a residual read; codes: a code tile is written)."""
    b_bytes = block_n * 128
    up = lambda x: (x + 1023) & ~1023                                              # noqa: E731
    stage = A_BYTES + (0 if prog_taps else b_bytes)
    if a_tx:
        stage = up(a_tx)
    ring_off = prog_taps * (b_bytes // 2 if pair else b_bytes)
    if a_tx and not prog_taps:
        ring_off = (3 if pair else 2) * up(a_tx + packed_tail)
        stage = b_bytes
    fixed = ring_off + 4 * ((EPI_F32 if f32 else 0) + (EPI_CODES if codes else 0)) + CODE_TABLE + 2048
    return min((SMEM_BUDGET - fixed) // stage, MAX_STAGES) >= 2


def conv_plan(case, sms=B200_SMS, n256=False, pair3=False, pair=True, f32=True, codes=False):
    """What tq_conv2d_codes_fused_enc / tq_conv2d_planes_i8_enc launch for this case: the variant, the kernel instance
    (BLOCK_N, MODE, RELU, KIND, CG), the box, the tile counts, the accumulator groups and the persistent grid.
    n256 / pair3 / pair: the switches TQ_CONV_N256=1, TQ_CONV_PAIR3=1, TQ_CONV_PAIR=0 (pair=False).  f32 / codes: the
    epilogue staging of the launch (default: the fp32-only launch; a residual needs the fp32 tile too)."""
    f32 = f32 or case.res
    Ho, Wo = _out_hw(case)
    N, H, W, C, Cout, R, S, s, p = case.N, case.H, case.W, case.C, case.Cout, case.k, case.k, case.stride, case.pad
    kind = case.kind
    kc = _cdiv(C, 128 if kind else 64)
    n_groups = case.planes[0] + case.planes[1] - 1 if kind else case.groups
    box, m_tiles = _pick_box(N, Ho, Wo, s)
    block_n = 64 if Cout <= 64 else (256 if n256 and kind == 0 and case.groups == 1 and Cout % 256 == 0 else 128)
    n_tiles = _cdiv(Cout, block_n)
    half = sms // 2

    def pairs_ok(m):
        return (m + 1) // 2 * n_tiles >= half

    prog = kind == 0 and n_groups == 1 and Cout <= 64 and R * S * kc <= 12
    halo = cg2 = packed = False
    if prog and kc == 1 and s == 1 and R * S > 1:
        hbox, hm = _pick_box_halo(N, Ho, Wo, R, S)
        if hbox is not None and hm * 100 <= m_tiles * 116:
            c2 = pair3 and pair and Cout % 16 == 0 and pairs_ok(hm)
            if _smem_fits(block_n, R * S, (hbox[0] + S - 1) * (hbox[1] + R - 1) * 128, 0, c2, f32, codes):
                box, m_tiles, halo, cg2 = hbox, hm, True, c2
    if (kind == 0 and not prog and not halo and block_n == 128 and s == 1 and R == 3 and S == 3 and p == 1 and N >= 2
            and 2 * (W + 1) * (H + 1) <= 128):
        nb = min(128 // ((W + 1) * (H + 1)), N)
        c2 = pair and pairs_ok(_cdiv(N, nb))
        if _smem_fits(block_n, 0, nb * (W + 1) * (H + 1) * 128, ((R - 1) * (W + 1) + S) * 128, c2, f32, codes):
            box, m_tiles, halo, packed, cg2 = (W, H, nb), _cdiv(N, nb), True, True, c2
    if kind == 0 and not prog and not halo and block_n == 128 and s == 1 and R * S > 1:
        hbox, hm = _pick_box_halo(N, Ho, Wo, R, S)
        if hbox is not None and hm * 100 <= m_tiles * 116:
            c2 = pair and pairs_ok(hm)
            if _smem_fits(block_n, 0, (hbox[0] + S - 1) * (hbox[1] + R - 1) * 128, 0, c2, f32, codes):
                box, m_tiles, halo, cg2 = hbox, hm, True, c2
    if prog and kc != 1:                       # resident weights take one channel block per tap: back to streaming
        prog = halo = cg2 = False
    if kind:
        mode = 0
    elif prog:
        mode = 3 if halo else 1
    else:
        mode = 4 if halo else 0
    cg = 2 if cg2 else 1
    variant = VARIANTS[(block_n, mode, kind, cg)]
    acc_cols = n_groups * block_n
    acc_stages = 3 if 3 * acc_cols <= 512 else (2 if 2 * acc_cols <= 512 else 1)
    if cg == 2:
        supers = (m_tiles + 1) // 2 * n_tiles
        grid = 2 * min(supers, half)
        per_cta = _cdiv(supers, grid // 2)
    else:
        grid = min(m_tiles * n_tiles, sms)
        per_cta = _cdiv(m_tiles * n_tiles, grid)
    return {"variant": variant, "instance": (block_n, mode, bool(case.act), kind, cg), "box": box, "m_tiles": m_tiles,
            "n_tiles": n_tiles, "n_groups": n_groups, "packed": packed, "grid": grid, "tiles_per_cta": per_cta,
            "acc_stages": acc_stages, "kc_blocks": kc, "out": (Ho, Wo)}


# ---- the cases ---------------------------------------------------------------------------------------------------

# (N, H, W, C, Cout, k, stride, pad, groups (kind::f16) or (planes_a, planes_w) (kind::i8)), per intended variant
SPECS = {
    "CV_64_M1": [
        (1, 1, 1, 8, 4, 1, 1, 0, 1), (2, 9, 13, 16, 12, 1, 1, 0, 1), (3, 11, 12, 24, 40, 1, 1, 0, 1),
        (1, 17, 17, 8, 16, 3, 2, 1, 1), (2, 15, 16, 24, 64, 3, 2, 2, 1), (1, 12, 12, 16, 40, 2, 2, 0, 1),
        (1, 3, 3, 8, 4, 3, 2, 0, 1), (1, 130, 1, 16, 48, 1, 1, 0, 1), (1, 1, 300, 8, 40, 1, 1, 0, 1),
        (4, 5, 5, 16, 40, 3, 1, 1, 1), (2, 16, 8, 64, 16, 1, 2, 1, 1), (1, 9, 9, 48, 64, 2, 2, 1, 1),
        (4, 120, 128, 8, 16, 1, 1, 0, 1)],
    "CV_64_M3": [
        (1, 3, 3, 16, 12, 3, 1, 0, 1), (1, 1, 1, 8, 4, 3, 1, 1, 1), (2, 14, 14, 8, 40, 3, 1, 1, 1),
        (1, 16, 14, 24, 16, 3, 1, 1, 1), (1, 17, 14, 16, 64, 3, 1, 1, 1), (1, 15, 14, 8, 12, 3, 1, 1, 1),
        (2, 30, 31, 64, 64, 2, 1, 0, 1), (1, 20, 33, 32, 40, 3, 1, 1, 1), (1, 12, 12, 16, 12, 3, 1, 2, 1),
        (1, 10, 126, 8, 4, 3, 1, 0, 1), (2, 9, 9, 48, 16, 2, 1, 1, 1), (1, 2, 2, 24, 48, 2, 1, 0, 1),
        (230, 14, 14, 8, 16, 3, 1, 1, 1),
        # a 3-row halo of 128 pixels beside nine resident weight tiles fits the codes-only staging alone: MODE 3 for the
        # codes-only launch, MODE 1 for the other two
        (1, 3, 128, 64, 64, 3, 1, 0, 1)],
    "CV_64_M0": [
        (1, 9, 9, 8, 12, 5, 1, 2, 1), (2, 7, 7, 16, 40, 5, 2, 3, 1), (1, 7, 7, 8, 4, 7, 1, 0, 1),
        (1, 13, 13, 16, 16, 7, 2, 3, 1), (1, 11, 11, 72, 40, 3, 1, 1, 1), (2, 9, 9, 72, 12, 3, 1, 1, 2),
        (1, 10, 10, 72, 64, 1, 1, 0, 1), (2, 5, 7, 136, 40, 1, 1, 0, 1), (1, 9, 9, 200, 64, 3, 1, 1, 4),
        (1, 6, 6, 200, 12, 3, 2, 1, 2), (1, 8, 8, 136, 4, 2, 1, 0, 1), (2, 11, 11, 72, 48, 1, 1, 0, 2),
        (1, 5, 9, 200, 16, 1, 2, 0, 4), (4, 120, 128, 8, 16, 5, 1, 2, 1)],
    "CV_128_M0": [
        (1, 1, 1, 8, 68, 1, 1, 0, 1), (2, 9, 13, 72, 132, 1, 1, 0, 2), (1, 7, 7, 200, 260, 1, 1, 0, 4),
        (1, 15, 15, 16, 196, 3, 2, 1, 1), (2, 14, 14, 200, 72, 3, 2, 1, 4), (1, 11, 11, 24, 72, 5, 2, 3, 1),
        (1, 14, 14, 8, 128, 7, 2, 3, 1), (2, 8, 8, 136, 136, 2, 2, 0, 1), (4, 5, 5, 16, 200, 3, 1, 0, 1),
        (1, 9, 9, 72, 132, 3, 2, 1, 2), (1, 3, 3, 200, 256, 3, 2, 1, 2), (1, 2, 130, 16, 68, 1, 1, 0, 1),
        (1, 5, 259, 8, 132, 3, 2, 1, 1), (4, 120, 128, 8, 72, 1, 1, 0, 1),
        # 7x7 on maps about 128 pixels wide: the halo buffers do not fit beside the ring, the streaming plan stays
        (1, 2, 122, 8, 72, 7, 1, 3, 1), (1, 1, 120, 8, 196, 7, 1, 4, 1), (74, 2, 122, 8, 128, 7, 1, 3, 1)],
    "CV_128_M4": [
        (1, 3, 3, 16, 68, 3, 1, 0, 1), (1, 14, 14, 8, 132, 3, 1, 1, 1), (1, 16, 14, 24, 256, 3, 1, 1, 1),
        (1, 12, 12, 16, 68, 5, 1, 2, 1), (1, 2, 67, 8, 72, 7, 1, 3, 1), (1, 1, 43, 8, 196, 7, 1, 4, 1),
        (1, 9, 9, 72, 136, 2, 1, 0, 2), (1, 10, 10, 72, 128, 3, 1, 1, 2), (1, 14, 14, 200, 68, 3, 1, 1, 4),
        (2, 7, 7, 16, 72, 3, 1, 1, 1), (5, 7, 7, 200, 132, 3, 1, 1, 4), (3, 5, 6, 72, 128, 3, 1, 1, 2),
        (3, 1, 1, 24, 200, 3, 1, 1, 1), (1, 16, 14, 136, 260, 3, 1, 1, 1)],
    "CV_128_M4_PAIR": [
        (80, 14, 14, 8, 68, 3, 1, 1, 1), (147, 10, 10, 8, 72, 3, 1, 1, 1), (293, 7, 7, 8, 68, 3, 1, 1, 1),
        (365, 4, 4, 200, 136, 3, 1, 1, 4), (147, 7, 7, 72, 136, 3, 1, 1, 2), (37, 14, 14, 200, 196, 2, 1, 0, 4),
        (37, 12, 12, 16, 132, 5, 1, 2, 1), (74, 2, 67, 8, 128, 7, 1, 3, 1), (1568, 1, 1, 24, 260, 3, 1, 1, 1),
        (147, 9, 9, 72, 200, 3, 1, 1, 2), (444, 10, 10, 8, 72, 3, 1, 1, 1), (700, 7, 7, 16, 128, 3, 1, 1, 1)],
    "CV_I8_64": [
        (1, 1, 1, 16, 4, 1, 1, 0, (1, 1)), (2, 9, 11, 48, 40, 3, 1, 1, (2, 1)), (1, 7, 7, 16, 12, 7, 2, 3, (1, 2)),
        (1, 9, 9, 144, 64, 5, 1, 2, (2, 2)), (3, 14, 14, 16, 16, 2, 2, 0, (1, 1)), (1, 12, 12, 208, 48, 3, 2, 1, (1, 2)),
        (2, 10, 10, 32, 40, 3, 1, 2, (2, 2)), (1, 6, 9, 80, 64, 1, 1, 0, (2, 1)), (4, 120, 128, 16, 40, 1, 1, 0, (2, 2))],
    "CV_I8_128": [
        (1, 1, 1, 16, 68, 1, 1, 0, (1, 1)), (2, 9, 13, 144, 132, 3, 1, 1, (2, 2)), (1, 10, 10, 48, 260, 5, 1, 2, (2, 1)),
        (1, 14, 14, 16, 196, 7, 2, 3, (1, 2)), (2, 8, 8, 208, 72, 2, 1, 0, (1, 1)), (2, 7, 7, 32, 128, 3, 1, 1, (1, 2)),
        (1, 11, 11, 80, 136, 3, 2, 2, (2, 2)), (3, 5, 5, 16, 200, 3, 1, 1, (2, 1)), (4, 120, 128, 16, 68, 1, 1, 0, (1, 1))],
}
# cases with a fixed activation (so that each RELU value of an instance meets them); `big`: the plane engine at the int32
# limit, K * act_max * wgt_max just below 2^31 and one output channel's patch at that bound
EXTRA_SPECS = {
    "CV_64_M0": [((1, 13, 11, 72, 40, 1, 1, 0, 2), False, False), ((1, 13, 11, 200, 16, 1, 1, 0, 4), True, False)],
    "CV_128_M0": [((1, 9, 15, 200, 136, 1, 1, 0, 4), True, False)],
    "CV_128_M4": [((1, 15, 14, 16, 132, 3, 1, 1, 1), False, False), ((1, 15, 14, 200, 68, 3, 1, 1, 4), True, False)],
    "CV_128_M4_PAIR": [((37, 15, 14, 200, 136, 3, 1, 1, 4), False, False)],
    "CV_I8_64": [((1, 1, 1, 1008, 16, 1, 1, 0, (2, 2)), False, True), ((1, 3, 3, 1040, 8, 3, 1, 0, (2, 1)), "relu6", True),
                 ((1, 13, 11, 16, 40, 1, 1, 0, (1, 1)), False, False), ((1, 13, 11, 48, 12, 1, 1, 0, (2, 1)), True, False)],
    "CV_I8_128": [((1, 5, 5, 512, 72, 3, 1, 0, (1, 2)), False, True), ((2, 3, 3, 112, 136, 3, 1, 0, (2, 2)), True, True),
                  ((1, 13, 11, 16, 68, 1, 1, 0, (1, 1)), False, False), ((2, 13, 11, 32, 136, 3, 1, 1, (1, 2)), True, False)],
}
# the instances only a switch reaches (run in child processes), and single CTAs where pairs are the default
ENV_SPECS = {
    "CV_256_M0": [(2, 9, 9, 16, 256, 3, 1, 1, 1), (1, 7, 7, 72, 512, 1, 1, 0, 1), (3, 7, 7, 24, 256, 3, 1, 1, 1),
                  (1, 6, 6, 200, 256, 3, 2, 1, 1)],
    "CV_64_M3_PAIR": [(80, 14, 14, 8, 48, 3, 1, 1, 1), (147, 10, 10, 16, 16, 3, 1, 1, 1),
                      (150, 12, 12, 24, 64, 3, 1, 2, 1), (460, 14, 14, 8, 32, 3, 1, 1, 1)],
    "CV_128_M4": [(444, 10, 10, 8, 72, 3, 1, 1, 1), (700, 7, 7, 16, 128, 3, 1, 1, 1), (300, 9, 9, 72, 132, 3, 1, 1, 2),
                  (450, 7, 7, 200, 68, 3, 1, 1, 4)],
}
ENV_OF = {"CV_256_M0": {"TQ_CONV_N256": "1"}, "CV_64_M3_PAIR": {"TQ_CONV_PAIR3": "1"}, "CV_128_M4": {"TQ_CONV_PAIR": "0"}}
PLAN_KW = {"CV_256_M0": {"n256": True}, "CV_64_M3_PAIR": {"pair3": True}, "CV_128_M4": {"pair": False}}


def _make_cases(specs, extra_specs=None, seed0=5000, counters=None):
    counters = collections.defaultdict(int) if counters is None else counters
    cases = []

    def add(spec, act=None, big=False, plan_kw=None):
        N, H, W, C, Cout, k, s, p, gp = spec
        kind = 1 if isinstance(gp, tuple) else 0
        variant = conv_plan(ConvCase(N, H, W, C, Cout, k, s, p, kind, 1 if kind else gp, gp if kind else (1, 1), False,
                                     1, "", False, False, "", 1, 0, False, 0), **(plan_kw or {}))["variant"]
        j = counters[variant]
        counters[variant] += 1
        a = ACT_SEQ[j % 4] if act is None else act
        inst = (variant, bool(a))
        c = counters[inst]
        counters[inst] += 1
        cc = counters[inst + ("codes",)]
        if Cout % 8 == 0:
            counters[inst + ("codes",)] += 1
        bits = BITS[cc % len(BITS)]
        if kind:
            pa, pw = gp
            signed = j % 2 == 1
            act_max = 1024 if pa == 2 else 127
        else:
            signed = j % 3 == 2
            act_max = 1024 if signed else 2 ** (ABITS[j % len(ABITS)] if gp == 1 else (10, 9)[j % 2])
        cases.append(ConvCase(N, H, W, C, Cout, k, s, p, kind, 1 if kind else gp, gp if kind else (1, 1), signed,
                              act_max, EPILOGUES[c % 4], (c + c // 4) % 2 == 1, a, ENCS[cc % 3], bits,
                              (0, 1, bits, bits + 2)[(cc + cc // 4) % 4], big, seed0 + len(cases)))

    for variant, lst in specs.items():
        for spec in lst:
            add(spec, plan_kw=PLAN_KW.get(variant) if extra_specs is None else None)
        for spec, act, big in (extra_specs or {}).get(variant, ()):
            add(spec, act, big=big)
    return cases


CASES = _make_cases(SPECS, EXTRA_SPECS)
ENV_CASES = {v: _make_cases({v: lst}, seed0=9000 + 100 * i) for i, (v, lst) in enumerate(ENV_SPECS.items())}
# every variant also meets both RELU values among the switch cases
for _v, _cs in ENV_CASES.items():
    ENV_CASES[_v] = [c._replace(act=(False, True)[i % 2] if i < 2 else c.act) for i, c in enumerate(_cs)]


def _case_id(c):
    g = f"g{c.groups}" if c.kind == 0 else f"p{c.planes[0]}{c.planes[1]}"
    return (f"{'i8' if c.kind else 'f16'}-N{c.N}-{c.H}x{c.W}-C{c.C}-Co{c.Cout}-k{c.k}s{c.stride}p{c.pad}-{g}-"
            f"{'s' if c.signed else 'u'}{c.act_max}-{c.epi}{'-res' if c.res else ''}-{c.act or 'noact'}-"
            f"{c.enc}-b{c.bits}t{c.terms}{'-big' if c.big else ''}")


# ---- data and reference ----------------------------------------------------------------------------------------

def _l1(w):
    """(pos, neg) [Cout, C/64 blocks]: sums of the positive / negative weight codes per output channel and 64-channel
    block over all taps (tq_conv_weight_l1)."""
    RS, Cout, C = w.shape
    kcb = _cdiv(C, 64)
    wp = np.zeros((RS, Cout, kcb * 64), dtype=np.int64)
    wp[:, :, :C] = w
    pos = np.maximum(wp, 0).reshape(RS, Cout, kcb, 64).sum(axis=(0, 3))
    neg = np.maximum(-wp, 0).reshape(RS, Cout, kcb, 64).sum(axis=(0, 3))
    return pos, neg


def chunk_bounds(w, act_max, signed, groups):
    """Per K chunk: act_max * max over output channels of the chunk's worst partial sum, and that channel."""
    pos, neg = _l1(w)
    Cout, kcb = pos.shape
    p = pos.reshape(Cout, groups, kcb // groups).sum(2)
    n = neg.reshape(Cout, groups, kcb // groups).sum(2)
    worst = p + n if signed else np.maximum(p, n)
    return [float(act_max) * float(worst[:, g].max()) for g in range(groups)], worst.argmax(0), p, n


def proven_groups(w, act_max, signed):
    """plan_weight's choice: the fewest groups whose every chunk is proven below 2^24 (None: the plane engine)."""
    Cout, C = w.shape[1], w.shape[2]
    kcb = _cdiv(C, 64)
    block_n = 64 if Cout <= 64 else 128
    for g in (1, 2, 4, 8):
        if kcb % g or g * block_n > (512 if block_n == 128 else 256):
            continue
        if max(chunk_bounds(w, act_max, signed, g)[0]) < EXACT:
            return g
    return None


def _interior(case):
    """An output position of the last image whose whole receptive field lies inside the image, else the centre one;
    returns (oh, ow, valid taps (r, s))."""
    Ho, Wo = _out_hw(case)

    def first(n_out, n_in):
        for o in range(n_out):
            if o * case.stride - case.pad >= 0 and o * case.stride - case.pad + case.k <= n_in:
                return o
        return n_out // 2

    oh, ow = first(Ho, case.H), first(Wo, case.W)
    taps = [(r, s) for r in range(case.k) for s in range(case.k)
            if 0 <= oh * case.stride - case.pad + r < case.H and 0 <= ow * case.stride - case.pad + s < case.W]
    return oh, ow, taps


def _codes(rng, shape, act_max, signed):
    lo = -act_max if signed else 0
    a = rng.integers(lo, act_max + 1, shape)
    a = np.where(rng.random(shape) < 0.5, 0, a).reshape(-1)
    ends = np.array([act_max, 1, act_max - 1] + ([-act_max, -1] if signed else [0]))
    pick = rng.choice(a.size, size=min(a.size, 3 * ends.size), replace=False)
    a[pick] = np.resize(ends, pick.size)
    return a.reshape(shape).astype(np.int64)


def _f16_weights(rng, case, taps_ok):
    """Integer weights [k*k, Cout, C] of the largest amplitude for which plan_weight proves exactly case.groups chunks
    (taps that never meet the image at the patch position are zero, so that the patch can reach every bound)."""
    RS = case.k * case.k
    u = rng.uniform(-1.0, 1.0, (RS, case.Cout, case.C))
    mask = np.zeros(RS, dtype=bool)
    for r, s in taps_ok:
        mask[r * case.k + s] = True
    u[~mask] = 0.0

    def at(A):
        return np.rint(u * A).astype(np.int64)

    def fits(A):
        g = proven_groups(at(A), case.act_max, case.signed)
        return g is not None and g <= case.groups

    lo, hi = 1, 2047
    if fits(hi):
        lo = hi
    else:
        while hi - lo > 1:                     # the bound grows with the amplitude: largest amplitude that still fits
            mid = (lo + hi) // 2
            lo, hi = (mid, hi) if fits(mid) else (lo, mid)
    w = at(lo)
    got = proven_groups(w, case.act_max, case.signed)
    assert got == case.groups, (_case_id(case), "weights cannot be drawn for", case.groups, "groups: got", got, lo)
    return w


def _setup(case):
    """Device operands of the case, its plan and its CPU reference (fp32 output, codes, facts about the patch)."""
    from oracle import fused_emul
    from oracle import tq_oracle as O
    from term_quantization_b200 import conv_codes
    rng = np.random.default_rng(case.seed)
    Ho, Wo = _out_hw(case)
    RS = case.k * case.k
    act = _codes(rng, (case.N, case.H, case.W, case.C), case.act_max, case.signed)
    oh, ow, taps = _interior(case)
    info = {}
    if case.kind == 0:
        w = _f16_weights(rng, case, taps)
        bounds, co_star, p, n = chunk_bounds(w, case.act_max, case.signed, case.groups)
        kcpg = _cdiv(case.C, 64) // case.groups
        for g in range(case.groups):                 # adversarial patch: chunk g's channels drive co_star[g] to its bound
            co = int(co_star[g])
            lo_c, hi_c = g * kcpg * 64, min(case.C, (g + 1) * kcpg * 64)
            for r, s in taps:
                wv = w[r * case.k + s, co, lo_c:hi_c]
                if case.signed:
                    v = np.sign(wv) * case.act_max
                elif p[co, g] >= n[co, g]:
                    v = (wv > 0) * case.act_max
                else:
                    v = (wv < 0) * case.act_max
                act[case.N - 1, oh * case.stride - case.pad + r, ow * case.stride - case.pad + s, lo_c:hi_c] = v
        info.update(bounds=bounds, co_star=co_star, kcpg=kcpg)
    else:
        pa, pw = case.planes
        K = case.C * RS
        wmax = 2047 if pw == 2 else 127
        wmax = min(wmax, (2 ** 31 - 1) // (K * case.act_max))
        assert wmax >= (128 if pw == 2 else 1), (_case_id(case), "no weight range for", case.planes)
        w = rng.integers(-wmax, wmax + 1, (RS, case.Cout, case.C))
        w.reshape(-1)[rng.choice(w.size, size=min(w.size, 4), replace=False)] = [wmax, -wmax, wmax, -wmax][:min(w.size, 4)]
        if case.big:                                 # output channel 0 at +-wmax, the patch at +-act_max against it
            w[:, 0, :] = rng.choice(np.array([-wmax, wmax]), (RS, case.C))
            for r, s in taps:
                act[case.N - 1, oh * case.stride - case.pad + r, ow * case.stride - case.pad + s, :] = (
                    np.sign(w[r * case.k + s, 0, :]) * case.act_max)
            if not case.signed:                      # unsigned codes: both operands of channel 0 positive
                act = np.abs(act)
                w[:, 0, :] = np.abs(w[:, 0, :])
        info.update(wmax=wmax)
    acc = fused_emul.conv_exact(act, w, (case.k, case.k), case.stride, case.pad)
    info["acc"] = acc
    info["patch"] = (case.N - 1, oh, ow, taps)
    M = 8.0
    q = float(np.quantile(np.abs(acc), 0.99)) if acc.size > 1 else float(np.abs(acc).max())
    scale = float(np.float32(M / max(q, 1.0)))
    bias = (rng.standard_normal(case.Cout) * M / 4).astype(np.float32) if "bias" in case.epi else None
    bn = None
    if "bn" in case.epi:
        bn = ((rng.uniform(0.5, 1.5, case.Cout) * rng.choice([-1.0, 1.0], case.Cout)).astype(np.float32),
              (rng.standard_normal(case.Cout) * M / 4).astype(np.float32))
    res = (rng.standard_normal((case.N, Ho, Wo, case.Cout)) * M / 4).astype(np.float32) if case.res else None
    # the fp32 chain, one IEEE step at a time
    t = acc.astype(np.float32) * np.float32(scale)
    if bias is not None:
        t = t + bias
    if bn is not None:
        t = O.fma_channels(t, bn[0], bn[1])
    if res is not None:
        t = t + res
    t = np.ascontiguousarray(fused_emul._act(t, case.act), dtype=np.float32)
    sf = float(np.float32(M / 2 ** case.bits * (0.37, 1.0, 2.9)[case.seed % 3]))
    quant = (sf, case.bits, case.terms, case.enc)
    c_ref = emul_encode(t, quant) if case.Cout % 8 == 0 else None
    wt = torch.from_numpy(w.astype(np.float16)).cuda()
    if case.kind == 0:
        plan = conv_codes.plan_weight(wt, case.act_max, signed_act=case.signed, engine="f16")
    else:
        plan = conv_codes.plan_weight(wt, case.act_max, signed_act=case.signed, engine="i8")
    dev = {"act": torch.from_numpy(act.astype(np.float16)).cuda(), "wgt": wt, "plan": plan, "scale": scale,
           "bias": None if bias is None else torch.from_numpy(bias).cuda(),
           "bn": None if bn is None else tuple(torch.from_numpy(v).cuda() for v in bn),
           "res": None if res is None else torch.from_numpy(res).cuda()}
    return dev, quant, t, c_ref, info


def _run(case, dev, want_f32=True, next_quant=None):
    from term_quantization_b200 import conv_codes
    return conv_codes.conv2d_codes_fused(dev["act"], dev["wgt"], (case.k, case.k), case.stride, case.pad, dev["scale"],
                                         bias=dev["bias"], bn=dev["bn"], residual=dev["res"], relu=case.act,
                                         want_f32=want_f32, next_quant=next_quant, plan=dev["plan"])


def _check_f32(got, want, what):
    got = got.cpu().numpy()
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not bits_equal(got, want):
        bad = np.flatnonzero(got.view(np.uint32).ravel() != want.view(np.uint32).ravel())
        i = int(bad[0])
        raise AssertionError(f"{what}: {bad.size} of {got.size} fp32 outputs differ, first at "
                             f"{tuple(int(v) for v in np.unravel_index(i, got.shape))}: "
                             f"got {got.ravel()[i]!r} want {want.ravel()[i]!r}")


def _check_codes(got, want, what):
    got = got.cpu().numpy().astype(np.int32)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got, want):
        bad = np.flatnonzero(got.ravel() != want.ravel())
        i = int(bad[0])
        raise AssertionError(f"{what}: {bad.size} of {got.size} codes differ, first at "
                             f"{tuple(int(v) for v in np.unravel_index(i, got.shape))}: "
                             f"got {got.ravel()[i]} want {want.ravel()[i]}")


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


def check_case(case, plan_kw=None):
    """Runs one case (fp32 + codes, codes only, fp32 only) against its reference; returns the plan it predicts."""
    dev, quant, t_ref, c_ref, info = _setup(case)
    plan = conv_plan(case, _sms(), **(plan_kw or {}))
    what = (_case_id(case), plan["variant"], "box", plan["box"], "groups", plan["n_groups"])
    wp = dev["plan"]
    if case.kind == 0:
        assert wp.engine == "f16" and wp.groups == case.groups, (what, wp)
        bounds = info["bounds"]
        assert wp.bound == max(bounds) and wp.bound < EXACT, (what, wp, bounds)
        if case.groups > 1:
            assert max(chunk_bounds(dev["wgt"].cpu().numpy().astype(np.int64), case.act_max, case.signed,
                                    case.groups // 2)[0]) >= EXACT, what
        # every chunk's real partial sum reaches its proven bound at the patch (the chunk -> block mapping is exercised)
        n, oh, ow, taps = info["patch"]
        a = dev["act"].cpu().numpy().astype(np.int64)
        w = dev["wgt"].cpu().numpy().astype(np.int64)
        for g, b in enumerate(bounds):
            co = int(info["co_star"][g])
            lo_c, hi_c = g * info["kcpg"] * 64, min(case.C, (g + 1) * info["kcpg"] * 64)
            part = sum(int(a[n, oh * case.stride - case.pad + r, ow * case.stride - case.pad + s, lo_c:hi_c]
                           @ w[r * case.k + s, co, lo_c:hi_c]) for r, s in taps)
            assert abs(part) >= 0.9 * b, (what, "chunk", g, part, b)
    else:
        assert wp.engine == "i8" and (2 if case.act_max > 127 else 1, wp.planes_w) == case.planes, (what, wp)
        if case.big:
            assert float(np.abs(info["acc"]).max()) > 2.0 ** 30, (what, float(np.abs(info["acc"]).max()))
    if c_ref is not None:
        out, codes = _run(case, dev, True, quant)
        _check_f32(out, t_ref, what)
        _check_codes(codes, c_ref, what)
        none, codes2 = _run(case, dev, False, quant)
        assert none is None
        _check_codes(codes2, c_ref, what + ("codes only",))
    out3, none = _run(case, dev, True, None)
    assert none is None
    _check_f32(out3, t_ref, what + ("fp32 only",))
    return plan


@pytest.mark.parametrize("case", CASES, ids=[f"c{i:03d}-{_case_id(c)}" for i, c in enumerate(CASES)])
def test_conv_against_exact_reference(case):
    check_case(case)


# ---- which instances the cases reach -----------------------------------------------------------------------------

def _edges(cases, plan_kw=None):
    """Per instance: the set of edge labels its cases meet."""
    out = collections.defaultdict(set)
    for c in cases:
        p = conv_plan(c, **(plan_kw or {}))
        key = (p["variant"], bool(c.act))
        Ho, Wo = p["out"]
        wb, hb, nb = p["box"]
        e = out[key]
        e.update({("epi", c.epi), ("res", c.res), ("act", c.act), ("k", c.k), ("stride", c.stride),
                  ("groups", p["n_groups"]), ("C", c.C), ("Cout%8", c.Cout % 8)})
        if c.kind:
            e.add(("planes", c.planes))
        if c.Cout % 8 == 0:
            e.update({("enc", c.enc), ("out", "codes")})
        e.add(("pad", "0" if c.pad == 0 else ("max" if c.pad == c.k // 2 + 1 else "mid")))
        if Ho == Wo == 1:
            e.add(("map", "1px"))
        if Wo % wb or Ho % hb:
            e.add(("tile", "partial"))
        if p["m_tiles"] > 1 and Wo % wb == 0 and Ho % hb == 0 and not p["packed"]:
            e.add(("tile", "full"))
        if p["tiles_per_cta"] >= 3:
            e.add(("tiles_per_cta", ">=3"))
        if c.Cout % 32:
            e.add(("chunk", "partial"))
        if p["packed"]:
            e.add(("packed", c.N % nb != 0))
        if VARIANTS.get((p["instance"][0], p["instance"][1], 0, 2)) == p["variant"] and p["m_tiles"] % 2:
            e.add(("pair", "odd"))
    return out


def test_every_default_instance_is_checked():
    """By the restated host rule the cases reach all 16 default instances, the packed halo single and paired, and
    every instance meets every epilogue entry and its tile, channel, filter and accumulator edges."""
    inst = collections.Counter((conv_plan(c)["variant"], bool(c.act)) for c in CASES)
    want = {(v, r) for v in DEFAULT_VARIANTS for r in (False, True)}
    print(f"default instances checked: {len(set(inst) & want)}/16", dict(sorted(inst.items())))
    assert set(inst) == want
    packed = {conv_plan(c)["variant"] for c in CASES if conv_plan(c)["packed"]}
    assert packed == {"CV_128_M4", "CV_128_M4_PAIR"}, packed
    edges = _edges(CASES)
    for (v, relu), e in sorted(edges.items()):
        need = {("epi", x) for x in EPILOGUES} | {("res", False), ("res", True), ("out", "codes"), ("Cout%8", 4),
                                                 ("tile", "partial"), ("chunk", "partial")}
        need |= {("act", "relu6"), ("act", True)} if relu else {("act", False)}
        need |= {("enc", x) for x in ENCS}
        if v.startswith("CV_I8"):
            pass
        else:
            need |= {("groups", 1)}
            if v in ("CV_64_M0", "CV_128_M0", "CV_128_M4", "CV_128_M4_PAIR"):
                need |= {("groups", 2), ("groups", 4)}
        assert need <= e, (v, relu, sorted(need - e))
    for v in DEFAULT_VARIANTS:
        e = edges[(v, False)] | edges[(v, True)]
        need = {("stride", 1), ("pad", "0"), ("map", "1px"), ("tile", "full")}
        if v not in ("CV_64_M3", "CV_128_M4", "CV_128_M4_PAIR"):
            need |= {("stride", 2), ("k", 1), ("pad", "max")}
        if v in ("CV_64_M0", "CV_128_M0", "CV_128_M4", "CV_128_M4_PAIR", "CV_I8_64", "CV_I8_128"):
            need |= {("k", 5), ("k", 7)}
        if v in ("CV_64_M1", "CV_64_M3", "CV_64_M0", "CV_128_M0", "CV_128_M4_PAIR", "CV_I8_64", "CV_I8_128"):
            need |= {("tiles_per_cta", ">=3")}
        if v.startswith("CV_I8"):
            need |= {("planes", pp) for pp in ((1, 1), (1, 2), (2, 1), (2, 2))}
        if v == "CV_128_M4_PAIR":
            need |= {("pair", "odd"), ("packed", True)}
        if v == "CV_128_M4":
            need |= {("packed", True)}
        assert need <= e, (v, sorted(need - e))
    chans = {c.C for c in CASES if c.kind == 0}
    assert {8, 16, 24, 72, 136, 200} <= chans
    couts = {c.Cout for c in CASES}
    assert {4, 12, 40, 68, 132, 196, 260} <= couts
    for v in ("CV_I8_64", "CV_I8_128"):
        assert any(c.big and conv_plan(c)["variant"] == v and c.act for c in CASES), v
        assert any(c.big and conv_plan(c)["variant"] == v and not c.act for c in CASES), v


def test_env_only_cases_reach_their_instances():
    """Under its switch every case of ENV_CASES reaches the instance it stands for, both RELU values of each: 4/4
    instances only a switch selects (and the single-CTA M4 kernel with several tiles per CTA)."""
    reached = set()
    for v, cases in ENV_CASES.items():
        for c in cases:
            p = conv_plan(c, **PLAN_KW[v])
            assert p["variant"] == v, (v, _case_id(c), p["variant"])
            assert conv_plan(c)["variant"] != v, (v, _case_id(c), "reached without the switch")
            reached.add((v, bool(c.act)))
    env_only = {(v, r) for v in ENV_VARIANTS for r in (False, True)}
    print(f"env-only instances checked: {len(reached & env_only)}/4")
    assert env_only <= reached
    assert any(conv_plan(c, pair=False)["tiles_per_cta"] >= 3 for c in ENV_CASES["CV_128_M4"])


_NAME = re.compile(r"conv_igemm_kernel\s*<\s*(\d+)\s*,\s*(\d+)\s*,\s*(true|false)\s*,\s*(\d+)\s*,\s*(\d+)\s*,"
                   r"\s*(true|false)\s*>")
_MANGLED = re.compile(r"conv_igemm_kernelILi(\d+)ELi(\d+)ELb([01])ELi(\d+)ELi(\d+)ELb([01])E")


def _launched(prof):
    """conv_igemm_kernel instances (BLOCK_N, MODE, RELU, KIND, CG) launched inside the profiler, with multiplicity."""
    got = collections.Counter()
    for ev in prof.key_averages():
        m = _NAME.search(ev.key) or _MANGLED.search(ev.key)
        if m:
            assert m[6] in ("false", "0"), ev.key              # no loss epilogue here
            got[(int(m[1]), int(m[2]), m[3] in ("true", "1"), int(m[4]), int(m[5]))] += ev.count
    return got


def profiled_instances(cases, plan_kw=None):
    """Runs the fp32-only launch of each case under torch.profiler: (launched Counter, predicted Counter)."""
    from torch.profiler import ProfilerActivity, profile
    ops = [(conv_plan(c, _sms(), **(plan_kw or {}))["instance"], c, _setup(c)) for c in cases]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _, c, (dev, _, _, _, _) in ops:
            _run(c, dev, True, None)
        torch.cuda.synchronize()
    for _, c, (dev, _, t_ref, _, _) in ops:
        _check_f32(_run(c, dev, True, None)[0], t_ref, _case_id(c))
    return _launched(prof), collections.Counter(inst for inst, _, _ in ops)


def default_reps():
    """One case of every default instance, and a packed one of each M4 kernel."""
    reps = {}
    for c in CASES:
        p = conv_plan(c)
        reps.setdefault((p["variant"], bool(c.act), p["packed"]), c)
    return reps


# The profiler runs in a child process, never in the pytest process: with a session of this file in the pytest process,
# the profiler test of test_dw_kernels_gpu.py that runs after it in the same process was seen to miss the first two
# kernels it launched.
_CHILD = r"""
import json, sys
sys.path[:0] = [{tests!r}, {root!r}]
import torch
import test_conv_kernels_gpu as T
v = {variant!r}
if v is None:
    cases, kw = list(T.default_reps().values()), {{}}
else:
    cases, kw = T.ENV_CASES[v], T.PLAN_KW[v]
    for c in cases:
        T.check_case(c, kw)
got, want = T.profiled_instances(cases, kw)
print("LAUNCHED", json.dumps(sorted([list(k), n] for k, n in got.items())))
print("PREDICTED", json.dumps(sorted([list(k), n] for k, n in want.items())))
assert got == want, (got, want)
"""


def _run_child(variant, env_extra):
    here = os.path.dirname(os.path.abspath(__file__))
    env = dict(os.environ, **env_extra)
    code = _CHILD.format(tests=here, root=os.path.dirname(here), variant=variant)
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    print(r.stdout[-4000:])
    assert r.returncode == 0, r.stderr[-6000:]
    assert "LAUNCHED" in r.stdout


def test_restated_host_rule_matches_the_launched_kernels():
    """One case of every default instance (and a packed one of each M4 kernel) runs under torch.profiler in a child
    process: the conv_igemm_kernel names launched must be exactly the instances conv_plan predicts, once each."""
    assert len({(v, r) for v, r, _ in default_reps()}) == 16
    _run_child(None, {})


@pytest.mark.parametrize("variant", sorted(ENV_CASES))
def test_switch_only_instances_in_a_child_process(variant):
    """TQ_CONV_N256=1 (BLOCK_N = 256), TQ_CONV_PAIR3=1 (resident-weight halo on CTA pairs) and TQ_CONV_PAIR=0 (single
    CTAs, several tiles per CTA on the streamed-weight halo kernel) are read once per process: their cases run in a
    child, exact against the reference and with the launched kernels matching conv_plan under the switch."""
    _run_child(variant, ENV_OF[variant])


# ---- tq_conv2d_codes_f16, the plain public entry point -----------------------------------------------------------

def test_conv2d_codes_f16_entry_point_equals_conv2d_codes():
    """tq_conv2d_codes_f16 (acc * scale + bias, fp32 out) on one case of each kind::f16 instance: equal to
    conv2d_codes and to the reference bit for bit."""
    from term_quantization_b200 import _lib, conv_codes
    reps = {}
    for c in CASES:
        p = conv_plan(c)
        if c.kind == 0 and not c.act:
            reps.setdefault(p["variant"], c._replace(epi="bias", res=False))
    assert set(reps) == {"CV_64_M0", "CV_64_M1", "CV_64_M3", "CV_128_M0", "CV_128_M4", "CV_128_M4_PAIR"}
    for v, c in sorted(reps.items()):
        dev, _, t_ref, _, _ = _setup(c)
        Ho, Wo = _out_hw(c)
        out = torch.full((c.N, Ho, Wo, c.Cout), float("nan"), device="cuda")
        with torch.cuda.device(out.device):
            rc = _lib.lib().tq_conv2d_codes_f16(dev["act"].data_ptr(), dev["wgt"].data_ptr(), dev["bias"].data_ptr(),
                                                out.data_ptr(), c.N, c.H, c.W, c.C, c.Cout, c.k, c.k, c.stride, c.pad,
                                                float(dev["scale"]), int(dev["plan"].groups),
                                                torch.cuda.current_stream().cuda_stream)
        _lib.check(rc)
        ref = conv_codes.conv2d_codes(dev["act"], dev["wgt"], dev["bias"], (c.k, c.k), c.stride, c.pad, dev["scale"],
                                      plan=dev["plan"])
        _check_f32(out, t_ref, (v, _case_id(c)))
        _check_f32(ref, t_ref, (v, _case_id(c), "conv2d_codes"))


# ---- refusals before any launch ----------------------------------------------------------------------------------

def test_refusals_leave_the_outputs_untouched():
    """Every argument the host refuses is refused before a kernel runs: the return code names it, the launch count
    does not move and sentinel-filled outputs stay as they were."""
    from term_quantization_b200 import _lib
    L = _lib.lib()
    stream = torch.cuda.current_stream().cuda_stream
    N, H, W = 1, 6, 6
    buf_a = torch.zeros(N * H * W * 1024 + 64, dtype=torch.float16, device="cuda")
    buf_w = torch.zeros(9 * 512 * 512 + 64, dtype=torch.float16, device="cuda")
    vec = torch.ones(1024 + 16, device="cuda")
    out = torch.full((N * H * W * 512 + 64,), 1234.5, device="cuda")
    codes = torch.full((N * H * W * 512 + 64,), 77.0, dtype=torch.float16, device="cuda")
    o0, c0 = out.clone(), codes.clone()
    P = lambda t, off=0: t.data_ptr() + off                                       # noqa: E731

    def f16(C, Cout, k=3, groups=1, out_p=None, codes_p=None, bias=None, bn_a=None, bn_b=None, sf=0.01, act=None):
        return L.tq_conv2d_codes_fused_enc(act or P(buf_a), P(buf_w), out_p, codes_p, bias, bn_a, bn_b, None, N, H, W, C,
                                           Cout, k, k, 1, 1, 1.0, 0, sf, 8, 3, _lib.ENC_HESE, groups, stream)

    def i8(C, Cout, act_max, wgt_max, pa=2, pw=2, k=3):
        return L.tq_conv2d_planes_i8_enc(P(buf_a), P(buf_w), pa, pw, P(out), None, None, None, None, None, N, H, W, C,
                                         Cout, k, k, 1, 1, 1.0, 0, 1.0, 1, 0, _lib.ENC_HESE, act_max, wgt_max, stream)

    I, U = _lib.TQ_ERR_INVALID, _lib.TQ_ERR_UNSUPPORTED
    cases = [
        ("C % 8", f16(12, 16, out_p=P(out)), U),
        ("Cout % 4", f16(16, 6, out_p=P(out)), U),
        ("codes with Cout % 8", f16(16, 12, out_p=P(out), codes_p=P(codes)), U),
        ("groups do not divide the channel blocks", f16(192, 64, groups=2, out_p=P(out)), I),
        ("groups x BLOCK_N 64 beyond tensor memory", f16(512, 64, groups=8, out_p=P(out)), U),
        ("groups x BLOCK_N 128 beyond tensor memory", f16(512, 128, groups=8, out_p=P(out)), U),
        ("bn_a without bn_b", f16(16, 16, out_p=P(out), bn_a=P(vec)), I),
        ("bn_b without bn_a", f16(16, 16, out_p=P(out), bn_b=P(vec)), I),
        ("misaligned output", f16(16, 16, out_p=P(out, 4)), I),
        ("misaligned codes", f16(16, 16, out_p=P(out), codes_p=P(codes, 2)), I),
        ("misaligned activations", f16(16, 16, out_p=P(out), act=P(buf_a, 8)), I),
        ("misaligned bias", f16(16, 16, out_p=P(out), bias=P(vec, 4)), I),
        ("i8 int32 bound", i8(128, 16, 1024, 2047), U),                       # 9 * 128 * 1024 * 2047 >= 2^31
        ("i8 int32 bound, one plane", i8(133152, 16, 127, 127, 1, 1, 1), U),            # 133152 * 127^2 >= 2^31
        ("next_sf below 2^-30 with codes", f16(16, 16, out_p=P(out), codes_p=P(codes), sf=2.0 ** -31), U),
        ("next_sf above 2^30 with codes", f16(16, 16, out_p=P(out), codes_p=P(codes), sf=2.0 ** 31), U),
    ]
    n0 = _lib.launch_count()
    torch.cuda.synchronize()
    for what, rc, want in cases:
        assert rc == want, (what, rc, L.tq_last_error())
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0
    assert torch.equal(out, o0) and torch.equal(codes, c0)
