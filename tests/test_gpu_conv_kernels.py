"""The tensor-core convolution kernels — conv_igemm_kernel (fprop and dgrad, csrc/conv_igemm.cu), conv_c64_kernel
(csrc/conv_c64.cu) and conv_wgrad_kernel with its two reduce kernels (csrc/conv_wgrad.cu) — element by element against
an fp64 reference, at every tile geometry their host planners select.

Geometry.  igemm_plan / c64_plan / wgrad_plan mirror the host planning (pick_block_n and the small-M narrowing,
conv_tile_geometry, halo / pair / double-M / epilogue groups / weight residency / stages / shared memory / cluster count,
add_tma, fold_il; the row-streaming eligibility; the weight-gradient split plan and reduce choice).  An unmarked test
asserts that the GPU matrix reaches every geometry class at 148 SMs; on the GPU the mirror is checked against what
launched: kernel name, grid and per-block shared memory from a torch.profiler trace, and the split count through
b2_conv_wgrad_workspace (splits x count x 4 bytes).

Reference.  One fp64 forward per case, on the bf16 operands the kernel reads (the packed weights themselves): every
launch is a sum of "parts", each a kxk tap loop of matrix products over gathered operand pixels — stride, input
sub-lattice (in_mul / in_off), tap offsets (custom pad), output placement (out_mul / out_off), fold phases and
row_offset are explicit indexing.  dgrad is torch.autograd.grad of the forward of the layer it differentiates (the
weights unpacked from the dgrad packing, taps flipped), wgrad the autograd weight gradient of the layer's forward; no
transposed-convolution formula is written by hand.  The epilogue rounds where the kernel rounds: bf16(act(acc + bias
[+ addend])) and, with add_after_act, bf16(bf16(act(acc + bias)) + addend) (conv_igemm.cu, the add_after_act branch of
the drain), the inner rounding straight-through.  Statistics: exact fp64 sums of the kernel's stored bf16 output over
the pixels the launch owns.

Bounds (per element, from the kernel's arithmetic).  An fp32 chain of n additions of terms t_i is within
n * u * sum|t_i| of the exact sum for a unit roundoff u; a full ulp per step (u = 2^-23) also covers truncating
accumulation inside the MMA.  conv_igemm / conv_c64: the accumulator is a chain of K / 16 MMAs (K = taps x 64-channel
blocks x 64, zero-filled past the channel count), then + bias and + addend: eps = (K / 16 + 3) * 2^-23 and
S = conv(|x|, |w|) + |bias| + |addend|; the bf16 store adds one ulp of the result, add_after_act one more of the inner
value.  wgrad: each split is a chain of pixels-per-split / 16 MMAs (twice that where the row-pair / fold modes feed one
accumulator from two MMA streams), the reduce adds the splits in fp32 (and dW in accumulate mode): eps = (n_acc + 1) *
2^-23 with n_acc = 4 * chunks per split (x 2) + splits + accumulate, S = the weight gradient of |x| against |dy|, fp32
output (no bf16 ulp).  Statistics: fp32 partials over at most 32 rows (8 / 4 / 2 / 1 tiles of N = 32 / 64 / 128 / 256,
conv_igemm.cu fold_stats), fp64 from there on: |err| <= 33 * 2^-23 * sum |v| (sum) and 33 * 2^-23 * sum v^2 (sum of
squares) of the stored values v.

Mutants.  Every GPU case also evaluates each applicable wrong reference and asserts that some checked element moves by
>= 10x its bound: padding wrapping into the neighbouring row / image, the halo-seam tap reading one pixel to the left,
the partial last 64-channel block dropped, the addend before the activation, clipped pixels counted in the statistics,
unflipped dgrad taps, transposed wgrad taps, a 64-pixel chunk dropped at a split boundary (on inputs whose
split-boundary chunks are scaled by 16), fold phases (a, b) swapped, and a non-zero dY row below the image in row-pair
mode.  The unmarked test runs the same machinery at small shapes on the CPU.
"""
import json
import math
import os
import re
import subprocess
import sys
import tempfile

import pytest
import torch

from test_gpu_bn_kernels import filled_workspace  # noqa: F401  (fixture)
from test_gpu_gate_kernels import _bits, _r, _st, _worst, ulp_bf16

SMS_B200 = 148
TILE_M = 128
SMEM_OPTIN = 232448
U23 = 2.0 ** -23
MUTANT_MARGIN = 10.0


def _env(name, dflt):
    """env_switch (host_util.cu): unset -> the default, otherwise atoi"""
    v = os.environ.get(name)
    if v is None:
        return dflt
    try:
        return int(v.strip() or 0)
    except ValueError:
        return 0


# ----------------------------------------------------------------------------------------------------------
# §1 the host planners, mirrored
# ----------------------------------------------------------------------------------------------------------
def _pow2ceil(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def tile_geometry(n, h, w, tile_pix):
    """conv_tile_geometry: (Wb, Hb, Nb, tw, th, tn)"""
    wb = min(_pow2ceil(w), tile_pix)
    rows = tile_pix // wb
    hb = min(_pow2ceil(h), rows)
    nb = rows // hb
    return wb, hb, nb, -(-w // wb), -(-h // hb), -(-n // nb)


def pick_block_n(cout, wide_rows):
    forced = _env("B200SEG_BLOCK_N", 0)
    if forced > 0 and cout % forced == 0 and not (forced > 128 and wide_rows):
        return forced
    for bn in (256, 128, 64, 32):
        if cout % bn == 0 and not (bn == 256 and wide_rows):
            return bn
    return 0


def c64_plan(a, sms):
    """conv_c64_try_launch: None when the layer goes to the generic kernel, else (stages, epi_groups, smem, grid)"""
    if _env("B200SEG_C64", 1) == 0:
        return None
    fold = a["fold"] == 1
    if fold and (a["k"] != 2 or a["c1"] != 0 or a["ldy"] != a["cout"] or _env("B200SEG_C64_FOLD", 1) == 0):
        return None
    if ((not fold and (a["k"] != 3 or a["fold"] != 0)) or a["cout"] != 64 or a["stride"] != 1 or a["out_mul"] != 1
            or a["in_mul"] != 1 or a["pad"] is not None or a["w"] % TILE_M or a["c0"] % 64 or a["c1"] % 64):
        return None
    if a["addend"] and (fold or a["add_after_act"]):
        return None
    cbt = (a["c0"] + a["c1"]) // 64
    if not 1 <= cbt <= 2 or _env("B200SEG_BLOCK_N", 0) != 0:
        return None
    rows_total = a["n"] * (a["w"] // TILE_M) * a["h"]
    if rows_total < 8 * sms or a["h"] < 4:
        return None
    tail = 320 + 16 + 64 * 4 + 192
    wres = (8 if fold else 9) * cbt * 8192
    epi = 2
    budget = SMEM_OPTIN - 1024 - tail - wres - 2 * TILE_M * 128
    if budget // 17408 < 3:
        epi, budget = 1, budget + TILE_M * 128
    stages = min(budget // 17408, 8)
    if stages < 2:
        return None
    return {"kernel": "conv_c64_kernel", "stages": stages, "epi_groups": epi, "grid": sms, "fold": int(fold),
            "smem": stages * 17408 + wres + epi * TILE_M * 128 + tail + 1024}


def igemm_plan(a, sms, max_pairs=None):
    """conv_igemm_launch (and the row-streaming kernel it tries first).  a: the launch's b2_conv_args as a dict."""
    c64 = c64_plan(a, sms)
    if c64 is not None:
        return c64
    max_pairs = sms // 2 if max_pairs is None else max_pairs
    k, fold, stride, cout = a["k"], a["fold"], a["stride"], a["cout"]
    p = {"kernel": None}
    bn = pick_block_n(cout, k == 3 and a["w"] >= TILE_M)
    wb, hb, nb, tw, th, tn = tile_geometry(a["n"], a["h"], a["w"], TILE_M)
    p.update(Wb=wb, Hb=hb, Nb=nb, tw=tw, th=th, tn=tn)
    taps = 16 if fold == 2 else k * k
    cbt = -(-a["c0"] // 64) + -(-a["c1"] // 64)
    m_tiles = tw * th * tn
    p["block_n0"] = bn
    if _env("B200SEG_BLOCK_N", 0) == 0 and _env("B200SEG_SMALL_M", 1) != 0:
        slots = sms // 2
        while bn > 64 and ((m_tiles * (4 if fold == 1 else 1) + 1) // 2) * (cout // bn) * 2 <= slots:
            bn //= 2
    n_tiles = cout // bn
    m_phase = m_tiles
    fold_il = int(fold == 1 and m_tiles % 2 == 0)
    if fold == 1:
        m_tiles *= 4
    halo = int(taps == 9 and stride == 1 and a["pad"] is None and hb == 1 and nb == 1 and wb == TILE_M)
    if halo:
        a_stage, b_stage, nk = -(-(TILE_M + 2) * 128 // 1024) * 1024, 3 * bn * 128, 3 * cbt
    else:
        a_stage, b_stage, nk = TILE_M * 128, bn * 128, taps * cbt
    ctile = TILE_M * bn * 2
    tail = 320 + 2 * 2 * 256 * 4 + 192
    dm = 0
    want = _env("B200SEG_DM", 2)
    if want and bn <= 128 and m_tiles >= _env("B200SEG_DM_MIN_TILES", 4 * sms) and not (fold == 1 and m_phase % 2):
        sb2 = 2 * a_stage + b_stage
        g2 = SMEM_OPTIN - 1024 - tail - 2 * ctile
        if g2 // sb2 >= 2 or (want == 2 and (g2 + ctile) // sb2 >= 2):
            dm = 1
    pair = 0
    want = _env("B200SEG_PAIR", 2)
    if want and m_tiles >= 2 and bn % 16 == 0 and (want >= 2 or bn == 256) and not (fold == 1 and m_phase % 2):
        pair, dm, b_stage = 1, 0, b_stage // 2
    stage_bytes = (2 if dm else 1) * a_stage + b_stage
    mma_clk = nk * (3 if halo else 1) * 4 * (bn // 2)
    epi_clk = 1750 + 36 * bn
    forced_g = _env("B200SEG_EPI_GROUPS", 0)
    epi = min(forced_g, 2) if forced_g > 0 else (2 if mma_clk * 5 < epi_clk * 6 else 1)
    if dm:
        epi = 2
    budget2 = SMEM_OPTIN - 1024 - tail - 2 * ctile
    if epi == 2 and budget2 // stage_bytes < 2:
        epi = 1
    if epi == 2 and pair and bn == 256 and forced_g == 0 and budget2 // stage_bytes < 4:
        epi = 1
    budget = SMEM_OPTIN - 1024 - tail - epi * ctile
    wres, wres_bytes = 0, 0
    wbytes = (4 if fold == 1 else 1) * nk * b_stage
    a_only = (2 if dm else 1) * a_stage
    if n_tiles == 1 and m_tiles >= 4 * sms and wbytes % 1024 == 0 and (budget - wbytes) // a_only >= 4:
        wres, wres_bytes, stage_bytes, budget = 1, wbytes, a_only, budget - wbytes
    stages = min(budget // stage_bytes, 12)
    if _env("B200SEG_MAX_STAGES", 0) >= 2:
        stages = min(stages, _env("B200SEG_MAX_STAGES", 0))
    assert stages >= 2, "tile configuration does not fit shared memory"
    csz = 2 if pair else 1
    clusters = sms // csz
    if pair:
        clusters = min(clusters, max_pairs)
    per_item = 2 if dm else csz
    total = -(-m_tiles // per_item) * n_tiles
    clusters = min(clusters, total)
    if clusters > n_tiles and total // clusters >= 16:
        clusters = (clusters // n_tiles) * n_tiles
    add_tma = int(bool(a["addend"]) and bn >= 64 and fold == 0 and a["out_mul"] == 1 and cout % 64 == 0)
    p.update(block_n=bn, n_tiles=n_tiles, m_tiles=m_tiles, m_tiles_phase=m_phase, fold_il=fold_il, halo=halo, dm=dm,
             pair=pair, epi_groups=epi, wres=wres, stages=stages, cbt=cbt, taps=taps, num_k_iters=nk,
             smem=stages * stage_bytes + epi * ctile + wres_bytes + tail + 1024, clusters=clusters, total=total,
             grid=clusters * csz, add_tma=add_tma, per_item=per_item,
             kernel=f"conv_igemm_kernel<{'true' if a['addend'] else 'false'}, {'true' if pair else 'false'}>")
    # a CTA meets more than one n-tile (and flushes its statistics when the slab changes) when the cluster count is not a
    # multiple of n_tiles and it has more than one item
    p["stats_flush"] = int(n_tiles > 1 and clusters % n_tiles != 0 and total > clusters)
    return p


def wgrad_plan(a, sms):
    """wgrad_plan (conv_wgrad.cu) + the reduce choice of b2_conv_wgrad"""
    k, xs = a["k"], a["x_stride"]
    cout, c0, c1 = a["cout"], a["c0"], a["c1"]
    wb, hb, nb, tw, th, tn = tile_geometry(a["n"], a["h"], a["w"], 64)
    num_chunks = tw * th * tn
    taps = k * k
    cbt = -(-c0 // 64) + -(-c1 // 64)
    pad_h = a["pad"][0] if a["pad"] is not None else (1 if k == 3 else 0)
    a_boxes = 1 if cout <= 64 else 2
    cpb = min(4 if k == 1 else 2, cbt)
    ncolb, gy = k * cpb, k
    rowpair = 0
    rp_ok = cout == 64 and xs == 1 and hb == 1 and nb == 1 and _env("B200SEG_WG_ROWPAIR", 1) != 0
    if rp_ok and k == 3 and pad_h == 1:
        rowpair, cpb = 2, 1
    elif rp_ok and k == 2:
        rowpair, cpb = 1, min(cbt, 2)
    if rowpair:
        ncolb, a_boxes, gy = rowpair * k * cpb, 2, 1
    fold = 0
    if a["fold"]:
        fold = 2 if cout == 64 else 1
        taps, rowpair, cpb = 16, 0, min(cbt, 2)
        ncolb, a_boxes, gy = (4 if fold == 1 else 3) * cpb, (2 if fold == 1 else 1), 4
    a_bytes = 4 * 8192 if fold == 1 else 2 * 8192
    gz = -(-cout // 128) * -(-cbt // cpb)
    base = gy * gz
    max_splits = (num_chunks + 7) // 8
    splits, best, s = 1, 0.0, 1
    while s <= max_splits and s * base <= 3 * sms + base:
        ctas = s * base
        eff = ctas / (-(-ctas // sms) * sms)
        if eff > best + 0.02:
            best, splits = eff, s
        s += 1
    cps = -(-num_chunks // splits)
    splits = -(-num_chunks // cps)
    count = cout * taps * (c0 + c1)
    xh = int(k == 3 and xs == 1 and a["pad"] is None and nb == 1 and wb >= 16 and (wb + 2) * hb * 128 <= 9 * 1024)
    nbox = rowpair if rowpair else cpb
    if fold:
        xh = int(nb == 1 and wb >= 16 and (wb + 2) * hb * 128 <= 9 * 1024)
        assert xh
    pair = int(_env("B200SEG_WG_PAIR", 1) != 0 and xh and (k == 3 or fold == 1) and not rowpair and fold != 2
               and cpb == 2 and cout % 256 == 0 and cbt % 2 == 0)
    b_stage = 9 * 1024 if pair else (nbox * 9 * 1024 if xh else ncolb * 8192)
    stages = min((200 * 1024) // (a_bytes + b_stage), 8)
    n4 = (count + 3) // 4
    return {"Wb": wb, "Hb": hb, "Nb": nb, "tw": tw, "th": th, "tn": tn, "num_chunks": num_chunks, "cpb": cpb,
            "rowpair": rowpair, "fold": fold, "xh": xh, "pair": pair, "splits": splits, "chunks_per_split": cps,
            "count": count, "grid": (gy * gz, splits), "stages": stages, "workspace": splits * count * 4,
            "smem": stages * (a_bytes + b_stage) + 256 + 1024,
            "kernel": f"conv_wgrad_kernel<{'true' if pair else 'false'}>",
            "reduce": "wgrad_reduce_wide_kernel" if n4 <= 16384 and splits >= 16 else "wgrad_reduce_kernel"}


# ----------------------------------------------------------------------------------------------------------
# the cases: b2_conv_args / b2_wgrad_args of one launch, as a dict
# ----------------------------------------------------------------------------------------------------------
def conv_case(name, kind, n, h, w, k, c0, cout, c1=0, stride=1, out_mul=1, out_off=(0, 0), in_mul=1, in_off=(0, 0),
              pad=None, fold=0, bias=True, addend=None, add_after_act=False, relu=True, stats=True, ld_x=0, ld_y=0,
              row_offset=0, rows_extra=0):
    """kind 'fprop' (wpk = the forward packing) or 'dgrad' (wpk = the dgrad packing, x0 = dY).  n, h, w: the conv
    grid (= the output grid of the launch before placement).  addend: None, 'add' or 'alias' (the output itself)."""
    return dict(name=name, kind=kind, n=n, h=h, w=w, k=k, c0=c0, c1=c1, cout=cout, stride=stride, out_mul=out_mul,
                out_off=out_off, in_mul=in_mul, in_off=in_off, pad=pad, fold=fold, bias=bias, addend=addend,
                add_after_act=add_after_act, relu=relu, stats=stats, ld_x=ld_x, ld_y=ld_y, row_offset=row_offset,
                rows_extra=rows_extra, ldy=cout + ld_y)


def wgrad_case(name, n, h, w, k, c0, cout, c1=0, x_stride=1, dy_mul=1, dy_off=(0, 0), pad=None, fold=False,
               accumulate=False, ld_dy=0):
    """n, h, w: the dY grid of the launch (the coarse grid with dy_mul / fold)"""
    return dict(name=name, kind="wgrad", n=n, h=h, w=w, k=k, c0=c0, c1=c1, cout=cout, x_stride=x_stride,
                dy_mul=dy_mul, dy_off=dy_off, pad=pad, fold=fold, accumulate=accumulate, ld_dy=ld_dy)


CONV_CASES = [
    # block_n and the small-M narrowing
    conv_case("bn256_3x3", "fprop", 4, 64, 64, 3, 64, 256),
    conv_case("smallm_1024", "fprop", 1, 16, 16, 3, 1024, 1024),
    conv_case("bn128_w64", "fprop", 4, 64, 64, 3, 64, 128, relu=False),
    conv_case("bn32_add_w32", "fprop", 2, 32, 32, 3, 64, 32, addend="add"),
    # tile shapes: halo row segments (two and three per row), multi-row, multi-image, clipping
    conv_case("halo_w256", "fprop", 2, 16, 256, 3, 64, 128),
    conv_case("halo_w384_2src", "fprop", 1, 12, 384, 3, 64, 128, c1=64),
    conv_case("w16", "fprop", 4, 16, 16, 3, 128, 64),
    conv_case("w8_multi_image", "fprop", 3, 8, 8, 3, 64, 128, bias=False),
    conv_case("img3x3_n7", "fprop", 7, 3, 3, 3, 64, 64),
    conv_case("clip_224", "fprop", 1, 224, 224, 3, 64, 128),
    conv_case("clip_20x28", "fprop", 2, 20, 28, 3, 64, 64),
    conv_case("clip_22x28_add", "fprop", 2, 22, 28, 3, 64, 128, addend="add"),
    # pair parity, single tile, epilogue groups, weight residency, statistics flush
    conv_case("pair_odd", "fprop", 3, 8, 16, 3, 64, 128),
    conv_case("single_tile", "fprop", 1, 8, 16, 3, 64, 128),
    conv_case("epi2_1x1", "fprop", 8, 32, 32, 1, 64, 128),
    conv_case("wres_3x3", "fprop", 5, 128, 128, 3, 64, 64),
    conv_case("stats_flush_192", "fprop", 2, 64, 64, 3, 64, 192),
    # addend: TMA, aliasing the output, after the activation, no ReLU
    conv_case("add_tma_1x1", "fprop", 2, 32, 64, 1, 128, 128, addend="add", relu=False),
    conv_case("add_alias_dgrad_1x1", "dgrad", 2, 32, 32, 1, 64, 128, addend="alias", bias=False, relu=False,
              stats=False),
    conv_case("add_after_act", "fprop", 2, 32, 128, 3, 64, 64, addend="add", add_after_act=True),
    # operands: two sources, row_offset, channel slices, partial channel blocks
    conv_case("dgrad_3x3_rowoff", "dgrad", 2, 32, 32, 3, 128, 64, row_offset=64, rows_extra=64, bias=False,
              relu=False, stats=False),
    conv_case("slices_ld", "fprop", 2, 16, 64, 3, 64, 64, ld_x=64, ld_y=64),
    conv_case("c0_32_stem", "fprop", 4, 32, 32, 1, 32, 64),
    conv_case("c0_152_stem", "fprop", 2, 32, 32, 1, 152, 64),
    # stride, placement, phases
    conv_case("stride2_3x3", "fprop", 2, 16, 16, 3, 64, 128, stride=2),
    conv_case("stride2_1x1", "fprop", 2, 16, 16, 1, 128, 64, stride=2, relu=False),
    conv_case("dgrad_2x2s2", "dgrad", 2, 16, 16, 2, 128, 64, stride=2, bias=False, relu=False, stats=False),
    conv_case("out_mul2_1x1", "fprop", 2, 16, 16, 1, 128, 64, out_mul=2, out_off=(1, 0), stats=True),
    conv_case("phase_dgrad_in_mul2", "dgrad", 2, 16, 32, 2, 128, 64, in_mul=2, in_off=(1, 0), pad=(1, 0),
              bias=False, relu=False, stats=False),
    conv_case("phase_dgrad_alias", "dgrad", 2, 16, 32, 2, 64, 128, in_mul=2, in_off=(0, 1), pad=(0, 1),
              addend="alias", bias=False, relu=False, stats=False),
    conv_case("phase_fprop_pad", "fprop", 2, 16, 32, 2, 64, 64, out_mul=2, out_off=(0, 1), pad=(1, 0)),
    # merged folded UpConv
    conv_case("fold1_il", "fprop", 2, 16, 32, 2, 64, 128, fold=1),
    conv_case("fold1_noil", "fprop", 3, 8, 16, 2, 64, 128, fold=1),
    conv_case("fold2", "dgrad", 2, 16, 32, 2, 128, 64, fold=2, bias=False, relu=False, stats=False),
    # the row-streaming kernel: test_gpu_c64.py CASES / FOLD_CASES, an addend, dgrad into a slice
    conv_case("c64_4x256", "fprop", 4, 256, 256, 3, 64, 64),
    conv_case("c64_5x251", "fprop", 5, 251, 128, 3, 64, 64, relu=False),
    conv_case("c64_3x203_2src", "fprop", 3, 203, 256, 3, 64, 64, c1=64),
    conv_case("c64_7x60", "fprop", 7, 60, 384, 3, 128, 64),
    conv_case("c64_37x33", "fprop", 37, 33, 128, 3, 64, 64),
    conv_case("c64_300x4", "fprop", 300, 4, 128, 3, 64, 64),
    conv_case("c64_add", "fprop", 5, 251, 128, 3, 64, 64, addend="add"),
    conv_case("c64_dgrad_slice", "dgrad", 5, 251, 128, 3, 64, 64, ld_y=64, bias=False, relu=False, stats=False),
    conv_case("c64_fold_10x128", "fprop", 10, 128, 128, 2, 128, 64, fold=1),
    conv_case("c64_fold_5x251", "fprop", 5, 251, 128, 2, 64, 64, fold=1),
    conv_case("c64_fold_3x150", "fprop", 3, 150, 256, 2, 128, 64, fold=1),
    conv_case("c64_fold_300x4", "fprop", 300, 4, 128, 2, 64, 64, fold=1),
    conv_case("c64_fold_37x33", "fprop", 37, 33, 128, 2, 128, 64, fold=1),
]

WGRAD_CASES = [
    wgrad_case("xh64x1_3x3", 2, 16, 64, 3, 64, 128),
    wgrad_case("xh32x2_3x3", 4, 32, 32, 3, 128, 128),
    wgrad_case("xh16x4_3x3", 4, 16, 16, 3, 64, 192),
    wgrad_case("nb4_3x3", 16, 4, 4, 3, 64, 128),
    wgrad_case("1x1_wide_reduce", 8, 64, 64, 1, 256, 64),
    wgrad_case("1x1_c0_152", 2, 32, 32, 1, 152, 64),
    wgrad_case("convT_xstride2", 2, 16, 16, 2, 64, 128, x_stride=2),
    wgrad_case("phase_dymul", 2, 16, 32, 2, 64, 128, dy_mul=2, dy_off=(1, 0), pad=(0, 1)),
    wgrad_case("rowpair2_oddH", 3, 17, 64, 3, 64, 64),
    wgrad_case("rowpair1_phase", 2, 16, 64, 2, 128, 64, dy_mul=2, dy_off=(0, 1), pad=(1, 0)),
    wgrad_case("wg_fold1", 2, 16, 32, 2, 128, 128, fold=True),
    wgrad_case("wg_fold2", 2, 16, 32, 2, 64, 64, fold=True),
    wgrad_case("pair256", 2, 32, 64, 3, 128, 256),
    wgrad_case("pair512_2src", 2, 16, 128, 3, 64, 512, c1=64),
    wgrad_case("one_split", 1, 8, 64, 3, 64, 128),
    wgrad_case("accumulate_2src", 2, 32, 64, 3, 64, 128, c1=64, accumulate=True),
    wgrad_case("dy_slice_cout64", 4, 32, 32, 3, 64, 64, ld_dy=64),
]

ALL_CASES = {c["name"]: c for c in CONV_CASES + WGRAD_CASES}
assert len(ALL_CASES) == len(CONV_CASES) + len(WGRAD_CASES)


def geometry(c, sms, max_pairs=None):
    return wgrad_plan(c, sms) if c["kind"] == "wgrad" else igemm_plan(c, sms, max_pairs)


def classes(c, sms):
    """the geometry classes a case reaches"""
    g = geometry(c, sms)
    out = set()
    if c["kind"] == "wgrad":
        if g["xh"] and not g["fold"]:
            out.add(f"wg_xh{g['Wb']}x{g['Hb']}")
        if not g["xh"] and g["Nb"] > 1:
            out.add("wg_nb>1")
        out |= {f"wg_{k}" for k, v in (("1x1", c["k"] == 1), ("xstride2", c["x_stride"] == 2),
                                       ("dymul", c["dy_mul"] == 2 and not c["fold"]),
                                       ("rowpair2", g["rowpair"] == 2), ("rowpair1", g["rowpair"] == 1),
                                       ("fold1", g["fold"] == 1), ("fold2", g["fold"] == 2),
                                       ("split1", g["splits"] == 1), ("splits_many", g["splits"] >= 16),
                                       ("accumulate", c["accumulate"]), ("two_src", c["c1"] > 0),
                                       ("cin_partial", (c["c0"] + c["c1"]) % 64 != 0),
                                       ("cout64", c["cout"] == 64), ("cout192", c["cout"] == 192),
                                       ("rowpair2_oddH", g["rowpair"] == 2 and c["h"] % 2 == 1)) if v}
        if g["pair"]:
            out.add(f"wg_pair{c['cout']}")
        out.add("wg_" + g["reduce"])
        return out
    out.add(g["kernel"].replace(" ", ""))
    if g["kernel"] == "conv_c64_kernel":
        out |= {"c64_fold" if g["fold"] else "c64", f"c64_epi{g['epi_groups']}"}
        if c["addend"]:
            out.add("c64_add")
        if c["kind"] == "dgrad" and c["ld_y"]:
            out.add("c64_dgrad_slice")
        return out
    out.add(f"block_n{g['block_n']}")
    if g["block_n"] != g["block_n0"]:
        out.add("small_m")
    if g["halo"]:
        out.add("halo" + ("_seam" if c["w"] > TILE_M else ""))
    if g["Hb"] > 1 and g["Nb"] == 1:
        out.add(f"multirow_w{g['Wb']}")
    if g["Nb"] > 1:
        out.add("multi_image" + ("_3x3" if c["h"] == 3 else ""))
    for k, v in (("clip_right", g["tw"] * g["Wb"] > c["w"]), ("clip_bottom", g["th"] * g["Hb"] > c["h"]),
                 ("clip_batch", g["tn"] * g["Nb"] > c["n"]), ("single_tile", g["m_tiles"] == 1),
                 ("wres", g["wres"]), ("dm", g["dm"]), ("add_tma", c["addend"] and g["add_tma"]),
                 ("add_rows", c["addend"] and not g["add_tma"]), ("add_alias", c["addend"] == "alias"),
                 ("add_after_act", c["add_after_act"]), ("no_bias", not c["bias"] and c["kind"] == "fprop"),
                 ("two_src", c["c1"] > 0), ("row_offset", c["row_offset"] > 0), ("slice_in", c["ld_x"] > 0),
                 ("slice_out", c["ld_y"] > 0), ("c0_partial", c["c0"] % 64 != 0), ("stride2", c["stride"] == 2),
                 ("dgrad_2x2s2", c["kind"] == "dgrad" and c["k"] == 2 and c["stride"] == 2),
                 ("out_mul", c["out_mul"] == 2), ("in_mul", c["in_mul"] == 2),
                 ("custom_pad", c["pad"] is not None), ("fold1_il", c["fold"] == 1 and g["fold_il"]),
                 ("fold1_noil", c["fold"] == 1 and not g["fold_il"]), ("fold2", c["fold"] == 2),
                 ("stats_flush", c["stats"] and g["stats_flush"]), ("relu", c["relu"]), ("no_relu", not c["relu"])):
        if v:
            out.add(k)
    if g["pair"]:
        out.add("pair_even" if g["m_tiles"] % 2 == 0 else "pair_odd")
    out.add(f"epi{g['epi_groups']}")
    return out


REQUIRED_CLASSES = {
    "conv_igemm_kernel<false,false>", "conv_igemm_kernel<false,true>", "conv_igemm_kernel<true,true>",
    "conv_c64_kernel", "block_n256", "block_n128", "block_n64", "block_n32", "small_m", "halo_seam",
    "multirow_w64", "multirow_w32", "multirow_w16", "multi_image", "multi_image_3x3", "clip_right", "clip_bottom",
    "clip_batch", "pair_even", "pair_odd", "single_tile", "epi1", "epi2", "wres", "stats_flush", "add_tma", "add_rows",
    "add_alias", "add_after_act", "relu", "no_relu", "no_bias", "two_src", "row_offset", "slice_in", "slice_out",
    "c0_partial", "stride2", "dgrad_2x2s2", "out_mul", "in_mul", "custom_pad", "fold1_il", "fold1_noil", "fold2",
    "c64", "c64_fold", "c64_add", "c64_dgrad_slice",
    "wg_xh64x1", "wg_xh32x2", "wg_xh16x4", "wg_nb>1", "wg_1x1", "wg_xstride2", "wg_dymul", "wg_rowpair2",
    "wg_rowpair2_oddH", "wg_rowpair1", "wg_fold1", "wg_fold2", "wg_pair256", "wg_pair512", "wg_split1",
    "wg_splits_many", "wg_wgrad_reduce_wide_kernel", "wg_wgrad_reduce_kernel", "wg_accumulate", "wg_two_src",
    "wg_cin_partial", "wg_cout64", "wg_cout192",
}

# with B200SEG_PAIR=0 the large N <= 128 layers run double-M work items (and wres_3x3 is one of them)
SWITCHES = {"B200SEG_C64": ["c64_5x251", "c64_add", "c64_dgrad_slice"],
            "B200SEG_C64_FOLD": ["c64_fold_5x251", "c64_fold_10x128"],
            "B200SEG_PAIR": ["wres_3x3", "bn128_w64", "halo_w256", "fold1_il", "clip_22x28_add", "c64_fold_300x4"],
            "B200SEG_WG_ROWPAIR": ["rowpair2_oddH", "rowpair1_phase", "dy_slice_cout64"],
            "B200SEG_WG_PAIR": ["pair256", "pair512_2src", "wg_fold1"]}


def test_mirror_reaches_every_class():
    """at 148 SMs the GPU matrix reaches every geometry class, and the switches-off subsets reach double-M and the
    generic kernel for the row-streaming shapes"""
    got = set()
    for c in ALL_CASES.values():
        got |= classes(c, SMS_B200)
    missing = REQUIRED_CLASSES - got
    assert not missing, sorted(missing)
    for c in ALL_CASES.values():
        print(c["name"], sorted(classes(c, SMS_B200)))
    saved = dict(os.environ)
    try:
        os.environ["B200SEG_PAIR"] = "0"
        assert igemm_plan(ALL_CASES["wres_3x3"], SMS_B200)["dm"] == 1
        os.environ["B200SEG_C64"] = "0"
        assert igemm_plan(ALL_CASES["c64_5x251"], SMS_B200)["kernel"].startswith("conv_igemm")
    finally:
        os.environ.clear()
        os.environ.update(saved)
    assert wgrad_plan(ALL_CASES["rowpair2_oddH"], SMS_B200)["rowpair"] == 2


# ----------------------------------------------------------------------------------------------------------
# §2 the reference (fp64, torch, any device)
# ----------------------------------------------------------------------------------------------------------
def _part(k, pad=None, stride=1, in_mul=1, in_off=(0, 0), out_mul=1, out_off=(0, 0), t0=0):
    pad = pad if pad is not None else ((k - 1) // 2, (k - 1) // 2)
    return dict(k=k, pad=pad, stride=stride, in_mul=in_mul, in_off=in_off, out_mul=out_mul, out_off=out_off, t0=t0)


def _tap_index(n, h, w, ih, iw, stride, dr, ds, dev, mutant=None, h0=0):
    """flat operand-pixel index of output (n, oh, ow) for one tap, n * ih * iw (the zero row) outside the image"""
    nn = torch.arange(n, device=dev).view(n, 1, 1)
    i = (stride * torch.arange(h0, h0 + h, device=dev) + dr).view(1, h, 1)
    j = (stride * torch.arange(w, device=dev) + ds).view(1, 1, w)
    if mutant == "seam" and ds == -1:
        ow = torch.arange(w, device=dev).view(1, 1, w)
        j = torch.where((ow % TILE_M == 0) & (ow > 0), j - 1, j)
    flat = (nn * ih + i) * iw + j
    if mutant == "wrap":
        valid = (flat >= 0) & (flat < n * ih * iw)
    else:
        valid = (i >= 0) & (i < ih) & (j >= 0) & (j < iw)
    return torch.where(valid, flat, torch.full_like(flat, n * ih * iw)).reshape(-1)


def conv_part(x, wt, part, h, w, mutant=None, h0=0):
    """x fp64 [n, H, W, C] (the full input), wt [taps, cout, C] -> [n, h, w, cout]: sum over taps (r, s) of the
    operand pixel (stride * oh + r - pad_h, stride * ow + s - pad_w) of the (in_off + in_mul * i) sub-lattice of x"""
    n, C = x.shape[0], x.shape[3]
    m, (oh_, ow_) = part["in_mul"], part["in_off"]
    og = x[:, oh_::m, ow_::m]
    ih, iw = og.shape[1], og.shape[2]
    flat = torch.cat([og.reshape(-1, C), og.new_zeros(1, C)])
    k, (ph, pw) = part["k"], part["pad"]
    out = None
    for o in range(k * k):
        idx = _tap_index(n, h, w, ih, iw, part["stride"], o // k - ph, o % k - pw, x.device, mutant, h0)
        term = flat[idx] @ wt[o].t()
        out = term if out is None else out + term
    return out.view(n, h, w, wt.shape[1])


def layer_forward(x, wt, parts, h, w, out_hw, mutant=None):
    """the launch / layer as a sum of placed parts: part p uses the taps wt[t0 : t0 + k * k] and lands on the
    (out_off + out_mul * i) sub-lattice of an out_hw output"""
    if len(parts) == 1 and parts[0]["out_mul"] == 1:
        p = parts[0]
        return conv_part(x, wt[p["t0"]:p["t0"] + p["k"] ** 2], p, h, w, mutant)
    y = x.new_zeros(x.shape[0], out_hw[0], out_hw[1], wt.shape[1])
    for p in parts:
        m, (a, b) = p["out_mul"], p["out_off"]
        y[:, a::m, b::m] = y[:, a::m, b::m] + conv_part(x, wt[p["t0"]:p["t0"] + p["k"] ** 2], p, h, w, mutant)
    return y


def fold_parts(fine_op=False):
    """the four 2x2 phase convolutions of a folded UpConv: phase (a, b) = taps 4 (2a + b) .. + 3, tap offsets
    (u - (1 - a), v - (1 - b)), output pixel (2h + a, 2w + b)"""
    return [_part(2, pad=(1 - a, 1 - b), out_mul=2, out_off=(a, b), t0=4 * (2 * a + b)) for a in (0, 1) for b in (0, 1)]


def launch_parts(c):
    """the parts of an fprop launch, in the kernel's own terms"""
    if c["fold"] == 1:
        return fold_parts()
    return [_part(c["k"], c["pad"], c["stride"], c["in_mul"], c["in_off"], c["out_mul"], c["out_off"])]


def dgrad_forward(c):
    """(parts, flip) of the forward layer whose input gradient a dgrad launch computes: the plain / phase convolutions
    with flipped taps (dgrad packing [k*k flipped][cin][cout]), or the four 1x1 placements of ConvTranspose2d(2, 2)
    (the 2x2 stride-2 dgrad, taps not flipped)"""
    if c["fold"] == 2:
        return fold_parts(), True
    if c["k"] == 2 and c["stride"] == 2:
        return [_part(1, out_mul=2, out_off=(i, j), t0=2 * i + j) for i in (0, 1) for j in (0, 1)], False
    if c["in_mul"] == 2:
        a, b = c["in_off"]
        return [_part(2, pad=(1 - a, 1 - b), out_mul=2, out_off=(a, b))], True
    return [_part(c["k"])], True


def forward_weights_from_dgrad(wd, parts, flip):
    """wd [taps, cin, cout] -> forward weights [taps, cout, cin] with each part's taps flipped (o -> k*k - 1 - o)"""
    out = wd.transpose(1, 2).clone()
    if flip:
        for p in parts:
            kk = p["k"] ** 2
            out[p["t0"]:p["t0"] + kk] = wd[p["t0"]:p["t0"] + kk].flip(0).transpose(1, 2)
    return out


def wgrad_parts(c):
    if c["fold"]:
        return fold_parts()
    if c["x_stride"] == 2:
        return [_part(2, pad=(0, 0), stride=2)]
    if c["dy_mul"] == 2:
        return [_part(2, pad=c["pad"], out_mul=2, out_off=c["dy_off"])]
    return [_part(c["k"], c["pad"])]


def epilogue(acc, bias, addend, relu, after, rounding=True):
    """act(acc + bias [+ addend]) or act(acc + bias) + addend, before the final bf16 rounding (the inner value, which
    the kernel rounds to bf16 before the addend joins, is straight-through); -> (value, inner value or None)"""
    v = acc + bias if bias is not None else acc
    if addend is not None and after:
        a = torch.relu(v) if relu else v
        return (_st(a, _r(a)) if rounding else a) + addend, a
    if addend is not None:
        v = v + addend
    return (torch.relu(v) if relu else v), None


def fprop_ref(t, c, mutant=None, rounding=True):
    """t: x [n, H, W, C0 + C1] fp64, wt [taps, cout, C], bias, addend (fp64, placed on the output grid).
    -> (pre-rounding output on the launch's output grid, S, the output-grid mask of the launch's pixels, one bf16 ulp
    of the inner rounding of add_after_act or 0)"""
    parts = launch_parts(c)
    wt = t["wt"]
    if mutant == "kblock":
        wt = wt.clone()
        wt[:, :, 64 * (c["c0"] // 64):c["c0"]] = 0
    if mutant == "phase_swap":
        wt = wt.clone()
        wt[4:8], wt[8:12] = t["wt"][8:12], t["wt"][4:8]
    oh, ow = out_extent(c)
    acc = layer_forward(t["x"], wt, parts, c["h"], c["w"], (oh, ow), mutant if mutant in ("wrap", "seam") else None)
    mag = layer_forward(t["x"].abs(), t["wt"].abs(), parts, c["h"], c["w"], (oh, ow))
    mask = own_mask(parts, c["n"], oh, ow, t["x"].device)
    bias = t.get("bias")
    add = t.get("addend")
    after = c["add_after_act"] != (mutant == "add_order")
    y, inner = epilogue(acc, bias, add, c["relu"], after, rounding)
    s = mag + (bias.abs() if bias is not None else 0) + (add.abs() if add is not None else 0)
    inner_ulp = ulp_bf16(inner.abs() + conv_eps(c) * s) if inner is not None else 0
    return y, s, mask, inner_ulp


def own_mask(parts, n, oh, ow, dev):
    """the output pixels a launch writes (None: all of them)"""
    if len(parts) == 1 and parts[0]["out_mul"] == 1:
        return None
    m = torch.zeros(n, oh, ow, 1, dtype=torch.bool, device=dev)
    for p in parts:
        mul, (a, b) = p["out_mul"], p["out_off"]
        m[:, a::mul, b::mul] = True
    return m


def out_extent(c):
    if c["fold"] == 1:
        return 2 * c["h"], 2 * c["w"]
    return c["h"] * c["out_mul"], c["w"] * c["out_mul"]


def dgrad_ref(t, c, mutant=None):
    """autograd of the forward layer at the dgrad launch's weights: t['x'] = dY (fp64, full fine tensor), t['wt'] =
    the dgrad packing [taps, rows, K] -> (dX rows [row_offset, row_offset + cout), S)"""
    parts, flip = dgrad_forward(c)
    if mutant == "unflipped":
        flip = not flip
    wd = t["wt"]
    if mutant == "phase_swap":
        wd = wd.clone()
        wd[4:8], wd[8:12] = t["wt"][8:12], t["wt"][4:8]
    dy = t["x"]
    n, hf, wf = dy.shape[:3]
    rows = wd.shape[1]

    def grad(dyv, wdv):
        xf = dy.new_zeros(n, c["h"], c["w"], rows, requires_grad=True)
        y = layer_forward(xf, forward_weights_from_dgrad(wdv, parts, flip), parts, c["h"], c["w"], (hf, wf),
                          mutant if mutant == "wrap" else None)
        assert y.shape == dyv.shape, (y.shape, dyv.shape)
        return torch.autograd.grad([y], [xf], [dyv])[0][..., c["row_offset"]:c["row_offset"] + c["cout"]]

    g = grad(dy, wd)
    mag = grad(dy.abs(), wd.abs())
    add = t.get("addend")
    y = g + add if add is not None else g
    return y, mag + (add.abs() if add is not None else 0), None, 0


def wgrad_ref(t, c, mutant=None):
    """autograd weight gradient of the layer's forward: t['x'] = X [n, H, W, C0 + C1], t['dy'] = the full dY tensor.
    -> dW in the kernel's layout ([cout][taps][cin], fold: [4][cout][4][cin]) and S"""
    parts = wgrad_parts(c)
    x, dy = t["x"], t["dy"]
    if mutant == "chunk":
        dy = dy * t["chunk_keep"]
    taps = 16 if c["fold"] else c["k"] ** 2

    def grad(xv, dyv, h_ext=0):
        wt = x.new_zeros(taps, c["cout"], x.shape[3], requires_grad=True)
        if h_ext:     # row-pair mutant: dY gets one more row below the image
            p = parts[0]
            y = conv_part(xv, wt, p, c["h"] + 1, c["w"])
        else:
            y = layer_forward(xv, wt, parts, c["h"], c["w"], dyv.shape[1:3])
        return torch.autograd.grad([y], [wt], [dyv])[0]

    g = grad(x, dy)
    if mutant == "rowpair_below":
        nxt = torch.roll(dy[:, :1], -1, dims=0)          # the next image's first row
        g = grad(x, torch.cat([dy, nxt], dim=1), h_ext=1)
    mag = grad(x.abs(), t["dy"].abs())
    if mutant == "transpose":
        k = c["k"]
        g = g.view(k, k, *g.shape[1:]).transpose(0, 1).reshape(g.shape)
    if mutant == "phase_swap":
        g = g.clone()
        g[4:8], g[8:12] = g[8:12].clone(), g[4:8].clone()

    def layout(v):
        if c["fold"]:
            return v.view(4, 4, c["cout"], -1).permute(0, 2, 1, 3)
        return v.permute(1, 0, 2)

    return layout(g), layout(mag)


# ----------------------------------------------------------------------------------------------------------
# bounds
# ----------------------------------------------------------------------------------------------------------
def conv_eps(c):
    cbt = -(-c["c0"] // 64) + -(-c["c1"] // 64)
    taps = 16 if c["fold"] == 2 else c["k"] ** 2
    return (taps * cbt * 4 + 3) * U23


def wgrad_eps(c, g):
    n_acc = 4 * g["chunks_per_split"] * (2 if g["rowpair"] or g["fold"] else 1) + g["splits"] + int(c["accumulate"])
    return (n_acc + 1) * U23


def conv_tol(ref, s, c, inner_ulp=0):
    """one bf16 ulp of the largest value the kernel's result can round from, + one of the inner value of
    add_after_act (the kernel and the reference may round it to neighbouring bf16 values), + eps * S"""
    e = conv_eps(c) * s
    return ulp_bf16(ref.abs() + e) + inner_ulp + e


def stats_tol(v):
    """fp32 partials over <= 32 rows, then fp64: [2, C] bound of the (sum, sum of squares) of the stored values v"""
    vd = v.double()
    return 33 * U23 * torch.stack([vd.abs().sum(0), (vd * vd).sum(0)])


# ----------------------------------------------------------------------------------------------------------
# inputs (any device) and mutants
# ----------------------------------------------------------------------------------------------------------
def _in_extent(c):
    if c["kind"] == "dgrad":
        if c["fold"] == 2 or c["in_mul"] == 2 or c["stride"] == 2:
            return 2 * c["h"], 2 * c["w"]
        return c["h"], c["w"]
    if c["fold"] == 1:
        return c["h"], c["w"]
    return c["h"] * c["stride"] * c["in_mul"], c["w"] * c["stride"] * c["in_mul"]


def make_conv_inputs(c, seed, device):
    """bf16 tensors as the kernel takes them and their fp64 copies for the reference"""
    gen = torch.Generator(device="cpu").manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=gen)
    hi, wi = _in_extent(c)
    cin = c["c0"] + c["c1"]
    taps = 16 if c["fold"] else c["k"] ** 2
    rows = c["cout"] + c["rows_extra"]
    ktot = -(-cin // 8) * 8
    xb = rn(c["n"], hi, wi, c["c0"] + c["ld_x"]).bfloat16()
    x0 = xb[..., c["ld_x"]:]                 # a channel slice at offset ld_x of a wider row when ld_x > 0
    x1 = rn(c["n"], hi, wi, c["c1"]).bfloat16() if c["c1"] else None
    wpk = (rn(taps, rows, ktot) / math.sqrt(cin * c["k"] ** 2)).bfloat16()
    wpk[..., cin:] = 0
    oh, ow = out_extent(c)
    ybuf = torch.full((c["n"], oh, ow, c["cout"] + c["ld_y"]), float("nan")).bfloat16()
    t = {"x0": x0, "x1": x1, "wpk": wpk, "ybuf": ybuf}
    if c["bias"]:
        t["bias"] = rn(c["cout"]).float()
    if c["addend"]:
        add = rn(c["n"], c["h"], c["w"], c["cout"]).bfloat16()
        if c["addend"] == "alias":
            ybuf = rn(c["n"], oh, ow, c["cout"] + c["ld_y"]).bfloat16()
            if c["ld_y"]:
                ybuf[..., :c["ld_y"]] = float("nan")
            t["ybuf"] = ybuf
        t["add"] = add
    t = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in t.items()}
    return t


def conv_ref_inputs(t, c):
    """fp64 tensors of the reference: the (concatenated) input, the weights [taps, rows, C] (forward or dgrad packing)
    and the addend on the launch's output grid"""
    x = t["x0"].double()
    if t["x1"] is not None:
        x = torch.cat([x, t["x1"].double()], dim=3)
    cin = c["c0"] + c["c1"]
    r = {"x": x}
    if c["kind"] == "fprop":
        r["wt"] = t["wpk"][:, c["row_offset"]:c["row_offset"] + c["cout"], :cin].double()
    else:
        r["wt"] = t["wpk"][..., :cin].double()
    if "bias" in t:
        r["bias"] = t["bias"].double()
    if c["addend"] == "alias":
        r["addend"] = t["ybuf"][..., c["ld_y"]:].double()
    elif c["addend"]:
        r["addend"] = t["add"].double()
    return r


def conv_mutants(c, g):
    m = []
    if c["kind"] == "fprop" and c["k"] > 1 and c["fold"] == 0 and g.get("Nb", 1) * g.get("Hb", 1) > 1 and \
            c["pad"] is None:
        m.append("wrap")
    if c["kind"] == "fprop" and c["k"] == 3 and c["w"] > TILE_M and c["stride"] == 1:
        m.append("seam")
    if c["c0"] % 64 and c["kind"] == "fprop":
        m.append("kblock")
    if c["addend"] and c["relu"]:
        m.append("add_order")
    if c["stats"] and c["bias"] and clipped_rows(c, g) > 0:
        m.append("stats_clip")
    if c["kind"] == "dgrad" and c["k"] > 1 and not (c["k"] == 2 and c["stride"] == 2):
        m.append("unflipped")          # (the 2x2 stride-2 dgrad is four 1x1 placements: nothing to flip)
    if c["fold"] in (1, 2):
        m.append("phase_swap")
    return m


def wgrad_mutants(c, g):
    m = []
    if c["k"] > 1 and not c["fold"]:
        m.append("transpose")
    if g["splits"] > 1 and not c["fold"]:
        m.append("chunk")
    if c["fold"]:
        m.append("phase_swap")
    if g["rowpair"] == 2 and c["h"] % 2 == 1:
        m.append("rowpair_below")
    return m


def clipped_rows(c, g):
    """accumulator rows of the launch's tiles that are outside the tensor (the ragged last tile of a pair excluded)"""
    if g["kernel"] == "conv_c64_kernel":
        return 0
    real = c["n"] * c["h"] * c["w"] * (4 if c["fold"] == 1 else 1)
    return g["m_tiles"] * TILE_M - real


def chunk_pixels(c, g, chunk):
    """(n, h, w) ranges of 64-pixel chunk `chunk` of the weight-gradient launch (the dY grid)"""
    t = chunk
    tw_i, t1 = t % g["tw"], t // g["tw"]
    th_i, tn_i = t1 % g["th"], t1 // g["th"]
    return ((tn_i * g["Nb"], (tn_i + 1) * g["Nb"]), (th_i * g["Hb"], (th_i + 1) * g["Hb"]),
            (tw_i * g["Wb"], (tw_i + 1) * g["Wb"]))


def make_wgrad_inputs(c, g, seed, device):
    """bf16 X (x0 | x1) and dY; the dY pixels of the first chunk of every split after the first are scaled by 16
    (exact), so that a dropped boundary chunk is far outside the bound; chunk_keep zeroes the first of them"""
    gen = torch.Generator(device="cpu").manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=gen)
    xs, dm = c["x_stride"], (2 if c["fold"] else c["dy_mul"])
    n, h, w = c["n"], c["h"], c["w"]
    x0 = rn(n, h * xs, w * xs, c["c0"]).bfloat16()
    x1 = rn(n, h * xs, w * xs, c["c1"]).bfloat16() if c["c1"] else None
    dyb = rn(n, h * dm, w * dm, c["cout"] + c["ld_dy"]).bfloat16()
    keep = torch.ones(n, h * dm, w * dm, 1)
    if g["splits"] > 1 and not c["fold"]:
        oh, ow = (c["dy_off"] if dm == 2 else (0, 0))
        for s in range(1, g["splits"]):
            (n0, n1), (h0, h1), (w0, w1) = chunk_pixels(c, g, s * g["chunks_per_split"])
            sl = (slice(n0, n1), slice(h0 * dm + oh, h1 * dm + oh, dm), slice(w0 * dm + ow, w1 * dm + ow, dm))
            dyb[sl] = (dyb[sl].float() * 16).bfloat16()
            if s == 1:
                keep[sl] = 0
    t = {"x0": x0, "x1": x1, "dyb": dyb, "dy": dyb[..., c["ld_dy"]:], "keep": keep}
    if c["accumulate"]:
        t["dw0"] = rn(*((4, c["cout"], 4, c["c0"] + c["c1"]) if c["fold"] else
                        (c["cout"], c["k"] ** 2, c["c0"] + c["c1"])))
    return {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in t.items()}


def wgrad_ref_inputs(t):
    x = t["x0"].double()
    if t["x1"] is not None:
        x = torch.cat([x, t["x1"].double()], dim=3)
    return {"x": x, "dy": t["dy"].double(), "chunk_keep": t["keep"].double()}


def conv_units(got, ref, tol, mask=None):
    """worst |got - ref| / tol over the launch's pixels"""
    err = got.double() - ref
    if mask is not None:
        err = err * mask
    return _worst(err, tol)


# ----------------------------------------------------------------------------------------------------------
# §2 the reference on its own (CPU)
# ----------------------------------------------------------------------------------------------------------
def _close(a, b, what):
    a, b = a.detach(), b.detach()
    assert float((a - b).abs().max()) <= 1e-10 * max(1.0, float(b.abs().max())), what


def _nchw(v):
    return v.permute(0, 3, 1, 2)


def _nhwc_(v):
    return v.permute(0, 2, 3, 1)


def test_reference_without_rounding_is_torch():
    """rounding off, the reference is torch: F.conv2d (padding, stride, two sources), the four UpConv phases are
    Upsample x2 + conv3x3 with the folded weights, the 2x2 stride-2 dgrad is conv_transpose2d's input gradient,
    and dgrad / wgrad of the plain and phase layers are torch autograd of F.conv2d / the upsampled conv"""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(0)
    rn = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    n, h, w, ci, co = 2, 6, 10, 12, 8
    for k in (1, 3):
        for stride in (1, 2):
            x = rn(n, h * stride, w * stride, ci)
            wt = rn(k * k, co, ci)
            W = wt.view(k, k, co, ci).permute(2, 3, 0, 1)
            c = conv_case("t", "fprop", n, h, w, k, 8, co, c1=ci - 8, stride=stride, addend="add")
            t = {"x": x, "wt": wt, "bias": rn(co), "addend": rn(n, h, w, co)}
            y = fprop_ref(t, c, rounding=False)[0]
            want = _nhwc_(F.conv2d(_nchw(x), W, t["bias"], stride=stride, padding=(k - 1) // 2)) + t["addend"]
            _close(y, torch.relu(want), f"fprop k={k} stride={stride}")
            if stride == 1:
                # dgrad: the kernel's dgrad packing [taps flipped][cin][cout] -> dX = autograd of F.conv2d
                dy = rn(n, h, w, co)
                wd = W.permute(2, 3, 1, 0).flip(0, 1).reshape(k * k, ci, co)
                cd = conv_case("d", "dgrad", n, h, w, k, co, ci, bias=False, relu=False)
                dx = dgrad_ref({"x": dy, "wt": wd}, cd)[0]
                xl = _nchw(x).clone().requires_grad_(True)
                F.conv2d(xl, W, padding=(k - 1) // 2).backward(_nchw(dy))
                _close(dx, _nhwc_(xl.grad), f"dgrad k={k}")
                # wgrad: dW [cout][taps][cin]
                cw = wgrad_case("w", n, h, w, k, ci, co)
                dw, _ = wgrad_ref({"x": x, "dy": dy}, cw)
                Wl = W.clone().requires_grad_(True)
                F.conv2d(_nchw(x), Wl, padding=(k - 1) // 2).backward(_nchw(dy))
                _close(dw, Wl.grad.permute(0, 2, 3, 1).reshape(co, k * k, ci), f"wgrad k={k}")
    # the folded UpConv: phases of Upsample x2 + conv3x3 (fold 1), its input gradient (fold 2), its weight gradient
    # (fold wgrad), checked through the folding W_ab[u][v] = sum_{r in R_a(u)} sum_{s in R_b(v)} W[r][s]
    W3 = rn(co, ci, 3, 3)
    R = [[[0], [1, 2]], [[0, 1], [2]]]
    wf = torch.zeros(16, co, ci, dtype=torch.float64)
    for a in (0, 1):
        for b in (0, 1):
            for u in (0, 1):
                for v in (0, 1):
                    wf[4 * (2 * a + b) + 2 * u + v] = sum(W3[:, :, r, s] for r in R[a][u] for s in R[b][v])
    x = rn(n, h, w, ci)
    c = conv_case("f", "fprop", n, h, w, 2, ci, co, fold=1, bias=False, relu=False)
    y = fprop_ref({"x": x, "wt": wf}, c, rounding=False)[0]
    up = lambda v: F.interpolate(_nchw(v), scale_factor=2, mode="nearest")
    _close(y, _nhwc_(F.conv2d(up(x), W3, padding=1)), "fold 1 = Upsample + conv3x3")
    for ph in range(4):
        a, b = ph >> 1, ph & 1
        cp = conv_case("p", "fprop", n, h, w, 2, ci, co, out_mul=2, out_off=(a, b), pad=(1 - a, 1 - b), bias=False,
                       relu=False)
        yp = fprop_ref({"x": x, "wt": wf[4 * ph:4 * ph + 4]}, cp, rounding=False)[0]
        _close(yp[:, a::2, b::2], y[:, a::2, b::2], f"phase {ph} fprop")
    dz = rn(n, 2 * h, 2 * w, co)
    wdf = wf.view(4, 4, co, ci).flip(1).transpose(2, 3).reshape(16, ci, co)   # [phase][flipped tap][cin][cout]
    c2 = conv_case("f2", "dgrad", n, h, w, 2, co, ci, fold=2, bias=False, relu=False)
    dx = dgrad_ref({"x": dz, "wt": wdf}, c2)[0]
    xl = _nchw(x).clone().requires_grad_(True)
    F.conv2d(F.interpolate(xl, scale_factor=2, mode="nearest"), W3, padding=1).backward(_nchw(dz))
    _close(dx, _nhwc_(xl.grad), "fold 2 = input gradient of Upsample + conv3x3")
    dsum = torch.zeros_like(dx)
    for ph in range(4):
        a, b = ph >> 1, ph & 1
        cp = conv_case("pd", "dgrad", n, h, w, 2, co, ci, in_mul=2, in_off=(a, b), pad=(a, b), bias=False, relu=False)
        dsum = dsum + dgrad_ref({"x": dz, "wt": wdf[4 * ph:4 * ph + 4]}, cp)[0]
    _close(dsum, dx, "the four phase dgrads sum to fold 2")
    cw = wgrad_case("fw", n, h, w, 2, ci, co, fold=True)
    dwe, _ = wgrad_ref({"x": x, "dy": dz}, cw)                                 # [4][cout][4][cin]
    Wl = W3.clone().requires_grad_(True)
    F.conv2d(up(x), Wl, padding=1).backward(_nchw(dz))
    dw9 = torch.zeros(co, ci, 3, 3, dtype=torch.float64)
    for a in (0, 1):
        for b in (0, 1):
            for u in (0, 1):
                for v in (0, 1):
                    for r in R[a][u]:
                        for s in R[b][v]:
                            dw9[:, :, r, s] += dwe[2 * a + b, :, 2 * u + v]
    _close(dw9, Wl.grad, "fold wgrad, unfolded = the weight gradient of Upsample + conv3x3")
    # ConvTranspose2d(k2, s2): the 2x2 stride-2 dgrad is its input gradient, x_stride 2 wgrad its weight gradient
    Wt = rn(ci, co, 2, 2)                      # ConvTranspose weight [in = ci][out = co]
    xc = rn(n, h, w, ci)
    dyf = rn(n, 2 * h, 2 * w, co)
    wd = Wt.permute(2, 3, 0, 1).reshape(4, ci, co)           # 'convT_d' packing [tap][cin][cout]
    cd = conv_case("t2", "dgrad", n, h, w, 2, co, ci, stride=2, bias=False, relu=False)
    dx = dgrad_ref({"x": dyf, "wt": wd}, cd)[0]
    xl = _nchw(xc).clone().requires_grad_(True)
    F.conv_transpose2d(xl, Wt, stride=2).backward(_nchw(dyf))
    _close(dx, _nhwc_(xl.grad), "2x2 stride-2 dgrad = conv_transpose2d input gradient")
    cw = wgrad_case("t2w", n, h, w, 2, co, ci, x_stride=2)
    dw, _ = wgrad_ref({"x": dyf, "dy": xc}, cw)             # [cin_T][4][cout_T]
    Wl = Wt.clone().requires_grad_(True)
    F.conv_transpose2d(_nchw(xc), Wl, stride=2).backward(_nchw(dyf))
    _close(dw, Wl.grad.permute(0, 2, 3, 1).reshape(ci, 4, co), "x_stride 2 wgrad = conv_transpose2d weight gradient")


# ----------------------------------------------------------------------------------------------------------
# mutant separation (CPU at small shapes, and in every GPU case)
# ----------------------------------------------------------------------------------------------------------
def conv_mutant_units(c, g, r, y, s, mask, got, got_stats=None, inner_ulp=0):
    """mutant -> max over checked elements of |mutant ref - kernel output| / bound"""
    ref_fn = fprop_ref if c["kind"] == "fprop" else dgrad_ref
    units = {}
    tol = conv_tol(y, s, c, inner_ulp)
    for m in conv_mutants(c, g):
        if m == "stats_clip":
            nclip = clipped_rows(c, g)
            bias = r["bias"]
            v = _r(torch.relu(bias) if c["relu"] else bias)
            st = got_stats + nclip * torch.stack([v, v * v])
            want = exact_stats(got, mask)
            units[m] = _worst(st - want, stats_tol(masked_rows(got, mask)))
            continue
        ym = ref_fn(r, c, mutant=m)[0]
        units[m] = conv_units(got, ym, tol, mask)
    return units


def masked_rows(v, mask):
    v = v.double().reshape(-1, v.shape[-1])
    if mask is not None:
        v = v[mask.reshape(-1)]
    return v


def exact_stats(v, mask=None):
    vd = masked_rows(v, mask)
    return torch.stack([vd.sum(0), (vd * vd).sum(0)])


def _cpu_small(c):
    """the case at a small extent that keeps its mode (CPU mutant check)"""
    s = dict(c)
    s["n"], s["h"], s["w"] = min(c["n"], 2), min(c["h"], 9), min(c["w"], 12)
    if c["kind"] == "wgrad":
        if c["fold"] or c["dy_mul"] == 2:
            s["h"], s["w"] = min(c["h"], 6), min(c["w"], 16)
        return s
    if c["w"] > TILE_M:
        s["w"] = 2 * TILE_M + 8                 # keeps a halo seam
        s["h"] = 2
        s["n"] = 1
    if c["h"] == 3:
        s["h"], s["w"], s["n"] = 3, 3, 3
    return s


@pytest.mark.parametrize("name", [c["name"] for c in CONV_CASES])
def test_conv_mutants_separate(name):
    """each applicable conv mutant moves some output (or statistic) by >= 10x its bound, with the kernel output
    emulated as the rounded reference, at a small extent of the case on the CPU (geometry of the full case)"""
    c = ALL_CASES[name]
    cs = _cpu_small(c)
    cs["c0"], cs["c1"] = min(c["c0"], 152), min(c["c1"], 64)
    cs["cout"] = min(c["cout"], 64)
    cs["rows_extra"] = min(c["rows_extra"], 64)
    if cs["kind"] == "dgrad" and cs["row_offset"]:
        cs["row_offset"] = cs["rows_extra"]
    t = make_conv_inputs(cs, 1, "cpu")
    r = conv_ref_inputs(t, cs)
    ref_fn = fprop_ref if cs["kind"] == "fprop" else dgrad_ref
    y, s, mask, iu = ref_fn(r, cs)
    got = _r(y)
    stats = exact_stats(got, mask) if cs["stats"] else None
    units = conv_mutant_units(cs, geometry(cs, SMS_B200), r, y, s, mask, got, stats, iu)
    assert conv_units(got, y, conv_tol(y, s, cs, iu), mask) <= 1
    print(name, {k: round(v, 1) for k, v in units.items()})
    for m, u in units.items():
        assert u >= MUTANT_MARGIN, (name, m, units)


@pytest.mark.parametrize("name", [c["name"] for c in WGRAD_CASES])
def test_wgrad_mutants_separate(name):
    c = ALL_CASES[name]
    cs = _cpu_small(c)
    cs["c0"], cs["c1"], cs["cout"] = min(c["c0"], 72), min(c["c1"], 16), min(c["cout"], 64)
    g = wgrad_plan(cs, SMS_B200)
    g["splits"], g["chunks_per_split"] = max(2, g["splits"]), max(1, g["num_chunks"] // 2)
    if g["num_chunks"] < 2:
        g["splits"] = 1
    t = make_wgrad_inputs(cs, g, 2, "cpu")
    r = wgrad_ref_inputs(t)
    dw, s = wgrad_ref(r, cs)
    tol = wgrad_eps(cs, g) * s
    units = {}
    for m in wgrad_mutants(cs, dict(g, rowpair=2 if c["name"].startswith("rowpair2") else g["rowpair"])):
        units[m] = _worst(wgrad_ref(r, cs, mutant=m)[0] - dw, tol)
    print(name, {k: round(v, 1) for k, v in units.items()})
    for m, u in units.items():
        assert u >= MUTANT_MARGIN, (name, m, units)


# ----------------------------------------------------------------------------------------------------------
# §3 the kernels (GPU)
# ----------------------------------------------------------------------------------------------------------
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def run_conv(c, t):
    """one launch through kernels.conv_igemm; -> (the whole output buffer, the launch's output slice, stats)"""
    from b200seg import kernels as K
    ybuf = t["ybuf"]
    y = ybuf[..., c["ld_y"]:] if c["ld_y"] else ybuf
    stats = torch.zeros(2, c["cout"], dtype=torch.float64, device="cuda") if c["stats"] else None
    add = None
    if c["addend"] == "alias":
        add = y
    elif c["addend"]:
        add = t["add"]
    K.conv_igemm(t["x0"], t["wpk"], c["cout"], c["k"], x1=t["x1"], bias=t.get("bias"), addend=add, stats=stats,
                 relu=c["relu"], out=y, row_offset=c["row_offset"], dgrad=c["kind"] == "dgrad", stride=c["stride"],
                 out_mul=c["out_mul"], out_off=c["out_off"], in_mul=c["in_mul"], in_off=c["in_off"], pad=c["pad"],
                 add_after_act=c["add_after_act"], fold=c["fold"])
    return ybuf, y, stats


def check_conv(c, seed=0, label=""):
    g = geometry(c, _sms())
    t = make_conv_inputs(c, seed, "cuda")
    r = conv_ref_inputs(t, c)          # before the launch: an aliased addend is the output's initial contents
    before = t["ybuf"].clone()
    ybuf, y, stats = run_conv(c, t)
    ref_fn = fprop_ref if c["kind"] == "fprop" else dgrad_ref
    with torch.no_grad() if c["kind"] == "fprop" else torch.enable_grad():
        ref, s, mask, iu = ref_fn(r, c)
    ref, s = ref.detach(), s.detach()
    tol = conv_tol(ref, s, c, iu)
    units = {"out": conv_units(y, ref, tol, mask)}
    # bytes the launch does not own keep their contents (NaN sentinel / the aliased tensor's other channels)
    keep = torch.ones(ybuf.shape, dtype=torch.bool, device="cuda")
    if mask is None:
        keep[..., c["ld_y"]:] = False
    else:
        keep[..., c["ld_y"]:] = ~mask
    assert torch.equal(_bits(ybuf)[keep], _bits(before)[keep]), (c["name"], "bytes outside the launch's output changed")
    if mask is not None:
        assert torch.isfinite(y.float()[mask.expand_as(y)]).all()
    else:
        assert torch.isfinite(y.float()).all()
    if stats is not None:
        want = exact_stats(y, mask)
        units["stats"] = _worst(stats - want, stats_tol(masked_rows(y, mask)))
    mut = conv_mutant_units(c, g, r, ref, s, mask, y, stats, iu)
    cls = sorted(classes(c, _sms()))
    print(f"{c['name']}{label}: {cls} worst err/bound " + ", ".join(f"{k} {v:.3g}" for k, v in units.items()) +
          " | mutants " + ", ".join(f"{k} {v:.3g}" for k, v in mut.items()))
    for k, v in units.items():
        assert v <= 1, (c["name"], k, units)
    for k, v in mut.items():
        assert v >= MUTANT_MARGIN, (c["name"], k, mut)
    return y, stats


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in CONV_CASES])
def test_conv_case(name):
    check_conv(ALL_CASES[name], seed=len(name))


def run_wgrad(c, t, ws_fill=None):
    """conv_wgrad; with ws_fill the workspace is allocated here and filled with that value first"""
    from b200seg import kernels as K
    out = t["dw0"].clone() if c["accumulate"] else None
    kw = dict(x1=t["x1"], out=out, accumulate=c["accumulate"], x_stride=c["x_stride"], dy_mul=c["dy_mul"],
              dy_off=c["dy_off"], pad=c["pad"], fold=c["fold"])
    if c["fold"]:
        kw["dy_mul"] = 2
    if ws_fill is None:
        return K.conv_wgrad(t["dy"], t["x0"], c["k"], **kw)
    real_empty = torch.empty

    def filled_empty(*a, **k):
        v = real_empty(*a, **k)
        if v.dtype == torch.uint8:
            v.view(torch.float32).fill_(ws_fill)
        return v

    torch.empty = filled_empty
    try:
        return K.conv_wgrad(t["dy"], t["x0"], c["k"], **kw)
    finally:
        torch.empty = real_empty


def check_wgrad(c, seed=0, label="", ws_fill=None):
    g = wgrad_plan(c, _sms())
    t = make_wgrad_inputs(c, g, seed, "cuda")
    dw = run_wgrad(c, t, ws_fill)
    r = wgrad_ref_inputs(t)
    ref, s = wgrad_ref(r, c)
    dw = dw.view(ref.shape)           # the merged fold launch writes [phase][cout][tap][cin]
    if c["accumulate"]:
        ref, s = ref + t["dw0"].double(), s + t["dw0"].double().abs()
    tol = wgrad_eps(c, g) * s
    u = _worst(dw.double() - ref, tol)
    mut = {}
    for m in wgrad_mutants(c, g):
        mref = wgrad_ref(r, c, mutant=m)[0] + (t["dw0"].double() if c["accumulate"] else 0)
        mut[m] = _worst(dw.double() - mref, tol)
    print(f"{c['name']}{label}: {sorted(classes(c, _sms()))} splits {g['splits']} worst err/bound dW {u:.3g} | "
          "mutants " + ", ".join(f"{k} {v:.3g}" for k, v in mut.items()))
    assert u <= 1, (c["name"], u)
    for k, v in mut.items():
        assert v >= MUTANT_MARGIN, (c["name"], k, mut)
    return dw


@pytest.mark.gpu
@pytest.mark.parametrize("name", [c["name"] for c in WGRAD_CASES])
def test_wgrad_case(name):
    check_wgrad(ALL_CASES[name], seed=len(name))


# ----------------------------------------------------------------------------------------------------------
# §4 the mirror against what launched (GPU): kernel names, grids and shared memory from a profiler trace, the split
# count from the workspace size
# ----------------------------------------------------------------------------------------------------------
_KNAME = re.compile(r"(conv_igemm_kernel<[^>]*>|conv_c64_kernel|conv_wgrad_kernel<[^>]*>|wgrad_reduce_wide_kernel|"
                    r"wgrad_reduce_kernel)")


def profiled_launches(calls, reps=3):
    """{label: [the library's kernels]} of ONE profiler session in which each labelled call runs `reps` times inside a
    record_function range that starts and ends with a device synchronise, so that the kernels of a call execute inside
    its range.  Kernels are assigned to a call by time, not by session: the activity records of a launch can reach
    the profiler after a short session has ended (a launch missing from its own session and showing up in the next
    one), and the session ends only after a pause that lets the last records arrive."""
    import time
    from torch.profiler import ProfilerActivity, profile, record_function
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for label, fn in calls:
            with record_function(f"conv-case:{label}"):
                torch.cuda.synchronize()
                for _ in range(reps):
                    fn()
                torch.cuda.synchronize()
            time.sleep(0.002)
        time.sleep(0.5)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            ev = json.load(f)["traceEvents"]
    ranges = [(e["name"][len("conv-case:"):], float(e["ts"]), float(e["ts"]) + float(e.get("dur", 0)))
              for e in ev if e.get("cat") == "user_annotation" and e.get("name", "").startswith("conv-case:")]
    out = {label: [] for label, _ in calls}
    for e in ev:
        if e.get("cat") != "kernel":
            continue
        m = _KNAME.search(e.get("name", ""))
        if not m:
            continue
        mid = float(e["ts"]) + 0.5 * float(e.get("dur", 0))
        for label, t0, t1 in ranges:
            if t0 <= mid <= t1:
                args = e.get("args", {})
                out[label].append({"name": m.group(1).replace(" ", ""), "grid": args.get("grid"),
                                   "smem": args.get("shared memory")})
    return out


def _wgrad_args(c):
    from b200seg import kernels as K
    a = K.WgradArgs()
    a.n, a.h, a.w, a.ksize = c["n"], c["h"], c["w"], c["k"]
    a.cout, a.lddy, a.c0, a.ldx0, a.c1, a.ldx1 = c["cout"], c["cout"] + c["ld_dy"], c["c0"], c["c0"], c["c1"], c["c1"]
    a.x_stride = c["x_stride"]
    a.dy_mul = 2 if c["fold"] else c["dy_mul"]
    a.dy_off_h, a.dy_off_w = c["dy_off"]
    if c["pad"] is not None:
        a.custom_pad, a.pad_h, a.pad_w = 1, c["pad"][0], c["pad"][1]
    a.fold = int(c["fold"])
    return a


@pytest.mark.gpu
def test_launches_match_mirror():
    """every case of the matrix launches the kernel, grid and shared memory the mirror predicts.  2-CTA clusters: the
    grid is capped by the number of co-resident clusters (cudaOccupancyMaxActiveClusters), which the trace of the
    largest one-n-tile pair launch reveals; every other pair launch must agree with that value."""
    from b200seg import _lib, kernels as K
    sms = _sms()
    calls, plans = [], {}
    for c in CONV_CASES:
        t = make_conv_inputs(c, 0, "cuda")
        run_conv(c, t)        # warm: module load, attributes
        calls.append((c["name"], (lambda c=c, t=t: run_conv(c, t))))
    for c in WGRAD_CASES:
        g = wgrad_plan(c, sms)
        assert int(_lib.load().b2_conv_wgrad_workspace(K.C.byref(_wgrad_args(c)))) == g["workspace"], c["name"]
        t = make_wgrad_inputs(c, g, 0, "cuda")
        run_wgrad(c, t)
        calls.append((c["name"], (lambda c=c, t=t: run_wgrad(c, t))))
    launched = profiled_launches(calls)
    # the cap on 2-CTA clusters, from the pair launch with the most work items and a single n-tile
    pairs = [c for c in CONV_CASES if geometry(c, sms).get("pair") and geometry(c, sms)["n_tiles"] == 1
             and geometry(c, sms)["total"] >= sms // 2]
    big = max(pairs, key=lambda c: geometry(c, sms)["total"])
    max_pairs = launched[big["name"]][0]["grid"][0] // 2 if launched[big["name"]] else None
    assert max_pairs is not None and 1 <= max_pairs <= sms // 2, (big["name"], launched[big["name"]])
    smem_seen = False
    for c in CONV_CASES:
        g = geometry(c, sms, max_pairs)
        ks = [k for k in launched[c["name"]] if k["name"].startswith("conv_")]
        assert ks and all(k == ks[0] for k in ks), (c["name"], ks)
        k = ks[0]
        assert k["name"] == g["kernel"].replace(" ", ""), (c["name"], k, g["kernel"])
        assert list(k["grid"]) == [g["grid"], 1, 1], (c["name"], k, g["grid"])
        if k["smem"] is not None:
            smem_seen = True
            assert k["smem"] == g["smem"], (c["name"], k["smem"], g["smem"])
        print(f"{c['name']}: {k['name']} grid {k['grid']} smem {k['smem']} (mirror {g['smem']})")
    for c in WGRAD_CASES:
        g = wgrad_plan(c, sms)
        ks = launched[c["name"]]
        names = sorted({k["name"] for k in ks})
        assert names == sorted([g["kernel"].replace(" ", ""), g["reduce"]]), (c["name"], names)
        ks = [k for k in ks if k["name"].startswith("conv_wgrad")]
        assert all(k == ks[0] for k in ks), (c["name"], ks)
        assert list(ks[0]["grid"]) == [g["grid"][0], g["grid"][1], 1], (c["name"], ks[0], g["grid"])
        if ks[0]["smem"] is not None:
            assert ks[0]["smem"] == g["smem"], (c["name"], ks[0]["smem"], g["smem"])
        print(f"{c['name']}: {names} grid {ks[0]['grid']} smem {ks[0]['smem']} splits {g['splits']}")
    print(f"per-block shared memory in the trace: {'yes' if smem_seen else 'no (name and grid checked only)'}; "
          f"co-resident 2-CTA clusters: {max_pairs}")


# ----------------------------------------------------------------------------------------------------------
# §5 switches off (read once per process: a child process) and deterministic mode
# ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("switch", sorted(SWITCHES))
def test_switched_off(switch):
    """the subset of the matrix under SWITCH=0, the mirror recomputed in the child (B200SEG_PAIR=0 is what runs
    double-M work items)"""
    env = dict(os.environ, **{switch: "0"})
    here = os.path.abspath(__file__)
    ids = [f"{here}::{'test_wgrad_case' if ALL_CASES[n]['kind'] == 'wgrad' else 'test_conv_case'}[{n}]"
           for n in SWITCHES[switch]]
    r = subprocess.run([sys.executable, "-m", "pytest", *ids, "-q", "-x", "-s", "-p", "no:cacheprovider"], env=env,
                       cwd=os.path.dirname(os.path.dirname(here)), capture_output=True, text=True, timeout=1800)
    print(r.stdout[-3000:])
    assert r.returncode == 0, (switch, r.stdout[-4000:], r.stderr[-2000:])
    if switch == "B200SEG_PAIR":
        assert "'dm'" in r.stdout, "no double-M launch in the child"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["stats_flush_192", "clip_22x28_add", "c64_5x251", "fold1_il", "bn256_3x3"])
def test_conv_stats_deterministic(filled_workspace, name):  # noqa: F811
    """deterministic mode: the statistics (and outputs) bit-identical over two runs and between a NaN- and a
    zero-filled workspace, and within the bounds"""
    runs = []
    for v in (float("nan"), 0.0, 0.0):
        filled_workspace(v)
        runs.append(check_conv(ALL_CASES[name], seed=3, label=" deterministic"))
        torch.cuda.synchronize()
    (ya, sa), (yb, sb), (yc, sc) = runs
    assert torch.equal(_bits(sb), _bits(sc)) and torch.equal(_bits(sa), _bits(sb)), name
    assert torch.equal(_bits(yb), _bits(yc)) and torch.equal(_bits(ya), _bits(yb)), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["xh64x1_3x3", "1x1_wide_reduce", "accumulate_2src", "wg_fold1"])
def test_wgrad_deterministic(name):
    """dW bit-identical over two runs and between a NaN- and a zero-filled workspace (every partial tile slot is
    written before the reduce reads it)"""
    c = ALL_CASES[name]
    runs = [check_wgrad(c, seed=4, label=f" workspace {v}", ws_fill=v) for v in (float("nan"), 0.0, 0.0)]
    assert torch.equal(_bits(runs[1]), _bits(runs[2])) and torch.equal(_bits(runs[0]), _bits(runs[1])), name


@pytest.mark.gpu
def test_addend_with_output_placement_is_rejected():
    """an addend with out_mul > 1 would be read on the conv grid while the output is written on the placed grid: the
    library rejects the combination"""
    from b200seg import kernels as K
    c = ALL_CASES["out_mul2_1x1"]
    t = make_conv_inputs(c, 0, "cuda")
    add = torch.zeros(c["n"], c["h"], c["w"], c["cout"], dtype=torch.bfloat16, device="cuda")
    with pytest.raises(RuntimeError):
        K.conv_igemm(t["x0"], t["wpk"], c["cout"], 1, addend=add, out=t["ybuf"], out_mul=2, out_off=(1, 0))
