"""Per-element reference tests for every bde_gemm kernel instance: conv_tma_kernel (gemm_tc_conv.cu), gemm_tc_kernel
(gemm_tc.cu) and gemm_simt_kernel (gemm_simt.cu), with the tile dispatcher restated in Python and asserted on every launch.

Exact operands.  Activations are integers in [-8, 8], weights integers in [-4, 4] times 2^-e, biases integers times
2^-e.  With K * 8 * 4 + max|b| <= 2^23 in units of 2^-e every bf16 operand, every product and every fp32 partial sum is
exact in any order, so the float64 reference (computed on the GPU with cuDNN off: im2col + dgemm, exact for integers)
is exact as well, and the kernel must match it bit for bit:
    fp32 output   got == ref
    bf16 output   got == ref.to(bfloat16)  (round to nearest even; |ref| runs well past 256, so odd integers are ties)
The store forms use e = 0 (ReLU6 uses a small e so that both clamps and the interior are hit).  Epilogues with a
nonlinearity (ConvLSTM, ConvGRU, GELU, sigmoid) keep the exact pre-activation, scaled by 2^-e into the range where the
nonlinearity bends, and are gated only for the epilogue's approximation (tanh.approx: relative 2^-11, so the
tanh-based sigmoid is off by at most 2^-12 absolute; the GELU quintic: GELU_FORM |h|; bf16 stores: half an ulp).
LayerNorm-gather instances (ln_mode) cannot be exact: they use the propagated per-element gate of the fused-attention
tests (fp32 two-pass statistics, bf16 rounding of x-hat).

Every case also checks that plausible mistakes FAIL: taps transposed (ky <-> kx), the neighbouring image's rows in the
halo instead of zeros, a0 and a1 swapped, the last 64-wide K block dropped.  That shows the operands are not degenerate.

Every output buffer is NaN-filled with NaN margins before and after the view: every element of the view must be written
and the margins must stay NaN.  A second launch of the same call must give identical bits.

expected_instance() restates the dispatch of gemm_tcgen05 / fill_params (gemm_tc.cu) and conv_tma_eligible /
conv_tma_launch (gemm_tc_conv.cu), including their environment switches and their dependence on the SM count; each GPU
case asserts that the profiler saw exactly that one GEMM instance.  Cases near a threshold derive their batch from the
SM count so that they stay on the intended side of it.  The test ids name all 84 instances of
profiles/sass/{gemm_tc_conv,gemm_tc,gemm_simt}.kernels.txt (test_instance_ids_cover_the_build); none is UNREACHABLE.

On a B200 (1000 W power limit) every exact case matched bit for bit (err/gate 0), including the two cases whose A
operand and output exceed 2^31 elements; the gated epilogues reached at most 0.98 of their gate (the bf16 half-ulp term,
tight by construction), and the file took 10 s including start-up.  The LayerNorm cases with c0 = 64 and an N tile of
at most 128 found the one-stage tile's epilogue staging running past its shared memory (fixed in TileCfg).
"""
import math
import os
import re
import zlib

import pytest
import torch
import torch.nn.functional as F

from test_gpu_fused_attention_mlp import U32, ln_ref, store, token_rows
from test_gpu_kernel_forms import BF, DEV, F64, GELU_FORM, R_BF16, TANH_APPROX, gpu, launched, pack

# bde2vid.h
EPI_STORE, EPI_LSTM, EPI_GRU_UR = 0, 1, 3
ACT_NONE, ACT_RELU, ACT_RELU6, ACT_GELU, ACT_SIGMOID = 0, 1, 2, 3, 4
E_SIG = 2.0 ** -12 + 8 * U32   # 0.5 tanh.approx(x / 2) + 0.5: absolute
TINY = 1e-300
MARGIN = 4096                  # NaN elements before and after every output view
B200_SMS = 148


# ---------------------------------------------------------------------------------------------------------------------
# instance names
# ---------------------------------------------------------------------------------------------------------------------
def inst_name(t):
    """("tma", BN, HALO, EPI, PAIR, NSUB) / ("tc", BN, TMA_B, DEEP, CH) / ("simt", T) -> the name in the SASS listings."""
    b = lambda v: "true" if v else "false"  # noqa: E731
    if t[0] == "tma":
        return "conv_tma_kernel<%d, %s, %d, %s, %d>" % (t[1], b(t[2]), t[3], b(t[4]), t[5])
    if t[0] == "tc":
        return "gemm_tc_kernel<%d, %s, %s, %d>" % (t[1], b(t[2]), b(t[3]), t[4])
    return "gemm_simt_kernel<%s>" % t[1]


_GEMM = re.compile(r"(conv_tma_kernel|gemm_tc_kernel|gemm_simt_kernel)(?:<([^<>()]*)>|I((?:L[ib]\d+E|f|13__nv_bfloat16)+)E)")


def gemm_instances(names):
    """Instance tuples of the bde_gemm kernels among ``names`` (demangled or mangled)."""
    out = set()
    for n in names:
        for m in _GEMM.finditer(n):
            base, dem, man = m.groups()
            if dem is not None:
                args = [a.strip() for a in dem.split(",")]
            else:
                args = []
                for k, v, f, bf in re.findall(r"L([ib])(\d+)E|(f)|13(__nv_bfloat16)", man):
                    args.append("float" if f else bf if bf else v if k == "i" else ("true" if v == "1" else "false"))
            tf = lambda s: s in ("true", "1")  # noqa: E731
            if base == "conv_tma_kernel" and len(args) == 5:
                out.add(("tma", int(args[0]), tf(args[1]), int(args[2]), tf(args[3]), int(args[4])))
            elif base == "gemm_tc_kernel" and len(args) == 4:
                out.add(("tc", int(args[0]), tf(args[1]), tf(args[2]), int(args[3])))
            elif base == "gemm_simt_kernel" and len(args) == 1:
                out.add(("simt", args[0]))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the dispatcher, restated
# ---------------------------------------------------------------------------------------------------------------------
def _cdiv(a, b):
    return -(-a // b)


def expected_instance(call, n_sm, env=None):
    """The instance bde_gemm launches for ``call`` on a part with ``n_sm`` SMs under the environment ``env``.
    call keys: engine ("tc" | "simt"), dtype ("bf16" | "f32"), n_img, h, w, c0, c1, n, k, s, pad, k_order, epi, act,
    out_f32, residual, ln."""
    env = env or {}

    def flag(name, dflt):                       # env_flag (gemm_tc.cu)
        v = env.get(name, "")
        return dflt if v == "" else v[0] == "1"

    def ival(name, dflt):                       # env_int (gemm_tc_conv.cu)
        v = env.get(name, "")
        return int(v) if v else dflt

    if call["engine"] == "simt":
        return ("simt", "float" if call["dtype"] == "f32" else "__nv_bfloat16")
    n_img, k, s, pad, N = call["n_img"], call["k"], call["s"], call["pad"], call["n"]
    c0, c1 = call["c0"], call["c1"]
    ho, wo = (call["h"] + 2 * pad - k) // s + 1, (call["w"] + 2 * pad - k) // s + 1
    ln, epi, out_f32, res = call["ln"], call["epi"], call["out_f32"], call["residual"]
    # conv_tma_eligible
    tma = not ln and flag("BDE2VID_CONV_TMA", True)
    if k == 1:
        tma = tma and s == 1 and pad == 0 and not out_f32 and not res and flag("BDE2VID_CONV_1X1", True)
    else:
        tma = tma and 3 <= k <= 5 and call["k_order"] == 1
    tma = tma and c0 % 64 == 0 and c1 % 64 == 0 and (s == 1 or (s == 2 and flag("BDE2VID_CONV_S2", True)))
    tma = tma and ho >= 8 and wo >= 8 and N % 32 == 0
    if tma:                                     # conv_tma_launch
        halo = s == 1 and flag("BDE2VID_CONV_HALO", True)
        swap = ival("BDE2VID_CONV_SWAP", 1) != 0
        d1, d2 = (ho, wo) if swap else (wo, ho)
        bn_max = 256 if N % 256 == 0 else 128 if N % 128 == 0 else 64 if N % 64 == 0 else 32
        nsub = 1
        if (halo and bn_max <= 128 and flag("BDE2VID_CONV_DUAL", True) and d2 > 16
                and n_img * _cdiv(d1, 8) * _cdiv(d2, 32) * (N // bn_max) >= n_sm):
            nsub = 2
        mt = n_img * _cdiv(d1, 8) * _cdiv(d2, 16 * nsub)
        pair = flag("BDE2VID_CONV_PAIR", False) and mt >= 2 and halo and bn_max == 256 and nsub == 1
        cs = 2 if pair else 1
        bn = bn_max
        while nsub == 1 and not pair and bn > 64 and 2 * _cdiv(mt, cs) * (N // bn) <= n_sm // cs:
            bn //= 2
        f = ival("BDE2VID_CONV_BN", 0)
        if f in (32, 64, 128, 256) and N % f == 0 and nsub == 1 and not pair:
            bn = f
        ep = 0
        if flag("BDE2VID_CONV_EPI_SPEC", True):
            if epi == EPI_LSTM:
                ep = 1
            elif epi == EPI_STORE and not out_f32 and not res and call["act"] in (ACT_NONE, ACT_RELU, ACT_RELU6):
                ep = 2
        return ("tma", bn, halo, ep, pair, nsub)
    # gemm_tcgen05 / fill_params
    tile2d = k > 1 and ho >= 8 and wo >= 16 and flag("BDE2VID_TC_TILE2D", True)
    m_tiles = n_img * _cdiv(wo, 16) * _cdiv(ho, 8) if tile2d else _cdiv(n_img * ho * wo, 128)
    K = k * k * (c0 + c1)
    num_kb = _cdiv(K, 64)
    bn = 128 if N % 128 == 0 else 64 if N % 64 == 0 else 32
    if N % 256 == 0 and K >= 512 and m_tiles * (N // 256) >= 100:
        bn = 256
    f = ival("BDE2VID_TC_BN", 0)
    if f in (32, 64, 128, 256) and N % f == 0:
        bn = f
    tma_b = not env.get("BDE2VID_TC_B_CPASYNC", "").startswith("1")
    if ln:
        bn = 256 if N % 256 == 0 else 192 if N % 192 == 0 else 128 if N % 128 == 0 else 64 if N % 64 == 0 else 32
        return ("tc", bn, tma_b, False, {1: 1, 2: 2}.get(c0 // 64, 4))
    small = m_tiles * (N // bn) <= n_sm and num_kb >= 8
    deep = (tile2d and flag("BDE2VID_TC_DEEP", False)) or (small and flag("BDE2VID_TC_DEEP_SMALL", True))
    return ("tc", bn, tma_b, deep, 0)


# ---------------------------------------------------------------------------------------------------------------------
# cases
# ---------------------------------------------------------------------------------------------------------------------
def case(inst, label, n_img, h, w, c0, n, k=3, s=1, c1=0, engine="tc", dtype="bf16", k_order=None, epi=EPI_STORE,
         act=ACT_NONE, out_f32=False, env=None, a0_ld=0, a1_ld=0):
    """One bde_gemm call.  ``n_img`` may be a function of the SM count (boundary cases)."""
    if k_order is None:
        k_order = 1 if (engine == "tc" and c0 % 64 == 0 and c1 % 64 == 0) else 0
    return dict(inst=inst, label=label, n_img=n_img, h=h, w=w, c0=c0, c1=c1, n=n, k=k, s=s, pad=k // 2, engine=engine,
                dtype=dtype, k_order=k_order, epi=epi, act=act, out_f32=out_f32, env=env or {}, a0_ld=a0_ld, a1_ld=a1_ld,
                residual=False, ln=False)


def resolve(cs, n_sm):
    r = dict(cs)
    if callable(r["n_img"]):
        r["n_img"] = r["n_img"](n_sm)
    return r


def _persistent_imgs(n_sm):
    """16 x 16 maps (2 tiles each): at least 3 x n_sm tiles and not a multiple of n_sm."""
    n = _cdiv(3 * n_sm, 2)
    return n + 1 if (2 * n) % n_sm == 0 else n


T, Fl = True, False
L, G = EPI_LSTM, EPI_GRU_UR
TMA_CASES = [
    # ---- tap mode (HALO = false): stride 2, or BDE2VID_CONV_HALO=0
    case(("tma", 32, Fl, 0, Fl, 1), "s2_33x45_c64+128", 2, 33, 45, 64, 96, s=2, c1=128, out_f32=True),
    case(("tma", 32, Fl, 1, Fl, 1), "s2_5x5_lstm", 2, 33, 33, 64, 96, k=5, s=2, epi=L),
    case(("tma", 32, Fl, 2, Fl, 1), "halo0_swap0_19x27", 3, 19, 27, 64, 32, env={"BDE2VID_CONV_HALO": "0", "BDE2VID_CONV_SWAP": "0"}),
    case(("tma", 64, Fl, 0, Fl, 1), "s2_pitched_a0", 2, 33, 33, 64, 64, s=2, out_f32=True, a0_ld=128),
    case(("tma", 64, Fl, 1, Fl, 1), "s2_lstm_35x50", 1, 35, 50, 128, 64, s=2, epi=L),
    case(("tma", 64, Fl, 2, Fl, 1), "s2_5x5_relu6", 2, 33, 33, 64, 192, k=5, s=2, act=ACT_RELU6),
    case(("tma", 128, Fl, 0, Fl, 1), "s2_gelu_bn128", 2, 33, 33, 64, 128, s=2, act=ACT_GELU, env={"BDE2VID_CONV_BN": "128"}),
    case(("tma", 128, Fl, 1, Fl, 1), "s2_lstm_many_tiles", lambda n: n // 12 + 1, 33, 33, 64, 128, s=2, epi=L),
    case(("tma", 128, Fl, 2, Fl, 1), "halo0_relu_bn128", 2, 20, 40, 64, 384, act=ACT_RELU,
         env={"BDE2VID_CONV_HALO": "0", "BDE2VID_CONV_BN": "128"}),
    case(("tma", 256, Fl, 0, Fl, 1), "s2_bn256", 2, 33, 33, 128, 256, s=2, out_f32=True, env={"BDE2VID_CONV_BN": "256"}),
    case(("tma", 256, Fl, 1, Fl, 1), "s2_lstm_many_tiles", lambda n: n // 12 + 1, 33, 33, 64, 256, s=2, epi=L),
    case(("tma", 256, Fl, 2, Fl, 1), "halo0_5x5_c192+64", 1, 17, 30, 192, 256, k=5, c1=64,
         env={"BDE2VID_CONV_HALO": "0", "BDE2VID_CONV_BN": "256"}),
    # ---- halo mode, one 8 x 16 tile per CTA
    case(("tma", 32, T, 0, Fl, 1), "swap0_21x35", 2, 21, 35, 64, 32, out_f32=True, env={"BDE2VID_CONV_SWAP": "0"}),
    case(("tma", 32, T, 1, Fl, 1), "lstm_c64+128_pitched_a1", 1, 17, 22, 64, 96, c1=128, a1_ld=192, epi=L),
    case(("tma", 32, T, 2, Fl, 1), "one_8x16_tile", 1, 8, 16, 64, 32),
    case(("tma", 64, T, 0, Fl, 1), "persistent_5x5_c256", _persistent_imgs, 16, 16, 256, 64, k=5, out_f32=True),
    case(("tma", 64, T, 1, Fl, 1), "lstm_c64+64", 1, 9, 19, 64, 64, c1=64, epi=L),
    case(("tma", 64, T, 2, Fl, 1), "1x1_relu", 2, 19, 26, 128, 64, k=1, act=ACT_RELU),
    case(("tma", 64, T, 2, Fl, 1), "dual_threshold_below", lambda n: _cdiv(n, 15) - 1, 40, 70, 64, 64),
    case(("tma", 128, T, 0, Fl, 1), "n256_narrowed_to_128", lambda n: n // 30, 33, 44, 64, 256, c1=64, out_f32=True),
    case(("tma", 128, T, 1, Fl, 1), "lstm_n128", lambda n: n // 30 + 1, 33, 44, 64, 128, c1=64, epi=L),
    case(("tma", 128, T, 2, Fl, 1), "5x5_relu6_bn128", 1, 40, 16, 64, 384, k=5, act=ACT_RELU6, env={"BDE2VID_CONV_BN": "128"}),
    case(("tma", 256, T, 0, Fl, 1), "n256_kept", lambda n: n // 30 + 1, 33, 44, 64, 256, out_f32=True),
    case(("tma", 256, T, 1, Fl, 1), "convlstm_gates", lambda n: n // 30 + 1, 33, 44, 64, 256, c1=64, epi=L),
    case(("tma", 256, T, 2, Fl, 1), "c192+64_pitched_a1_bn256", 1, 20, 36, 192, 256, c1=64, a1_ld=128,
         env={"BDE2VID_CONV_BN": "256"}),
    # ---- dual tiles (NSUB = 2)
    case(("tma", 32, T, 0, Fl, 2), "d2_40", lambda n: _cdiv(n, 6), 24, 40, 64, 32, out_f32=True),
    case(("tma", 32, T, 1, Fl, 2), "lstm_d2_40", lambda n: _cdiv(n, 18), 24, 40, 64, 96, epi=L),
    case(("tma", 32, T, 2, Fl, 2), "swap0_37x27", lambda n: _cdiv(n, 8), 37, 27, 64, 32, env={"BDE2VID_CONV_SWAP": "0"}),
    case(("tma", 64, T, 0, Fl, 2), "d2_40_c128", lambda n: _cdiv(n, 4), 16, 40, 128, 64, out_f32=True),
    case(("tma", 64, T, 1, Fl, 2), "lstm_40x70", lambda n: _cdiv(n, 15), 40, 70, 64, 64, epi=L),
    case(("tma", 64, T, 2, Fl, 2), "dual_threshold_above", lambda n: _cdiv(n, 15), 40, 70, 64, 64),
    case(("tma", 128, T, 0, Fl, 2), "d2_72", lambda n: _cdiv(n, 9), 24, 72, 64, 128, out_f32=True),
    case(("tma", 128, T, 1, Fl, 2), "lstm_33x44", lambda n: _cdiv(n, 10), 33, 44, 64, 128, epi=L),
    case(("tma", 128, T, 2, Fl, 2), "n384_relu", lambda n: _cdiv(n, 18), 17, 40, 64, 384, act=ACT_RELU),
    # ---- CTA pairs (cta_group::2)
    case(("tma", 256, T, 0, T, 1), "3_tiles_dummy", 1, 8, 48, 64, 256, out_f32=True, env={"BDE2VID_CONV_PAIR": "1"}),
    case(("tma", 256, T, 1, T, 1), "lstm_2_tiles", 1, 8, 32, 64, 256, c1=64, epi=L, env={"BDE2VID_CONV_PAIR": "1"}),
    case(("tma", 256, T, 2, T, 1), "33x44x3", 3, 33, 44, 128, 256, env={"BDE2VID_CONV_PAIR": "1"}),
]
CP = {"BDE2VID_TC_B_CPASYNC": "1"}
TC_CASES = [
    case(("tc", 32, T, Fl, 0), "ctot40_c24+16", 2, 19, 37, 24, 96, c1=16),
    case(("tc", 32, T, T, 0), "linear_6x10_small_grid", 5, 6, 10, 96, 32, out_f32=True),
    case(("tc", 32, Fl, Fl, 0), "dense_K200", 1, 1000, 1, 200, 32, k=1, env=CP),
    case(("tc", 32, Fl, T, 0), "deep_env_c32+64", 2, 24, 40, 32, 96, c1=64, out_f32=True,
         env=dict(CP, BDE2VID_TC_DEEP="1")),
    case(("tc", 64, T, Fl, 0), "dense_gelu", 1, 1000, 1, 192, 192, k=1, act=ACT_GELU),
    case(("tc", 64, T, T, 0), "linear_5x5_relu6", 3, 7, 7, 64, 64, k=5, act=ACT_RELU6),
    case(("tc", 64, Fl, Fl, 0), "s2_ctot40_sigmoid", 3, 33, 33, 40, 64, s=2, act=ACT_SIGMOID, env=CP),
    case(("tc", 64, Fl, T, 0), "deep_env_lstm", 2, 20, 36, 64, 64, c1=64, k_order=0, epi=L,
         env=dict(CP, BDE2VID_TC_DEEP="1")),
    case(("tc", 128, T, Fl, 0), "c64+64_kmajor", lambda n: n // 12 + 1, 22, 50, 64, 128, c1=64, k_order=0, out_f32=True),
    case(("tc", 128, T, Fl, 0), "bn256_rule_99_tiles", 1, 72, 176, 64, 256, k_order=0, out_f32=True),
    case(("tc", 128, T, Fl, 0), "small_grid_plus_1", lambda n: n * 128 + 1, 1, 1, 512, 128, k=1, out_f32=True),
    case(("tc", 128, T, T, 0), "small_grid_exact", lambda n: n * 128, 1, 1, 512, 128, k=1, out_f32=True),
    case(("tc", 128, T, T, 0), "deep_env_5x5_gru", 2, 17, 33, 16, 384, k=5, c1=8, epi=G, env={"BDE2VID_TC_DEEP": "1"}),
    case(("tc", 128, Fl, Fl, 0), "dense_f32", 1, 700, 1, 256, 128, k=1, out_f32=True, env=CP),
    case(("tc", 128, Fl, T, 0), "dense_small_grid", 1, 256, 1, 512, 128, k=1, env=CP),
    case(("tc", 256, T, Fl, 0), "bn256_rule_200_tiles", lambda n: n // 100 + 1, 80, 160, 64, 256, k_order=0, out_f32=True),
    case(("tc", 256, T, T, 0), "bn256_rule_100_tiles_small_grid", 1, 80, 160, 64, 256, k_order=0, out_f32=True),
    case(("tc", 256, T, T, 0), "bn_env_deep_env", 2, 16, 32, 40, 256, env={"BDE2VID_TC_BN": "256", "BDE2VID_TC_DEEP": "1"}),
    case(("tc", 256, Fl, Fl, 0), "dense_bn_env", 1, 300, 1, 64, 512, k=1, out_f32=True,
         env=dict(CP, BDE2VID_TC_BN="256")),
    case(("tc", 256, Fl, T, 0), "dense_100_tiles_small_grid", 1, 100 * 128 - 5, 1, 512, 256, k=1, out_f32=True, env=CP),
]
SIMT_CASES = [
    case(("simt", "float"), "c24+16_n100", 2, 13, 17, 24, 100, c1=16, engine="simt", dtype="f32", out_f32=True),
    case(("simt", "float"), "lstm", 2, 11, 14, 32, 64, c1=32, engine="simt", dtype="f32", epi=L),
    case(("simt", "__nv_bfloat16"), "5x5_chunk_major", 2, 15, 21, 64, 64, k=5, engine="simt", k_order=1),
]
CONV_CASES = TMA_CASES + TC_CASES + SIMT_CASES


def case_id(cs):
    return "%s-%s" % (inst_name(cs["inst"]), cs["label"])


# LayerNorm-gather instances: (N -> BN) x c0 -> CH x weight tile by TMA or cp.async
LN_N = {32: 96, 64: 320, 128: 128, 192: 192, 256: 256}


def _ln_cases():
    out = []
    i = 0
    for bn, N in sorted(LN_N.items()):
        for c0 in (64, 128, 256):
            for tma_b in (True, False):
                D = i % 8 + 1
                ntok = 49 if i % 2 == 0 else 1
                nwin = (3 + i % 4) if ntok == 49 else 150 + 7 * i
                if (nwin * D * ntok) % 128 == 0:
                    nwin += 1
                ident = D == 1 and i % 4 == 0      # ln_tok_map = NULL: plain rows
                out.append(dict(inst=("tc", bn, tma_b, False, {64: 1, 128: 2, 256: 4}[c0]), N=N, c0=c0, D=D, ntok=ntok,
                                nwin=nwin, ident=ident, none_slot=(i % D) if D > 1 else None, out_f32=i % 3 != 0,
                                env={} if tma_b else dict(CP), label="D%d_ntok%d_rows%d" % (D, ntok, nwin * D * ntok)))
                i += 1
    return out


LN_CASES = _ln_cases()


def ln_call(lc):
    return dict(engine="tc", dtype="bf16", n_img=1, h=lc["nwin"] * lc["D"] * lc["ntok"], w=1, c0=lc["c0"], c1=0,
                n=lc["N"], k=1, s=1, pad=0, k_order=0, epi=EPI_STORE, act=ACT_NONE, out_f32=lc["out_f32"],
                residual=False, ln=True)


# 64-bit addressing: A operand and output each hold more than 2^31 elements (8200 images x 64 x 64 x 64 channels)
BIG_CASES = [
    case(("tma", 64, T, 2, Fl, 2), "beyond_2^31", 8200, 64, 64, 64, 64),
    case(("tc", 64, T, Fl, 0), "beyond_2^31", 8200, 64, 64, 64, 64, k_order=0),
]

# instances no legal call can reach, with the reason
UNREACHABLE = {}


# ---------------------------------------------------------------------------------------------------------------------
# operands and references
# ---------------------------------------------------------------------------------------------------------------------
def _seed(label):
    return zlib.crc32(label.encode()) & 0x7FFFFFFF


def _exact_store(cs):
    return cs["epi"] == EPI_STORE and cs["act"] in (ACT_NONE, ACT_RELU)


def conv_rows(x, w, b, s, pad):
    """float64 convolution as rows [M, N] in NHWC pixel order; cuDNN off (im2col + dgemm: exact for integers)."""
    with torch.backends.cudnn.flags(enabled=False):
        y = F.conv2d(x, w, b, stride=s, padding=pad)
    return y.permute(0, 2, 3, 1).reshape(-1, w.shape[0])


def halo_from_neighbours(x, pad):
    """x with its top / bottom padding taken from the previous / next image instead of zeros (the flat-index mistake)."""
    z = torch.zeros_like(x[:1])
    prev = torch.cat([z, x[:-1]])[:, :, x.shape[2] - pad:, :]
    nxt = torch.cat([x[1:], z])[:, :, :pad, :]
    return torch.cat([prev, x, nxt], 2)


def last_block_mask(ci, k, k_order, K):
    """Boolean [ci * k * k] over the unpacked weight (c, ky, kx) that marks the columns of the last 64-wide K block."""
    idx = (torch.arange(ci * k * k, dtype=torch.float32) + 1).view(1, ci, k, k)
    pk, _ = pack(idx, torch.float32, k_order == 1)
    cols = pk[0, 64 * ((K - 1) // 64):K].long().cpu() - 1
    m = torch.zeros(ci * k * k, dtype=torch.bool)
    m[cols] = True
    return m


class Operands:
    """Device operands of one call and their float64 values (on the device)."""

    def __init__(self, cs, imgs=None):
        g = torch.Generator(device=DEV).manual_seed(_seed(case_id(cs)))
        n, h, w, c0, c1, N, k = cs["n_img"], cs["h"], cs["w"], cs["c0"], cs["c1"], cs["n"], cs["k"]
        ci = c0 + c1
        K = k * k * ci
        dt = torch.float32 if cs["dtype"] == "f32" else BF
        self.K = K
        if _exact_store(cs):
            e = 0
        else:   # pre-activation std ~ 3: where the nonlinearities bend (ReLU6: both clamps and the interior)
            e = max(0, round(math.log2(12.6 * math.sqrt(K) / 3.0)))
        assert K * 32 + 64 <= 2 ** 23
        self.scale = 2.0 ** -e

        def ints(shape, lo, hi, dtype):
            return torch.randint(lo, hi + 1, shape, generator=g, device=DEV, dtype=torch.int8).to(dtype)

        # every operand lives at the start of a larger allocation, so that a read past its end (up to one image or
        # one 128-row tile) stays inside the allocation and shows up as a wrong value
        extra = max(2, _cdiv(128, h * w) + 1)

        def source(c, ld):
            if ld:   # channel slice [ld - c, ld) of a wider map; the other channels hold values the kernel must not read
                full = torch.full((n + extra, h, w, ld), 100.0, dtype=dt, device=DEV)
                full[..., ld - c:] = ints((n + extra, h, w, c), -8, 8, dt)
                return full[:n, ..., ld - c:]
            return ints((n + extra, h, w, c), -8, 8, dt)[:n]

        self.a0 = source(c0, cs["a0_ld"])
        self.a1 = source(c1, cs["a1_ld"]) if c1 else None
        wt = ints((N, ci, k, k), -4, 4, F64) * self.scale
        self.wt = wt
        self.b64 = ints((N,), -64, 64, F64) * self.scale
        self.b = self.b64.float()
        self.w, self.ld = pack(wt, dt, cs["k_order"] == 1)
        ho = (h + 2 * cs["pad"] - k) // cs["s"] + 1
        wo = (w + 2 * cs["pad"] - k) // cs["s"] + 1
        self.M, self.hw = n * ho * wo, ho * wo
        self.tail_rows = 128 + self.hw      # rows past the end a wrong tile mapping can reach: one tile, one image
        hid = N // 4 if cs["epi"] == EPI_LSTM else N // 2 if cs["epi"] == EPI_GRU_UR else N
        self.hid = hid
        self.cprev = None
        if cs["epi"] in (EPI_LSTM, EPI_GRU_UR):   # c_prev / h_prev in [-2, 2], exact in fp32
            self.cprev = (ints((self.M + self.tail_rows, hid), -16, 16, torch.float32) / 8)[:self.M]
        self.imgs = list(range(n)) if imgs is None else imgs

    def x64(self, imgs=None):
        imgs = self.imgs if imgs is None else imgs
        xs = [self.a0[imgs]] + ([self.a1[imgs]] if self.a1 is not None else [])
        return torch.cat([t.to(F64) for t in xs], -1).permute(0, 3, 1, 2)

    def rows(self, imgs):
        """Output row indices of the images ``imgs``."""
        return torch.cat([torch.arange(i * self.hw, (i + 1) * self.hw, device=DEV) for i in imgs])


def pre_ref(cs, op, wrong=None):
    """Exact pre-activation rows [M', N] (M' = rows of op.imgs); ``wrong`` names a plausible mistake."""
    x, wt, s, pad = op.x64(), op.wt, cs["s"], cs["pad"]
    if wrong == "taps_transposed":
        wt = wt.transpose(-1, -2)
    elif wrong == "a0_a1_swapped":
        c0 = cs["c0"]
        x = torch.cat([x[:, c0:], x[:, :c0]], 1)
    elif wrong == "last_k_block_dropped":
        m = last_block_mask(wt.shape[1], cs["k"], cs["k_order"], op.K).to(DEV)
        wt = (wt.reshape(wt.shape[0], -1) * (~m).to(F64)).view_as(wt)
    elif wrong == "neighbour_halo":
        x = halo_from_neighbours(x, pad)
        return conv_rows(x, wt, op.b64, s, (0, pad))
    return conv_rows(x, wt, op.b64, s, pad)


def wrongs_of(cs, op):
    out = ["last_k_block_dropped"]
    if cs["k"] > 1:
        assert not torch.equal(op.wt, op.wt.transpose(-1, -2))
        out.append("taps_transposed")
    if len(op.imgs) >= 2 and cs["pad"] > 0:
        out.append("neighbour_halo")
    if cs["c1"] and cs["c1"] == cs["c0"]:
        out.append("a0_a1_swapped")
    return out


def expected_outputs(cs, op, pre):
    """{output name: (reference, gate or None for an exact comparison)} from the pre-activation rows."""
    bf = cs["dtype"] == "bf16"
    r = R_BF16 if bf else 0.0
    if cs["epi"] == EPI_LSTM:
        cp = op.cprev[op.rows(op.imgs)].to(F64) if len(op.imgs) != cs["n_img"] else op.cprev.to(F64)
        si, sf, so, tg = torch.sigmoid(pre[:, 0::4]), torch.sigmoid(pre[:, 1::4]), torch.sigmoid(pre[:, 2::4]), torch.tanh(pre[:, 3::4])
        c = sf * cp + si * tg
        tc = torch.tanh(c)
        h = so * tc
        e_c = E_SIG * (cp.abs() + tg.abs()) + si * tg.abs() * TANH_APPROX + 4 * U32 * ((sf * cp).abs() + (si * tg).abs())
        e_h = E_SIG * tc.abs() + so * (TANH_APPROX * tc.abs() + e_c) + 4 * U32 * h.abs()
        return {"out": (h, r * h.abs() + 1.01 * e_h + TINY), "c": (c, e_c + U32 * c.abs() + TINY)}
    if cs["epi"] == EPI_GRU_UR:
        hp = op.cprev.to(F64)
        u, hr = torch.sigmoid(pre[:, 0::2]), hp * torch.sigmoid(pre[:, 1::2])
        e_hr = hp.abs() * E_SIG + 4 * U32 * hr.abs()
        return {"out": (hr, r * hr.abs() + 1.01 * e_hr + TINY), "c": (u, E_SIG + TINY)}
    act = cs["act"]
    if act in (ACT_NONE, ACT_RELU, ACT_RELU6):
        ref = pre if act == ACT_NONE else pre.clamp(min=0.0) if act == ACT_RELU else pre.clamp(0.0, 6.0)
        return {"out": (ref, None)}
    if act == ACT_GELU:
        ref = F.gelu(pre)
        e = (GELU_FORM + 0.5 * TANH_APPROX + 16 * U32) * pre.abs()
    else:
        ref = torch.sigmoid(pre)
        e = 16 * U32 * ref.abs()
    out_r = 0.0 if cs["out_f32"] else r
    return {"out": (ref, out_r * ref.abs() + 1.01 * e + TINY)}


# ---------------------------------------------------------------------------------------------------------------------
# outputs, launch, comparison
# ---------------------------------------------------------------------------------------------------------------------
class Out:
    """A [rows, cols] view into a NaN-filled buffer with NaN margins on both sides; the one after the view holds at
    least ``tail_rows`` rows, so that a stray write past the end stays inside the buffer and is seen."""

    def __init__(self, rows, cols, dtype, tail_rows=128):
        self.tail = max(MARGIN, tail_rows * cols)
        self.buf = torch.full((MARGIN + rows * cols + self.tail,), float("nan"), dtype=dtype, device=DEV)
        self.view = self.buf[MARGIN:MARGIN + rows * cols].view(rows, cols)

    def verify(self, name):
        n_unwritten = int(torch.isnan(self.view).sum())
        assert n_unwritten == 0, "%s: %d elements of the output were not written" % (name, n_unwritten)
        n_stray = int((~torch.isnan(self.buf[:MARGIN])).sum() + (~torch.isnan(self.buf[-self.tail:])).sum())
        assert n_stray == 0, "%s: %d writes landed outside the output view" % (name, n_stray)

    def untouched(self):
        return bool(torch.isnan(self.buf).all())


def alloc_outputs(cs, op):
    dt = torch.float32 if cs["dtype"] == "f32" else BF
    if cs["epi"] in (EPI_LSTM, EPI_GRU_UR):
        return {"out": Out(op.M, op.hid, dt, op.tail_rows), "c": Out(op.M, op.hid, torch.float32, op.tail_rows)}
    return {"out": Out(op.M, cs["n"], torch.float32 if cs["out_f32"] else dt, op.tail_rows)}


def launch(cs, op, outs):
    from bde2vid_b200 import ops
    kw = dict(n_img=cs["n_img"], h_in=cs["h"], w_in=cs["w"], c0=cs["c0"], n=cs["n"], ksize=cs["k"], stride=cs["s"],
              pad=cs["pad"], w_ld=op.ld, epi=cs["epi"], act=cs["act"], out_f32=cs["out_f32"], k_order=cs["k_order"],
              engine=ops.ENGINE_SIMT if cs["engine"] == "simt" else ops.ENGINE_TCGEN05,
              dtype=torch.float32 if cs["dtype"] == "f32" else BF, a0_ld=cs["a0_ld"], a1_ld=cs["a1_ld"])
    if cs["c1"]:
        kw.update(a1=op.a1, c1=cs["c1"])
    if "c" in outs:
        kw.update(c_prev=op.cprev, c_out=outs["c"].view)
    ops.gemm(op.a0, op.w, op.b, outs["out"].view, **kw)


def clear_switches(monkeypatch, env):
    for k in list(os.environ):
        if k.startswith("BDE2VID_CONV_") or k.startswith("BDE2VID_TC_"):
            monkeypatch.delenv(k)
    for k, v in env.items():
        monkeypatch.setenv(k, v)


def run_routed(fn, inst):
    """fn() under the profiler; assert that exactly one GEMM instance ran and that it is ``inst``."""
    _, names = launched(fn)
    gemm_names = [n for n in names if re.search(r"conv_tma_kernel|gemm_tc_kernel|gemm_simt_kernel", n)]
    got = gemm_instances(gemm_names)
    assert got == {inst} and len(gemm_names) == 1, (inst_name(inst), sorted(gemm_names))


def compare(name, got, ref, gate, dtype, wrongs=()):
    """Exact (gate None: got == ref rounded to the output type) or gated per-element comparison; every wrong reference
    in ``wrongs`` (name, reference) must fail it.  Returns the largest err / gate (0 for a passing exact case)."""
    got = got.to(F64)
    if gate is None:
        want = ref.to(dtype).to(F64)
        bad = got != want
        nb = int(bad.sum())
        if nb:
            i = int(bad.reshape(-1).nonzero()[0])
            raise AssertionError("%s: %d of %d elements differ; first at flat index %d: got %r, want %r (exact %r)"
                                 % (name, nb, got.numel(), i, float(got.reshape(-1)[i]), float(want.reshape(-1)[i]),
                                    float(ref.reshape(-1)[i])))
        for wn, wr in wrongs:
            assert (got != wr.to(dtype).to(F64)).any(), "%s: the wrong reference '%s' matches too" % (name, wn)
        return 0.0
    ratio = float(((got - ref).abs() / gate).max())
    assert ratio <= 1.0, "%s: err/gate %.3f" % (name, ratio)
    for wn, wr in wrongs:
        rw = float(((got - wr).abs() / gate).max())
        assert rw > 1.0, "%s: the wrong reference '%s' passes the gate too (err/gate %.3f)" % (name, wn, rw)
    return ratio


def check_case(cs, op, outs, wrong_pres=()):
    name = case_id(cs)
    pre = pre_ref(cs, op)
    exp = expected_outputs(cs, op, pre)
    wexp = [(wn, expected_outputs(cs, op, wp)) for wn, wp in wrong_pres]
    worst = 0.0
    rows = op.rows(op.imgs) if len(op.imgs) != cs["n_img"] else None
    for key, (ref, gate) in exp.items():
        o = outs[key]
        o.verify("%s %s" % (name, key))
        got = o.view if rows is None else o.view[rows]
        wr = [(wn, we[key][0]) for wn, we in wexp]
        worst = max(worst, compare("%s %s" % (name, key), got, ref, gate, o.view.dtype, wr))
        if gate is None and o.view.dtype == BF and cs["act"] == ACT_NONE:
            # real rounding happened, ties included: odd integers beyond 256
            assert ((ref.abs() > 256) & (torch.remainder(ref, 2) == 1)).any(), name
    print("%-90s err/gate %.3f" % (name, worst))


# ---------------------------------------------------------------------------------------------------------------------
# GPU cases
# ---------------------------------------------------------------------------------------------------------------------
def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


@gpu
@pytest.mark.parametrize("cs", CONV_CASES, ids=case_id)
def test_gemm_instance(cs, monkeypatch):
    """One bde_gemm call per case: the instance the dispatcher restatement predicts is the one that runs, the outputs
    match the exact reference (or the epilogue gate) in every element, nothing outside the outputs is written, the
    plausible mistakes fail, and a second launch is bit-identical."""
    cs = resolve(cs, sm_count())
    clear_switches(monkeypatch, cs["env"])
    inst = expected_instance(cs, sm_count(), cs["env"])
    assert inst == cs["inst"], (inst_name(inst), inst_name(cs["inst"]))
    op = Operands(cs)
    outs = alloc_outputs(cs, op)
    run_routed(lambda: launch(cs, op, outs), inst)
    check_case(cs, op, outs, [(wn, pre_ref(cs, op, wn)) for wn in wrongs_of(cs, op)])
    again = alloc_outputs(cs, op)
    launch(cs, op, again)
    for key in outs:
        assert torch.equal(outs[key].buf.view(torch.uint8), again[key].buf.view(torch.uint8)), "repeat launch differs"


@gpu
@pytest.mark.parametrize("lc", LN_CASES, ids=lambda lc: "%s-%s" % (inst_name(lc["inst"]), lc["label"]))
def test_ln_gather_instance(lc, monkeypatch):
    """LayerNorm-gather A operand (ln_mode): rows m = (win * D + d) * n_tok + tok of frame d through the token map, None
    frames and -1 tokens as zero rows.  Gate: the propagated bound of the fp32 two-pass statistics and the bf16 x-hat
    (ln_ref / store of the fused-attention tests), then E_ACC of the product's mass."""
    from bde2vid_b200 import ops
    from test_gpu_kernel_forms import E_ACC
    clear_switches(monkeypatch, lc["env"])
    name = "%s-%s" % (inst_name(lc["inst"]), lc["label"])
    call = ln_call(lc)
    inst = expected_instance(call, sm_count(), lc["env"])
    assert inst == lc["inst"], (inst_name(inst), name)
    g = torch.Generator().manual_seed(_seed(name))
    C, N, D, ntok, nwin = lc["c0"], lc["N"], lc["D"], lc["ntok"], lc["nwin"]
    P = 97
    frames = [token_rows(P, C, g).to(DEV) for _ in range(D)]
    if lc["none_slot"] is not None:
        frames[lc["none_slot"]] = None
    M = nwin * D * ntok
    if lc["ident"]:
        frames = [token_rows(M, C, g).to(DEV)]
        tmap = None
        x = frames[0].to(F64)
    else:
        tm = torch.randint(0, P, (nwin, ntok), generator=g)
        tm[torch.rand(nwin, ntok, generator=g) < 0.15] = -1
        tmap = tm.to(torch.int32).to(DEV)
        x = torch.zeros(nwin, D, ntok, C, dtype=F64, device=DEV)
        for d, f in enumerate(frames):
            if f is not None:
                x[:, d] = f.to(F64)[tm.clamp(min=0).to(DEV)] * (tm >= 0).to(DEV).unsqueeze(-1).to(F64)
        x = x.reshape(M, C)
    w = (torch.randint(-4, 5, (N, C), generator=g).to(F64) / 32).to(DEV)
    b = (torch.randint(-64, 65, (N,), generator=g).to(F64) / 32).to(DEV)
    pw, ld = pack(w.view(N, C, 1, 1), BF, False)
    out = Out(M, N, torch.float32 if lc["out_f32"] else BF)

    def run():
        ops.gemm(None, pw, b.float(), out.view, n_img=1, h_in=M, w_in=1, c0=C, n=N, w_ld=ld, out_f32=lc["out_f32"],
                 engine=ops.ENGINE_TCGEN05, dtype=BF, ln_frames=frames, ln_tok_map=tmap, ln_n_tok=ntok)
    run_routed(run, inst)
    out.verify(name)
    xhat, e_x = ln_ref(x)
    xr, dx = store(xhat, e_x, BF)

    def lin(wm):
        a = xr @ wm.t() + b
        e = E_ACC * (xr.abs() @ wm.abs().t() + b.abs()) + dx @ wm.abs().t()
        return a, e
    a, e = lin(w)
    if lc["out_f32"]:
        ref, gate = a, e + U32 * a.abs() + TINY
    else:
        ref, gate = store(a, e, BF)
        gate = gate + TINY
    w_drop = w.clone()
    w_drop[:, C - 64:] = 0
    wrong = lin(w_drop)[0]
    r = compare(name, out.view, ref, gate, out.view.dtype, [("last_k_block_dropped", wrong)])
    print("%-90s err/gate %.3f" % (name, r))
    first, out = out, Out(M, N, out.view.dtype)       # run() writes to the new buffer
    run()
    assert torch.equal(first.buf.view(torch.uint8), out.buf.view(torch.uint8)), "repeat launch differs"


@gpu
@pytest.mark.parametrize("cs", BIG_CASES, ids=case_id)
def test_gemm_beyond_2_31_elements(cs, monkeypatch):
    """A operand and output of more than 2^31 elements each: the 64-bit address arithmetic.  Compares the first image,
    the images just before and after the 2^31-element mark and the last one, exactly; every output element must be
    written and the margins untouched."""
    free, _ = torch.cuda.mem_get_info()
    need = 24 << 30
    if free < need:
        print("skipped: %.1f GB free, %.1f GB needed" % (free / 2 ** 30, need / 2 ** 30))
        pytest.skip("%.1f GB of device memory free, %.1f GB needed" % (free / 2 ** 30, need / 2 ** 30))
    clear_switches(monkeypatch, cs["env"])
    inst = expected_instance(cs, sm_count(), cs["env"])
    assert inst == cs["inst"], inst_name(inst)
    per_img = cs["h"] * cs["w"] * cs["c0"]
    mark = (1 << 31) // per_img
    op = Operands(cs, imgs=[0, mark - 1, mark, mark + 1, cs["n_img"] - 1])
    assert op.a0.numel() > (1 << 31) and op.M * cs["n"] > (1 << 31)
    outs = alloc_outputs(cs, op)
    run_routed(lambda: launch(cs, op, outs), inst)
    check_case(cs, op, outs)
    del outs, op
    torch.cuda.empty_cache()


@gpu
def test_refused_calls(monkeypatch):
    """Calls the tcgen05 engine cannot serve raise RuntimeError and leave the NaN-filled output untouched."""
    from bde2vid_b200 import _lib, ops
    clear_switches(monkeypatch, {})
    g = torch.Generator(device=DEV).manual_seed(7)
    x = torch.randint(-8, 9, (1, 16, 16, 256), generator=g, device=DEV).to(BF)
    wbuf = torch.randint(-4, 5, (512 * 1664 + 64,), generator=g, device=DEV).to(BF)
    bias = torch.zeros(512, device=DEV)
    frames = [torch.randn(64, 96, generator=g, device=DEV)]

    def call(N=64, c0=64, k=3, w_ld=None, w_off=0, a0_ld=0, k_order=1, src=None):
        K = k * k * c0
        ld = w_ld if w_ld is not None else _cdiv(K, 64) * 64
        w = wbuf[w_off:w_off + N * ld].view(N, ld)
        a0 = (x[..., :c0].contiguous() if src is None else src)
        out = Out(16 * 16, N, BF)
        with pytest.raises(RuntimeError):
            ops.gemm(a0, w, bias, out.view, n_img=1, h_in=16, w_in=16, c0=c0, n=N, ksize=k, pad=k // 2, w_ld=ld,
                     engine=ops.ENGINE_TCGEN05, dtype=BF, k_order=k_order, a0_ld=a0_ld)
        assert out.untouched()

    call(N=48)                                      # N % 32 != 0
    call(k=1, w_ld=96)                              # w_ld not a multiple of 64
    call(w_ld=512)                                  # w_ld < K (576)
    call(w_off=32)                                  # weights 64 bytes past a 128-byte boundary
    call(c0=12, k_order=0)                          # c % 8 != 0
    call(k=7, c0=64)                                # 7 x 7
    call(k_order=0, a0_ld=128, src=x[..., :128][..., 64:])   # pitched source on the gemm_tc_kernel route
    # LayerNorm mode: c0 = 96, and ln_D = 9 (beyond the descriptor's 8 frame slots: raw descriptor)
    out = Out(64, 64, torch.float32)
    w = wbuf[:64 * 128].view(64, 128)
    with pytest.raises(RuntimeError):
        ops.gemm(None, w, bias, out.view, n_img=1, h_in=64, w_in=1, c0=96, n=64, w_ld=128, out_f32=True,
                 engine=ops.ENGINE_TCGEN05, dtype=BF, ln_frames=frames)
    assert out.untouched()
    lib = _lib.require_device()
    f64 = torch.randn(64, 64, generator=g, device=DEV)
    d = _lib.GemmDesc()
    d.engine, d.dtype = ops.ENGINE_TCGEN05, _lib.BDE_DTYPE[BF]
    d.ln_mode, d.ln_D, d.ln_n_tok = 1, 9, 1
    for i in range(8):
        d.ln_frames[i] = f64.data_ptr()
    d.c0, d.n_img, d.h_in, d.w_in, d.h_out, d.w_out, d.ksize, d.stride = 64, 1, 64, 1, 64, 1, 1, 1
    d.w, d.bias, d.n, d.w_ld = _lib.ptr(wbuf[:64 * 64].view(64, 64)), _lib.ptr(bias), 64, 64
    d.out_f32, d.out = 1, _lib.ptr(out.view)
    with pytest.raises(RuntimeError):
        _lib.check(lib.bde_gemm(_lib.C.byref(d), _lib.stream_ptr()), "bde_gemm")
    torch.cuda.synchronize()
    assert out.untouched()


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def _call(n_img, h, w, c0, n, k=3, s=1, c1=0, engine="tc", k_order=1, epi=EPI_STORE, act=ACT_NONE, out_f32=False,
          ln=False):
    return dict(engine=engine, dtype="bf16", n_img=n_img, h=h, w=w, c0=c0, c1=c1, n=n, k=k, s=s, pad=k // 2,
                k_order=k_order, epi=epi, act=act, out_f32=out_f32, residual=False, ln=ln)


# (call, env, instance) worked out by hand from gemm_tc_conv.cu / gemm_tc.cu for a 148-SM B200
DISPATCH_TABLE = [
    # dual tiles: 10 images x 5 x 3 tile pairs = 150 >= 148; 9 images: 135
    (_call(10, 40, 70, 64, 64), {}, ("tma", 64, True, 2, False, 2)),
    (_call(9, 40, 70, 64, 64), {}, ("tma", 64, True, 2, False, 1)),
    (_call(10, 40, 70, 64, 64), {"BDE2VID_CONV_DUAL": "0"}, ("tma", 64, True, 2, False, 1)),
    # ConvLSTM gates, N = 256 on 33 x 44 (15 tiles per image): narrowed while 2 x tiles x N / BN <= 148
    (_call(1, 33, 44, 64, 256, c1=64, epi=EPI_LSTM), {}, ("tma", 64, True, 1, False, 1)),
    (_call(4, 33, 44, 64, 256, c1=64, epi=EPI_LSTM), {}, ("tma", 128, True, 1, False, 1)),
    (_call(5, 33, 44, 64, 256, c1=64, epi=EPI_LSTM), {}, ("tma", 256, True, 1, False, 1)),
    (_call(1, 33, 44, 64, 256, c1=64, epi=EPI_LSTM), {"BDE2VID_CONV_BN": "256"}, ("tma", 256, True, 1, False, 1)),
    (_call(1, 33, 44, 64, 256, c1=64, epi=EPI_LSTM), {"BDE2VID_CONV_EPI_SPEC": "0"}, ("tma", 64, True, 0, False, 1)),
    (_call(1, 33, 44, 64, 256, c1=64), {"BDE2VID_CONV_PAIR": "1"}, ("tma", 256, True, 2, True, 1)),
    (_call(1, 8, 16, 64, 256), {"BDE2VID_CONV_PAIR": "1"}, ("tma", 64, True, 2, False, 1)),   # one tile: no pair
    # store epilogue: fp32 output / GELU -> generic; stride 2 / HALO=0 -> tap mode
    (_call(1, 33, 44, 64, 64, out_f32=True), {}, ("tma", 64, True, 0, False, 1)),
    (_call(1, 33, 44, 64, 64, act=ACT_GELU), {}, ("tma", 64, True, 0, False, 1)),
    (_call(1, 33, 44, 64, 64, act=ACT_RELU6), {}, ("tma", 64, True, 2, False, 1)),
    (_call(1, 33, 44, 64, 96, s=2), {}, ("tma", 32, False, 2, False, 1)),
    (_call(1, 33, 44, 64, 64), {"BDE2VID_CONV_HALO": "0"}, ("tma", 64, False, 2, False, 1)),
    # h_out 8 vs 7: the edge of TMA-conv eligibility (7 rows: linear M tiles, 9 K blocks, 1 CTA -> deep)
    (_call(1, 8, 20, 64, 64), {}, ("tma", 64, True, 2, False, 1)),
    (_call(1, 7, 20, 64, 64), {}, ("tc", 64, True, True, 0)),
    (_call(1, 8, 20, 64, 64, k_order=0), {}, ("tc", 64, True, True, 0)),
    (_call(1, 8, 20, 64, 64), {"BDE2VID_CONV_TMA": "0"}, ("tc", 64, True, True, 0)),
    (_call(1, 8, 20, 96, 64, k_order=0), {}, ("tc", 64, True, True, 0)),
    (_call(1, 16, 16, 64, 64, k=7, k_order=0), {}, ("tc", 64, True, True, 0)),
    # gemm_tc BN = 256: N % 256 == 0, K >= 512, m_tiles * N / 256 >= 100
    (_call(2, 80, 160, 64, 256, k_order=0), {}, ("tc", 256, True, False, 0)),
    (_call(1, 80, 160, 64, 256, k_order=0), {}, ("tc", 256, True, True, 0)),         # 100 CTAs <= 148, 9 K blocks: deep
    (_call(1, 72, 176, 64, 256, k_order=0), {}, ("tc", 128, True, False, 0)),
    (_call(1, 80, 160, 56, 256, k_order=0), {}, ("tc", 128, True, False, 0)),       # K = 504
    (_call(1, 80, 160, 64, 256, k_order=0), {"BDE2VID_TC_BN": "64"}, ("tc", 64, True, False, 0)),
    (_call(1, 80, 160, 64, 256, k_order=0), {"BDE2VID_TC_BN": "96"}, ("tc", 256, True, True, 0)),
    # small-grid deep: m_tiles * N / BN <= 148 and num_kb >= 8
    (_call(1, 148 * 128, 1, 512, 128, k=1, out_f32=True), {}, ("tc", 128, True, True, 0)),
    (_call(1, 148 * 128 + 1, 1, 512, 128, k=1, out_f32=True), {}, ("tc", 128, True, False, 0)),
    (_call(1, 148 * 128, 1, 448, 128, k=1, out_f32=True), {}, ("tc", 128, True, False, 0)),
    (_call(1, 148 * 128, 1, 512, 128, k=1, out_f32=True), {"BDE2VID_TC_DEEP_SMALL": "0"}, ("tc", 128, True, False, 0)),
    (_call(1, 148 * 128, 1, 512, 128, k=1), {}, ("tc", 128, True, True, 0)),         # w_out = 1 < 8: not a TMA conv
    (_call(2, 40, 64, 40, 64, k_order=0), {"BDE2VID_TC_DEEP": "1"}, ("tc", 64, True, True, 0)),
    (_call(2, 40, 64, 40, 64, k_order=0), {"BDE2VID_TC_B_CPASYNC": "1"}, ("tc", 64, False, False, 0)),
    # LayerNorm BN from N, CH from c0
    (_call(1, 300, 1, 64, 96, k=1, ln=True), {}, ("tc", 32, True, False, 1)),
    (_call(1, 300, 1, 128, 192, k=1, ln=True), {}, ("tc", 192, True, False, 2)),
    (_call(1, 300, 1, 256, 320, k=1, ln=True), {"BDE2VID_TC_B_CPASYNC": "1"}, ("tc", 64, False, False, 4)),
    (_call(1, 300, 1, 256, 256, k=1, ln=True), {"BDE2VID_TC_BN": "64"}, ("tc", 256, True, False, 4)),
    (_call(1, 30, 1, 256, 256, k=1, ln=True), {}, ("tc", 256, True, False, 4)),      # never deep
    # SIMT
    (dict(_call(1, 8, 8, 8, 8), engine="simt", dtype="f32"), {}, ("simt", "float")),
    (dict(_call(1, 8, 8, 8, 8), engine="simt"), {}, ("simt", "__nv_bfloat16")),
]


@pytest.mark.parametrize("i", range(len(DISPATCH_TABLE)))
def test_dispatch_table(i):
    """expected_instance against instances derived by hand from the dispatch code, at 148 SMs."""
    call, env, want = DISPATCH_TABLE[i]
    got = expected_instance(call, B200_SMS, env)
    assert got == want, (inst_name(got), inst_name(want))


@pytest.mark.parametrize("n_sm", [132, 148, 160])
def test_cases_stay_on_their_side(n_sm):
    """Every case reaches its declared instance whatever the SM count the batch is derived from."""
    for cs in CONV_CASES + BIG_CASES:
        r = resolve(cs, n_sm)
        assert expected_instance(r, n_sm, r["env"]) == r["inst"], (case_id(cs), n_sm)
    for lc in LN_CASES:
        assert expected_instance(ln_call(lc), n_sm, lc["env"]) == lc["inst"], lc["label"]


def test_persistent_case_wraps():
    """The persistent case gives every CTA at least 3 tiles, unequal counts, and 100 K blocks per tile (weight ring
    of at most 8 stages wraps inside a tile)."""
    for n_sm in (132, 148, 160):
        n = _persistent_imgs(n_sm)
        groups = 2 * n
        assert groups >= 3 * n_sm and groups % n_sm != 0
    assert 25 * 256 // 64 == 100


def test_exact_operand_bound():
    """K * max|a| * max|w| + max|b| <= 2^23 (in units of the weight scale) for every case."""
    for cs in CONV_CASES + BIG_CASES:
        K = cs["k"] ** 2 * (cs["c0"] + cs["c1"])
        assert K * 8 * 4 + 64 <= 2 ** 23, case_id(cs)


def test_instance_parser():
    """The parser reads demangled and mangled names of all three kernel families."""
    names = {
        "void bde::tc::conv_tma_kernel<64, true, 2, false, 2>(CUtensorMap_st, CUtensorMap_st, CUtensorMap_st, "
        "bde::tc::CvParams)": ("tma", 64, True, 2, False, 2),
        "_ZN3bde2tc15conv_tma_kernelILi256ELb1ELi1ELb1ELi1EEEv14CUtensorMap_stS2_S2_NS0_8CvParamsE":
            ("tma", 256, True, 1, True, 1),
        "void bde::tc::gemm_tc_kernel<192, false, false, 4>(CUtensorMap_st, bde::tc::TcParams)": ("tc", 192, False, False, 4),
        "_ZN3bde2tc14gemm_tc_kernelILi128ELb1ELb0ELi0EEEv14CUtensorMap_stNS0_8TcParamsE": ("tc", 128, True, False, 0),
        "void bde::(anonymous namespace)::gemm_simt_kernel<float>(bde::(anonymous namespace)::GemmParams)": ("simt", "float"),
        "_ZN3bde12_GLOBAL__N_116gemm_simt_kernelI13__nv_bfloat16EEvNS0_10GemmParamsE": ("simt", "__nv_bfloat16"),
        "_ZN3bde12_GLOBAL__N_116gemm_simt_kernelIfEEvNS0_10GemmParamsE": ("simt", "float"),
    }
    for n, want in names.items():
        assert gemm_instances([n]) == {want}, (n, gemm_instances([n]))
        assert inst_name(want) in n or "I" in n
    assert gemm_instances(["void bde::tc::mlp_fused256_kernel<2>(CUtensorMap_st)"]) == set()


def test_instance_ids_cover_the_build():
    """The instances this file reaches plus UNREACHABLE are exactly the bde_gemm instances the build contains."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    built = set()
    for f in ("gemm_tc_conv", "gemm_tc", "gemm_simt"):
        with open(os.path.join(root, "profiles", "sass", f + ".kernels.txt")) as fh:
            for line in fh:
                if not line.startswith("#") and line.strip():
                    built |= gemm_instances([line.split("  ")[0]])
    ours = {cs["inst"] for cs in CONV_CASES} | {lc["inst"] for lc in LN_CASES} | set(UNREACHABLE)
    assert len(built) == 84, len(built)
    assert ours == built, sorted(inst_name(t) for t in ours ^ built)
