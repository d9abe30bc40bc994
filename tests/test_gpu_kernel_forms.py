"""Kernel-level references for the GEMM epilogue, activation and source forms the models launch, and for the
element-wise / gather entry points around the GEMMs.

Every case compares one launch with a float64 CPU reference of the same operation whose operands are rounded exactly
as the kernel consumes them (bf16 for the tcgen05 engine and the bf16 SIMT engine, fp32 for the fp32 SIMT engine), under
a PER-ELEMENT gate

    |got - ref| <= r * |ref| + e * mass,     mass = conv(|x|, |w|) + |b|   (float64)

with r = 2^-8 for a bf16 store (round to nearest: at most half an ulp of 8 significant bits) and r = 0 for an fp32 one,
and e covering the fp32 accumulation.  Documented approximations of the bf16 engine widen a gate by their own bound
(tanh.approx: relative 2^-11; the GELU quintic: 5.4e-5 absolute on the normal CDF, DESIGN.md section 2).  Each case
prints the largest ratio err / gate it saw.  Every family also checks that a plausibly wrong reference FAILS the same
gate, so that the gate is known to tell the difference, and every case asserts (with torch.profiler) which kernel
actually served it, so that a dispatch change cannot move a case to another kernel unnoticed.

The CPU tests at the end check the reference helpers against the oracle functions they restate.
"""
import functools
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import oracle_torch as O

DEV = "cuda"
F64 = torch.float64
BF = torch.bfloat16
gpu = pytest.mark.gpu

# gate constants.  Every case prints its max err/gate; calibrated once on a B200 (1000 W power limit): bf16 stores reach
# 0.99 of the gate (the half-ulp term is tight by construction), fp32 outputs use 0.02 - 0.2 of it (GEMMs 0.031, ConvGRU
# u 0.016, h' 0.042, window_reduce 0.028, pred 0.019), the tensor-core attention 0.76, LayerNorm with mean 1e3 / std 0.1
# rows 0.90, the chained ConvGRU step against O.convgru_step 0.19; frame metrics agree with the oracle to 1e-14.
R_BF16 = 2.0 ** -8          # bf16 store: half an ulp, relative
E_ACC = 1e-5                # fp32 accumulation, relative to the absolute mass of the sum
TANH_APPROX = 2.0 ** -11    # tanh.approx.f32, relative
GELU_FORM = 5.4e-5          # fitted-quintic GELU of the bf16 engine, absolute on Phi(x)


# ---------------------------------------------------------------------------------------------------------------------
# shared machinery
# ---------------------------------------------------------------------------------------------------------------------
def rnd(t, dtype):
    """t rounded to the element type a kernel consumes, returned as float64."""
    return t.to(dtype).to(F64)


def nhwc(x, dtype):
    return x.permute(0, 2, 3, 1).contiguous().to(DEV, dtype)


def nchw64(t):
    return t.to(F64).cpu().permute(0, 3, 1, 2)


def gate_ratio(got, ref, gate):
    """max(|got - ref| / gate); > 1 means the gate fails somewhere."""
    got, ref, gate = got.to(F64).cpu(), ref.to(F64).cpu(), gate.to(F64).cpu()
    assert torch.isfinite(got).all(), "non-finite output"
    return float(((got - ref).abs() / gate).max())


def check(name, got, ref, gate, wrong=None):
    """Assert the per-element gate; with ``wrong`` (a plausibly wrong reference) also assert that it fails the gate."""
    r = gate_ratio(got, ref, gate)
    print("%-60s err/gate %.3f" % (name, r))
    assert r <= 1.0, "%s: err/gate %.3f" % (name, r)
    if wrong is not None:
        rw = gate_ratio(got, wrong, gate)
        assert rw > 1.0, "%s: the wrong reference passes the gate too (err/gate %.3f)" % (name, rw)


_TMA = re.compile(r"conv_tma_kernel(?:<(\d+), (true|false), (\d+), (true|false), (\d+)>|ILi(\d+)ELb([01])ELi(\d+)ELb([01])ELi(\d+)E)")


def launched(fn):
    """Run fn() under torch.profiler (CUDA activity only) and return (fn's result, names of the kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, {e.name for e in prof.events()}


def tma_forms(names):
    """[(BN, halo, EPI, pair, NSUB)] of every conv_tma_kernel instance among ``names``."""
    out = []
    for n in names:
        m = _TMA.search(n)
        if m:
            g = [x for x in m.groups() if x is not None]
            out.append((int(g[0]), g[1] in ("true", "1"), int(g[2]), g[3] in ("true", "1"), int(g[4])))
    return out


def has_kernel(names, base):
    """True if a kernel whose (demangled or mangled) name contains ``base`` as a whole identifier ran."""
    pat = re.compile(r"(?<![A-Za-z0-9_])%s(?![A-Za-z0-9_])|\d%s(?=I|E|v)" % (base, base))
    return any(pat.search(n) for n in names)


def assert_route(names, route):
    """route: ("simt", "float" | "bf16"), ("tc",), ("tma", EPI, NSUB | None, BN | None), or ("kernel", base name)."""
    kind = route[0]
    if kind == "simt":
        simt = [n for n in names if "gemm_simt_kernel" in n]
        assert simt, names
        assert all(("bfloat16" in n) == (route[1] == "bf16") for n in simt), simt
        assert not tma_forms(names) and not has_kernel(names, "gemm_tc_kernel"), names
    elif kind == "tc":
        assert has_kernel(names, "gemm_tc_kernel") and not tma_forms(names), names
    elif kind == "tma":
        forms = tma_forms(names)
        assert forms and not has_kernel(names, "gemm_tc_kernel"), names
        for bn, _halo, epi, _pair, nsub in forms:
            assert epi == route[1], (forms, route)
            assert route[2] is None or nsub == route[2], (forms, route)
            assert route[3] is None or bn == route[3], (forms, route)
    else:
        assert has_kernel(names, route[1]), (route, names)


def conv64(x_list, w, b, stride=1):
    """float64 convolution over the channel concat of x_list (NCHW) and its absolute mass conv(|x|, |w|) + |b|."""
    x = torch.cat(x_list, 1)
    pad = w.shape[-1] // 2
    y = F.conv2d(x, w, b, stride=stride, padding=pad)
    mass = F.conv2d(x.abs(), w.abs(), None if b is None else b.abs(), stride=stride, padding=pad)
    return y, mass


def act64(y, act):
    from bde2vid_b200 import ops
    return {ops.ACT_NONE: lambda t: t, ops.ACT_RELU: F.relu, ops.ACT_RELU6: lambda t: t.clamp(0.0, 6.0),
            ops.ACT_GELU: F.gelu, ops.ACT_SIGMOID: torch.sigmoid}[act](y)


# engine forms of bde_gemm: (engine, operand dtype, environment, chunk-major K when the channels allow it)
ENGINES = {
    "simt_f32": ("simt", torch.float32, {}),
    "simt_bf16": ("simt", BF, {}),
    "tc": ("tc", BF, {"BDE2VID_CONV_TMA": "0"}),
    "tma": ("tma", BF, {}),
    "tma_generic": ("tma", BF, {"BDE2VID_CONV_EPI_SPEC": "0"}),
}


def engine_setup(name, monkeypatch):
    from bde2vid_b200 import ops
    kind, dtype, env = ENGINES[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    return (ops.ENGINE_SIMT if kind == "simt" else ops.ENGINE_TCGEN05), dtype, kind


def pack(w, dtype, chunk_major):
    from bde2vid_b200.engine import _pack_conv
    return _pack_conv(w.to(torch.float32).to(DEV), dtype, chunk_major=chunk_major)


def out_hw(h, w, k, s):
    return (h + 2 * (k // 2) - k) // s + 1, (w + 2 * (k // 2) - k) // s + 1


# ---------------------------------------------------------------------------------------------------------------------
# 1. bde_gemm forms
# ---------------------------------------------------------------------------------------------------------------------
# n, cin, cout, h, w, k, stride, expected NSUB of the TMA conv kernel
ACT_SHAPES = {
    "3x3": (2, 64, 64, 20, 28, 3, 1, 1),
    "5x5s2": (2, 64, 128, 33, 44, 5, 2, 1),
    "1x1": (2, 128, 64, 19, 26, 1, 1, 1),
    # 10 images x 5 x 3 tile pairs = 150 >= 148 SMs: the dual-tile form (two 8 x 16 tiles per CTA)
    "dual": (10, 64, 64, 40, 70, 3, 1, 2),
}


@functools.lru_cache(maxsize=None)
def _act_operands(shape, dtype):
    n, ci, co, h, w, k, s, _ = ACT_SHAPES[shape]
    g = torch.Generator().manual_seed(ci + co + h + k)
    x = rnd(torch.randn(n, ci, h, w, generator=g, dtype=F64), dtype)
    wt = rnd(torch.randn(co, ci, k, k, generator=g, dtype=F64) * (4.0 / (ci * k * k) ** 0.5), dtype)
    b = (2.0 + 0.5 * torch.randn(co, generator=g, dtype=F64)).float().to(F64)
    pre, mass = conv64([x], wt, b, s)
    return x, wt, b, pre, mass


@gpu
@pytest.mark.parametrize("engine", sorted(ENGINES))
@pytest.mark.parametrize("shape", sorted(ACT_SHAPES))
def test_gemm_activations(shape, engine, monkeypatch):
    """NONE / RELU / RELU6 / GELU / SIGMOID in the store epilogue of every engine.  Pre-activations are spread over
    (-inf, 0), (0, 6) and (6, inf), each holding >= 10 % of the outputs, so that both clamps of ReLU6 are exercised.
    TMA conv: NONE / RELU / RELU6 take the specialised store epilogue (EPI 2) unless BDE2VID_CONV_EPI_SPEC=0, GELU /
    SIGMOID always the generic one (EPI 0).
    Max err/gate observed on a B200 (1000 W): 0.99 on the bf16 engines (the half-ulp store term, which is reached by
    construction), 0.031 on the fp32 SIMT engine; GELU on the tcgen05 engine 0.91."""
    from bde2vid_b200 import ops
    n, ci, co, h, w, k, s, nsub = ACT_SHAPES[shape]
    eng, dtype, kind = engine_setup(engine, monkeypatch)
    x, wt, b, pre, mass = _act_operands(shape, dtype)
    frac = [float((pre < 0).double().mean()), float(((pre > 0) & (pre < 6)).double().mean()), float((pre > 6).double().mean())]
    assert min(frac) >= 0.10, frac
    cm = kind != "simt"
    pw, ld = pack(wt, dtype, cm)
    a0 = nhwc(x, dtype)
    bd = b.float().to(DEV)
    ho, wo = out_hw(h, w, k, s)
    bf = dtype == BF
    for act in (ops.ACT_NONE, ops.ACT_RELU, ops.ACT_RELU6, ops.ACT_GELU, ops.ACT_SIGMOID):
        out = torch.full((n, ho, wo, co), float("nan"), dtype=dtype, device=DEV)

        def run():
            ops.gemm(a0, pw, bd, out, n_img=n, h_in=h, w_in=w, c0=ci, n=co, ksize=k, stride=s, pad=k // 2, w_ld=ld, act=act,
                     engine=eng, dtype=dtype, k_order=int(cm))
        _, names = launched(run)
        if kind == "simt":
            assert_route(names, ("simt", "bf16" if bf else "float"))
        elif kind == "tc":
            assert_route(names, ("tc",))
        else:
            spec = engine == "tma" and act in (ops.ACT_NONE, ops.ACT_RELU, ops.ACT_RELU6)
            assert_route(names, ("tma", 2 if spec else 0, nsub, None))
        ref = act64(pre, act)
        lip = 0.25 if act == ops.ACT_SIGMOID else 1.13      # Lipschitz bound of the activation (GELU: 1.13)
        gate = (R_BF16 if bf else 2.0 ** -23) * ref.abs() + E_ACC * lip * mass
        if act == ops.ACT_GELU and kind != "simt":
            gate = gate + (GELU_FORM + 0.5 * TANH_APPROX) * pre.abs()
        wrong = None
        if act == ops.ACT_RELU6:
            wrong = F.relu(pre)                               # ReLU instead of ReLU6
        elif act == ops.ACT_RELU:
            wrong = pre.clamp(0.0, 6.0)
        elif act == ops.ACT_NONE:
            wrong = F.relu(pre)
        else:
            wrong = act64(pre - b.view(1, -1, 1, 1), act)     # bias dropped
        check("act %d %s %s" % (act, shape, engine), nchw64(out), ref, gate, wrong)


# ---- ConvGRU step ---------------------------------------------------------------------------------------------------
def gru_ur_ref(x, h_op, h_master, wu, bu, wr, br):
    """First ConvGRU launch (BDE_EPI_GRU_UR) in float64: u = sigmoid(update), hr = h_master * sigmoid(reset), where the
    convolutions read cat[x, h_op] and the pointwise product the fp32 master h.  Returns (u, hr, mass_u, mass_r)."""
    pu, mu = conv64([x, h_op], wu, bu)
    pr, mr = conv64([x, h_op], wr, br)
    return torch.sigmoid(pu), h_master * torch.sigmoid(pr), mu, mr


def gru_out_ref(x, hr_op, h_master, u, wo, bo):
    """Second launch (BDE_EPI_GRU_OUT): h' = h (1 - u) + tanh(conv(cat[x, hr]) + bo) u.  Returns (h', o, mass_o)."""
    po, mo = conv64([x, hr_op], wo, bo)
    o = torch.tanh(po)
    return h_master * (1 - u) + o * u, o, mo


def gru_step_ref(x, h, wu, bu, wr, br, wo, bo, operand=lambda t: t):
    """Both launches chained; ``operand`` rounds what the convolutions read (h, h * r) as the kernels do."""
    if h is None:
        h = torch.zeros(x.shape[0], wu.shape[0], x.shape[2], x.shape[3], dtype=x.dtype)
    u, hr, _, _ = gru_ur_ref(x, operand(h), h, wu, bu, wr, br)
    return gru_out_ref(x, operand(hr), h, u, wo, bo)[0]


# hidden C, B, h, w, engine form, forced N tile (BDE2VID_CONV_BN)
GRU_CASES = [
    (64, 4, 33, 44, "tma", None),
    (128, 2, 17, 22, "tma", None),
    (256, 1, 9, 19, "tma", None),
    (64, 2, 17, 22, "tma", "32"),
    (128, 1, 9, 19, "tma", "64"),
    (32, 2, 17, 22, "tc", None),      # FireNet: channels padded to 32, c0 % 64 != 0 -> gemm_tc_kernel
    (32, 4, 33, 44, "tc", None),
    (32, 1, 9, 19, "simt_f32", None),
]


@gpu
@pytest.mark.parametrize("C,B,h,w,form,bn", GRU_CASES)
def test_convgru_step(C, B, h, w, form, bn, monkeypatch):
    """ConvGRU step as _chain_step issues it: [update | reset] conv with rows n = 2c + g (EPI_GRU_UR -> u fp32, h * r),
    then the out-gate conv over cat[x, h * r] (EPI_GRU_OUT -> h' fp32 master + operand copy).  First step with
    c_prev = None and an all-zero h operand, second step fed with the first step's h' / master.  On the TMA conv x is the
    pitched channel half of a [.., 2C] map (a0_ld = 2C), as the merged encoder conv writes it.  Each launch is checked
    against its own float64 reference (the OUT launch from the kernel's own u and h * r), the chained step against
    O.convgru_step.  Gates widen by tanh.approx (sigmoid = 0.5 tanh(x / 2) + 0.5: absolute 2^-12)."""
    from bde2vid_b200 import ops
    if bn is not None:
        monkeypatch.setenv("BDE2VID_CONV_BN", bn)
    eng = ops.ENGINE_SIMT if form == "simt_f32" else ops.ENGINE_TCGEN05
    dtype = torch.float32 if form == "simt_f32" else BF
    bf = dtype == BF
    cm = form == "tma"
    g = torch.Generator().manual_seed(C * 7 + B + h)
    K = 2 * C * 9
    wu = torch.randn(C, 2 * C, 3, 3, generator=g, dtype=F64) * (2.0 / K ** 0.5)
    wr = torch.randn(C, 2 * C, 3, 3, generator=g, dtype=F64) * (2.0 / K ** 0.5)
    wo = torch.randn(C, 2 * C, 3, 3, generator=g, dtype=F64) * (2.0 / K ** 0.5)
    wu, wr, wo = rnd(wu, dtype), rnd(wr, dtype), rnd(wo, dtype)
    bu, br, bo = [(0.3 * torch.randn(C, generator=g, dtype=F64)).float().to(F64) for _ in range(3)]
    # packed as the engine does it (engine.py gru_layers)
    pur, ldu = pack(torch.stack([wu, wr], 1).reshape(2 * C, 2 * C, 3, 3), dtype, cm)
    bur = torch.stack([bu, br], 1).reshape(-1).float().to(DEV)
    po, ldo = pack(wo, dtype, cm)
    bod = bo.float().to(DEV)
    xs = [rnd(torch.randn(B, C, h, w, generator=g, dtype=F64), dtype) for _ in range(2)]
    if cm:
        wide = [torch.cat([torch.randn(B, C, h, w, generator=g, dtype=F64), x], 1) for x in xs]
        xin = [nhwc(t, dtype)[..., C:] for t in wide]     # channel half [C, 2C) of a [.., 2C] map
        pitch = dict(a0_ld=2 * C)
    else:
        xin, pitch = [nhwc(x, dtype) for x in xs], {}
    zero = torch.zeros(B, h, w, C, dtype=dtype, device=DEV)
    route = ("tma", 0, None, int(bn) if bn else None) if form == "tma" else ("tc",) if form == "tc" else ("simt", "float")
    gate_bf = R_BF16 if bf else 2.0 ** -23
    sig_ap = 0.5 * TANH_APPROX if bf else 2.0 ** -22

    def step(k, h_op, h_master_dev):
        u = torch.full((B, h, w, C), float("nan"), device=DEV)
        hr = torch.full((B, h, w, C), float("nan"), dtype=dtype, device=DEV)
        hout = torch.full((B, h, w, C), float("nan"), dtype=dtype, device=DEV)
        hm = torch.full((B, h, w, C), float("nan"), device=DEV)

        def run():
            ops.gemm(xin[k], pur, bur, hr, n_img=B, h_in=h, w_in=w, c0=C, n=2 * C, ksize=3, pad=1, w_ld=ldu, a1=h_op, c1=C,
                     epi=ops.EPI_GRU_UR, c_prev=h_master_dev, c_out=u, engine=eng, dtype=dtype, k_order=int(cm), **pitch)
            ops.gemm(xin[k], po, bod, hout, n_img=B, h_in=h, w_in=w, c0=C, n=C, ksize=3, pad=1, w_ld=ldo, a1=hr, c1=C,
                     epi=ops.EPI_GRU_OUT, c_prev=h_master_dev, residual=u, c_out=hm, engine=eng, dtype=dtype, k_order=int(cm),
                     **pitch)
        _, names = launched(run)
        assert_route(names, route)
        return u, hr, hout, hm

    h_master = torch.zeros(B, C, h, w, dtype=F64)
    results = []
    for k in range(2):
        h_op_dev = zero if k == 0 else results[-1][2]
        hm_dev = None if k == 0 else results[-1][3]
        u, hr, hout, hm = step(k, h_op_dev, hm_dev)
        x = xs[k]
        h_op = nchw64(h_op_dev)
        u_ref, hr_ref, mu, mr = gru_ur_ref(x, h_op, h_master, wu, bu, wr, br)
        # wrong reference: update and reset rows swapped
        u_sw, hr_sw, _, _ = gru_ur_ref(x, h_op, h_master, wr, br, wu, bu)
        check("gru UR u   C%d B%d %dx%d %s bn%s step%d" % (C, B, h, w, form, bn, k), nchw64(u), u_ref,
              sig_ap + 0.25 * E_ACC * mu + 2.0 ** -23, u_sw)
        hr_gate = gate_bf * hr_ref.abs() + h_master.abs() * (sig_ap + 0.25 * E_ACC * mr) + 1e-30
        check("gru UR h*r C%d B%d %dx%d %s bn%s step%d" % (C, B, h, w, form, bn, k), nchw64(hr), hr_ref, hr_gate,
              hr_sw if k > 0 else None)
        # OUT launch from the kernel's own u and h * r
        hk_ref, o_ref, mo = gru_out_ref(x, nchw64(hr), h_master, nchw64(u), wo, bo)
        ua = nchw64(u).abs()
        g32 = ua * ((TANH_APPROX if bf else 2.0 ** -22) * o_ref.abs() + E_ACC * mo) + 2.0 ** -22 * (h_master.abs() + ua * o_ref.abs())
        wrong_out = h_master * nchw64(u) + o_ref * (1 - nchw64(u))              # u and 1 - u exchanged
        check("gru OUT h' fp32 C%d B%d %dx%d %s bn%s step%d" % (C, B, h, w, form, bn, k), nchw64(hm), hk_ref, g32, wrong_out)
        check("gru OUT h' op   C%d B%d %dx%d %s bn%s step%d" % (C, B, h, w, form, bn, k), nchw64(hout), hk_ref,
              gate_bf * hk_ref.abs() + g32)
        # the chained step against the oracle's cell: its gap to the mixed-precision chain is the operand rounding
        sd = {"g.update_gate.weight": wu, "g.update_gate.bias": bu, "g.reset_gate.weight": wr, "g.reset_gate.bias": br,
              "g.out_gate.weight": wo, "g.out_gate.bias": bo}
        oracle = O.convgru_step(sd, "g", x, None if k == 0 else h_master)
        mixed = gru_step_ref(x, h_master, wu, bu, wr, br, wo, bo, operand=lambda t: rnd(t, dtype))
        # (the per-launch gates above are the tight ones; 2^-7 covers kernel and reference rounding h * r to bf16 on
        # different sides of a tie, and the u / h * r errors carried into h')
        comp_gate = (mixed - oracle).abs() + 2.0 ** -7 + gate_bf * oracle.abs()
        check("gru step vs O.convgru_step C%d B%d %dx%d %s bn%s step%d" % (C, B, h, w, form, bn, k), nchw64(hm), oracle,
              comp_gate)
        results.append((u, hr, hout, hm))
        h_master = nchw64(hm)
    if form == "tma" and bn is None and C == 64:
        # programmatic dependent launch: the OUT launch reads u (written by the UR launch) with __ldg after
        # griddepcontrol.wait.  Same chain with PDL disabled: bit-identical.
        monkeypatch.setenv("BDE2VID_PDL", "0")
        u2, hr2, hout2, hm2 = step(1, results[0][2], results[0][3])
        assert torch.equal(u2, results[1][0]) and torch.equal(hr2, results[1][1])
        assert torch.equal(hout2, results[1][2]) and torch.equal(hm2, results[1][3])


# ---- residual forms -------------------------------------------------------------------------------------------------
RES_CASES = [
    # engine form, C, B, h, w, expected route
    ("tma", 64, 2, 20, 28),
    ("tma", 128, 1, 17, 22),
    ("tc", 64, 2, 20, 28),
    ("tc", 32, 2, 17, 22),
    ("simt_bf16", 32, 2, 17, 22),
    ("simt_f32", 64, 1, 17, 22),
]


@gpu
@pytest.mark.parametrize("form,C,B,h,w", RES_CASES)
def test_residual_forms(form, C, B, h, w, monkeypatch):
    """(a) res_mode = 1: a residual of the operand type added BEFORE the activation (E2VID / FireNet ResidualBlock,
    relu(conv2(y) + x)).  (b) out_f32 + fp32 residual added after the (absent) activation + a bf16 copy in out2, on a
    3 x 3 conv (the residual tail, x = x + conv2(.)), and (c) the same in place (out is residual).  On the TMA conv all
    of them take the generic epilogue (EPI 0)."""
    from bde2vid_b200 import ops
    eng, dtype, kind = engine_setup(form, monkeypatch)
    bf = dtype == BF
    cm = kind != "simt" and C % 64 == 0
    g = torch.Generator().manual_seed(C + B + h + 3)
    x = rnd(torch.randn(B, C, h, w, generator=g, dtype=F64), dtype)
    wt = rnd(torch.randn(C, C, 3, 3, generator=g, dtype=F64) * (1.5 / (9 * C) ** 0.5), dtype)
    b = (0.2 * torch.randn(C, generator=g, dtype=F64)).float().to(F64)
    res = rnd(torch.randn(B, C, h, w, generator=g, dtype=F64), dtype)
    pw, ld = pack(wt, dtype, cm)
    bd = b.float().to(DEV)
    pre, mass = conv64([x], wt, b)
    route = ("tma", 0, None, None) if kind == "tma" else ("tc",) if kind == "tc" else ("simt", "bf16" if bf else "float")
    rb = R_BF16 if bf else 2.0 ** -23
    common = dict(n_img=B, h_in=h, w_in=w, c0=C, n=C, ksize=3, pad=1, w_ld=ld, engine=eng, dtype=dtype, k_order=int(cm))
    a0 = nhwc(x, dtype)
    # (a) res_mode = 1
    out = torch.full((B, h, w, C), float("nan"), dtype=dtype, device=DEV)
    _, names = launched(lambda: ops.gemm(a0, pw, bd, out, act=ops.ACT_RELU, residual=nhwc(res, dtype), res_mode=1, **common))
    assert_route(names, route)
    ref = F.relu(pre + res)
    check("res_mode=1 relu %s C%d" % (form, C), nchw64(out), ref, rb * ref.abs() + E_ACC * (mass + res.abs()) + 1e-30,
          F.relu(pre) + res)                                   # activation applied before the residual
    # (b) out_f32 + fp32 residual + out2
    r32 = torch.randn(B, C, h, w, generator=g, dtype=F64).float().to(F64)
    o32 = torch.full((B, h, w, C), float("nan"), device=DEV)
    o2 = torch.full((B, h, w, C), float("nan"), dtype=dtype, device=DEV)
    _, names = launched(lambda: ops.gemm(a0, pw, bd, o32, out_f32=True, residual=nhwc(r32, torch.float32), out2=o2, **common))
    assert_route(names, route)
    ref = pre + r32
    g32 = E_ACC * (mass + r32.abs()) + 2.0 ** -23 * ref.abs()
    check("out_f32+res %s C%d" % (form, C), nchw64(o32), ref, g32, pre)     # residual dropped
    check("out2 %s C%d" % (form, C), nchw64(o2), ref, rb * ref.abs() + g32, pre + 2 * r32)
    # (c) in place: out aliases the fp32 residual
    xs = nhwc(r32, torch.float32)
    _, names = launched(lambda: ops.gemm(a0, pw, bd, xs, out_f32=True, residual=xs, out2=o2, **common))
    assert_route(names, route)
    check("in-place res %s C%d" % (form, C), nchw64(xs), ref, g32, pre)


# ---- two A sources --------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k_order", [0, 1])
@pytest.mark.parametrize("C", [64, 128, 256])
def test_concat_fusion_1x1(C, k_order, monkeypatch):
    """Decoder concat fusion: 1 x 1 conv over cat[skip, x] with two DIFFERENT sources (TMA conv, specialised store),
    then the Q2 form (decoder 0 sees cat[feat, feat]: a0 is a1), then a pitched a1 (a1_ld)."""
    from bde2vid_b200 import ops
    n, h, w = 3, 18, 27
    g = torch.Generator().manual_seed(C + k_order)
    s0 = rnd(torch.randn(n, C, h, w, generator=g, dtype=F64), BF)
    s1 = rnd(torch.randn(n, C, h, w, generator=g, dtype=F64) * 2 + 1, BF)
    wt = rnd(torch.randn(C, 2 * C, 1, 1, generator=g, dtype=F64) / (2 * C) ** 0.5, BF)
    b = (0.3 * torch.randn(C, generator=g, dtype=F64)).float().to(F64)
    pw, ld = pack(wt, BF, bool(k_order))
    bd = b.float().to(DEV)
    common = dict(n_img=n, h_in=h, w_in=w, c0=C, c1=C, n=C, w_ld=ld, engine=ops.ENGINE_TCGEN05, dtype=BF, k_order=k_order)
    a0, a1 = nhwc(s0, BF), nhwc(s1, BF)
    out = torch.full((n, h, w, C), float("nan"), dtype=BF, device=DEV)
    _, names = launched(lambda: ops.gemm(a0, pw, bd, out, a1=a1, **common))
    assert_route(names, ("tma", 2, None, None))
    ref, mass = conv64([s0, s1], wt, b)
    check("concat 1x1 C%d k%d" % (C, k_order), nchw64(out), ref, R_BF16 * ref.abs() + E_ACC * mass,
          conv64([s1, s0], wt, b)[0])                                          # sources exchanged
    # Q2: the same tensor twice
    _, names = launched(lambda: ops.gemm(a0, pw, bd, out, a1=a0, **common))
    assert_route(names, ("tma", 2, None, None))
    ref, mass = conv64([s0, s0], wt, b)
    check("concat 1x1 Q2 C%d k%d" % (C, k_order), nchw64(out), ref, R_BF16 * ref.abs() + E_ACC * mass,
          conv64([s0, s1], wt, b)[0])
    # pitched second source: channels [C, 2C) of a [.., 2C] map
    wide = torch.cat([rnd(torch.randn(n, C, h, w, generator=g, dtype=F64), BF), s1], 1)
    a1w = nhwc(wide, BF)[..., C:]
    _, names = launched(lambda: ops.gemm(a0, pw, bd, out, a1=a1w, a1_ld=2 * C, **common))
    assert_route(names, ("tma", 2, None, None))
    ref, mass = conv64([s0, s1], wt, b)
    check("concat 1x1 pitched a1 C%d k%d" % (C, k_order), nchw64(out), ref, R_BF16 * ref.abs() + E_ACC * mass,
          conv64([s0, wide[:, :C]], wt, b)[0])                                  # the wrong half of the wide map


@gpu
@pytest.mark.parametrize("form", ["tma", "tma_generic", "tc"])
def test_two_source_3x3_unequal(form, monkeypatch):
    """3 x 3 conv over two sources with c0 != c1 (64 + 128), ReLU6, and with a pitched a1."""
    from bde2vid_b200 import ops
    eng, dtype, _ = engine_setup(form, monkeypatch)
    n, c0, c1, co, h, w = 2, 64, 128, 64, 21, 30
    g = torch.Generator().manual_seed(11)
    s0 = rnd(torch.randn(n, c0, h, w, generator=g, dtype=F64), BF)
    s1 = rnd(torch.randn(n, c1, h, w, generator=g, dtype=F64), BF)
    wt = rnd(torch.randn(co, c0 + c1, 3, 3, generator=g, dtype=F64) * (4.0 / (9 * (c0 + c1)) ** 0.5), BF)
    b = (2.0 + 0.5 * torch.randn(co, generator=g, dtype=F64)).float().to(F64)
    pw, ld = pack(wt, BF, True)
    bd = b.float().to(DEV)
    route = ("tc",) if form == "tc" else ("tma", 2 if form == "tma" else 0, None, None)
    pre, mass = conv64([s0, s1], wt, b)
    ref = pre.clamp(0.0, 6.0)
    gate = R_BF16 * ref.abs() + E_ACC * mass
    common = dict(n_img=n, h_in=h, w_in=w, c0=c0, c1=c1, n=co, ksize=3, pad=1, w_ld=ld, engine=eng, dtype=BF, k_order=1,
                  act=ops.ACT_RELU6)
    out = torch.full((n, h, w, co), float("nan"), dtype=BF, device=DEV)
    _, names = launched(lambda: ops.gemm(nhwc(s0, BF), pw, bd, out, a1=nhwc(s1, BF), **common))
    assert_route(names, route)
    # wrong: the first 64 channels of source 1 read in place of source 0
    check("3x3 two-source 64+128 %s" % form, nchw64(out), ref, gate, conv64([s1[:, :c0], s1], wt, b)[0].clamp(0.0, 6.0))
    if form != "tc":      # the cp.async engine refuses pitched sources (test_gpu_gemm.py)
        wide = torch.cat([s1, rnd(torch.randn(n, 64, h, w, generator=g, dtype=F64), BF)], 1)
        _, names = launched(lambda: ops.gemm(nhwc(s0, BF), pw, bd, out, a1=nhwc(wide, BF)[..., :c1], a1_ld=c1 + 64, **common))
        assert_route(names, route)
        check("3x3 two-source pitched a1 %s" % form, nchw64(out), ref, gate)


# ---------------------------------------------------------------------------------------------------------------------
# 2. element-wise and gather entry points
# ---------------------------------------------------------------------------------------------------------------------
def window_tokens(frames, tm, c):
    """[nwin, ntok, c] float64 token matrix of every frame (None = all-zero frame, map < 0 = zero token)."""
    out = []
    for f in frames:
        src = torch.zeros(int(tm.max()) + 1, c, dtype=F64) if f is None else f.to(F64)
        t = src[tm.clamp(min=0).long()] * (tm >= 0).unsqueeze(-1).to(F64)
        out.append(t)
    return out


def window_reduce_ref(frames, tm, c, X, w, b):
    """bde_window_reduce in float64: conv[o] = b[o] + sum_tok w[o, tok] x[tok, o // X] per (window, frame) -- the
    grouped Conv2d(C, X*C, window, groups=C) -- then the reference's view of [C*X] as [X, C] (index j*C + c).
    Returns (out [nwin, D, X, c], mass)."""
    ch = torch.arange(c * X) // X
    outs, masses = [], []
    for t in window_tokens(frames, tm, c):
        tg = t[:, :, ch]                                         # [nwin, ntok, c*X]
        conv = torch.einsum("wto,ot->wo", tg, w) + b
        mass = torch.einsum("wto,ot->wo", tg.abs(), w.abs()) + b.abs()
        outs.append(conv.view(-1, X, c))
        masses.append(mass.view(-1, X, c))
    return torch.stack(outs, 1), torch.stack(masses, 1)


@gpu
@pytest.mark.parametrize("c", [64, 256])
@pytest.mark.parametrize("X", [1, 4, 9])
@pytest.mark.parametrize("D", [1, 2, 3])
def test_window_reduce(D, X, c):
    """nwindow_size feature reduction on plain and dilated token maps, frame 1 all-zero (None) when D > 1; then the
    CUDA-core window attention over the n_kv = D * X reduced tokens against float64 softmax attention."""
    from bde2vid_b200 import ops
    from bde2vid_b200.engine import window_token_map
    B, H, W = 2, 11, 16
    g = torch.Generator().manual_seed(D * 100 + X * 10 + c)
    frames = [torch.randn(B * H * W, c, generator=g) for _ in range(D)]
    if D > 1:
        frames[1] = None
    w = torch.randn(c * X, 49, generator=g) / 7.0
    b = torch.randn(c * X, generator=g) * 0.1
    for dil in (False, True):
        tm, _ = window_token_map(B, H, W, (7, 7), dil, DEV)
        nwin = tm.shape[0]
        out = torch.full((nwin, D, X, c), float("nan"), device=DEV)
        _, names = launched(lambda: ops.window_reduce([None if f is None else f.to(DEV) for f in frames], tm.view(-1), nwin, 49,
                                                      c, X, w.to(DEV), b.to(DEV), out))
        assert_route(names, ("kernel", "window_reduce_kernel"))
        ref, mass = window_reduce_ref(frames, tm.cpu(), c, X, w.to(F64), b.to(F64))
        wrong = None
        if X > 1:   # the natural c*X + j view of the [C*X] vector instead of the reference's j*C + c
            wrong = ref.reshape(nwin, D, X * c).view(nwin, D, c, X).transpose(2, 3)
        check("window_reduce D%d X%d c%d dil%d" % (D, X, c, dil), out, ref, E_ACC * mass + 2.0 ** -23 * ref.abs(), wrong)
    if D * X in (8, 27):
        heads = 16
        hd = c // heads
        n_kv = D * X
        for dtype in (torch.float32, BF):
            q = rnd(torch.randn(nwin, 49, c, generator=g, dtype=F64) * hd ** -0.5, dtype)
            kv = rnd(torch.randn(nwin, n_kv, 2 * c, generator=g, dtype=F64), dtype)
            bias = torch.randn(heads, 49, n_kv, generator=g, dtype=F64).float().to(F64)
            qh = q.view(nwin, 49, heads, hd).permute(0, 2, 1, 3)
            kh = kv[..., :c].reshape(nwin, n_kv, heads, hd).permute(0, 2, 1, 3)
            vh = kv[..., c:].reshape(nwin, n_kv, heads, hd).permute(0, 2, 1, 3)
            p = torch.softmax(qh @ kh.transpose(-1, -2) + bias, -1)
            ref = (p @ vh).permute(0, 2, 1, 3).reshape(nwin, 49, c)
            mass = (p @ vh.abs()).permute(0, 2, 1, 3).reshape(nwin, 49, c)
            wrong = (torch.softmax(qh @ kh.transpose(-1, -2), -1) @ vh).permute(0, 2, 1, 3).reshape(nwin, 49, c)
            o = torch.full((nwin, 49, c), float("nan"), dtype=dtype, device=DEV)
            _, names = launched(lambda: ops.window_attention(q.to(DEV, dtype), kv.to(DEV, dtype),
                                                             bias.permute(0, 2, 1).contiguous().float().to(DEV), nwin, 49,
                                                             n_kv, c, heads, o))
            assert_route(names, ("kernel", "window_attention_kernel"))
            rb = R_BF16 if dtype == BF else 2.0 ** -23
            check("window_attention n_kv=%d c%d %s" % (n_kv, c, dtype), o, ref, rb * ref.abs() + E_ACC * mass, wrong)


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, BF])
@pytest.mark.parametrize("c", [32, 64])
def test_pred_sigmoid(c, dtype):
    """predI + output activation: skip 'sum' (wt_head None: w . (x + head)) and 'concat' (folded [wt | wt_head]),
    ACT_SIGMOID and ACT_NONE ('Identity'), over pixel counts around the 128-thread block."""
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(c + (dtype == BF))
    for n_pix in (1, 127, 129, 1000):
        x = rnd(torch.randn(n_pix, c, generator=g, dtype=F64), dtype)
        hd = rnd(torch.randn(n_pix, c, generator=g, dtype=F64), dtype)
        wt = (torch.randn(c, generator=g, dtype=F64) * 0.3).float().to(F64)
        wh = (torch.randn(c, generator=g, dtype=F64) * 0.3).float().to(F64)
        b = torch.randn(1, generator=g, dtype=F64).float().to(F64)
        for concat in (False, True):
            for act in (ops.ACT_SIGMOID, ops.ACT_NONE):
                img = torch.full((n_pix,), float("nan"), device=DEV)
                _, names = launched(lambda: ops.pred_sigmoid(x.to(DEV, dtype), hd.to(DEV, dtype), wt.float().to(DEV), b.float().to(DEV),
                                                             c, n_pix, img, wt_head=wh.float().to(DEV) if concat else None, act=act))
                assert_route(names, ("kernel", "pred_sigmoid_kernel"))
                if concat:
                    pre, mass = x @ wt + hd @ wh + b, x.abs() @ wt.abs() + hd.abs() @ wh.abs() + b.abs()
                    wrong_pre = x @ wh + hd @ wt + b                      # wt / wt_head exchanged
                else:
                    pre, mass = (x + hd) @ wt + b, (x.abs() + hd.abs()) @ wt.abs() + b.abs()
                    wrong_pre = x @ wt + b                                # head dropped
                f = torch.sigmoid if act == ops.ACT_SIGMOID else (lambda t: t)
                ref = f(pre)
                gate = E_ACC * mass * (0.25 if act == ops.ACT_SIGMOID else 1.0) + 2.0 ** -23 * ref.abs()
                wrong = f(wrong_pre)
                if n_pix == 1:
                    wrong = None      # one pixel can land on either side by chance
                check("pred_sigmoid c%d %s n%d concat%d act%d" % (c, dtype, n_pix, concat, act), img, ref, gate, wrong)


UP_COMBOS = [   # (skip dtype | None, x dtype, dst dtype): every combination bde_upsample2x_sum accepts
    (None, torch.float32, torch.float32), (torch.float32, torch.float32, torch.float32),
    (None, torch.float32, BF), (None, BF, BF), (torch.float32, torch.float32, BF), (torch.float32, BF, BF),
    (BF, torch.float32, BF), (BF, BF, BF),
]


@gpu
@pytest.mark.parametrize("combo", range(len(UP_COMBOS)))
def test_upsample2x_sum_forms(combo):
    """dst = bilinear_x2(skip + x_scale * x) (align_corners=False) for every (skip, x, dst) dtype combination, crossed with
    x_scale in {1, 2}, c in {4, 12, 32, 64, 256} (c % 8 != 0 takes the generic kernel), h in {1, 8, 9, 17}, w in {1, 13, 176}
    (w * c / 8 > 256: rows wider than one block; h / w = 1: clamped taps).  The block kernel serves bf16 outputs with
    c % 8 == 0, the generic one everything else."""
    from bde2vid_b200 import ops
    sk_t, x_t, d_t = UP_COMBOS[combo]
    g = torch.Generator().manual_seed(combo)
    worst = 0.0
    for c in (4, 12, 32, 64, 256):
        block = d_t == BF and c % 8 == 0
        routed = False
        for h in (1, 8, 9, 17):
            for w in (1, 13, 176):
                for xs in (1.0, 2.0):
                    x = rnd(torch.randn(1, c, h, w, generator=g, dtype=F64), x_t)
                    sk = None if sk_t is None else rnd(torch.randn(1, c, h, w, generator=g, dtype=F64), sk_t)
                    src = xs * x + (0 if sk is None else sk)
                    amass = xs * x.abs() + (0 if sk is None else sk.abs())
                    ref = F.interpolate(src, scale_factor=2, mode="bilinear", align_corners=False)
                    mass = F.interpolate(amass, scale_factor=2, mode="bilinear", align_corners=False)
                    dst = torch.full((1, 2 * h, 2 * w, c), float("nan"), dtype=d_t, device=DEV)

                    def run():
                        ops.upsample2x_sum(None if sk is None else nhwc(sk, sk_t), nhwc(x, x_t), xs, 1, h, w, c, dst)
                    if not routed and w == 176:
                        _, names = launched(run)
                        assert_route(names, ("kernel", "upsample2x_sum_block_kernel" if block else "upsample2x_sum_kernel"))
                        assert has_kernel(names, "upsample2x_sum_kernel") != block
                        routed = True
                    else:
                        run()
                    rb = R_BF16 if d_t == BF else 0.0
                    gate = rb * ref.abs() + 2.0 ** -21 * mass + 1e-30
                    r = gate_ratio(nchw64(dst), ref, gate)
                    worst = max(worst, r)
                    assert r <= 1.0, ("upsample", combo, c, h, w, xs, r)
                    if h > 1 and w > 1 and xs == 2.0:
                        # discrimination: the nearest-neighbour x2 (and x_scale ignored) must fail
                        near = F.interpolate(src, scale_factor=2, mode="nearest")
                        assert gate_ratio(nchw64(dst), near, gate) > 1.0
                        wrong = F.interpolate(x + (0 if sk is None else sk), scale_factor=2, mode="bilinear", align_corners=False)
                        assert gate_ratio(nchw64(dst), wrong, gate) > 1.0
    print("upsample2x_sum combo %s err/gate %.3f" % (UP_COMBOS[combo], worst))


@gpu
@pytest.mark.parametrize("dtype", [torch.float32, BF])
@pytest.mark.parametrize("c", [32, 64, 96, 128, 256, 1024])
def test_layernorm_forms(c, dtype):
    """Row LayerNorm: the vectorised forms (c = 64 / 128 / 256, several rows per warp) and the one-row-per-warp kernel
    (any other c), row counts that are not multiples of the rows per warp / per block, and rows with mean 1e3 and
    std 0.1, where a one-pass E[x^2] - mean^2 variance in fp32 would be meaningless.  Gate: the fp32 mean carries
    ~u sqrt(c) mean|x| of summation error, i.e. u sqrt(c) mean|x| / sigma relative on the output."""
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(c + (dtype == BF))
    vec = c in (64, 128, 256)
    gamma = torch.randn(c, generator=g).float()
    beta = torch.randn(c, generator=g).float()
    for rows in (1, 5, 37, 1003):
        for shifted in (False, True):
            x = torch.randn(rows, c, generator=g, dtype=F64) * (0.1 if shifted else 2.0) + (1e3 if shifted else 0.5)
            x = x.float()
            out = torch.full((rows, c), float("nan"), dtype=dtype, device=DEV)
            _, names = launched(lambda: ops.layernorm(x.to(DEV), rows, c, gamma.to(DEV), beta.to(DEV), out))
            assert_route(names, ("kernel", "ln_gather_qkv_kernel" if vec else "layernorm_kernel"))
            assert has_kernel(names, "layernorm_kernel") != vec
            x64 = x.to(F64)
            ref = F.layer_norm(x64, (c,), gamma.to(F64), beta.to(F64), 1e-5)
            sigma = x64.var(1, correction=0, keepdim=True).add(1e-5).sqrt()
            rel = 4 * 2.0 ** -24 * c ** 0.5 * (1 + x64.abs().mean(1, keepdim=True) / sigma)
            gate = (R_BF16 if dtype == BF else 2.0 ** -22) * ref.abs() + gamma.abs().to(F64) * rel + 1e-6 * beta.abs().to(F64)
            wrong = None
            if dtype == torch.float32 and not shifted and c >= 64:
                # unbiased (c - 1) variance instead of the biased one
                wrong = (x64 - x64.mean(1, keepdim=True)) / x64.var(1, correction=1, keepdim=True).add(1e-5).sqrt() \
                    * gamma.to(F64) + beta.to(F64)
            if shifted and rows > 1:
                # one-pass variance in fp32
                xf = x
                var1 = ((xf * xf).mean(1, keepdim=True) - xf.mean(1, keepdim=True) ** 2).clamp(min=0)
                wrong = ((xf - xf.mean(1, keepdim=True)) / (var1 + 1e-5).sqrt() * gamma + beta).to(F64)
            check("layernorm c%d %s rows%d shifted%d" % (c, dtype, rows, shifted), out, ref, gate, wrong)


@gpu
@pytest.mark.parametrize("H,W,Hp,Wp,y0,x0", [(7, 40, 12, 48, 2, 5), (33, 7, 40, 16, 4, 3), (7, 7, 9, 9, 1, 2),
                                              (45, 70, 64, 96, 9, 13), (32, 64, 32, 64, 0, 0)])
def test_frame_metrics_forms(H, W, Hp, Wp, y0, x0):
    """Per-frame MSE / SSIM against O.mse / O.ssim_uniform7 in float64 with data_range 1 and 2 (the reference's default),
    identical frames (MSE 0, SSIM 1), constant frames (zero variance), one valid SSIM row / column (H or W = 7), sizes
    that are not multiples of the 32-pixel tile and nonzero crop offsets."""
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(H * W + y0)
    pred = torch.rand(4, Hp, Wp, generator=g)
    gt = torch.rand(4, H, W, generator=g)
    gt[1] = pred[1, y0:y0 + H, x0:x0 + W]            # identical
    pred[2].fill_(0.25)                              # constant prediction
    gt[2].fill_(0.75)                                # constant ground truth
    gt[3] = (pred[3, y0:y0 + H, x0:x0 + W] * 0.5 + 0.1 * gt[3]).contiguous()   # correlated
    for dr in (1.0, 2.0):
        out, names = launched(lambda: ops.frame_metrics(pred.to(DEV), gt.to(DEV), y0, x0, dr))
        assert_route(names, ("kernel", "frame_metrics_kernel"))
        out = out.cpu()
        for i in range(4):
            crop = pred[i, y0:y0 + H, x0:x0 + W].to(F64)
            mse = float(((crop - gt[i].to(F64)) ** 2).mean())
            ssim = O.ssim_uniform7(crop, gt[i].to(F64), dr)
            print("frame_metrics %dx%d dr%.0f frame %d: mse err %.2e ssim err %.2e" % (H, W, dr, i, abs(out[i, 0] - mse),
                                                                                       abs(out[i, 1] - ssim)))
            assert abs(float(out[i, 0]) - mse) <= 1e-12 * max(mse, 1e-30) + 1e-15
            assert abs(float(out[i, 1]) - ssim) <= 1e-10
            if i != 1:
                # data_range 1 instead of 2 (or 2 instead of 1) gives a different SSIM
                assert abs(float(out[i, 1]) - O.ssim_uniform7(crop, gt[i].to(F64), 3.0 - dr)) > 1e-6
        assert float(out[1, 0]) == 0.0 and abs(float(out[1, 1]) - 1.0) <= 1e-12


@gpu
@pytest.mark.parametrize("cin", [1, 5, 6])
def test_head_conv_forms(cin):
    """Direct 5 x 5 head conv from the planar voxel grid: ACT_NONE and ACT_RELU6 with pre-activations on both sides of
    both clamps, cin in {1, 5, 6} (odd counts leave a zero-weight half channel pair)."""
    from bde2vid_b200 import ops
    n, h, w = 2, 37, 45
    g = torch.Generator().manual_seed(cin)
    vox = torch.randn(n, cin, h, w, generator=g)
    wt = torch.randn(32, cin, 5, 5, generator=g) * (4.0 / (25 * cin) ** 0.5)
    b = 2.0 + 0.5 * torch.randn(32, generator=g)
    pre, mass = conv64([rnd(vox, BF)], rnd(wt, BF), b.to(F64))
    frac = [float((pre < 0).double().mean()), float(((pre > 0) & (pre < 6)).double().mean()), float((pre > 6).double().mean())]
    assert min(frac) >= 0.10, frac
    for act in (ops.ACT_NONE, ops.ACT_RELU6):
        out = torch.full((n, h, w, 32), float("nan"), dtype=BF, device=DEV)
        _, names = launched(lambda: ops.head_conv(vox.to(DEV), wt.to(DEV), b.to(DEV), out, act=act))
        assert_route(names, ("kernel", "head_conv_kernel"))
        ref = pre if act == ops.ACT_NONE else pre.clamp(0.0, 6.0)
        wrong = F.relu(pre)
        check("head_conv cin%d act%d" % (cin, act), nchw64(out), ref, R_BF16 * ref.abs() + E_ACC * mass, wrong)


@gpu
def test_pack_voxel_and_cast_bit_exact():
    """bde_pack_voxel_nhwc (planar fp32 -> NHWC with zero channel padding) and bde_cast are pure conversions: bit-exact
    against torch's round-to-nearest-even for every supported pair, at sizes that are not multiples of the 256-thread
    block; an unsupported dtype pair is refused."""
    from bde2vid_b200 import _lib, ops
    g = torch.Generator().manual_seed(5)
    for (N, bins, Hp, Wp, cpad) in ((3, 5, 13, 19, 8), (1, 6, 7, 37, 8), (2, 1, 5, 3, 4)):
        vox = torch.randn(N, bins, Hp, Wp, generator=g) * 3
        vox[0, 0, 0, :3] = torch.tensor([1.0 + 2 ** -8, -(1.0 + 3 * 2 ** -8), 1e-40])   # ties and a subnormal
        for dtype in (torch.float32, BF):
            out, names = launched(lambda: ops.pack_voxel_nhwc(vox.to(DEV), cpad, dtype))
            assert_route(names, ("kernel", "pack_voxel_kernel"))
            ref = torch.zeros(N, Hp, Wp, cpad)
            ref[..., :bins] = vox.permute(0, 2, 3, 1)
            assert torch.equal(out.cpu().view(torch.int16 if dtype == BF else torch.int32),
                               ref.to(dtype).view(torch.int16 if dtype == BF else torch.int32))
    for n in (1, 255, 257, 1000):
        src = torch.randn(n, generator=g) * 100
        src[0] = 1.0 + 2 ** -8
        for s_t, d_t in ((torch.float32, BF), (BF, torch.float32), (torch.float32, torch.float32)):
            s = src.to(s_t).to(DEV)
            d = torch.full((n,), float("nan"), dtype=d_t, device=DEV)
            _, names = launched(lambda: ops.cast(s, d))
            assert_route(names, ("kernel", "cast_kernel"))
            ref = s.cpu().to(d_t)
            iv = torch.int16 if d_t == BF else torch.int32
            assert torch.equal(d.cpu().view(iv), ref.view(iv))
    with pytest.raises(RuntimeError, match="unsupported dtype pair"):
        ops.cast(torch.zeros(8, dtype=BF, device=DEV), torch.zeros(8, dtype=BF, device=DEV))
    lib = _lib.load()
    vox = torch.zeros(1, 2, 3, 3, device=DEV)
    out = torch.zeros(1, 3, 3, 4, device=DEV)
    assert lib.bde_pack_voxel_nhwc(_lib.ptr(vox), 1, 2, 3, 3, 4, _lib.ptr(out), 7, _lib.stream_ptr()) != 0


@gpu
@pytest.mark.parametrize("C", [64, 256])
@pytest.mark.parametrize("q_ind", [0, 1, 2])
def test_window_attention_mma_qkv(C, q_ind):
    """Tensor-core attention reading q / k / v from the merged [n_win * n_kv, 3C] projection buffer, query rows at
    q_row0 = q_ind * 49, against float64 softmax attention.  Gate: P and V enter the second MMA as fp16 (2 x 2^-11
    relative on sum p |v|) on top of the bf16 store."""
    from bde2vid_b200 import ops
    heads, D, nq = 16, 3, 49
    hd, n_kv, nwin = C // heads, D * nq, 23
    g = torch.Generator().manual_seed(C + q_ind)
    qkv = rnd(torch.randn(nwin, n_kv, 3 * C, generator=g, dtype=F64), BF)
    qkv[..., :C] *= hd ** -0.5
    qkv = rnd(qkv, BF)
    bias = torch.randn(heads, nq, n_kv, generator=g, dtype=F64).float().to(F64)
    bp = ops.pad_bias_for_mma(bias.float().to(DEV), n_kv)
    out = torch.full((nwin, nq, C), float("nan"), dtype=BF, device=DEV)
    _, names = launched(lambda: ops.window_attention_mma_qkv(qkv.view(nwin * n_kv, 3 * C).to(DEV, BF), bp, nwin, nq, n_kv,
                                                             q_ind * nq, C, heads, out))
    assert_route(names, ("kernel", "window_attention_mma_kernel"))

    def attn(q_rows):
        qh = qkv[:, q_rows, :C].reshape(nwin, nq, heads, hd).permute(0, 2, 1, 3)
        kh = qkv[..., C:2 * C].reshape(nwin, n_kv, heads, hd).permute(0, 2, 1, 3)
        vh = qkv[..., 2 * C:].reshape(nwin, n_kv, heads, hd).permute(0, 2, 1, 3)
        p = torch.softmax(qh @ kh.transpose(-1, -2) + bias, -1)
        return (p @ vh).permute(0, 2, 1, 3).reshape(nwin, nq, C), (p @ vh.abs()).permute(0, 2, 1, 3).reshape(nwin, nq, C)
    ref, mass = attn(slice(q_ind * nq, (q_ind + 1) * nq))
    wrong, _ = attn(slice(((q_ind + 1) % D) * nq, ((q_ind + 1) % D + 1) * nq))   # another frame's query rows
    check("attention mma qkv C%d q_ind %d" % (C, q_ind), out, ref, R_BF16 * ref.abs() + 2.0 ** -9 * mass + E_ACC * mass, wrong)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: the reference helpers against the oracle functions they restate
# ---------------------------------------------------------------------------------------------------------------------
def test_gru_reference_matches_oracle():
    g = torch.Generator().manual_seed(0)
    C, B, h, w = 8, 2, 5, 7
    sd = {"g.update_gate.weight": torch.randn(C, 2 * C, 3, 3, generator=g, dtype=F64),
          "g.update_gate.bias": torch.randn(C, generator=g, dtype=F64),
          "g.reset_gate.weight": torch.randn(C, 2 * C, 3, 3, generator=g, dtype=F64),
          "g.reset_gate.bias": torch.randn(C, generator=g, dtype=F64),
          "g.out_gate.weight": torch.randn(C, 2 * C, 3, 3, generator=g, dtype=F64),
          "g.out_gate.bias": torch.randn(C, generator=g, dtype=F64)}
    ws = [sd["g." + k] for k in ("update_gate.weight", "update_gate.bias", "reset_gate.weight", "reset_gate.bias",
                                 "out_gate.weight", "out_gate.bias")]
    x = torch.randn(B, C, h, w, generator=g, dtype=F64)
    for state in (None, torch.randn(B, C, h, w, generator=g, dtype=F64)):
        ref = O.convgru_step(sd, "g", x, state)
        assert torch.allclose(gru_step_ref(x, state, *ws), ref, rtol=0, atol=1e-12)
    # the engine's interleaved packing (rows n = 2c + g) puts update in even and reset in odd rows
    wi = torch.stack([ws[0], ws[2]], 1).reshape(2 * C, 2 * C, 3, 3)
    assert torch.equal(wi[0::2], ws[0]) and torch.equal(wi[1::2], ws[2])


@pytest.mark.parametrize("X", [1, 4, 9])
def test_window_reduce_reference_matches_grouped_conv(X):
    """window_reduce_ref restates the oracle's grouped convolution (oracle_torch.py attention_block: Conv2d(C, X*C,
    window, groups=C) over every (frame, window), result viewed as [X, C])."""
    from bde2vid_b200.engine import window_token_map
    g = torch.Generator().manual_seed(X)
    B, H, W, C, D = 1, 9, 15, 8, 2
    frames = [torch.randn(B * H * W, C, generator=g, dtype=F64), None]
    rw = torch.randn(C * X, 1, 7, 7, generator=g, dtype=F64)
    rb = torch.randn(C * X, generator=g, dtype=F64)
    for dil in (False, True):
        tm, _ = window_token_map(B, H, W, (7, 7), dil, "cpu")
        nwin = tm.shape[0]
        tok = window_tokens(frames, tm, C)
        img = torch.stack([t.reshape(nwin, 7, 7, C).permute(0, 3, 1, 2) for t in tok], 0).contiguous()
        red = F.conv2d(img.view(-1, C, 7, 7), rw, rb, groups=C).view(D, nwin, X, C).permute(1, 0, 2, 3)
        mine, _ = window_reduce_ref(frames, tm, C, X, rw.view(C * X, 49), rb)
        assert torch.allclose(mine, red, rtol=0, atol=1e-12)


def test_concat_prediction_folding_matches_two_convs():
    """engine.py folds predI's two 1 x 1 convolutions (2c -> c, then c -> 1, nothing in between) into one [2c] vector
    and one bias: w_eff = W2 W1, split as (x | head) weights.  In float64 this equals the oracle's two convolutions
    over cat[x, head] (oracle_torch.py bde2vid_forward)."""
    g = torch.Generator().manual_seed(3)
    c, n, h, w = 16, 2, 5, 6
    W1 = torch.randn(c, 2 * c, 1, 1, generator=g, dtype=F64)
    b1 = torch.randn(c, generator=g, dtype=F64)
    W2 = torch.randn(1, c, 1, 1, generator=g, dtype=F64)
    b2 = torch.randn(1, generator=g, dtype=F64)
    x = torch.randn(n, c, h, w, generator=g, dtype=F64)
    head = torch.randn(n, c, h, w, generator=g, dtype=F64)
    two = F.conv2d(F.conv2d(torch.cat([x, head], 1), W1, b1), W2, b2)
    pw = W2.reshape(-1)
    w_eff = pw @ W1.reshape(c, 2 * c)
    pred_w, pred_wh, pred_b = w_eff[:c], w_eff[c:], pw @ b1 + b2
    one = torch.einsum("nchw,c->nhw", x, pred_w) + torch.einsum("nchw,c->nhw", head, pred_wh) + pred_b
    assert torch.allclose(one, two[:, 0], rtol=0, atol=1e-12)
    # exchanging the halves (head first) is a different map
    wrong = torch.einsum("nchw,c->nhw", x, pred_wh) + torch.einsum("nchw,c->nhw", head, pred_w) + pred_b
    assert not torch.allclose(wrong, two[:, 0], rtol=0, atol=1e-3)


def test_route_parser_reads_both_name_forms():
    """The route assertions read kernel names as the profiler reports them, demangled or mangled."""
    dem = "void bde::tc::conv_tma_kernel<64, true, 2, false, 2>(CUtensorMap, CUtensorMap, CUtensorMap, bde::tc::CvParams)"
    man = "_ZN3bde2tc15conv_tma_kernelILi128ELb0ELi0ELb0ELi1EEEv14CUtensorMap_stS2_S2_NS0_8CvParamsE"
    assert tma_forms({dem}) == [(64, True, 2, False, 2)]
    assert tma_forms({man}) == [(128, False, 0, False, 1)]
    assert has_kernel({"void bde::upsample2x_sum_block_kernel<float, float>(...)"}, "upsample2x_sum_block_kernel")
    assert not has_kernel({"void bde::upsample2x_sum_block_kernel<float, float>(...)"}, "upsample2x_sum_kernel")
    assert has_kernel({"_ZN3bde21upsample2x_sum_kernelIffE"}, "upsample2x_sum_kernel")
    assert not has_kernel({"void bde::ln_gather_qkv_kernel<float, 8>(...)"}, "layernorm_kernel")
