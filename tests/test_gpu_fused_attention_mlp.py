"""Kernel-level float64 references for the fused window-attention kernels (bde_window_attention_fused,
bde_window_attention_fused_kvpre: attn_fused.cu, attn_tc256.cu) and the fused transformer MLPs (bde_mlp_fused,
bde_mlp_fused_sum: mlp_fused.cu), one case per kernel instance, in the call forms the engine makes.

The references restate DTransformer.py:183-207 (WindowAttention3D) and 279-306 (the block's shortcut and MLP) in plain
float64 torch on the operands exactly as the kernels receive them: fp32 frames, bf16 wqkv with the LayerNorm affine and
the q scale folded in, fp32 bqkv, the compact fp32 bias table [heads, D, 169] indexed analytically, bf16 wproj, fp32
bproj; bf16 w1 (norm2 folded in), fp32 b1, bf16 w2, fp32 b2.  Zero tokens (map -1, or a None frame) enter the LayerNorm
as zeros and their keys stay in the softmax, as in the oracle.

Gates are PER ELEMENT.  The kernels store several intermediates in narrow types; the reference stores the same ones
(mirrored stores) and gives each an allowance only where its rounding is undetermined:

    flip(a, e, dtype) = |rnd(a + e) - rnd(a - e)|     (0 where both neighbours round alike, one ulp where they do not)
    ar = rnd(a),  delta_a = e_a + flip(a, e_a)        for a float64 value a the kernel computes to within e_a

Rounding points.  Attention: xhat -> bf16; q, k -> bf16; v -> fp16 (satfinite); the unnormalised p -> fp16; o -> bf16
(o_out, or in front of the projection).  MLP: xhat -> bf16; the GELU output -> bf16.  First-order propagation:

    LayerNorm  e_xhat = |xhat| (rho / 2 + R_SQRT + 2u) + dmu * rstd,  dmu = (L + 1) u mean|x|,
               rho = (L + 6) u + dmu^2 / (var + 1e-5)       (two-pass fp32 statistics; L = C / 8 + 3 is the longest
               add chain: one lane sums C / 8 values, then three shuffle levels)
    q, k, v    e = E_ACC (|xr| |W|^T + |b|) + delta_xr |W|^T
    scores     e_s = E_ACC (|qr| |kr|^T + |bias|) + delta_q |kr|^T + |qr| delta_k^T + u (|s| + 2 max_row |s|)
               (the last term: fp32 rounding of the exp2 argument s log2e - m)
    o          e_o = sum_j [p_j (e_s,j + 2 u_h + E_EX2) + H_SUB] |vr_j - o| + sum_j p_j delta_v,j
                     + E_ACC (sum_j p_j |vr_j| + |o|) + (E_RCP + u) |o|
               2 u_h covers the fp16 p, which enters numerator and denominator alike; H_SUB the absolute rounding of a
               p below the fp16 normal range; the denominator is >= 1.  Nothing here depends on the order in which the
               keys are visited, so the online softmax of attn_tc256.cu / the segmented one of the C = 64 kernel need
               no mirroring.
    projection e_y = E_ACC (|or| |Wp|^T + |bp|) + delta_or |Wp|^T;  the fp32 update x + (acc + bp) adds u (|x| + 2|y|)
    MLP        e_h as q; fast_gelu adds (GELU_FORM + TANH_APPROX / 2 + 16 u) |h| + GELU_LIP e_h before the hidden bf16
               store; fc2 as the projection; the sum_io form adds one fp32 rounding u |sum|; sum_t is bit-exact
               against sum_io.to(bf16).

Constants (u = 2^-24, u_h = 2^-11 are the fp32 / fp16 unit roundoffs):
    E_ACC     1e-5    fp32 accumulation, relative to the absolute mass of the sum (test_gpu_kernel_forms.py)
    R_SQRT    2^-22   rsqrt.approx.f32 (PTX ISA: max relative error 2^-22.9) and rsqrtf (CUDA C Programming Guide: 2 ulp)
    E_EX2     2^-22   ex2.approx.ftz.f32 (PTX ISA: max relative error 2 ulp over the full range)
    E_RCP     2^-23   rcp.approx.ftz.f32 (PTX ISA: max relative error 1 ulp)
    H_SUB     2^-25   half the spacing of fp16 subnormals
    GELU_FORM 5.4e-5  the fitted quintic of fast_gelu, absolute on Phi(x) (DESIGN.md section 2), valid with the
                      polynomial frozen beyond |x| = 5
    TANH_APPROX 2^-11 tanh.approx.f32, relative (PTX ISA)
    GELU_LIP  1.13    max |GELU'(x)| (1.1289 at x = 1.4)
    16 u      the handful of fp32 roundings in fast_gelu's argument (|r| <= 1.5 |x|) and its final fma

On a B200 (1000 W power limit) the largest err / gate seen was 0.996 on the bf16 o_out stores (a one-ulp flip against
a gate of ulp + e, tight by construction), 0.17 on the fp32 updates of the C = 64 kernels, 0.03 on those of the C = 256
kernels, 0.18 / 0.08 on the C = 64 / C = 256 MLPs.

Every case prints its largest err / gate and asserts, with torch.profiler, which kernel instance served it; the test ids
name the instances (all 24 of profiles/sass/{attn_fused,attn_tc256,mlp_fused}.kernels.txt).  Each family also checks that
a plausibly wrong reference fails the same gate.  (tanh-GELU is not among them: it differs from erf-GELU by at most
1.8e-4 |h|, inside the 2.4e-4 |h| that tanh.approx alone is allowed, so no sound gate can separate the two.)

The CPU tests at the end pin the references (without roundings, exact GELU) to O.attention_block, check the flip helper
and the kernel-name parser.
"""
import re

import pytest
import torch
import torch.nn.functional as F

from oracle import oracle_torch as O
from test_gpu_kernel_forms import BF, DEV, E_ACC, F64, GELU_FORM, TANH_APPROX, check, gate_ratio, gpu, launched, rnd

F16 = torch.float16
U32 = 2.0 ** -24
U_H = 2.0 ** -11
R_SQRT = 2.0 ** -22
E_EX2 = 2.0 ** -22
E_RCP = 2.0 ** -23
H_SUB = 2.0 ** -25
GELU_LIP = 1.13
LN_EPS = 1e-5
TINY = 1e-300          # gate of an element that must be bit-unchanged


# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------
def flip(a, e, dtype):
    """One ulp of ``dtype`` where a +- e round differently, else 0."""
    return (rnd(a + e, dtype) - rnd(a - e, dtype)).abs()


def store(a, e, dtype, exact=False):
    """Mirrored store: (rnd(a), e + flip(a, e)); ``exact``: no rounding at all."""
    if exact:
        return a, torch.zeros_like(a)
    return rnd(a, dtype), e + flip(a, e, dtype)


def ln_ref(x, ln_eps=LN_EPS):
    """Affine-free LayerNorm over the last dim in float64 and the error bound of the kernels' fp32 two-pass form."""
    C = x.shape[-1]
    L = C // 8 + 3
    mu = x.mean(-1, keepdim=True)
    d = x - mu
    var = (d * d).mean(-1, keepdim=True)
    rstd = (var + ln_eps).rsqrt()
    xhat = d * rstd
    dmu = (L + 1) * U32 * x.abs().mean(-1, keepdim=True)
    rho = (L + 6) * U32 + dmu ** 2 / (var + ln_eps)
    return xhat, xhat.abs() * (0.5 * rho + R_SQRT + 2 * U32) + dmu * rstd


def linear_ref(xr, dx, w, b, dtype, exact=False):
    """Mirrored store of xr w^T + b (fp32 accumulation) with its delta."""
    a = xr @ w.t() + b
    e = E_ACC * (xr.abs() @ w.abs().t() + b.abs()) + dx @ w.abs().t()
    return store(a, e, dtype, exact)


def rel_index():
    """Analytic 13 x 13 relative offset of (query token, key token) of a 7 x 7 window (DTransformer.py:139-152)."""
    a = torch.arange(7)
    ai, bi = a.repeat_interleave(7), a.repeat(7)
    return (ai[:, None] - ai[None, :] + 6) * 13 + (bi[:, None] - bi[None, :] + 6)


def win_tokens(f, tm):
    """[nwin, 49, C] tokens of frame f (float64 [P, C] or None) through the token map (-1 = zero token)."""
    if f is None:
        return None
    return f[tm.clamp(min=0)] * (tm >= 0).unsqueeze(-1).to(F64)


def attn_ref(frames, q_slot, tm, wqkv, bqkv, tbl, wproj, bproj, heads, kvpre=None, exact=False, ln_eps=LN_EPS,
             wrong=None, chunk=None):
    """Attention half in float64 with mirrored stores.  frames: D float64 [P, C] maps or None; tm: long [nwin, 49];
    wqkv / wproj: float64 values of the bf16 weights; kvpre: per slot None or float64 [P, 2C] k | v rows (bf16 values;
    the query slot is ignored).  wrong: None, "mirror_tbl", "softmax_per_frame" or "drop_zero_keys".
    Returns (o, d_o [nwin * 49, C], y, e_y [nwin * 49, C]); y and e_y are None without wproj."""
    D = len(frames)
    C = wqkv.shape[1]
    hd = C // heads
    nwin = tm.shape[0]
    N = D * 49
    dev = tm.device
    rel = rel_index().to(dev)
    tb = tbl.flip(1) if wrong == "mirror_tbl" else tbl
    bias = torch.cat([tb[:, d][:, rel] for d in range(D)], 2)                                 # [heads, 49, N]
    Wq, Wk, Wv = wqkv[:C], wqkv[C:2 * C], wqkv[2 * C:]
    bq, bk, bv = bqkv[:C], bqkv[C:2 * C], bqkv[2 * C:]
    if chunk is None:
        chunk = max(1, 2 ** 25 // (heads * 49 * N * hd))
    outs = []
    for w0 in range(0, nwin, chunk):
        t = tm[w0:w0 + chunk]
        nw = t.shape[0]
        ks, dks, vs, dvs, valid = [], [], [], [], []
        for d in range(D):
            src = win_tokens(frames[d], t) if (kvpre is None or d == q_slot) else None
            valid.append((t >= 0) & (frames[d] is not None if kvpre is None or d == q_slot else kvpre[d] is not None))
            if kvpre is not None and d != q_slot:
                # precomputed neighbour k | v as given (bf16); zero tokens take the bias rounded to bf16
                kvz = torch.cat([rnd(bk, BF), rnd(bv, BF)]).expand(nw, 49, 2 * C)
                kv = kvz if kvpre[d] is None else torch.where((t >= 0).unsqueeze(-1), kvpre[d][t.clamp(min=0)], kvz)
                ks.append(kv[..., :C])
                dks.append(torch.zeros_like(kv[..., :C]))
                vs.append(rnd(kv[..., C:], F16))
                dvs.append(torch.zeros_like(kv[..., :C]))
                continue
            if src is None:
                src = torch.zeros(nw, 49, C, dtype=F64, device=dev)
            xhat, ex = ln_ref(src, ln_eps)
            xr, dx = store(xhat, ex, BF, exact)
            if d == q_slot:
                q, dq = linear_ref(xr, dx, Wq, bq, BF, exact)
            k, dk = linear_ref(xr, dx, Wk, bk, BF, exact)
            v, dv = linear_ref(xr, dx, Wv, bv, F16, exact)
            ks.append(k)
            dks.append(dk)
            vs.append(v)
            dvs.append(dv)

        def heads_of(z):
            return z.reshape(nw, z.shape[1], heads, hd).permute(0, 2, 1, 3)
        qh, dqh = heads_of(q), heads_of(dq)
        kh, dkh = heads_of(torch.cat(ks, 1)), heads_of(torch.cat(dks, 1))
        vh, dvh = heads_of(torch.cat(vs, 1)), heads_of(torch.cat(dvs, 1))
        s = qh @ kh.transpose(-1, -2) + bias
        e_s = (E_ACC * (qh.abs() @ kh.abs().transpose(-1, -2) + bias.abs()) + dqh @ kh.abs().transpose(-1, -2)
               + qh.abs() @ dkh.transpose(-1, -2))
        e_s = e_s + U32 * (s.abs() + 2 * s.abs().amax(-1, keepdim=True))
        if wrong == "drop_zero_keys":
            s = s.masked_fill(~torch.cat(valid, 1).view(nw, 1, 1, N), float("-inf"))
        if wrong == "softmax_per_frame":
            p = torch.cat([torch.softmax(s[..., d * 49:(d + 1) * 49], -1) for d in range(D)], -1) / D
        else:
            p = torch.softmax(s, -1)
        o = p @ vh                                                                            # [nw, heads, 49, hd]
        wdev = p * (e_s + 2 * U_H + E_EX2) + H_SUB
        e_o = (wdev.unsqueeze(-1) * (vh.unsqueeze(2) - o.unsqueeze(3)).abs()).sum(3)
        e_o = e_o + p @ dvh + E_ACC * (p @ vh.abs() + o.abs()) + (E_RCP + U32) * o.abs()
        o = o.permute(0, 2, 1, 3).reshape(nw * 49, C)
        e_o = e_o.permute(0, 2, 1, 3).reshape(nw * 49, C)
        outs.append((o, e_o))
    o = torch.cat([a for a, _ in outs])
    e_o = torch.cat([b for _, b in outs])
    orr, d_o = store(o, e_o, BF, exact)
    if wproj is None:
        return orr, d_o, None, None
    y, e_y = linear_ref(orr, d_o, wproj, bproj, F64, True)
    e_y = E_ACC * (orr.abs() @ wproj.abs().t() + bproj.abs()) + d_o @ wproj.abs().t()
    return orr, d_o, y, e_y


def scatter_update(before, shortcut, tm, y, e_y):
    """(ref, gate) of the fp32 map after x[pix] = shortcut[pix] + y: covered pixels gated, the others bit-unchanged."""
    ref = before.clone()
    gate = torch.full_like(before, TINY)
    pix = tm.reshape(-1)
    sel = pix >= 0
    p = pix[sel]
    xs = shortcut[p]
    yy = y[sel]
    ref[p] = xs + yy
    gate[p] = e_y[sel] + U32 * (xs.abs() + 2 * yy.abs())
    return ref, gate


def gelu_form_gate(h):
    return (GELU_FORM + 0.5 * TANH_APPROX + 16 * U32) * h.abs()


def mlp_ref(x, w1, b1, w2, b2, exact=False, ln_eps=LN_EPS, gelu=F.gelu):
    """x + fc2(GELU(fc1(LN(x)))) in float64 with mirrored stores; returns (ref, gate, h)."""
    xhat, ex = ln_ref(x, ln_eps)
    xr, dx = store(xhat, ex, BF, exact)
    h = xr @ w1.t() + b1
    e_h = E_ACC * (xr.abs() @ w1.abs().t() + b1.abs()) + dx @ w1.abs().t()
    g = gelu(h)
    gr, dg = store(g, gelu_form_gate(h) + GELU_LIP * e_h, BF, exact)
    y = gr @ w2.t() + b2
    e_y = E_ACC * (gr.abs() @ w2.abs().t() + b2.abs()) + dg @ w2.abs().t()
    ref = x + y
    return ref, e_y + U32 * (x.abs() + 2 * y.abs()), h


# ---------------------------------------------------------------------------------------------------------------------
# kernel instances
# ---------------------------------------------------------------------------------------------------------------------
_KERNEL = re.compile(r"(attn_fused_kernel|attn_win256_tc_kernel|attn_win256_kernel|mlp_fused256_kernel|mlp_fused_kernel)"
                     r"(?:<([^<>]*)>|I((?:L[ib]\d+E)+)E)?")


def instances(names):
    """Instance strings (``base<arg, ...>`` as in profiles/sass/*.kernels.txt) of the fused kernels among ``names``,
    from demangled (``attn_fused_kernel<64, 4, 7, false>``) or mangled (``attn_fused_kernelILi64ELi4ELi7ELb0EE``) names."""
    out = set()
    for n in names:
        for m in _KERNEL.finditer(n):
            base, dem, man = m.groups()
            if dem is not None:
                args = [a.strip() for a in dem.split(",")]
            elif man is not None:
                args = [v if k == "i" else ("true" if v == "1" else "false") for k, v in re.findall(r"L([ib])(\d+)E", man)]
            else:
                args = None
            out.add(base if not args else "%s<%s>" % (base, ", ".join(args)))
    return out


def run_routed(fn, inst):
    """fn() under the profiler; assert that exactly the fused instance ``inst`` ran."""
    _, names = launched(fn)
    got = instances(names)
    print("profiled:", [n for n in names if instances([n])])
    assert got == {inst}, (inst, got, sorted(names))


def sm_count():
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------
# attention inputs
# ---------------------------------------------------------------------------------------------------------------------
def token_rows(P, C, g):
    """Rows with a non-zero mean and a per-row standard deviation spread log-uniformly over [1e-3, 1e2]: below
    sqrt(1e-5) = 3.2e-3 the LayerNorm epsilon dominates the variance."""
    std = 10.0 ** (5 * torch.rand(P, 1, generator=g, dtype=F64) - 3)
    mean = 0.5 * torch.randn(P, 1, generator=g, dtype=F64) + 0.3
    return (mean + std * torch.randn(P, C, generator=g, dtype=F64)).float()


class AttnSetup:
    """Operands of one attention block as the engine passes them (device tensors) and their float64 values."""

    def __init__(self, C, D, P, seed, tbl_scale):
        g = torch.Generator().manual_seed(seed)
        heads = 16
        hd = C // heads
        self.C, self.D, self.P, self.heads = C, D, P, heads
        self.frames = [token_rows(P, C, g).to(DEV) for _ in range(D)]
        w = torch.randn(3 * C, C, generator=g, dtype=F64) / C ** 0.5
        w[:C] *= hd ** -0.5
        self.wqkv = w.to(BF).to(DEV)
        self.bqkv = (0.1 * torch.randn(3 * C, generator=g)).to(DEV)
        self.tbl = (tbl_scale * torch.randn(heads, D, 169, generator=g)).to(DEV)
        self.wproj = (torch.randn(C, C, generator=g, dtype=F64) / C ** 0.5).to(BF).to(DEV)
        self.bproj = (0.1 * torch.randn(C, generator=g)).to(DEV)

    def f64(self, t):
        return None if t is None else t.to(F64)

    def ref(self, frames, q_slot, tm, proj=True, **kw):
        return attn_ref([self.f64(f) for f in frames], q_slot, tm.long(), self.f64(self.wqkv), self.f64(self.bqkv),
                        self.f64(self.tbl), self.f64(self.wproj) if proj else None, self.f64(self.bproj), self.heads, **kw)

    def launch(self, frames, q_slot, tm, xs=None, o_out=None):
        from bde2vid_b200 import ops
        ops.window_attention_fused(frames, q_slot, tm.view(-1), tm.shape[0], self.C, self.heads, self.wqkv, self.bqkv,
                                   self.tbl, None if o_out is not None else self.wproj,
                                   None if o_out is not None else self.bproj, xs=xs, o_out=o_out)


def tmap(B, H, W, dilated):
    from bde2vid_b200.engine import window_token_map
    return window_token_map(B, H, W, (7, 7), dilated, DEV)[0]


def run_update(S, frames, q_slot, tm, inst, direct, name, wrongs=(), **kw):
    """One projected launch (in place on a copy of the query frame, or direct: query frame = frames[q_slot], xs a
    NaN-filled separate map), checked against the reference; returns the output map."""
    q = frames[q_slot]
    q0 = q.clone()
    if direct:
        xs = torch.full_like(q, float("nan"))
        fr = list(frames)
    else:
        xs = q.clone()
        fr = list(frames)
        fr[q_slot] = xs
    run_routed(lambda: S.launch(fr, q_slot, tm, xs=xs, **kw), inst)
    if direct:
        assert torch.equal(q, q0), "the query frame was written"
        assert bool((tm.reshape(-1) >= 0).sum() == q.shape[0]), "direct form needs a map that covers every pixel"
    _, _, y, e_y = S.ref(frames, q_slot, tm)
    before = torch.full_like(q0, float("nan")).to(F64) if direct else q0.to(F64)
    ref, gate = scatter_update(before, q0.to(F64), tm.long(), y, e_y)
    if direct:
        gate = torch.where(torch.isnan(ref), torch.full_like(gate, TINY), gate)
    for wr in wrongs:
        if wr == "neighbour_shortcut":
            other = frames[(q_slot + 1) % len(frames)]
            wref, _ = scatter_update(before, torch.zeros_like(before) if other is None else other.to(F64), tm.long(), y, e_y)
        elif wr == "ln_eps":
            wref, _ = scatter_update(before, q0.to(F64), tm.long(), *S.ref(frames, q_slot, tm, ln_eps=1e-6)[2:])
        else:
            wref, _ = scatter_update(before, q0.to(F64), tm.long(), *S.ref(frames, q_slot, tm, wrong=wr)[2:])
        rw = gate_ratio(xs, wref, gate)
        assert rw > 1.0, "%s: the wrong reference '%s' passes the gate too (err/gate %.3f)" % (name, wr, rw)
    check(name, xs, ref, gate)
    return xs


ATTN64 = ["attn_fused_kernel<64, 4, %d, false>" % nt for nt in (7, 13, 19)]
ATTN64_PERS = ["attn_fused_kernel<64, 4, %d, true>" % nt for nt in (7, 13, 19)]
TC256 = ["attn_win256_tc_kernel<%d, %d>" % (nt, cl) for nt in (7, 13, 19) for cl in (1, 2)]
WIN256 = ["attn_win256_kernel<%d, false>" % nt for nt in (7, 13, 19)]
KVPRE = ["attn_win256_kernel<%d, true>" % nt for nt in (13, 19)]
HG256 = ["attn_fused_kernel<256, 16, %d, false>" % nt for nt in (7, 13, 19)]
MLP64 = "mlp_fused_kernel"
MLP256 = ["mlp_fused256_kernel<%d>" % cl for cl in (1, 2, 4)]
NT_D = {7: 1, 13: 2, 19: 3}


def nt_of(inst):
    return int(re.search(r"<(?:64, 4, |256, 16, )?(\d+)", inst).group(1))


# ---------------------------------------------------------------------------------------------------------------------
# C = 64, 16 heads of 4 channels (level 1)
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("inst", ATTN64)
def test_attn64(inst):
    """attn_fused_kernel<64, 4, NT, false> on the model's level-1 map (132 x 176: 494 ragged windows): q_slot at every
    position, a None frame in each non-query slot, plain and dilated maps, in-place and direct forms, bias tables at
    scale 0.02 and 1.0."""
    D = NT_D[nt_of(inst)]
    H, W = 132, 176
    tms = {dil: tmap(1, H, W, dil) for dil in (False, True)}
    assert tms[False].shape[0] == 494
    run = 0
    for q_slot in range(D):
        for zero in [None] + [z for z in range(D) if z != q_slot]:
            S = AttnSetup(64, D, H * W, seed=100 * D + 10 * q_slot + (0 if zero is None else zero + 1),
                          tbl_scale=0.02 if run % 2 else 1.0)
            frames = list(S.frames)
            if zero is not None:
                frames[zero] = None
            for dil in (False, True):
                wrongs = ()
                if D == 3 and q_slot == 0 and zero == 2 and not dil:
                    wrongs = ("mirror_tbl", "softmax_per_frame", "neighbour_shortcut", "drop_zero_keys", "ln_eps")
                elif D == 1 and not dil:
                    wrongs = ("drop_zero_keys", "ln_eps")
                run_update(S, frames, q_slot, tms[dil], inst, direct=not dil,
                           name="%s q%d zero%s dil%d tbl%d" % (inst, q_slot, zero, dil, run % 2), wrongs=wrongs)
            run += 1


@gpu
@pytest.mark.parametrize("inst", ATTN64_PERS)
def test_attn64_persistent(inst, monkeypatch):
    """attn_fused_kernel<64, 4, NT, true> (BDE2VID_ATTN64_PERSIST=1) on two level-1 maps (988 windows: each of the
    2 x SMs halves walks several) sliced to an odd (987) and an even (988) window count, in place: bit-identical to the
    one-window-per-CTA form, within the gate of the reference, and the pixels of the sliced-off window bit-unchanged.
    n_win = 1 falls back to the per-window kernel."""
    NT = nt_of(inst)
    D = NT_D[NT]
    q_slot = D // 2
    H, W = 132, 176
    S = AttnSetup(64, D, 2 * H * W, seed=7 + NT, tbl_scale=1.0)
    frames = list(S.frames)
    if D > 1:
        frames[(q_slot + 1) % D] = None
    full = tmap(2, H, W, True)
    assert full.shape[0] == 988
    for n in (987, 988):
        tm = full[:n].contiguous()
        monkeypatch.setenv("BDE2VID_ATTN64_PERSIST", "1")
        xp = run_update(S, frames, q_slot, tm, inst, direct=False, name="%s n_win %d" % (inst, n))
        monkeypatch.setenv("BDE2VID_ATTN64_PERSIST", "0")
        xs = frames[q_slot].clone()
        fr = list(frames)
        fr[q_slot] = xs
        run_routed(lambda: S.launch(fr, q_slot, tm, xs=xs), "attn_fused_kernel<64, 4, %d, false>" % NT)
        assert torch.equal(xp, xs), "persistent and one-window-per-CTA forms differ"
    monkeypatch.setenv("BDE2VID_ATTN64_PERSIST", "1")
    run_update(S, frames, q_slot, full[:1].contiguous(), "attn_fused_kernel<64, 4, %d, false>" % NT, direct=False,
               name="%s n_win 1 -> per-window kernel" % inst)


# ---------------------------------------------------------------------------------------------------------------------
# C = 256, 16 heads of 16 channels (level 3)
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("inst", TC256)
def test_attn256_tc(inst, monkeypatch):
    """attn_win256_tc_kernel<NT, CL>: the automatic cluster choice (CL = 2 while 2 n_win <= SMs) on its side of the
    boundary, reached by slicing rows of the token map, the model's 33 x 44 map (35 windows per image, padding in the
    plain windows) plain and dilated, in-place and direct, then the other cluster size forced on the same operands,
    repeat launches bit-identical."""
    NT, CL = [int(v) for v in re.findall(r"\d+", inst.split("<")[1])]
    D = NT_D[NT]
    q_slot = min(1, D - 1)
    sms = sm_count()
    H, W = 33, 44
    B = 1 if CL == 2 else 3
    # (the wrong references below need the large-scale table: at 0.02 the mirrored slot's table moves the scores by
    # less than the gate; the checkpoint-like scale is covered by the boundary case)
    S = AttnSetup(256, D, B * H * W, seed=300 + NT + CL, tbl_scale=1.0)
    frames = list(S.frames)
    plain, dil = tmap(B, H, W, False), tmap(B, H, W, True)
    assert (2 * plain.shape[0] <= sms) == (CL == 2)
    wr = ("mirror_tbl",) if D > 1 else ("drop_zero_keys",)
    run_update(S, frames, q_slot, plain, inst, direct=True, name="%s plain direct" % inst, wrongs=wr)
    if D == 3:
        frames[2] = None
    run_update(S, frames, q_slot, dil, inst, direct=False, name="%s dilated in place" % inst)
    # the boundary of the automatic choice: n_win = SMs / 2 -> CL 2, one window more -> CL 1 (in place, sliced map)
    Sb = AttnSetup(256, D, 3 * H * W, seed=301 + NT, tbl_scale=0.02)
    n = sms // 2 + (1 if CL == 1 else 0)
    run_update(Sb, list(Sb.frames), q_slot, tmap(3, H, W, False)[:n].contiguous(), inst, direct=False,
               name="%s n_win %d (SMs %d)" % (inst, n, sms))
    # forced: this instance on the other side of the boundary, and the other one on this side
    other = 3 - CL
    Bf = 1 if CL == 1 else 3
    tm_f = tmap(Bf, H, W, False)
    Sf = AttnSetup(256, D, Bf * H * W, seed=302 + NT, tbl_scale=1.0)
    outs = {}
    for cl in (CL, other):
        monkeypatch.setenv("BDE2VID_ATTN_TC256_CLUSTER", str(cl))
        outs[cl] = run_update(Sf, list(Sf.frames), q_slot, tm_f, "attn_win256_tc_kernel<%d, %d>" % (NT, cl), direct=False,
                              name="%s forced CL %d" % (inst, cl))
    xs = Sf.frames[q_slot].clone()
    fr = list(Sf.frames)
    fr[q_slot] = xs
    monkeypatch.setenv("BDE2VID_ATTN_TC256_CLUSTER", str(CL))
    Sf.launch(fr, q_slot, tm_f, xs=xs)
    torch.cuda.synchronize()
    assert torch.equal(xs, outs[CL]), "repeat launch differs"


@gpu
@pytest.mark.parametrize("inst", WIN256)
def test_attn256_mma(inst, monkeypatch):
    """attn_win256_kernel<NT, false> (BDE2VID_ATTN_TC256=0), 33 x 44 plain (direct) and dilated (in place)."""
    monkeypatch.setenv("BDE2VID_ATTN_TC256", "0")
    NT = nt_of(inst)
    D = NT_D[NT]
    q_slot = D - 1
    H, W = 33, 44
    S = AttnSetup(256, D, 2 * H * W, seed=400 + NT, tbl_scale=1.0)
    frames = list(S.frames)
    wr = ("mirror_tbl", "neighbour_shortcut") if D > 1 else ("drop_zero_keys",)
    run_update(S, frames, q_slot, tmap(2, H, W, False), inst, direct=True, name="%s plain direct" % inst, wrongs=wr)
    if D > 1:
        frames[0] = None
    run_update(S, frames, q_slot, tmap(2, H, W, True), inst, direct=False, name="%s dilated in place" % inst)


@gpu
@pytest.mark.parametrize("inst", KVPRE)
def test_attn256_kvpre(inst):
    """attn_win256_kernel<NT, true>: precomputed neighbour k | v rows (bf16) at pitch 2C and at the wider pitch of the
    engine's kv_past slice (block 1 of 3), one None neighbour, q_slot in {0, 1, D - 1}, in place and direct."""
    from bde2vid_b200 import ops
    NT = nt_of(inst)
    D = NT_D[NT]
    C = 256
    H, W = 33, 44
    P = 2 * H * W
    S = AttnSetup(C, D, P, seed=500 + NT, tbl_scale=1.0)
    W64 = S.wqkv[C:].to(F64)
    kvs = []
    for d in range(D):      # k | v of every frame as the engine precomputes them: LayerNorm + rows [C, 3C), bf16
        kv = (ln_ref(S.frames[d].to(F64))[0].to(BF).to(F64) @ W64.t() + S.bqkv[C:].to(F64)).to(BF)
        wide = torch.zeros(P, 6 * C, dtype=BF, device=DEV)
        wide[:, 2 * C:4 * C] = kv
        kvs.append((kv.contiguous(), wide[:, 2 * C:4 * C]))
    for i, q_slot in enumerate(sorted({0, 1, D - 1})):
        for dil in (False, True):
            tm = tmap(2, H, W, dil)
            kv = [None if d == q_slot else kvs[d][(i + int(dil)) % 2] for d in range(D)]
            zero = [d for d in range(D) if d != q_slot][int(dil) % (D - 1)]
            if dil:
                kv[zero] = None
            direct = not dil
            q = S.frames[q_slot]
            q0 = q.clone()
            xs = torch.full_like(q, float("nan")) if direct else q.clone()
            xq = q if direct else xs
            run_routed(lambda: ops.window_attention_fused_kvpre(xq, kv, q_slot, tm.view(-1), tm.shape[0], C, 16, S.wqkv,
                                                                S.bqkv, S.tbl, S.wproj, S.bproj, xs), inst)
            assert torch.equal(q, q0)
            kv64 = [None if t is None else t.to(F64) for t in kv]
            frames64 = [q0 if d == q_slot else None for d in range(D)]
            _, _, y, e_y = S.ref(frames64, q_slot, tm, kvpre=kv64)
            before = torch.full_like(q0, float("nan")).to(F64) if direct else q0.to(F64)
            ref, gate = scatter_update(before, q0.to(F64), tm.long(), y, e_y)
            name = "%s q%d dil%d pitch %d" % (inst, q_slot, dil, kv[(q_slot + 1) % D].stride(0) if kv[(q_slot + 1) % D] is not None else 0)
            if dil:
                # the bias table of the mirrored frame slot
                _, _, yw, _ = S.ref(frames64, q_slot, tm, kvpre=kv64, wrong="mirror_tbl")
                wref, _ = scatter_update(before, q0.to(F64), tm.long(), yw, e_y)
                assert gate_ratio(xs, wref, gate) > 1.0, name
            check(name, xs, ref, gate)


@gpu
@pytest.mark.parametrize("inst", HG256)
def test_attn256_head_groups(inst):
    """attn_fused_kernel<256, 16, NT, false>: the per-head-group form that writes the bf16 attention output o_out
    (the projection then runs as a GEMM), gated on the bf16 o store.  The token map has 35 plain windows of the 33 x 44
    map plus three windows that are entirely padding."""
    NT = nt_of(inst)
    D = NT_D[NT]
    H, W = 33, 44
    S = AttnSetup(256, D, H * W, seed=600 + NT, tbl_scale=1.0)
    tm = torch.cat([tmap(1, H, W, False), torch.full((3, 49), -1, dtype=torch.int32, device=DEV)]).contiguous()
    for q_slot in sorted({0, D - 1}):
        frames = list(S.frames)
        if D > 1:
            frames[(q_slot + 1) % D] = None
        ob = torch.full((tm.shape[0] * 49, 256), float("nan"), dtype=BF, device=DEV)
        run_routed(lambda: S.launch(frames, q_slot, tm, o_out=ob), inst)
        o, d_o, _, _ = S.ref(frames, q_slot, tm, proj=False)
        gate = d_o + TINY
        name = "%s o_out q%d" % (inst, q_slot)
        rw = gate_ratio(ob, S.ref(frames, q_slot, tm, proj=False, ln_eps=1e-6)[0], gate)
        assert rw > 1.0, "%s: LayerNorm eps 1e-6 passes too (%.3f)" % (name, rw)
        if D > 1:
            rw = gate_ratio(ob, S.ref(frames, q_slot, tm, proj=False, wrong="mirror_tbl")[0], gate)
            assert rw > 1.0, "%s: the mirrored slot's bias table passes too (%.3f)" % (name, rw)
        check(name, ob, o, gate)


@gpu
def test_attn_refused_calls():
    """A None query frame with the projection, and an unsupported (c, heads, D), are refused."""
    from bde2vid_b200 import ops
    S = AttnSetup(64, 3, 14 * 14, seed=1, tbl_scale=0.02)
    tm = tmap(1, 14, 14, False)
    xs = S.frames[1].clone()
    with pytest.raises(RuntimeError):
        S.launch([S.frames[0], None, S.frames[2]], 1, tm, xs=xs)
    with pytest.raises(RuntimeError):
        ops.window_attention_fused(S.frames, 1, tm.view(-1), tm.shape[0], 128, 16, S.wqkv, S.bqkv, S.tbl, S.wproj, S.bproj,
                                   xs=xs)
    with pytest.raises(RuntimeError):
        ops.window_attention_fused(S.frames + [S.frames[0]], 1, tm.view(-1), tm.shape[0], 64, 16, S.wqkv, S.bqkv, S.tbl,
                                   S.wproj, S.bproj, xs=xs)
    assert torch.equal(xs, S.frames[1])


# ---------------------------------------------------------------------------------------------------------------------
# fused MLPs
# ---------------------------------------------------------------------------------------------------------------------
class MlpSetup:
    def __init__(self, C, seed):
        g = torch.Generator().manual_seed(seed)
        Hd = 4 * C
        self.C, self.Hd = C, Hd
        self.w1 = (2.5 * torch.randn(Hd, C, generator=g, dtype=F64) / C ** 0.5).to(BF).to(DEV)
        self.b1 = (0.1 * torch.randn(Hd, generator=g)).to(DEV)
        self.w2 = (torch.randn(C, Hd, generator=g, dtype=F64) / Hd ** 0.5).to(BF).to(DEV)
        self.b2 = (0.1 * torch.randn(C, generator=g)).to(DEV)
        self.g = g

    def rows(self, n):
        return token_rows(n, self.C, self.g).to(DEV)

    def launch(self, x, sum_io=None, sum_t=None):
        from bde2vid_b200 import ops
        ops.mlp_fused(x, x.shape[0], self.C, self.Hd, self.w1, self.b1, self.w2, self.b2, sum_io=sum_io, sum_t=sum_t)

    def ref(self, x, **kw):
        return mlp_ref(x.to(F64), self.w1.to(F64), self.b1.to(F64), self.w2.to(F64), self.b2.to(F64), **kw)


def mlp_forms(M, x0, inst, name, wrong=False):
    """In place, sum_io only and sum_io + sum_t on copies of x0: the same x, each within the gate."""
    ref, gate, h = M.ref(x0)
    outs = []
    for form in ("in place", "sum_io", "sum_io + sum_t"):
        x = x0.clone()
        s0 = torch.randn(x0.shape, generator=M.g).to(DEV) * 3 if form != "in place" else None
        sm = None if s0 is None else s0.clone()
        st = torch.full(x0.shape, float("nan"), dtype=BF, device=DEV) if form == "sum_io + sum_t" else None
        run_routed(lambda: M.launch(x, sm, st), inst)
        if form == "in place":
            if wrong:
                rw = gate_ratio(x, M.ref(x0, ln_eps=1e-6)[0], gate)
                assert rw > 1.0, "%s: LayerNorm eps 1e-6 passes too (%.3f)" % (name, rw)
            check("%s %s" % (name, form), x, ref, gate)
        else:
            assert torch.equal(x, outs[0]), "%s: %s changes x" % (name, form)
            sref = s0.to(F64) + ref
            check("%s %s: sum_io" % (name, form), sm, sref, gate + U32 * sref.abs() + TINY)
            if st is not None:
                assert torch.equal(st, sm.to(BF))
        outs.append(x)
    return outs[0], float(h.abs().max())


@gpu
@pytest.mark.parametrize("rows", ["1", "127", "128", "129", "2SM-1", "2SM", "2SM+1"])
def test_mlp64(rows):
    """mlp_fused_kernel (C = 64, hidden 256): ragged and exact 128-row tiles, and tile counts just below, at and above
    2 x SMs (the persistent grid), so that persistent CTAs walk more than one tile; in place, sum_io, sum_io + sum_t."""
    sms = sm_count()
    n = {"2SM-1": (2 * sms - 1) * 128, "2SM": 2 * sms * 128, "2SM+1": (2 * sms + 1) * 128 + 5}.get(rows) or int(rows)
    M = MlpSetup(64, seed=n)
    x0 = M.rows(n)
    _, hmax = mlp_forms(M, x0, MLP64, "%s rows %d" % (MLP64, n), wrong=n >= 128)
    if n >= 1000:
        assert hmax >= 8.0, hmax


@gpu
@pytest.mark.parametrize("inst", MLP256)
def test_mlp256(inst, monkeypatch):
    """mlp_fused256_kernel<CL>: row counts on both sides of the automatic choice (CL 4 while tiles * 4 <= SMs, CL 2
    while tiles * 2 <= SMs, BM = 128 rows), then CL forced on other row counts with the sum forms, repeat launches and
    BDE2VID_PDL=0 bit-identical."""
    CL = int(inst.split("<")[1][0])
    sms = sm_count()
    auto = {4: [1, (sms // 4) * 128], 2: [(sms // 4) * 128 + 1, (sms // 2) * 128], 1: [(sms // 2) * 128 + 1]}[CL]
    M = MlpSetup(256, seed=900 + CL)
    for n in auto:
        x0 = M.rows(n)
        mlp_forms(M, x0, inst, "%s auto rows %d" % (inst, n), wrong=n > 1)
    monkeypatch.setenv("BDE2VID_MLP256_CLUSTER", str(CL))
    n = {4: (sms // 2) * 128 + 77, 2: 300, 1: 4 * 128 + 3}[CL]
    x0 = M.rows(n)
    x, hmax = mlp_forms(M, x0, inst, "%s forced rows %d" % (inst, n))
    assert hmax >= 8.0, hmax
    xr = x0.clone()
    M.launch(xr)
    monkeypatch.setenv("BDE2VID_PDL", "0")
    xp = x0.clone()
    M.launch(xp)
    torch.cuda.synchronize()
    assert torch.equal(xr, x) and torch.equal(xp, x)


# ---------------------------------------------------------------------------------------------------------------------
# CPU tests
# ---------------------------------------------------------------------------------------------------------------------
def _block_sd(C, heads, D, g):
    from bde2vid_b200.synth import relative_position_index
    p = "blk."
    sd = {p + "attn.relative_position_bias_table": 0.5 * torch.randn((2 * D - 1) * 169, heads, generator=g, dtype=F64),
          p + "attn.relative_position_index": relative_position_index(D, 7, 7)}
    for ln in ("attn.norm_q", "attn.norm_kv", "norm2"):
        sd[p + ln + ".weight"] = 1 + 0.2 * torch.randn(C, generator=g, dtype=F64)
        sd[p + ln + ".bias"] = 0.2 * torch.randn(C, generator=g, dtype=F64)
    for name, (o, i) in {"attn.q": (C, C), "attn.kv": (2 * C, C), "attn.proj": (C, C), "mlp.fc1": (4 * C, C),
                         "mlp.fc2": (C, 4 * C)}.items():
        sd[p + name + ".weight"] = torch.randn(o, i, generator=g, dtype=F64) / i ** 0.5
        sd[p + name + ".bias"] = 0.1 * torch.randn(o, generator=g, dtype=F64)
    return sd


def compact_table(sd, D, q_ind, heads):
    """[heads, D, 169] table rebuilt from relative_position_index (every analytic offset must read one entry)."""
    table = sd["blk.attn.relative_position_bias_table"]
    index = sd["blk.attn.relative_position_index"]
    rel = rel_index().reshape(-1)
    tbl = torch.full((heads, D, 169), float("nan"), dtype=F64)
    for d in range(D):
        idx = index[q_ind * 49:(q_ind + 1) * 49, d * 49:(d + 1) * 49].reshape(-1)
        tbl[:, d, rel] = table[idx].t()
        assert torch.equal(tbl[:, d, rel], table[idx].t()), "one relative offset reads two table entries"
    assert not torch.isnan(tbl).any()
    return tbl


@pytest.mark.parametrize("D,q_ind,dilated", [(2, 0, False), (2, 1, True), (3, 1, False), (3, 0, True), (3, 2, False)])
def test_reference_vs_oracle(D, q_ind, dilated):
    """The attention-half and MLP references without roundings (exact GELU), on the engine's folding
    (engine.py:273-287) and compact tables rebuilt from relative_position_index, equal O.attention_block in float64."""
    C, heads, B, H, W = 64, 16, 2, 9, 16
    g = torch.Generator().manual_seed(D * 10 + q_ind + 100 * dilated)
    sd = _block_sd(C, heads, D, g)
    frames = [torch.randn(B, C, H, W, generator=g, dtype=F64) * 1.5 + 0.3 for _ in range(D)]
    oracle = O.attention_block(sd, "blk", frames, q_ind, heads, dilated)
    p = "blk.attn."
    sc = (C // heads) ** -0.5
    Wq, bq, Wkv, bkv = sd[p + "q.weight"], sd[p + "q.bias"], sd[p + "kv.weight"], sd[p + "kv.bias"]
    gq, btq, gk, btk = sd[p + "norm_q.weight"], sd[p + "norm_q.bias"], sd[p + "norm_kv.weight"], sd[p + "norm_kv.bias"]
    wqkv = torch.cat([sc * Wq * gq[None, :], Wkv * gk[None, :]], 0)
    bqkv = torch.cat([sc * (Wq @ btq + bq), Wkv @ btk + bkv], 0)
    tbl = compact_table(sd, D, q_ind, heads)
    # the engine's own construction of the compact table from the bias-table rows of each frame offset
    tab = sd[p + "relative_position_bias_table"]
    eng = torch.stack([tab[((q_ind - d) + D - 1) * 169:((q_ind - d) + D) * 169] for d in range(D)], 0).permute(2, 0, 1)
    assert torch.equal(eng, tbl)
    from bde2vid_b200.engine import window_token_map
    tm = window_token_map(B, H, W, (7, 7), dilated, "cpu")[0].long()
    flat = [f.permute(0, 2, 3, 1).reshape(B * H * W, C) for f in frames]
    _, _, y, _ = attn_ref(flat, q_ind, tm, wqkv, bqkv, tbl, sd[p + "proj.weight"], sd[p + "proj.bias"], heads, exact=True)
    x = flat[q_ind].clone()
    pix = tm.reshape(-1)
    x[pix[pix >= 0]] += y[pix >= 0]
    W1, b1 = sd["blk.mlp.fc1.weight"], sd["blk.mlp.fc1.bias"]
    g2, bt2 = sd["blk.norm2.weight"], sd["blk.norm2.bias"]
    out, _, _ = mlp_ref(x, W1 * g2[None, :], W1 @ bt2 + b1, sd["blk.mlp.fc2.weight"], sd["blk.mlp.fc2.bias"], exact=True)
    got = out.reshape(B, H, W, C).permute(0, 3, 1, 2)
    err = float(((got - oracle).abs() / oracle.abs().clamp(min=1)).max())
    assert err <= 1e-12, err


@pytest.mark.parametrize("dtype", [BF, F16])
def test_flip(dtype):
    """flip is 0 away from ties and one ulp at a tie (and where a rounding boundary lies within +- e).  rnd goes through
    fp32 as the kernels' stores do, so e below fp32 resolution does not separate the neighbours of a tie."""
    one = torch.tensor([1.0], dtype=F64)
    ulp = 2.0 ** -7 if dtype == BF else 2.0 ** -10
    assert float(flip(one, torch.tensor([ulp / 8]), dtype)) == 0.0
    tie = one + ulp / 2
    assert float(flip(tie, torch.tensor([2.0 ** -20]), dtype)) == ulp
    assert float(flip(tie + ulp / 4, torch.tensor([2.0 ** -20]), dtype)) == 0.0
    assert float(flip(tie + ulp / 4, torch.tensor([ulp / 2]), dtype)) == ulp
    x = torch.tensor([3.0 + ulp], dtype=F64)       # in [2, 4) the ulp is 2 ulp(1): 3 + ulp(1) is a tie
    assert float(flip(x, torch.tensor([2.0 ** -20]), dtype)) == 2 * ulp
    s = store(tie, torch.tensor([2.0 ** -20]), dtype)
    assert float(s[1]) == ulp + 2.0 ** -20 and float(s[0]) in (1.0, 1.0 + ulp)


# kernel names as torch.profiler reported them on a B200
_PROFILED_NAMES = {
    "void bde::(anonymous namespace)::attn_fused_kernel<64, 4, 13, true>(bde::(anonymous namespace)::FusedAttnParams)":
        "attn_fused_kernel<64, 4, 13, true>",
    "void bde::(anonymous namespace)::attn_fused_kernel<256, 16, 19, false>(bde::(anonymous namespace)::FusedAttnParams)":
        "attn_fused_kernel<256, 16, 19, false>",
    "void bde::(anonymous namespace)::attn_win256_kernel<13, true>(bde::(anonymous namespace)::FusedAttnParams)":
        "attn_win256_kernel<13, true>",
    "void bde::tc::(anonymous namespace)::attn_win256_tc_kernel<19, 1>(CUtensorMap_st, CUtensorMap_st, "
    "bde::tc::(anonymous namespace)::TcAttnParams)": "attn_win256_tc_kernel<19, 1>",
    "void bde::tc::mlp_fused256_kernel<2>(CUtensorMap_st, CUtensorMap_st, bde::tc::Mlp3Params)": "mlp_fused256_kernel<2>",
    "bde::tc::mlp_fused_kernel(CUtensorMap_st, CUtensorMap_st, bde::tc::MlpParams)": "mlp_fused_kernel",
}


def test_instance_parser():
    """The parser reads the template arguments of the fused kernels in the demangled and the mangled form."""
    dem = {
        "void bde::(anonymous namespace)::attn_fused_kernel<64, 4, 19, true>(bde::(anonymous namespace)::FusedAttnParams)":
            "attn_fused_kernel<64, 4, 19, true>",
        "void bde::tc::attn_win256_tc_kernel<13, 2>(CUtensorMap_st, CUtensorMap_st, bde::tc::TcAttnParams)":
            "attn_win256_tc_kernel<13, 2>",
    }
    man = {   # symbol names of the sm_100a build (cuobjdump -sass)
        "_ZN3bde46_GLOBAL__N__b80b0db7_13_attn_fused_cu_44e2f06b17attn_fused_kernelILi256ELi16ELi7ELb0EEEvNS0_15FusedAttnParamsE":
            "attn_fused_kernel<256, 16, 7, false>",
        "_ZN3bde46_GLOBAL__N__b80b0db7_13_attn_fused_cu_44e2f06b18attn_win256_kernelILi19ELb1EEEvNS0_15FusedAttnParamsE":
            "attn_win256_kernel<19, true>",
        "_ZN3bde2tc46_GLOBAL__N__1f88433e_13_attn_tc256_cu_87ba617621attn_win256_tc_kernelILi7ELi2EEEv14CUtensorMap_stS3_NS1_12TcAttnParamsE":
            "attn_win256_tc_kernel<7, 2>",
        "_ZN3bde2tc19mlp_fused256_kernelILi4EEEv14CUtensorMap_stS2_NS0_10Mlp3ParamsE": "mlp_fused256_kernel<4>",
        "_ZN3bde2tc16mlp_fused_kernelE14CUtensorMap_stS1_NS0_9MlpParamsE": "mlp_fused_kernel",
    }
    for n, want in list(dem.items()) + list(man.items()) + list(_PROFILED_NAMES.items()):
        assert instances([n]) == {want}, (n, instances([n]))
    assert instances(["void bde::tc::gemm_tc_kernel<1>(bde::tc::TcParams)"]) == set()


def test_instance_ids_cover_the_build():
    """The test ids of this file name every fused instance the build contains."""
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    listed = set()
    for f in ("attn_fused", "attn_tc256", "mlp_fused"):
        with open(os.path.join(root, "profiles", "sass", f + ".kernels.txt")) as fh:
            for line in fh:
                if not line.startswith("#") and line.strip():
                    listed |= instances([line.split("  ")[0]])
    ours = set(ATTN64 + ATTN64_PERS + TC256 + WIN256 + KVPRE + HG256 + [MLP64] + MLP256)
    assert len(listed) == 24 and listed == ours, (sorted(listed ^ ours))
