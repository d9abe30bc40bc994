"""GPU parity: element-wise / gather / attention kernels vs functional torch on the CPU."""
import pytest
import torch
import torch.nn.functional as F

from oracle import oracle_torch as O

pytestmark = pytest.mark.gpu
DEV = "cuda"
DTYPES = [torch.float32, torch.bfloat16]


def nhwc(x, dtype=torch.float32):
    return x.permute(0, 2, 3, 1).contiguous().to(DEV, dtype)


def nchw(x):
    return x.float().cpu().permute(0, 3, 1, 2)


@pytest.mark.parametrize("dtype", DTYPES)
def test_upsample2x_sum(dtype):
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(0)
    n, c, h, w = 2, 64, 9, 13
    skip = torch.randn(n, c, h, w, generator=g)
    x = torch.randn(n, c, h, w, generator=g)
    xr = x.to(dtype).float()
    ref = F.interpolate(skip + xr, scale_factor=2, mode="bilinear", align_corners=False)
    dst = torch.zeros(n, 2 * h, 2 * w, c, dtype=dtype, device=DEV)
    ops.upsample2x_sum(nhwc(skip), nhwc(x, dtype), 1.0, n, h, w, c, dst)
    torch.cuda.synchronize()
    tol = 1e-5 if dtype == torch.float32 else 4e-2
    assert (nchw(dst) - ref).abs().max() <= tol
    # quirk Q2: skip = None, x_scale = 2 (fp32 source)
    ref2 = F.interpolate(2 * skip, scale_factor=2, mode="bilinear", align_corners=False)
    ops.upsample2x_sum(None, nhwc(skip), 2.0, n, h, w, c, dst)
    torch.cuda.synchronize()
    assert (nchw(dst) - ref2).abs().max() <= tol


@pytest.mark.parametrize("dtype", DTYPES)
def test_pred_sigmoid_and_add(dtype):
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(1)
    P, c = 1000, 32
    x = torch.randn(P, c, generator=g).to(dtype)
    hd = torch.randn(P, c, generator=g).to(dtype)
    wt = torch.randn(c, generator=g) * 0.3
    b = torch.randn(1, generator=g)
    img = torch.zeros(P, device=DEV)
    ops.pred_sigmoid(x.to(DEV), hd.to(DEV), wt.to(DEV), b.to(DEV), c, P, img)
    ref = torch.sigmoid((x.float() + hd.float()) @ wt + b)
    torch.cuda.synchronize()
    assert (img.cpu() - ref).abs().max() <= 2e-6
    a32 = torch.randn(P, c, generator=g)
    of = torch.zeros(P, c, device=DEV)
    ot = torch.zeros(P, c, device=DEV, dtype=dtype)
    ops.add(x.to(DEV), a32.to(DEV), out_f32=of, out_t=None if dtype == torch.float32 else ot, dtype=dtype)
    torch.cuda.synchronize()
    assert (of.cpu() - (x.float() + a32)).abs().max() <= 1e-6
    if dtype != torch.float32:
        assert (ot.float().cpu() - (x.float() + a32)).abs().max() <= 3e-2


@pytest.mark.parametrize("H,W", [(12, 20), (9, 13), (7, 30), (33, 44)])
def test_window_token_map_matches_oracle(H, W):
    """Host logic cross-check (runs on the GPU box because the product module needs the device for the map)."""
    from bde2vid_b200.engine import window_token_map
    for dil in (False, True):
        mine, g = window_token_map(2, H, W, (7, 7), dil, "cpu")
        idx, ok, g2 = O.window_token_map(H, W, dil)
        nwin = idx.shape[0]
        assert mine.shape == (2 * nwin, 49)
        assert torch.equal(mine[:nwin].long(), idx)
        second = torch.where(idx >= 0, idx + H * W, idx)
        assert torch.equal(mine[nwin:].long(), second)


@pytest.mark.parametrize("dtype", DTYPES)
def test_ln_gather_and_layernorm(dtype):
    from bde2vid_b200 import ops
    from bde2vid_b200.engine import window_token_map
    g = torch.Generator().manual_seed(2)
    B, C, H, W, D = 2, 64, 9, 13, 3
    frames = [torch.randn(B * H * W, C, generator=g) for _ in range(D)]
    frames[2] = None
    gamma, beta = torch.randn(C, generator=g), torch.randn(C, generator=g)
    for dil in (False, True):
        tm, geo = window_token_map(B, H, W, (7, 7), dil, DEV)
        nwin = tm.shape[0]
        out = torch.zeros(nwin, D, 49, C, dtype=dtype, device=DEV)
        ops.ln_gather([None if f is None else f.to(DEV) for f in frames], tm, nwin, 49, C, gamma.to(DEV), beta.to(DEV), out)
        torch.cuda.synchronize()
        tmc = tm.cpu().long()
        for d in range(D):
            src = torch.zeros(B * H * W, C) if frames[d] is None else frames[d]
            tok = src[tmc.clamp(min=0).reshape(-1)].reshape(nwin, 49, C) * (tmc >= 0).unsqueeze(-1)
            ref = F.layer_norm(tok, (C,), gamma, beta, 1e-5)
            err = (out[:, d].float().cpu() - ref).abs().max()
            assert err <= (2e-5 if dtype == torch.float32 else 5e-2), (dil, d, float(err))
    x = torch.randn(500, 256, generator=g) * 3 + 1
    g2, b2 = torch.randn(256, generator=g), torch.randn(256, generator=g)
    o = torch.zeros(500, 256, dtype=dtype, device=DEV)
    ops.layernorm(x.to(DEV), 500, 256, g2.to(DEV), b2.to(DEV), o)
    torch.cuda.synchronize()
    assert (o.float().cpu() - F.layer_norm(x, (256,), g2, b2, 1e-5)).abs().max() <= (3e-5 if dtype == torch.float32 else 6e-2)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C,heads,D", [(64, 16, 3), (256, 16, 3), (128, 16, 5), (64, 16, 2)])
def test_window_attention(dtype, C, heads, D):
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(C + D)
    nwin, nq = 5, 49
    nkv = D * 49
    hd = C // heads
    q = (torch.randn(nwin, nq, C, generator=g) * hd ** -0.5).to(dtype)
    kv = torch.randn(nwin, nkv, 2 * C, generator=g).to(dtype)
    bias = torch.randn(heads, nq, nkv, generator=g)
    qh = q.float().view(nwin, nq, heads, hd).permute(0, 2, 1, 3)
    kh = kv.float()[..., :C].reshape(nwin, nkv, heads, hd).permute(0, 2, 1, 3)
    vh = kv.float()[..., C:].reshape(nwin, nkv, heads, hd).permute(0, 2, 1, 3)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) + bias, -1) @ vh).permute(0, 2, 1, 3).reshape(nwin, nq, C)
    out = torch.zeros(nwin, nq, C, dtype=dtype, device=DEV)
    ops.window_attention(q.to(DEV), kv.to(DEV), bias.permute(0, 2, 1).contiguous().to(DEV), nwin, nq, nkv, C, heads, out)
    torch.cuda.synchronize()
    assert (out.float().cpu() - ref).abs().max() <= (2e-5 if dtype == torch.float32 else 2e-2)


@pytest.mark.parametrize("C,heads,D", [(64, 16, 3), (256, 16, 3), (128, 16, 3), (64, 16, 2), (64, 16, 1)])
def test_window_attention_mma(C, heads, D):
    """Tensor-core attention core (bf16 mma.sync) vs fp32 softmax attention on the same bf16 inputs."""
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(C + 7 * D)
    nwin, nq = 37, 49
    nkv = D * 49
    hd = C // heads
    q = (torch.randn(nwin, nq, C, generator=g) * hd ** -0.5).to(torch.bfloat16)
    kv = torch.randn(nwin, nkv, 2 * C, generator=g).to(torch.bfloat16)
    bias = torch.randn(heads, nq, nkv, generator=g)
    qh = q.float().view(nwin, nq, heads, hd).permute(0, 2, 1, 3)
    kh = kv.float()[..., :C].reshape(nwin, nkv, heads, hd).permute(0, 2, 1, 3)
    vh = kv.float()[..., C:].reshape(nwin, nkv, heads, hd).permute(0, 2, 1, 3)
    ref = (torch.softmax(qh @ kh.transpose(-1, -2) + bias, -1) @ vh).permute(0, 2, 1, 3).reshape(nwin, nq, C)
    out = torch.full((nwin, nq, C), 7.0, dtype=torch.bfloat16, device=DEV)
    bp = ops.pad_bias_for_mma(bias.to(DEV), nkv)
    assert bp is not None and bp.shape[1] == 64
    ops.window_attention_mma(q.to(DEV), kv.to(DEV), bp, nwin, nq, nkv, C, heads, out)
    torch.cuda.synchronize()
    err = (out.float().cpu() - ref).abs().max()
    print("attention mma", C, heads, D, float(err))
    assert err <= 3e-2


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("C", [64, 128, 256])
def test_ln_gather_qkv(dtype, C):
    from bde2vid_b200 import ops
    from bde2vid_b200.engine import window_token_map
    g = torch.Generator().manual_seed(C)
    B, H, W, D, qs = 2, 9, 13, 3, 1
    frames = [torch.randn(B * H * W, C, generator=g) for _ in range(D)]
    frames[0] = None
    gk, bk, gq, bq = (torch.randn(C, generator=g) for _ in range(4))
    for dil in (False, True):
        tm, _ = window_token_map(B, H, W, (7, 7), dil, DEV)
        nwin = tm.shape[0]
        okv = torch.zeros(nwin, D, 49, C, dtype=dtype, device=DEV)
        oq = torch.zeros(nwin, 49, C, dtype=dtype, device=DEV)
        ops.ln_gather_qkv([None if f is None else f.to(DEV) for f in frames], qs, tm, nwin, 49, C, gk.to(DEV), bk.to(DEV),
                          gq.to(DEV), bq.to(DEV), okv, oq)
        torch.cuda.synchronize()
        tmc = tm.cpu().long()
        tol = 2e-5 if dtype == torch.float32 else 5e-2
        for d in range(D):
            src = torch.zeros(B * H * W, C) if frames[d] is None else frames[d]
            tok = src[tmc.clamp(min=0).reshape(-1)].reshape(nwin, 49, C) * (tmc >= 0).unsqueeze(-1)
            assert (okv[:, d].float().cpu() - F.layer_norm(tok, (C,), gk, bk, 1e-5)).abs().max() <= tol
            if d == qs:
                assert (oq.float().cpu() - F.layer_norm(tok, (C,), gq, bq, 1e-5)).abs().max() <= tol


# 1 / 129: ragged tiles; 23232 / 92928: one / four 132 x 176 maps; 37965 = 296 full tiles + a ragged one: every persistent CTA of the
# C = 64 kernel (2 per SM) walks more than one tile
@pytest.mark.parametrize("rows", [1, 128, 129, 1000, 23232, 37965, 92928])
@pytest.mark.parametrize("C", [64, 256])
def test_mlp_fused(rows, C):
    """x += fc2(GELU(fc1(LN(x)))) in one tcgen05 kernel vs fp32 torch on bf16-rounded weights (DTransformer.py:279-304);
    C = 64 / hidden 256 (level 1) and C = 256 / hidden 1024 (level 3, hidden chunked through shared memory)."""
    from bde2vid_b200 import ops
    g = torch.Generator().manual_seed(rows + C)
    Hd = 4 * C
    x = torch.randn(rows, C, generator=g) * 2 + 0.3
    gamma, beta = 1 + 0.2 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)
    W1, b1 = torch.randn(Hd, C, generator=g) / C ** 0.5, torch.randn(Hd, generator=g) * 0.1
    W2, b2 = torch.randn(C, Hd, generator=g) / Hd ** 0.5, torch.randn(C, generator=g) * 0.1
    w1f = (W1 * gamma[None, :]).to(torch.bfloat16)
    b1f = W1 @ beta + b1
    w2f = W2.to(torch.bfloat16)
    xn = F.layer_norm(x, (C,), eps=1e-5).to(torch.bfloat16).float()
    hid = F.gelu(xn @ w1f.float().t() + b1f).to(torch.bfloat16).float()
    ref = x + hid @ w2f.float().t() + b2
    xd = x.to(DEV).contiguous()
    ops.mlp_fused(xd, rows, C, Hd, w1f.to(DEV).contiguous(), b1f.to(DEV), w2f.to(DEV).contiguous(), b2.to(DEV))
    torch.cuda.synchronize()
    err = float((xd.cpu() - ref).abs().max())
    print("mlp_fused", rows, C, err)
    assert err <= 2e-2     # bf16 rounding of the hidden activations at values of order 1..8
    full = x + F.gelu(F.layer_norm(x, (C,), gamma, beta, 1e-5) @ W1.t() + b1) @ W2.t() + b2
    assert float((xd.cpu() - full).abs().max()) <= 6e-2
    # fused "x + merged" (..._V5.py:166-169): sum_io += x_new, sum_t = bf16(sum_io); x itself as without the option
    merged = torch.randn(rows, C, generator=g)
    x2, sm = x.to(DEV).contiguous(), merged.to(DEV).contiguous()
    st = torch.zeros(rows, C, dtype=torch.bfloat16, device=DEV)
    ops.mlp_fused(x2, rows, C, Hd, w1f.to(DEV).contiguous(), b1f.to(DEV), w2f.to(DEV).contiguous(), b2.to(DEV), sum_io=sm, sum_t=st)
    torch.cuda.synchronize()
    assert torch.equal(x2, xd)
    assert float((sm.cpu() - (xd.cpu() + merged)).abs().max()) <= 1e-5
    assert torch.equal(st, sm.to(torch.bfloat16))
    if C == 256:
        # hidden dimension split over a thread-block cluster (BDE2VID_MLP256_CLUSTER = 1 / 2 / 4): the partial fc2 accumulators
        # are summed into x in CL phases separated by cluster barriers, in a fixed order -> deterministic; the split only
        # changes the fp32 summation order of the K = 1024 product
        import os
        outs = {}
        for cl in ("1", "2", "4"):
            os.environ["BDE2VID_MLP256_CLUSTER"] = cl
            for rep in range(2):
                xc = x.to(DEV).contiguous()
                ops.mlp_fused(xc, rows, C, Hd, w1f.to(DEV).contiguous(), b1f.to(DEV), w2f.to(DEV).contiguous(), b2.to(DEV))
                torch.cuda.synchronize()
                if rep == 0:
                    outs[cl] = xc
                else:
                    assert torch.equal(outs[cl], xc), "cluster %s not deterministic" % cl
            assert float((outs[cl].cpu() - ref).abs().max()) <= 2e-2
            assert float((outs[cl] - outs["1"]).abs().max()) <= 1e-4
        del os.environ["BDE2VID_MLP256_CLUSTER"]


@pytest.mark.parametrize("shape", [(3, 5, 40, 56), (2, 5, 33, 47), (1, 3, 16, 32), (2, 6, 19, 70)])
def test_head_conv(shape):
    """5x5 head convolution straight from planar fp32 voxels (mma.sync, bf16 operands) vs torch conv2d on the same
    bf16-rounded operands (...V5.py:116; ConvLayer submodules.py:85-114)."""
    from bde2vid_b200 import ops
    n, cin, h, w = shape
    g = torch.Generator().manual_seed(sum(shape))
    vox = torch.randn(n, cin, h, w, generator=g) * (torch.rand(n, cin, h, w, generator=g) < 0.4)   # sparse, signed, like voxels
    wt = torch.randn(32, cin, 5, 5, generator=g) / (25 * cin) ** 0.5
    b = torch.randn(32, generator=g) * 0.1
    ref = F.relu(F.conv2d(vox.to(torch.bfloat16).float(), wt.to(torch.bfloat16).float(), b, padding=2))
    out = torch.zeros(n, h, w, 32, dtype=torch.bfloat16, device=DEV)
    ops.head_conv(vox.to(DEV).contiguous(), wt.to(DEV).contiguous(), b.to(DEV), out, act=ops.ACT_RELU)
    torch.cuda.synchronize()
    got = out.float().cpu().permute(0, 3, 1, 2)
    err = float((got - ref).abs().max())
    print("head_conv", shape, err, float(ref.abs().max()))
    assert err <= 1e-2 * max(1.0, float(ref.abs().max()))


@pytest.mark.parametrize("H,W,Hp,Wp", [(260, 346, 264, 352), (180, 240, 184, 240), (33, 47, 40, 48)])
def test_frame_metrics_vs_oracle(H, W, Hp, Wp):
    """Device MSE / SSIM of the centre crop vs the oracle restatement (evaluate/metrics.py:42-65)."""
    from bde2vid_b200 import ops
    from oracle import oracle_torch as O
    g = torch.Generator().manual_seed(H + W)
    n = 3
    pred = torch.rand(n, Hp, Wp, generator=g)
    y0, x0 = Hp // 2 - H // 2, Wp // 2 - W // 2
    gt = (pred[:, y0:y0 + H, x0:x0 + W] + 0.1 * torch.randn(n, H, W, generator=g)).clamp(0, 1).contiguous()
    out = ops.frame_metrics(pred.to(DEV), gt.to(DEV), y0, x0, 1.0).cpu()
    for i in range(n):
        crop = pred[i, y0:y0 + H, x0:x0 + W]
        assert abs(float(out[i, 0]) - O.mse(crop, gt[i])) <= 1e-7
        assert abs(float(out[i, 1]) - O.ssim_uniform7(crop, gt[i])) <= 1e-6


@pytest.mark.parametrize("dilated,zero_frame", [(False, None), (True, 2), (False, 0)])
def test_window_attention_whole_window_kernel_c256(dilated, zero_frame):
    """C = 256: the whole-window kernel (tcgen05 projections, projection + scatter fused; one CTA or one 2-CTA cluster
    per window) against an fp32 torch restatement of DTransformer.py:183-207, 294-299 (NOT another CUDA kernel).  70 windows, plain
    and dilated token maps, a missing neighbour frame.  The per-head-group kernel is checked against the same reference."""
    from bde2vid_b200 import ops
    from bde2vid_b200.engine import window_token_map
    g = torch.Generator().manual_seed(5 + int(dilated))
    B, h, w, C, heads, D, q_ind = 2, 35, 49, 256, 16, 3, 1
    P = B * h * w
    tm, _ = window_token_map(B, h, w, (7, 7), dilated, DEV)
    nwin = tm.shape[0]
    assert nwin >= 64
    frames = [(torch.randn(P, C, generator=g) * 1.5 + 0.2).to(DEV) for _ in range(D)]
    if zero_frame is not None:
        frames[zero_frame] = None
    wq_f = torch.randn(3 * C, C, generator=g) / C ** 0.5
    wq_f[:C] *= (C // heads) ** -0.5            # the engine folds the q scale head_dim^-0.5 into the q rows (engine.py)
    wqkv = wq_f.to(torch.bfloat16).to(DEV)
    bqkv = (torch.randn(3 * C, generator=g) * 0.1).to(DEV)
    table = torch.randn((2 * D - 1) * 169, heads, generator=g) * 0.5
    rows = [table[((q_ind - d) + D - 1) * 169:((q_ind - d) + D) * 169] for d in range(D)]
    tbl = torch.stack(rows, 0).permute(2, 0, 1).contiguous().to(DEV)          # [heads, D, 169]
    wproj = (torch.randn(C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(DEV)
    bproj = (torch.randn(C, generator=g) * 0.1).to(DEV)
    xs0 = frames[q_ind].clone()
    # reference: plain fp32 torch following DTransformer.py:183-207 (norm_q / norm_kv + q / kv Linear, scaled q k^T +
    # relative-position bias, softmax, attn v, proj) and :294-299 (window_reverse, crop, shortcut).  The LayerNorm affine
    # and the q scale are already folded into wqkv / bqkv by the caller (engine.py), so LN here has no affine.
    idx = tm.view(nwin, 49).long()
    keep = idx >= 0
    hd = C // heads

    def win_tokens(fr):                       # [nwin, 49, C]; zero-padding tokens are all-zero BEFORE the LayerNorm
        if fr is None:
            return torch.zeros(nwin, 49, C, device=DEV)
        return fr[idx.clamp(min=0)] * keep.unsqueeze(-1)

    fr_list = [xs0 if d == q_ind else frames[d] for d in range(D)]
    xhat = torch.cat([F.layer_norm(win_tokens(f), (C,), eps=1e-5) for f in fr_list], 1)       # [nwin, D*49, C]
    qkv_ref = xhat @ wqkv.float().t() + bqkv                                                   # rows q | k | v
    q = qkv_ref[:, q_ind * 49:(q_ind + 1) * 49, :C].reshape(nwin, 49, heads, hd).permute(0, 2, 1, 3)
    k = qkv_ref[:, :, C:2 * C].reshape(nwin, D * 49, heads, hd).permute(0, 2, 1, 3)
    v = qkv_ref[:, :, 2 * C:].reshape(nwin, D * 49, heads, hd).permute(0, 2, 1, 3)
    a_ = torch.arange(7, device=DEV)
    ai, bi = a_.repeat_interleave(7), a_.repeat(7)                                            # token -> (row, col)
    rel = (ai[:, None] - ai[None, :] + 6) * 13 + (bi[:, None] - bi[None, :] + 6)              # [49 q, 49 k]
    bias = torch.cat([tbl[:, d][:, rel] for d in range(D)], 2)                                # [heads, 49, D*49]
    attn = torch.softmax(q @ k.transpose(-2, -1) + bias.unsqueeze(0), dim=-1)
    o = (attn @ v).permute(0, 2, 1, 3).reshape(nwin * 49, C)
    proj = o @ wproj.float().t() + bproj
    ref = xs0.clone()
    flat, kflat = idx.reshape(-1), keep.reshape(-1)
    ref[flat[kflat]] += proj[kflat]
    fr = list(frames)
    upd = float((ref - xs0).abs().max())
    assert upd > 0.1                                  # the attention path really contributes
    # whole-window kernel, in place on a copy of the query frame: one CTA per window, and one window per 2-CTA cluster (the
    # head groups split, partial projections summed into x in two phases -- the default while 2 * nwin CTAs fit one wave)
    import os
    got = {}
    for cl in ("1", "2"):
        os.environ["BDE2VID_ATTN_TC256_CLUSTER"] = cl
        try:
            for rep in range(2):
                xs = xs0.clone()
                fr[q_ind] = xs
                ops.window_attention_fused(fr, q_ind, tm.view(-1), nwin, C, heads, wqkv, bqkv, tbl, wproj, bproj, xs=xs)
                torch.cuda.synchronize()
                if rep == 0:
                    got[cl] = xs
                else:
                    assert torch.equal(xs, got[cl]), "cluster %s: not deterministic" % cl
        finally:
            del os.environ["BDE2VID_ATTN_TC256_CLUSTER"]
        err = float((got[cl] - ref).abs().max())
        print("win256 cluster", cl, dilated, zero_frame, err, upd)
        # pure fp32 reference, bf16 operands in the kernel (xhat, q, k, o rounded to bf16, p / v to fp16, two chained K = 256
        # products): gate relative to the size of the update the attention half makes
        assert err <= 1.5e-2 * max(1.0, upd), (cl, err, upd)
    assert float((got["1"] - got["2"]).abs().max()) <= 1e-4 * max(1.0, upd)   # only the fp32 order of the projection sum differs
    # the per-head-group kernel (o only) against the same fp32 reference
    ob = torch.zeros(nwin * 49, C, dtype=torch.bfloat16, device=DEV)
    fr[q_ind] = xs0
    ops.window_attention_fused(fr, q_ind, tm.view(-1), nwin, C, heads, wqkv, bqkv, tbl, o_out=ob)
    torch.cuda.synchronize()
    assert float((ob.float() - o).abs().max()) <= 1.5e-2 * max(1.0, float(o.abs().max()))


@pytest.mark.parametrize("dilated,zero_frame,D,q_ind", [(False, None, 3, 1), (True, 2, 3, 1), (False, 0, 3, 1), (True, None, 2, 0),
                                                        (False, None, 1, 0)])
def test_window_attention_fused_c64_vs_fp32_torch(dilated, zero_frame, D, q_ind):
    """C = 64, 16 heads of 4 channels (level 1): attn_fused_kernel<64, 4, NT> -- gather + LayerNorm + q/k/v + softmax(q k^T +
    bias) v + projection + scatter in ONE launch -- against an fp32 torch restatement of DTransformer.py:183-207, 294-299.
    A repeat launch must agree bit for bit."""
    from bde2vid_b200 import ops
    from bde2vid_b200.engine import window_token_map
    g = torch.Generator().manual_seed(11 + int(dilated) + D)
    B, h, w, C, heads = 3, 33, 45, 64, 16
    P = B * h * w
    tm, _ = window_token_map(B, h, w, (7, 7), dilated, DEV)
    nwin = tm.shape[0]
    assert nwin > 100
    frames = [(torch.randn(P, C, generator=g) * 1.5 + 0.2).to(DEV) for _ in range(D)]
    if zero_frame is not None:
        frames[zero_frame] = None
    hd = C // heads
    wq_f = torch.randn(3 * C, C, generator=g) / C ** 0.5
    wq_f[:C] *= hd ** -0.5
    wqkv = wq_f.to(torch.bfloat16).to(DEV)
    bqkv = (torch.randn(3 * C, generator=g) * 0.1).to(DEV)
    tbl = (torch.randn(heads, D, 169, generator=g) * 0.5).to(DEV)
    wproj = (torch.randn(C, C, generator=g) / C ** 0.5).to(torch.bfloat16).to(DEV)
    bproj = (torch.randn(C, generator=g) * 0.1).to(DEV)
    xs0 = frames[q_ind].clone()
    idx = tm.view(nwin, 49).long()
    keep = idx >= 0

    def win_tokens(fr):
        if fr is None:
            return torch.zeros(nwin, 49, C, device=DEV)
        return fr[idx.clamp(min=0)] * keep.unsqueeze(-1)

    fr_list = [xs0 if d == q_ind else frames[d] for d in range(D)]
    xhat = torch.cat([F.layer_norm(win_tokens(f), (C,), eps=1e-5) for f in fr_list], 1)
    qkv_ref = xhat @ wqkv.float().t() + bqkv
    q = qkv_ref[:, q_ind * 49:(q_ind + 1) * 49, :C].reshape(nwin, 49, heads, hd).permute(0, 2, 1, 3)
    k = qkv_ref[:, :, C:2 * C].reshape(nwin, D * 49, heads, hd).permute(0, 2, 1, 3)
    v = qkv_ref[:, :, 2 * C:].reshape(nwin, D * 49, heads, hd).permute(0, 2, 1, 3)
    a_ = torch.arange(7, device=DEV)
    ai, bi = a_.repeat_interleave(7), a_.repeat(7)
    rel = (ai[:, None] - ai[None, :] + 6) * 13 + (bi[:, None] - bi[None, :] + 6)
    bias = torch.cat([tbl[:, d][:, rel] for d in range(D)], 2)
    attn = torch.softmax(q @ k.transpose(-2, -1) + bias.unsqueeze(0), dim=-1)
    o = (attn @ v).permute(0, 2, 1, 3).reshape(nwin * 49, C)
    proj = o @ wproj.float().t() + bproj
    ref = xs0.clone()
    flat, kflat = idx.reshape(-1), keep.reshape(-1)
    ref[flat[kflat]] += proj[kflat]
    upd = float((ref - xs0).abs().max())
    assert upd > 0.1
    got = None
    for rep in range(2):
        xs = xs0.clone()
        fr = list(frames)
        fr[q_ind] = xs
        ops.window_attention_fused(fr, q_ind, tm.view(-1), nwin, C, heads, wqkv, bqkv, tbl, wproj, bproj, xs=xs)
        torch.cuda.synchronize()
        if rep == 0:
            got = xs
        else:
            assert torch.equal(xs, got), "not deterministic"
    err = float((got - ref).abs().max())
    print("attn64", dilated, zero_frame, D, err, upd)
    assert err <= 1.5e-2 * max(1.0, upd), (err, upd)
