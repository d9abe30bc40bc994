"""Sequence executor for the BDE2VID generator.

Implements the level-by-level bidirectional schedule of
model/BDE2VID/bde2vid_cross_scale_propogation_V5.py:100-241 on top of the C-ABI kernels:

  A  head conv, batched over all T frames                                  (:116)
  B  per level: encoder conv batched over T, then the two ConvLSTM chains  (:122-135), the
     ff + fb merge (:137-147) and the in-place sequential window attention (:151-169, quirks Q1,Q4)
  C  decoders + prediction, batched over chunks of frames                  (:183-197, quirk Q2)

All buffers are allocated once per (T, B, Hp, Wp) "plan"; the whole forward is captured into a
CUDA graph on its second use so that replay costs one launch from the host.
Weights are repacked once per engine (K-major [Cout, kh*kw*Cin], gate-interleaved LSTM rows,
query scale folded into q, relative-position bias pre-gathered).
"""
import functools
import os
import warnings
from collections import OrderedDict

import torch

from . import ops
from .synth import relative_position_index
from .ops import (ACT_GELU, ACT_NONE, ACT_RELU, ACT_RELU6, ENGINE_SIMT, ENGINE_TCGEN05, EPI_GRU_OUT, EPI_GRU_UR,
                  EPI_LSTM, EPI_SCATTER, EPI_STORE)

K_ALIGN = 64      # packed weight rows are zero-padded to a multiple of this (tcgen05 K block)
VOX_CPAD = 8      # voxel channels padded 5 -> 8 so that a pixel is one 16-byte bf16 chunk


def window_geometry(H, W, ws):
    """Symmetric zero padding to window multiples (DTransformer.py:254-266)."""
    wh = H if H <= ws[0] else ws[0]
    ww = W if W <= ws[1] else ws[1]
    pad_h = (wh - H % wh) % wh
    pad_w = (ww - W % ww) % ww
    return dict(wh=wh, ww=ww, pt=pad_h // 2, pl=pad_w // 2, nH=(H + pad_h) // wh, nW=(W + pad_w) // ww)


def window_token_map(B, H, W, ws, dilated, device):
    """int32 [B*nWin, wh*ww]: row of the [B*H*W, C] feature matrix feeding every window token, -1 for
    tokens on zero padding.  Plain windows: token (a,b) of window (i,j) <-> padded pixel
    (wh*i+a, ww*j+b); dilated windows (odd blocks, DTransformer.py:362, window_partition :53-59):
    padded pixel (wh*i+2a, ww*j+2b) of the map padded by one more window bottom/right."""
    g = window_geometry(H, W, ws)
    wh, ww, nH, nW = g["wh"], g["ww"], g["nH"], g["nW"]
    step = 2 if dilated else 1
    i = torch.arange(nH).view(nH, 1, 1, 1)
    j = torch.arange(nW).view(1, nW, 1, 1)
    a = torch.arange(wh).view(1, 1, wh, 1)
    b = torch.arange(ww).view(1, 1, 1, ww)
    r = (wh * i + step * a - g["pt"]).expand(nH, nW, wh, ww)
    c = (ww * j + step * b - g["pl"]).expand(nH, nW, wh, ww)
    ok = (r >= 0) & (r < H) & (c >= 0) & (c < W)
    idx = torch.where(ok, r * W + c, torch.full_like(r, -1)).reshape(1, nH * nW, wh * ww)
    boff = (torch.arange(B) * (H * W)).view(B, 1, 1)
    full = torch.where(idx >= 0, idx + boff, idx.expand(B, -1, -1))
    return full.reshape(B * nH * nW, wh * ww).to(torch.int32).contiguous().to(device), g


def _pack_conv(w, dtype, cin_pad=None, chunk_major=False):
    """[Cout, Cin, kh, kw] -> K-major [Cout, Kpad], zero padded to K_ALIGN.
    k = (ky*kw + kx)*Cin + c by default; with ``chunk_major`` (Cin % 64 == 0, ``k_order=1`` of bde_gemm)
    k = (c // 64)*(kh*kw*64) + (ky*kw + kx)*64 + c % 64."""
    co, ci, kh, kw = w.shape
    w = w.permute(0, 2, 3, 1)
    if cin_pad is not None and cin_pad > ci:
        w = torch.nn.functional.pad(w, (0, cin_pad - ci))
    if chunk_major:
        assert w.shape[-1] % 64 == 0
        w = w.reshape(co, kh * kw, w.shape[-1] // 64, 64).permute(0, 2, 1, 3)
    w = w.reshape(co, -1)
    K = w.shape[1]
    Kp = (K + K_ALIGN - 1) // K_ALIGN * K_ALIGN
    out = torch.zeros(co, Kp, dtype=dtype, device=w.device)
    out[:, :K] = w.to(dtype)
    return out.contiguous(), Kp


def _pack_linear(w, dtype, scale=1.0):
    n, K = w.shape
    Kp = (K + K_ALIGN - 1) // K_ALIGN * K_ALIGN
    out = torch.zeros(n, Kp, dtype=dtype, device=w.device)
    out[:, :K] = (w * scale).to(dtype)
    return out.contiguous(), Kp


def _fold_norm(conv, holder):
    """Effective (weight, bias) of conv2d followed by the eval-mode norm_layer of a ConvLayer / UpsampleConvLayer
    (submodules.py:100-111, 133-145): BatchNorm2d (affine, running statistics) or InstanceNorm2d(track_running_stats=True)
    (running statistics, no affine) are per-channel affine maps  y = (x - mean) / sqrt(var + eps) * g + b."""
    w = conv.weight.detach().float()
    b = conv.bias.detach().float() if conv.bias is not None else torch.zeros(w.shape[0], device=w.device)
    nl = getattr(holder, "norm_layer", None) if holder is not None else None
    if nl is None:
        return w, b
    scale = 1.0 / torch.sqrt(nl.running_var.detach().float() + nl.eps)
    if getattr(nl, "weight", None) is not None:
        scale = scale * nl.weight.detach().float()
    shift = -nl.running_mean.detach().float() * scale
    if getattr(nl, "bias", None) is not None:
        shift = shift + nl.bias.detach().float()
    return w * scale.view(-1, 1, 1, 1), b * scale + shift


def _f32(t):
    return t.detach().to(torch.float32).contiguous()


class _Layer:
    """Packed weights of one conv / linear."""

    def __init__(self, w, w_ld, bias, n, ksize=1, stride=1, pad=0, k_order=0):
        self.w, self.w_ld, self.bias, self.n = w, w_ld, bias, n
        self.ksize, self.stride, self.pad, self.k_order = ksize, stride, pad, k_order


def _run_layer(layer, a0, out, n_img, h, w, c0, *, engine, dtype, **kw):
    """``out`` = ``layer`` applied to the NHWC map ``a0`` [n_img, h, w, c0] by bde_gemm (``kw``: ops.gemm's other options)."""
    return ops.gemm(a0, layer.w, layer.bias, out, n_img=n_img, h_in=h, w_in=w, c0=c0, n=layer.n, ksize=layer.ksize,
                    stride=layer.stride, pad=layer.pad, w_ld=layer.w_ld, k_order=layer.k_order, engine=engine, dtype=dtype,
                    **kw)


def _packed_conv(w, b, stride, dt, tc, chunk_ok, cin_pad=None):
    """Packs conv weights w [Cout, Cin, k, k]: chunk-major K (the L1-friendly im2col order of the tcgen05 convs) where
    ``chunk_ok`` allows it."""
    k = w.shape[-1]
    cm = tc and chunk_ok
    pw, ld = _pack_conv(w, dt, cin_pad, chunk_major=cm)
    return _Layer(pw, ld, b.contiguous(), w.shape[0], k, stride, k // 2, k_order=int(cm))


def _conv_layer(holder, stride, dt, tc, cin_pad=None):
    """``holder``: a ConvLayer-like container (conv2d [+ norm_layer], folded in) or a bare nn.Conv2d."""
    conv = getattr(holder, "conv2d", holder)
    w, b = _fold_norm(conv, holder if conv is not holder else None)
    return _packed_conv(w, b, stride, dt, tc, w.shape[-1] > 1 and w.shape[1] % 64 == 0, cin_pad)


def _merged_conv_layer(hold_f, hold_b, stride, dt, tc):
    """forward + backward encoder convs read the same input (...V5.py:129-130): one GEMM with N doubled;
    output channels [0, C) = forward, [C, 2C) = backward."""
    wf, bf = _fold_norm(hold_f.conv2d, hold_f)
    wb, bb = _fold_norm(hold_b.conv2d, hold_b)
    w = torch.cat([wf, wb], 0)
    return _packed_conv(w, torch.cat([bf, bb], 0), stride, dt, tc, w.shape[-1] > 1 and w.shape[1] % 64 == 0)


def _lstm_layer(conv, dt, tc):
    """ConvLSTM gates conv with rows reordered so that n = 4*c + gate (gate order in, remember, out, cell:
    submodules.py:320)."""
    w = conv.weight.detach().float()
    hid = w.shape[0] // 4
    w = w.view(4, hid, *w.shape[1:]).permute(1, 0, 2, 3, 4).reshape(4 * hid, *w.shape[1:])
    b = conv.bias.detach().float().view(4, hid).t().reshape(-1)
    return _packed_conv(w, b, 1, dt, tc, hid % 64 == 0)


def _gru_layers(blk, dt, tc, grow=None):
    """ConvGRU (submodules.py:337-375) as two convolutions: [update | reset] with rows interleaved n = 2c + g
    (BDE_EPI_GRU_UR) and out_gate (BDE_EPI_GRU_OUT).  ``grow`` maps each gate's (weight, bias) before packing."""
    wb = [(c.weight.detach().float(), c.bias.detach().float()) for c in (blk.update_gate, blk.reset_gate, blk.out_gate)]
    (wu, bu), (wr, br), (wo, bo) = [grow(w, b) for w, b in wb] if grow is not None else wb
    hid = wu.shape[0]
    w = torch.stack([wu, wr], 1).reshape(2 * hid, *wu.shape[1:])
    b = torch.stack([bu, br], 1).reshape(-1)
    return _packed_conv(w, b, 1, dt, tc, hid % 64 == 0), _packed_conv(wo, bo, 1, dt, tc, hid % 64 == 0)


def _lin_layer(lin, dt, scale=1.0):
    w, ld = _pack_linear(lin.weight.detach().float(), dt, scale)
    return _Layer(w, ld, _f32(lin.bias * scale), lin.weight.shape[0])


class Engine:
    def __init__(self, gen, precision):
        from . import _lib
        _lib.require_device()
        if precision not in ("bf16", "fp32", "bf16-simt"):
            raise ValueError("precision must be 'bf16' (tcgen05 tensor cores), 'fp32' (CUDA-core parity mode) or "
                             "'bf16-simt' (debug)")
        self.precision = precision
        self.dtype = torch.float32 if precision == "fp32" else torch.bfloat16
        self.gemm_engine = ENGINE_TCGEN05 if precision == "bf16" else ENGINE_SIMT
        cfg = gen.cfg
        self.cfg = cfg
        self.device = gen.head.conv2d.weight.device
        if self.device.type != "cuda":
            raise RuntimeError("BDE2VID (bde2vid_b200) must be on a CUDA device before forward(); no CPU path exists")
        self.L = cfg["num_encoders"]
        self.bc = cfg["basechannels"]
        self.bins = cfg["num_bins"]
        self.ks = cfg["ks"]
        self.buf = cfg["buffer_index"]
        self.q_ind = cfg["q_idx"]
        self.D = len(self.buf)
        self.heads = cfg["num_heads"]
        self.ws = cfg["window_size"]
        self.depths = cfg["depths"]
        self.rec = cfg.get("recurrent_block_type", "convlstm")        # 'convlstm' | 'convgru' | None (useRC=False)
        self.concat = cfg.get("skip_type", "sum") == "concat"
        self.nwindow_size = cfg.get("nwindow_size")
        self.net_act = cfg.get("net_act", ACT_RELU)
        self.out_act = cfg.get("out_act", ops.ACT_SIGMOID)
        self.fuse_attn = os.environ.get("BDE2VID_FUSED_ATTN", "1") != "0"
        self.fuse_mlp = os.environ.get("BDE2VID_FUSED_MLP", "1") != "0"
        self.fuse_win256 = os.environ.get("BDE2VID_ATTN_WIN256", "1") != "0"
        # the whole-window C = 256 kernel (tcgen05 projections, attn_tc256.cu) is used from this many windows up; the mma.sync
        # form it replaced only paid off from 64 windows (one CTA per window), the tcgen05 form wins at every size measured
        # (35 windows: 31.7 us vs 64.5 us per launch; tools/attn_tc256_probe.py)
        self.win256_min = int(os.environ.get("BDE2VID_WIN256_MIN", "1" if os.environ.get("BDE2VID_ATTN_TC256", "1") != "0" else "64"))
        # precomputed neighbour k | v for the level-3 attention (bde_window_attention_fused_kvpre): OFF by default.
        # Measured on B200 (round 1): the attention kernel stays at 66 us per launch with 60 % fewer MMAs and a 5-deep
        # weight prefetch (it is bound by barrier / shared-memory latency at 16 warps per SM, not by the projections),
        # while the extra LayerNorm + 1x1-conv launches cost ~12 us per frame: 1982 vs 2021 frames/s.
        self.kv_pre = os.environ.get("BDE2VID_ATTN_KVPRE", "0") != "0"
        if self.bins > VOX_CPAD:
            raise NotImplementedError("num_bins > %d" % VOX_CPAD)
        dt = self.dtype
        tc = self.gemm_engine == ENGINE_TCGEN05
        self.gemm = functools.partial(_run_layer, engine=self.gemm_engine, dtype=dt)
        with torch.no_grad():
            self.head = _conv_layer(gen.head, 1, dt, tc, cin_pad=VOX_CPAD)
            # dedicated first-layer kernel (planar fp32 voxels -> NHWC bf16, no packing pass): 32 channels, 5x5
            hw, hb_ = _fold_norm(gen.head.conv2d, gen.head)
            self.head_direct = None
            if (tc and hw.shape[0] == 32 and hw.shape[-1] == 5 and hw.shape[1] <= 6 and self.net_act in (ACT_RELU, ACT_RELU6)
                    and os.environ.get("BDE2VID_HEAD_CONV", "1") != "0"):
                self.head_direct = (hw.contiguous(), hb_.contiguous())
            self.enc = []
            for l in range(self.L):
                fe, be = gen.forward_encoder[l], gen.backward_encoder[l]
                fc, bcv = (fe.conv, be.conv) if self.rec is not None else (fe, be)
                e = dict(f_conv=_conv_layer(fc, 2, dt, tc), b_conv=_conv_layer(bcv, 2, dt, tc))
                if self.rec == "convlstm":
                    e.update(f_lstm=_lstm_layer(fe.recurrent_block.Gates, dt, tc),
                             b_lstm=_lstm_layer(be.recurrent_block.Gates, dt, tc))
                elif self.rec == "convgru":
                    e.update(f_gru=_gru_layers(fe.recurrent_block, dt, tc), b_gru=_gru_layers(be.recurrent_block, dt, tc))
                # the merged form feeds the chains through pitched TMA descriptors: recurrent encoders only
                if tc and self.rec is not None and os.environ.get("BDE2VID_MERGE_ENC", "1") != "0":
                    e["fb_conv"] = _merged_conv_layer(fc, bcv, 2, dt, tc)
                self.enc.append(e)
            self.attn = []
            n_tok = self.ws[0] * self.ws[1]
            for l in range(self.L):
                blocks = []
                if self.depths[l] > 0:
                    C = self.bc * 2 ** (l + 1)
                    hd = C // self.heads
                    # kv tokens per frame: the window's tokens, or nwin0 * nwin1 after the reduction conv (DTransformer.py:172-175)
                    n_kvf = n_tok if self.nwindow_size is None else self.nwindow_size[0] * self.nwindow_size[1]
                    use_mma = (self.nwindow_size is None and dt == torch.bfloat16 and n_tok <= 64 and hd in (4, 8, 16)
                               and self.heads % 2 == 0 and ops.attention_mma_bias_stride(self.D * n_tok) > 0)
                    # fused front end (tcgen05 only): LayerNorm folded into the projections.
                    #   Linear(LN(x)) = (W diag(gamma)) xhat + (W beta + b),  xhat = (x - mean) / sqrt(var + eps)
                    # q and kv share xhat, so ONE GEMM with N = 3C produces [q | k | v] for every kv token.
                    # Blocks without it take the unfused route (see attention_routes).
                    fused = tc and use_mma and C in (64, 128, 256)
                    for blk in gen.feat_attns[l].blocks:
                        a = blk.attn
                        # weights of every route: proj and fc2 always; the rest only where the block's route can use them
                        b = dict(proj=_lin_layer(a.proj, dt), fc2=_lin_layer(blk.mlp.fc2, dt), tbl=None)
                        # (DTransformer.py:195-197: only the first N = D * n_kvf columns of the index are used)
                        idx = a.relative_position_index[self.q_ind * n_tok:(self.q_ind + 1) * n_tok, :self.D * n_kvf]
                        bias = a.relative_position_bias_table.detach().float()[idx.reshape(-1)]
                        bias_hmn = bias.reshape(n_tok, self.D * n_kvf, self.heads).permute(2, 0, 1).contiguous()
                        if use_mma:
                            b["bias_mma"] = ops.pad_bias_for_mma(bias_hmn, self.D * n_tok)
                        if fused:
                            sc = hd ** -0.5
                            Wq, bq = a.q.weight.detach().float(), a.q.bias.detach().float()
                            Wkv, bkv = a.kv.weight.detach().float(), a.kv.bias.detach().float()
                            gq, btq = a.norm_q.weight.detach().float(), a.norm_q.bias.detach().float()
                            gk, btk = a.norm_kv.weight.detach().float(), a.norm_kv.bias.detach().float()
                            Wqkv = torch.cat([sc * Wq * gq[None, :], Wkv * gk[None, :]], 0)
                            bqkv = torch.cat([sc * (Wq @ btq + bq), Wkv @ btk + bkv], 0)
                            w, ld = _pack_linear(Wqkv, dt)
                            b["qkv"] = _Layer(w, ld, bqkv.contiguous(), 3 * C)
                            # rows [C, 3C) = k | v: the projection of the neighbour frames, precomputable outside the chain
                            b["kv_l"] = _Layer(w[C:], ld, bqkv[C:].contiguous(), 2 * C)
                            W1, b1 = blk.mlp.fc1.weight.detach().float(), blk.mlp.fc1.bias.detach().float()
                            g2, bt2 = blk.norm2.weight.detach().float(), blk.norm2.bias.detach().float()
                            w, ld = _pack_linear(W1 * g2[None, :], dt)
                            b["fc1_ln"] = _Layer(w, ld, (W1 @ bt2 + b1).contiguous(), 4 * C)
                            # fully fused attention half (gather + LN + q/k/v + attention [+ proj + scatter]): needs the
                            # analytic relative-position index so that the bias can be rebuilt from the compact table
                            if (self.fuse_attn and ops.window_attention_fused_supported(C, self.heads, n_tok, self.D)
                                    and tuple(self.ws) == (7, 7)
                                    and torch.equal(a.relative_position_index.cpu(),
                                                    relative_position_index(self.D, 7, 7))):
                                rel = 13 * 13
                                tab = a.relative_position_bias_table.detach().float()
                                rows = [tab[((self.q_ind - d) + self.D - 1) * rel:((self.q_ind - d) + self.D) * rel]
                                        for d in range(self.D)]
                                b["tbl"] = torch.stack(rows, 0).permute(2, 0, 1).contiguous()       # [heads, D, 169]
                        else:
                            b.update(nq_g=_f32(a.norm_q.weight), nq_b=_f32(a.norm_q.bias),
                                     nkv_g=_f32(a.norm_kv.weight), nkv_b=_f32(a.norm_kv.bias),
                                     q=_lin_layer(a.q, dt, hd ** -0.5), kv=_lin_layer(a.kv, dt),
                                     n2_g=_f32(blk.norm2.weight), n2_b=_f32(blk.norm2.bias), fc1=_lin_layer(blk.mlp.fc1, dt))
                            if not use_mma:
                                b["bias"] = bias_hmn.permute(0, 2, 1).contiguous()       # [heads, D*n_kvf, n_tok]
                            if self.nwindow_size is not None:
                                rc = a.reduction_conv
                                b["red"] = (_f32(rc.weight.reshape(rc.weight.shape[0], -1)), _f32(rc.bias), n_kvf)
                        blocks.append(b)
                self.attn.append(blocks)
                # all blocks' k | v projections stacked: one LayerNorm-GEMM per finished frame (the "past" neighbour)
                if blocks and all("kv_l" in b for b in blocks):
                    w_all = torch.cat([b["kv_l"].w for b in blocks], 0).contiguous()
                    b_all = torch.cat([b["kv_l"].bias for b in blocks], 0).contiguous()
                    blocks[0]["kv_all"] = _Layer(w_all, blocks[0]["kv_l"].w_ld, b_all, w_all.shape[0])
            # last level with depth 0: ParseLayer + ResidualBlockNoBN x n (...V5.py:77-80, 261-282)
            self.tail = None
            if self.depths[-1] == 0:
                self.tail = [(_conv_layer(rb.conv1, 1, dt, tc), _conv_layer(rb.conv2, 1, dt, tc))
                             for rb in list(gen.feat_attns[-1])[1:]]
            self.dec = [_conv_layer(gen.decoders[i][1], 1, dt, tc) for i in range(self.L)]
            # skip_type 'concat': 1x1 fusion convolution over cat[skip, x] in front of every decoder (...V5.py:86-93)
            self.dec_fus = [_conv_layer(gen.decoders[i][0], 1, dt, tc) for i in range(self.L)] if self.concat else None
            pw, pb = gen.predI[1].weight.detach().float().reshape(-1), gen.predI[1].bias.detach().float()
            if self.concat:
                # predI = conv1x1(2bc -> bc) then conv1x1(bc -> 1) with nothing in between: one [2bc] vector
                W1 = gen.predI[0].weight.detach().float().reshape(self.bc, 2 * self.bc)
                b1 = gen.predI[0].bias.detach().float()
                w_eff = pw @ W1
                self.pred_w, self.pred_wh = w_eff[:self.bc].contiguous(), w_eff[self.bc:].contiguous()
                self.pred_b = (pw @ b1 + pb).reshape(1).contiguous()
            else:
                self.pred_w, self.pred_wh, self.pred_b = pw.contiguous(), None, pb.contiguous()
        # plans (buffers + CUDA graph per (T, B, Hp, Wp, slot)) are kept in an LRU bounded in bytes: the reference driver
        # with subseq_L=None calls the model with a different T per file (eval_models_seq.py:216-221)
        self.plans = OrderedDict()
        # budget: BDE2VID_PLAN_CACHE_GB, else 60 % of the device's memory (108 GB on a B200: two streams x eight 100-window
        # sequences keep ~2 x 33 GB of plans alive and must not evict each other inside a step)
        gb = os.environ.get("BDE2VID_PLAN_CACHE_GB")
        if gb is not None:
            self.plan_cache_bytes = int(float(gb) * 2 ** 30)
        elif torch.cuda.is_available():
            self.plan_cache_bytes = int(0.6 * torch.cuda.get_device_properties(self.device).total_memory)
        else:
            self.plan_cache_bytes = 64 * 2 ** 30
        self.dec_chunk = 8

    # ------------------------------------------------------------------------------------
    def plan(self, T, B, Hp, Wp, slot=0):
        """``slot`` selects an independent set of buffers + graph, so that several sequences can be
        in flight at once on different CUDA streams (one slot per stream)."""
        key = (T, B, Hp, Wp, slot)
        p = self.plans.get(key)
        if p is None:
            p = _Plan(self, T, B, Hp, Wp)
            self.plans[key] = p
            # evict least-recently-used plans (never the one just built) until the cache fits its byte budget
            total = sum(q.nbytes for q in self.plans.values())
            for k in list(self.plans.keys()):
                if total <= self.plan_cache_bytes or k == key:
                    break
                total -= self.plans[k].nbytes
                self.plans.pop(k).release()
        else:
            self.plans.move_to_end(key)
        return p

    def forward(self, vox_list, use_graph=True, slot=0):
        """vox_list: T tensors [B, bins, Hp, Wp] float32 (CUDA).  Returns T tensors [B, 1, Hp, Wp]."""
        T = len(vox_list)
        if T == 0:
            return []
        v0 = vox_list[0]
        if not v0.is_cuda:
            raise RuntimeError("BDE2VID.forward needs CUDA tensors (the reference driver moves voxels with "
                               ".to(device), eval_models_seq.py:204); no CPU path exists")
        B, bins, Hp, Wp = v0.shape
        if bins != self.bins:
            raise ValueError("expected %d voxel bins, got %d" % (self.bins, bins))
        S = 2 ** self.L
        if Hp % S or Wp % S:
            raise ValueError("input %dx%d must be padded to a multiple of %d (Croper.pad)" % (Hp, Wp, S))
        p = self.plan(T, B, Hp, Wp, slot)
        torch.stack([v.to(torch.float32) for v in vox_list], dim=0, out=p.vox_in)
        p.run(use_graph, from_events=False)
        img = p.img.clone().view(T, B, 1, Hp, Wp)
        return list(img.unbind(0))

    def forward_events(self, xs, ys, ts, ps, offsets, H, W, crop, use_graph=True, slot=0, normalize=None, hot_mask=None):
        """Fused path: raw events -> frames (voxeliser writes the padded grids the UNet reads)."""
        return self.forward_events_batch([(xs, ys, ts, ps, offsets)], H, W, crop, use_graph, slot, normalize, hot_mask)[0]

    def forward_events_batch(self, seqs, H, W, crop, use_graph=True, slot=0, normalize=None, hot_mask=None, pair=None):
        """B independent sequences (each a tuple xs, ys, ts, ps, offsets with the same number of windows)
        processed as one batch: every kernel of the schedule runs once for all B sequences.  Returns a list
        (per sequence) of T frames [1, 1, Hp, Wp].  Event arrays: loader format (four float32 arrays) or the on-disk
        dtypes (int16 x / y, float64 t, bool p).  ``normalize``: None | 'legacy' | 'robust' | ('robust', low, top)
        (the loader's LegacyNorm / RobustNorm voxel transforms); ``hot_mask``: optional float32 [H, W] hot-pixel mask."""
        B = len(seqs)
        T = seqs[0][4].numel() - 1
        if any(s[4].numel() - 1 != T for s in seqs):
            raise ValueError("sequences batched together must have the same number of windows")
        Hp, Wp = crop.height_crop_size, crop.width_crop_size
        p = self.plan(T, B, Hp, Wp, slot if pair is None else ("pair", pair.rank, slot))
        p.pair = pair
        p.set_events(seqs, H, W, crop.padding_top, crop.padding_left, normalize, hot_mask)
        p.run(use_graph and (pair is None or pair.graph), from_events=True)
        img = p.img.clone().view(T, B, 1, 1, Hp, Wp)
        return [list(img[:, b].unbind(0)) for b in range(B)]


class PairSplit:
    """Two GPUs share ONE sequence (SURVEY.md section 8, row f4).  Time cannot be split (the bidirectional recurrence and the
    in-place attention chain, ...V5.py:119-169), but per level the two recurrent chains are independent of each other:

      * rank 0 of the pair runs the FORWARD chain of every level, rank 1 the BACKWARD chain;
      * after the chains of a level the hidden-state sequences are exchanged (``hf`` from rank 0, ``hb`` from rank 1: one
        NCCL broadcast each over NVLink, T x B x h x w x C bf16) and both ranks form ``ff + fb``;
      * the attention chain of the level is sequential in t and needs every frame: both ranks run it, redundantly and
        bit-identically (same kernels, same inputs);
      * the decoder chunks (frames [c Tc, (c + 1) Tc)) alternate between the ranks; the frames meet in one all-reduce(sum)
        over the image buffer whose foreign chunks are zero (x + 0 is exact), so both ranks return all T frames.

    Head conv and the (merged) encoder convs are batched over all frames and cheap; both ranks run them.  ``graph``: capture
    the schedule incl. the NCCL calls in a CUDA graph (off by default: eager launches)."""

    def __init__(self, rank, group=None, src_ranks=(0, 1), graph=False):
        assert rank in (0, 1)
        self.rank, self.group, self.src_ranks, self.graph = rank, group, tuple(src_ranks), graph

    def owns_direction(self, rev):
        return self.rank == (1 if rev else 0)

    def owns_chunk(self, chunk_index):
        return chunk_index % 2 == self.rank

    def broadcast(self, t, owner):
        import torch.distributed as dist
        dist.broadcast(t, src=self.src_ranks[owner], group=self.group)

    def sum_frames(self, img):
        import torch.distributed as dist
        dist.all_reduce(img, op=dist.ReduceOp.SUM, group=self.group)


# kernel routes of one attention block (attention_routes; _Plan._attention_block runs them)
KVPRE = "kvpre"        # window_attention_fused_kvpre: neighbour k | v precomputed once per frame (BDE2VID_ATTN_KVPRE=1)
WHOLE = "whole"        # window_attention_fused, projection + scatter in the kernel
SPLIT = "split"        # window_attention_fused to the window output, then the proj + scatter GEMM
QKV = "qkv"            # LayerNorm-gather qkv GEMM, window_attention_mma_qkv, proj + scatter GEMM
UNFUSED = "unfused"    # LayerNorm gathers, q and kv GEMMs, attention kernel, proj + scatter, LayerNorm, fc1, fc2


def attention_routes(eng, l, C, nwin):
    """The kernel route of every attention block of level ``l`` (C channels, ``nwin`` windows per frame), and whether
    the blocks of the fused routes run their MLP as one kernel (else as two GEMMs)."""
    blocks = eng.attn[l]
    mlp_fused = eng.fuse_mlp and ops.mlp_fused_supported(C, 4 * C)
    if (C == 256 and eng.fuse_win256 and eng.kv_pre and nwin >= 64 and list(eng.buf) == [-1, 0, 1] and eng.q_ind == 1
            and all(b["tbl"] is not None for b in blocks)):
        return [KVPRE] * len(blocks), mlp_fused
    # C = 256: the whole-window kernel (gather + LN once per window, projection + scatter fused) once there are enough
    # windows to fill the SMs with one CTA each; below that (a single sequence has 35 level-3 windows) the per-head-group
    # kernel's 4 CTAs per window finish sooner
    whole = C == 64 or (eng.fuse_win256 and nwin >= eng.win256_min)
    return [(WHOLE if whole else SPLIT) if b["tbl"] is not None else QKV if "qkv" in b else UNFUSED
            for b in blocks], mlp_fused


class _Plan:
    """Static buffers + launch sequence for one (T, B, Hp, Wp)."""

    def __init__(self, eng, T, B, Hp, Wp):
        self.eng, self.T, self.B, self.Hp, self.Wp = eng, T, B, Hp, Wp
        dev, dt = eng.device, eng.dtype
        f32 = torch.float32
        self.nbytes = 0

        def E(*s, dtype=dt, zero=False):
            t = (torch.zeros if zero else torch.empty)(*s, dtype=dtype, device=dev)
            self.nbytes += t.numel() * t.element_size()
            return t

        N = T * B
        self.vox_in = E(T, B, eng.bins, Hp, Wp, dtype=f32)
        self.vox8 = E(N, Hp, Wp, VOX_CPAD) if eng.head_direct is None else None
        self.head = E(N, Hp, Wp, eng.bc)
        self.img = E(N, Hp, Wp, dtype=f32)
        self.lv = []
        for l in range(eng.L):
            h, w, C = Hp >> (l + 1), Wp >> (l + 1), eng.bc * 2 ** (l + 1)
            # merged forward / backward encoder conv: the recurrent chains then read channel halves of one [.., 2C] map,
            # which only the TMA conv kernel can do (it needs C % 64 == 0 and a map of at least 8 x 8)
            merged = ("fb_conv" in eng.enc[l] and C % 64 == 0 and h >= 8 and w >= 8
                      and os.environ.get("BDE2VID_CONV_TMA", "1") != "0")
            efb = E(N, h, w, 2 * C) if merged else None      # [.., :C] forward encoder conv, [.., C:] backward
            d = dict(h=h, w=w, C=C, efb=efb,
                     ef=None if merged else E(N, h, w, C), eb=None if merged else E(N, h, w, C),
                     feat=E(N, h, w, C, dtype=f32))
            if eng.rec is not None:
                # hf / hb: hidden state of every frame (the chains' output); cf / cb: fp32 ping-pong of the ConvLSTM cell
                # state, or of the ConvGRU hidden state's fp32 master copy
                d.update(hf=E(N, h, w, C), hb=E(N, h, w, C),
                         cf=[E(B, h, w, C, dtype=f32) for _ in range(2)], cb=[E(B, h, w, C, dtype=f32) for _ in range(2)],
                         zero=E(B, h, w, C, zero=True))
            if eng.rec == "convgru":
                d.update(uf=E(B, h, w, C, dtype=f32), ub=E(B, h, w, C, dtype=f32), hrf=E(B, h, w, C), hrb=E(B, h, w, C))
            d["feat_t"] = d["feat"] if dt == f32 else E(N, h, w, C)
            if eng.depths[l] > 0:
                ws = eng.ws
                if h < ws[0] or w < ws[1]:
                    raise NotImplementedError(
                        "feature map %dx%d at attention level %d is smaller than the %dx%d window; the reference "
                        "fails on such inputs too (relative_position_index is built for full windows)" % (h, w, l, *ws))
                tm_plain, g = window_token_map(B, h, w, ws, False, dev)
                tm_dil, _ = window_token_map(B, h, w, ws, True, dev)
                nwin = tm_plain.shape[0]
                ntok = ws[0] * ws[1]
                P = B * h * w
                routes, mlp_fused = attention_routes(eng, l, C, nwin)
                d.update(tm=[tm_plain, tm_dil], nwin=nwin, ntok=ntok, routes=routes, mlp_fused=mlp_fused,
                         xs=E(P, C, dtype=f32), ob=E(nwin * ntok, C))
                # scratch of the routes the blocks take
                if QKV in routes:
                    d["qkv"] = E(nwin * eng.D * ntok, 3 * C)
                if UNFUSED in routes:
                    n_kvf = ntok if eng.nwindow_size is None else eng.nwindow_size[0] * eng.nwindow_size[1]
                    d.update(qn=E(nwin * ntok, C), kvn=E(nwin * eng.D * n_kvf, C), qb=E(nwin * ntok, C),
                             kvb=E(nwin * eng.D * n_kvf, 2 * C))
                    if eng.nwindow_size is not None:
                        d["kvr"] = E(nwin * eng.D * n_kvf, C, dtype=f32)
                if UNFUSED in routes or not mlp_fused:
                    d.update(yn=E(P, C), hid=E(P, 4 * C))
                if KVPRE in routes:
                    # precomputed neighbour k | v: future frames for every block and frame, past frame ping-pong
                    d["kv_fut"] = E(len(routes), T, P, 2 * C)
                    d["kv_past"] = [E(P, len(routes) * 2 * C) for _ in range(2)]
                    d["xn_all"] = E(T * P, C)          # LayerNorm'ed (no affine: folded into the weights) features, bf16
                    d["ln_one"] = torch.ones(C, dtype=f32, device=dev)
                    d["ln_zero"] = torch.zeros(C, dtype=f32, device=dev)
            elif l == eng.L - 1 and eng.tail is not None:
                P = B * h * w
                # ResidualBlockNoBN tail: running x (fp32 + operand copy) and the conv1 output
                d.update(tl_x=E(B, h, w, C, dtype=f32), tl_xb=E(B, h, w, C), tl_y=E(B, h, w, C),
                         tl_zero=E(B, h, w, C, dtype=f32, zero=True))
                d["tl_zerob"] = d["tl_zero"] if dt == f32 else E(B, h, w, C, zero=True)
            self.lv.append(d)
        Tc = min(eng.dec_chunk, T)
        self.Tc = Tc
        self.dec = []
        for i in range(eng.L):
            l_in = eng.L - 1 - i                     # level whose resolution the decoder input has
            h, w, C = self.lv[l_in]["h"], self.lv[l_in]["w"], self.lv[l_in]["C"]
            dd = dict(h=h, w=w, C=C, up=E(Tc * B, 2 * h, 2 * w, C), out=E(Tc * B, 2 * h, 2 * w, C // 2))
            if eng.concat:
                dd["fus"] = E(Tc * B, h, w, C)
            self.dec.append(dd)
        self.graphs = {}
        self.runs = {}
        self.pair = None                # PairSplit: this plan runs its share of a sequence split over two GPUs
        self.ev = None
        self.ev_kind = None
        self.norm = (0, 0.0, 95.0)      # voxel normalisation of the fused events path: (mode, low_perc, top_perc)
        self.hot_mask = None
        self.oob = E(1, dtype=torch.int32, zero=True)
        self.oob_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.oob_event = None
        self.side = torch.cuda.Stream(device=dev)
        # two-stream schedule (backward chain / decoders on `side`); False serialises everything on one stream
        self.overlap = os.environ.get("BDE2VID_OVERLAP", "1") != "0"

    def release(self):
        """Drop the CUDA graph and every buffer (LRU eviction)."""
        self.graphs.clear()
        self.lv, self.dec, self.ev = [], [], None
        self.vox_in = self.vox8 = self.head = self.img = None

    # ------------------------------------------------------------------------------------
    def check_oob(self):
        """Events outside the sensor are dropped by the fused path (the reference's index_put_ raises IndexError).  The
        count of the previous run is copied to pinned host memory asynchronously and examined here, at the next call:
        BDE2VID_STRICT_OOB=1 waits for it and raises like the reference, otherwise a finished count != 0 warns."""
        if self.oob_event is None:
            return
        strict = os.environ.get("BDE2VID_STRICT_OOB", "0") == "1"
        if strict:
            self.oob_event.synchronize()
        if self.oob_event.query():
            n = int(self.oob_host.item())
            self.oob_event = None
            if n:
                msg = "%d events outside the sensor were dropped by the fused voxeliser" % n
                if strict:
                    raise IndexError(msg)
                warnings.warn(msg)

    def set_events(self, seqs, H, W, pad_top, pad_left, normalize=None, hot_mask=None):
        """Stage the events of the B sequences into static buffers (host or device sources; the copies are
        asynchronous on the current stream) so that the captured graph can include the voxeliser.  Event arrays are
        either the loader format (four float32 arrays) or the on-disk dtypes (int16, int16, float64, bool / uint8)."""
        assert len(seqs) == self.B
        self.check_oob()
        n = max(s[0].numel() for s in seqs)
        dev = self.eng.device
        geom = (H, W, pad_top, pad_left)
        raw = seqs[0][0].dtype != torch.float32
        dts = (torch.int16, torch.int16, torch.float64, torch.uint8) if raw else (torch.float32,) * 4
        norm = (0, 0.0, 95.0)
        if normalize is not None:
            mode = {"legacy": ops.NORM_LEGACY, "LegacyNorm": ops.NORM_LEGACY, "robust": ops.NORM_ROBUST,
                    "RobustNorm": ops.NORM_ROBUST}[normalize if isinstance(normalize, str) else normalize[0]]
            lo, hi = (0.0, 95.0) if isinstance(normalize, str) else (float(normalize[1]), float(normalize[2]))
            norm = (mode, lo, hi)
        if (self.ev is None or self.ev_cap < n or self.ev_geom != geom or self.ev_kind != raw or self.norm != norm
                or (hot_mask is None) != (self.hot_mask is None)):
            self.ev_cap = max(int(n * 1.25) + 16, 1024)
            self.ev = [[torch.zeros(self.ev_cap, dtype=d, device=dev) for d in dts] for _ in range(self.B)]
            self.ev_off = [torch.zeros(self.T + 1, dtype=torch.int64, device=dev) for _ in range(self.B)]
            self.ev_geom, self.ev_kind, self.norm = geom, raw, norm
            self.hot_mask = None if hot_mask is None else torch.empty(H, W, dtype=torch.float32, device=dev)
            self.graphs.pop(True, None)
            self.runs[True] = 0
        if hot_mask is not None:
            self.hot_mask.copy_(hot_mask, non_blocking=True)
        for b, (xs, ys, ts, ps, offsets) in enumerate(seqs):
            m = xs.numel()
            for dst, src in zip(self.ev[b], (xs, ys, ts, ps)):
                dst[:m].copy_(src.view(torch.uint8) if src.dtype == torch.bool else src, non_blocking=True)
            self.ev_off[b].copy_(offsets, non_blocking=True)

    def run(self, use_graph, from_events):
        self.runs[from_events] = self.runs.get(from_events, 0) + 1
        if not use_graph:
            self._enqueue(from_events)
        else:
            if from_events not in self.graphs and self.runs[from_events] >= 2:
                g = torch.cuda.CUDAGraph()
                torch.cuda.synchronize()
                with torch.cuda.graph(g):
                    self._enqueue(from_events)
                self.graphs[from_events] = g
            if from_events in self.graphs:
                self.graphs[from_events].replay()
            else:
                self._enqueue(from_events)
        if from_events:
            self.oob_host.copy_(self.oob, non_blocking=True)
            self.oob_event = torch.cuda.Event()
            self.oob_event.record()

    # ------------------------------------------------------------------------------------
    def _chain_step(self, d, layer_key, e, xin, pitch, hbuf, cbuf, t, tprev, k, rev):
        """One recurrent step of one direction: ConvLSTM (gates conv + pointwise update in one launch) or ConvGRU (two
        launches: [update | reset] conv -> u, h * r;  out_gate conv -> h')."""
        eng, B = self.eng, self.B
        h, w, C = d["h"], d["w"], d["C"]
        first = k == 0
        hprev = d["zero"] if first else hbuf[tprev * B:(tprev + 1) * B]
        if eng.rec == "convlstm":
            eng.gemm(e[layer_key + "_lstm"], xin, hbuf[t * B:(t + 1) * B], B, h, w, C, a1=hprev, c1=C, epi=EPI_LSTM,
                      c_prev=None if first else cbuf[(k + 1) & 1], c_out=cbuf[k & 1], **pitch)
            self.launches += 1
            return
        ur, og = e[layer_key + "_gru"]
        u, hr = (d["ub"], d["hrb"]) if rev else (d["uf"], d["hrf"])
        hm_prev = None if first else cbuf[(k + 1) & 1]
        eng.gemm(ur, xin, hr, B, h, w, C, a1=hprev, c1=C, epi=EPI_GRU_UR, c_prev=hm_prev, c_out=u, **pitch)
        eng.gemm(og, xin, hbuf[t * B:(t + 1) * B], B, h, w, C, a1=hr, c1=C, epi=EPI_GRU_OUT, c_prev=hm_prev, residual=u,
                  c_out=cbuf[k & 1], **pitch)
        self.launches += 2

    def _enqueue(self, from_events):
        eng, T, B, Hp, Wp = self.eng, self.T, self.B, self.Hp, self.Wp
        N = T * B
        self.launches = 0
        if from_events:
            H, W, pt, pl = self.ev_geom
            self.oob.zero_()
            # sequence b writes windows t = 0..T-1 at vox_in[t, b]: window stride = B grids.  min_events = 3 is the loader
            # contract (h5_dataset.py:219-221): windows with fewer than 3 events give an all-zero grid
            for b in range(B):
                xs, ys, ts, ps = self.ev[b]
                ops.voxelize_seq_into(xs, ys, ts, ps, self.ev_off[b], eng.bins, H, W, pt, pl, Hp, Wp,
                                      self.vox_in[0, b], B * eng.bins * Hp * Wp, oob_count=self.oob, min_events=3,
                                      hot_mask=self.hot_mask)
                self.launches += 1
            if self.norm[0]:
                # LegacyNorm / RobustNorm of the loader (transform_voxel, h5_dataset.py:226), per window, in place
                ops.voxel_normalize(self.vox_in, H, W, pt, pl, self.norm[0], self.norm[1], self.norm[2],
                                    window_stride=eng.bins * Hp * Wp, n_windows=N)
                self.launches += 1
        # A: head conv + activation over all frames (...V5.py:116)
        if eng.head_direct is not None:
            ops.head_conv(self.vox_in.view(N, eng.bins, Hp, Wp), eng.head_direct[0], eng.head_direct[1], self.head, act=eng.net_act)
            self.launches += 1
        else:
            ops.pack_voxel_nhwc(self.vox_in.view(N, eng.bins, Hp, Wp), VOX_CPAD, eng.dtype, out=self.vox8)
            eng.gemm(eng.head, self.vox8, self.head, N, Hp, Wp, VOX_CPAD, act=eng.net_act)
            self.launches += 2
        x, xc, xh, xw = self.head, eng.bc, Hp, Wp
        for l in range(eng.L):
            d, e = self.lv[l], eng.enc[l]
            h, w, C = d["h"], d["w"], d["C"]
            # the two recurrent chains (sequential in t; gates conv + pointwise fused in one kernel) are independent
            # of each other: the backward direction (conv + chain) runs on a second stream
            main = torch.cuda.current_stream()
            side = self.side if self.overlap else main
            merged = d["efb"] is not None
            if merged:
                # both directions' encoder convs in one launch over all T (same input, N doubled); each chain then reads
                # its channel half of the [.., 2C] map through a pitched TMA descriptor
                eng.gemm(e["fb_conv"], x, d["efb"], N, xh, xw, xc, act=eng.net_act)
                self.launches += 1
            side.wait_stream(main)
            pair = self.pair
            for (strm, key, conv, src, rev) in ((main, "f", e["f_conv"], d["ef"], False), (side, "b", e["b_conv"], d["eb"], True)):
                if pair is not None and eng.rec is not None and not pair.owns_direction(rev):
                    continue                      # the other GPU of the pair runs this direction (PairSplit)
                with torch.cuda.stream(main if pair is not None else strm):
                    if not merged:
                        # encoder conv is not recurrent: one launch over all T (...V5.py:129-130, conv part)
                        eng.gemm(conv, x, src, N, xh, xw, xc, act=eng.net_act)
                        self.launches += 1
                    if eng.rec is None:
                        continue                  # useRC=False: the encoder is the ConvLayer alone (...V5.py:255-257)
                    hbuf, cbuf = (d["hb"], d["cb"]) if rev else (d["hf"], d["cf"])
                    for k in range(T):
                        t, tprev = (T - 1 - k, T - k) if rev else (k, k - 1)
                        if merged:
                            xin = d["efb"][t * B:(t + 1) * B, :, :, (C if rev else 0):(2 * C if rev else C)]
                            pitch = dict(a0_ld=2 * C)
                        else:
                            xin, pitch = src[t * B:(t + 1) * B], {}
                        self._chain_step(d, key, e, xin, pitch, hbuf, cbuf, t, tprev, k, rev)
            main.wait_stream(side)
            if pair is not None and eng.rec is not None:
                pair.broadcast(d["hf"], 0)
                pair.broadcast(d["hb"], 1)
            # merged = ff + fb (...V5.py:137-147)
            ff, fb = (d["ef"], d["eb"]) if eng.rec is None else (d["hf"], d["hb"])
            ops.add(ff, fb, out_f32=d["feat"], out_t=None if eng.dtype == torch.float32 else d["feat_t"], dtype=eng.dtype)
            self.launches += 1
            last = l == eng.L - 1
            if eng.depths[l] > 0:
                # the last level's frames are final as soon as their attention step is done: the decoders of a
                # finished chunk of frames run on the side stream while the (latency-bound) chain continues
                self._attention_level(l, self._decode_chunk_async if last else None)
            elif last and eng.tail is not None:
                self._tail_level(l, self._decode_chunk_async)
            x, xc, xh, xw = d["feat_t"], C, h, w
        if self.overlap:
            torch.cuda.current_stream().wait_stream(self.side)
        if self.pair is not None:
            self.pair.sum_frames(self.img)

    def _tail_level(self, l, on_frame_done):
        """Last level with depth 0 (...V5.py:77-80, 151-169, 261-282): per frame, in order, x = feats_buffer[0] (ParseLayer:
        the frame at offset buffer_index[0], all-zero outside the sequence, already updated if it is a past frame --
        quirk Q5 with Q1 / Q4), then num_res_blocks x (x = x + conv2(act(conv1(x)))), then merged[t] = x + merged[t]."""
        eng, T, B = self.eng, self.T, self.B
        d = self.lv[l]
        h, w, C = d["h"], d["w"], d["C"]
        P = B * h * w
        feat = d["feat"].view(T, P * C)
        feat_t = d["feat_t"].view(T, P * C)
        lowp = eng.dtype != torch.float32
        for t in range(T):
            src_t = t + eng.buf[0]
            if 0 <= src_t < T:
                x32, xop = feat[src_t].view(B, h, w, C), feat_t[src_t].view(B, h, w, C)
            else:
                x32, xop = d["tl_zero"], d["tl_zerob"]
            for (c1, c2) in eng.tail:
                eng.gemm(c1, xop, d["tl_y"], B, h, w, C, act=eng.net_act)
                # conv2 + bias + residual (fp32, after the absent activation): x = x + conv2(.)
                eng.gemm(c2, d["tl_y"], d["tl_x"], B, h, w, C, out_f32=True, residual=x32,
                          out2=d["tl_xb"] if lowp else None)
                x32, xop = d["tl_x"], d["tl_xb"] if lowp else d["tl_x"]
                self.launches += 2
            ops.add(x32.view(-1), feat[t], out_f32=feat[t], out_t=feat_t[t] if lowp else None, dtype=eng.dtype)
            self.launches += 1
            on_frame_done(t)

    def _decode_chunk_async(self, t):
        """Called after frame t of the last level is final; launches the decoder of a completed chunk."""
        T, Tc = self.T, self.Tc
        if (t + 1) % Tc != 0 and t != T - 1:
            return
        t0 = (t // Tc) * Tc
        if self.pair is not None and not self.pair.owns_chunk(t // Tc):
            self.img[t0 * self.B:(min(t0 + Tc, T)) * self.B].zero_()     # the other GPU's chunk: zero for the final all-reduce(sum)
            return
        if not self.overlap:
            self._decode_chunk(t0)
            return
        self.side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(self.side):
            self._decode_chunk(t0)

    def _decode_chunk(self, t0):
        """C: decoders + prediction for frames [t0, t0 + Tc) (...V5.py:183-197)."""
        eng, T, B, Hp, Wp = self.eng, self.T, self.B, self.Hp, self.Wp
        n = min(self.Tc, T - t0) * B
        s = slice(t0 * B, t0 * B + n)
        cur = None
        for i in range(eng.L):
            dd = self.dec[i]
            l_in = eng.L - 1 - i
            if eng.concat:
                # skip_concat: fusion conv1x1 over cat[skip, x] (two GEMM sources), then bilinear x2 + conv (...V5.py:86-93).
                # Quirk Q2: decoder 0 sees cat[feat, feat]
                skip = self.lv[l_in]["feat_t"][s]
                xin = skip if i == 0 else cur
                eng.gemm(eng.dec_fus[i], skip, dd["fus"][:n], n, dd["h"], dd["w"], dd["C"], a1=xin, c1=dd["C"])
                ops.upsample2x_sum(None, dd["fus"][:n], 1.0, n, dd["h"], dd["w"], dd["C"], dd["up"][:n])
                self.launches += 1
            else:
                feat = self.lv[l_in]["feat"][s]
                if i == 0:    # quirk Q2: the last level is appended twice -> decoder 0 sees feat + feat
                    ops.upsample2x_sum(None, feat, 2.0, n, dd["h"], dd["w"], dd["C"], dd["up"][:n])
                else:
                    ops.upsample2x_sum(feat, cur, 1.0, n, dd["h"], dd["w"], dd["C"], dd["up"][:n])
            eng.gemm(eng.dec[i], dd["up"][:n], dd["out"][:n], n, 2 * dd["h"], 2 * dd["w"], dd["C"], act=ACT_RELU6)
            cur = dd["out"][:n]
            self.launches += 2
        ops.pred_sigmoid(cur, self.head[s], eng.pred_w, eng.pred_b, eng.bc, n * Hp * Wp, self.img[s], wt_head=eng.pred_wh,
                         act=eng.out_act)
        self.launches += 1

    def _mlp(self, blk, d, xs, P, C, sum_io=None, sum_t=None):
        """xs += fc2(GELU(fc1(LN(xs)))) (DTransformer.py:279-283,302-304): one fused kernel where supported.
        Returns True when the optional "x + merged" sum (sum_io += xs, sum_t = bf16) was fused into that kernel."""
        eng = self.eng
        if d["mlp_fused"]:
            ops.mlp_fused(xs, P, C, 4 * C, blk["fc1_ln"].w, blk["fc1_ln"].bias, blk["fc2"].w, blk["fc2"].bias,
                          sum_io=sum_io, sum_t=sum_t)
            self.launches += 1
            return sum_io is not None
        else:
            eng.gemm(blk["fc1_ln"], None, d["hid"], 1, P, 1, C, act=ACT_GELU, ln_frames=[xs])
            eng.gemm(blk["fc2"], d["hid"], xs, 1, P, 1, 4 * C, out_f32=True, residual=xs)
            self.launches += 2
        return False

    def _attention_level(self, l, on_frame_done=None):
        """In-place sequential multi-frame window attention (...V5.py:151-169; DTransformer.py:254-389)."""
        eng, T, B = self.eng, self.T, self.B
        d = self.lv[l]
        h, w, C = d["h"], d["w"], d["C"]
        P = B * h * w
        feat = d["feat"].view(T, P, C)
        feat_t = d["feat_t"].view(T, P, C)
        xs, routes = d["xs"], d["routes"]
        pre = KVPRE in routes
        if pre:
            # k | v of the (pre-attention) future neighbours, all frames at once per block
            # (one LayerNorm pass, then per block a 1x1 convolution over the [T*B, h, w, C] map on the TMA conv kernel)
            ops.layernorm(feat.view(T * P, C), T * P, C, d["ln_one"], d["ln_zero"], d["xn_all"])
            for i, blk in enumerate(eng.attn[l]):
                eng.gemm(blk["kv_l"], d["xn_all"], d["kv_fut"][i].view(T * P, 2 * C), T * B, h, w, C)
            self.launches += 1 + len(eng.attn[l])
        for t in range(T):
            # past neighbours are already post-attention (updated in place), future ones are not: quirk Q1
            frames = [feat[t + o] if 0 <= t + o < T else None for o in eng.buf]      # None = all-zero map (Q4)
            qsrc = frames[eng.q_ind]
            # the first block (plain windows: every pixel belongs to exactly one window) of the fused-projection kernels
            # reads the query frame / shortcut straight from feat[t] and writes x: no copy of feat[t] into xs
            direct0 = qsrc is not None and routes[0] in (WHOLE, KVPRE)
            if not direct0:
                if qsrc is None:
                    xs.zero_()
                else:
                    ops.cast(qsrc, xs)
                self.launches += 1
            sum_done = False
            for i, (blk, route) in enumerate(zip(eng.attn[l], routes)):
                # the last block's fused MLP also does "x + merged[t]" (feat[t] += x, bf16 copy) -- bf16 engine only
                last = i == len(routes) - 1 and eng.dtype != torch.float32
                sum_args = (feat[t], feat_t[t]) if last else (None, None)
                fr = list(frames)
                fr[eng.q_ind] = qsrc if (direct0 and i == 0) else xs
                sum_done = self._attention_block(route, i, blk, d, fr, t, sum_args)
            # x + merged[t], stored back in place (...V5.py:166-169), unless the last MLP kernel already did it
            if not sum_done:
                ops.add(xs, feat[t], out_f32=feat[t], out_t=None if eng.dtype == torch.float32 else feat_t[t],
                        dtype=eng.dtype)
                self.launches += 1
            if pre and t + 1 < T:
                # this frame is final: its k | v for every block of the next step (the "past" neighbour there)
                xn_t = d["xn_all"][t * P:(t + 1) * P]      # (its pre-attention copy is not needed any more)
                ops.layernorm(feat[t], P, C, d["ln_one"], d["ln_zero"], xn_t)
                eng.gemm(eng.attn[l][0]["kv_all"], xn_t, d["kv_past"][t & 1], B, h, w, C)
                self.launches += 2
            if on_frame_done is not None:
                on_frame_done(t)

    def _attention_block(self, route, i, blk, d, fr, t, sum_args):
        """Block ``i`` at frame ``t`` along its route, in place on xs (``fr``: its input frames).  Returns True when the
        block's MLP kernel also did the "x + merged" sum of ``sum_args``."""
        eng, C, nwin, ntok, D, xs = self.eng, d["C"], d["nwin"], d["ntok"], self.eng.D, d["xs"]
        P = xs.shape[0]
        tm = d["tm"][i & 1]
        if route == UNFUSED:
            n_kvf = ntok
            if "red" in blk:
                # nwindow_size (DTransformer.py:172-175): q from the window's tokens, kv from the "feature reduction"
                # conv of every frame's window (raw tokens), then norm_kv
                rw, rb, n_kvf = blk["red"]
                ops.ln_gather([fr[eng.q_ind]], tm, nwin, ntok, C, blk["nq_g"], blk["nq_b"], d["qn"])
                ops.window_reduce(fr, tm.view(-1), nwin, ntok, C, n_kvf, rw, rb, d["kvr"])
                ops.layernorm(d["kvr"], nwin * D * n_kvf, C, blk["nkv_g"], blk["nkv_b"], d["kvn"])
                self.launches += 3
            elif C in (64, 128, 256):
                ops.ln_gather_qkv(fr, eng.q_ind, tm, nwin, ntok, C, blk["nkv_g"], blk["nkv_b"], blk["nq_g"],
                                  blk["nq_b"], d["kvn"], d["qn"])
                self.launches += 1
            else:
                ops.ln_gather([fr[eng.q_ind]], tm, nwin, ntok, C, blk["nq_g"], blk["nq_b"], d["qn"])
                ops.ln_gather(fr, tm, nwin, ntok, C, blk["nkv_g"], blk["nkv_b"], d["kvn"])
                self.launches += 2
            eng.gemm(blk["q"], d["qn"], d["qb"], 1, nwin * ntok, 1, C)
            eng.gemm(blk["kv"], d["kvn"], d["kvb"], 1, nwin * D * n_kvf, 1, C)
            if "bias_mma" in blk:
                ops.window_attention_mma(d["qb"], d["kvb"], blk["bias_mma"], nwin, ntok, D * ntok, C, eng.heads, d["ob"])
            else:
                ops.window_attention(d["qb"], d["kvb"], blk["bias"], nwin, ntok, D * n_kvf, C, eng.heads, d["ob"])
            # proj + window_reverse + crop + shortcut: x[pixel] += proj(o); uncovered pixels keep x
            eng.gemm(blk["proj"], d["ob"], xs, 1, nwin * ntok, 1, C, epi=EPI_SCATTER, row_map=tm.view(-1))
            ops.layernorm(xs, P, C, blk["n2_g"], blk["n2_b"], d["yn"])
            eng.gemm(blk["fc1"], d["yn"], d["hid"], 1, P, 1, C, act=ACT_GELU)
            eng.gemm(blk["fc2"], d["hid"], xs, 1, P, 1, 4 * C, out_f32=True, residual=xs)
            self.launches += 7
            return False
        if route == KVPRE:
            kv = [None] * D
            if t >= 1:
                kv[0] = d["kv_past"][(t - 1) & 1][:, i * 2 * C:(i + 1) * 2 * C]
            if t + 1 < self.T:
                kv[2] = d["kv_fut"][i, t + 1]
            ops.window_attention_fused_kvpre(fr[eng.q_ind], kv, eng.q_ind, tm.view(-1), nwin, C, eng.heads, blk["qkv"].w,
                                             blk["qkv"].bias, blk["tbl"], blk["proj"].w, blk["proj"].bias, xs)
            self.launches += 1
        elif route == WHOLE:
            ops.window_attention_fused(fr, eng.q_ind, tm.view(-1), nwin, C, eng.heads, blk["qkv"].w, blk["qkv"].bias,
                                       blk["tbl"], blk["proj"].w, blk["proj"].bias, xs=xs)
            self.launches += 1
        elif route == SPLIT:
            ops.window_attention_fused(fr, eng.q_ind, tm.view(-1), nwin, C, eng.heads, blk["qkv"].w, blk["qkv"].bias,
                                       blk["tbl"], o_out=d["ob"])
            eng.gemm(blk["proj"], d["ob"], xs, 1, nwin * ntok, 1, C, epi=EPI_SCATTER, row_map=tm.view(-1))
            self.launches += 2
        else:   # QKV: [window gather + LayerNorm + q/k/v projection] -> attention -> proj + scatter
            eng.gemm(blk["qkv"], None, d["qkv"], 1, nwin * D * ntok, 1, C, ln_frames=fr, ln_tok_map=tm.view(-1),
                     ln_n_tok=ntok)
            ops.window_attention_mma_qkv(d["qkv"], blk["bias_mma"], nwin, ntok, D * ntok, eng.q_ind * ntok, C, eng.heads,
                                         d["ob"])
            eng.gemm(blk["proj"], d["ob"], xs, 1, nwin * ntok, 1, C, epi=EPI_SCATTER, row_map=tm.view(-1))
            self.launches += 3
        return self._mlp(blk, d, xs, P, C, *sum_args)
