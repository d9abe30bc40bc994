"""Python-side wrappers of the C ABI (one function per entry point of include/bde2vid.h).

All tensors are contiguous CUDA tensors owned by PyTorch; the wrappers only pass pointers and
sizes and enqueue on ``torch.cuda.current_stream()``.  Nothing here computes on the host.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import (ACT_GELU, ACT_NONE, ACT_RELU, ACT_RELU6, ACT_SIGMOID, BDE_DTYPE, BF16, ENGINE_SIMT,  # noqa: F401
                   ENGINE_TCGEN05, EPI_GRU_OUT, EPI_GRU_UR, EPI_LSTM, EPI_SCATTER, EPI_STORE, F32, TORCH_DTYPE, check, ptr, stream_ptr)


def voxelize_seq(xs, ys, ts, ps, offsets, num_bins, H, W, pad_top=0, pad_left=0, Hp=None, Wp=None, out=None,
                 oob_count=None, algo=0, min_events=1):
    """float32 event arrays + int64 CSR offsets [T+1] -> float32 [T, bins, Hp, Wp].  ``min_events``: windows with fewer
    events give zeros (1 = the bare reference function, 3 = the loader contract h5_dataset.py:219-221)."""
    lib = _lib.require_device()
    Hp = H + pad_top if Hp is None else Hp
    Wp = W + pad_left if Wp is None else Wp
    T = offsets.numel() - 1
    for t in (xs, ys, ts, ps):
        assert t.dtype == torch.float32 and t.is_cuda
    assert offsets.dtype == torch.int64 and offsets.is_cuda
    if out is None:
        out = torch.empty((T, num_bins, Hp, Wp), dtype=torch.float32, device=xs.device)
    assert out.shape == (T, num_bins, Hp, Wp) and out.dtype == torch.float32
    check(lib.bde_voxelize_seq(ptr(xs), ptr(ys), ptr(ts), ptr(ps), ptr(offsets), T, num_bins, H, W, pad_top, pad_left,
                               Hp, Wp, ptr(out), ptr(oob_count), algo, min_events, stream_ptr()), "bde_voxelize_seq")
    return out


def voxelize_seq_into(xs, ys, ts, ps, offsets, num_bins, H, W, pad_top, pad_left, Hp, Wp, out_view, window_stride,
                      oob_count=None, algo=0, min_events=1, hot_mask=None):
    """Voxelise one sequence into a strided destination: ``out_view`` is the tensor element where window 0's grid
    starts and consecutive windows are ``window_stride`` floats apart (batch buffers [T, B, bins, Hp, Wp]).
    Event arrays: four float32 tensors (loader format) or the on-disk dtypes int16 / int16 / float64 / bool|uint8
    (bde_voxelize_raw_strided)."""
    lib = _lib.require_device()
    T = offsets.numel() - 1
    if xs.dtype == torch.float32:
        assert ys.dtype == ts.dtype == ps.dtype == torch.float32
        fn, name = lib.bde_voxelize_seq_strided, "bde_voxelize_seq_strided"
    else:
        assert xs.dtype == torch.int16 and ys.dtype == torch.int16 and ts.dtype == torch.float64 \
            and ps.dtype in (torch.bool, torch.uint8), "raw events must be int16 / int16 / float64 / bool"
        fn, name = lib.bde_voxelize_raw_strided, "bde_voxelize_raw_strided"
    assert hot_mask is None or (hot_mask.dtype == torch.float32 and hot_mask.shape == (H, W))
    check(fn(ptr(xs), ptr(ys), ptr(ts), ptr(ps), ptr(offsets), T, num_bins, H, W, pad_top, pad_left, Hp, Wp,
             C.c_void_p(out_view.data_ptr()), window_stride, ptr(oob_count), algo, min_events, ptr(hot_mask), stream_ptr()), name)


def voxelize_raw(xs, ys, ts, ps, offsets, num_bins, H, W, pad_top=0, pad_left=0, Hp=None, Wp=None, out=None,
                 oob_count=None, algo=0, min_events=3, hot_mask=None):
    """On-disk event dtypes (int16 x / y, float64 t, bool p) + CSR offsets -> float32 [T, bins, Hp, Wp]; the loader's
    conversions (h5_dataset.py:222-225, :414) happen in the kernel."""
    Hp = H + pad_top if Hp is None else Hp
    Wp = W + pad_left if Wp is None else Wp
    T = offsets.numel() - 1
    if out is None:
        out = torch.empty((T, num_bins, Hp, Wp), dtype=torch.float32, device=xs.device)
    voxelize_seq_into(xs, ys, ts, ps, offsets, num_bins, H, W, pad_top, pad_left, Hp, Wp, out, num_bins * Hp * Wp,
                      oob_count=oob_count, algo=algo, min_events=min_events, hot_mask=hot_mask)
    return out


NORM_LEGACY, NORM_ROBUST = 1, 2


def voxel_normalize(grids, H, W, pad_top, pad_left, mode, low_perc=0.0, top_perc=95.0, window_stride=None, n_windows=None,
                    stats=None):
    """In-place LegacyNorm / RobustNorm of every window's sensor area (see bde_voxel_normalize).  ``grids``: float32
    [T, bins, Hp, Wp] contiguous, or any float32 view whose window 0 starts at its first element when ``window_stride`` /
    ``n_windows`` (floats between windows, number of windows) are given with bins / Hp / Wp taken from its last 3 dims."""
    lib = _lib.require_device()
    bins, Hp, Wp = grids.shape[-3:]
    if window_stride is None:
        assert grids.is_contiguous()
        window_stride = bins * Hp * Wp
        n_windows = grids.numel() // window_stride
    assert grids.dtype == torch.float32
    check(lib.bde_voxel_normalize(C.c_void_p(grids.data_ptr()), window_stride, n_windows, bins, H, W, pad_top, pad_left, Hp, Wp,
                                  mode, float(low_perc), float(top_perc), ptr(stats), stream_ptr()), "bde_voxel_normalize")
    return grids


def hot_pixel_mask(xs, ys, ps, H, W, num_hot):
    """get_hot_event_mask (event_utils.py:100-116) on the device: float32 [H, W] of {0, 1}."""
    lib = _lib.require_device()
    assert xs.dtype == torch.int16 and ys.dtype == torch.int16 and ps.dtype in (torch.bool, torch.uint8)
    mask = torch.empty(H, W, dtype=torch.float32, device=xs.device)
    scratch = torch.empty(H, W, dtype=torch.float32, device=xs.device)
    check(lib.bde_hot_pixel_mask(ptr(xs), ptr(ys), ptr(ps), xs.numel(), H, W, int(num_hot), ptr(mask), ptr(scratch),
                                 stream_ptr()), "bde_hot_pixel_mask")
    return mask


def pack_voxel_nhwc(vox, c_pad, dtype, out=None):
    """[N, bins, Hp, Wp] float32 planar -> [N, Hp, Wp, c_pad] NHWC of ``dtype``."""
    lib = _lib.require_device()
    N, bins, Hp, Wp = vox.shape
    if out is None:
        out = torch.empty((N, Hp, Wp, c_pad), dtype=dtype, device=vox.device)
    check(lib.bde_pack_voxel_nhwc(ptr(vox), N, bins, Hp, Wp, c_pad, ptr(out), BDE_DTYPE[dtype], stream_ptr()),
          "bde_pack_voxel_nhwc")
    return out


def frame_metrics(pred, gt, y0, x0, data_range):
    """pred float32 [n, Hp, Wp] (padded model output), gt float32 [n, H, W] -> float64 [n, 2] = (mse, ssim) per frame
    of pred[:, y0:y0+H, x0:x0+W] vs gt (evaluate/metrics.py:42-65)."""
    lib = _lib.require_device()
    n, Hp, Wp = pred.shape
    _, H, W = gt.shape
    assert pred.dtype == torch.float32 and gt.dtype == torch.float32 and pred.is_contiguous() and gt.is_contiguous()
    out = torch.zeros(n, 2, dtype=torch.float64, device=pred.device)
    check(lib.bde_frame_metrics(ptr(pred), ptr(gt), n, H, W, Hp, Wp, y0, x0, float(data_range), ptr(out), stream_ptr()),
          "bde_frame_metrics")
    return out


def head_conv(vox, w, bias, out, act=ACT_RELU):
    """float32 planar [N, Cin, H, W] voxels x float32 [32, Cin, 5, 5] weights -> bf16 NHWC [N, H, W, 32]."""
    lib = _lib.require_device()
    N, cin, H, W = vox.shape
    cout, _, k, _ = w.shape
    assert vox.dtype == torch.float32 and w.dtype == torch.float32 and out.dtype == torch.bfloat16
    assert vox.is_contiguous() and w.is_contiguous() and out.is_contiguous()
    check(lib.bde_head_conv(ptr(vox), ptr(w), ptr(bias), ptr(out), N, cin, H, W, cout, k, act, stream_ptr()), "bde_head_conv")
    return out


def gemm(a0, w, bias, out, *, n_img, h_in, w_in, c0, n, ksize=1, stride=1, pad=0, a1=None, c1=0, w_ld=0,
         epi=EPI_STORE, act=ACT_NONE, out_f32=False, residual=None, c_prev=None, c_out=None, row_map=None,
         out2=None, engine=ENGINE_SIMT, dtype=None, k_order=0, ln_frames=None, ln_tok_map=None, ln_n_tok=1,
         res_mode=0, a0_ld=0, a1_ld=0):
    """Implicit-GEMM conv / linear (see bde_gemm in include/bde2vid.h).  Returns (h_out, w_out).
    ``ln_frames`` (list of float32 [*, c0] tensors or None) switches the A operand to the fused
    LayerNorm-gather form (``a0`` is then ignored and may be None)."""
    lib = _lib.require_device()
    d = _lib.GemmDesc()
    d.engine = engine
    d.dtype = BDE_DTYPE[a0.dtype if dtype is None else dtype]
    # a pitched source is a channel slice of a wider NHWC map: not contiguous by construction, only its base matters
    d.a0 = C.c_void_p(a0.data_ptr()) if (a0_ld and a0 is not None) else ptr(a0)
    d.a1 = C.c_void_p(a1.data_ptr()) if (a1_ld and a1 is not None) else ptr(a1)
    if ln_frames is not None:
        d.ln_mode, d.ln_D, d.ln_n_tok = 1, len(ln_frames), ln_n_tok
        for i, f in enumerate(ln_frames):
            d.ln_frames[i] = None if f is None else f.data_ptr()
        d.ln_tok_map = ptr(ln_tok_map)
    d.c0, d.c1 = c0, c1
    d.n_img, d.h_in, d.w_in = n_img, h_in, w_in
    d.h_out = (h_in + 2 * pad - ksize) // stride + 1
    d.w_out = (w_in + 2 * pad - ksize) // stride + 1
    d.ksize, d.stride, d.pad = ksize, stride, pad
    d.w, d.bias, d.n, d.w_ld, d.k_order = ptr(w), ptr(bias), n, w_ld, k_order
    d.epi, d.act, d.out_f32 = epi, act, int(out_f32)
    d.out, d.residual, d.c_prev, d.c_out = ptr(out), ptr(residual), ptr(c_prev), ptr(c_out)
    d.row_map, d.out2, d.res_mode = ptr(row_map), ptr(out2), res_mode
    d.a0_ld, d.a1_ld = a0_ld, a1_ld
    check(lib.bde_gemm(C.byref(d), stream_ptr()), "bde_gemm")
    return d.h_out, d.w_out


def add(a, b, out_f32=None, out_t=None, dtype=torch.float32):
    lib = _lib.require_device()
    n = a.numel()
    assert b.numel() == n
    check(lib.bde_add(ptr(a), int(a.dtype == torch.float32), ptr(b), int(b.dtype == torch.float32), ptr(out_f32),
                      ptr(out_t), n, BDE_DTYPE[dtype], stream_ptr()), "bde_add")


def upsample2x_sum(skip, x, x_scale, n_img, h, w, c, dst):
    lib = _lib.require_device()
    check(lib.bde_upsample2x_sum(ptr(skip), int(skip is not None and skip.dtype == torch.float32), ptr(x),
                                 int(x.dtype == torch.float32), float(x_scale), n_img, h, w, c, ptr(dst),
                                 BDE_DTYPE[dst.dtype], stream_ptr()), "bde_upsample2x_sum")
    return dst


def shuffle2x_sum(g, skip, n_img, h, w, c, dst):
    """dst [n_img, 2h, 2w, c] = phase shuffle of g [n_img, h, w, 4c] (+ skip, same shape as dst); see bde_shuffle2x_sum."""
    lib = _lib.require_device()
    assert g.dtype == dst.dtype and (skip is None or skip.dtype == dst.dtype), "g, skip and dst must share one dtype"
    check(lib.bde_shuffle2x_sum(ptr(g), ptr(skip), n_img, h, w, c, ptr(dst), BDE_DTYPE[dst.dtype], stream_ptr()),
          "bde_shuffle2x_sum")
    return dst


def pred_sigmoid(x, head, wt, bias, c, n_pix, img, wt_head=None, act=ACT_SIGMOID):
    lib = _lib.require_device()
    check(lib.bde_pred_sigmoid(ptr(x), ptr(head), ptr(wt), ptr(wt_head), ptr(bias), c, n_pix, ptr(img), BDE_DTYPE[x.dtype],
                               act, stream_ptr()), "bde_pred_sigmoid")
    return img


def window_reduce(frames, tok_map, n_win, n_tok, c, X, w, b, out):
    """Depthwise whole-window "feature reduction" (nwindow_size) -> float32 [n_win, D, X, c]; see bde_window_reduce."""
    lib = _lib.require_device()
    D = len(frames)
    arr = (C.c_void_p * D)(*[None if f is None else f.data_ptr() for f in frames])
    check(lib.bde_window_reduce(arr, D, ptr(tok_map), n_win, n_tok, c, X, ptr(w), ptr(b), ptr(out), stream_ptr()),
          "bde_window_reduce")
    return out


def ln_gather(frames, tok_map, n_win, n_tok, c, gamma, beta, out):
    """frames: list of float32 [*, c] tensors or None (zero frame)."""
    lib = _lib.require_device()
    D = len(frames)
    arr = (C.c_void_p * D)(*[None if f is None else f.data_ptr() for f in frames])
    check(lib.bde_ln_gather(arr, D, ptr(tok_map), n_win, n_tok, c, ptr(gamma), ptr(beta), ptr(out),
                            BDE_DTYPE[out.dtype], stream_ptr()), "bde_ln_gather")
    return out


def layernorm(x, rows, c, gamma, beta, out):
    lib = _lib.require_device()
    check(lib.bde_layernorm(ptr(x), rows, c, ptr(gamma), ptr(beta), ptr(out), BDE_DTYPE[out.dtype], stream_ptr()),
          "bde_layernorm")
    return out


def window_attention(q, kv, bias_t, n_win, n_q, n_kv, c, heads, out):
    lib = _lib.require_device()
    check(lib.bde_window_attention(ptr(q), ptr(kv), ptr(bias_t), n_win, n_q, n_kv, c, heads, ptr(out),
                                   BDE_DTYPE[out.dtype], stream_ptr()), "bde_window_attention")
    return out


def ln_gather_qkv(frames, q_slot, tok_map, n_win, n_tok, c, g_kv, b_kv, g_q, b_q, out_kv, out_q):
    """Fused window gather + norm_kv (all frames) + norm_q (query slot)."""
    lib = _lib.require_device()
    D = len(frames)
    arr = (C.c_void_p * D)(*[None if f is None else f.data_ptr() for f in frames])
    check(lib.bde_ln_gather_qkv(arr, D, q_slot, ptr(tok_map), n_win, n_tok, c, ptr(g_kv), ptr(b_kv), ptr(g_q), ptr(b_q),
                                ptr(out_kv), ptr(out_q), BDE_DTYPE[out_kv.dtype], stream_ptr()), "bde_ln_gather_qkv")


def attention_mma_bias_stride(n_kv):
    return _lib.load().bde_window_attention_mma_bias_stride(n_kv)


def pad_bias_for_mma(bias_hmn, n_kv):
    """[heads, n_q, n_kv] float32 -> [heads, 64, stride] with -1e30 on the key padding."""
    stride = attention_mma_bias_stride(n_kv)
    if stride == 0:
        return None
    heads, n_q, _ = bias_hmn.shape
    out = torch.zeros(heads, 64, stride, dtype=torch.float32, device=bias_hmn.device)
    out[:, :, n_kv:] = -1e30
    out[:, :n_q, :n_kv] = bias_hmn
    return out.contiguous()


def window_attention_mma(q, kv, bias_padded, n_win, n_q, n_kv, c, heads, out):
    lib = _lib.require_device()
    assert q.dtype == torch.bfloat16
    check(lib.bde_window_attention_mma(ptr(q), ptr(kv), ptr(bias_padded), n_win, n_q, n_kv, c, heads, ptr(out),
                                       stream_ptr()), "bde_window_attention_mma")
    return out


def window_attention_mma_qkv(qkv, bias_padded, n_win, n_q, n_kv, q_row0, c, heads, out):
    lib = _lib.require_device()
    assert qkv.dtype == torch.bfloat16
    check(lib.bde_window_attention_mma_qkv(ptr(qkv), ptr(bias_padded), n_win, n_q, n_kv, q_row0, c, heads, ptr(out),
                                           stream_ptr()), "bde_window_attention_mma_qkv")
    return out


def window_attention_fused_supported(c, heads, n_tok, D):
    return _lib.load().bde_window_attention_fused_supported(c, heads, n_tok, D) == 1


def window_attention_fused(frames, q_slot, tok_map, n_win, c, heads, wqkv, bqkv, bias_tbl, wproj=None, bproj=None,
                           xs=None, o_out=None):
    """Fused gather + LayerNorm + q/k/v + window attention (+ proj + scatter for c == 64); see include/bde2vid.h."""
    lib = _lib.require_device()
    D = len(frames)
    arr = (C.c_void_p * D)(*[None if f is None else f.data_ptr() for f in frames])
    check(lib.bde_window_attention_fused(arr, D, q_slot, ptr(tok_map), n_win, c, heads, ptr(wqkv), ptr(bqkv), ptr(bias_tbl),
                                         ptr(wproj), ptr(bproj), ptr(xs), ptr(o_out), stream_ptr()),
          "bde_window_attention_fused")


def mlp_fused_supported(c, hidden):
    return _lib.load().bde_mlp_fused_supported(c, hidden) == 1


def mlp_fused(x, rows, c, hidden, w1, b1, w2, b2, sum_io=None, sum_t=None):
    """x (float32 [rows, c]) += fc2(GELU(fc1(LayerNorm(x)))) in place; see include/bde2vid.h.  With ``sum_io`` (float32
    [rows, c]) the kernel also does sum_io += x_new and, if given, sum_t = bf16(sum_io)  ("x + merged", ...V5.py:166-169)."""
    lib = _lib.require_device()
    assert x.dtype == torch.float32
    if sum_io is None:
        check(lib.bde_mlp_fused(ptr(x), rows, c, hidden, ptr(w1), ptr(b1), ptr(w2), ptr(b2), stream_ptr()), "bde_mlp_fused")
        return
    assert sum_io.dtype == torch.float32 and (sum_t is None or sum_t.dtype == torch.bfloat16)
    check(lib.bde_mlp_fused_sum(ptr(x), rows, c, hidden, ptr(w1), ptr(b1), ptr(w2), ptr(b2), ptr(sum_io), ptr(sum_t), stream_ptr()),
          "bde_mlp_fused_sum")


def cast(src, dst):
    lib = _lib.require_device()
    check(lib.bde_cast(ptr(src), BDE_DTYPE[src.dtype], ptr(dst), BDE_DTYPE[dst.dtype], src.numel(), stream_ptr()),
          "bde_cast")
    return dst
