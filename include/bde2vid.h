/*
 * bde2vid.h -- C ABI of libbde2vid_sm100.so: hand-written sm_100a kernels for the BDE2VID
 * inference hot path (event voxelisation + bidirectional recurrent conv UNet forward).
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch types.  The reference
 * (gaopinghai/BDE2VID) is pure Python/PyTorch, so "the FFI a maintainer would bind" is a
 * ctypes stub (see INTEGRATION.md); every entry point cites the reference code it replaces.
 *
 * Conventions
 *   - all pointers are DEVICE pointers unless the name ends in _host;
 *   - `stream` is a cudaStream_t passed as void*; every call only enqueues work;
 *   - return value 0 = ok, negative = error (see bde_last_error());
 *   - the library never allocates or frees device memory: callers own every buffer;
 *   - activations are NHWC ("pixels x channels"), element type selected by `dtype`.
 */
#ifndef BDE2VID_H_
#define BDE2VID_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BDE_ABI_VERSION 3

/* element types of activation / weight buffers */
enum { BDE_F32 = 0, BDE_BF16 = 1 };

/* activations applied in GEMM epilogues */
enum { BDE_ACT_NONE = 0, BDE_ACT_RELU = 1, BDE_ACT_RELU6 = 2, BDE_ACT_GELU = 3, BDE_ACT_SIGMOID = 4 };

/* epilogue kinds of bde_gemm */
enum {
  BDE_EPI_STORE = 0,   /* out[m,n] = act(acc + bias[n]) (+ residual[m,n])                       */
  BDE_EPI_LSTM = 1,    /* N = 4*hidden, gate-interleaved rows; ConvLSTM pointwise update         */
  BDE_EPI_SCATTER = 2, /* out_f32[row_map[m], n] += acc + bias[n]   (rows with map < 0 dropped)  */
  /* ConvGRU (model/BDE2VID/submodules.py:337-375, model/e2vid/submodules.py ConvGRU) as two fused convolutions:    */
  BDE_EPI_GRU_UR = 3,  /* N = 2*hidden, rows interleaved n = 2*c + g (g = 0 update_gate, 1 reset_gate):           */
                       /*   c_out[m,c] = u = sigmoid(update)  (fp32);  out[m,c] = h_prev[m,c] * sigmoid(reset)    */
                       /*   (`dtype`; the second source of the out_gate convolution).  h_prev = c_prev (fp32).    */
  BDE_EPI_GRU_OUT = 4  /* N = hidden: o = tanh(acc + bias);  h' = h_prev * (1 - u) + o * u;  h_prev = c_prev     */
                       /*   (fp32, NULL = zeros), u = residual (fp32); c_out = h' (fp32 master), out = h' (`dtype`) */
};

/* GEMM engines */
enum { BDE_ENGINE_SIMT = 0, BDE_ENGINE_TCGEN05 = 1 };

const char* bde_last_error(void);
int bde_abi_version(void);
/* 1 if the device of the current context is compute capability 10.x, else 0 (negative on error) */
int bde_device_ok(void);

/* --------------------------------------------------------------------------------------------
 * Voxeliser.  Replaces events_to_voxel_torch (events_contrast_maximization/utils/event_utils.py
 * :466-509) and its callee events_to_image_torch (:330-376), for a whole sequence in one launch,
 * and the zero padding of Croper.pad (utils_func/inference_utils.py:104-111).
 *
 *   xs, ys, ts, ps : float32[n_events]   loader format (h5_dataset.py:222-225,:414): x,y hold
 *                    integers, ts is relative to the window's first event, ps is +-1
 *   offsets        : int64[T+1]          CSR window boundaries into the event arrays
 *   out            : float32[T, num_bins, Hp, Wp]; the H x W sensor area sits at (pad_top,
 *                    pad_left); every byte of `out` is written (padding = 0)
 *   oob_count      : optional int32[1], incremented for every event outside the sensor (the
 *                    reference raises IndexError from index_put_; such events are dropped here)
 *   algo           : 0 = auto (= 2), 1 = shared-memory row-band tiles + warp aggregation, 2 = memset + global
 *                    RED.ADD.F32 (L2 executes the reductions; 128-bit event loads; windows processed in L2-sized
 *                    chunks), 3 = cluster / distributed-shared-memory grid, 4 = cluster zero + global reductions,
 *                    5 = algorithm 2 with a warp-level pre-reduction of lanes that hit the same cell
 *   min_events     : windows with fewer events produce an all-zero grid.  1 reproduces the bare function
 *                    (dt == 0 gives the reference's NaNs); 3 is the loader contract (h5_dataset.py:219-221:
 *                    `if len(xs) < 3: voxel = zeros`) that the fused events -> frames path must keep.
 */
int bde_voxelize_seq(const float* xs, const float* ys, const float* ts, const float* ps,
                     const int64_t* offsets, int T, int num_bins, int H, int W,
                     int pad_top, int pad_left, int Hp, int Wp,
                     float* out, int* oob_count, int algo, int min_events, void* stream);

/* Same, with `out_window_stride` floats between the grids of consecutive windows (>= bins*Hp*Wp).  Lets B
 * sequences be voxelised straight into one [T, B, bins, Hp, Wp] batch buffer (stride B*bins*Hp*Wp).
 *   hot_mask : optional float32 [H, W] of {0, 1}: the loader's hot-pixel mask (h5_dataset.py:163-172, :364
 *              `voxel_grid * self.hot_events_mask`, the same mask for every bin); events on masked pixels are
 *              dropped (algorithms 2 / 5). */
int bde_voxelize_seq_strided(const float* xs, const float* ys, const float* ts, const float* ps,
                             const int64_t* offsets, int T, int num_bins, int H, int W,
                             int pad_top, int pad_left, int Hp, int Wp,
                             float* out, size_t out_window_stride, int* oob_count, int algo, int min_events,
                             const float* hot_mask, void* stream);

/* Event ingest in the reference's ON-DISK dtypes (events_contrast_maximization/tools/event_packagers.py:44-47:
 * events/xs, ys int16; events/ts float64 seconds; events/ps bool), 13 bytes per event instead of 16.  The loader's
 * conversions (data_loader/h5_dataset.py:204-226, :410-415) happen in registers, bit-exactly:
 *   x, y -> float32;  t -> float32(ts - ts[first event of the window]) (float64 subtraction, then the cast);
 *   p -> ps * 2.0 - 1.0.   `offsets` are the per-frame event_idx windows (h5_dataset.py:448-455) as CSR.
 * Replaces DynamicH5Dataset.__getitem__'s voxelisation on DataLoader workers + the per-window H2D of dense grids
 * (eval_models_seq.py:204).  algo: 0 / 2 / 5 as above. */
int bde_voxelize_raw_strided(const int16_t* xs, const int16_t* ys, const double* ts, const uint8_t* ps,
                             const int64_t* offsets, int T, int num_bins, int H, int W,
                             int pad_top, int pad_left, int Hp, int Wp,
                             float* out, size_t out_window_stride, int* oob_count, int algo, int min_events,
                             const float* hot_mask, void* stream);

/* Voxel normalisation variants of the loader, applied per window on the sensor area of the padded grids, in place
 * (the padding ring stays zero: the reference normalises before Croper.pad).
 *   mode 1 = LegacyNorm (utils_func/data_augmentation.py:311-330): mean / std over the NON-ZERO cells,
 *            x = (x != 0) * (x - mean) / std   (unchanged when there are no non-zero cells or std == 0)
 *   mode 2 = RobustNorm(low_perc, top_perc) (utils_func/utils.py:7-51): t = k-th smallest value with
 *            k = 1 + round(.01 * q * (numel - 1)) (exact order statistic over the bins*H*W cells, radix select);
 *            unchanged when t_max == t_min == 0, else x = (clamp(x, t_min, t_max) - t_min) / (t_max + 1e-6)
 *   grids: float32, window w at grids + w * window_stride, [bins, Hp, Wp] with the sensor at (pad_top, pad_left)
 *   stats: optional float32 [T, 4] receiving (mean, std, count, 0) or (t_min, t_max, 0, 0) per window */
int bde_voxel_normalize(float* grids, size_t window_stride, int T, int num_bins, int H, int W, int pad_top, int pad_left,
                        int Hp, int Wp, int mode, float low_perc, float top_perc, float* stats, void* stream);

/* Hot-pixel mask of the loader (events_contrast_maximization/utils/event_utils.py:100-116 get_hot_event_mask,
 * h5_dataset.py:163-172): accumulate the polarities of the first n events into an image, then clear the num_hot
 * largest pixels one argmax at a time (first index wins ties, as np.argmax).  Event formats as bde_voxelize_raw_strided
 * (ps in {0,1} -> +-1).  mask: float32 [H, W] output of {0, 1};  scratch: float32 [H, W]. */
int bde_hot_pixel_mask(const int16_t* xs, const int16_t* ys, const uint8_t* ps, int64_t n, int H, int W, int num_hot,
                       float* mask, float* scratch, void* stream);

/* Head convolution straight from the voxeliser's planar grid (model/BDE2VID/bde2vid_cross_scale_propogation_V5.py:116,
 * ConvLayer model/BDE2VID/submodules.py:85-114):  out = act(conv5x5(vox) + bias)
 *   vox : float32 [n_img, cin, h, w] planar (cin = num_bins <= 6)    w : float32 [32, cin, 5, 5] (checkpoint layout)
 *   out : bf16 NHWC [n_img, h, w, 32]                                act: BDE_ACT_NONE / RELU / RELU6
 * Operands are rounded to bf16, accumulation is fp32 (mma.sync).  Replaces bde_pack_voxel_nhwc + bde_gemm for the
 * 5-channel first layer, where an im2col gather moves 16 bytes per tap. */
int bde_head_conv(const float* vox, const float* w, const float* bias, void* out, int n_img, int cin, int h, int w_px,
                  int cout, int ksize, int act, void* stream);

/* planar voxel grids float32[T, bins, Hp, Wp] -> NHWC with channels padded to c_pad (zeros),
 * element type `dtype`.  Feeds the head convolution (bde2vid_cross_scale_propogation_V5.py:116). */
int bde_pack_voxel_nhwc(const float* vox, int T, int bins, int Hp, int Wp, int c_pad,
                        void* out, int dtype, void* stream);

/* --------------------------------------------------------------------------------------------
 * Implicit-GEMM convolution / linear layer.
 *
 *   C[m, n] = sum_k A[m, k] * Wp[n, k],   m = (img, oy, ox),  k = (tap, channel)
 *
 * A is gathered on the fly from one or two NHWC sources (two sources = the channel concat of
 * ConvLSTM, model/BDE2VID/submodules.py:316, without materialising it).  Replaces every
 * nn.Conv2d / nn.Linear on the path: ConvLayer (submodules.py:85-114), ConvLSTM.Gates (:317),
 * UpsampleConvLayer.conv2d (:139), predI, and the q/kv/proj/fc1/fc2 Linears of
 * model/BDE2VID/DTransformer.py:188-204,28-36.
 */
typedef struct bde_gemm_desc {
  int engine;            /* BDE_ENGINE_*                                                        */
  int dtype;             /* element type of a0/a1/w and of `out` unless out_f32                  */
  /* A operand */
  const void* a0;        /* NHWC [n_img, h_in, w_in, c0]                                         */
  const void* a1;        /* optional second source [n_img, h_in, w_in, c1] (c1 = 0 -> unused)    */
  int c0, c1;
  int n_img, h_in, w_in, h_out, w_out;
  int ksize, stride, pad;
  /* B operand: packed weights [n, ksize*ksize*(c0+c1)], K-major, k = (ky*ksize+kx)*(c0+c1)+c    */
  const void* w;
  const float* bias;     /* float32[n] (always fp32), may be NULL                                */
  int n;
  int w_ld;              /* row pitch of w in elements (>= K; 0 means K).  The tcgen05 engine    */
                         /* needs w_ld % 64 == 0 with zero padding beyond K.                    */
  int k_order;           /* 0: k = (tap, channel) as above.  1: k = (chunk, tap, channel % 64) with  */
                         /* chunk = channel / 64 (needs c0 % 64 == c1 % 64 == 0): all taps of one    */
                         /* 64-channel slab are consecutive, which lets the tcgen05 engine serve the */
                         /* im2col re-reads of a pixel tile from L1.                                 */
  /* LayerNorm-gather A operand (tcgen05 engine only).  ln_mode = 1: a0 is ignored and                */
  /*   A[m, :] = (x - mean(x)) / sqrt(var(x) + 1e-5),  x = ln_frames[d][ln_tok_map[win*n_tok + tok], :]   */
  /* with m = (win*ln_D + d)*ln_n_tok + tok (float32 rows of c0 channels; NULL frame or map < 0 = zero   */
  /* token, which stays all-zero).  ln_tok_map = NULL means the identity map (plain rows, ln_D = 1).  */
  /* The LayerNorm affine is NOT applied: fold gamma into w and beta into bias (W diag(g), W b + bias).  */
  /* Replaces window_partition + norm_q / norm_kv (DTransformer.py:41-60, 183-184) and norm2 (:281).     */
  int ln_mode;
  int ln_D;
  int ln_n_tok;
  const float* ln_frames[8];
  const int* ln_tok_map;
  /* epilogue */
  int epi;               /* BDE_EPI_*                                                            */
  int act;               /* BDE_ACT_* (STORE only)                                               */
  int out_f32;           /* STORE: write float32 instead of `dtype`                              */
  void* out;             /* STORE: [M, n]; LSTM: h_out [M, hidden] (dtype); SCATTER: f32 [P, n]  */
  const void* residual;  /* STORE: optional [M, n] residual, see res_mode                        */
  const float* c_prev;   /* LSTM: float32 [M, hidden] or NULL (= zeros)                          */
  float* c_out;          /* LSTM: float32 [M, hidden]                                            */
  const int* row_map;    /* SCATTER: int32 [M] destination row or -1                             */
  void* out2;            /* STORE+out_f32: optional second copy of the result in `dtype`         */
  int res_mode;          /* STORE: 0 = `residual` is float32, added AFTER the activation (attention  */
                         /* MLP, DTransformer.py:302-304); 1 = `residual` has element type `dtype`   */
                         /* and is added BEFORE the activation (ResidualBlock,                        */
                         /* model/e2vid/submodules.py:234-247: out = relu(conv2(..) + x))            */
  int a0_ld, a1_ld;      /* pixel pitch of a0 / a1 in elements (0 = c0 / c1): lets a source be a      */
                         /* channel slice of a wider NHWC buffer (the forward / backward encoder convs */
                         /* write one [.., 2C] map, each ConvLSTM chain reads its half).  Only the      */
                         /* TMA convolution kernel of the tcgen05 engine accepts a pitch != c.          */
} bde_gemm_desc;

int bde_gemm(const bde_gemm_desc* desc, void* stream);

/* Per-frame MSE and SSIM of the centre-cropped prediction against the ground truth, on the device
 * (eval_models_seq.py:242-258; evaluate/metrics.py:42-65: F.mse_loss, skimage structural_similarity defaults: 7x7
 * uniform window, K1 = .01, K2 = .03, sample covariance, mean over the valid interior; data_range as given).
 *   pred float32 [n, Hp, Wp] (crop window at (y0, x0), size H x W = Croper.crop)   gt float32 [n, H, W]
 *   out  float64 [n, 2] = (mse, ssim) per frame; accumulated atomically, the caller zeroes it first. */
int bde_frame_metrics(const float* pred, const float* gt, int n, int H, int W, int Hp, int Wp, int y0, int x0,
                      double data_range, double* out, void* stream);

/* Measurement hook: between bde_profile_begin(max) and bde_profile_end every tcgen05 bde_gemm launch is
 * bracketed by a pair of CUDA events on its stream; bde_profile_end returns the summed kernel time (ms)
 * and the number of launches.  Not for use under stream capture. */
int bde_profile_begin(int max_launches);
int bde_profile_end(double* total_ms, int* n_launches);
/* Algorithmic work of the launches profiled since bde_profile_begin: sum of 2 * M * n * ksize^2 * (c0 + c1). */
int bde_profile_flops(double* flops);

/* --------------------------------------------------------------------------------------------
 * Element-wise / gather kernels around the GEMMs.
 */

/* sum = a + b over n elements (bidirectional merge ff + fb, ...V5.py:144; attention residual
 * x + merged, ...V5.py:166).  a / b are float32 when the *_f32 flag is set, else `dtype`.
 * The fp32 sum goes to out_f32 and/or a `dtype` copy to out_t (either may be NULL; in-place ok). */
int bde_add(const void* a, int a_f32, const void* b, int b_f32, float* out_f32, void* out_t, size_t n,
            int dtype, void* stream);

/* dst = bilinear_x2(skip + x)  with align_corners=False (submodules.py:138 fed by skip_sum,
 * ...V5.py:191-194); skip, x: NHWC [n_img, h, w, c] of `dtype`; either may also be float32 when
 * the *_f32 flag is set; dst NHWC [n_img, 2h, 2w, c] of `dtype`.  x_scale multiplies x (Q2: the
 * last level is added to itself -> skip = x, handled by passing skip = NULL, x_scale = 2). */
int bde_upsample2x_sum(const void* skip, int skip_f32, const void* x, int x_f32, float x_scale,
                       int n_img, int h, int w, int c, void* dst, int dtype, void* stream);

/* Pixel shuffle of a stride-2 transposed convolution computed as four stride-1 phase convolutions on the
 * low-resolution map (TransposedConvLayer of model/e2vid/submodules.py, E2VID's use_upsample_conv=False), plus the
 * skip_sum that feeds the next decoder (model/e2vid/unet.py):
 *   dst[b, 2i+py, 2j+px, :] = g[b, i, j, (2py+px)*c : (2py+px+1)*c]  (+ skip[b, 2i+py, 2j+px, :])
 * g NHWC [n_img, h, w, 4c]; skip (NULL = none) and dst NHWC [n_img, 2h, 2w, c]; all three of `dtype`, 16-byte
 * aligned; c % 8 == 0.  A bf16 sum is formed in fp32 and rounded once. */
int bde_shuffle2x_sum(const void* g, const void* skip, int n_img, int h, int w, int c, void* dst, int dtype,
                      void* stream);

/* img[p] = act(bias + sum_c wt[c] * x[p,c] + wt_head[c] * head[p,c])  (predI + output activation, ...V5.py:195-197)
 * x, head NHWC [P, c] of `dtype`; img float32[P].  wt_head = NULL means wt (skip_type 'sum': w . (x + head)); with
 * skip_type 'concat' the two 1x1 convolutions of predI (...V5.py:92-97: fusion 2c -> c, then c -> 1, no activation in
 * between) are folded by the caller into one [2c] vector (wt | wt_head) and one bias.  act: BDE_ACT_SIGMOID or BDE_ACT_NONE
 * (ACTIVATION registry 'Sigmoid' / 'Identity', model/BDE2VID/activaions.py). */
int bde_pred_sigmoid(const void* x, const void* head, const float* wt, const float* wt_head, const float* bias, int c,
                     size_t n_pix, float* img, int dtype, int act, void* stream);

/* "Feature reduction" of WindowAttention3D when nwindow_size is set (DTransformer.py:128-131, 172-175): the depthwise
 * whole-window convolution Conv2d(C, X*C, kernel = window, groups = C) that turns the n_tok tokens of every (window,
 * frame) into X tokens, including the reference's reinterpretation of the [C*X] output vector as [X, C].
 *   frames_host : HOST array of D device pointers float32 [P, c] (NULL = all-zero frame);  tok_map int32 [n_win * n_tok]
 *   w float32 [c*X, n_tok] (reduction_conv.weight [C*X, 1, wh, ww] flattened), b float32 [c*X]
 *   out float32 [n_win, D, X, c]  (kv token index d*X + j', before norm_kv) */
int bde_window_reduce(const float* const* frames_host, int D, const int* tok_map, int n_win, int n_tok, int c, int X,
                      const float* w, const float* b, float* out, void* stream);

/* Window-token gather + LayerNorm (DTransformer.py:41-60 window_partition, :183-184 norm_q/kv).
 *   frames[d]  : float32 NHWC [h*w, c] feature map of buffer slot d, or NULL (= all-zero frame)
 *   tok_map    : int32 [n_win * n_tok] source pixel per window token or -1 (zero token)
 *   out        : `dtype` [n_win, D, n_tok, c]  (kv token index d*n_tok + a*ww + b)
 * Each token (including zero tokens) is normalised over c with (gamma, beta), eps 1e-5. */
int bde_ln_gather(const float* const* frames_host, int D, const int* tok_map, int n_win, int n_tok,
                  int c, const float* gamma, const float* beta, void* out, int dtype, void* stream);

/* Fused form used by the executor: one pass produces the kv tokens of all D frames (norm_kv) and the
 * q tokens of frame `q_slot` (norm_q; same mean / rstd, different affine).  c in {64, 128, 256}.
 *   out_kv : `dtype` [n_win, D, n_tok, c];  out_q : `dtype` [n_win, n_tok, c] */
int bde_ln_gather_qkv(const float* const* frames_host, int D, int q_slot, const int* tok_map, int n_win,
                      int n_tok, int c, const float* g_kv, const float* b_kv, const float* g_q,
                      const float* b_q, void* out_kv, void* out_q, int dtype, void* stream);

/* Row-wise LayerNorm of a float32 [rows, c] matrix -> `dtype` (norm2, DTransformer.py:281). */
int bde_layernorm(const float* x, size_t rows, int c, const float* gamma, const float* beta,
                  void* out, int dtype, void* stream);

/* Window multi-head attention core (DTransformer.py:192-203):
 *   q   : `dtype` [n_win, n_q, c]      (already scaled by head_dim^-0.5)
 *   kv  : `dtype` [n_win, n_kv, 2c]    (k = [..., :c], v = [..., c:])
 *   bias: float32 [heads, n_kv, n_q]   relative-position bias, pre-gathered and transposed
 *   out : `dtype` [n_win, n_q, c]      softmax(q k^T + bias) v, heads concatenated
 */
int bde_window_attention(const void* q, const void* kv, const float* bias, int n_win, int n_q,
                         int n_kv, int c, int heads, void* out, int dtype, void* stream);

/* Tensor-core form of the same op for bf16 (mma.sync m16n8k16, scores kept in registers).
 *   bias_padded: float32 [heads, 64, stride] with stride = bde_window_attention_mma_bias_stride(n_kv),
 *                bias_padded[h, m, n] = bias for n < n_kv, a large negative number (-1e30) for
 *                n_kv <= n < stride (masks the key padding), anything finite for m >= n_q.
 * Supports n_q <= 64, n_kv <= 152, head_dim in {4, 8, 16}, even head count;
 * bde_window_attention_mma_bias_stride returns 0 for an unsupported n_kv. */
int bde_window_attention_mma_bias_stride(int n_kv);
int bde_window_attention_mma(const void* q, const void* kv, const float* bias_padded, int n_win, int n_q,
                             int n_kv, int c, int heads, void* out, void* stream);

/* Same, reading q / k / v from ONE merged projection buffer qkv: bf16 [n_win * n_kv, 3c] whose row
 * w * n_kv + n holds [q | k | v] of kv token n of window w (the fused LayerNorm + qkv GEMM writes it);
 * the n_q query rows of a window start at row q_row0 (= q_slot * n_q) inside the window. */
int bde_window_attention_mma_qkv(const void* qkv, const float* bias_padded, int n_win, int n_q, int n_kv,
                                 int q_row0, int c, int heads, void* out, void* stream);

/* Fused attention half of one SwinTransformerBlock3D (DTransformer.py:254-299): window gather through
 * tok_map (plain or dilated windows, -1 = zero-padding token) + norm_q / norm_kv + q / kv Linear +
 * softmax(q k^T + relative-position bias) v, all inside one kernel (q, k, v stay in shared memory).
 *   frames_host : HOST array of D device pointers, float32 [P, c] per buffered frame (NULL = all-zero
 *                 frame, ...V5.py:160-161); frames_host[q_slot] is the running x of the block
 *   tok_map     : int32 [n_win * 49]
 *   wqkv, bqkv  : bf16 [3c, c] / float32 [3c]: rows q | k | v with the LayerNorm affine and the q scale
 *                 folded in (W diag(gamma), W beta + b), as for bde_gemm's ln_mode
 *   bias_tbl    : float32 [heads, D, 169]: bias_tbl[h, d, (aq-ak+6)*13 + (bq-bk+6)] =
 *                 relative_position_bias_table[((q_slot - d) + D - 1)*169 + ..., h]  (DTransformer.py:139-152,195-199)
 *   c == 64 : wproj bf16 [c, c], bproj float32 [c]; xs float32 [P, c] (= frames_host[q_slot]) receives
 *             xs[pix] += proj(attn)[token] + bproj for every covered pixel (window_reverse + crop + shortcut)
 *   c == 256: o_out bf16 [n_win * 49, c] receives the attention output (heads concatenated); the caller
 *             runs proj as a bde_gemm with BDE_EPI_SCATTER.  With wproj, bproj and xs given instead, the
 *             projection is fused as for c == 64 (one whole-window tcgen05 kernel); wqkv and wproj must then
 *             be 128-byte aligned (the call fails otherwise)
 * Supported: 7x7 windows, D <= 3, (c, heads) with c in {64, 256} and head_dim = c / 64 * 4 (4 or 16);
 * bde_window_attention_fused_supported returns 1 for a supported shape. */
int bde_window_attention_fused_supported(int c, int heads, int n_tok, int D);
int bde_window_attention_fused(const float* const* frames_host, int D, int q_slot, const int* tok_map, int n_win,
                               int c, int heads, const void* wqkv, const float* bqkv, const float* bias_tbl,
                               const void* wproj, const float* bproj, float* xs, void* o_out, void* stream);

/* Fused MLP half of a SwinTransformerBlock3D (DTransformer.py:279-283,302-304), in place on the fp32
 * residual stream:  x[m, :] += fc2(GELU(fc1(LayerNorm(x[m, :]))))   for x float32 [rows, c].
 *   w1, b1 : bf16 [hidden, c] / float32 [hidden] with norm2's affine folded in (W diag(gamma), W beta + b)
 *   w2, b2 : bf16 [c, hidden] / float32 [c]
 * Both GEMMs run on tcgen05; the hidden activation stays in shared memory.  Implemented for c = 64,
 * hidden = 256 (bde_mlp_fused_supported); other shapes use two bde_gemm calls (ln_mode + GELU, residual). */
int bde_mlp_fused_supported(int c, int hidden);
int bde_mlp_fused(float* x, size_t rows, int c, int hidden, const void* w1, const float* b1, const void* w2,
                  const float* b2, void* stream);
/* Same, and additionally (after the last block of a frame, ..._V5.py:166-169 "x + merged"): sum_io[m] += x_new[m]
 * (float32 [rows, c], in place) and, when sum_t != NULL, sum_t[m] = bf16(sum_io[m]). */
int bde_mlp_fused_sum(float* x, size_t rows, int c, int hidden, const void* w1, const float* b1, const void* w2,
                      const float* b2, float* sum_io, void* sum_t, void* stream);

/* float32 -> dtype copy/cast (and back); n elements */
int bde_cast(const void* src, int src_dtype, void* dst, int dst_dtype, size_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BDE2VID_H_ */
