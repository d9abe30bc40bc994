// Bandwidth-bound kernels around the GEMMs: bidirectional merge, bilinear x2 + skip sum,
// prediction head, window-token gather + LayerNorm, row LayerNorm, casts.
#include "common.cuh"

namespace bde {

// ---------------------------------------------------------------------------------------------
// out = a + b   (ff + fb, bde2vid_cross_scale_propogation_V5.py:144)
// ---------------------------------------------------------------------------------------------
template <typename T, typename TA, typename TB>
__global__ void add_kernel(const TA* a, const TB* b, float* out_f32, T* out_t, size_t n4) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n4) return;
  float4 x = load4<TA>(a + i * 4), y = load4<TB>(b + i * 4);
  float4 s = make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
  if (out_f32 != nullptr) store4<float>(out_f32 + i * 4, s);
  if (out_t != nullptr) store4<T>(out_t + i * 4, s);
}

// ---------------------------------------------------------------------------------------------
// dst = bilinear_x2(skip + x_scale * x), align_corners=False (submodules.py:138; SURVEY A.6):
//   out[2i]   = .25*in[max(i-1,0)] + .75*in[i]
//   out[2i+1] = .75*in[i]          + .25*in[min(i+1,n-1)]
// F.interpolate computes source index (dst+0.5)/2-0.5 clamped at 0, lambda from it; the weights
// above are the exact values of that formula for scale 2.
// ---------------------------------------------------------------------------------------------
template <typename T, typename TS, typename TX>
__global__ void upsample2x_sum_kernel(const TS* __restrict__ skip, const TX* __restrict__ x, float x_scale,
                                      int h, int w, int c4, T* __restrict__ dst, size_t total) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // over n_img * 2h * 2w * c4
  if (i >= total) return;
  int cq = (int)(i % c4);
  size_t pix = i / c4;
  int ox = (int)(pix % (2 * w));
  size_t r = pix / (2 * w);
  int oy = (int)(r % (2 * h));
  size_t img = r / (2 * h);
  // source taps
  int y0, y1, x0, x1;
  float wy0, wy1, wx0, wx1;
  if (oy & 1) { y0 = oy >> 1; y1 = min(y0 + 1, h - 1); wy0 = 0.75f; wy1 = 0.25f; }
  else        { y1 = oy >> 1; y0 = max(y1 - 1, 0);     wy0 = 0.25f; wy1 = 0.75f; }
  if (ox & 1) { x0 = ox >> 1; x1 = min(x0 + 1, w - 1); wx0 = 0.75f; wx1 = 0.25f; }
  else        { x1 = ox >> 1; x0 = max(x1 - 1, 0);     wx0 = 0.25f; wx1 = 0.75f; }
  auto fetch = [&](int yy, int xx) {
    size_t o = (((size_t)img * h + yy) * w + xx) * (size_t)(c4 * 4) + cq * 4;
    float4 v = load4<TX>(x + o);
    v.x *= x_scale; v.y *= x_scale; v.z *= x_scale; v.w *= x_scale;
    if (skip != nullptr) {
      float4 s = load4<TS>(skip + o);
      v.x += s.x; v.y += s.y; v.z += s.z; v.w += s.w;
    }
    return v;
  };
  float4 a = fetch(y0, x0), b = fetch(y0, x1), cc = fetch(y1, x0), d = fetch(y1, x1);
  // torch: horizontal lerp inside vertical lerp: w_y0*(w_x0*a + w_x1*b) + w_y1*(w_x0*c + w_x1*d)
  float4 o;
  o.x = wy0 * (wx0 * a.x + wx1 * b.x) + wy1 * (wx0 * cc.x + wx1 * d.x);
  o.y = wy0 * (wx0 * a.y + wx1 * b.y) + wy1 * (wx0 * cc.y + wx1 * d.y);
  o.z = wy0 * (wx0 * a.z + wx1 * b.z) + wy1 * (wx0 * cc.z + wx1 * d.z);
  o.w = wy0 * (wx0 * a.w + wx1 * b.w) + wy1 * (wx0 * cc.w + wx1 * d.w);
  store4<T>(dst + pix * (size_t)(c4 * 4) + cq * 4, o);
}


// Faster form for bf16 outputs with c % 8 == 0: one thread per INPUT pixel and 8 channels produces the 2 x 2 output
// pixels it maps to from its 3 x 3 neighbourhood (2.25 source reads per output instead of 4, 16-byte loads / stores,
// 32-bit index math from the block coordinates).  Same arithmetic order as the kernel above.
template <typename TV>
__device__ __forceinline__ void load8f(const TV* p, float (&v)[8]);
template <>
__device__ __forceinline__ void load8f<float>(const float* p, float (&v)[8]) {
  const float4 a = *reinterpret_cast<const float4*>(p), b = *reinterpret_cast<const float4*>(p + 4);
  v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
template <>
__device__ __forceinline__ void load8f<__nv_bfloat16>(const __nv_bfloat16* p, float (&v)[8]) {
  const uint4 r = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}

// Thread = (input column, 8 channels); the block walks kUpRows input rows with a ROLLING window of three summed rows
// (x * scale + skip, columns prev / this / next) in registers: 6 vector loads per input row instead of the 18 of the
// one-row-per-thread form, which re-fetched and re-summed the whole 3 x 3 neighbourhood for every input pixel.
constexpr int kUpRows = 8;
template <typename TS, typename TX>
__global__ void __launch_bounds__(256) upsample2x_sum_block_kernel(const TS* __restrict__ skip, const TX* __restrict__ x, float x_scale,
                                                                     int h, int w, int c8, __nv_bfloat16* __restrict__ dst) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // over w * c8 of one input row
  if (idx >= w * c8) return;
  const int ix = idx / c8, cq = idx - ix * c8;
  const int iy0 = blockIdx.y * kUpRows, img = blockIdx.z;
  const int iy1 = min(iy0 + kUpRows, h);
  const int c = c8 * 8;
  const int xs[3] = {max(ix - 1, 0), ix, min(ix + 1, w - 1)};   // source columns (prev, this, next), clamped
  auto load_row = [&](int r, float (&row)[3][8]) {
    r = min(max(r, 0), h - 1);
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      const size_t o = (((size_t)img * h + r) * w + xs[b]) * (size_t)c + cq * 8;
      load8f<TX>(x + o, row[b]);
#pragma unroll
      for (int e = 0; e < 8; ++e) row[b][e] *= x_scale;
      if (skip != nullptr) {
        float sk[8];
        load8f<TS>(skip + o, sk);
#pragma unroll
        for (int e = 0; e < 8; ++e) row[b][e] += sk[e];
      }
    }
  };
  float v[3][3][8];   // rows (prev, this, next) x columns (prev, this, next)
  load_row(iy0 - 1, v[0]);
  load_row(iy0, v[1]);
  for (int iy = iy0; iy < iy1; ++iy) {
    load_row(iy + 1, v[2]);
    // output (2 iy + dy, 2 ix + dx): dy = 0 -> rows (prev .25, this .75); dy = 1 -> rows (this .75, next .25); same for columns
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int y0 = dy, y1 = dy + 1, x0 = dx, x1 = dx + 1;   // indices into the 3 x 3 neighbourhood
        const float wy0 = dy ? 0.75f : 0.25f, wy1 = dy ? 0.25f : 0.75f;
        const float wx0 = dx ? 0.75f : 0.25f, wx1 = dx ? 0.25f : 0.75f;
        float o[8];
#pragma unroll
        for (int e = 0; e < 8; ++e)
          o[e] = wy0 * (wx0 * v[y0][x0][e] + wx1 * v[y0][x1][e]) + wy1 * (wx0 * v[y1][x0][e] + wx1 * v[y1][x1][e]);
        uint4 pk;
        __nv_bfloat162 t0 = __floats2bfloat162_rn(o[0], o[1]), t1 = __floats2bfloat162_rn(o[2], o[3]);
        __nv_bfloat162 t2 = __floats2bfloat162_rn(o[4], o[5]), t3 = __floats2bfloat162_rn(o[6], o[7]);
        pk.x = *reinterpret_cast<uint32_t*>(&t0); pk.y = *reinterpret_cast<uint32_t*>(&t1);
        pk.z = *reinterpret_cast<uint32_t*>(&t2); pk.w = *reinterpret_cast<uint32_t*>(&t3);
        const size_t op = (((size_t)img * 2 * h + (2 * iy + dy)) * (2 * w) + (2 * ix + dx)) * (size_t)c + cq * 8;
        *reinterpret_cast<uint4*>(dst + op) = pk;
      }
#pragma unroll
    for (int b = 0; b < 3; ++b)
#pragma unroll
      for (int e = 0; e < 8; ++e) { v[0][b][e] = v[1][b][e]; v[1][b][e] = v[2][b][e]; }
  }
}

// ---------------------------------------------------------------------------------------------
// Pixel shuffle of a stride-2 transposed convolution run as four phase convolutions on the low-resolution map
// (TransposedConvLayer, model/e2vid/submodules.py), plus the skip that feeds the next decoder (skip_sum, unet.py):
//   dst[b, 2i+py, 2j+px, :] = g[b, i, j, (2py+px)*c : (2py+px+1)*c]  (+ skip[b, 2i+py, 2j+px, :])
// Thread = one 16-byte vector of a destination row, so every row is stored coalesced; blockIdx.y walks the rows.
// The bf16 sum is formed in fp32 and rounded once, as torch's bf16 add does.
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ uint4 add16(uint4 a, uint4 b);
template <>
__device__ __forceinline__ uint4 add16<float>(uint4 a, uint4 b) {
  const float4 x = *reinterpret_cast<const float4*>(&a), y = *reinterpret_cast<const float4*>(&b);
  const float4 s = make_float4(x.x + y.x, x.y + y.y, x.z + y.z, x.w + y.w);
  return *reinterpret_cast<const uint4*>(&s);
}
template <>
__device__ __forceinline__ uint4 add16<__nv_bfloat16>(uint4 a, uint4 b) {
  const uint32_t x[4] = {a.x, a.y, a.z, a.w}, y[4] = {b.x, b.y, b.z, b.w};
  uint32_t r[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 p = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&x[i]));
    const float2 q = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&y[i]));
    const __nv_bfloat162 s = __floats2bfloat162_rn(p.x + q.x, p.y + q.y);
    r[i] = *reinterpret_cast<const uint32_t*>(&s);
  }
  return make_uint4(r[0], r[1], r[2], r[3]);
}

template <typename T>
__global__ void __launch_bounds__(256) shuffle2x_sum_kernel(const T* __restrict__ g, const T* __restrict__ skip, int h, int w,
                                                            int cv, int rows, T* __restrict__ dst) {
  constexpr int V = 16 / sizeof(T);                          // elements per vector
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;     // over the 2w * cv vectors of one destination row
  if (idx >= 2 * w * cv) return;
  const int ox = idx / cv, q = idx - ox * cv;
  const int c = cv * V;
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {       // r = img * 2h + oy
    const int img = r / (2 * h), oy = r - img * 2 * h;
    const size_t src = (((size_t)img * h + (oy >> 1)) * w + (ox >> 1)) * (size_t)(4 * c) +
                       (size_t)(((oy & 1) * 2 + (ox & 1)) * c + q * V);
    const size_t o = (size_t)r * (size_t)(2 * w) * c + (size_t)idx * V;
    uint4 v = __ldg(reinterpret_cast<const uint4*>(g + src));
    if (skip != nullptr) v = add16<T>(v, __ldg(reinterpret_cast<const uint4*>(skip + o)));
    *reinterpret_cast<uint4*>(dst + o) = v;
  }
}

// ---------------------------------------------------------------------------------------------
// img = sigmoid(bias + wt . (x + head))   (predI 1x1 conv + Sigmoid, ...V5.py:195-197)
// one thread per pixel; c <= 256, multiple of 4
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void pred_sigmoid_kernel(const T* __restrict__ x, const T* __restrict__ head,
                                    const float* __restrict__ wt, const float* __restrict__ wt_head,
                                    const float* __restrict__ bias, int c, size_t n_pix, float* __restrict__ img, int act) {
  extern __shared__ float sw[];   // [2][c]: weights of x, weights of head
  for (int i = threadIdx.x; i < c; i += blockDim.x) {
    sw[i] = wt[i];
    sw[c + i] = wt_head != nullptr ? wt_head[i] : wt[i];
  }
  __syncthreads();
  size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n_pix) return;
  float acc = bias[0];
  const T* xp = x + p * c;
  const T* hp = head + p * c;
  if (wt_head == nullptr) {       // skip_sum: w . (x + head), the reference's order
    for (int k = 0; k < c; k += 4) {
      float4 a = load4<T>(xp + k), b = load4<T>(hp + k);
      acc = fmaf(sw[k + 0], a.x + b.x, acc);
      acc = fmaf(sw[k + 1], a.y + b.y, acc);
      acc = fmaf(sw[k + 2], a.z + b.z, acc);
      acc = fmaf(sw[k + 3], a.w + b.w, acc);
    }
  } else {                        // skip_concat: the two 1x1 convolutions folded into one [2c] vector
    for (int k = 0; k < c; k += 4) {
      float4 a = load4<T>(xp + k), b = load4<T>(hp + k);
      acc = fmaf(sw[k + 0], a.x, acc); acc = fmaf(sw[c + k + 0], b.x, acc);
      acc = fmaf(sw[k + 1], a.y, acc); acc = fmaf(sw[c + k + 1], b.y, acc);
      acc = fmaf(sw[k + 2], a.z, acc); acc = fmaf(sw[c + k + 2], b.z, acc);
      acc = fmaf(sw[k + 3], a.w, acc); acc = fmaf(sw[c + k + 3], b.w, acc);
    }
  }
  img[p] = act == BDE_ACT_SIGMOID ? sigmoid_f(acc) : acc;
}

// ---------------------------------------------------------------------------------------------
// Window "feature reduction" of WindowAttention3D with nwin_size set (DTransformer.py:128-131, 172-175): a depthwise
// convolution whose kernel covers the whole window, Conv2d(C, X*C, kernel = window, groups = C), turns the n_tok tokens of
// a (frame, window) into X = nwin0 * nwin1 tokens.  The reference then VIEWS the [C*X] output vector (index o = c*X + j)
// as [X, C] (index j'*C + c'), which this kernel reproduces: out[(win*D + d)*X + j', c'] = conv[o = j'*C + c'],
// conv[o] = b[o] + sum_tok w[o, tok] * x[d, win, tok, o / X].   One warp per (win, d, j'); zero tokens contribute 0.
// ---------------------------------------------------------------------------------------------
struct FramePtrs8 {
  const float* f[8];
};
__global__ void __launch_bounds__(256) window_reduce_kernel(FramePtrs8 frames, int D, const int* __restrict__ tok_map, int n_tok, int c,
                                                            int X, const float* __restrict__ w, const float* __restrict__ b,
                                                            float* __restrict__ out, size_t total_rows) {
  const size_t row = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // (win, d, j')
  const int lane = threadIdx.x & 31;
  if (row >= total_rows) return;
  const int jp = (int)(row % X);
  const size_t wd = row / X;
  const int d = (int)(wd % D);
  const size_t win = wd / D;
  const float* fr = frames.f[d];
  const int* tm = tok_map + win * n_tok;
  for (int cp = lane; cp < c; cp += 32) {
    const int o = jp * c + cp;
    const int ch = o / X;
    float acc = b != nullptr ? b[o] : 0.f;
    if (fr != nullptr) {
      const float* wo = w + (size_t)o * n_tok;
      for (int t = 0; t < n_tok; ++t) {
        const int src = tm[t];
        if (src >= 0) acc = fmaf(wo[t], fr[(size_t)src * c + ch], acc);
      }
    }
    out[row * c + cp] = acc;
  }
}

// ---------------------------------------------------------------------------------------------
// LayerNorm helpers: one warp per row of c <= 1024 channels (c % 32 == 0 not required)
// ---------------------------------------------------------------------------------------------
constexpr int kMaxPerLane = 32;  // c <= 1024

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T>
__device__ __forceinline__ void ln_row(const float* __restrict__ src /* may be nullptr = zeros */, int c,
                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                       T* __restrict__ dst, int lane) {
  float v[kMaxPerLane];
  int cnt = 0;
  float s = 0.f;
  for (int k = lane; k < c; k += 32, ++cnt) {
    v[cnt] = src != nullptr ? src[k] : 0.f;
    s += v[cnt];
  }
  float mean = warp_sum(s) / (float)c;
  float q = 0.f;
  for (int i = 0; i < cnt; ++i) {
    float d = v[i] - mean;
    q += d * d;
  }
  float var = warp_sum(q) / (float)c;
  float rstd = 1.0f / sqrtf(var + 1e-5f);
  int i = 0;
  for (int k = lane; k < c; k += 32, ++i) dst[k] = from_f32<T>((v[i] - mean) * rstd * gamma[k] + beta[k]);
}

struct FramePtrs {
  const float* f[8];
};

// window_partition (DTransformer.py:41-60) + norm_q / norm_kv (:183-184)
template <typename T>
__global__ void ln_gather_kernel(FramePtrs frames, int D, const int* __restrict__ tok_map, int n_tok, int c,
                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                 T* __restrict__ out, size_t total_rows) {
  size_t row = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // (win, d, tok)
  int lane = threadIdx.x & 31;
  if (row >= total_rows) return;
  int tok = (int)(row % n_tok);
  size_t r = row / n_tok;
  int d = (int)(r % D);
  size_t win = r / D;
  int pix = tok_map[win * n_tok + tok];
  const float* fr = frames.f[d];
  const float* src = (fr != nullptr && pix >= 0) ? fr + (size_t)pix * c : nullptr;
  ln_row<T>(src, c, gamma, beta, out + row * c, lane);
}

// Fused q + kv variant: norm_q and norm_kv of the query frame share mean / rstd, so one pass over the
// window tokens writes the kv tokens of every frame and, for the query slot, the q tokens as well.
// Vectorised: each lane owns 8 consecutive channels, LPT = C / 8 lanes cooperate on one token and a
// warp handles 32 / LPT tokens at once (C = 64 -> 4 tokens per warp), which keeps 4x more
// independent loads in flight per warp than the one-token-per-warp form.
template <int LPT>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int o = LPT / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T, int LPT>
__global__ void __launch_bounds__(256) ln_gather_qkv_kernel(
    FramePtrs frames, int D, int q_slot, const int* __restrict__ tok_map, int n_tok,
    const float* __restrict__ g_kv, const float* __restrict__ b_kv, const float* __restrict__ g_q,
    const float* __restrict__ b_q, T* __restrict__ out_kv, T* __restrict__ out_q, size_t total_rows) {
  constexpr int C = 8 * LPT;
  constexpr int TPW = 32 / LPT;  // tokens per warp
  const int lane = threadIdx.x & 31;
  const int sub = lane / LPT, ll = lane % LPT;
  const size_t warp_id = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const size_t row = warp_id * TPW + sub;  // (win, d, tok)
  const bool live = row < total_rows;
  int d = 0;
  size_t wt = 0;  // win * n_tok + tok
  const float* src = nullptr;
  if (live) {
    const int tok = (int)(row % n_tok);
    const size_t r = row / n_tok;
    d = (int)(r % D);
    const size_t win = r / D;
    wt = win * n_tok + tok;
    const int pix = tok_map != nullptr ? __ldg(tok_map + wt) : (int)wt;  // nullptr = identity (plain rows)
    const float* fr = frames.f[0];
#pragma unroll
    for (int i = 1; i < 8; ++i) fr = (d == i) ? frames.f[i] : fr;  // no dynamic indexing of the by-value struct
    if (fr != nullptr && pix >= 0) src = fr + (size_t)pix * C + ll * 8;
  }
  float v[8];
  if (src != nullptr) {
    const float4 t0 = *reinterpret_cast<const float4*>(src), t1 = *reinterpret_cast<const float4*>(src + 4);
    v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
  } else {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) s += v[i];
  const float mean = group_sum<LPT>(s) / (float)C;
  float qq = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    v[i] -= mean;
    qq += v[i] * v[i];
  }
  const float rstd = 1.0f / sqrtf(group_sum<LPT>(qq) / (float)C + 1e-5f);
  if (!live) return;
  auto emit = [&](const float* gm, const float* bt, T* dst) {
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(gm + ll * 8)), g1 = __ldg(reinterpret_cast<const float4*>(gm + ll * 8 + 4));
    const float4 c0 = __ldg(reinterpret_cast<const float4*>(bt + ll * 8)), c1 = __ldg(reinterpret_cast<const float4*>(bt + ll * 8 + 4));
    store4<T>(dst, make_float4(v[0] * rstd * g0.x + c0.x, v[1] * rstd * g0.y + c0.y, v[2] * rstd * g0.z + c0.z,
                               v[3] * rstd * g0.w + c0.w));
    store4<T>(dst + 4, make_float4(v[4] * rstd * g1.x + c1.x, v[5] * rstd * g1.y + c1.y, v[6] * rstd * g1.z + c1.z,
                                   v[7] * rstd * g1.w + c1.w));
  };
  emit(g_kv, b_kv, out_kv + row * C + ll * 8);
  if (d == q_slot && out_q != nullptr) emit(g_q, b_q, out_q + wt * (size_t)C + ll * 8);
}

template <typename T>
__global__ void layernorm_kernel(const float* __restrict__ x, size_t rows, int c, const float* __restrict__ gamma,
                                 const float* __restrict__ beta, T* __restrict__ out) {
  size_t row = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  ln_row<T>(x + row * c, c, gamma, beta, out + row * c, lane);
}

template <typename TS, typename TD>
__global__ void cast_kernel(const TS* __restrict__ src, TD* __restrict__ dst, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = from_f32<TD>(to_f32<TS>(src[i]));
}

}  // namespace bde

using namespace bde;

template <typename T>
static int launch_add(const void* a, int a_f32, const void* b, int b_f32, float* out_f32, void* out_t, size_t n4,
                      cudaStream_t s) {
  unsigned blocks = (unsigned)ceil_div(n4, 256);
  if (a_f32 && b_f32)
    add_kernel<T, float, float><<<blocks, 256, 0, s>>>((const float*)a, (const float*)b, out_f32, (T*)out_t, n4);
  else if (a_f32 && !b_f32)
    add_kernel<T, float, T><<<blocks, 256, 0, s>>>((const float*)a, (const T*)b, out_f32, (T*)out_t, n4);
  else if (!a_f32 && b_f32)
    add_kernel<T, T, float><<<blocks, 256, 0, s>>>((const T*)a, (const float*)b, out_f32, (T*)out_t, n4);
  else
    add_kernel<T, T, T><<<blocks, 256, 0, s>>>((const T*)a, (const T*)b, out_f32, (T*)out_t, n4);
  return check_launch("add_kernel");
}

extern "C" int bde_add(const void* a, int a_f32, const void* b, int b_f32, float* out_f32, void* out_t, size_t n,
                       int dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(n % 4 == 0, "bde_add: n must be a multiple of 4");
  BDE_REQUIRE(a != nullptr && b != nullptr, "bde_add: null input");
  if (n == 0) return 0;
  if (dtype == BDE_F32) return launch_add<float>(a, 1, b, 1, out_f32, out_t, n / 4, s);
  return launch_add<__nv_bfloat16>(a, a_f32, b, b_f32, out_f32, out_t, n / 4, s);
}

template <typename T>
static int launch_upsample(const void* skip, int skip_f32, const void* x, int x_f32, float x_scale, int n_img, int h,
                           int w, int c, void* dst, cudaStream_t s) {
  size_t total = (size_t)n_img * 2 * h * 2 * w * (c / 4);
  unsigned blocks = (unsigned)ceil_div(total, 256);
  T* d = (T*)dst;
  if (sizeof(T) == 2 && c % 8 == 0 && h <= 65535 && n_img <= 65535) {
    // block form (bf16 output): thread = input pixel x 8 channels
    dim3 grid((unsigned)ceil_div((size_t)w * (c / 8), 256), (unsigned)ceil_div(h, kUpRows), (unsigned)n_img);
    __nv_bfloat16* db = (__nv_bfloat16*)dst;
    if (skip_f32 && x_f32)
      upsample2x_sum_block_kernel<float, float><<<grid, 256, 0, s>>>((const float*)skip, (const float*)x, x_scale, h, w, c / 8, db);
    else if (skip_f32 && !x_f32)
      upsample2x_sum_block_kernel<float, __nv_bfloat16><<<grid, 256, 0, s>>>((const float*)skip, (const __nv_bfloat16*)x, x_scale, h, w, c / 8, db);
    else if (!skip_f32 && x_f32)
      upsample2x_sum_block_kernel<__nv_bfloat16, float><<<grid, 256, 0, s>>>((const __nv_bfloat16*)skip, (const float*)x, x_scale, h, w, c / 8, db);
    else
      upsample2x_sum_block_kernel<__nv_bfloat16, __nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)skip, (const __nv_bfloat16*)x, x_scale, h, w, c / 8, db);
    return check_launch("upsample2x_sum_block_kernel");
  }
  if (skip_f32 && x_f32)
    upsample2x_sum_kernel<T, float, float><<<blocks, 256, 0, s>>>((const float*)skip, (const float*)x, x_scale, h, w, c / 4, d, total);
  else if (skip_f32 && !x_f32)
    upsample2x_sum_kernel<T, float, T><<<blocks, 256, 0, s>>>((const float*)skip, (const T*)x, x_scale, h, w, c / 4, d, total);
  else if (!skip_f32 && x_f32)
    upsample2x_sum_kernel<T, T, float><<<blocks, 256, 0, s>>>((const T*)skip, (const float*)x, x_scale, h, w, c / 4, d, total);
  else
    upsample2x_sum_kernel<T, T, T><<<blocks, 256, 0, s>>>((const T*)skip, (const T*)x, x_scale, h, w, c / 4, d, total);
  return check_launch("upsample2x_sum_kernel");
}

extern "C" int bde_upsample2x_sum(const void* skip, int skip_f32, const void* x, int x_f32, float x_scale, int n_img,
                                  int h, int w, int c, void* dst, int dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(c % 4 == 0, "bde_upsample2x_sum: c must be a multiple of 4");
  BDE_REQUIRE(x != nullptr && dst != nullptr, "bde_upsample2x_sum: null pointer");
  if (n_img == 0) return 0;
  if (dtype == BDE_F32) return launch_upsample<float>(skip, 1, x, 1, x_scale, n_img, h, w, c, dst, s);
  return launch_upsample<__nv_bfloat16>(skip, skip_f32, x, x_f32, x_scale, n_img, h, w, c, dst, s);
}

extern "C" int bde_shuffle2x_sum(const void* g, const void* skip, int n_img, int h, int w, int c, void* dst, int dtype,
                                 void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(g != nullptr && dst != nullptr, "bde_shuffle2x_sum: null pointer");
  BDE_REQUIRE(c > 0 && c % 8 == 0, "bde_shuffle2x_sum: c must be a positive multiple of 8 (got %d)", c);
  BDE_REQUIRE(n_img >= 0 && h >= 0 && w >= 0, "bde_shuffle2x_sum: bad sizes");
  BDE_REQUIRE(dtype == BDE_F32 || dtype == BDE_BF16, "bde_shuffle2x_sum: bad dtype %d", dtype);
  BDE_REQUIRE(((uintptr_t)g | (uintptr_t)skip | (uintptr_t)dst) % 16 == 0, "bde_shuffle2x_sum: buffers must be 16-byte aligned");
  const size_t rows = (size_t)n_img * 2 * h;
  BDE_REQUIRE(rows < ((size_t)1 << 31) && (size_t)2 * w * c < ((size_t)1 << 31), "bde_shuffle2x_sum: map too large");
  if (rows == 0 || w == 0) return 0;
  const int esize = dtype == BDE_F32 ? 4 : 2;
  const int cv = c * esize / 16;
  const dim3 grid((unsigned)ceil_div((size_t)2 * w * cv, 256), (unsigned)(rows < 65535 ? rows : 65535));
  if (dtype == BDE_F32)
    shuffle2x_sum_kernel<float><<<grid, 256, 0, s>>>((const float*)g, (const float*)skip, h, w, cv, (int)rows, (float*)dst);
  else
    shuffle2x_sum_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>((const __nv_bfloat16*)g, (const __nv_bfloat16*)skip, h, w, cv,
                                                             (int)rows, (__nv_bfloat16*)dst);
  return check_launch("shuffle2x_sum_kernel");
}

extern "C" int bde_pred_sigmoid(const void* x, const void* head, const float* wt, const float* wt_head, const float* bias, int c,
                                size_t n_pix, float* img, int dtype, int act, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(c % 4 == 0 && c <= 4096, "bde_pred_sigmoid: bad channel count");
  BDE_REQUIRE(act == BDE_ACT_SIGMOID || act == BDE_ACT_NONE, "bde_pred_sigmoid: activation must be SIGMOID or NONE");
  if (n_pix == 0) return 0;
  unsigned blocks = (unsigned)ceil_div(n_pix, 128);
  const size_t smem = (size_t)2 * c * sizeof(float);
  if (dtype == BDE_F32)
    pred_sigmoid_kernel<float><<<blocks, 128, smem, s>>>((const float*)x, (const float*)head, wt, wt_head, bias, c, n_pix, img, act);
  else
    pred_sigmoid_kernel<__nv_bfloat16><<<blocks, 128, smem, s>>>((const __nv_bfloat16*)x, (const __nv_bfloat16*)head, wt, wt_head, bias, c, n_pix, img, act);
  return check_launch("pred_sigmoid_kernel");
}

extern "C" int bde_window_reduce(const float* const* frames_host, int D, const int* tok_map, int n_win, int n_tok, int c, int X,
                                 const float* w, const float* b, float* out, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(D >= 1 && D <= 8 && X >= 1 && c >= 1 && n_tok >= 1, "bde_window_reduce: bad sizes");
  BDE_REQUIRE(tok_map != nullptr && w != nullptr && out != nullptr, "bde_window_reduce: null pointer");
  FramePtrs8 fp;
  for (int i = 0; i < 8; ++i) fp.f[i] = i < D ? frames_host[i] : nullptr;
  const size_t rows = (size_t)n_win * D * X;
  if (rows == 0) return 0;
  window_reduce_kernel<<<(unsigned)ceil_div(rows * 32, 256), 256, 0, s>>>(fp, D, tok_map, n_tok, c, X, w, b, out, rows);
  return check_launch("window_reduce_kernel");
}

extern "C" int bde_ln_gather(const float* const* frames_host, int D, const int* tok_map, int n_win, int n_tok, int c,
                             const float* gamma, const float* beta, void* out, int dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(D >= 1 && D <= 8, "bde_ln_gather: D must be in [1, 8]");
  BDE_REQUIRE(c <= 32 * kMaxPerLane, "bde_ln_gather: c too large");
  FramePtrs fp;
  for (int i = 0; i < 8; ++i) fp.f[i] = i < D ? frames_host[i] : nullptr;
  size_t rows = (size_t)n_win * D * n_tok;
  if (rows == 0) return 0;
  unsigned blocks = (unsigned)ceil_div(rows * 32, 256);
  if (dtype == BDE_F32)
    ln_gather_kernel<float><<<blocks, 256, 0, s>>>(fp, D, tok_map, n_tok, c, gamma, beta, (float*)out, rows);
  else
    ln_gather_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(fp, D, tok_map, n_tok, c, gamma, beta, (__nv_bfloat16*)out, rows);
  return check_launch("ln_gather_kernel");
}

template <typename T>
static int launch_ln_gather_qkv(const FramePtrs& fp, int D, int q_slot, const int* tok_map, int n_tok, int c,
                                const float* g_kv, const float* b_kv, const float* g_q, const float* b_q, void* out_kv,
                                void* out_q, size_t rows, cudaStream_t s) {
#define BDE_LNQKV(LPT_)                                                                                              \
  ln_gather_qkv_kernel<T, LPT_><<<(unsigned)ceil_div(ceil_div(rows, 32 / LPT_) * 32, 256), 256, 0, s>>>(                \
      fp, D, q_slot, tok_map, n_tok, g_kv, b_kv, g_q, b_q, (T*)out_kv, (T*)out_q, rows)
  if (c == 64) BDE_LNQKV(8);
  else if (c == 128) BDE_LNQKV(16);
  else if (c == 256) BDE_LNQKV(32);
  else BDE_REQUIRE(false, "bde_ln_gather_qkv: c must be 64, 128 or 256 (use bde_ln_gather otherwise)");
#undef BDE_LNQKV
  return check_launch("ln_gather_qkv_kernel");
}

extern "C" int bde_ln_gather_qkv(const float* const* frames_host, int D, int q_slot, const int* tok_map, int n_win,
                                 int n_tok, int c, const float* g_kv, const float* b_kv, const float* g_q,
                                 const float* b_q, void* out_kv, void* out_q, int dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(D >= 1 && D <= 8 && q_slot >= 0 && q_slot < D, "bde_ln_gather_qkv: bad D / q_slot");
  FramePtrs fp;
  for (int i = 0; i < 8; ++i) fp.f[i] = i < D ? frames_host[i] : nullptr;
  size_t rows = (size_t)n_win * D * n_tok;
  if (rows == 0) return 0;
  if (dtype == BDE_F32)
    return launch_ln_gather_qkv<float>(fp, D, q_slot, tok_map, n_tok, c, g_kv, b_kv, g_q, b_q, out_kv, out_q, rows, s);
  return launch_ln_gather_qkv<__nv_bfloat16>(fp, D, q_slot, tok_map, n_tok, c, g_kv, b_kv, g_q, b_q, out_kv, out_q, rows, s);
}

extern "C" int bde_layernorm(const float* x, size_t rows, int c, const float* gamma, const float* beta, void* out,
                             int dtype, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  BDE_REQUIRE(c <= 32 * kMaxPerLane, "bde_layernorm: c too large");
  if (rows == 0) return 0;
  if (c == 64 || c == 128 || c == 256) {
    // vectorised path: the plain-rows case of the gather kernel (identity map, one "frame")
    FramePtrs fp;
    for (int i = 0; i < 8; ++i) fp.f[i] = i == 0 ? x : nullptr;
    if (dtype == BDE_F32)
      return launch_ln_gather_qkv<float>(fp, 1, 0, nullptr, 1, c, gamma, beta, gamma, beta, out, nullptr, rows, s);
    return launch_ln_gather_qkv<__nv_bfloat16>(fp, 1, 0, nullptr, 1, c, gamma, beta, gamma, beta, out, nullptr, rows, s);
  }
  unsigned blocks = (unsigned)ceil_div(rows * 32, 256);
  if (dtype == BDE_F32)
    layernorm_kernel<float><<<blocks, 256, 0, s>>>(x, rows, c, gamma, beta, (float*)out);
  else
    layernorm_kernel<__nv_bfloat16><<<blocks, 256, 0, s>>>(x, rows, c, gamma, beta, (__nv_bfloat16*)out);
  return check_launch("layernorm_kernel");
}

extern "C" int bde_cast(const void* src, int src_dtype, void* dst, int dst_dtype, size_t n, void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n == 0) return 0;
  unsigned blocks = (unsigned)ceil_div(n, 256);
  if (src_dtype == BDE_F32 && dst_dtype == BDE_BF16)
    cast_kernel<float, __nv_bfloat16><<<blocks, 256, 0, s>>>((const float*)src, (__nv_bfloat16*)dst, n);
  else if (src_dtype == BDE_BF16 && dst_dtype == BDE_F32)
    cast_kernel<__nv_bfloat16, float><<<blocks, 256, 0, s>>>((const __nv_bfloat16*)src, (float*)dst, n);
  else if (src_dtype == BDE_F32 && dst_dtype == BDE_F32)
    cast_kernel<float, float><<<blocks, 256, 0, s>>>((const float*)src, (float*)dst, n);
  else
    BDE_REQUIRE(false, "bde_cast: unsupported dtype pair");
  return check_launch("cast_kernel");
}
