// Shared pieces of the tcgen05 implicit-GEMM kernels: parameters, PTX wrappers, tile geometry,
// UMMA descriptors and the fused quad epilogue.  Included by gemm_tc.cu (one tile per CTA), gemm_tc_conv.cu
// (persistent TMA-fed convolutions with an overlapped epilogue) and mlp_fused.cu.
#pragma once
#include <cuda.h>
#include <cudaTypedefs.h>

#include "common.cuh"

namespace bde {
namespace tc {

constexpr int BM = 128;
constexpr int BK = 64;  // bf16 elements = 128 bytes = one swizzle row
constexpr int kNumProducerWarps = 8;
constexpr int kNumProducerThreads = kNumProducerWarps * 32;
constexpr int kRowsPerThread = BM / (kNumProducerWarps * 4);  // 4
constexpr int kThreads = kNumProducerThreads + 64;
constexpr int kTmaWarp = kNumProducerWarps, kMmaWarp = kNumProducerWarps + 1;

struct TcParams {
  const __nv_bfloat16* a0;
  const __nv_bfloat16* a1;
  const __nv_bfloat16* w;  // only used when !kBTma
  const float* bias;
  int c0, c1, ctot;
  int n_img, h_in, w_in, h_out, w_out, ksize, stride, pad;
  int M, N, K, w_ld, num_kb;
  int tiles_x, tiles_y;  // > 0: M tiles are 8 x 16 output-pixel patches (L1-friendly halo reuse); 0: 128 consecutive pixels
  uint32_t ypat_all;     // bit (ky * ksize) set for every ky: multiplying by an x-bit mask replicates it per row
  int dense;             // 1x1, stride 1, pad 0: A is a plain [M, K] matrix
  int k_order;           // 0: k = (tap, channel);  1: k = (64-channel chunk, tap, channel in chunk)
  int epi, act, out_f32;
  void* out;
  void* out2;
  const void* residual;
  int res_mode;
  const float* c_prev;
  float* c_out;
  const int* row_map;
  // LayerNorm-gather A operand (kLn kernels): A[m, :] = (x - mean) / sqrt(var + 1e-5) of the fp32 row that
  // token m = (win, d, tok) maps to (affine folded into the weights by the caller); zero tokens stay 0.
  const float* ln_f[8];
  const int* ln_map;
  int ln_D, ln_ntok;
  long long* dbg;  // optional per-CTA phase timestamps (clock64), 8 slots per CTA, for bring-up profiling
};

#define BDE_DBG(slot)                                                                     \
  do {                                                                                    \
    if (p.dbg != nullptr) p.dbg[((size_t)blockIdx.y * gridDim.x + blockIdx.x) * 8 + (slot)] = clock64(); \
  } while (0)

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
// Same wait with a sleep between polls, for the single-purpose warps (TMA producer, MMA issuer) whose waits are long: a warp
// spinning on try_wait is always ready to issue and takes the scheduler slots of the worker warps on its sub-partition.
__device__ __forceinline__ void mbar_wait_backoff(uint32_t bar, uint32_t parity, uint32_t ns = 64) {
  uint32_t done = 0;
  while (true) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (done) break;
    __nanosleep(ns);
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
// arrive on `bar` once all cp.async issued so far by this thread have landed (counted in the
// barrier's expected arrivals: .noinc)
__device__ __forceinline__ void cp_async_mbar_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// Guard for single-thread tcgen05 / TMA issue.  With a predicate that comes from elect.sync ptxas emits the
// uniform-datapath instructions (UTCHMMA, UTCBAR, UTMALDG) directly; under `if (lane == 0)` it wraps each of them in an
// ELECT ... BRA.U.ANY waterfall loop (~40 issue cycles apiece).  True in exactly one (the lowest) lane of the converged warp
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred P1;\n\t"
      "elect.sync _|P1, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P1;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 x bf16 -> fp32
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows of 128 bytes, 8-row groups 1024 bytes apart.
// (cute::UMMA::SmemDescriptor: start[0,14) LBO[16,30) SBO[32,46) version[46,48)=1 layout[61,64)=2)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
  d |= (uint64_t)1 << 16;            // leading byte offset (ignored for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;  // stride byte offset: 8 rows * 128 B
  d |= (uint64_t)1 << 46;            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;            // SWIZZLE_128B
  return d;
}
// cute::UMMA::InstrDescriptor for kind::f16: c=F32 [4,6)=1, a=BF16 [7,10)=1, b=BF16 [10,13)=1,
// a/b K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

constexpr int kTileH = 8, kTileW = 16;  // 2-D M tile (kTileH * kTileW == BM)

// M-tile geometry.  The CTA-uniform part (integer divisions) is computed once; mapping a tile row to
// its output pixel is then a handful of adds.  Three modes:
//   2-D    : the tile is an 8 x 16 patch of output pixels of one image (convolutions)
//   dense  : 1x1 / stride 1 / no padding: the "pixel" index is the row index itself (linear layers)
//   linear : 128 consecutive output pixels in raster order (small images)
struct TileGeom {
  int img, oy0, ox0;  // 2-D mode
  int m0;             // dense / linear mode
  __device__ __forceinline__ void init(const TcParams& p, int tile) {
    img = oy0 = ox0 = 0;
    m0 = tile * BM;
    if (p.tiles_x > 0) {
      const int per_img = p.tiles_x * p.tiles_y;
      img = tile / per_img;
      const int t = tile - img * per_img;
      const int ty = t / p.tiles_x;
      oy0 = ty * kTileH;
      ox0 = (t - ty * p.tiles_x) * kTileW;
    }
  }
  // returns false for rows outside the problem; m = linear output index (epilogue addressing)
  __device__ __forceinline__ bool row_pixel(const TcParams& p, int row, int& im, int& oy, int& ox, int& m) const {
    if (p.tiles_x > 0) {
      im = img;
      oy = oy0 + (row >> 4);
      ox = ox0 + (row & 15);
      m = (im * p.h_out + oy) * p.w_out + ox;
      return oy < p.h_out && ox < p.w_out;
    }
    m = m0 + row;
    if (m >= p.M) return false;
    if (p.dense) {  // no spatial structure needed
      im = 0; oy = m; ox = 0;
      return true;
    }
    const int hw = p.h_out * p.w_out;
    im = m / hw;
    const int rem = m - im * hw;
    oy = rem / p.w_out;
    ox = rem - oy * p.w_out;
    return true;
  }
};

// kDeep = false: few stages so that two CTAs share an SM (mainloop of one overlaps the epilogue of the
//                other) -- used for linear layers, whose A operand has no reuse.
// kDeep = true : one CTA per SM with a deep pipeline; the smaller shared-memory carve-out leaves
//                >= 64 KB of L1 so that the im2col re-reads of a 2-D pixel tile (each input pixel is
//                needed by up to k*k taps) are served by L1 instead of L2.
// kLn = true : the LayerNorm-gather producer fills all K blocks of the tile at once (K = C <= 256), so it
//                needs >= 4 stages.
template <int BN, bool kDeep, int kLn = 0>
struct TileCfg {
  static constexpr int kStages = kLn > 0 ? kLn : kDeep ? (BN >= 256 ? 4 : (BN >= 128 ? 5 : (BN >= 64 ? 6 : 8)))
                                       : (BN >= 256 ? 4 : (BN >= 128 ? 3 : 4));
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStageBytes = kABytes + kBBytes;
  // the epilogue transposes its accumulator chunks in the operand region (8 producer warps x 32 rows x 36 floats) once the
  // main loop is done; a one-stage LayerNorm tile with BN <= 128 has fewer operand bytes than that
  static constexpr int kEpiBytes = kNumProducerWarps * 32 * 36 * 4;
  static constexpr int kOperandBytes = kStages * kStageBytes > kEpiBytes ? kStages * kStageBytes : kEpiBytes;
  static constexpr int kSmemBytes = kOperandBytes + 1024 /*align slack*/ + 256 /*barriers*/ + BN * 4 /*bias*/;
  static constexpr int kTmemCols = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));
};

// fast transcendental forms for the bf16 path (relative error ~1e-6, far below bf16 resolution)
__device__ __forceinline__ float fast_sigmoid(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }
__device__ __forceinline__ float fast_tanh(float x) { return 1.0f - __fdividef(2.0f, __expf(2.0f * x) + 1.0f); }
// single-MUFU forms for the ConvLSTM gate math (tanh.approx.f32: max relative error 2^-11, a quarter of the bf16
// rounding that h undergoes anyway): sigmoid(x) = 0.5 tanh(x / 2) + 0.5.  5 MUFU per cell instead of 10.
__device__ __forceinline__ float mufu_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float mufu_sigmoid(float x) { return fmaf(mufu_tanh(0.5f * x), 0.5f, 0.5f); }

// Exact-erf GELU (DTransformer.py:345-346, nn.GELU approximate='none') for the bf16 path, as x * sigmoid(p(x)) with an
// odd degree-5 polynomial p fitted (minimax over [-6, 6], scipy least squares) to the logit of the normal CDF
// (|error of the form| <= 5.4e-5), and sigmoid(p) = 0.5 + 0.5 tanh(p / 2) so that ONE MUFU op (tanh.approx, relative
// error 2^-11) serves an element: the ex2 + rcp form kept the XU pipe busy for 2 x 8 cycles per warp instruction and made
// the GELU epilogues of both fused MLP kernels MUFU-bound (4 K cycles per 128 x 128 chunk, round-2 phase counters).
// Absolute error <= 0.5 |x| 2^-11, below the bf16 rounding (2^-9 |gelu|) except in the far negative tail where it stays
// under 1.3e-3.  The fp32 parity engine keeps erff.
__device__ __forceinline__ float fast_gelu(float x) {
  const float x2 = fminf(x * x, 25.0f);   // beyond |x| = 5 the polynomial factor is frozen: the argument stays monotone and tanh saturates
  const float r = x * fmaf(x2, fmaf(x2, -3.81888e-4f, 3.72153e-2f), 7.972375e-1f);   // p(x) / 2
  const float h = 0.5f * x;
  return fmaf(h, mufu_tanh(r), h);
}

__device__ __forceinline__ uint4 pack8_bf16(const float* v) {
  uint4 pk;
  __nv_bfloat162 t0 = __floats2bfloat162_rn(v[0], v[1]);
  __nv_bfloat162 t1 = __floats2bfloat162_rn(v[2], v[3]);
  __nv_bfloat162 t2 = __floats2bfloat162_rn(v[4], v[5]);
  __nv_bfloat162 t3 = __floats2bfloat162_rn(v[6], v[7]);
  pk.x = *reinterpret_cast<uint32_t*>(&t0);
  pk.y = *reinterpret_cast<uint32_t*>(&t1);
  pk.z = *reinterpret_cast<uint32_t*>(&t2);
  pk.w = *reinterpret_cast<uint32_t*>(&t3);
  return pk;
}

// ------------------------------------------------------------------------------------------
// Epilogue on 4 consecutive columns [nb, nb+4) of output row m (after the shared-memory transpose every
// lane owns such a quad, 8 lanes cover 32 contiguous columns of one row -> coalesced global traffic).
// For the LSTM epilogue the quad is exactly (in, remember, out, cell) of hidden channel nb / 4.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void epilogue_quad(const TcParams& p, int m, int nb, float4 acc, float4 b, int dst_row) {
  float v0 = acc.x + b.x, v1 = acc.y + b.y, v2 = acc.z + b.z, v3 = acc.w + b.w;
  if (p.epi == BDE_EPI_STORE) {
    const size_t o = (size_t)m * p.N + nb;
    if (p.res_mode == 1 && p.residual != nullptr) {  // pre-activation residual in the operand type (bf16)
      const uint2 rr = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p.residual) + o);
      const float2 r0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rr.x));
      const float2 r1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rr.y));
      v0 += r0.x; v1 += r0.y; v2 += r1.x; v3 += r1.y;
    }
    if (p.act == BDE_ACT_RELU) {
      v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f);
    } else if (p.act == BDE_ACT_RELU6) {
      v0 = fminf(fmaxf(v0, 0.f), 6.f); v1 = fminf(fmaxf(v1, 0.f), 6.f);
      v2 = fminf(fmaxf(v2, 0.f), 6.f); v3 = fminf(fmaxf(v3, 0.f), 6.f);
    } else if (p.act == BDE_ACT_GELU) {
      v0 = fast_gelu(v0); v1 = fast_gelu(v1); v2 = fast_gelu(v2); v3 = fast_gelu(v3);
    } else if (p.act != BDE_ACT_NONE) {
      v0 = apply_act(v0, p.act); v1 = apply_act(v1, p.act); v2 = apply_act(v2, p.act); v3 = apply_act(v3, p.act);
    }
    if (p.res_mode == 0 && p.residual != nullptr) {
      const float4 r = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.residual) + o);
      v0 += r.x; v1 += r.y; v2 += r.z; v3 += r.w;
    }
    if (p.out_f32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + o) = make_float4(v0, v1, v2, v3);
    __nv_bfloat16* dstb = p.out_f32 ? reinterpret_cast<__nv_bfloat16*>(p.out2) : reinterpret_cast<__nv_bfloat16*>(p.out);
    if (dstb != nullptr) {
      const __nv_bfloat162 t0 = __floats2bfloat162_rn(v0, v1), t1 = __floats2bfloat162_rn(v2, v3);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&t0);
      pk.y = *reinterpret_cast<const uint32_t*>(&t1);
      *reinterpret_cast<uint2*>(dstb + o) = pk;
    }
  } else if (p.epi == BDE_EPI_LSTM) {
    // (submodules.py:320-332)  c = sig(remember) * c_prev + sig(in) * tanh(cell);  h = sig(out) * tanh(c)
    const size_t o = (size_t)m * (p.N >> 2) + (nb >> 2);
    const float cprev = p.c_prev != nullptr ? p.c_prev[o] : 0.f;
    const float c = fast_sigmoid(v1) * cprev + fast_sigmoid(v0) * fast_tanh(v3);
    const float h = fast_sigmoid(v2) * fast_tanh(c);
    p.c_out[o] = c;
    reinterpret_cast<__nv_bfloat16*>(p.out)[o] = __float2bfloat16_rn(h);
  } else {  // BDE_EPI_SCATTER
    if (dst_row >= 0) {
      float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (size_t)dst_row * p.N + nb);
      float4 cur = *dst;
      cur.x += v0; cur.y += v1; cur.z += v2; cur.w += v3;
      *dst = cur;
    }
  }
}

// ---- epilogue with pre-fetched auxiliary operand --------------------------------------------------------------
// The global READS of an epilogue (LSTM: c_prev; STORE: fp32 or pre-activation residual; SCATTER: the destination's
// current value) alias the kernel's own stores as far as the compiler can tell, so inside an unrolled row loop every
// read would wait for the previous row's store to issue and for its own latency: ~700 cycles x rows.  The callers
// therefore fetch the operand of all 8 rows of a chunk up front (aux_load, independent loads in flight together) and
// hand it to the math here.
__device__ __forceinline__ float4 aux_load(const TcParams& p, int m, int nb, int dst_row) {
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  if (p.epi == BDE_EPI_LSTM) {
    if (p.c_prev != nullptr) a.x = p.c_prev[(size_t)m * (p.N >> 2) + (nb >> 2)];
  } else if (p.epi == BDE_EPI_GRU_UR) {   // h_prev of the two hidden channels of this quad
    if (p.c_prev != nullptr) {
      const float2 h2 = *reinterpret_cast<const float2*>(p.c_prev + (size_t)m * (p.N >> 1) + (nb >> 1));
      a.x = h2.x; a.y = h2.y;
    }
  } else if (p.epi == BDE_EPI_GRU_OUT) {  // h_prev of the four hidden channels
    if (p.c_prev != nullptr) a = *reinterpret_cast<const float4*>(p.c_prev + (size_t)m * p.N + nb);
  } else if (p.epi == BDE_EPI_STORE) {
    if (p.residual != nullptr) {
      const size_t o = (size_t)m * p.N + nb;
      if (p.res_mode == 1) {
        const uint2 rr = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p.residual) + o);
        const float2 r0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rr.x));
        const float2 r1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&rr.y));
        a = make_float4(r0.x, r0.y, r1.x, r1.y);
      } else {
        a = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.residual) + o);
      }
    }
  } else if (p.epi == BDE_EPI_SCATTER && dst_row >= 0) {
    a = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.out) + (size_t)dst_row * p.N + nb);
  }
  return a;
}

__device__ __forceinline__ void epilogue_quad_aux(const TcParams& p, int m, int nb, float4 acc, float4 b, int dst_row, float4 aux) {
  float v0 = acc.x + b.x, v1 = acc.y + b.y, v2 = acc.z + b.z, v3 = acc.w + b.w;
  if (p.epi == BDE_EPI_STORE) {
    const size_t o = (size_t)m * p.N + nb;
    if (p.res_mode == 1) { v0 += aux.x; v1 += aux.y; v2 += aux.z; v3 += aux.w; }
    if (p.act == BDE_ACT_RELU) {
      v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); v2 = fmaxf(v2, 0.f); v3 = fmaxf(v3, 0.f);
    } else if (p.act == BDE_ACT_RELU6) {
      v0 = fminf(fmaxf(v0, 0.f), 6.f); v1 = fminf(fmaxf(v1, 0.f), 6.f);
      v2 = fminf(fmaxf(v2, 0.f), 6.f); v3 = fminf(fmaxf(v3, 0.f), 6.f);
    } else if (p.act == BDE_ACT_GELU) {
      v0 = fast_gelu(v0); v1 = fast_gelu(v1); v2 = fast_gelu(v2); v3 = fast_gelu(v3);
    } else if (p.act != BDE_ACT_NONE) {
      v0 = apply_act(v0, p.act); v1 = apply_act(v1, p.act); v2 = apply_act(v2, p.act); v3 = apply_act(v3, p.act);
    }
    if (p.res_mode == 0) { v0 += aux.x; v1 += aux.y; v2 += aux.z; v3 += aux.w; }   // aux is zero without a residual
    if (p.out_f32) *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + o) = make_float4(v0, v1, v2, v3);
    __nv_bfloat16* dstb = p.out_f32 ? reinterpret_cast<__nv_bfloat16*>(p.out2) : reinterpret_cast<__nv_bfloat16*>(p.out);
    if (dstb != nullptr) {
      const __nv_bfloat162 t0 = __floats2bfloat162_rn(v0, v1), t1 = __floats2bfloat162_rn(v2, v3);
      uint2 pk;
      pk.x = *reinterpret_cast<const uint32_t*>(&t0);
      pk.y = *reinterpret_cast<const uint32_t*>(&t1);
      *reinterpret_cast<uint2*>(dstb + o) = pk;
    }
  } else if (p.epi == BDE_EPI_LSTM) {
    const size_t o = (size_t)m * (p.N >> 2) + (nb >> 2);
    const float c = fmaf(mufu_sigmoid(v1), aux.x, mufu_sigmoid(v0) * mufu_tanh(v3));
    const float h = mufu_sigmoid(v2) * mufu_tanh(c);
    p.c_out[o] = c;
    reinterpret_cast<__nv_bfloat16*>(p.out)[o] = __float2bfloat16_rn(h);
  } else if (p.epi == BDE_EPI_GRU_UR) {
    // ConvGRU, first conv (submodules.py:371-373): quad = (update, reset) of hidden channels nb/2, nb/2 + 1
    const size_t o = (size_t)m * (p.N >> 1) + (nb >> 1);
    *reinterpret_cast<float2*>(p.c_out + o) = make_float2(mufu_sigmoid(v0), mufu_sigmoid(v2));
    *reinterpret_cast<__nv_bfloat162*>(reinterpret_cast<__nv_bfloat16*>(p.out) + o) =
        __floats2bfloat162_rn(aux.x * mufu_sigmoid(v1), aux.y * mufu_sigmoid(v3));
  } else if (p.epi == BDE_EPI_GRU_OUT) {
    // ConvGRU, second conv (submodules.py:374-375): h' = h (1 - u) + tanh(out_gate) u
    const size_t o = (size_t)m * p.N + nb;
    const float4 u = __ldg(reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.residual) + o));
    const float h0 = fmaf(aux.x, 1.0f - u.x, mufu_tanh(v0) * u.x), h1 = fmaf(aux.y, 1.0f - u.y, mufu_tanh(v1) * u.y);
    const float h2 = fmaf(aux.z, 1.0f - u.z, mufu_tanh(v2) * u.z), h3 = fmaf(aux.w, 1.0f - u.w, mufu_tanh(v3) * u.w);
    *reinterpret_cast<float4*>(p.c_out + o) = make_float4(h0, h1, h2, h3);
    const __nv_bfloat162 t0 = __floats2bfloat162_rn(h0, h1), t1 = __floats2bfloat162_rn(h2, h3);
    uint2 pk;
    pk.x = *reinterpret_cast<const uint32_t*>(&t0);
    pk.y = *reinterpret_cast<const uint32_t*>(&t1);
    *reinterpret_cast<uint2*>(reinterpret_cast<__nv_bfloat16*>(p.out) + o) = pk;
  } else if (dst_row >= 0) {  // BDE_EPI_SCATTER
    *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (size_t)dst_row * p.N + nb) =
        make_float4(aux.x + v0, aux.y + v1, aux.z + v2, aux.w + v3);
  }
}

// host helpers implemented in gemm_tc.cu
int get_weight_tmap(const void* w, int n, int w_ld, int bn, CUtensorMap* out);
bool env_flag(const char* name, bool dflt);
bool b_via_tma();
// fills TcParams from the public descriptor (validation included); returns 0 or a negative error
int fill_params(const bde_gemm_desc* d, TcParams& p, bool& ln);
extern long long* g_dbg;
extern size_t g_dbg_ctas;

}  // namespace tc
}  // namespace bde
